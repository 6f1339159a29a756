#!/usr/bin/env python3
"""
Generates tests/golden/bc_kat.json and tests/golden/bc_arrays.npz from the REAL reference's bloom_compress.py (bc),
imported through oracle/refshim.py, for the bloom_compress drop-in:

    python tests/golden/make_golden_bc.py

Everything stored is an output of unmodified reference code (numpy 2.3, Pillow 12.2, xxhash 3.7):
  * bc.BloomFilterCompressor._binarize_image masks for every supported layout and a threshold sweep
  * compress_image payloads (images saved as PNG, read back by the reference) and decompress_image outputs,
    plus one payload with its witness cut short (the reference raises IndexError)
  * compress_text / decompress_text payloads
  * the run_compression_tests vectors (n = 100 000, p = .1 .. .4), seeded
  * nested RationalBloomFilter probes / activation, and the stdout of one coded and one raw compress
"""
import contextlib
import hashlib
import io
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "..")))
from oracle import refshim  # noqa: E402

ivc, rbf, bc, fvc = refshim.load()
from PIL import Image  # noqa: E402  (the reference's dependency)

BC = bc.BloomFilterCompressor


def sha(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def quiet(fn, *a, **kw):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **kw)


# (name, shape, dtype); ragged n everywhere so that the last mask word is partial
BIN_IMAGES = [("u8_37x53", (37, 53), "uint8"), ("rgb_48x80", (48, 80, 3), "uint8"), ("rgba_48x80", (48, 80, 4), "uint8"),
              ("la_33x65", (33, 65, 2), "uint8"), ("one_40x72", (40, 72, 1), "uint8"), ("u16_40x72", (40, 72), "uint16"),
              ("bool_16x16", (16, 16), "bool")]
THRESHOLDS = [127, 0, 254, 255, -1, 300, 127.5, float("nan")]

# (name, PIL mode, channels, p of bright pixels): p = 0 and p = 0.4 take the raw branch
CODEC_IMAGES = [("L_p0", "L", 1, 0.0), ("L_p05", "L", 1, 0.05), ("RGB_p01", "RGB", 3, 0.01), ("RGB_p15", "RGB", 3, 0.15),
                ("RGBA_p05", "RGBA", 4, 0.05), ("RGBA_p30", "RGBA", 4, 0.30), ("LA_p10", "LA", 2, 0.10), ("L_p40", "L", 1, 0.40)]
CODEC_HW = (48, 64)


def bin_image(shape, dtype, seed):
    rng = np.random.default_rng(seed)
    if dtype == "bool":
        return rng.random(shape) < 0.3
    hi = 256 if dtype == "uint8" else 65536
    return rng.integers(0, hi, shape).astype(dtype)


def sparse_bright(ch, p, seed):
    """dark background with a fraction p of bright pixels (all channels bright)."""
    rng = np.random.default_rng(seed)
    h, w = CODEC_HW
    img = rng.integers(0, 100, (h, w, ch))
    bright = rng.random((h, w)) < p
    img[bright] = rng.integers(200, 256, (int(bright.sum()), ch))
    img = img.astype(np.uint8)
    return img[:, :, 0] if ch == 1 else img


def main():
    kat = {"binarize": [], "images": [], "text": [], "synthetic": [], "filters": [], "stdout": {}}
    arrays = {}
    for s, (name, shape, dt) in enumerate(BIN_IMAGES):
        img = bin_image(shape, dt, 1000 + s)
        arrays["bin_" + name] = img
        for t in THRESHOLDS:
            m = BC._binarize_image(img, t)
            kat["binarize"].append({"image": name, "threshold": repr(t), "sha": sha(m.astype(np.uint8)),
                                    "ones": int(m.sum()), "n": int(m.size)})
    comp = BC()
    with tempfile.TemporaryDirectory() as td:
        for s, (name, mode, ch, p) in enumerate(CODEC_IMAGES):
            img = sparse_bright(ch, p, 2000 + s)
            path = os.path.join(td, name + ".png")
            Image.fromarray(img, mode=mode).save(path)
            loaded = np.array(Image.open(path))
            assert np.array_equal(loaded, img)
            arrays["img_" + name] = loaded
            data, ratio = quiet(comp.compress_image, path, 127)
            dec = quiet(comp.decompress_image, data)
            kat["images"].append({"name": name, "mode": mode, "payload": data.hex(), "ratio": ratio.hex() if isinstance(ratio, float) else float(ratio).hex(),
                                  "decoded_sha": sha(dec), "decoded_dtype": str(dec.dtype), "decoded_shape": list(dec.shape)})
    # a coded payload with the witness cut short: the decoder runs past the end of the witness list
    coded = next(r for r in kat["images"] if r["name"] == "RGB_p15")
    short = bytes.fromhex(coded["payload"])[:-3]
    try:
        quiet(comp.decompress_image, short)
        err = None
    except Exception as e:      # noqa: BLE001
        err = type(e).__name__
    assert err == "IndexError", err
    kat["short_witness"] = {"payload": short.hex(), "error": err}

    ctrl = "".join(np.random.default_rng(7).choice(["\x00", "\x01", "\x02", "\x04", "\x08", "\x10"], 300))
    for name, text, depth in [("ascii", "The quick brown fox jumps over the lazy dog. " * 4, 8), ("utf8_16", "Grüße, 世界! ∑ω", 16),
                              ("nonascii_8", "naïve café ☕", 8), ("control", ctrl, 8), ("empty", "", 8)]:
        data, ratio = quiet(comp.compress_text, text, depth)
        back = quiet(comp.decompress_text, data)
        kat["text"].append({"name": name, "text": text, "bit_depth": depth, "payload": data.hex(), "ratio": float(ratio).hex(),
                            "decoded": back})

    n = 100000
    for i, p in enumerate([0.1, 0.2, 0.3, 0.4]):
        seed = 3000 + i
        x = (np.random.default_rng(seed).random(n) < p).astype(np.uint8)
        bm, wit, dens, nn, ratio = quiet(comp.compress, x)
        k, l = BC._calculate_optimal_params(n, dens)
        dec = quiet(comp.decompress, bm, wit, nn, k)
        kat["synthetic"].append({"seed": seed, "n": n, "p_gen": p, "density": float(dens).hex(), "ratio": float(ratio).hex(),
                                 "k": float(k).hex(), "l": int(l), "bitmap_sha": sha(np.asarray(bm, dtype=np.uint8)),
                                 "witness_len": len(wit), "witness_sha": sha(np.asarray(wit, dtype=np.uint8)),
                                 "lossless": bool(np.array_equal(x, dec))})

    for size, k in [(1000, 2.3), (997, 3.0), (65536, 4.71), (12345, 0.4)]:
        f = BC.RationalBloomFilter(size, k)
        items = list(range(0, 60)) + [99, 100, 101, 12345, 999999, 4294967295]
        kat["filters"].append({"size": size, "k": k, "items": items,
                               "probes": [[int(f._get_hash_indices(it, i)) for i in range(f.floor_k + 1)] for it in items],
                               "activation": [bool(f._determine_activation(it)) for it in items]})

    for name, p in [("coded", 0.05), ("raw", 0.4)]:
        x = (np.random.default_rng(4000).random(5000) < p).astype(np.uint8)
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            comp.compress(x)
        kat["stdout"][name] = {"seed": 4000, "n": 5000, "p_gen": p, "text": buf.getvalue()}

    with open(os.path.join(HERE, "bc_kat.json"), "w") as f:
        json.dump(kat, f, indent=0, sort_keys=True)
    np.savez_compressed(os.path.join(HERE, "bc_arrays.npz"), **arrays)
    print("wrote bc_kat.json, bc_arrays.npz")


if __name__ == "__main__":
    main()
