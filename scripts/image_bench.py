#!/usr/bin/env python3
"""
Throughput of the bi-level image codec (bloom_compress drop-in) on one GPU.

A seeded batch of 4K-sized sparse-bright images -- half RGB 3840x2160x3, half grey 3840x2160, each group larger than the
126 MB L2, so K1 reads from HBM -- is coded with compress_images and decoded with decompress_images.  Reports one JSON line
(also written to <out>/image_bench.json):

  * compress_images: images/s and Mpx/s by wall clock (upload, encode, batched fetch and the host container assembly) and by
    device events (rbf_stream_stage_ms of the last encode of each group);
  * k_binarize: bytes moved (C*S bytes read + 1/8 byte written per pixel) over its event span, and that over the HBM peak
    (MEASURED_PEAKS.json when present, else bench.py's fallback -- the field says which);
  * decompress_images: images/s by wall clock over the payloads that decode.  The decoder takes k from the payload's float32
    (bc:427, 461), as the reference does; at 4K the rounded k often lets more positions pass than the witness holds and the
    reference raises IndexError -- the count of such payloads is reported;
  * parity: three images against the C coder (encode, and decode on the float32 k) and decode_verify (exact k) of both groups;
    how many decodable payloads come back equal to their mask is reported beside them;
  * the C coder's CPU time for one image (the single-threaded CPU arm);
  * the card name and power limit (nvidia-smi query).

    python scripts/image_bench.py --out DIR [--images 64] [--reps 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import measured_peaks  # noqa: E402
from tests.test_bloom_compress_host import binarize_image  # noqa: E402  (numpy restatement of bc:67-87)


def sparse_bright(shape, p, seed):
    rng = np.random.default_rng(seed)
    img = rng.integers(0, 100, shape, dtype=np.uint8)
    bright = rng.random(shape[:2]) < p
    img[bright] = 255
    return img


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:       # noqa: BLE001
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--images", type=int, default=64)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    from new_bloom_filter_repo_b200 import _cabi, bloom_compress as bcm
    from oracle import c_oracle as co

    H, W = 2160, 3840
    half = a.images // 2
    shapes = [(H, W, 3)] * half + [(H, W)] * (a.images - half)
    ps = [0.01, 0.02, 0.05, 0.1]
    imgs = [sparse_bright(s, ps[i % len(ps)], 500 + i) for i, s in enumerate(shapes)]
    npx = H * W * len(imgs)
    in_bytes = sum(im.nbytes for im in imgs)
    comp = bcm.BloomFilterCompressor()
    comp.max_batch_images, comp.max_batch_bytes = len(imgs), in_bytes      # one encode per group: decode_verify covers all of it

    payloads = comp.compress_images(imgs)                       # warm-up: module load, stream allocation
    streams = {k: st for k, st in comp._streams.streams.items() if k[2] > 0}          # the two encode streams (RGB, grey)
    verify = {str(k[:3]): int(st.decode_verify().sum()) for k, st in streams.items()}
    decodable = []
    for i, (p, _) in enumerate(payloads):
        try:
            comp.decompress_images([p])
            decodable.append(i)
        except IndexError:
            pass

    wall, dev, k1 = [], [], []
    for _ in range(a.reps):
        t0 = time.perf_counter()
        payloads = comp.compress_images(imgs)
        wall.append(time.perf_counter() - t0)
        st = [s.stage_ms() for s in streams.values()]
        dev.append(sum(s["encode_total"] for s in st) / 1e3)
        k1.append(sum(s["k1_threshold"] for s in st) / 1e3)
    dwall = []
    for _ in range(a.reps):
        t0 = time.perf_counter()
        decs = comp.decompress_images([payloads[i][0] for i in decodable])
        dwall.append(time.perf_counter() - t0)

    lossless = sum(np.array_equal(d.reshape(-1), binarize_image(imgs[i], 127) * 255) for d, i in zip(decs, decodable))
    oracle_ok, cpu_s = True, None
    for i in (0, half // 2, len(imgs) - 1):
        m = binarize_image(imgs[i], 127)
        t0 = time.perf_counter()
        ob, ow, op, on, oratio, ok, ol = co.compress(m, seeds=_cabi.BC_SEEDS)
        cpu_s = time.perf_counter() - t0 if cpu_s is None else cpu_s
        bitmap, witness, p, n, k, shape = comp._unpack_compressed_data(payloads[i][0])
        oracle_ok &= np.array_equal(bitmap, ob) and np.array_equal(np.asarray(witness, np.uint8), ow)
        out = np.zeros(n, dtype=np.uint8)
        bm, wt = np.ascontiguousarray(bitmap, np.uint8), np.ascontiguousarray(witness, np.uint8)
        used = co.lib().orc_decompress_kl(bm.ctypes.data, len(bm), wt.ctypes.data, len(wt), n, float(k), 0, 1, 999, out.ctypes.data)
        oracle_ok &= (used > len(wt)) == (i not in decodable)
        if i in decodable:
            oracle_ok &= np.array_equal(decs[decodable.index(i)].reshape(-1), out * 255)

    peak, peak_src = measured_peaks()
    k1_bytes = in_bytes + npx / 8
    best_wall, best_dev, best_k1, best_dec = min(wall), min(dev), min(k1), min(dwall)
    res = {
        "metric": "image_codec_4k", "card": card(), "images": len(imgs), "shape_rgb": [H, W, 3], "shape_grey": [H, W],
        "compress_images_per_s_wall": len(imgs) / best_wall, "compress_mpx_per_s_wall": npx / best_wall / 1e6,
        "compress_images_per_s_device": len(imgs) / best_dev, "compress_mpx_per_s_device": npx / best_dev / 1e6,
        "k_binarize_ms": best_k1 * 1e3, "k_binarize_gb_per_s": k1_bytes / best_k1 / 1e9,
        "k_binarize_share_of_hbm_peak": k1_bytes / best_k1 / 1e9 / peak, "hbm_peak_gb_per_s": peak, "hbm_peak_source": peak_src,
        "decompress_images_per_s_wall": len(decodable) / best_dec, "decode_payloads_timed": len(decodable),
        "decode_index_errors_float32_k": len(imgs) - len(decodable), "decoded_equal_to_mask": int(lossless),
        "cpu_c_coder_s_per_image": cpu_s, "cpu_c_coder_images_per_s": 1.0 / cpu_s,
        "parity": {"c_coder_3_images": bool(oracle_ok), "decode_verify_zero": all(v == 0 for v in verify.values())},
        "reps": a.reps, "wall_s": wall, "device_s": dev,
    }
    line = json.dumps(res)
    with open(os.path.join(a.out, "image_bench.json"), "w") as f:
        f.write(line + "\n")
    print(line)
    return 0 if all(res["parity"].values()) else 1


if __name__ == "__main__":
    sys.exit(main())
