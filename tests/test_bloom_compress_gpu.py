"""GPU tests of the bloom_compress drop-in (bloom_compress.py, bc): k_binarize against the reference's masks, compress_image /
decompress_image / text payloads byte-exact against the reference's, the batch API against the one-image calls, the image
stream at 4K-class sizes against the C coder, and the refusals of image streams."""
import contextlib
import io

import numpy as np
import pytest

from tests.test_bloom_compress_host import _threshold, binarize_image
from tests.util import golden_json, golden_npz, sha

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def bcm():
    from new_bloom_filter_repo_b200 import bloom_compress
    return bloom_compress


@pytest.fixture()
def comp(bcm):
    return bcm.BloomFilterCompressor()


def quiet(fn, *a, **kw):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **kw)


def test_binarize_fixture(bcm):
    kat, arr = golden_json("bc_kat.json"), golden_npz("bc_arrays.npz")
    for rec in kat["binarize"]:
        m = bcm.BloomFilterCompressor._binarize_image(arr["bin_" + rec["image"]], _threshold(rec))
        assert m.dtype == np.uint8 and m.size == rec["n"]
        assert (sha(m), int(m.sum())) == (rec["sha"], rec["ones"]), rec


def test_image_payloads_fixture(comp):
    kat, arr = golden_json("bc_kat.json"), golden_npz("bc_arrays.npz")
    imgs = [arr["img_" + r["name"]] for r in kat["images"]]
    for rec, img in zip(kat["images"], imgs):
        data, ratio = quiet(comp.compress_image, img, 127)
        assert data.hex() == rec["payload"], rec["name"]
        assert float(ratio).hex() == rec["ratio"], rec["name"]
        dec = comp.decompress_image(data)
        assert (sha(dec), str(dec.dtype), list(dec.shape)) == (rec["decoded_sha"], rec["decoded_dtype"], rec["decoded_shape"])
    batch = comp.compress_images(imgs)
    assert [d.hex() for d, _ in batch] == [r["payload"] for r in kat["images"]]
    decs = comp.decompress_images([d for d, _ in batch])
    assert [sha(d) for d in decs] == [r["decoded_sha"] for r in kat["images"]]


def test_compress_image_path_form(comp, tmp_path):
    Image = pytest.importorskip("PIL.Image")
    kat, arr = golden_json("bc_kat.json"), golden_npz("bc_arrays.npz")
    for rec in kat["images"]:
        path = tmp_path / (rec["name"] + ".png")
        Image.fromarray(arr["img_" + rec["name"]], mode=rec["mode"]).save(path)
        out = tmp_path / (rec["name"] + ".bloom")
        data, _ = quiet(comp.compress_image, str(path), 127, str(out))
        assert data.hex() == rec["payload"] and out.read_bytes() == data
        png = tmp_path / (rec["name"] + "_dec.png")
        dec = comp.decompress_image(data, str(png))
        assert np.array_equal(np.array(Image.open(png)), dec)


def test_corrupt_payload_raises_index_error(comp):
    kat = golden_json("bc_kat.json")
    short = bytes.fromhex(kat["short_witness"]["payload"])
    with pytest.raises(IndexError):
        comp.decompress_image(short)
    good = bytes.fromhex(kat["images"][1]["payload"])
    with pytest.raises(IndexError):
        comp.decompress_images([good, short])
    # a well-formed container whose witness is too short for its filter: caught on the batched device path
    bitmap, witness, p, n, k, shape = comp._unpack_compressed_data(bytes.fromhex(kat["images"][3]["payload"]))
    cut = comp._pack_compressed_data(bitmap, witness[:len(witness) // 2], p, n, k, shape)
    with pytest.raises(IndexError):
        comp.decompress_images([good, cut])


def test_text_fixture(comp):
    kat = golden_json("bc_kat.json")
    for rec in kat["text"]:
        data, ratio = quiet(comp.compress_text, rec["text"], rec["bit_depth"])
        assert data.hex() == rec["payload"], rec["name"]
        assert float(ratio).hex() == rec["ratio"]
        assert comp.decompress_text(data) == rec["decoded"]


def test_synthetic_vectors_and_stdout(comp):
    kat = golden_json("bc_kat.json")
    for rec in kat["synthetic"]:
        x = (np.random.default_rng(rec["seed"]).random(rec["n"]) < rec["p_gen"]).astype(np.uint8)
        bm, wit, dens, n, ratio = quiet(comp.compress, x)
        assert (float(dens).hex(), float(ratio).hex()) == (rec["density"], rec["ratio"])
        assert sha(np.asarray(bm, dtype=np.uint8)) == rec["bitmap_sha"]
        assert (len(wit), sha(np.asarray(wit, dtype=np.uint8))) == (rec["witness_len"], rec["witness_sha"])
        k, l = comp._calculate_optimal_params(n, dens)
        assert (float(k).hex(), l) == (rec["k"], rec["l"])
        assert np.array_equal(comp.decompress(bm, wit, n, k), x) == rec["lossless"]
    for rec in kat["stdout"].values():
        x = (np.random.default_rng(rec["seed"]).random(rec["n"]) < rec["p_gen"]).astype(np.uint8)
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            comp.compress(x)
        assert buf.getvalue() == rec["text"]


def test_nested_filter(bcm):
    for rec in golden_json("bc_kat.json")["filters"]:
        f = bcm.BloomFilterCompressor.RationalBloomFilter(rec["size"], rec["k"])
        for it, probes, act in zip(rec["items"], rec["probes"], rec["activation"]):
            assert [f._get_hash_indices(it, i) for i in range(f.floor_k + 1)] == probes
            assert f._determine_activation(it) == act


def c_decode(bitmap, witness, n, k):
    """The C decoder (bc:307-346 with bc's seeds) -> (mask, Bloom-test passes)."""
    import ctypes as C
    from oracle import c_oracle as co
    bm = np.ascontiguousarray(bitmap, dtype=np.uint8)
    wt = np.ascontiguousarray(witness, dtype=np.uint8)
    out = np.zeros(n, dtype=np.uint8)
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)       # noqa: E731
    consumed = co.lib().orc_decompress_kl(ptr(bm), len(bm), ptr(wt), len(wt), n, float(k), 0, 1, 999, ptr(out))
    return out, int(consumed)


def _sparse(shape, p, seed, dtype=np.uint8):
    rng = np.random.default_rng(seed)
    hi = 100 if dtype == np.uint8 else 20000
    img = rng.integers(0, hi, shape).astype(dtype)
    bright = rng.random(shape[:2]) < p
    img[bright] = np.iinfo(dtype).max
    return img


def test_batch_equals_single_across_chunks_and_shapes(comp):
    imgs = [_sparse((40, 72, 3), 0.05, 1), _sparse((33, 65), 0.1, 2), _sparse((40, 72, 3), 0.2, 3), _sparse((33, 65), 0.0, 4),
            _sparse((40, 72, 3), 0.4, 5), _sparse((40, 72, 3), 0.01, 6), _sparse((33, 65), 0.05, 7, np.uint16),
            _sparse((40, 72, 3), 0.12, 8), _sparse((20, 30, 4), 0.07, 9), np.zeros((0, 5), np.uint8)]
    single = [quiet(comp.compress_image, im, 100) for im in imgs]
    comp.max_batch_images = 3                              # three chunks of the (40, 72, 3) group
    batch = comp.compress_images(imgs, threshold=100)
    assert [(d, r) for d, r in batch] == single
    payloads = [d for d, _ in batch[:-1]]
    decs = comp.decompress_images(payloads)
    for im, d in zip(imgs, decs):
        assert np.array_equal(d, binarize_image(im, 100).reshape(im.shape[:2]) * 255)
        assert d.dtype == np.uint8


@pytest.mark.parametrize("shape", [(2048, 2048, 3), (2160, 3840), (4096, 4096, 4)])
def test_image_stream_at_scale(shape):
    from new_bloom_filter_repo_b200 import FrameStream, _cabi
    from new_bloom_filter_repo_b200 import bloom_compress as bcm
    from oracle import c_oracle as co
    ps = [5e-5, 0.01, 0.05, 0.2, 0.4]
    imgs = np.stack([_sparse(shape, p, 100 + i) for i, p in enumerate(ps)])
    h, w = shape[:2]
    ch = shape[2] if len(shape) == 3 else 1
    st = FrameStream(h, w, ch, np.uint8, max_frames=len(ps), images=True)
    st.upload(imgs.reshape(len(ps), h, w, ch))
    idx = list(range(len(ps)))
    res = st.encode(idx, idx, 127, seeds=_cabi.BC_SEEDS)
    bms, wts, masks = st.fetch_batch(0, len(ps), want_masks=True)
    assert not st.decode_verify().any()
    for j, im in enumerate(imgs):
        mask = np.unpackbits(masks[j], bitorder="little")[:h * w]
        ref = binarize_image(im, 127)
        assert np.array_equal(mask, ref), j
        assert res[j].ones == int(ref.sum())
        ob, ow, op, on, oratio, ok, ol = co.compress(ref, seeds=_cabi.BC_SEEDS)
        assert (res[j].l, res[j].wlen, res[j].raw) == (ol, len(ow), ol == 0)
        if ol:
            assert bms[j, :(ol + 7) // 8].tobytes() == np.packbits(ob).tobytes()
            assert wts[j, :(len(ow) + 7) // 8].tobytes() == np.packbits(ow).tobytes()
    # rbf_stream_decode with the encoder's exact k reproduces every coded mask
    coded = [j for j in idx if not res[j].raw]
    dm, used = st.decode([res[j].l for j in coded], [res[j].wlen for j in coded], [res[j].k for j in coded], bms[coded], wts[coded],
                         seeds=_cabi.BC_SEEDS)
    for t, j in enumerate(coded):
        assert used[t] == res[j].wlen
        assert np.array_equal(np.unpackbits(dm[t], bitorder="little")[:h * w], binarize_image(imgs[j], 127))
    # the public decode takes k from the payload's float32, as the reference does (bc:427, 461): compare with the C decoder on
    # that k, including the IndexError when the rounded k lets more positions pass than the witness holds
    comp = bcm.BloomFilterCompressor()
    for (data, _), im in zip(comp.compress_images(list(imgs)), imgs):
        bitmap, witness, p, n, k, _ = comp._unpack_compressed_data(data)
        if not witness:
            assert np.array_equal(comp.decompress_images([data])[0], bitmap.reshape(h, w) * 255)
            continue
        out, consumed = c_decode(bitmap, witness, n, k)
        if consumed > len(witness):
            with pytest.raises(IndexError):
                comp.decompress_images([data])
        else:
            assert np.array_equal(comp.decompress_images([data])[0].reshape(-1), out * 255)
    st.close()


def test_image_stream_refusals():
    from new_bloom_filter_repo_b200 import FrameStream, RbfError, _cabi
    st = FrameStream(16, 16, 3, np.uint8, max_frames=2, images=True)
    for key in ("gray_mode", "mask_mode"):
        with pytest.raises(RbfError, match="-6"):
            st.set_option(key, 1)
    st.upload(np.zeros((2, 16, 16, 3), np.uint8))
    with pytest.raises(RbfError, match="-1"):
        st.encode([0], [1], 127, seeds=_cabi.BC_SEEDS)
    with pytest.raises(RbfError, match="-6"):
        st.encode_host(np.zeros((2, 16, 16, 3), np.uint8), 127)
    for C, S in [(5, 1), (2, 2), (3, 2), (0, 2)]:          # (0, 1) is the decode-only stream below
        with pytest.raises(RbfError):
            FrameStream(8, 8, C, np.uint8 if S == 1 else np.uint16, max_frames=1, images=True)
    with pytest.raises(RbfError):                          # frame streams still refuse 2- and 4-channel frames
        FrameStream(8, 8, 4, np.uint8, max_frames=2)
    st.close()
    dec = FrameStream(16, 16, 0, np.uint8, max_frames=2, images=True)       # decode-only: no image store
    with pytest.raises(RbfError, match="-6"):
        dec.upload(np.zeros((1, 16, 16, 0), np.uint8))
    with pytest.raises(RbfError, match="-6"):
        dec.encode([0], [0], 127, seeds=_cabi.BC_SEEDS)
    dec.close()


def test_stream_cache_is_bounded_and_closable(comp):
    imgs = [_sparse((16 + i, 40, 3), 0.05, 20 + i) for i in range(6)]
    payloads = [comp.compress_images([im])[0][0] for im in imgs]
    assert len(comp._streams.streams) == comp._streams.capacity == 4          # least recently used shapes were freed
    for im, data in zip(imgs, payloads):
        assert np.array_equal(comp.decompress_images([data])[0], binarize_image(im, 127).reshape(im.shape[:2]) * 255)
    assert all(k[2] == 0 for k in list(comp._streams.streams)[-4:])          # decodes use image-store-free streams
    comp.close()
    assert not comp._streams.streams
    assert comp.compress_images(imgs[:1])[0][0] == payloads[0]
