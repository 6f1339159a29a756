"""CPU tests (-m "not gpu") of the bloom_compress drop-in: a numpy restatement of _binarize_image (bc:67-87) pinned to the
reference's masks, the drop-in's container parsers and text glue against the reference's payloads, and the input checks that
refuse an image before any device work."""
import math

import numpy as np
import pytest

from tests.util import golden_json, golden_npz, sha

from new_bloom_filter_repo_b200.bloom_compress import BloomFilterCompressor as BC


def binarize_image(image: np.ndarray, threshold) -> np.ndarray:
    """bc:67-87 restated: gray = floor(channel mean) for C > 1 (8-bit samples), the sample itself otherwise; 1 where gray > t."""
    a = np.asarray(image)
    if a.ndim > 2 and a.shape[2] > 1:
        gray = a.astype(np.int64).sum(axis=2) // a.shape[2]
    else:
        gray = a.astype(np.int64)
    t = float(threshold)
    if math.isnan(t):
        return np.zeros(gray.size, dtype=np.uint8)
    return (gray > math.floor(t)).astype(np.uint8).reshape(-1)


def _threshold(rec):
    return float(rec["threshold"]) if "." in rec["threshold"] or rec["threshold"] == "nan" else int(rec["threshold"])


def test_binarize_restatement_matches_reference():
    kat, arr = golden_json("bc_kat.json"), golden_npz("bc_arrays.npz")
    assert len(kat["binarize"]) == 7 * 8
    for rec in kat["binarize"]:
        m = binarize_image(arr["bin_" + rec["image"]], _threshold(rec))
        assert (sha(m), int(m.sum())) == (rec["sha"], rec["ones"]), rec


def test_unpack_image_payloads():
    kat, arr = golden_json("bc_kat.json"), golden_npz("bc_arrays.npz")
    comp = BC.__new__(BC)                                  # the parsers need no device
    for rec in kat["images"]:
        data = bytes.fromhex(rec["payload"])
        bitmap, witness, p, n, k, shape = comp._unpack_compressed_data(data)
        img = arr["img_" + rec["name"]]
        assert shape == img.shape and n == img.shape[0] * img.shape[1]
        assert comp._pack_compressed_data(bitmap, witness, p, n, k, shape) == data
        mask = binarize_image(img, 127)
        if len(witness) == 0:                              # raw branch: the payload holds the mask itself (l = n)
            assert np.array_equal(bitmap, mask) and k == 0.0
        else:
            assert sum(witness) == mask.sum()              # every set position passes the Bloom test
            assert (mask.reshape(img.shape[:2]) * 255).shape == tuple(rec["decoded_shape"])
    coded = [r for r in kat["images"] if comp._unpack_compressed_data(bytes.fromhex(r["payload"]))[1]]
    assert len(coded) >= 4


def test_text_payloads_and_debinarize():
    kat = golden_json("bc_kat.json")
    comp = BC.__new__(BC)
    for rec in kat["text"]:
        data = bytes.fromhex(rec["payload"])
        bitmap, witness, p, n, k, text_length, bit_depth = comp._unpack_text_data(data)
        assert (text_length, bit_depth) == (len(rec["text"]), rec["bit_depth"])
        assert comp._pack_text_data(bitmap, witness, p, n, k, text_length, bit_depth) == data
        bits = BC._binarize_text(rec["text"], rec["bit_depth"])
        assert len(bits) == n
        if len(witness) == 0:
            assert BC._debinarize_text(bitmap, bit_depth)[:text_length] == rec["decoded"]
    names = {r["name"]: r for r in kat["text"]}
    assert names["nonascii_8"]["decoded"] == "na?ve caf? ?"
    assert comp._unpack_text_data(bytes.fromhex(names["control"]["payload"]))[1]        # actually coded


@pytest.mark.parametrize("image", [np.zeros((4, 4, 3), np.uint16), np.zeros((2, 2, 2, 2), np.uint8), np.zeros((4, 4), np.int32),
                                   np.zeros((4, 4), np.float32), np.zeros((4, 4, 5), np.uint8), np.zeros((), np.uint8)])
def test_binarize_refusals_before_device(image):
    with pytest.raises(ValueError):
        BC._binarize_image(image, 127)
    with pytest.raises(ValueError):
        BC.__new__(BC).compress_images([np.zeros((4, 4), np.uint8), image])
