"""
Drop-in for the reference's bloom_compress.py (bc), its bi-level image and text codec:

    BloomFilterCompressor                   bc:13-618
      RationalBloomFilter (nested)          bc:144-239   integer indices, seeds 0 / 1 / 999
      compress / decompress                 bc:241-346   the improved_video_compressor drop-in's device coder, bc's seeds
      compress_image / decompress_image     bc:348-416   K1 = k_binarize (bc:67-87) on an image stream, then K2 -> K3 -> K3b
      compress_text / decompress_text       bc:490-555   text masks go through the single-mask coder (rbf_compress_mask)
    run_compression_tests                   bc:621-727   without the matplotlib figure

Same names, arguments, return shapes, exceptions and printed lines (bc prints unconditionally, bc:258, 268-269, 300-303).
New here, and the reason to code images on a GPU: compress_images / decompress_images code a whole batch -- one upload, one
encode and one batched copy per group of equally shaped images -- with results byte-identical to the one-image calls.

Deliberate difference (DESIGN.md section 6): _binarize_image refuses with ValueError what it cannot reproduce exactly --
multi-channel images with samples wider than 8 bits (numpy's float -> uint8 cast of a mean above 255 is
implementation-defined), more than 3 dimensions, more than 4 channels, and sample types other than uint8 / uint16 / bool.
"""
from __future__ import annotations

import io
import struct
import time
from collections import OrderedDict
from typing import Dict, List, Optional, Tuple

import numpy as np

from . import _cabi
from . import improved_video_compressor as _ivc
from .stream import FrameStream

class _StreamCache:
    """Image streams by (H, W, channels, sample type, k1_only); the least recently used is closed, and its device memory freed,
    once more than `capacity` are held.  channels = 0 is a decode-only stream (no image store)."""

    def __init__(self, capacity: int):
        self.capacity = capacity
        self.streams: "OrderedDict[tuple, FrameStream]" = OrderedDict()

    def get(self, h: int, w: int, ch: int, dtype, count: int, k1_only: bool = False) -> FrameStream:
        """A stream holding at least `count` images."""
        key = (h, w, ch, np.dtype(dtype).str, bool(k1_only))
        st = self.streams.pop(key, None)
        if st is not None and st.max_frames < count:
            st.close()
            st = None
        if st is None:
            st = FrameStream(h, w, ch, dtype, max_frames=count, k1_only=k1_only, images=True)
        self.streams[key] = st
        while len(self.streams) > self.capacity:
            self.streams.popitem(last=False)[1].close()
        return st

    def clear(self) -> None:
        for st in self.streams.values():
            st.close()
        self.streams.clear()


_BINARIZE_STREAMS = _StreamCache(2)          # _binarize_image is a static method: one small cache of one-image streams


def _image_layout(image) -> Tuple[np.ndarray, Tuple[int, int, int]]:
    """-> (samples as uint8 / uint16, (H, W, C)) of an image _binarize_image accepts; ValueError otherwise."""
    a = np.asarray(image)
    if a.ndim == 0 or a.ndim > 3:
        raise ValueError(f"images are 1-, 2- or 3-dimensional arrays, not {a.ndim}-dimensional")
    if a.dtype == np.bool_:
        a = a.view(np.uint8)                                  # numpy stores bool as 0/1 bytes: same comparison results
    elif a.dtype.kind == "u" and a.dtype.itemsize in (1, 2):
        a = a.astype(np.uint8 if a.dtype.itemsize == 1 else np.uint16, copy=False)   # native byte order
    else:
        raise ValueError(f"image samples must be uint8, uint16 or bool, not {a.dtype}")
    ch = a.shape[2] if a.ndim == 3 else 1
    if ch > 4:
        raise ValueError(f"images have at most 4 channels, not {ch}")
    if ch > 1 and a.dtype.itemsize != 1:
        raise ValueError("multi-channel images need 8-bit samples: the reference's uint8 cast of a mean above 255 "
                         "(bloom_compress.py:81) is implementation-defined")
    h, w = (1, a.shape[0]) if a.ndim == 1 else (a.shape[0], a.shape[1])
    return a, (h, w, ch)


def _image_hw(original_shape) -> Tuple[int, int]:
    if len(original_shape) > 2:                               # bc:404-408 (a 1-D or 0-D shape raises ValueError there too)
        height, width = original_shape[:2]
    else:
        height, width = original_shape
    return height, width


class BloomFilterCompressor(_ivc.BloomFilterCompressor):
    """bc.BloomFilterCompressor (bc:13-618)."""

    P_STAR = 0.32453                                          # bc:23

    class RationalBloomFilter(_ivc.RationalBloomFilter):
        """bc.BloomFilterCompressor.RationalBloomFilter (bc:144-239): the ivc filter with h1/h2 seeds 0 / 1 (bc:163-164)
        and activation seed 999 (bc:195)."""

        def __init__(self, size: int, k_star: float):
            super().__init__(size, k_star, seeds=_cabi.BC_SEEDS)

    def __init__(self):
        super().__init__(verbose=False, seeds=_cabi.BC_SEEDS)
        self.max_batch_images = 64                            # images per device batch of compress_images / decompress_images
        self.max_batch_bytes = 1 << 30                        # and at most this many bytes of samples per batch
        self._streams = _StreamCache(4)                       # device streams of this compressor, by image shape

    def close(self) -> None:
        """Free the device streams this compressor holds (they are also freed when it is garbage-collected)."""
        self._streams.clear()

    @staticmethod
    def _calculate_optimal_params(n: int, p: float) -> Tuple[float, int]:       # bc:30-64
        return _ivc.calculate_optimal_params(n, p)

    @staticmethod
    def _binarize_image(image: np.ndarray, threshold: int = 127) -> np.ndarray:  # bc:67-87
        """Flat uint8 0/1 mask of (gray > threshold), computed by k_binarize on the device."""
        a, (h, w, ch) = _image_layout(image)
        if a.size == 0:
            return np.zeros(0, dtype=np.uint8)
        st = _BINARIZE_STREAMS.get(h, w, ch, a.dtype, 1, k1_only=True)
        st.upload(a.reshape(1, h, w, ch))
        st.encode([0], [0], float(threshold), seeds=_cabi.BC_SEEDS)
        return st.fetch(0)[2]

    @staticmethod
    def _binarize_text(text: str, bit_depth: int = 8) -> np.ndarray:             # bc:89-112
        data = text.encode("ascii", errors="replace") if bit_depth == 8 else text.encode("utf-8")
        return np.unpackbits(np.frombuffer(data, dtype=np.uint8))

    @staticmethod
    def _debinarize_text(binary_array: np.ndarray, bit_depth: int = 8) -> str:   # bc:114-142
        bits = np.asarray(binary_array)
        if len(bits) % 8:
            bits = np.pad(bits, (0, 8 - len(bits) % 8), "constant")
        data = np.packbits(bits).tobytes()
        return data.decode("ascii" if bit_depth == 8 else "utf-8", errors="replace")

    # ------------------------------------------------------------------ the 0/1-vector coder
    def _report(self, p, n: int, k: float, l: int, wlen: int, raw: bool) -> None:
        """The lines bc.compress prints (bc:258, 268-269, 300-303); nothing for the p <= 1e-4 / n = 0 raw branch (bc:264-266)."""
        if raw:
            if p >= self.P_STAR:
                print(f"Density {p:.4f} is >= threshold {self.P_STAR}, compression not effective")
            return
        print(f"Input length: {n}, Density: {p:.4f}")
        print(f"Optimal parameters: k={k:.4f}, l={l}")
        print(f"Bloom filter size: {l} bits")
        print(f"Witness size: {wlen} bits")
        print(f"Compression ratio: {(l + wlen) / n:.4f}")
        print(f"Bloom filter test pass rate: {wlen / n:.4f}")      # every Bloom-test pass adds one witness bit (bc:287-293)

    def compress(self, binary_input: np.ndarray):                                 # bc:241-305
        """-> (bloom_filter_bitmap, witness, density, input_length, compression_ratio).  bc has no `l >= n` guard (bc:264)
        where ivc has one (ivc:223), but it cannot fire for n >= 2: l / n <= 0.317 for every p in (1e-4, P_STAR), and n < 2
        has p in {0, 1} -- so the device coder, which applies the ivc gate, already behaves as bc."""
        out = super().compress(binary_input)
        bitmap, witness, p, n, ratio = out
        raw = len(witness) == 0 and ratio == 1.0
        k = self._calculate_optimal_params(n, p)[0] if not raw else 0.0
        self._report(p, n, k, len(bitmap), len(witness), raw)
        return out

    # ------------------------------------------------------------------ images
    def _image_payload(self, r, bm_row, wt_row, mask_row, shape) -> Tuple[bytes, float]:
        """bc:369-376 for one encoded image: the container of _pack_compressed_data from the device's packbits rows."""
        n = r.n
        k, _ = self._calculate_optimal_params(n, r.p)                               # bc:372
        if r.raw:                                             # bc:257-266: the mask itself, l = n bits
            bits = np.packbits(np.unpackbits(mask_row, bitorder="little")[:n]).tobytes()
            return self._header(r.p, n, k, shape, n, 0) + bits, 1.0
        nb, nw = (r.l + 7) // 8, (r.wlen + 7) // 8
        return self._header(r.p, n, k, shape, r.l, r.wlen) + bm_row[:nb].tobytes() + wt_row[:nw].tobytes(), (r.l + r.wlen) / n

    @staticmethod
    def _header(p, n, k, shape, l, wlen) -> bytes:            # bc:424-441
        return (struct.pack("!fIfB", p, n, k, len(shape)) + b"".join(struct.pack("!I", d) for d in shape)
                + struct.pack("!II", l, wlen))

    def _chunk(self, frame_bytes: int) -> int:
        return max(1, min(int(self.max_batch_images), int(self.max_batch_bytes) // max(1, frame_bytes)))

    def _encode_images(self, images, threshold) -> List[Tuple[bytes, float, object]]:
        """(payload, ratio, PairResult or None) per image, in input order; equally shaped images share device batches."""
        layouts = [_image_layout(img) for img in images]      # every ValueError before any device work
        out: List[Optional[tuple]] = [None] * len(images)
        groups: Dict[tuple, List[int]] = {}
        for i, (a, hwc) in enumerate(layouts):
            if a.size == 0:                                   # n = 0: p = nan, the raw branch (bc:253-266) without a device
                bm, wt, p, n, ratio = self.compress(np.zeros(0, dtype=np.uint8))
                out[i] = (self._header(p, 0, 0, np.shape(images[i]), 0, 0), ratio, None)
            else:
                groups.setdefault(hwc + (a.dtype.str,), []).append(i)
        thr = float(threshold)
        for (h, w, ch, dt), idx in groups.items():
            chunk = self._chunk(h * w * ch * np.dtype(dt).itemsize)
            st = self._streams.get(h, w, ch, dt, min(chunk, len(idx)))
            for c0 in range(0, len(idx), chunk):
                part = idx[c0:c0 + chunk]
                st.upload(np.stack([layouts[i][0].reshape(h, w, ch) for i in part]))
                slots = list(range(len(part)))
                res = st.encode(slots, slots, thr, seeds=_cabi.BC_SEEDS)
                any_raw = any(r.raw for r in res)
                bms, wts, masks = st.fetch_batch(0, len(part), want_masks=any_raw)
                for j, i in enumerate(part):
                    data, ratio = self._image_payload(res[j], bms[j], wts[j], masks[j] if any_raw else None, np.shape(images[i]))
                    out[i] = (data, ratio, res[j])
        return out

    def compress_images(self, images, threshold: int = 127) -> List[Tuple[bytes, float]]:
        """compress_image for many images (arrays) at once, silently: [(compressed_data_bytes, compression_ratio)] in input order,
        byte-identical to compress_image of each."""
        return [(data, ratio) for data, ratio, _ in self._encode_images(list(images), threshold)]

    def compress_image(self, image_path, threshold: int = 127, output_path: Optional[str] = None) -> Tuple[bytes, float]:
        """bc:348-383.  `image_path` may also be the image array itself."""
        if isinstance(image_path, np.ndarray):
            img = image_path
        else:
            from PIL import Image
            img = np.array(Image.open(image_path))
        data, ratio, r = self._encode_images([img], threshold)[0]
        if r is not None:
            self._report(r.p, r.n, self._calculate_optimal_params(r.n, r.p)[0], r.l, r.wlen, r.raw)
        if output_path:
            with open(output_path, "wb") as f:
                f.write(data)
        return data, ratio

    @staticmethod
    def _parse_image_payload(data: bytes):
        """The fields of a bc:418-452 container: (p, n, k, shape, l, wlen, bitmap bytes, witness bytes); a short payload reads
        short, exactly like bc:454-488's buffer.read."""
        buf = io.BytesIO(data)
        p, n, k = struct.unpack("!fIf", buf.read(12))
        (nd,) = struct.unpack("!B", buf.read(1))
        shape = tuple(struct.unpack("!I", buf.read(4))[0] for _ in range(nd))
        l, wlen = struct.unpack("!I", buf.read(4))[0], struct.unpack("!I", buf.read(4))[0]
        return p, n, k, shape, l, wlen, buf.read((l + 7) // 8), buf.read((wlen + 7) // 8)

    def _unpack_compressed_data(self, data: bytes) -> Tuple:                      # bc:454-488
        p, n, k, shape, l, wlen, bb, wb = self._parse_image_payload(data)
        bloom_bitmap = np.unpackbits(np.frombuffer(bb, dtype=np.uint8))[:l]
        witness = np.unpackbits(np.frombuffer(wb, dtype=np.uint8))[:wlen].tolist()
        return bloom_bitmap, witness, p, n, k, shape

    def _pack_compressed_data(self, bloom_bitmap: np.ndarray, witness: list, p: float, n: int, k: float,
                              original_shape: Tuple) -> bytes:                      # bc:418-452
        return (self._header(p, n, k, original_shape, len(bloom_bitmap), len(witness)) + np.packbits(bloom_bitmap).tobytes()
                + np.packbits(np.array(witness, dtype=np.uint8)).tobytes())

    def _decompress_one(self, data: bytes) -> np.ndarray:                         # bc:397-410
        bloom_bitmap, witness, p, n, k, shape = self._unpack_compressed_data(data)
        flat = self.decompress(bloom_bitmap, witness, n, k)
        return flat.reshape(_image_hw(shape)) * 255

    def decompress_images(self, payloads) -> List[np.ndarray]:
        """decompress_image for many payloads at once: [uint8 (H, W) image of 0 / 255] in input order.  Well-formed coded
        payloads of one (H, W) share device batches (rbf_stream_decode); anything else -- raw payloads, short or corrupt
        ones -- takes the one-payload path, so errors are the reference's.  The first error in input order is raised."""
        payloads = list(payloads)
        out: List[object] = [None] * len(payloads)
        groups: Dict[Tuple[int, int], List[tuple]] = {}
        for i, data in enumerate(payloads):
            try:
                p, n, k, shape, l, wlen, bb, wb = self._parse_image_payload(data)
                h, w = _image_hw(shape)
                batchable = (wlen > 0 and 1 <= l <= n and wlen <= n and h * w == n and len(bb) == (l + 7) // 8
                             and len(wb) == (wlen + 7) // 8 and 0.0 <= k <= 1e6)
            except Exception:
                batchable = False
            if batchable:
                groups.setdefault((h, w), []).append((i, l, wlen, k, bb, wb))
                continue
            try:
                out[i] = self._decompress_one(data)
            except Exception as e:                            # noqa: BLE001  (re-raised below, in input order)
                out[i] = e
        for (h, w), items in groups.items():
            n = h * w
            chunk = self._chunk(n)
            st = self._streams.get(h, w, 0, np.uint8, min(chunk, len(items)))      # decode-only: no image store
            for c0 in range(0, len(items), chunk):
                part = items[c0:c0 + chunk]
                bslot = max(16, (max(len(it[4]) for it in part) + 15) // 16 * 16)
                wslot = max(16, (max(len(it[5]) for it in part) + 15) // 16 * 16)
                bms = np.zeros((len(part), bslot), dtype=np.uint8)
                wts = np.zeros((len(part), wslot), dtype=np.uint8)
                for j, it in enumerate(part):
                    bms[j, :len(it[4])] = np.frombuffer(it[4], dtype=np.uint8)
                    wts[j, :len(it[5])] = np.frombuffer(it[5], dtype=np.uint8)
                masks, consumed = st.decode([it[1] for it in part], [it[2] for it in part], [it[3] for it in part], bms, wts,
                                            seeds=_cabi.BC_SEEDS)
                for j, it in enumerate(part):
                    if consumed[j] > it[2]:                   # bc:342: witness[witness_idx] runs past the end
                        out[it[0]] = IndexError("list index out of range")
                    else:
                        out[it[0]] = np.unpackbits(masks[j], bitorder="little")[:n].reshape(h, w) * 255
        for r in out:
            if isinstance(r, Exception):
                raise r
        return out

    def decompress_image(self, compressed_data: bytes, output_path: Optional[str] = None) -> np.ndarray:   # bc:385-416
        img = self.decompress_images([compressed_data])[0]
        if output_path:
            from PIL import Image
            Image.fromarray(img.astype(np.uint8)).save(output_path)
        return img

    # ------------------------------------------------------------------ text
    def compress_text(self, text: str, bit_depth: int = 8, output_path: Optional[str] = None) -> Tuple[bytes, float]:   # bc:490-524
        bloom_bitmap, witness, p, n, ratio = self.compress(self._binarize_text(text, bit_depth))
        k, _ = self._calculate_optimal_params(n, p)
        data = self._pack_text_data(bloom_bitmap, witness, p, n, k, len(text), bit_depth)
        if output_path:
            with open(output_path, "wb") as f:
                f.write(data)
        return data, ratio

    def decompress_text(self, compressed_data: bytes, output_path: Optional[str] = None) -> str:              # bc:526-555
        bloom_bitmap, witness, p, n, k, text_length, bit_depth = self._unpack_text_data(compressed_data)
        text = self._debinarize_text(self.decompress(bloom_bitmap, witness, n, k), bit_depth)[:text_length]
        if output_path:
            with open(output_path, "w", encoding="utf-8") as f:
                f.write(text)
        return text

    def _pack_text_data(self, bloom_bitmap: np.ndarray, witness: list, p: float, n: int, k: float, text_length: int,
                        bit_depth: int) -> bytes:                                   # bc:557-587
        return (struct.pack("!fIfIBII", p, n, k, text_length, bit_depth, len(bloom_bitmap), len(witness))
                + np.packbits(bloom_bitmap).tobytes() + np.packbits(np.array(witness, dtype=np.uint8)).tobytes())

    def _unpack_text_data(self, data: bytes) -> Tuple:                            # bc:589-618
        buf = io.BytesIO(data)
        p, n, k, text_length, bit_depth, l, wlen = struct.unpack("!fIfIBII", buf.read(25))
        bloom_bitmap = np.unpackbits(np.frombuffer(buf.read((l + 7) // 8), dtype=np.uint8))[:l]
        witness = np.unpackbits(np.frombuffer(buf.read((wlen + 7) // 8), dtype=np.uint8))[:wlen].tolist()
        return bloom_bitmap, witness, p, n, k, text_length, bit_depth


def run_compression_tests():                                                      # bc:621-727, without the figure
    compressor = BloomFilterCompressor()
    print("Test 1: Synthetic binary data")
    print("============================")
    n = 100000
    for p in [0.1, 0.2, 0.3, 0.4]:
        print(f"\nDensity p = {p}")
        binary_data = np.random.choice([0, 1], size=n, p=[1 - p, p])
        t0 = time.time()
        bloom_bitmap, witness, density, input_length, ratio = compressor.compress(binary_data)
        compress_time = time.time() - t0
        k, _ = compressor._calculate_optimal_params(n, density)
        t0 = time.time()
        decompressed = compressor.decompress(bloom_bitmap, witness, input_length, k)
        decompress_time = time.time() - t0
        print(f"Lossless reconstruction: {np.array_equal(binary_data, decompressed)}")
        print(f"Compression ratio: {ratio:.4f}")
        print(f"Compression time: {compress_time:.4f}s")
        print(f"Decompression time: {decompress_time:.4f}s")
        if density >= compressor.P_STAR:
            print(f"Note: Density {density:.4f} is above threshold {compressor.P_STAR:.4f}")
            print("No actual compression was performed (ratio should be 1.0)")
    try:
        print("\nTest 2: Image compression")
        print("========================")
        from PIL import Image
        test_image = np.zeros((100, 100), dtype=np.uint8)
        test_image[25:75, 25:75] = 255
        test_image[40:60, 40:60] = 0
        Image.fromarray(test_image).save("test_image.png")
        binary_data = compressor._binarize_image(test_image, threshold=127)
        density = np.sum(binary_data) / len(binary_data)
        print(f"Image density: {density:.4f}")
        if density >= compressor.P_STAR:
            print(f"Note: Image density {density:.4f} is above threshold {compressor.P_STAR:.4f}")
            print("Compression may not be effective")
        print("\nCompressing test image...")
        compressed_data, ratio = compressor.compress_image("test_image.png", threshold=127, output_path="test_image.bloom")
        print("\nDecompressing test image...")
        decompressed_image = compressor.decompress_image(compressed_data, output_path="test_image_decompressed.png")
        is_lossless = np.array_equal(binary_data, decompressed_image.flatten() / 255)
        print(f"Lossless reconstruction: {is_lossless}")
        print(f"Compression ratio: {ratio:.4f}")
    except Exception as e:
        print(f"Error in image compression test: {e}")
        import traceback
        traceback.print_exc()


if __name__ == "__main__":
    run_compression_tests()
