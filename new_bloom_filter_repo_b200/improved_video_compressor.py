"""
Drop-in for the reference's improved_video_compressor.py on the rational-Bloom hot path:

    RationalBloomFilter      ivc:39-138    (integer indices, seeds 0x12345678 / 0x87654321 / 999)
    BloomFilterCompressor    ivc:140-307   (compress / decompress of a 0/1 vector)
    VideoFrameCompressor     ivc:671-1234  (_calculate_frame_diff, _apply_frame_diff,
                                            _compress/_decompress_frame_differences, keyframe codec)
    ImprovedVideoCompressor  ivc:309-523   (compress_video / decompress_video / verify_lossless)

Same names, arguments, return shapes and error behaviour; the per-pixel thresholding, the XXH64
double hashing, the probabilistic floor(k*)+1'th probe and the bit-array set/test run as sm_100a
kernels behind the C ABI (include/rbf_b200.h).  No host implementation of those exists in this
package: without librbf_b200.so and a B200 every entry point raises.

Where the reference is unwired (SURVEY.md section 0): `VideoFrameCompressor.bloom_compressor` is
assigned here (the reference never does), and `ImprovedVideoCompressor.compress_video` gains the
keyframe / inter-frame loop the reference's `keyframe_interval` argument promises; with
`keyframe_interval=1` its output is byte-identical to the reference's (all keyframes, ivc:390).
"""
from __future__ import annotations

import ctypes as C
import io
import math
import os
import struct
import time
import zlib
from typing import Dict, List, Optional, Tuple

import numpy as np

from . import _cabi
from .fixed_video_compressor import FixedVideoCompressor, YUVFrame
from .rational_bloom_filter import _DeviceFilter
from .stream import FrameStream


class RationalBloomFilter:
    """ivc.RationalBloomFilter (ivc:39-138).  `bit_array` is fetched from / written to the device copy."""

    def __init__(self, size: int, k_star: float, seeds=None):
        self.size = size                                      # ivc:55
        self.k_star = k_star                                  # ivc:56
        self.floor_k = math.floor(k_star)                     # ivc:57
        self.p_activation = k_star - self.floor_k             # ivc:58
        self.h1_seed = 0x12345678 if seeds is None else seeds[0]   # ivc:62
        self.h2_seed = 0x87654321 if seeds is None else seeds[1]   # ivc:63
        self._act_seed = 999 if seeds is None else seeds[2]        # ivc:94
        self._dev = _DeviceFilter(size, k_star, (self.h1_seed, self.h2_seed, self._act_seed))

    @property
    def bit_array(self) -> np.ndarray:                        # ivc:59 (np.uint8[size], one byte per bit)
        """A read-only snapshot of the device bits: in-place writes (`f.bit_array[i] = 1`) would be lost, so they raise;
        assign a whole array instead (`f.bit_array = bits`, as ivc:290 does)."""
        a = self._dev.get_bits()
        a.setflags(write=False)
        return a

    @bit_array.setter
    def bit_array(self, bits) -> None:                        # `bloom_filter.bit_array = bloom_bitmap`, ivc:290
        self._dev.set_bits(bits)

    def _get_hash_indices(self, item: int, i: int) -> int:    # ivc:65-81
        b = str(item).encode("utf-8")
        return _cabi.lib().rbf_probe_index(_cabi.xxh64(b, self.h1_seed), _cabi.xxh64(b, self.h2_seed), int(i), int(self.size))

    def _determine_activation(self, item: int) -> bool:       # ivc:83-97
        return _cabi.xxh64(str(item).encode("utf-8"), self._act_seed) < _cabi.activation_threshold(self.p_activation)

    @staticmethod
    def _split(indices):
        """uint32 items go to the decimal-index kernels; anything else the reference would hash as str(item) -- negative or
        >= 2**32 integers -- goes through the string kernels, so `str(item)` semantics hold for every int."""
        arr = np.asarray(indices)
        if arr.dtype.kind in "iu" and arr.size and (arr.dtype.kind == "u" or int(arr.min()) >= 0) and int(arr.max()) < 2 ** 32:
            return arr.astype(np.uint32, copy=False).reshape(-1), None
        if arr.size == 0:
            return np.zeros(0, dtype=np.uint32), None
        return None, [str(int(x)) if isinstance(x, (int, np.integer)) else str(x) for x in np.asarray(indices, dtype=object).reshape(-1)]

    def add_index(self, index: int) -> None:                  # ivc:99-114
        self.add_indices([index])

    def check_index(self, index: int) -> bool:                # ivc:116-138
        return bool(self.check_indices([index])[0])

    def add_indices(self, indices) -> None:                   # batch form: one launch
        u32, strs = self._split(indices)
        if strs is None:
            self._dev.add_indices(u32)
        else:
            self._dev.add_strings(strs)

    def check_indices(self, indices) -> np.ndarray:
        u32, strs = self._split(indices)
        if strs is None:
            return self._dev.check_indices(u32).astype(bool)
        return self._dev.check_strings(strs).astype(bool)


def calculate_optimal_params(n: int, p: float) -> Tuple[float, int]:
    """BloomFilterCompressor._calculate_optimal_params, expression for expression (ivc:161-196; bloom_compress.py:30-64 is the
    same code)."""
    if p <= 0.0001:
        return 0, 0
    if p >= BloomFilterCompressor.P_STAR:
        return 0, 0
    q = 1 - p
    L = math.log(2)
    k = math.log2(q * (L ** 2) / p)
    if math.isnan(k) or k <= 0:
        return 0, 0
    gamma = 1 / L
    l = int(p * n * k * gamma)
    return max(0.1, k), max(1, l)


class BloomFilterCompressor:
    """ivc.BloomFilterCompressor (ivc:140-307)."""

    P_STAR = 0.32453                                          # ivc:150

    def __init__(self, verbose: bool = False, seeds=_cabi.IVC_SEEDS):
        self.verbose = verbose
        self._seeds = seeds

    def _calculate_optimal_params(self, n: int, p: float) -> Tuple[float, int]:   # ivc:161-196
        return calculate_optimal_params(n, p)

    def compress(self, binary_input: np.ndarray, k_l_override=None):             # ivc:198-266
        """-> (bloom_filter_bitmap, witness, density, input_length, compression_ratio)"""
        arr = np.asarray(binary_input)
        n = len(arr)
        if n == 0:                                            # the reference divides 0/0 -> nan and falls through to the
            with np.errstate(invalid="ignore", divide="ignore"):   # raw-passthrough branch (ivc:212, ivc:188-189, ivc:223-225)
                p = np.float64(0.0) / np.float64(0.0)
            return binary_input, [], p, 0, 1.0
        m8 = np.ascontiguousarray(arr, dtype=np.uint8)
        if m8.size and m8.max() > 1:
            raise ValueError("binary_input must hold 0/1 values")
        info = _cabi.MaskInfo()
        bitmap = np.empty(n, dtype=np.uint8)
        witness = np.empty(n, dtype=np.uint8)
        sd = _cabi.seeds_struct(self._seeds)
        ko, lo = (0.0, 0) if k_l_override is None else (float(k_l_override[0]), int(k_l_override[1]))
        _cabi.check(_cabi.lib().rbf_compress_mask(_cabi.ctx(), _cabi.ptr(m8), n, C.byref(sd), ko, lo, C.byref(info),
                                                  _cabi.ptr(bitmap), _cabi.ptr(witness)), _cabi.ctx())
        p = np.float64(info.p)
        self.last_info = info
        if info.raw:                                          # ivc:215-218, ivc:223-225
            if self.verbose and p >= self.P_STAR:
                print(f"Density {p:.4f} is >= threshold {self.P_STAR}, compression not effective")
            return binary_input, [], p, n, 1.0
        l, wlen = int(info.l), int(info.wlen)
        if self.verbose:
            print(f"Input length: {n}, Density: {p:.4f}")
            print(f"Optimal parameters: k={info.k:.4f}, l={l}")
            print(f"Bloom filter size: {l} bits")
            print(f"Witness size: {wlen} bits")
        ratio = (l + wlen) / n                                # ivc:256-258
        return bitmap[:l].copy(), list(witness[:wlen]), p, n, ratio

    def decompress(self, bloom_bitmap: np.ndarray, witness: list, n: int, k: float) -> np.ndarray:   # ivc:268-307
        if len(witness) == 0:                                 # ivc:282-284
            return bloom_bitmap
        bm = np.ascontiguousarray(np.asarray(bloom_bitmap, dtype=np.uint8))
        wt = np.ascontiguousarray(np.asarray(witness, dtype=np.uint8))
        out = np.empty(n, dtype=np.uint8)
        consumed = C.c_uint64()
        sd = _cabi.seeds_struct(self._seeds)
        _cabi.check(_cabi.lib().rbf_decompress_mask(_cabi.ctx(), _cabi.ptr(bm), len(bm), _cabi.ptr(wt), len(wt), int(n),
                                                    float(k), C.byref(sd), _cabi.ptr(out), C.byref(consumed)), _cabi.ctx())
        if consumed.value > len(wt):                          # the reference's witness[witness_idx] raises here
            raise IndexError("list index out of range")
        return out


def _frame_data(frame) -> np.ndarray:
    return frame.data if hasattr(frame, "yuv_info") else np.asarray(frame)


class VideoFrameCompressor:
    """The inter-frame pieces of ivc.VideoFrameCompressor (ivc:671-1234)."""

    def __init__(self, noise_tolerance: float = 10.0, keyframe_interval: int = 30, min_diff_threshold: float = 3.0,
                 max_diff_threshold: float = 30.0, bloom_threshold_modifier: float = 1.0, num_threads: int = None,
                 use_direct_yuv: bool = False, verbose: bool = False):
        self.noise_tolerance = noise_tolerance
        self.keyframe_interval = keyframe_interval
        self.min_diff_threshold = min_diff_threshold
        self.max_diff_threshold = max_diff_threshold
        self.bloom_threshold_modifier = bloom_threshold_modifier
        self.use_direct_yuv = use_direct_yuv
        self.verbose = verbose
        self.num_threads = max(1, (os.cpu_count() or 2) - 1) if num_threads is None else max(1, num_threads)  # ivc:714-717
        self.bloom_compressor = BloomFilterCompressor(verbose=False)   # the attribute ivc:927 needs
        self._streams: Dict[tuple, FrameStream] = {}

    def _estimate_noise_level(self, frame: np.ndarray) -> float:                  # ivc:727-746
        """N3: the 5x5 median runs on the device (k_median5, bit-exact with cv2.medianBlur); the float32 std is numpy's,
        exactly as in the reference."""
        a = np.ascontiguousarray(_frame_data(frame))
        if a.ndim != 2 or a.dtype not in (np.uint8, np.uint16):
            raise NotImplementedError("noise estimate is implemented for 2-D uint8/uint16 planes (the Y / gray plane)")
        smoothed = np.empty_like(a)
        _cabi.check(_cabi.lib().rbf_median_blur5(_cabi.ctx(), _cabi.ptr(a), a.shape[0], a.shape[1], a.dtype.itemsize,
                                                 _cabi.ptr(smoothed)), _cabi.ctx())
        noise = a.astype(np.float32) - smoothed.astype(np.float32)                 # ivc:741
        return np.std(noise)                                                       # ivc:744

    def _adaptive_diff_threshold(self, frame: np.ndarray) -> float:               # ivc:748-766
        noise_level = self._estimate_noise_level(frame)
        return max(self.min_diff_threshold, min(self.max_diff_threshold, noise_level * self.noise_tolerance))

    def _stream_for(self, shape, dtype, k1_only: bool = False, gray: bool = False) -> FrameStream:
        """Cached 2-frame device store per (shape, dtype, options).  Options are per-stream state of the C ABI, so several
        compressors (or threads with their own compressor) never flip a shared switch."""
        key = (tuple(shape), np.dtype(dtype).str, bool(k1_only), bool(gray))
        s = self._streams.get(key)
        if s is None:
            ch = shape[2] if len(shape) == 3 else 1
            s = FrameStream(shape[0], shape[1], ch, dtype, max_frames=2, max_pairs=1, k1_only=k1_only, gray_mode=gray)
            self._streams[key] = s
        return s

    @staticmethod
    def _bgr2gray(a: np.ndarray) -> np.ndarray:
        """cv2.cvtColor(a, cv2.COLOR_BGR2GRAY) for uint8/uint16 (OpenCV's 15-bit fixed point; ivc:794-795) -- used on the host
        only to feed the adaptive-threshold noise estimate; the mask itself is computed by K1 in gray mode."""
        x = a.astype(np.uint32)
        return ((x[:, :, 0] * 3735 + x[:, :, 1] * 19235 + x[:, :, 2] * 9798 + 16384) >> 15).astype(a.dtype)

    def _calculate_frame_diff(self, prev_frame, curr_frame, threshold: Optional[float] = None):
        """ivc:768-847 -> (binary_diff uint8 HxW, changed_values, diff_density).  The mask is computed by K1: on the first
        channel (Y) for `use_direct_yuv` frames, on the BGR->gray conversion otherwise (ivc:788-795), or on the single plane."""
        pd, cd = _frame_data(prev_frame), _frame_data(curr_frame)
        is_color = pd.ndim > 2 and pd.shape[2] > 1
        gray = is_color and not (self.use_direct_yuv and pd.shape[2] >= 3)
        if gray and pd.shape[2] != 3:
            raise NotImplementedError("BGR->gray masks are implemented for 3-channel frames (cv2.COLOR_BGR2GRAY, ivc:794-795)")
        if pd.dtype not in (np.uint8, np.uint16) or pd.shape != cd.shape or pd.dtype != cd.dtype:
            raise ValueError("frames must be equal-shape uint8/uint16 arrays")
        if threshold is None:                                  # ivc:804-805: adaptive threshold from the current Y / gray plane
            plane = (self._bgr2gray(cd) if gray else cd[:, :, 0].copy()) if is_color else cd.copy()
            threshold = self._adaptive_diff_threshold(plane)
        st = self._stream_for(pd.shape, pd.dtype, k1_only=True, gray=gray)
        st.upload(np.stack([pd, cd]))
        res = st.encode([0], [1], float(threshold))[0]
        _, _, flat = st.fetch(0)                               # k1_only stream: the mask is the only output
        binary_diff = flat.reshape(pd.shape[0], pd.shape[1]).astype(np.uint8)
        vals = st.gather_changed(1)[0]                        # N1: ordered gather on the device (ivc:810-842)
        if is_color and self.use_direct_yuv and hasattr(curr_frame, "yuv_info"):
            changed = vals.astype(np.uint8)                   # ivc:825 allocates uint8: 16-bit samples are truncated there too
        else:
            changed = vals.copy()                             # ivc:832-842 keep the frame dtype
        density = res.ones / binary_diff.size                  # ivc:845
        self._last_pair_result = res
        return binary_diff, changed, density

    def _apply_frame_diff(self, base_frame, diff_mask: np.ndarray, changed_values: np.ndarray):   # ivc:849-909
        """N2: the scatter runs on the device (k_gather_scatter); the result is a copy of base_frame's type."""
        nxt = base_frame.copy()
        data = _frame_data(nxt)
        vals = np.asarray(changed_values)
        if data.dtype not in (np.uint8, np.uint16) or vals.dtype != data.dtype or not (data.ndim == 2 or data.shape[2] == 3):
            rows, cols = np.where(diff_mask == 1)              # formats outside the device store: host indexing
            ch = data.shape[2] if data.ndim == 3 else 1
            if len(vals) == len(rows) * ch:
                data[rows, cols] = vals.reshape(-1, ch) if ch > 1 else vals
        else:
            st = self._stream_for(data.shape, data.dtype, k1_only=True)
            st.upload(np.ascontiguousarray(data)[None], first=0)
            st.apply_diff(0, 1, diff_mask, vals)               # value-count mismatch leaves the base unchanged (ivc:882)
            data[...] = st.download(1)
        if self.use_direct_yuv and hasattr(nxt, "yuv_info") and data.ndim == 3:
            nxt.yuv_info["y_plane"] = data[:, :, 0].copy()
            nxt.yuv_info["u_plane"] = data[:, :, 1].copy()
            nxt.yuv_info["v_plane"] = data[:, :, 2].copy()
        return nxt

    def _compress_frame_differences(self, binary_diff: np.ndarray, changed_values: np.ndarray) -> Tuple[bytes, float]:
        """ivc:911-967: `<f` p | `<I` n | `<f` k | `<I` l | `<I` |w| | packbits(bitmap) | packbits(witness) | zlib(values)."""
        flat = binary_diff.flatten()
        bitmap, witness, p, n, _ = self.bloom_compressor.compress(flat)
        buf = io.BytesIO()
        buf.write(struct.pack("<f", p))
        buf.write(struct.pack("<I", n))
        k, l = self.bloom_compressor._calculate_optimal_params(n, p)     # ivc:937
        buf.write(struct.pack("<f", k))
        buf.write(struct.pack("<I", len(bitmap)))
        buf.write(struct.pack("<I", len(witness)))
        bb = np.packbits(bitmap).tobytes()
        buf.write(struct.pack("<I", len(bb)))
        buf.write(bb)
        wb = np.packbits(np.array(witness, dtype=np.uint8)).tobytes()
        buf.write(struct.pack("<I", len(wb)))
        buf.write(wb)
        vb = zlib.compress(changed_values.tobytes(), level=9)
        buf.write(struct.pack("<I", len(vb)))
        buf.write(struct.pack("<I", len(changed_values)))
        buf.write(vb)
        original_size = n + len(changed_values) * 8
        return buf.getvalue(), buf.tell() * 8 / original_size

    def _decompress_frame_differences(self, compressed_data: bytes, frame_shape, k_exact: Optional[float] = None):
        """ivc:969-1027.  `k_exact` (not in the reference) overrides the float32 k of the payload -- the reference
        decodes with the rounded k (ivc:938/986), which can break the round trip (SURVEY.md hard part 3i)."""
        buf = io.BytesIO(compressed_data)
        p = struct.unpack("<f", buf.read(4))[0]
        n = struct.unpack("<I", buf.read(4))[0]
        k = struct.unpack("<f", buf.read(4))[0]
        bitmap_length = struct.unpack("<I", buf.read(4))[0]
        witness_length = struct.unpack("<I", buf.read(4))[0]
        bsz = struct.unpack("<I", buf.read(4))[0]
        bloom_bitmap = np.unpackbits(np.frombuffer(buf.read(bsz), dtype=np.uint8))[:bitmap_length]
        wsz = struct.unpack("<I", buf.read(4))[0]
        witness = np.unpackbits(np.frombuffer(buf.read(wsz), dtype=np.uint8))[:witness_length].tolist()
        vsz = struct.unpack("<I", buf.read(4))[0]
        vcount = struct.unpack("<I", buf.read(4))[0]
        changed = np.frombuffer(zlib.decompress(buf.read(vsz)), dtype=np.uint8)[:vcount]
        if witness_length > 0:
            flat = self.bloom_compressor.decompress(bloom_bitmap, witness, n, k if k_exact is None else k_exact)
        else:
            flat = bloom_bitmap
        if len(frame_shape) == 3 and frame_shape[2] > 1:
            binary_diff = flat.reshape((frame_shape[0], frame_shape[1]))
        else:
            binary_diff = flat.reshape(frame_shape)
        return binary_diff, changed

    def compress_frame(self, frame, is_keyframe: bool = True):                    # ivc:1029-1104
        if not is_keyframe:
            raise ValueError("Non-keyframe compression should be handled by compress_video")
        body = FixedVideoCompressor(verbose=False).compress_frame(frame)
        data = struct.pack("<B", 1) + body                                         # ivc:1053: type tag 1 = keyframe
        meta = {"type": "keyframe", "shape": frame.shape, "original_size": frame.nbytes, "compressed_size": len(data),
                "compression_ratio": len(data) / frame.nbytes, "has_yuv_info": hasattr(frame, "yuv_info")}
        return data, meta

    def decompress_frame(self, compressed_data: bytes):                            # ivc:1106-1234
        if compressed_data[0] != 1:
            raise ValueError(f"Unknown frame type: {compressed_data[0]}")
        frame = FixedVideoCompressor(verbose=False).decompress_frame(compressed_data[1:])
        if hasattr(frame, "yuv_info") and not self.use_direct_yuv:                 # ivc:1163
            return frame.data
        return frame


_INTER_TAG_V1 = b"\xff\xff\xff\xffRBF1"   # round-1 layout: raw-passthrough masks stored as plain np.packbits bytes
_INTER_TAG = b"\xff\xff\xff\xffRBF2"      # current: raw-passthrough masks zlib-compressed (a static scene costs ~1 KB, not n/8 B)
# neither can be a FixedVideoCompressor payload (height 0xFFFFFFFF).  NOTE: inter payloads exist only in this implementation --
# the reference's decoder knows keyframes only (ivc:1124); files written with keyframe_interval=1 are interchangeable.


class ImprovedVideoCompressor:
    """ivc.ImprovedVideoCompressor (ivc:309-523) with the GOP loop wired in.

    Frame i is a keyframe when i % keyframe_interval == 0 (zlib codec, byte-identical to the reference's
    payload); otherwise it is coded against the ORIGINAL previous frame: K1 mask -> Bloom + witness coder ->
    changed pixel values (zlib).  `inter_frame_mode`:
      "lossless"  (default) mask = any byte of the pixel differs, so reconstruction is always exact;
      "reference" mask = |dY| > inter_frame_threshold exactly as _calculate_frame_diff (ivc:788-808); a frame whose
                  unflagged pixels changed (chroma-only or sub-threshold changes) falls back to a keyframe.
    The entropy stage (zlib level 9, ivc:956 / fvc:31) stays on the CPU but runs in a thread pool (`num_threads`; zlib
    releases the GIL), and a group of `batch_size` inter frames costs ONE encode call and ONE batched device->host copy.
    """

    def __init__(self, noise_tolerance: float = 10.0, keyframe_interval: int = 30, min_diff_threshold: float = 3.0,
                 max_diff_threshold: float = 30.0, bloom_threshold_modifier: float = 1.0, batch_size: int = 30,
                 num_threads: int = None, use_direct_yuv: bool = False, verbose: bool = False):
        self.noise_tolerance = noise_tolerance
        self.keyframe_interval = keyframe_interval
        self.min_diff_threshold = min_diff_threshold
        self.max_diff_threshold = max_diff_threshold
        self.bloom_threshold_modifier = bloom_threshold_modifier
        self.batch_size = batch_size
        self.num_threads = max(1, min(32, (os.cpu_count() or 2))) if num_threads is None else max(1, int(num_threads))
        self.use_direct_yuv = use_direct_yuv
        self.verbose = verbose
        self.compressor = FixedVideoCompressor(verbose=verbose)                    # ivc:356
        self.inter_frame_mode = "lossless"
        self.inter_frame_threshold = 0.0
        _cabi.ctx()                                                                 # fail now if there is no B200

    # ------------------------------------------------------------------ encode
    @staticmethod
    def _inter_payload(shape, itemsize, ch, r, bm_row, wt_row, mask_row, values) -> bytes:
        """Assemble one inter-frame payload (runs in a worker thread; the zlib calls release the GIL)."""
        vz = zlib.compress(values.tobytes(), 9)
        hdr = _INTER_TAG + struct.pack("<IIIBB", shape[0], shape[1], itemsize, ch, 1 if r.raw else 0)
        body = struct.pack("<dIIQ", r.k, r.l, r.wlen, r.ones)
        if r.raw:                                              # passthrough branch (ivc:215-225): the mask itself, np.packbits order
            n = shape[0] * shape[1]
            raw_bits = np.packbits(np.unpackbits(mask_row, bitorder="little")[:n]).tobytes()
            rz = zlib.compress(raw_bits, 9)
            body += struct.pack("<I", len(rz)) + rz + struct.pack("<I", 0)
        else:
            nb, nw = (r.l + 7) // 8, (r.wlen + 7) // 8
            body += struct.pack("<I", nb) + bm_row[:nb].tobytes() + struct.pack("<I", nw) + wt_row[:nw].tobytes()
        body += struct.pack("<II", len(vz), values.size) + vz
        return hdr + body

    def _encode_inter_frames(self, datas: List[np.ndarray], inter: List[int], pool) -> Dict[int, object]:
        """Futures of the inter-frame payloads for frame indices `inter` (each coded against frame i-1); None = keyframe instead."""
        out: Dict[int, object] = {}
        if not inter:
            return out
        shape, dtype = datas[0].shape, datas[0].dtype
        ch = shape[2] if len(shape) == 3 else 1
        group = max(2, int(self.batch_size))
        st = FrameStream(shape[0], shape[1], ch, dtype, max_frames=2 * group, max_pairs=group,
                         mask_mode=1 if self.inter_frame_mode == "lossless" else 0)
        try:
            for g0 in range(0, len(inter), group):
                idxs = inter[g0:g0 + group]
                need = sorted(set(idxs) | {i - 1 for i in idxs})
                slot = {f: s for s, f in enumerate(need)}
                st.upload(np.stack([datas[f] for f in need]))
                res = st.encode([slot[i - 1] for i in idxs], [slot[i] for i in idxs], float(self.inter_frame_threshold))
                gathered = st.gather_changed(len(idxs))            # N1: changed values of every pair, one launch, one copy
                any_raw = any(r.raw for r in res)
                bms, wts, masks = st.fetch_batch(0, len(idxs), want_masks=any_raw)   # one D2H per kind, one sync per group
                for j, i in enumerate(idxs):
                    r = res[j]
                    if r.resid and self.inter_frame_mode != "lossless":
                        out[i] = None                              # not exactly representable: keyframe instead
                        continue
                    out[i] = pool.submit(self._inter_payload, shape, dtype.itemsize, ch, r, bms[j], wts[j],
                                         masks[j] if (masks is not None and r.raw) else None, gathered[j])
        finally:
            st.close()
        return out

    def compress_video(self, frames: List[np.ndarray], output_path: str = None, input_color_space: str = "BGR") -> Dict:
        if not frames:
            raise ValueError("No frames provided for compression")                 # ivc:372-373
        start_time = time.time()
        if input_color_space.upper() == "YUV":                                      # ivc:378-384 (wraps in place)
            self.use_direct_yuv = True
            for i in range(len(frames)):
                if not hasattr(frames[i], "yuv_info"):
                    frames[i] = self.compressor.add_yuv_info_to_frame(frames[i])
        original_size = sum(frame.nbytes for frame in frames)
        datas = [np.ascontiguousarray(_frame_data(f)) for f in frames]
        ki = max(1, int(self.keyframe_interval))
        uniform = all(d.shape == datas[0].shape and d.dtype == datas[0].dtype for d in datas) and \
            datas[0].dtype in (np.uint8, np.uint16) and (datas[0].ndim == 2 or datas[0].shape[2] == 3)
        inter = [i for i in range(len(frames)) if i % ki != 0] if uniform else []
        from concurrent.futures import ThreadPoolExecutor
        compressed_frames: List[bytes] = []
        keyframes = 0
        with ThreadPoolExecutor(self.num_threads) as pool:
            # keyframes (zlib level 9 of whole frames, fvc:31) start in the pool first; the GPU encodes the groups meanwhile
            inter_set = set(inter)
            key_jobs = {i: self.compressor.compress_frame_async(frames[i], pool) for i in range(len(frames)) if i not in inter_set}
            payloads = self._encode_inter_frames(datas, inter, pool)
            for i, f in enumerate(frames):
                fut = payloads.get(i)
                if fut is None:
                    kj = key_jobs.get(i)
                    pl = kj() if kj is not None else self.compressor.compress_frame(f)
                    keyframes += 1
                else:
                    pl = fut.result()
                compressed_frames.append(pl)
        if output_path:                                                             # ivc:393-406
            os.makedirs(os.path.dirname(os.path.abspath(output_path)), exist_ok=True)
            with open(output_path, "wb") as fh:
                fh.write(b"BFVC")
                fh.write(struct.pack("<I", len(frames)))
                for c in compressed_frames:
                    fh.write(struct.pack("<I", len(c)))
                    fh.write(c)
        if output_path and os.path.exists(output_path):
            compressed_size = os.path.getsize(output_path)
        else:
            compressed_size = sum(len(c) for c in compressed_frames) + 4 + 4 + 4 * len(compressed_frames)   # ivc:413-415
        self._last_compressed_frames = compressed_frames
        ratio = compressed_size / original_size
        dt = time.time() - start_time
        results = {"frame_count": len(frames), "original_size": original_size, "compressed_size": compressed_size,
                   "compression_ratio": ratio, "space_savings": 1.0 - ratio, "compression_time": dt,
                   "frames_per_second": len(frames) / dt if dt > 0 else float("inf"), "keyframes": keyframes,
                   "keyframe_ratio": keyframes / len(frames), "output_path": output_path,
                   "color_space": input_color_space, "overall_ratio": ratio}       # ivc:424-437
        if self.verbose:
            print(f"Compression Ratio: {ratio:.4f}  keyframes: {keyframes}/{len(frames)}")
        return results

    # ------------------------------------------------------------------ decode
    def _decode_inter(self, payload: bytes, prev):
        v1 = payload[:len(_INTER_TAG_V1)] == _INTER_TAG_V1
        pos = len(_INTER_TAG)
        h, w, isz, ch, raw = struct.unpack_from("<IIIBB", payload, pos)
        pos += struct.calcsize("<IIIBB")
        k, l, wlen, ones = struct.unpack_from("<dIIQ", payload, pos)
        pos += struct.calcsize("<dIIQ")
        (bl,) = struct.unpack_from("<I", payload, pos); pos += 4
        bbytes = np.frombuffer(payload, dtype=np.uint8, count=bl, offset=pos); pos += bl
        (wl,) = struct.unpack_from("<I", payload, pos); pos += 4
        wbytes = np.frombuffer(payload, dtype=np.uint8, count=wl, offset=pos); pos += wl
        vlen, vcount = struct.unpack_from("<II", payload, pos); pos += 8
        dtype = np.uint8 if isz == 1 else np.uint16
        values = np.frombuffer(zlib.decompress(payload[pos:pos + vlen]), dtype=dtype)[:vcount]
        n = h * w
        pdata = _frame_data(prev)
        exp_shape = (h, w, ch) if ch > 1 else (h, w)
        if pdata.shape != exp_shape or pdata.dtype != np.dtype(dtype):
            raise ValueError(f"inter frame {exp_shape}/{np.dtype(dtype)} does not match the previous frame {pdata.shape}/{pdata.dtype}")
        if values.size != ones * ch:
            raise ValueError(f"corrupt inter frame: {values.size} changed values for {ones} changed pixels x {ch} channels")
        if raw:
            rbits = bbytes if v1 else np.frombuffer(zlib.decompress(bbytes.tobytes()), dtype=np.uint8)
            mask = np.unpackbits(rbits)[:n]
        else:
            bitmap = np.unpackbits(bbytes)[:l]
            witness = np.unpackbits(wbytes)[:wlen]
            mask = BloomFilterCompressor().decompress(bitmap, witness, n, k)
        st = getattr(self, "_dec_stream", None)
        if st is None or (st.H, st.W, st.C, st.dtype) != (h, w, ch, np.dtype(dtype)):
            st = FrameStream(h, w, ch, dtype, max_frames=2, max_pairs=1, k1_only=True)
            self._dec_stream, self._dec_slot, self._dec_src = st, 0, None
        if self._dec_src is not prev:                             # previous frame is not the one resident on the device
            st.upload(np.ascontiguousarray(pdata)[None], first=0)
            self._dec_slot = 0
        nxt_slot = 1 - self._dec_slot
        applied = st.apply_diff(self._dec_slot, nxt_slot, mask, values)     # N2: scatter on the device
        if applied != ones:                                       # the reference would silently return the base frame (ivc:882)
            self._dec_src = None
            raise ValueError(f"corrupt inter frame: the decoded mask selects {int(np.count_nonzero(mask))} pixels, the payload "
                             f"announces {ones}")
        out = st.download(nxt_slot)
        self._dec_slot = nxt_slot
        res = YUVFrame(out) if hasattr(prev, "yuv_info") else out
        self._dec_src = res
        return res

    def decompress_video(self, input_path: str = None, output_path: Optional[str] = None,
                         compressed_frames: List[bytes] = None, metadata: Dict = None) -> List[np.ndarray]:
        if input_path and os.path.exists(input_path):                              # ivc:471-485
            with open(input_path, "rb") as fh:
                magic = fh.read(4)
                if magic != b"BFVC":
                    raise ValueError(f"Invalid file format: {magic}")
                count = struct.unpack("<I", fh.read(4))[0]
                compressed_frames = []
                for _ in range(count):
                    size = struct.unpack("<I", fh.read(4))[0]
                    compressed_frames.append(fh.read(size))
        if not compressed_frames:
            raise ValueError("No compressed frames provided")                       # ivc:487-488
        frames = []
        for c in compressed_frames:
            if c[:len(_INTER_TAG)] in (_INTER_TAG, _INTER_TAG_V1):
                if not frames:
                    raise ValueError("inter frame without a preceding frame")
                frames.append(self._decode_inter(c, frames[-1]))
            else:
                frames.append(self.compressor.decompress_frame(c))
        if output_path:
            self.save_frames_as_video(frames, output_path)
        return frames

    def verify_lossless(self, original_frames, decompressed_frames) -> Dict:       # ivc:506-523
        return self.compressor.verify_lossless(original_frames, decompressed_frames)

    def save_frames_as_video(self, frames, output_path: str, fps: int = 30) -> str:   # ivc:525-581 (host glue, cv2)
        import cv2
        if not frames:
            raise ValueError("No frames provided")
        os.makedirs(os.path.dirname(os.path.abspath(output_path)), exist_ok=True)
        h, w = frames[0].shape[:2]
        color = len(frames[0].shape) > 2
        out = cv2.VideoWriter(output_path, cv2.VideoWriter_fourcc(*"mp4v"), fps, (w, h), isColor=color)
        if not out.isOpened():
            raise ValueError(f"Could not create video writer for {output_path}")
        for f in frames:
            d = _frame_data(f)
            if color and hasattr(f, "yuv_info") and self.use_direct_yuv:
                d = cv2.cvtColor(d, cv2.COLOR_YUV2BGR)
            elif not color:
                d = cv2.cvtColor(d, cv2.COLOR_GRAY2BGR)
            elif d.shape[2] == 3 and not hasattr(f, "yuv_info"):
                d = cv2.cvtColor(d, cv2.COLOR_RGB2BGR)
            out.write(d)
        out.release()
        return output_path
