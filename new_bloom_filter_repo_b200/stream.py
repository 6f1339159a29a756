"""
FrameStream: Python handle on the C ABI's rbf_stream -- a device-resident store of
interleaved H x W x C frames plus the per-pair outputs of the batched hot path
(K1 threshold -> exact (k, l, T) on the host -> K2 insert -> K3 query -> K3b witness).
No PyTorch; device memory belongs to the C library.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import numpy as np

from . import _cabi
from ._cabi import MaskInfo


class PairResult:
    """What BloomFilterCompressor.compress returns for one frame pair (ivc:266), in wire form."""
    __slots__ = ("n", "ones", "resid", "l", "wlen", "p", "k", "raw", "floor_k", "act_T")

    def __init__(self, mi: MaskInfo):
        self.n, self.ones, self.resid, self.l, self.wlen = int(mi.n), int(mi.ones), int(mi.resid), int(mi.l), int(mi.wlen)
        self.p, self.k, self.raw, self.floor_k, self.act_T = float(mi.p), float(mi.k), bool(mi.raw), int(mi.floor_k), int(mi.act_T)

    def __repr__(self):
        return "PairResult(n=%d ones=%d l=%d wlen=%d k=%r raw=%s)" % (self.n, self.ones, self.l, self.wlen, self.k, self.raw)


class FrameStream:
    def __init__(self, height: int, width: int, channels: int = 3, dtype=np.uint8, max_frames: int = 2,
                 max_pairs: Optional[int] = None, k1_only: bool = False, mask_mode: int = 0, gray_mode: bool = False,
                 images: bool = False):
        """images=True: a stream of single images (rbf_stream_create_images) -- "pair" i of encode() is image curr_idx[i]
        (prev_idx == curr_idx) and K1 is _binarize_image (bloom_compress.py:67-87); max_frames images, as many pairs."""
        dt = np.dtype(dtype)
        if dt not in (np.dtype(np.uint8), np.dtype(np.uint16)):
            raise ValueError("frames must be uint8 or uint16")
        self.H, self.W, self.C, self.dtype = int(height), int(width), int(channels), dt
        self.max_frames = int(max_frames)
        self.max_pairs = int(max_pairs if max_pairs is not None else max(1, max_frames - 1))
        self.npix = self.H * self.W
        self._h = C.c_void_p()
        if images:
            self.max_pairs = self.max_frames
            _cabi.check(_cabi.lib().rbf_stream_create_images(_cabi.ctx(), self.H, self.W, self.C, dt.itemsize, self.max_frames,
                                                             C.byref(self._h)), _cabi.ctx())
        else:
            _cabi.check(_cabi.lib().rbf_stream_create(_cabi.ctx(), self.H, self.W, self.C, dt.itemsize, self.max_frames,
                                                      self.max_pairs, C.byref(self._h)), _cabi.ctx())
        self._infos = (MaskInfo * self.max_pairs)()
        self.pairs = 0
        self.k1_only = bool(k1_only)
        for key, val in (("k1_only", int(bool(k1_only))), ("mask_mode", int(mask_mode)), ("gray_mode", int(bool(gray_mode)))):
            self.set_option(key, val)

    def set_option(self, key: str, value: int) -> None:
        """Per-stream option of the C ABI (rbf_stream_set_option): k1_only, mask_mode, gray_mode."""
        _cabi.check(_cabi.lib().rbf_stream_set_option(self._h, key.encode(), int(value)), _cabi.ctx())
        if key == "k1_only":
            self.k1_only = bool(value)

    def close(self):
        if getattr(self, "_h", None):
            _cabi.lib().rbf_stream_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ data movement
    def upload(self, frames: np.ndarray, first: int = 0) -> None:
        """frames: [count, H, W, C] (or [H, W, C]) contiguous array of the stream's dtype."""
        a = np.ascontiguousarray(frames)
        if a.ndim == 3 and self.C > 1 or (a.ndim == 2 and self.C == 1):
            a = a[None]
        if a.dtype != self.dtype or a.shape[1:3] != (self.H, self.W):
            raise ValueError("frame shape/dtype mismatch: %r %r" % (a.shape, a.dtype))
        _cabi.check(_cabi.lib().rbf_stream_upload(self._h, int(first), int(a.shape[0]), _cabi.ptr(a)), _cabi.ctx())

    # ------------------------------------------------------------------ the hot path
    def encode(self, prev_idx: Sequence[int], curr_idx: Sequence[int], threshold: float,
               seeds=_cabi.IVC_SEEDS, k_override=None, l_override=None) -> List[PairResult]:
        p = np.ascontiguousarray(np.asarray(prev_idx, dtype=np.uint32))
        c = np.ascontiguousarray(np.asarray(curr_idx, dtype=np.uint32))
        if p.shape != c.shape or p.ndim != 1:
            raise ValueError("prev_idx and curr_idx must be 1-D and equally long")
        sd = _cabi.seeds_struct(seeds)
        ko = lo = None
        if k_override is not None:
            ko = np.ascontiguousarray(np.asarray(k_override, dtype=np.float64))
            lo = np.ascontiguousarray(np.asarray(l_override, dtype=np.uint64))
        _cabi.check(_cabi.lib().rbf_stream_encode(self._h, _cabi.ptr(p), _cabi.ptr(c), p.size, float(threshold), C.byref(sd),
                                                  _cabi.ptr(ko) if ko is not None else None,
                                                  _cabi.ptr(lo) if lo is not None else None, self._infos), _cabi.ctx())
        self.pairs = int(p.size)
        return [PairResult(self._infos[i]) for i in range(self.pairs)]

    def encode_consecutive(self, nframes: int, threshold: float, **kw) -> List[PairResult]:
        idx = np.arange(nframes, dtype=np.uint32)
        return self.encode(idx[:-1], idx[1:], threshold, **kw)

    def fetch(self, pair: int, want_mask: bool = True):
        """-> (bitmap_packbits uint8[ceil(l/8)], witness_packbits uint8[ceil(wlen/8)], mask uint8[n] or None)."""
        mi = self._infos[pair]
        if self.k1_only:                                   # the encode stopped after K1: only the mask exists
            bm, wt = np.zeros(0, dtype=np.uint8), np.zeros(0, dtype=np.uint8)
        else:
            bm = np.zeros((int(mi.l) + 7) // 8, dtype=np.uint8)
            wt = np.zeros((int(mi.wlen) + 7) // 8, dtype=np.uint8)
        mk = np.zeros((self.npix + 7) // 8, dtype=np.uint8) if want_mask else None
        _cabi.check(_cabi.lib().rbf_stream_fetch(self._h, int(pair), _cabi.ptr(bm) if bm.size else None,
                                                 _cabi.ptr(wt) if wt.size else None,
                                                 _cabi.ptr(mk) if mk is not None else None), _cabi.ctx())
        mask = np.unpackbits(mk, bitorder="little")[: self.npix] if mk is not None else None
        return bm, wt, mask

    def fetch_batch(self, first: int, count: int, want_masks: bool = False):
        """Packed outputs of pairs [first, first+count) with one D2H copy per kind and one sync:
        -> (bitmaps uint8[count, bslot], witnesses uint8[count, wslot], masks uint8[count, ceil(n/8)] or None);
        pair j's bitmap is bitmaps[j, :ceil(l_j/8)] (np.packbits order), its witness witnesses[j, :ceil(wlen_j/8)]."""
        infos = [self._infos[first + j] for j in range(count)]
        bslot = max(16, (max((int(m.l) + 7) // 8 for m in infos) + 15) // 16 * 16)
        wslot = max(16, (max((int(m.wlen) + 7) // 8 for m in infos) + 15) // 16 * 16)
        bm = np.zeros((count, bslot), dtype=np.uint8)
        wt = np.zeros((count, wslot), dtype=np.uint8)
        mslot = (self.npix + 7) // 8
        mk = np.zeros((count, mslot), dtype=np.uint8) if want_masks else None
        coded = not self.k1_only
        _cabi.check(_cabi.lib().rbf_stream_fetch_batch(self._h, int(first), int(count), _cabi.ptr(bm) if coded else None, bslot,
                                                       _cabi.ptr(wt) if coded else None, wslot,
                                                       _cabi.ptr(mk) if mk is not None else None, mslot), _cabi.ctx())
        return bm, wt, mk

    def decode_verify(self, pairs: Optional[int] = None) -> np.ndarray:
        """Decode every encoded pair on the GPU from its own bitmap + witness (ivc:268-307) and
        return the number of mismatching mask words per pair (all zeros == round trip holds)."""
        n = self.pairs if pairs is None else int(pairs)
        out = np.zeros(n, dtype=np.uint64)
        _cabi.check(_cabi.lib().rbf_stream_decode_verify(self._h, n, _cabi.ptr(out)), _cabi.ctx())
        return out

    def decode(self, l, wlen, k, bitmaps: np.ndarray, witnesses: np.ndarray, seeds=_cabi.IVC_SEEDS):
        """Decode caller-supplied payloads of this stream's n positions at once (ivc:268-307, bc:307-346):
        payload i = (l[i], wlen[i], k[i]) with its packbits bitmap in bitmaps[i] and witness in witnesses[i] (uint8 [count, slot]).
        -> (masks uint8[count, ceil(n/8)] little bit order, consumed uint64[count] = Bloom-test passes per payload)."""
        lv = np.ascontiguousarray(np.asarray(l, dtype=np.uint64))
        wv = np.ascontiguousarray(np.asarray(wlen, dtype=np.uint64))
        kv = np.ascontiguousarray(np.asarray(k, dtype=np.float64))
        bm = np.ascontiguousarray(bitmaps, dtype=np.uint8)
        wt = np.ascontiguousarray(witnesses, dtype=np.uint8)
        count = lv.size
        if not (wv.size == kv.size == count == bm.shape[0] == wt.shape[0]):
            raise ValueError("l, wlen, k, bitmaps and witnesses must describe the same payloads")
        mslot = (self.npix + 7) // 8
        masks = np.empty((count, mslot), dtype=np.uint8)
        consumed = np.zeros(count, dtype=np.uint64)
        sd = _cabi.seeds_struct(seeds)
        _cabi.check(_cabi.lib().rbf_stream_decode(self._h, count, _cabi.ptr(lv), _cabi.ptr(wv), _cabi.ptr(kv), C.byref(sd),
                                                  _cabi.ptr(bm), bm.shape[1], _cabi.ptr(wt), wt.shape[1], _cabi.ptr(masks), mslot,
                                                  _cabi.ptr(consumed)), _cabi.ctx())
        self.pairs = 0
        return masks, consumed

    # ------------------------------------------------------------------ N1 / N2 (SURVEY 8f)
    def gather_changed(self, pairs: Optional[int] = None) -> List[np.ndarray]:
        """Per encoded pair: interleaved channel values of the current frame at the mask's set positions (ivc:810-842)."""
        n = self.pairs if pairs is None else int(pairs)
        offs = np.zeros(n + 1, dtype=np.uint64)
        _cabi.check(_cabi.lib().rbf_stream_gather_changed(self._h, n, None, 0, _cabi.ptr(offs)), _cabi.ctx())
        buf = np.empty(int(offs[-1]), dtype=np.uint8)
        if buf.size:
            _cabi.check(_cabi.lib().rbf_stream_gather_changed(self._h, n, _cabi.ptr(buf), buf.size, _cabi.ptr(offs)), _cabi.ctx())
        return [buf[int(offs[i]):int(offs[i + 1])].view(self.dtype) for i in range(n)]

    def apply_diff(self, base_frame: int, out_frame: int, mask: np.ndarray, values: np.ndarray) -> int:
        """store[out_frame] = store[base_frame] with masked pixels replaced by `values` (ivc:849-909); returns pixels applied."""
        mk = np.packbits(np.ascontiguousarray(mask, dtype=np.uint8).reshape(-1), bitorder="little")
        vals = np.ascontiguousarray(values).view(np.uint8).reshape(-1)
        applied = C.c_uint64()
        _cabi.check(_cabi.lib().rbf_stream_apply_diff(self._h, int(base_frame), int(out_frame), _cabi.ptr(mk),
                                                      _cabi.ptr(vals) if vals.size else None, vals.size, C.byref(applied)), _cabi.ctx())
        return int(applied.value)

    def download(self, frame: int) -> np.ndarray:
        shape = (self.H, self.W, self.C) if self.C > 1 else (self.H, self.W)
        out = np.empty(shape, dtype=self.dtype)
        _cabi.check(_cabi.lib().rbf_stream_download(self._h, int(frame), _cabi.ptr(out)), _cabi.ctx())
        return out

    def stage_ms(self) -> dict:
        out = (C.c_double * 6)()
        _cabi.check(_cabi.lib().rbf_stream_stage_ms(self._h, out), _cabi.ctx())
        return dict(zip(("k1_threshold", "front_k1_host_k2", "k2_insert", "k3_query", "k3b_witness", "encode_total"),
                        [float(x) for x in out]))

    def encode_host(self, frames: np.ndarray, threshold: float, seeds=_cabi.IVC_SEEDS, bitmap_slot: int = 0,
                    witness_slot: int = 0, out_bitmaps: np.ndarray = None, out_witness: np.ndarray = None):
        """End-to-end call: host frames in, packed bitmaps/witnesses back in host slots (copies included)."""
        a = np.ascontiguousarray(frames)
        nfr = a.shape[0]
        sd = _cabi.seeds_struct(seeds)
        _cabi.check(_cabi.lib().rbf_stream_encode_host(
            self._h, _cabi.ptr(a), nfr, float(threshold), C.byref(sd), self._infos,
            _cabi.ptr(out_bitmaps) if out_bitmaps is not None else None, int(bitmap_slot),
            _cabi.ptr(out_witness) if out_witness is not None else None, int(witness_slot)), _cabi.ctx())
        self.pairs = nfr - 1
        return [PairResult(self._infos[i]) for i in range(self.pairs)]
