"""
new_bloom_filter_repo_b200 -- B200-native (sm_100a) implementation of the rational-Bloom-filter
insert/query hot path of ross39/new_bloom_filter_repo, behind the reference's own Python API.

    from new_bloom_filter_repo_b200 import ImprovedVideoCompressor, RationalBloomFilter

Host code is Python calling hand-written CUDA through a C ABI (include/rbf_b200.h) with ctypes.
There is no CPU fallback: importing is cheap, but every entry point needs librbf_b200.so and a B200.
"""
from . import _cabi
from . import bloom_compress
from ._cabi import RbfError
from .improved_video_compressor import (BloomFilterCompressor, ImprovedVideoCompressor, VideoFrameCompressor)
from .improved_video_compressor import RationalBloomFilter as IndexRationalBloomFilter
from .rational_bloom_filter import RationalBloomFilter, StandardBloomFilter
from .fixed_video_compressor import FixedVideoCompressor, YUVFrame
from .stream import FrameStream, PairResult

__all__ = ["ImprovedVideoCompressor", "VideoFrameCompressor", "BloomFilterCompressor", "IndexRationalBloomFilter",
           "RationalBloomFilter", "StandardBloomFilter", "FixedVideoCompressor", "YUVFrame", "FrameStream",
           "PairResult", "RbfError"]
