// rbf_kernels.cuh -- device-side job descriptors and launcher prototypes shared by
// rbf_kernels.cu (kernels) and rbf_api.cu (C ABI + host pipeline).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "rbf_hash.cuh"

namespace rbf {

// One Bloom filter (= one inter-frame mask, or one user filter).  Device-resident array.
// Internal bit order everywhere on the device is LSB-first in little-endian 32-bit words
// (bit j -> word j>>5, bit j&31); conversion to the reference's np.packbits order
// (MSB-first per byte, ivc:945,951) is a per-byte bit reversal done once on the way out.
struct FrameJob {
    uint32_t n;           // positions (H*W)
    uint32_t l;           // Bloom size in bits; 0 => raw passthrough (ivc:215-225), no work
    uint32_t floor_k;     // ivc:57
    uint32_t has_act;     // p_activation > 0
    uint64_t act_T;       // h < act_T  <=>  h/(2^64-1) < p_activation   (ivc:95-97)
    uint64_t seed1, seed2, seedA;   // ivc:62-63, ivc:94
    FastMod fm;           // m = l
    const uint32_t* mask; // n bits, natural packing, >= 16 B zero padding after the last word
    uint32_t* bits;       // l bits (ceil(l/32) words rounded up to 16 B), zeroed before insert
    uint32_t* pass;       // Bloom-test pass mask, century-padded: 4 words (128 bit) per 100 positions
    uint32_t* witness;    // witness bit stream (K3b output / K4b input), zeroed before K3b
    uint32_t* out_mask;   // decode output, natural packing, zeroed before K4b
    uint32_t wlen_in;     // decode: number of valid witness bits
    uint32_t neg_m;       // 2^32 - l, for the one-instruction remainder step of the query kernels
};

// One frame pair for the threshold kernel (ivc:788-808).
struct PairJob {
    const uint8_t* prev;
    const uint8_t* curr;
    uint32_t* mask;       // n bits natural packing
};

struct GatherJob {
    const uint32_t* mask;     // n bits, natural packing
    const uint8_t* frame;     // gather: source (curr) frame; scatter: unused
    uint8_t* values;          // gather: output; scatter: input (rank-ordered pixel values)
    uint8_t* out_frame;       // scatter: destination frame (already holds the base frame)
    uint32_t npix;
    uint32_t pix_bytes;
};


// launchers (all asynchronous on `st`); return cudaError_t of the launch
cudaError_t launch_threshold(const PairJob* d_pairs, int F, uint32_t npix, int channels, int sample_bytes,
                             int thr_int, int any_mode, int gray_mode, uint32_t* d_ones, uint32_t* d_resid, int variant,
                             int sm_count, int ctas_per_sm, cudaStream_t st);
// single-image K1 (bloom_compress.py:67-87): PairJob::curr is the image, prev is unused; thr_int = floor of the Python threshold
cudaError_t launch_binarize(const PairJob* d_images, int F, uint32_t npix, int channels, int sample_bytes, int thr_int,
                            uint32_t* d_ones, int sm_count, int ctas_per_sm, cudaStream_t st);
cudaError_t launch_insert(const FrameJob* d_jobs, int F, uint32_t max_centuries, int variant, int sm_count, cudaStream_t st);
cudaError_t launch_query(const FrameJob* d_jobs, const uint32_t* d_cent_prefix, int F, uint32_t total_centuries,
                         uint32_t max_l_bits, int variant, int sm_count, int smem_bytes_cap, int tile_warps, cudaStream_t st);
cudaError_t launch_witness(const FrameJob* d_jobs, int F, uint32_t max_centuries, int sm_count, uint32_t* d_scratch, uint32_t* d_wlen,
                           cudaStream_t st);
cudaError_t launch_expand(const FrameJob* d_jobs, int F, uint32_t max_centuries, int sm_count, uint32_t* d_scratch, uint32_t* d_consumed,
                          cudaStream_t st);
uint32_t gather_chunks(uint32_t npix);
cudaError_t launch_gather_scatter(const GatherJob* d_jobs, int F, int scatter, uint32_t npix, uint32_t pix_bytes, uint32_t* d_counts,
                                  uint32_t* d_totals, cudaStream_t st);
cudaError_t launch_median5(const void* d_in, uint32_t pix_stride, uint32_t H, uint32_t W, int sample_bytes, void* d_out, cudaStream_t st);
cudaError_t launch_bitrev(uint32_t* d_words, size_t nwords, cudaStream_t st);
cudaError_t launch_unpack_bits(const uint32_t* d_words, uint8_t* d_out, size_t nbits, cudaStream_t st);
cudaError_t launch_unpack_bits_msb(const uint32_t* d_words, uint8_t* d_out, size_t nbits, cudaStream_t st);
cudaError_t launch_popcount(const uint32_t* d_words, size_t nwords, uint32_t* d_out, cudaStream_t st);
cudaError_t launch_count_diff(const uint32_t* a, const uint32_t* b, size_t stride_words, size_t nwords, int F,
                              uint32_t* d_out, cudaStream_t st);
cudaError_t launch_pack_bytes(const uint8_t* d_bytes, uint32_t* d_words, size_t nbits, cudaStream_t st);

// explicit-item kernels (drop-in RationalBloomFilter.add_index/check_index, rbf add/contains)
cudaError_t launch_items_u32(const FrameJob* d_job, const uint32_t* d_items, uint32_t count, uint8_t* d_result,
                             int insert, cudaStream_t st);
cudaError_t launch_items_str(const FrameJob* d_job, const uint8_t* d_blob, const uint64_t* d_offs, uint32_t count,
                             uint8_t* d_result, int insert, int standard_k, cudaStream_t st);
cudaError_t launch_hash_debug(const uint32_t* d_items, uint32_t count, uint64_t seed, uint64_t* d_out, int mode,
                              cudaStream_t st);

// exchange over peer memory: store `pairs` slots of slot_w words into recv[r] + dst_off_w of every rank, then signal `seq`
cudaError_t launch_push_slots(const uint32_t* d_bits, size_t stride_w, uint32_t slot_w, uint32_t pairs, uint32_t* const* recv,
                              uint32_t* const* flags, int nranks, int rank, size_t dst_off_w, uint32_t seq, int sm_count, cudaStream_t st);
cudaError_t launch_peer_wait(const uint32_t* d_flags, int nranks, uint32_t seq, long long timeout_cycles, uint32_t* d_err, cudaStream_t st);

int query_max_smem_bytes();

}  // namespace rbf
