/*
 * rbf_b200.h -- C ABI of the B200-native rational-Bloom-filter hot path.
 *
 * The reference (ross39/new_bloom_filter_repo @ 7e37ed8) is pure Python and has no FFI:
 * its "plugin interface" for this path is the Python class surface in
 * improved_video_compressor.py (ivc) and rational_bloom_filter.py (rbf).  Every entry
 * point below names the reference function(s) it replaces (file:line); INTEGRATION.md
 * shows the ctypes binding a maintainer adds on the reference side.
 *
 * Conventions
 *   - plain C types only; every function returns RBF_OK (0) or a negative rbf_status and never
 *     throws.  rbf_last_error(ctx) / rbf_last_global_error() return the message.
 *   - the caller owns host buffers; a context / stream / filter owns its device buffers.
 *   - one context per host thread (not internally thread-safe, like the single-threaded
 *     reference); one context is bound to one CUDA device and one CUDA stream.
 *   - there is NO CPU fallback: without a usable CUDA device rbf_ctx_create fails.
 *   - bit arrays cross this boundary either "unpacked" (one uint8 0/1 per bit, the
 *     reference's in-memory form, ivc:59) or "packbits" (numpy.packbits order, MSB first,
 *     the reference's wire form, ivc:945,951).  The name of each parameter says which.
 */
#ifndef RBF_B200_H
#define RBF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RBF_ABI_VERSION 2

typedef enum {
    RBF_OK = 0,
    RBF_ERR_INVALID = -1,     /* bad argument */
    RBF_ERR_CUDA = -2,        /* CUDA runtime error */
    RBF_ERR_NO_DEVICE = -3,   /* no usable GPU (there is no CPU fallback) */
    RBF_ERR_NCCL = -4,
    RBF_ERR_OOM = -5,
    RBF_ERR_STATE = -6
} rbf_status;

typedef struct rbf_ctx rbf_ctx;
typedef struct rbf_filter rbf_filter;
typedef struct rbf_stream rbf_stream;

/* Hash seeds of a filter variant: ivc:62-63 + ivc:94 (0x12345678, 0x87654321, 999);
 * rbf:100-101 + rbf:134 (0, 1, ceil(k*)); bloom_compress.py:163-164,195 (0, 1, 999). */
typedef struct {
    uint64_t h1, h2, act;
} rbf_seeds;

/* Per-mask result of the Bloom+witness coder, mirrors the tuple returned by
 * BloomFilterCompressor.compress (ivc:266) plus the parameters it derived. */
typedef struct {
    uint64_t n;        /* input length (ivc:208) */
    uint64_t ones;     /* np.sum(binary_input) (ivc:211) */
    uint64_t resid;    /* pixels with mask==0 whose bytes differ (inter-frame losslessness check; 0 for mask input) */
    uint64_t l;        /* Bloom length in bits (ivc:193); 0 when raw */
    uint64_t wlen;     /* witness length in bits (ivc:253) */
    uint64_t act_T;    /* activation threshold: h < act_T <=> h/(2^64-1) < p_activation (ivc:95-97) */
    double p;          /* density (ivc:212) */
    double k;          /* k* (ivc:185); 0 when raw */
    uint32_t floor_k;  /* ivc:57 */
    uint32_t raw;      /* 1: passthrough branch (ivc:215-218 or ivc:223-225): bitmap is the input, witness empty */
} rbf_mask_info;

/* ------------------------------------------------------------------ library / context */
int rbf_abi_version(void);
const char* rbf_last_global_error(void);
int rbf_ctx_create(int device_ordinal, rbf_ctx** out);
void rbf_ctx_destroy(rbf_ctx* ctx);
const char* rbf_last_error(const rbf_ctx* ctx);
int rbf_device_info(rbf_ctx* ctx, char* name, int name_len, int* sm_count, int* cc_major, int* cc_minor,
                    uint64_t* total_mem_bytes);
/* options: "k1_variant" (0 = vectorised loads, 1 = TMA bulk-copy ring), "query_smem_bytes" (cap), "query_variant",
 * "insert_variant", "host_chunk_frames", "encode_ranges" (1..8: K1/K2 pipelining depth of rbf_stream_encode),
 * "k1_ctas_per_sm" / "pipe_k1_ctas_per_sm" (K1 grid caps); "k1_only" / "mask_mode" here are only the defaults that
 * streams created afterwards inherit -- per-stream state lives in rbf_stream_set_option. */
int rbf_set_option(rbf_ctx* ctx, const char* key, int64_t value);
int64_t rbf_get_counter(rbf_ctx* ctx, const char* key);   /* "kernel_launches", "h2d_bytes", "d2h_bytes" */
int rbf_reset_counters(rbf_ctx* ctx);
int rbf_sync(rbf_ctx* ctx);
/* device-side timing on the context's stream (CUDA events) */
int rbf_timer_start(rbf_ctx* ctx);
int rbf_timer_stop_ms(rbf_ctx* ctx, double* ms);

/* ------------------------------------------------------------------ exact host-side scalars (no GPU) */
/* xxhash.xxh64_intdigest(data, seed) -- ivc:77,78,94; rbf:27,115,116,134 */
uint64_t rbf_xxh64(const void* data, uint64_t len, uint64_t seed);
/* xxh64 of str(item): straight route and the century/decade/finish route the kernels use */
uint64_t rbf_hash_decimal(uint32_t item, uint64_t seed);
uint64_t rbf_hash_decimal_century(uint32_t item, uint64_t seed);
/* RationalBloomFilter._get_hash_indices: (h1 + i*h2) % size over unbounded ints -- ivc:81 */
uint32_t rbf_probe_index(uint64_t h1, uint64_t h2, uint32_t i, uint32_t size);
/* RationalBloomFilter._determine_activation as a threshold -- ivc:94-97 */
uint64_t rbf_activation_threshold(double p_activation);
/* BloomFilterCompressor.compress gating + _calculate_optimal_params -- ivc:208-225, ivc:161-196.
 * Returns 1 when the Bloom coder applies, 0 for the raw-passthrough branches. */
int rbf_optimal_params(uint64_t n, uint64_t ones, double* p, double* k, uint64_t* l);

/* ------------------------------------------------------------------ device memory helpers */
int rbf_malloc(rbf_ctx* ctx, size_t bytes, void** dptr);
int rbf_free(rbf_ctx* ctx, void* dptr);
int rbf_malloc_host(rbf_ctx* ctx, size_t bytes, void** hptr);   /* pinned */
int rbf_free_host(rbf_ctx* ctx, void* hptr);
int rbf_memcpy_h2d(rbf_ctx* ctx, void* dptr, const void* hptr, size_t bytes);
int rbf_memcpy_d2h(rbf_ctx* ctx, void* hptr, const void* dptr, size_t bytes);
int rbf_memset(rbf_ctx* ctx, void* dptr, int value, size_t bytes);

/* ------------------------------------------------------------------ one filter (drop-in RationalBloomFilter)
 * ivc.RationalBloomFilter.__init__ / add_index / check_index / bit_array  (ivc:47-138)
 * rbf.RationalBloomFilter.add / contains (rbf:139-182), rbf.StandardBloomFilter (rbf:13-41, standard_k > 0) */
int rbf_filter_create(rbf_ctx* ctx, uint64_t size, double k_star, const rbf_seeds* seeds, rbf_filter** out);
void rbf_filter_destroy(rbf_filter* f);
int rbf_filter_add_indices(rbf_filter* f, const uint32_t* items, uint32_t count);
int rbf_filter_check_indices(rbf_filter* f, const uint32_t* items, uint32_t count, uint8_t* out01);
int rbf_filter_add_strings(rbf_filter* f, const uint8_t* blob, const uint64_t* offsets, uint32_t count, int standard_k);
int rbf_filter_check_strings(rbf_filter* f, const uint8_t* blob, const uint64_t* offsets, uint32_t count, int standard_k,
                             uint8_t* out01);
int rbf_filter_get_bits(rbf_filter* f, uint8_t* unpacked_out);        /* size bytes of 0/1 */
int rbf_filter_set_bits(rbf_filter* f, const uint8_t* unpacked_in);   /* `bloom_filter.bit_array = bitmap`, ivc:290 */

/* ------------------------------------------------------------------ mask coder (drop-in BloomFilterCompressor)
 * compress (ivc:198-266): mask_unpacked[n] (0/1) -> info, bitmap_unpacked_out[l], witness_unpacked_out[wlen].
 * Output buffers must hold n bytes each.  k_override > 0 replaces _calculate_optimal_params with
 * (k_override, l_override)  (BASELINE config 5). */
int rbf_compress_mask(rbf_ctx* ctx, const uint8_t* mask_unpacked, uint64_t n, const rbf_seeds* seeds, double k_override,
                      uint64_t l_override, rbf_mask_info* info, uint8_t* bitmap_unpacked_out,
                      uint8_t* witness_unpacked_out);
/* decompress (ivc:268-307): bitmap_unpacked[l], witness_unpacked[wlen], n, k -> mask_unpacked_out[n].
 * *consumed = number of positions that passed the Bloom test (the reference raises IndexError when > wlen). */
int rbf_decompress_mask(rbf_ctx* ctx, const uint8_t* bitmap_unpacked, uint64_t l, const uint8_t* witness_unpacked,
                        uint64_t wlen, uint64_t n, double k, const rbf_seeds* seeds, uint8_t* mask_unpacked_out,
                        uint64_t* consumed);

/* ------------------------------------------------------------------ frame stream (the batched hot path)
 * A stream owns a device-resident store of `max_frames` interleaved H x W x C frames (uint8 or
 * little-endian uint16 samples) and the per-pair outputs.  rbf_stream_encode runs, for every
 * (prev, curr) pair:   K1 VideoFrameCompressor._calculate_frame_diff mask part (ivc:788-808)
 *                      -> BloomFilterCompressor.compress (ivc:198-266) on the flattened mask (ivc:924-927). */
int rbf_stream_create(rbf_ctx* ctx, uint32_t height, uint32_t width, uint32_t channels, uint32_t sample_bytes,
                      uint32_t max_frames, uint32_t max_pairs, rbf_stream** out);
/* A stream of single images for BloomFilterCompressor.compress_image (bloom_compress.py:348-383): "pair" i of
 * rbf_stream_encode is image curr_idx[i] (prev_idx must equal curr_idx) and K1 is _binarize_image (bc:67-87) --
 * gray > threshold with gray = floor(mean of the C samples) for C > 1 (8-bit samples) and the sample itself for C = 1.
 * C in 1..4 with 1-byte samples, or C = 1 with 2-byte samples; the store holds max_images images (and pairs).
 * C = 0 (1-byte samples) makes a decode-only stream for rbf_stream_decode: it keeps the per-image bit-array, witness and
 * mask slots but no image store (upload, encode, apply_diff and median5 return RBF_ERR_STATE; download copies nothing).
 * Encode / fetch / fetch_batch / decode_verify / stage_ms / k1_only work as for frame streams; "mask_mode",
 * "gray_mode" and rbf_stream_encode_host are refused with RBF_ERR_STATE. */
int rbf_stream_create_images(rbf_ctx* ctx, uint32_t height, uint32_t width, uint32_t channels, uint32_t sample_bytes,
                             uint32_t max_images, rbf_stream** out);
void rbf_stream_destroy(rbf_stream* s);
/* per-stream options (no process-global state: two compressors in one process do not interfere):
 *   "k1_only"   1: rbf_stream_encode stops after K1 (mask + counts) -- VideoFrameCompressor._calculate_frame_diff (ivc:784-808);
 *               infos report wlen = 0 and rbf_stream_fetch refuses bitmap / witness pointers
 *   "mask_mode" 0: |dY| > threshold (ivc:808); 1: additionally any byte of the pixel differs (lossless GOP mode)
 *   "gray_mode" 1: 3-channel frames are BGR and the mask is taken on cv2.cvtColor(.., COLOR_BGR2GRAY) (ivc:792-795),
 *               OpenCV's fixed point (3735 B + 19235 G + 9798 R + 16384) >> 15 for 8- and 16-bit samples */
int rbf_stream_set_option(rbf_stream* s, const char* key, int64_t value);
int rbf_stream_upload(rbf_stream* s, uint32_t first_frame, uint32_t count, const void* host_frames);
int rbf_stream_frame_ptr(rbf_stream* s, uint32_t frame, void** dptr);
/* threshold: the Python float compared with `diff > threshold` (ivc:808).  k_override/l_override: NULL or [pairs]. */
int rbf_stream_encode(rbf_stream* s, const uint32_t* prev_idx, const uint32_t* curr_idx, uint32_t pairs, double threshold,
                      const rbf_seeds* seeds, const double* k_override, const uint64_t* l_override, rbf_mask_info* infos_out);
/* end-to-end variant: frames come from (pinned) host memory, packed outputs go back to host, copies inside */
int rbf_stream_encode_host(rbf_stream* s, const void* host_frames, uint32_t nframes, double threshold, const rbf_seeds* seeds,
                           rbf_mask_info* infos_out, uint8_t* bitmaps_packbits_out, uint64_t bitmap_slot_bytes,
                           uint8_t* witness_packbits_out, uint64_t witness_slot_bytes);
/* copy one pair's outputs to the host: bitmap/witness in packbits order (ceil(l/8), ceil(wlen/8) bytes),
 * mask as little-bit-order packed bytes (ceil(n/8)); any pointer may be NULL */
int rbf_stream_fetch(rbf_stream* s, uint32_t pair, uint8_t* bitmap_packbits, uint8_t* witness_packbits,
                     uint8_t* mask_packed_little);
/* the same for pairs [first, first+count) at once: output k of a kind lands at base + k*slot_bytes (slot_bytes bytes are copied
 * per pair, capped at the device slot); one synchronisation for the whole batch.  NULL pointers are skipped. */
int rbf_stream_fetch_batch(rbf_stream* s, uint32_t first, uint32_t count, uint8_t* bitmaps_packbits, uint64_t bitmap_slot_bytes,
                           uint8_t* witness_packbits, uint64_t witness_slot_bytes, uint8_t* masks_packed_little,
                           uint64_t mask_slot_bytes);
/* decode the pairs encoded by the last rbf_stream_encode from their own bitmap + witness (ivc:268-307) and
 * compare with the stored masks on the device: mismatches_out[pair] = differing mask words */
int rbf_stream_decode_verify(rbf_stream* s, uint32_t pairs, uint64_t* mismatches_out);
/* decode `count` caller-supplied payloads of the stream's n = H*W positions at once (BloomFilterCompressor.decompress,
 * bc:307-346 / ivc:268-307): payload i is (l[i], wlen[i], k[i]) with its bitmap at bitmaps_packbits + i*bitmap_slot_bytes and its
 * witness at witness_packbits + i*witness_slot_bytes (np.packbits order).  The decoded mask lands little-bit-order packed at
 * masks_packed_little + i*mask_slot_bytes; consumed_out[i] = positions that passed the Bloom test (the reference raises
 * IndexError when that exceeds wlen[i]).  Requires 1 <= l <= n and wlen <= n.  Overwrites the outputs of the last encode. */
int rbf_stream_decode(rbf_stream* s, uint32_t count, const uint64_t* l, const uint64_t* wlen, const double* k, const rbf_seeds* seeds,
                      const uint8_t* bitmaps_packbits, uint64_t bitmap_slot_bytes, const uint8_t* witness_packbits,
                      uint64_t witness_slot_bytes, uint8_t* masks_packed_little, uint64_t mask_slot_bytes, uint64_t* consumed_out);
int rbf_stream_bitmap_region(rbf_stream* s, void** dptr, uint64_t* stride_bytes);
/* device time (CUDA events) of the stages of the last rbf_stream_encode, ms.  K1 and K2 are pipelined over ranges of pairs
 * on two streams, so their spans overlap:
 * out = { K1 span, everything in front of K3 (K1 + host (k,l,T) round trips + K2 as overlapped), K2 span, K3 query,
 *         K3b witness, whole encode } */
int rbf_stream_stage_ms(rbf_stream* s, double out[6]);

/* ---- SURVEY 8(f) rows N1 / N2, device side
 * N1  changed-value gather of VideoFrameCompressor._calculate_frame_diff (ivc:810-842): for each pair of the last
 *     encode, the interleaved channel values (native sample type) of the CURRENT frame at the mask's set positions, in
 *     row-major order.  offsets_out[pairs+1] = byte offsets per pair; values_out == NULL only fills the offsets. */
int rbf_stream_gather_changed(rbf_stream* s, uint32_t pairs, uint8_t* values_out, uint64_t values_capacity,
                              uint64_t* offsets_out);
/* N2  VideoFrameCompressor._apply_frame_diff (ivc:849-909): store[out_frame] = store[base_frame] with the pixels selected
 *     by the mask (n bits, little bit order) replaced by `values` in rank order; when the value count does not match the
 *     mask the base frame is copied unchanged (ivc:882) and *applied_pixels = 0. */
int rbf_stream_apply_diff(rbf_stream* s, uint32_t base_frame, uint32_t out_frame, const uint8_t* mask_packed_little,
                          const uint8_t* values, uint64_t values_bytes, uint64_t* applied_pixels);
int rbf_stream_download(rbf_stream* s, uint32_t frame, void* host_out);
/* N3  the 5x5 median of cv2.medianBlur in VideoFrameCompressor._estimate_noise_level (ivc:738): replicated border, 13th
 *     smallest of 25, exact for uint8 / uint16.  The float32 std of (frame - median) stays in numpy (ivc:741-744). */
int rbf_median_blur5(rbf_ctx* ctx, const void* plane_in, uint32_t height, uint32_t width, uint32_t sample_bytes, void* plane_out);
int rbf_stream_median5(rbf_stream* s, uint32_t frame, void* plane_out);   /* channel 0 of a resident frame */

/* ------------------------------------------------------------------ multi-GPU (one process per GPU)
 * frames are sharded across ranks; the per-rank Bloom bit arrays are exchanged with ONE ncclAllGather
 * over NVLink.  NCCL is dlopen'ed (libnccl.so.2); the unique id travels over the caller's own channel. */
int rbf_nccl_unique_id(uint8_t id_out[128]);
int rbf_nccl_init(rbf_ctx* ctx, const uint8_t id[128], int rank, int nranks);
int rbf_nccl_allgather(rbf_ctx* ctx, const void* d_send, void* d_recv, uint64_t bytes_per_rank);
/* compact `pairs` bitmap slots (slot_bytes each) into d_send and all-gather them into d_recv.  Enqueued on the context's
 * communication stream so that the next rbf_stream_encode overlaps the exchange; d_recv is complete after rbf_sync,
 * rbf_timer_stop_ms or rbf_memcpy_d2h. */
int rbf_stream_allgather_bitmaps(rbf_stream* s, uint32_t pairs, uint64_t slot_bytes, void* d_send, void* d_recv);
int rbf_nccl_destroy(rbf_ctx* ctx);

/* The same exchange without NCCL on the data path: every rank maps the receive buffers and flag arrays of all ranks
 * (CUDA IPC; the 64-byte handles travel over the caller's channel, like the NCCL id) and
 * rbf_stream_allgather_bitmaps becomes ONE kernel that stores this rank's slots straight into every rank's
 * receive buffer over NVLink, followed by a system-scope release of a sequence number into each rank's flag array.
 *   receive buffer: 2 halves x nranks x pairs x slot_bytes (cudaMalloc via rbf_malloc); exchange number q lands in
 *   half q & 1 (rbf_peer_gather_half), so a rank may still read exchange q-1 while its peers deliver q;
 *   flag array: nranks uint32, zeroed by its owner before the handles are exchanged.
 * All ranks must use the same pairs and slot_bytes (a multiple of 16).  As with the NCCL form the call only enqueues work; the
 * other ranks' slots are complete after rbf_sync / rbf_timer_stop_ms / rbf_memcpy_d2h, which return an error if a peer
 * did not deliver within ~3 s instead of hanging.
 * CONTRACT: a rank must have finished reading exchange q-1 (copied it out, or consumed it on the context's stream) before it
 * calls exchange q+1 -- exchange q+1 reuses the half that held q-1; the library only guarantees that no rank overwrites a half
 * before every rank has signalled the exchange in between.  Validated at 2 and 8 GPUs (profiles/r02_n{2,8}_*_p2p.json). */
int rbf_peer_export(rbf_ctx* ctx, const void* d_ptr, uint8_t handle_out[64]);
int rbf_peer_open(rbf_ctx* ctx, const uint8_t handle[64], void** d_ptr_out);
int rbf_peer_close(rbf_ctx* ctx, void* d_ptr);
int rbf_peer_gather_init(rbf_ctx* ctx, int rank, int nranks, void* const* recv_ptrs, void* const* flag_ptrs);
int rbf_peer_gather_half(rbf_ctx* ctx, uint32_t* half_out);
int rbf_peer_gather_shutdown(rbf_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* RBF_B200_H */
