// rbf_api.cu -- the C ABI (include/rbf_b200.h) and the host side of the pipeline.
// Host code mirrors the reference's float expressions exactly (compile with -ffp-contract=off).
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/rbf_b200.h"
#include "rbf_kernels.cuh"

using namespace rbf;

// ------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

struct rbf_ctx {
    int device = -1;
    cudaStream_t st = nullptr;
    cudaStream_t st_copy = nullptr;   // H2D of frame chunks in rbf_stream_encode_host
    cudaStream_t st_comm = nullptr;   // slot packing + ncclAllGather of rbf_stream_allgather_bitmaps (overlaps the next encode)
    cudaEvent_t ev_enc = nullptr, ev_pack = nullptr, ev_comm = nullptr;
    bool pack_pending = false, comm_pending = false;
    // exchange over NVLink peer memory (rbf_peer_gather_init): receive buffers / flag arrays of all ranks as mapped here
    int peer_nranks = 0, peer_rank = 0;
    uint32_t* peer_recv[16] = {nullptr};
    uint32_t* peer_flags[16] = {nullptr};
    uint32_t peer_seq = 0;
    bool peer_wait_pending = false;
    uint32_t* peer_err = nullptr;     // mapped pinned word, set by k_peer_wait on time-out
    int host_chunk_frames = 32;
    cudaStream_t st_k1 = nullptr;     // pipelined encode: K1 of the later ranges + the witness memset run here, beside K2 on `st`
    cudaStream_t st_d2h = nullptr;    // rbf_stream_encode_host: result copies of chunk i overlap the kernels of chunk i+1
    cudaEvent_t ev_fork = nullptr, ev_wit = nullptr, ev_k1[8] = {nullptr}, ev_d2h = nullptr;
    int encode_ranges = 1;            // rbf_stream_encode: K1/K2 pipelined over this many ranges of pairs (1 = serial, the default: K1 (HBM)
                                      // and K2 (L2 atomics) slow each other down when they overlap -- profiles/r02_kbench_pipeline.jsonl)
    int k1_ctas_per_sm = 32;          // grid cap of K1 (pipelined encodes use pipe_k1_ctas_per_sm so that K2 finds room beside it)
    int pipe_k1_ctas_per_sm = 4;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaDeviceProp prop;
    int sm_count = 0;
    int k1_variant = 0;
    int insert_variant = 1; // 1: dense warp-compacted K2 (one RED.OR per probe; default); 0: per-lane K2
    int query_variant = 5;  // 0: per-lane; 1: staged A->B->C rings, L2 tail; 2: staged + 2-CTA DSMEM clusters; 3: dense A+B, ring before C;
                            // 4: decade tiles of round 1 (m <= 2^23, else 1); 5: decade tiles with carried stage-B batches (half tiles
                            // for 2^23 < m <= 2^24, ring kernel beyond); 6: half-decade tiles for every m <= 2^24
    int k1_only = 0;        // stop after K1 (mask + counts): VideoFrameCompressor._calculate_frame_diff
    int mask_mode = 0;      // 0: |dY| > thr (ivc:808); 1: additionally any byte of the pixel differs
    int query_smem_cap = 0;
    int query_warps = 0;    // warps per CTA of the tile query kernel (0 = its compiled maximum, 28)
    int kq_ranges = 1;      // > 1: K2 of range r+1 runs beside K3 of range r (see stream_encode_pipelined)
    char err[512];
    int64_t launches = 0, h2d = 0, d2h = 0;
    std::vector<void*> scratch;
    std::vector<size_t> scratch_sz;
    // NCCL (dlopen'ed)
    void* nccl_lib = nullptr;
    void* nccl_comm = nullptr;
    int nranks = 1, rank = 0;
};

static int set_err(rbf_ctx* c, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    snprintf(g_err, sizeof g_err, "%s", buf);
    if (c) snprintf(c->err, sizeof c->err, "%s", buf);
    return code;
}
#define CK(ctx, call)                                                                                           \
    do {                                                                                                        \
        cudaError_t e__ = (call);                                                                               \
        if (e__ != cudaSuccess)                                                                                 \
            return set_err(ctx, e__ == cudaErrorMemoryAllocation ? RBF_ERR_OOM : RBF_ERR_CUDA, "%s:%d %s: %s", \
                           __FILE__, __LINE__, #call, cudaGetErrorString(e__));                               \
    } while (0)
#define LAUNCH(ctx, call)  \
    do {                   \
        CK(ctx, call);     \
        (ctx)->launches++; \
    } while (0)

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

static int scratch_get(rbf_ctx* c, int slot, size_t bytes, void** out) {
    if ((int)c->scratch.size() <= slot) { c->scratch.resize(slot + 1, nullptr); c->scratch_sz.resize(slot + 1, 0); }
    if (c->scratch_sz[slot] < bytes) {
        if (c->scratch[slot]) CK(c, cudaFree(c->scratch[slot]));
        c->scratch[slot] = nullptr; c->scratch_sz[slot] = 0;
        size_t nb = align_up(bytes + (bytes >> 2), 256);
        CK(c, cudaMalloc(&c->scratch[slot], nb));
        c->scratch_sz[slot] = nb;
    }
    *out = c->scratch[slot];
    return RBF_OK;
}
// ------------------------------------------------------------------------------------------
// exact host-side scalars
// ------------------------------------------------------------------------------------------
// correctly rounded double of h / (2^64 - 1): Python int/int true division (ivc:95).  The exact
// quotient is h*2^-64*(1 + 2^-64 + ...), a hair above h*2^-64, so round h to 53 bits, ties up.
static double unit_div(uint64_t h) {
    if (h == 0) return 0.0;
    const int bl = 64 - __builtin_clzll(h);
    if (bl <= 53) return ldexp((double)h, -64);
    const int sh = bl - 53;
    uint64_t top = h >> sh;
    const uint64_t rem = h & ((1ULL << sh) - 1), half = 1ULL << (sh - 1);
    if (rem >= half) top += 1;
    return ldexp((double)top, sh - 64);
}

extern "C" uint64_t rbf_activation_threshold(double p_act) {
    if (!(p_act > 0.0)) return 0;                       // also NaN
    if (unit_div(UINT64_MAX) < p_act) return UINT64_MAX;
    uint64_t lo = 0, hi = UINT64_MAX;                   // smallest h with unit_div(h) >= p_act
    while (lo < hi) {
        const uint64_t mid = lo + (hi - lo) / 2;
        if (unit_div(mid) < p_act) lo = mid + 1; else hi = mid;
    }
    return lo;
}

static const double kPStar = 0.32453;                  // ivc:150

// _calculate_optimal_params (ivc:161-196); returns l (0 => the (0, 0) result)
static uint64_t optimal_kl(uint64_t n, double p, double* k_out) {
    *k_out = 0.0;
    if (p <= 0.0001) return 0;
    if (p >= kPStar) return 0;
    const double q = 1 - p;
    const double L = log(2.0);
    const double k = log2(q * pow(L, 2.0) / p);         // ivc:185
    if (isnan(k) || k <= 0) return 0;
    const double gamma = 1 / L;
    const double lf = p * (double)n * k * gamma;        // ivc:193, evaluated left to right
    const uint64_t l = (uint64_t)lf;
    *k_out = k > 0.1 ? k : 0.1;
    return l > 1 ? l : 1;
}

extern "C" int rbf_optimal_params(uint64_t n, uint64_t ones, double* p_out, double* k_out, uint64_t* l_out) {
    const double p = (double)ones / (double)n;          // ivc:212
    double k = 0.0;
    uint64_t l = 0;
    int coded = 0;
    if (!(p >= kPStar)) {                               // ivc:215
        l = optimal_kl(n, p, &k);
        if (!(l == 0 || l >= n)) coded = 1;             // ivc:223
    }
    if (!coded) { k = 0.0; l = 0; }
    if (p_out) *p_out = p;
    if (k_out) *k_out = k;
    if (l_out) *l_out = l;
    return coded;
}

extern "C" uint64_t rbf_xxh64(const void* data, uint64_t len, uint64_t seed) {
    return xxh64_bytes((const uint8_t*)data, (uint32_t)len, seed);
}
extern "C" uint64_t rbf_hash_decimal(uint32_t item, uint64_t seed) { return xxh64_decimal(item, seed); }
extern "C" uint64_t rbf_hash_decimal_century(uint32_t item, uint64_t seed) {
    const Century c = make_century(item / 100u);
    return finish(c.kind, decade_state(c, century_state(c, seed), seed, (item / 10u) % 10u), seed, item % 10u);
}
extern "C" uint32_t rbf_probe_index(uint64_t h1, uint64_t h2, uint32_t i, uint32_t size) {
    if (size == 0) return 0;
    return probe_index(h1, h2, i, make_fastmod(size));
}
extern "C" int rbf_abi_version(void) { return RBF_ABI_VERSION; }
extern "C" const char* rbf_last_global_error(void) { return g_err; }

// fill the filter part of a job from (size, k*)  (ivc:47-63)
static void job_set_filter(FrameJob& J, uint64_t size, double k_star, const rbf_seeds& sd) {
    J.l = (uint32_t)size;
    const double fl = floor(k_star);
    J.floor_k = (uint32_t)(fl < 0 ? 0 : fl);
    const double p_act = k_star - fl;                   // ivc:58
    J.has_act = p_act > 0.0 ? 1u : 0u;
    J.act_T = rbf_activation_threshold(p_act);
    J.seed1 = sd.h1; J.seed2 = sd.h2; J.seedA = sd.act;
    J.fm = make_fastmod((uint32_t)size);
    J.neg_m = 0u - (uint32_t)size;
}

// ------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------
extern "C" int rbf_ctx_create(int device, rbf_ctx** out) {
    if (!out) return set_err(nullptr, RBF_ERR_INVALID, "rbf_ctx_create: out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return set_err(nullptr, RBF_ERR_NO_DEVICE, "no CUDA device available (%s); this library has no CPU fallback",
                       e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return set_err(nullptr, RBF_ERR_INVALID, "device %d out of range [0,%d)", device, ndev);
    rbf_ctx* c = new rbf_ctx();
    c->err[0] = 0;
    c->device = device;
    if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaGetDeviceProperties(&c->prop, device)) != cudaSuccess) {
        delete c;
        return set_err(nullptr, RBF_ERR_CUDA, "cudaSetDevice/GetDeviceProperties: %s", cudaGetErrorString(e));
    }
    if (c->prop.major < 10) {
        int maj = c->prop.major, mn = c->prop.minor;
        delete c;
        return set_err(nullptr, RBF_ERR_NO_DEVICE, "device is sm_%d%d; this library is built for sm_100a only", maj, mn);
    }
    c->sm_count = c->prop.multiProcessorCount;
    c->query_smem_cap = query_max_smem_bytes();
    if ((e = cudaStreamCreateWithFlags(&c->st, cudaStreamNonBlocking)) != cudaSuccess ||
        (e = cudaEventCreate(&c->ev0)) != cudaSuccess || (e = cudaEventCreate(&c->ev1)) != cudaSuccess) {
        delete c;
        return set_err(nullptr, RBF_ERR_CUDA, "stream/event create: %s", cudaGetErrorString(e));
    }
    *out = c;
    return RBF_OK;
}

extern "C" void rbf_ctx_destroy(rbf_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    rbf_nccl_destroy(c);
    for (void* p : c->scratch) if (p) cudaFree(p);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->st) cudaStreamDestroy(c->st);
    if (c->st_k1) cudaStreamDestroy(c->st_k1);
    if (c->st_d2h) cudaStreamDestroy(c->st_d2h);
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_wit) cudaEventDestroy(c->ev_wit);
    if (c->ev_d2h) cudaEventDestroy(c->ev_d2h);
    for (auto& e : c->ev_k1) if (e) cudaEventDestroy(e);
    if (c->st_copy) cudaStreamDestroy(c->st_copy);
    if (c->st_comm) { cudaStreamSynchronize(c->st_comm); cudaStreamDestroy(c->st_comm); }
    if (c->ev_enc) cudaEventDestroy(c->ev_enc);
    if (c->ev_pack) cudaEventDestroy(c->ev_pack);
    if (c->ev_comm) cudaEventDestroy(c->ev_comm);
    if (c->peer_err) cudaFreeHost(c->peer_err);
    delete c;
}
extern "C" const char* rbf_last_error(const rbf_ctx* c) { return c ? c->err : g_err; }

extern "C" int rbf_device_info(rbf_ctx* c, char* name, int name_len, int* sm_count, int* cc_major, int* cc_minor,
                               uint64_t* total_mem) {
    if (!c) return set_err(nullptr, RBF_ERR_INVALID, "ctx is NULL");
    if (name && name_len > 0) snprintf(name, name_len, "%s", c->prop.name);
    if (sm_count) *sm_count = c->sm_count;
    if (cc_major) *cc_major = c->prop.major;
    if (cc_minor) *cc_minor = c->prop.minor;
    if (total_mem) *total_mem = c->prop.totalGlobalMem;
    return RBF_OK;
}
extern "C" int rbf_set_option(rbf_ctx* c, const char* key, int64_t v) {
    if (!c || !key) return set_err(c, RBF_ERR_INVALID, "rbf_set_option: NULL");
    if (!strcmp(key, "k1_variant")) { c->k1_variant = (int)v; return RBF_OK; }
    if (!strcmp(key, "query_variant")) { c->query_variant = (int)(v < 0 ? 0 : (v > 6 ? 6 : v)); return RBF_OK; }
    if (!strcmp(key, "insert_variant")) { c->insert_variant = v ? 1 : 0; return RBF_OK; }
    if (!strcmp(key, "host_chunk_frames")) { c->host_chunk_frames = (int)v; return RBF_OK; }
    if (!strcmp(key, "k1_only")) { c->k1_only = v ? 1 : 0; return RBF_OK; }        // default of streams created afterwards
    if (!strcmp(key, "mask_mode")) { c->mask_mode = v ? 1 : 0; return RBF_OK; }    // (per-stream: rbf_stream_set_option)
    if (!strcmp(key, "query_warps")) { c->query_warps = (int)v; return RBF_OK; }
    if (!strcmp(key, "kq_ranges")) { c->kq_ranges = (int)(v < 1 ? 1 : (v > 8 ? 8 : v)); return RBF_OK; }
    if (!strcmp(key, "encode_ranges")) { c->encode_ranges = (int)(v < 1 ? 1 : (v > 8 ? 8 : v)); return RBF_OK; }
    if (!strcmp(key, "k1_ctas_per_sm")) { c->k1_ctas_per_sm = (int)(v < 1 ? 1 : (v > 64 ? 64 : v)); return RBF_OK; }
    if (!strcmp(key, "pipe_k1_ctas_per_sm")) { c->pipe_k1_ctas_per_sm = (int)(v < 1 ? 1 : (v > 64 ? 64 : v)); return RBF_OK; }
    if (!strcmp(key, "query_smem_bytes")) {
        c->query_smem_cap = (int)((v <= 0 || v > query_max_smem_bytes()) ? query_max_smem_bytes() : v);
        return RBF_OK;
    }
    return set_err(c, RBF_ERR_INVALID, "unknown option %s", key);
}
extern "C" int64_t rbf_get_counter(rbf_ctx* c, const char* key) {
    if (!c || !key) return -1;
    if (!strcmp(key, "kernel_launches")) return c->launches;
    if (!strcmp(key, "h2d_bytes")) return c->h2d;
    if (!strcmp(key, "d2h_bytes")) return c->d2h;
    return -1;
}
extern "C" int rbf_reset_counters(rbf_ctx* c) { if (!c) return RBF_ERR_INVALID; c->launches = c->h2d = c->d2h = 0; return RBF_OK; }
// before the bit arrays are overwritten: the slot packing of a pending all-gather must have read them
static int wait_pack(rbf_ctx* c) {
    if (c->pack_pending) { CK(c, cudaStreamWaitEvent(c->st, c->ev_pack, 0)); c->pack_pending = false; }
    return RBF_OK;
}
// make the context's stream wait for an all-gather still running on the communication stream
static const long long kPeerTimeoutCycles = 6000000000LL;    // ~3 s of SM clocks: a lost peer must not hang the GPU
static int join_comm(rbf_ctx* c) {
    if (c->comm_pending) { CK(c, cudaStreamWaitEvent(c->st, c->ev_comm, 0)); c->comm_pending = false; c->pack_pending = false; }
    if (c->peer_wait_pending) {                                // the other ranks' slots of the last exchange
        LAUNCH(c, launch_peer_wait(c->peer_flags[c->peer_rank], c->peer_nranks, c->peer_seq, kPeerTimeoutCycles, c->peer_err, c->st));
        c->peer_wait_pending = false;
    }
    return RBF_OK;
}
static int check_peer_err(rbf_ctx* c) {                        // call after the stream has been synchronised
    if (c->peer_err && *(volatile uint32_t*)c->peer_err) {
        *(volatile uint32_t*)c->peer_err = 0;
        return set_err(c, RBF_ERR_NCCL, "peer exchange timed out: a rank did not deliver its slots");
    }
    return RBF_OK;
}
extern "C" int rbf_sync(rbf_ctx* c) {
    if (!c) return RBF_ERR_INVALID;
    if (int r = join_comm(c)) return r;
    CK(c, cudaStreamSynchronize(c->st));
    return check_peer_err(c);
}
extern "C" int rbf_timer_start(rbf_ctx* c) { if (!c) return RBF_ERR_INVALID; CK(c, cudaEventRecord(c->ev0, c->st)); return RBF_OK; }
extern "C" int rbf_timer_stop_ms(rbf_ctx* c, double* ms) {
    if (!c || !ms) return RBF_ERR_INVALID;
    if (int r = join_comm(c)) return r;
    CK(c, cudaEventRecord(c->ev1, c->st));
    CK(c, cudaEventSynchronize(c->ev1));
    float f = 0;
    CK(c, cudaEventElapsedTime(&f, c->ev0, c->ev1));
    *ms = f;
    return check_peer_err(c);
}

// memory
extern "C" int rbf_malloc(rbf_ctx* c, size_t bytes, void** d) { if (!c || !d) return RBF_ERR_INVALID; CK(c, cudaSetDevice(c->device)); CK(c, cudaMalloc(d, bytes ? bytes : 1)); return RBF_OK; }
extern "C" int rbf_free(rbf_ctx* c, void* d) { if (!c) return RBF_ERR_INVALID; if (d) CK(c, cudaFree(d)); return RBF_OK; }
extern "C" int rbf_malloc_host(rbf_ctx* c, size_t bytes, void** h) { if (!c || !h) return RBF_ERR_INVALID; CK(c, cudaMallocHost(h, bytes ? bytes : 1)); return RBF_OK; }
extern "C" int rbf_free_host(rbf_ctx* c, void* h) { if (!c) return RBF_ERR_INVALID; if (h) CK(c, cudaFreeHost(h)); return RBF_OK; }
extern "C" int rbf_memcpy_h2d(rbf_ctx* c, void* d, const void* h, size_t n) {
    if (!c) return RBF_ERR_INVALID;
    CK(c, cudaMemcpyAsync(d, h, n, cudaMemcpyHostToDevice, c->st)); CK(c, cudaStreamSynchronize(c->st)); c->h2d += n; return RBF_OK;
}
extern "C" int rbf_memcpy_d2h(rbf_ctx* c, void* h, const void* d, size_t n) {
    if (!c) return RBF_ERR_INVALID;
    if (int r = join_comm(c)) return r;
    CK(c, cudaMemcpyAsync(h, d, n, cudaMemcpyDeviceToHost, c->st)); CK(c, cudaStreamSynchronize(c->st)); c->d2h += n;
    return check_peer_err(c);
}
extern "C" int rbf_memset(rbf_ctx* c, void* d, int v, size_t n) { if (!c) return RBF_ERR_INVALID; CK(c, cudaMemsetAsync(d, v, n, c->st)); return RBF_OK; }

// ------------------------------------------------------------------------------------------
// one filter
// ------------------------------------------------------------------------------------------
struct rbf_filter {
    rbf_ctx* c;
    uint64_t size;
    FrameJob job;          // host copy
    FrameJob* d_job;
    uint32_t* d_bits;      // LSB-first
    size_t words;
};

extern "C" int rbf_filter_create(rbf_ctx* c, uint64_t size, double k_star, const rbf_seeds* sd, rbf_filter** out) {
    if (!c || !sd || !out) return set_err(c, RBF_ERR_INVALID, "rbf_filter_create: NULL argument");
    if (size == 0 || size > 0xffffffffULL) return set_err(c, RBF_ERR_INVALID, "filter size %llu outside [1, 2^32)", (unsigned long long)size);
    if (!(k_star >= 0.0) || k_star > 1e6) return set_err(c, RBF_ERR_INVALID, "k_star %g not supported", k_star);
    CK(c, cudaSetDevice(c->device));
    rbf_filter* f = new rbf_filter();
    f->c = c; f->size = size; f->words = align_up((size + 31) / 32 + 8, 32);
    memset(&f->job, 0, sizeof f->job);
    job_set_filter(f->job, size, k_star, *sd);
    f->job.n = 0;
    cudaError_t e = cudaMalloc(&f->d_bits, f->words * 4);
    if (e == cudaSuccess) e = cudaMalloc(&f->d_job, sizeof(FrameJob));
    if (e != cudaSuccess) { delete f; return set_err(c, RBF_ERR_OOM, "rbf_filter_create: %s", cudaGetErrorString(e)); }
    f->job.bits = f->d_bits;
    CK(c, cudaMemsetAsync(f->d_bits, 0, f->words * 4, c->st));
    CK(c, cudaMemcpyAsync(f->d_job, &f->job, sizeof(FrameJob), cudaMemcpyHostToDevice, c->st));
    CK(c, cudaStreamSynchronize(c->st));
    *out = f;
    return RBF_OK;
}
extern "C" void rbf_filter_destroy(rbf_filter* f) {
    if (!f) return;
    cudaFree(f->d_bits); cudaFree(f->d_job);
    delete f;
}
static int filter_items_u32(rbf_filter* f, const uint32_t* items, uint32_t count, uint8_t* out, int insert) {
    rbf_ctx* c = f->c;
    if (count == 0) return RBF_OK;
    void *d_items, *d_res;
    int rc;
    if ((rc = scratch_get(c, 0, (size_t)count * 4, &d_items))) return rc;
    if ((rc = scratch_get(c, 1, (size_t)count, &d_res))) return rc;
    CK(c, cudaMemcpyAsync(d_items, items, (size_t)count * 4, cudaMemcpyHostToDevice, c->st)); c->h2d += (size_t)count * 4;
    LAUNCH(c, launch_items_u32(f->d_job, (const uint32_t*)d_items, count, (uint8_t*)d_res, insert, c->st));
    if (!insert) { CK(c, cudaMemcpyAsync(out, d_res, count, cudaMemcpyDeviceToHost, c->st)); c->d2h += count; }
    CK(c, cudaStreamSynchronize(c->st));
    return RBF_OK;
}
extern "C" int rbf_filter_add_indices(rbf_filter* f, const uint32_t* items, uint32_t count) {
    if (!f || (!items && count)) return set_err(f ? f->c : nullptr, RBF_ERR_INVALID, "rbf_filter_add_indices: NULL");
    return filter_items_u32(f, items, count, nullptr, 1);
}
extern "C" int rbf_filter_check_indices(rbf_filter* f, const uint32_t* items, uint32_t count, uint8_t* out) {
    if (!f || ((!items || !out) && count)) return set_err(f ? f->c : nullptr, RBF_ERR_INVALID, "rbf_filter_check_indices: NULL");
    return filter_items_u32(f, items, count, out, 0);
}
static int filter_items_str(rbf_filter* f, const uint8_t* blob, const uint64_t* offs, uint32_t count, int standard_k,
                            uint8_t* out, int insert) {
    rbf_ctx* c = f->c;
    if (count == 0) return RBF_OK;
    const size_t blob_bytes = (size_t)offs[count];
    void *d_blob, *d_offs, *d_res;
    int rc;
    if ((rc = scratch_get(c, 0, blob_bytes + 16, &d_blob))) return rc;
    if ((rc = scratch_get(c, 1, (size_t)count, &d_res))) return rc;
    if ((rc = scratch_get(c, 2, ((size_t)count + 1) * 8, &d_offs))) return rc;
    if (blob_bytes) { CK(c, cudaMemcpyAsync(d_blob, blob, blob_bytes, cudaMemcpyHostToDevice, c->st)); }
    CK(c, cudaMemcpyAsync(d_offs, offs, ((size_t)count + 1) * 8, cudaMemcpyHostToDevice, c->st));
    c->h2d += blob_bytes + ((size_t)count + 1) * 8;
    LAUNCH(c, launch_items_str(f->d_job, (const uint8_t*)d_blob, (const uint64_t*)d_offs, count, (uint8_t*)d_res, insert,
                               standard_k, c->st));
    if (!insert) { CK(c, cudaMemcpyAsync(out, d_res, count, cudaMemcpyDeviceToHost, c->st)); c->d2h += count; }
    CK(c, cudaStreamSynchronize(c->st));
    return RBF_OK;
}
extern "C" int rbf_filter_add_strings(rbf_filter* f, const uint8_t* blob, const uint64_t* offs, uint32_t count, int standard_k) {
    if (!f || (!offs && count)) return set_err(f ? f->c : nullptr, RBF_ERR_INVALID, "rbf_filter_add_strings: NULL");
    return filter_items_str(f, blob, offs, count, standard_k, nullptr, 1);
}
extern "C" int rbf_filter_check_strings(rbf_filter* f, const uint8_t* blob, const uint64_t* offs, uint32_t count,
                                        int standard_k, uint8_t* out) {
    if (!f || ((!offs || !out) && count)) return set_err(f ? f->c : nullptr, RBF_ERR_INVALID, "rbf_filter_check_strings: NULL");
    return filter_items_str(f, blob, offs, count, standard_k, out, 0);
}
extern "C" int rbf_filter_get_bits(rbf_filter* f, uint8_t* out) {
    if (!f || !out) return set_err(f ? f->c : nullptr, RBF_ERR_INVALID, "rbf_filter_get_bits: NULL");
    rbf_ctx* c = f->c;
    void* d_bytes; int rc;
    if ((rc = scratch_get(c, 0, f->size, &d_bytes))) return rc;
    LAUNCH(c, launch_unpack_bits(f->d_bits, (uint8_t*)d_bytes, f->size, c->st));
    CK(c, cudaMemcpyAsync(out, d_bytes, f->size, cudaMemcpyDeviceToHost, c->st)); c->d2h += f->size;
    CK(c, cudaStreamSynchronize(c->st));
    return RBF_OK;
}
extern "C" int rbf_filter_set_bits(rbf_filter* f, const uint8_t* in) {
    if (!f || !in) return set_err(f ? f->c : nullptr, RBF_ERR_INVALID, "rbf_filter_set_bits: NULL");
    rbf_ctx* c = f->c;
    void* d_bytes; int rc;
    if ((rc = scratch_get(c, 0, f->size, &d_bytes))) return rc;
    CK(c, cudaMemcpyAsync(d_bytes, in, f->size, cudaMemcpyHostToDevice, c->st)); c->h2d += f->size;
    CK(c, cudaMemsetAsync(f->d_bits, 0, f->words * 4, c->st));
    LAUNCH(c, launch_pack_bytes((const uint8_t*)d_bytes, f->d_bits, f->size, c->st));
    CK(c, cudaStreamSynchronize(c->st));
    return RBF_OK;
}

// ------------------------------------------------------------------------------------------
// mask coder (host buffers)
// ------------------------------------------------------------------------------------------

static size_t bit_words_padded(uint64_t nbits) { return align_up((nbits + 31) / 32 + 8, 32); }   // >= 32 B of padding, 128 B multiple
static size_t pass_words(uint64_t n) { return align_up(((n + 99) / 100) * 4, 32); }

extern "C" int rbf_compress_mask(rbf_ctx* c, const uint8_t* mask, uint64_t n, const rbf_seeds* sd, double k_override,
                                 uint64_t l_override, rbf_mask_info* info, uint8_t* bitmap_out, uint8_t* witness_out) {
    if (!c || !mask || !sd || !info) return set_err(c, RBF_ERR_INVALID, "rbf_compress_mask: NULL argument");
    if (n == 0 || n > 0xffffff00ULL) return set_err(c, RBF_ERR_INVALID, "n = %llu outside [1, 2^32-256]", (unsigned long long)n);
    CK(c, cudaSetDevice(c->device));
    memset(info, 0, sizeof *info);
    info->n = n;
    const size_t mw = bit_words_padded(n), pw = pass_words(n);
    void *d_bytes, *d_mask, *d_bits, *d_pass, *d_wit, *d_small;
    int rc;
    if ((rc = scratch_get(c, 0, n, &d_bytes)) || (rc = scratch_get(c, 3, mw * 4, &d_mask)) ||
        (rc = scratch_get(c, 4, mw * 4, &d_bits)) || (rc = scratch_get(c, 5, pw * 4, &d_pass)) ||
        (rc = scratch_get(c, 6, mw * 4, &d_wit)) || (rc = scratch_get(c, 7, 4096, &d_small)))
        return rc;
    uint32_t* d_cnt = (uint32_t*)d_small;                         // [0] ones, [1] wlen
    uint32_t* d_prefix = d_cnt + 4;                               // [2] cent_prefix
    FrameJob* d_job = (FrameJob*)((uint8_t*)d_small + 256);
    CK(c, cudaMemcpyAsync(d_bytes, mask, n, cudaMemcpyHostToDevice, c->st)); c->h2d += n;
    CK(c, cudaMemsetAsync(d_mask, 0, mw * 4, c->st));
    CK(c, cudaMemsetAsync(d_cnt, 0, 16, c->st));
    LAUNCH(c, launch_pack_bytes((const uint8_t*)d_bytes, (uint32_t*)d_mask, n, c->st));
    LAUNCH(c, launch_popcount((const uint32_t*)d_mask, (n + 31) / 32, d_cnt, c->st));
    uint32_t h_cnt[4] = {0, 0, 0, 0};
    CK(c, cudaMemcpyAsync(h_cnt, d_cnt, 16, cudaMemcpyDeviceToHost, c->st)); c->d2h += 16;
    CK(c, cudaStreamSynchronize(c->st));
    info->ones = h_cnt[0];
    double p, k; uint64_t l;
    int coded = rbf_optimal_params(n, info->ones, &p, &k, &l);
    info->p = p;
    if (k_override > 0.0 && !(p >= kPStar)) { k = k_override; l = l_override; coded = !(l == 0 || l >= n); }
    if (!coded) { info->raw = 1; return RBF_OK; }
    info->k = k; info->l = l;
    FrameJob J; memset(&J, 0, sizeof J);
    J.n = (uint32_t)n;
    job_set_filter(J, l, k, *sd);
    J.mask = (const uint32_t*)d_mask; J.bits = (uint32_t*)d_bits; J.pass = (uint32_t*)d_pass; J.witness = (uint32_t*)d_wit;
    info->floor_k = J.floor_k; info->act_T = J.act_T;
    const uint32_t ncent = (uint32_t)((n + 99) / 100);
    uint32_t h_prefix[2] = {0, ncent};
    CK(c, cudaMemcpyAsync(d_job, &J, sizeof J, cudaMemcpyHostToDevice, c->st));
    CK(c, cudaMemcpyAsync(d_prefix, h_prefix, 8, cudaMemcpyHostToDevice, c->st));
    CK(c, cudaMemsetAsync(d_bits, 0, bit_words_padded(l) * 4, c->st));
    CK(c, cudaMemsetAsync(d_wit, 0, mw * 4, c->st));
    LAUNCH(c, launch_insert(d_job, 1, ncent, c->insert_variant, c->sm_count, c->st));
    LAUNCH(c, launch_query(d_job, d_prefix, 1, ncent, (uint32_t)l, c->query_variant, c->sm_count, c->query_smem_cap, c->query_warps, c->st));
    LAUNCH(c, launch_witness(d_job, 1, ncent, c->sm_count, (uint32_t*)((uint8_t*)d_small + 1024), d_cnt + 1, c->st)); c->launches += 2;
    CK(c, cudaMemcpyAsync(h_cnt, d_cnt, 16, cudaMemcpyDeviceToHost, c->st)); c->d2h += 16;
    CK(c, cudaStreamSynchronize(c->st));
    info->wlen = h_cnt[1];
    // after K3b both streams are in packbits order; hand them back unpacked (ivc:266 returns bit_array, witness)
    if (bitmap_out) {
        LAUNCH(c, launch_unpack_bits_msb((const uint32_t*)d_bits, (uint8_t*)d_bytes, l, c->st));
        CK(c, cudaMemcpyAsync(bitmap_out, d_bytes, l, cudaMemcpyDeviceToHost, c->st)); c->d2h += l;
        CK(c, cudaStreamSynchronize(c->st));
    }
    if (witness_out && info->wlen) {
        LAUNCH(c, launch_unpack_bits_msb((const uint32_t*)d_wit, (uint8_t*)d_bytes, info->wlen, c->st));
        CK(c, cudaMemcpyAsync(witness_out, d_bytes, info->wlen, cudaMemcpyDeviceToHost, c->st)); c->d2h += info->wlen;
        CK(c, cudaStreamSynchronize(c->st));
    }
    return RBF_OK;
}

extern "C" int rbf_decompress_mask(rbf_ctx* c, const uint8_t* bitmap, uint64_t l, const uint8_t* witness, uint64_t wlen,
                                   uint64_t n, double k, const rbf_seeds* sd, uint8_t* out, uint64_t* consumed) {
    if (!c || !bitmap || !sd || !out || (!witness && wlen)) return set_err(c, RBF_ERR_INVALID, "rbf_decompress_mask: NULL argument");
    if (n == 0 || n > 0xffffff00ULL || l == 0 || l > 0xffffffffULL) return set_err(c, RBF_ERR_INVALID, "bad n/l");
    if (!(k >= 0.0)) return set_err(c, RBF_ERR_INVALID, "bad k");
    CK(c, cudaSetDevice(c->device));
    const size_t mw = bit_words_padded(n), lw = bit_words_padded(l), ww = bit_words_padded(wlen), pw = pass_words(n);
    const size_t big = n > l ? (n > wlen ? n : wlen) : (l > wlen ? l : wlen);
    void *d_bytes, *d_out, *d_bits, *d_pass, *d_wit, *d_small;
    int rc;
    if ((rc = scratch_get(c, 0, big, &d_bytes)) || (rc = scratch_get(c, 3, mw * 4, &d_out)) ||
        (rc = scratch_get(c, 4, lw * 4, &d_bits)) || (rc = scratch_get(c, 5, pw * 4, &d_pass)) ||
        (rc = scratch_get(c, 6, ww * 4, &d_wit)) || (rc = scratch_get(c, 7, 4096, &d_small)))
        return rc;
    uint32_t* d_cnt = (uint32_t*)d_small;
    uint32_t* d_prefix = d_cnt + 4;
    FrameJob* d_job = (FrameJob*)((uint8_t*)d_small + 256);
    CK(c, cudaMemsetAsync(d_bits, 0, lw * 4, c->st));
    CK(c, cudaMemsetAsync(d_wit, 0, ww * 4, c->st));
    CK(c, cudaMemsetAsync(d_out, 0, mw * 4, c->st));
    CK(c, cudaMemcpyAsync(d_bytes, bitmap, l, cudaMemcpyHostToDevice, c->st)); c->h2d += l;
    LAUNCH(c, launch_pack_bytes((const uint8_t*)d_bytes, (uint32_t*)d_bits, l, c->st));
    if (wlen) {
        CK(c, cudaMemcpyAsync(d_bytes, witness, wlen, cudaMemcpyHostToDevice, c->st)); c->h2d += wlen;
        // witness values are used as bits: any non-zero byte other than 1 is not representable; the reference
        // stores whatever the list holds (ivc:303); np.unpackbits output is 0/1 (ivc:1001-1002)
        LAUNCH(c, launch_pack_bytes((const uint8_t*)d_bytes, (uint32_t*)d_wit, wlen, c->st));
    }
    FrameJob J; memset(&J, 0, sizeof J);
    J.n = (uint32_t)n;
    job_set_filter(J, l, k, *sd);
    J.bits = (uint32_t*)d_bits; J.pass = (uint32_t*)d_pass; J.witness = (uint32_t*)d_wit; J.out_mask = (uint32_t*)d_out;
    J.wlen_in = (uint32_t)wlen;
    const uint32_t ncent = (uint32_t)((n + 99) / 100);
    uint32_t h_prefix[2] = {0, ncent};
    CK(c, cudaMemcpyAsync(d_job, &J, sizeof J, cudaMemcpyHostToDevice, c->st));
    CK(c, cudaMemcpyAsync(d_prefix, h_prefix, 8, cudaMemcpyHostToDevice, c->st));
    LAUNCH(c, launch_query(d_job, d_prefix, 1, ncent, (uint32_t)l, c->query_variant, c->sm_count, c->query_smem_cap, c->query_warps, c->st));
    LAUNCH(c, launch_expand(d_job, 1, ncent, c->sm_count, (uint32_t*)((uint8_t*)d_small + 1024), d_cnt, c->st)); c->launches += 1;
    LAUNCH(c, launch_unpack_bits((const uint32_t*)d_out, (uint8_t*)d_bytes, n, c->st));
    uint32_t h_cnt = 0;
    CK(c, cudaMemcpyAsync(out, d_bytes, n, cudaMemcpyDeviceToHost, c->st)); c->d2h += n;
    CK(c, cudaMemcpyAsync(&h_cnt, d_cnt, 4, cudaMemcpyDeviceToHost, c->st));
    CK(c, cudaStreamSynchronize(c->st));
    if (consumed) *consumed = h_cnt;
    return RBF_OK;
}

// ------------------------------------------------------------------------------------------
// frame stream
// ------------------------------------------------------------------------------------------
struct rbf_stream {
    rbf_ctx* c;
    uint32_t H, W, C, S, max_frames, max_pairs;
    uint64_t npix, frame_bytes, frame_stride;
    uint8_t* d_frames = nullptr;
    size_t mask_stride_w = 0, pass_stride_w = 0;     // words per pair
    uint32_t *d_mask = nullptr, *d_bits = nullptr, *d_wit = nullptr, *d_pass = nullptr, *d_dec = nullptr;
    FrameJob* d_jobs = nullptr;
    PairJob* d_pairs = nullptr;
    uint32_t *d_prefix = nullptr, *d_ones = nullptr, *d_resid = nullptr, *d_wlen = nullptr, *d_chunkcnt = nullptr;
    // pinned host mirrors
    FrameJob* h_jobs = nullptr;
    PairJob* h_pairs = nullptr;
    uint32_t *h_prefix = nullptr, *h_ones = nullptr, *h_resid = nullptr, *h_wlen = nullptr;
    uint32_t last_pairs = 0, last_max_l = 0;
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    bool staged = false;
    // per-stream options (rbf_stream_set_option); defaults come from the context at creation
    int k1_only = 0;        // stop after K1 (mask + counts): VideoFrameCompressor._calculate_frame_diff
    int mask_mode = 0;      // 0: |dY| > thr (ivc:808); 1: additionally any byte of the pixel differs
    int gray_mode = 0;      // 1: the mask is taken on cv2.COLOR_BGR2GRAY of the pixel (ivc:792-795) instead of on sample 0
    bool images = false;    // rbf_stream_create_images: pair i is image curr_idx[i], K1 is k_binarize (bloom_compress.py:67-87)
    bool last_k1_only = false;
    size_t bits_hwm = 0, wit_hwm = 0;   // bytes per slot that may hold set bits (see stream_clear_outputs)
    bool wit_dirty_full = false;
    std::vector<cudaEvent_t> ev_copy;
    std::vector<rbf_mask_info> last_infos;
};

extern "C" void rbf_stream_destroy(rbf_stream* s) {
    if (!s) return;
    cudaSetDevice(s->c->device);
    cudaFree(s->d_frames); cudaFree(s->d_mask); cudaFree(s->d_bits); cudaFree(s->d_wit); cudaFree(s->d_pass); cudaFree(s->d_dec);
    cudaFree(s->d_jobs); cudaFree(s->d_pairs); cudaFree(s->d_prefix); cudaFree(s->d_ones); cudaFree(s->d_resid); cudaFree(s->d_wlen); cudaFree(s->d_chunkcnt);
    for (auto& e : s->ev) if (e) cudaEventDestroy(e);
    for (auto& e : s->ev_copy) if (e) cudaEventDestroy(e);
    cudaFreeHost(s->h_jobs); cudaFreeHost(s->h_pairs); cudaFreeHost(s->h_prefix); cudaFreeHost(s->h_ones); cudaFreeHost(s->h_resid); cudaFreeHost(s->h_wlen);
    delete s;
}

static int stream_alloc(rbf_ctx* c, uint32_t H, uint32_t W, uint32_t C, uint32_t S, uint32_t max_frames, uint32_t max_pairs,
                        rbf_stream** out) {
    const uint64_t npix = (uint64_t)H * W;
    if (npix > 0xffffff00ULL) return set_err(c, RBF_ERR_INVALID, "frame too large");
    CK(c, cudaSetDevice(c->device));
    rbf_stream* s = new rbf_stream();
    s->c = c; s->H = H; s->W = W; s->C = C; s->S = S; s->max_frames = max_frames; s->max_pairs = max_pairs;
    s->npix = npix; s->frame_bytes = npix * C * S; s->frame_stride = align_up(s->frame_bytes + 64, 256);
    s->mask_stride_w = bit_words_padded(npix);
    s->pass_stride_w = pass_words(npix);
    cudaError_t e = cudaSuccess;
    auto dalloc = [&](void** p, size_t bytes) { if (e == cudaSuccess) e = cudaMalloc(p, bytes); };
    auto halloc = [&](void** p, size_t bytes) { if (e == cudaSuccess) e = cudaMallocHost(p, bytes); };
    dalloc((void**)&s->d_frames, s->frame_stride * max_frames);
    dalloc((void**)&s->d_mask, s->mask_stride_w * 4 * max_pairs);
    dalloc((void**)&s->d_bits, s->mask_stride_w * 4 * max_pairs);
    dalloc((void**)&s->d_wit, s->mask_stride_w * 4 * max_pairs);
    dalloc((void**)&s->d_pass, s->pass_stride_w * 4 * max_pairs);
    dalloc((void**)&s->d_jobs, sizeof(FrameJob) * max_pairs);
    dalloc((void**)&s->d_pairs, sizeof(PairJob) * max_pairs);
    dalloc((void**)&s->d_prefix, 4 * (3 * (size_t)max_pairs + 32));
    dalloc((void**)&s->d_ones, 4 * (size_t)max_pairs);
    dalloc((void**)&s->d_resid, 4 * (size_t)max_pairs);
    dalloc((void**)&s->d_wlen, 4 * (size_t)max_pairs);
    dalloc((void**)&s->d_chunkcnt, 4 * 32 * (size_t)max_pairs);
    halloc((void**)&s->h_jobs, sizeof(FrameJob) * max_pairs);
    halloc((void**)&s->h_pairs, sizeof(PairJob) * max_pairs);
    halloc((void**)&s->h_prefix, 4 * (3 * (size_t)max_pairs + 32));
    halloc((void**)&s->h_ones, 4 * (size_t)max_pairs);
    halloc((void**)&s->h_resid, 4 * (size_t)max_pairs);
    halloc((void**)&s->h_wlen, 4 * (size_t)max_pairs);
    if (e != cudaSuccess) {
        rbf_stream_destroy(s);
        return set_err(c, e == cudaErrorMemoryAllocation ? RBF_ERR_OOM : RBF_ERR_CUDA, "rbf_stream_create: %s", cudaGetErrorString(e));
    }
    for (auto& ev : s->ev) CK(c, cudaEventCreate(&ev));
    memset(s->h_ones, 0, 4 * (size_t)max_pairs); memset(s->h_resid, 0, 4 * (size_t)max_pairs); memset(s->h_wlen, 0, 4 * (size_t)max_pairs);
    s->k1_only = c->k1_only; s->mask_mode = c->mask_mode;
    CK(c, cudaMemsetAsync(s->d_wlen, 0, 4 * (size_t)max_pairs, c->st));
    CK(c, cudaMemsetAsync(s->d_bits, 0, s->mask_stride_w * 4 * max_pairs, c->st));
    CK(c, cudaMemsetAsync(s->d_wit, 0, s->mask_stride_w * 4 * max_pairs, c->st));
    CK(c, cudaMemsetAsync(s->d_mask, 0, s->mask_stride_w * 4 * max_pairs, c->st));   // zero padding once
    CK(c, cudaStreamSynchronize(c->st));
    *out = s;
    return RBF_OK;
}

extern "C" int rbf_stream_create(rbf_ctx* c, uint32_t H, uint32_t W, uint32_t C, uint32_t S, uint32_t max_frames,
                                 uint32_t max_pairs, rbf_stream** out) {
    if (!c || !out) return set_err(c, RBF_ERR_INVALID, "rbf_stream_create: NULL");
    if (!(S == 1 || S == 2) || !(C == 1 || C == 3) || H == 0 || W == 0 || max_frames < 2 || max_pairs < 1)
        return set_err(c, RBF_ERR_INVALID, "unsupported frame format H=%u W=%u C=%u sample_bytes=%u", H, W, C, S);
    return stream_alloc(c, H, W, C, S, max_frames, max_pairs, out);
}

extern "C" int rbf_stream_create_images(rbf_ctx* c, uint32_t H, uint32_t W, uint32_t C, uint32_t S, uint32_t max_images,
                                        rbf_stream** out) {
    if (!c || !out) return set_err(c, RBF_ERR_INVALID, "rbf_stream_create_images: NULL");
    const bool fmt = (S == 1 && C <= 4) || (S == 2 && C == 1);          // C = 0: decode-only, no image store
    if (!fmt || H == 0 || W == 0 || max_images < 1)
        return set_err(c, RBF_ERR_INVALID, "unsupported image format H=%u W=%u C=%u sample_bytes=%u max_images=%u", H, W, C, S, max_images);
    if (int r = stream_alloc(c, H, W, C, S, max_images, max_images, out)) return r;
    (*out)->images = true;
    (*out)->mask_mode = 0;
    return RBF_OK;
}

extern "C" int rbf_stream_set_option(rbf_stream* s, const char* key, int64_t v) {
    if (!s || !key) return set_err(s ? s->c : nullptr, RBF_ERR_INVALID, "rbf_stream_set_option: NULL");
    if (!strcmp(key, "k1_only")) { s->k1_only = v ? 1 : 0; return RBF_OK; }
    if (s->images && v && (!strcmp(key, "mask_mode") || !strcmp(key, "gray_mode")))
        return set_err(s->c, RBF_ERR_STATE, "%s is a frame-pair option; image streams binarize one image", key);
    if (!strcmp(key, "mask_mode")) { s->mask_mode = v ? 1 : 0; return RBF_OK; }
    if (!strcmp(key, "gray_mode")) {
        if (v && s->C != 3) return set_err(s->c, RBF_ERR_INVALID, "gray_mode needs 3-channel frames");
        s->gray_mode = v ? 1 : 0;
        return RBF_OK;
    }
    return set_err(s->c, RBF_ERR_INVALID, "unknown stream option %s", key);
}

extern "C" int rbf_stream_upload(rbf_stream* s, uint32_t first, uint32_t count, const void* host) {
    if (!s || !host) return set_err(s ? s->c : nullptr, RBF_ERR_INVALID, "rbf_stream_upload: NULL");
    rbf_ctx* c = s->c;
    if (s->frame_bytes == 0) return set_err(c, RBF_ERR_STATE, "decode-only image stream (0 channels): it has no image store");
    if ((uint64_t)first + count > s->max_frames) return set_err(c, RBF_ERR_INVALID, "frames [%u,%u) exceed store of %u", first, first + count, s->max_frames);
    CK(c, cudaMemcpy2DAsync(s->d_frames + (size_t)first * s->frame_stride, s->frame_stride, host, s->frame_bytes, s->frame_bytes,
                            count, cudaMemcpyHostToDevice, c->st));
    c->h2d += (int64_t)s->frame_bytes * count;
    CK(c, cudaStreamSynchronize(c->st));
    return RBF_OK;
}
extern "C" int rbf_stream_frame_ptr(rbf_stream* s, uint32_t frame, void** dptr) {
    if (!s || !dptr || frame >= s->max_frames) return set_err(s ? s->c : nullptr, RBF_ERR_INVALID, "rbf_stream_frame_ptr: bad argument");
    *dptr = s->d_frames + (size_t)frame * s->frame_stride;
    return RBF_OK;
}
extern "C" int rbf_stream_bitmap_region(rbf_stream* s, void** dptr, uint64_t* stride) {
    if (!s) return RBF_ERR_INVALID;
    if (dptr) *dptr = s->d_bits;
    if (stride) *stride = s->mask_stride_w * 4;
    return RBF_OK;
}

// `diff > threshold` with integer diff and a Python float threshold (ivc:808)  ==  diff > floor(threshold)
static int threshold_to_int(double thr) {
    if (isnan(thr)) return 0x7fffffff;                 // every comparison with NaN is False
    if (thr < -1.0) return -1;                         // diff >= -32768 only for uint16 wrap; handled below
    if (thr > 1e9) return 0x7fffffff;
    return (int)floor(thr);
}

// ---- pieces of the batched encode ----------------------------------------------------------
static int stream_thr_int(const rbf_stream* s, double threshold) {
    int thr_int = threshold_to_int(threshold);
    if (s->S == 2 && threshold < -1.0)                  // int16 abs can be -32768 (ivc:801): keep exact floor
        thr_int = threshold < -40000.0 ? -40000 : (int)floor(threshold);
    return thr_int;
}

static int stream_fill_pairs(rbf_stream* s, uint32_t first, uint32_t count, const uint32_t* prev_idx, const uint32_t* curr_idx) {
    for (uint32_t i = 0; i < count; i++) {
        if (prev_idx[i] >= s->max_frames || curr_idx[i] >= s->max_frames)
            return set_err(s->c, RBF_ERR_INVALID, "pair %u references a frame outside the store", first + i);
        PairJob& P = s->h_pairs[first + i];
        P.prev = s->d_frames + (size_t)prev_idx[i] * s->frame_stride;
        P.curr = s->d_frames + (size_t)curr_idx[i] * s->frame_stride;
        P.mask = s->d_mask + (size_t)(first + i) * s->mask_stride_w;
    }
    return RBF_OK;
}

struct RangeTotals {
    uint32_t total_cent = 0, coded_pairs = 0, max_l = 0;
};

// host side of pairs [first, first+count): K1's counts -> (p, k, l, T) exactly as the reference computes them -> FrameJob.
// hp[i+1] = base_cent + centuries of the coded pairs among the first i+1 of the range (K3's work list).
static void stream_range_params(rbf_stream* s, uint32_t first, uint32_t count, const rbf_seeds* sd, const double* kov,
                                const uint64_t* lov, uint32_t* hp, uint32_t base_cent, RangeTotals* out) {
    const uint32_t n = (uint32_t)s->npix, ncent = (n + 99u) / 100u;
    if (s->last_infos.size() < (size_t)first + count) s->last_infos.resize((size_t)first + count);
    uint32_t total_cent = base_cent;
    hp[0] = base_cent;
    for (uint32_t i = 0; i < count; i++) {
        rbf_mask_info& in = s->last_infos[first + i];
        memset(&in, 0, sizeof in);
        in.n = n; in.ones = s->h_ones[first + i]; in.resid = s->h_resid[first + i];
        double p, k; uint64_t l;
        int coded = rbf_optimal_params(n, in.ones, &p, &k, &l);
        in.p = p;
        if (kov && kov[i] > 0.0 && !(p >= kPStar)) { k = kov[i]; l = lov ? lov[i] : 0; coded = !(l == 0 || l >= n); }
        FrameJob& J = s->h_jobs[first + i];
        memset(&J, 0, sizeof J);
        J.n = n;
        J.mask = s->d_mask + (size_t)(first + i) * s->mask_stride_w;
        J.bits = s->d_bits + (size_t)(first + i) * s->mask_stride_w;
        J.witness = s->d_wit + (size_t)(first + i) * s->mask_stride_w;
        J.pass = s->d_pass + (size_t)(first + i) * s->pass_stride_w;
        if (coded) {
            job_set_filter(J, l, k, *sd);
            in.k = k; in.l = l; in.floor_k = J.floor_k; in.act_T = J.act_T;
            total_cent += ncent; out->coded_pairs++;
            if (l > out->max_l) out->max_l = (uint32_t)l;
        } else {
            in.raw = 1;
        }
        hp[i + 1] = total_cent;
    }
    out->total_cent = total_cent - base_cent;
}

// Zero what K2 / K3b will OR into.  Nothing ever writes a bit array at or beyond bit l, or a witness at or beyond bit wlen,
// and both regions are fully zeroed at creation, so clearing [0, high-water mark) of every slot is enough.
static int stream_clear_outputs(rbf_stream* s, uint32_t first, uint32_t count, uint32_t max_l, cudaStream_t st) {
    rbf_ctx* c = s->c;
    const size_t stride = s->mask_stride_w * 4;
    const size_t need = align_up((size_t)((max_l + 31u) / 32u) * 4 + 64, 128);
    if (need > s->bits_hwm) s->bits_hwm = need;
    const size_t wb = s->bits_hwm < stride ? s->bits_hwm : stride;
    const size_t ww = (s->wit_dirty_full || s->wit_hwm > stride) ? stride : s->wit_hwm;
    CK(c, cudaMemset2DAsync(s->d_bits + (size_t)first * s->mask_stride_w, stride, 0, wb, count, st));
    if (ww) CK(c, cudaMemset2DAsync(s->d_wit + (size_t)first * s->mask_stride_w, stride, 0, ww, count, st));
    return RBF_OK;
}
static void stream_note_witness(rbf_stream* s, uint32_t first, uint32_t count) {      // after the encode has been synchronised
    for (uint32_t i = 0; i < count; i++) {
        const size_t nb = align_up((size_t)((s->h_wlen[first + i] + 31u) / 32u) * 4 + 64, 128);
        if (nb > s->wit_hwm) s->wit_hwm = nb;
    }
}

// Encode pairs [first, first+count) (slots of all per-pair arrays) serially on the context's stream; `pfx` is the slot of this
// range's century-prefix array (count+1 entries) inside h_prefix/d_prefix.  Used per chunk by rbf_stream_encode_host.
static int stream_encode_range(rbf_stream* s, uint32_t first, uint32_t count, uint32_t pfx, const uint32_t* prev_idx,
                               const uint32_t* curr_idx, double threshold, const rbf_seeds* sd, const double* kov,
                               const uint64_t* lov, bool record_events) {
    rbf_ctx* c = s->c;
    const uint32_t n = (uint32_t)s->npix;
    const int thr_int = stream_thr_int(s, threshold);
    if (int r = stream_fill_pairs(s, first, count, prev_idx, curr_idx)) return r;
    CK(c, cudaMemcpyAsync(s->d_pairs + first, s->h_pairs + first, sizeof(PairJob) * count, cudaMemcpyHostToDevice, c->st));
    CK(c, cudaMemsetAsync(s->d_ones + first, 0, 4 * (size_t)count, c->st));
    CK(c, cudaMemsetAsync(s->d_resid + first, 0, 4 * (size_t)count, c->st));
    if (record_events) { s->staged = false; CK(c, cudaEventRecord(s->ev[0], c->st)); }
    LAUNCH(c, launch_threshold(s->d_pairs + first, (int)count, n, (int)s->C, (int)s->S, thr_int, s->mask_mode, s->gray_mode,
                               s->d_ones + first, s->d_resid + first, c->k1_variant, c->sm_count, c->k1_ctas_per_sm, c->st));
    if (c->k1_variant == 1 && !s->gray_mode) c->launches++;              // tail kernel
    if (record_events) CK(c, cudaEventRecord(s->ev[1], c->st));
    CK(c, cudaMemcpyAsync(s->h_ones + first, s->d_ones + first, 4 * (size_t)count, cudaMemcpyDeviceToHost, c->st));
    CK(c, cudaMemcpyAsync(s->h_resid + first, s->d_resid + first, 4 * (size_t)count, cudaMemcpyDeviceToHost, c->st));
    c->d2h += 8 * (int64_t)count;
    CK(c, cudaStreamSynchronize(c->st));               // the one host round trip: (p, k, l, T) need libm's log2
    const uint32_t ncent = (n + 99u) / 100u;
    RangeTotals rt;
    uint32_t* hp = s->h_prefix + pfx;
    stream_range_params(s, first, count, sd, kov, lov, hp, 0, &rt);
    if (first + count > s->last_pairs || first == 0) s->last_pairs = first + count;
    if (rt.max_l > s->last_max_l || first == 0) s->last_max_l = rt.max_l;
    s->last_k1_only = s->k1_only != 0;
    if (rt.coded_pairs == 0 || s->k1_only) return RBF_OK;
    CK(c, cudaMemcpyAsync(s->d_jobs + first, s->h_jobs + first, sizeof(FrameJob) * count, cudaMemcpyHostToDevice, c->st));
    CK(c, cudaMemcpyAsync(s->d_prefix + pfx, hp, 4 * ((size_t)count + 1), cudaMemcpyHostToDevice, c->st));
    if (int r = wait_pack(c)) return r;                  // the slots of the last all-gather are packed
    if (int r = stream_clear_outputs(s, first, count, rt.max_l, c->st)) return r;
    if (record_events) CK(c, cudaEventRecord(s->ev[2], c->st));
    LAUNCH(c, launch_insert(s->d_jobs + first, (int)count, ncent, c->insert_variant, c->sm_count, c->st));
    if (record_events) CK(c, cudaEventRecord(s->ev[3], c->st));
    LAUNCH(c, launch_query(s->d_jobs + first, s->d_prefix + pfx, (int)count, rt.total_cent, rt.max_l, c->query_variant, c->sm_count,
                           c->query_smem_cap, c->query_warps, c->st));
    if (record_events) CK(c, cudaEventRecord(s->ev[4], c->st));
    s->wit_dirty_full = true;                            // until the witness lengths of this encode are known
    LAUNCH(c, launch_witness(s->d_jobs + first, (int)count, ncent, c->sm_count, s->d_chunkcnt + 32 * (size_t)first, s->d_wlen + first, c->st));
    c->launches += 2;                                   // pass-count + finalize kernels
    if (record_events) { CK(c, cudaEventRecord(s->ev[5], c->st)); s->staged = true; }
    CK(c, cudaMemcpyAsync(s->h_wlen + first, s->d_wlen + first, 4 * (size_t)count, cudaMemcpyDeviceToHost, c->st));
    c->d2h += 4 * (int64_t)count;
    return RBF_OK;
}

static int ensure_pipe_streams(rbf_ctx* c) {
    if (!c->st_k1) {
        CK(c, cudaStreamCreateWithFlags(&c->st_k1, cudaStreamNonBlocking));
        CK(c, cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
        for (auto& e : c->ev_k1) CK(c, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    return RBF_OK;
}

// The resident-stream encode, pipelined: K1 has no host dependency, so K1 of ALL ranges is enqueued up front on a second
// stream; as soon as a range's counts have landed the host derives its (k, l, T) and enqueues that range's K2 on the main
// stream, where it runs BESIDE K1 of the later ranges (K1 is HBM-bound with a grid that leaves SM slots free, K2 is
// issue/atomics-bound), and the host round trip is hidden behind both.  K3 and K3b are single launches over all pairs.
static int stream_encode_pipelined(rbf_stream* s, uint32_t pairs, const uint32_t* prev_idx, const uint32_t* curr_idx,
                                   double threshold, const rbf_seeds* sd, const double* kov, const uint64_t* lov) {
    rbf_ctx* c = s->c;
    const uint32_t n = (uint32_t)s->npix, ncent = (n + 99u) / 100u;
    const int thr_int = s->images ? threshold_to_int(threshold) : stream_thr_int(s, threshold);
    uint32_t R = (uint32_t)c->encode_ranges;
    if (R > 8u) R = 8u;
    if (pairs < 8u * R) R = 1u;                          // small jobs: nothing to hide behind
    if (int r = ensure_pipe_streams(c)) return r;
    if (int r = stream_fill_pairs(s, 0, pairs, prev_idx, curr_idx)) return r;
    CK(c, cudaMemcpyAsync(s->d_pairs, s->h_pairs, sizeof(PairJob) * pairs, cudaMemcpyHostToDevice, c->st));
    CK(c, cudaMemsetAsync(s->d_ones, 0, 4 * (size_t)pairs, c->st));
    CK(c, cudaMemsetAsync(s->d_resid, 0, 4 * (size_t)pairs, c->st));
    s->staged = false;
    CK(c, cudaEventRecord(s->ev[0], c->st));
    CK(c, cudaEventRecord(c->ev_fork, c->st));
    CK(c, cudaStreamWaitEvent(c->st_k1, c->ev_fork, 0));
    uint32_t lo[9];
    for (uint32_t r = 0; r <= R; r++) lo[r] = (uint32_t)(((uint64_t)pairs * r) / R);
    const int k1_cap = R > 1u ? c->pipe_k1_ctas_per_sm : c->k1_ctas_per_sm;
    for (uint32_t r = 0; r < R; r++) {
        const uint32_t f = lo[r], cnt = lo[r + 1] - lo[r];
        if (s->images) {
            LAUNCH(c, launch_binarize(s->d_pairs + f, (int)cnt, n, (int)s->C, (int)s->S, thr_int, s->d_ones + f, c->sm_count, k1_cap, c->st_k1));
        } else {
            LAUNCH(c, launch_threshold(s->d_pairs + f, (int)cnt, n, (int)s->C, (int)s->S, thr_int, s->mask_mode, s->gray_mode, s->d_ones + f,
                                       s->d_resid + f, c->k1_variant, c->sm_count, k1_cap, c->st_k1));
            if (c->k1_variant == 1 && !s->gray_mode) c->launches++;
        }
        CK(c, cudaMemcpyAsync(s->h_ones + f, s->d_ones + f, 4 * (size_t)cnt, cudaMemcpyDeviceToHost, c->st_k1));
        CK(c, cudaMemcpyAsync(s->h_resid + f, s->d_resid + f, 4 * (size_t)cnt, cudaMemcpyDeviceToHost, c->st_k1));
        CK(c, cudaEventRecord(c->ev_k1[r], c->st_k1));
    }
    CK(c, cudaEventRecord(s->ev[1], c->st_k1));           // end of the last K1
    c->d2h += 8 * (int64_t)pairs;
    s->last_infos.clear();
    s->last_pairs = pairs; s->last_max_l = 0;
    s->last_k1_only = s->k1_only != 0;
    RangeTotals all;
    uint32_t base_cent = 0;
    bool first_k2 = true;
    // K2 || K3 mode (kq_ranges > 1, serial K1): K2 is bound by L2 atomics with the SMs mostly waiting, K3 by instruction issue with
    // L2 idle; K2 of range q+1 is enqueued on the second stream and runs BESIDE K3 of range q (K3 is then launched with fewer
    // warps and a little less shared memory -- options query_warps / query_smem_bytes -- so that one K2 CTA fits next to it).
    uint32_t Q = (R == 1u && !s->k1_only) ? (uint32_t)c->kq_ranges : 1u;
    if (Q > 8u) Q = 8u;
    if (pairs < 8u * Q) Q = 1u;
    const bool kq = Q > 1u;
    for (uint32_t r = 0; r < R; r++) {
        const uint32_t f = lo[r], cnt = lo[r + 1] - lo[r];
        CK(c, cudaEventSynchronize(c->ev_k1[r]));         // this range's counts are on the host
        RangeTotals rt;
        stream_range_params(s, f, cnt, sd, kov, lov, s->h_prefix + f, base_cent, &rt);
        base_cent += rt.total_cent;
        all.coded_pairs += rt.coded_pairs;
        if (rt.max_l > all.max_l) all.max_l = rt.max_l;
        if (s->k1_only || rt.coded_pairs == 0) continue;
        CK(c, cudaStreamWaitEvent(c->st, c->ev_k1[r], 0)); // K2 reads the masks K1 wrote on the other stream
        CK(c, cudaMemcpyAsync(s->d_jobs + f, s->h_jobs + f, sizeof(FrameJob) * cnt, cudaMemcpyHostToDevice, c->st));
        if (first_k2) { if (int e = wait_pack(c)) return e; }
        if (int e = stream_clear_outputs(s, f, cnt, rt.max_l, c->st)) return e;
        if (first_k2) { CK(c, cudaEventRecord(s->ev[2], c->st)); first_k2 = false; }
        if (!kq) LAUNCH(c, launch_insert(s->d_jobs + f, (int)cnt, ncent, c->insert_variant, c->sm_count, c->st));
    }
    all.total_cent = base_cent;
    s->last_max_l = all.max_l;
    if (s->k1_only || all.coded_pairs == 0) {
        CK(c, cudaStreamWaitEvent(c->st, c->ev_k1[R - 1], 0));
        return RBF_OK;
    }
    CK(c, cudaMemcpyAsync(s->d_prefix, s->h_prefix, 4 * ((size_t)pairs + 1), cudaMemcpyHostToDevice, c->st));
    if (kq) {
        uint32_t qlo[9];
        for (uint32_t q = 0; q <= Q; q++) qlo[q] = (uint32_t)(((uint64_t)pairs * q) / Q);
        // per-range work lists for K3 (each starts at 0), behind the whole-encode list that decode_verify uses
        uint32_t* hp2 = s->h_prefix + pairs + 1;
        uint32_t off = 0, range_cent[8], range_off[8];
        for (uint32_t q = 0; q < Q; q++) {
            range_off[q] = off;
            const uint32_t b0 = s->h_prefix[qlo[q]];
            for (uint32_t i = qlo[q]; i <= qlo[q + 1]; i++) hp2[off++] = s->h_prefix[i] - b0;
            range_cent[q] = s->h_prefix[qlo[q + 1]] - b0;
        }
        CK(c, cudaMemcpyAsync(s->d_prefix + pairs + 1, hp2, 4 * (size_t)off, cudaMemcpyHostToDevice, c->st));
        CK(c, cudaEventRecord(c->ev_fork, c->st));            // jobs, prefix lists and cleared outputs are in place
        CK(c, cudaStreamWaitEvent(c->st_k1, c->ev_fork, 0));
        for (uint32_t q = 0; q < Q; q++) {
            const uint32_t f = qlo[q], cnt = qlo[q + 1] - qlo[q];
            LAUNCH(c, launch_insert(s->d_jobs + f, (int)cnt, ncent, c->insert_variant, c->sm_count, c->st_k1));
            CK(c, cudaEventRecord(c->ev_k1[q], c->st_k1));
            CK(c, cudaStreamWaitEvent(c->st, c->ev_k1[q], 0));
            if (q == 0) CK(c, cudaEventRecord(s->ev[3], c->st));
            LAUNCH(c, launch_query(s->d_jobs + f, s->d_prefix + pairs + 1 + range_off[q], (int)cnt, range_cent[q], all.max_l, c->query_variant,
                                   c->sm_count, c->query_smem_cap, c->query_warps, c->st));
        }
    } else {
        CK(c, cudaEventRecord(s->ev[3], c->st));
        LAUNCH(c, launch_query(s->d_jobs, s->d_prefix, (int)pairs, all.total_cent, all.max_l, c->query_variant, c->sm_count,
                               c->query_smem_cap, c->query_warps, c->st));
    }
    CK(c, cudaEventRecord(s->ev[4], c->st));
    s->wit_dirty_full = true;
    LAUNCH(c, launch_witness(s->d_jobs, (int)pairs, ncent, c->sm_count, s->d_chunkcnt, s->d_wlen, c->st));
    c->launches += 2;                                   // pass-count + finalize kernels
    CK(c, cudaEventRecord(s->ev[5], c->st));
    s->staged = true;
    CK(c, cudaMemcpyAsync(s->h_wlen, s->d_wlen, 4 * (size_t)pairs, cudaMemcpyDeviceToHost, c->st));
    c->d2h += 4 * (int64_t)pairs;
    return RBF_OK;
}

extern "C" int rbf_stream_encode(rbf_stream* s, const uint32_t* prev_idx, const uint32_t* curr_idx, uint32_t pairs,
                                 double threshold, const rbf_seeds* sd, const double* kov, const uint64_t* lov,
                                 rbf_mask_info* infos) {
    if (!s || !prev_idx || !curr_idx || !sd) return set_err(s ? s->c : nullptr, RBF_ERR_INVALID, "rbf_stream_encode: NULL");
    rbf_ctx* c = s->c;
    if (pairs == 0 || pairs > s->max_pairs) return set_err(c, RBF_ERR_INVALID, "pairs = %u outside [1, %u]", pairs, s->max_pairs);
    if (s->frame_bytes == 0) return set_err(c, RBF_ERR_STATE, "decode-only image stream (0 channels): nothing to encode");
    if (s->images)
        for (uint32_t i = 0; i < pairs; i++)
            if (prev_idx[i] != curr_idx[i]) return set_err(c, RBF_ERR_INVALID, "image stream: prev_idx[%u] != curr_idx[%u]", i, i);
    CK(c, cudaSetDevice(c->device));
    int rc = stream_encode_pipelined(s, pairs, prev_idx, curr_idx, threshold, sd, kov, lov);
    if (rc) { cudaStreamSynchronize(c->st_k1); cudaStreamSynchronize(c->st); return rc; }
    CK(c, cudaStreamSynchronize(c->st));
    const bool coded_run = !s->k1_only;
    if (coded_run) { stream_note_witness(s, 0, pairs); s->wit_dirty_full = false; }
    for (uint32_t i = 0; i < pairs; i++) {
        s->last_infos[i].wlen = (coded_run && !s->last_infos[i].raw) ? s->h_wlen[i] : 0;
        if (infos) infos[i] = s->last_infos[i];
    }
    return RBF_OK;
}

extern "C" int rbf_stream_stage_ms(rbf_stream* s, double out[6]) {
    if (!s || !out) return RBF_ERR_INVALID;
    rbf_ctx* c = s->c;
    if (!s->staged) return set_err(c, RBF_ERR_STATE, "no fully staged encode has run");
    CK(c, cudaEventSynchronize(s->ev[5]));
    auto span = [&](int a, int b, double* o) -> cudaError_t { float f = 0; cudaError_t e = cudaEventElapsedTime(&f, s->ev[a], s->ev[b]); *o = f; return e; };
    CK(c, span(0, 1, &out[0]));     // K1: first launch .. end of the last range (runs beside K2 of the earlier ranges)
    CK(c, span(0, 3, &out[1]));     // everything in front of K3: K1 + host (k, l, T) round trips + K2, as overlapped
    CK(c, span(2, 3, &out[2]));     // K2: first launch .. end of the last range
    CK(c, span(3, 4, &out[3]));     // K3
    CK(c, span(4, 5, &out[4]));     // K3b (pass count, witness, packbits order)
    CK(c, span(0, 5, &out[5]));     // whole encode
    return RBF_OK;
}

extern "C" int rbf_stream_fetch(rbf_stream* s, uint32_t pair, uint8_t* bitmap, uint8_t* witness, uint8_t* mask_little) {
    if (!s) return RBF_ERR_INVALID;
    rbf_ctx* c = s->c;
    if (pair >= s->last_pairs) return set_err(c, RBF_ERR_INVALID, "pair %u was not encoded", pair);
    if (s->last_k1_only && (bitmap || witness))
        return set_err(c, RBF_ERR_STATE, "the last encode stopped after K1 (k1_only): there is no bitmap / witness to fetch");
    const rbf_mask_info& in = s->last_infos[pair];
    if (bitmap && !in.raw) { size_t nb = (in.l + 7) / 8; CK(c, cudaMemcpyAsync(bitmap, s->d_bits + (size_t)pair * s->mask_stride_w, nb, cudaMemcpyDeviceToHost, c->st)); c->d2h += nb; }
    if (witness && !in.raw && in.wlen) { size_t nb = (in.wlen + 7) / 8; CK(c, cudaMemcpyAsync(witness, s->d_wit + (size_t)pair * s->mask_stride_w, nb, cudaMemcpyDeviceToHost, c->st)); c->d2h += nb; }
    if (mask_little) { size_t nb = (s->npix + 7) / 8; CK(c, cudaMemcpyAsync(mask_little, s->d_mask + (size_t)pair * s->mask_stride_w, nb, cudaMemcpyDeviceToHost, c->st)); c->d2h += nb; }
    CK(c, cudaStreamSynchronize(c->st));
    return RBF_OK;
}

// One strided copy per output kind for pairs [first, first+count) and ONE synchronisation (the GOP loop's batched fetch).
extern "C" int rbf_stream_fetch_batch(rbf_stream* s, uint32_t first, uint32_t count, uint8_t* bitmaps, uint64_t bitmap_slot,
                                      uint8_t* witness, uint64_t witness_slot, uint8_t* masks_little, uint64_t mask_slot) {
    if (!s) return RBF_ERR_INVALID;
    rbf_ctx* c = s->c;
    if (count == 0 || (uint64_t)first + count > s->last_pairs) return set_err(c, RBF_ERR_INVALID, "pairs [%u,%u) were not encoded", first, first + count);
    if (s->last_k1_only && (bitmaps || witness))
        return set_err(c, RBF_ERR_STATE, "the last encode stopped after K1 (k1_only): there is no bitmap / witness to fetch");
    const size_t stride = s->mask_stride_w * 4;
    auto copy2d = [&](uint8_t* dst, uint64_t slot, const uint32_t* src) -> cudaError_t {
        const size_t w = slot < stride ? (size_t)slot : stride;
        c->d2h += (int64_t)w * count;
        return cudaMemcpy2DAsync(dst, slot, (const uint8_t*)src + (size_t)first * stride, stride, w, count, cudaMemcpyDeviceToHost, c->st);
    };
    if (bitmaps && bitmap_slot) CK(c, copy2d(bitmaps, bitmap_slot, s->d_bits));
    if (witness && witness_slot) CK(c, copy2d(witness, witness_slot, s->d_wit));
    if (masks_little && mask_slot) CK(c, copy2d(masks_little, mask_slot, s->d_mask));
    CK(c, cudaStreamSynchronize(c->st));
    return RBF_OK;
}

extern "C" int rbf_stream_encode_host(rbf_stream* s, const void* host_frames, uint32_t nframes, double threshold,
                                      const rbf_seeds* sd, rbf_mask_info* infos, uint8_t* bitmaps, uint64_t bitmap_slot,
                                      uint8_t* witness, uint64_t witness_slot) {
    if (!s || !host_frames || !sd || nframes < 2) return set_err(s ? s->c : nullptr, RBF_ERR_INVALID, "rbf_stream_encode_host: bad argument");
    rbf_ctx* c = s->c;
    const uint32_t pairs = nframes - 1;
    if (nframes > s->max_frames || pairs > s->max_pairs) return set_err(c, RBF_ERR_INVALID, "stream too small for %u frames", nframes);
    CK(c, cudaSetDevice(c->device));
    if (!c->st_copy) CK(c, cudaStreamCreateWithFlags(&c->st_copy, cudaStreamNonBlocking));
    if (!c->st_d2h) { CK(c, cudaStreamCreateWithFlags(&c->st_d2h, cudaStreamNonBlocking)); CK(c, cudaEventCreateWithFlags(&c->ev_d2h, cudaEventDisableTiming)); }
    if (s->k1_only) return set_err(c, RBF_ERR_STATE, "rbf_stream_encode_host on a k1_only stream");
    if (s->images) return set_err(c, RBF_ERR_STATE, "rbf_stream_encode_host codes frame pairs; image streams use rbf_stream_encode");
    // chunks of frames: all H2D copies are queued on the copy stream up front (pinned source), the compute stream
    // encodes a chunk's pairs as soon as its frames have landed, so PCIe transfer and kernels overlap
    const uint32_t CH = c->host_chunk_frames > 1 ? (uint32_t)c->host_chunk_frames : 32u;
    const uint32_t nchunks = (nframes + CH - 1) / CH;
    while (s->ev_copy.size() < nchunks) { cudaEvent_t e; CK(c, cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); s->ev_copy.push_back(e); }
    const uint8_t* src = (const uint8_t*)host_frames;
    for (uint32_t k = 0; k < nchunks; k++) {
        const uint32_t f0 = k * CH, f1 = (f0 + CH < nframes) ? f0 + CH : nframes;
        CK(c, cudaMemcpy2DAsync(s->d_frames + (size_t)f0 * s->frame_stride, s->frame_stride, src + (size_t)f0 * s->frame_bytes,
                                s->frame_bytes, s->frame_bytes, f1 - f0, cudaMemcpyHostToDevice, c->st_copy));
        CK(c, cudaEventRecord(s->ev_copy[k], c->st_copy));
    }
    c->h2d += (int64_t)s->frame_bytes * nframes;
    s->last_infos.clear();
    s->last_pairs = 0; s->last_max_l = 0;
    const size_t stride = s->mask_stride_w * 4;
    std::vector<uint32_t> pi, ci;
    for (uint32_t k = 0; k < nchunks; k++) {
        const uint32_t f0 = k * CH, f1 = (f0 + CH < nframes) ? f0 + CH : nframes;
        const uint32_t p0 = f0 == 0 ? 0 : f0 - 1, p1 = f1 - 1;      // pairs (i, i+1) whose current frame is in this chunk
        if (p1 <= p0) continue;
        const uint32_t cnt = p1 - p0;
        pi.resize(cnt); ci.resize(cnt);
        for (uint32_t i = 0; i < cnt; i++) { pi[i] = p0 + i; ci[i] = p0 + i + 1; }
        CK(c, cudaStreamWaitEvent(c->st, s->ev_copy[k], 0));
        int rc = stream_encode_range(s, p0, cnt, p0 + k, pi.data(), ci.data(), threshold, sd, nullptr, nullptr, false);
        if (rc) return rc;
        // the packed results of this chunk go back on their own stream, beside the kernels of the next chunk
        CK(c, cudaEventRecord(c->ev_d2h, c->st));
        CK(c, cudaStreamWaitEvent(c->st_d2h, c->ev_d2h, 0));
        if (bitmaps && bitmap_slot) {
            const size_t w = bitmap_slot < stride ? bitmap_slot : stride;
            CK(c, cudaMemcpy2DAsync(bitmaps + (size_t)p0 * bitmap_slot, bitmap_slot, (const uint8_t*)s->d_bits + (size_t)p0 * stride, stride,
                                    w, cnt, cudaMemcpyDeviceToHost, c->st_d2h));
            c->d2h += (int64_t)w * cnt;
        }
        if (witness && witness_slot) {
            const size_t w = witness_slot < stride ? witness_slot : stride;
            CK(c, cudaMemcpy2DAsync(witness + (size_t)p0 * witness_slot, witness_slot, (const uint8_t*)s->d_wit + (size_t)p0 * stride, stride,
                                    w, cnt, cudaMemcpyDeviceToHost, c->st_d2h));
            c->d2h += (int64_t)w * cnt;
        }
    }
    CK(c, cudaEventRecord(c->ev_d2h, c->st_d2h));        // the caller's timer / next call on `st` sees the copies done
    CK(c, cudaStreamWaitEvent(c->st, c->ev_d2h, 0));
    CK(c, cudaStreamSynchronize(c->st));
    stream_note_witness(s, 0, pairs);
    s->wit_dirty_full = false;
    // one contiguous prefix array for later decode_verify over all pairs
    {
        const uint32_t ncent = (uint32_t)((s->npix + 99) / 100);
        uint32_t tot = 0;
        s->h_prefix[0] = 0;
        for (uint32_t i = 0; i < pairs; i++) { if (!s->last_infos[i].raw) tot += ncent; s->h_prefix[i + 1] = tot; }
        CK(c, cudaMemcpyAsync(s->d_prefix, s->h_prefix, 4 * ((size_t)pairs + 1), cudaMemcpyHostToDevice, c->st));
        CK(c, cudaStreamSynchronize(c->st));
    }
    for (uint32_t i = 0; i < pairs; i++) {
        if (!s->last_infos[i].raw) s->last_infos[i].wlen = s->h_wlen[i];
        if (infos) infos[i] = s->last_infos[i];
    }
    return RBF_OK;
}

// Decode slots [0, pairs) of the bit-array / witness regions (packbits order; h_jobs and d_prefix / h_prefix describe the filters)
// into d_dec (ivc:268-307, bc:307-346); the number of Bloom-test passes of each lands in d_wlen.  Leaves the slots LSB-first.
static int stream_decode_slots(rbf_stream* s, uint32_t pairs, uint32_t max_l, const uint64_t* wlen) {
    rbf_ctx* c = s->c;
    const size_t stride_w = s->mask_stride_w;
    if (!s->d_dec) CK(c, cudaMalloc((void**)&s->d_dec, stride_w * 4 * s->max_pairs));
    CK(c, cudaMemsetAsync(s->d_dec, 0, stride_w * 4 * pairs, c->st));
    // bitmap and witness sit in packbits order after K3b; the kernels work LSB-first
    if (int r = wait_pack(c)) return r;
    LAUNCH(c, launch_bitrev(s->d_bits, stride_w * pairs, c->st));
    LAUNCH(c, launch_bitrev(s->d_wit, stride_w * pairs, c->st));
    for (uint32_t i = 0; i < pairs; i++) {
        FrameJob& J = s->h_jobs[i];
        J.out_mask = s->d_dec + (size_t)i * stride_w;
        J.wlen_in = (uint32_t)wlen[i];
        J.mask = nullptr;                               // a real decode knows no mask (ivc:286-304)
    }
    CK(c, cudaMemcpyAsync(s->d_jobs, s->h_jobs, sizeof(FrameJob) * pairs, cudaMemcpyHostToDevice, c->st));
    const uint32_t total_cent = s->h_prefix[pairs];
    LAUNCH(c, launch_query(s->d_jobs, s->d_prefix, (int)pairs, total_cent, max_l, c->query_variant, c->sm_count, c->query_smem_cap, c->query_warps, c->st));
    LAUNCH(c, launch_expand(s->d_jobs, (int)pairs, (uint32_t)((s->npix + 99) / 100), c->sm_count, s->d_chunkcnt, s->d_wlen, c->st));
    c->launches += 1;
    return RBF_OK;
}

extern "C" int rbf_stream_decode_verify(rbf_stream* s, uint32_t pairs, uint64_t* mismatches) {
    if (!s || !mismatches) return set_err(s ? s->c : nullptr, RBF_ERR_INVALID, "rbf_stream_decode_verify: NULL");
    rbf_ctx* c = s->c;
    if (pairs == 0 || pairs > s->last_pairs) return set_err(c, RBF_ERR_INVALID, "only %u pairs were encoded", s->last_pairs);
    CK(c, cudaSetDevice(c->device));
    const size_t stride_w = s->mask_stride_w;
    std::vector<uint64_t> wlen(pairs);
    for (uint32_t i = 0; i < pairs; i++) wlen[i] = s->last_infos[i].wlen;
    if (int r = stream_decode_slots(s, pairs, s->last_max_l, wlen.data())) return r;
    void* d_cnt; int rc;
    if ((rc = scratch_get(c, 7, 4 * (size_t)pairs + 4096, &d_cnt))) return rc;
    CK(c, cudaMemsetAsync(d_cnt, 0, 4 * (size_t)pairs, c->st));
    LAUNCH(c, launch_count_diff(s->d_mask, s->d_dec, stride_w, (s->npix + 31) / 32, (int)pairs, (uint32_t*)d_cnt, c->st));
    LAUNCH(c, launch_bitrev(s->d_bits, stride_w * pairs, c->st));
    LAUNCH(c, launch_bitrev(s->d_wit, stride_w * pairs, c->st));
    std::vector<uint32_t> h(pairs);
    CK(c, cudaMemcpyAsync(h.data(), d_cnt, 4 * (size_t)pairs, cudaMemcpyDeviceToHost, c->st));
    CK(c, cudaStreamSynchronize(c->st));
    for (uint32_t i = 0; i < pairs; i++) mismatches[i] = s->last_infos[i].raw ? 0 : h[i];
    return RBF_OK;
}

extern "C" int rbf_stream_decode(rbf_stream* s, uint32_t count, const uint64_t* l, const uint64_t* wlen, const double* k,
                                 const rbf_seeds* sd, const uint8_t* bitmaps, uint64_t bitmap_slot, const uint8_t* witness,
                                 uint64_t witness_slot, uint8_t* masks_little, uint64_t mask_slot, uint64_t* consumed) {
    if (!s || !l || !wlen || !k || !sd || !bitmaps || !witness || !masks_little || !consumed)
        return set_err(s ? s->c : nullptr, RBF_ERR_INVALID, "rbf_stream_decode: NULL");
    rbf_ctx* c = s->c;
    if (count == 0 || count > s->max_pairs) return set_err(c, RBF_ERR_INVALID, "count = %u outside [1, %u]", count, s->max_pairs);
    const uint64_t n = s->npix, mbytes = (n + 7) / 8;
    const size_t stride = s->mask_stride_w * 4;
    uint64_t max_l = 0;
    for (uint32_t i = 0; i < count; i++) {
        // l > n or wlen > n only come from a corrupt payload; the single-mask decoder (rbf_decompress_mask) takes those
        if (l[i] == 0 || l[i] > n || wlen[i] > n || !(k[i] >= 0.0) || k[i] > 1e6)
            return set_err(c, RBF_ERR_INVALID, "image %u: l=%llu wlen=%llu k=%g outside the stream's range (n=%llu)", i,
                           (unsigned long long)l[i], (unsigned long long)wlen[i], k[i], (unsigned long long)n);
        if ((l[i] + 7) / 8 > bitmap_slot || (wlen[i] + 7) / 8 > witness_slot)
            return set_err(c, RBF_ERR_INVALID, "image %u: bitmap / witness larger than its slot", i);
        if (l[i] > max_l) max_l = l[i];
    }
    if (mask_slot < mbytes) return set_err(c, RBF_ERR_INVALID, "mask slot %llu < %llu bytes", (unsigned long long)mask_slot, (unsigned long long)mbytes);
    CK(c, cudaSetDevice(c->device));
    if (int r = wait_pack(c)) return r;
    // the payloads replace the outputs of the last encode: no fetch / decode_verify of it from here on
    s->last_pairs = 0; s->last_infos.clear(); s->staged = false;
    const size_t bw = bitmap_slot < stride ? (size_t)bitmap_slot : stride, ww = witness_slot < stride ? (size_t)witness_slot : stride;
    if (bw > s->bits_hwm) s->bits_hwm = bw;               // the next encode clears what was written here
    if (ww > s->wit_hwm) s->wit_hwm = ww;
    CK(c, cudaMemcpy2DAsync(s->d_bits, stride, bitmaps, bitmap_slot, bw, count, cudaMemcpyHostToDevice, c->st));
    CK(c, cudaMemcpy2DAsync(s->d_wit, stride, witness, witness_slot, ww, count, cudaMemcpyHostToDevice, c->st));
    c->h2d += (int64_t)(bw + ww) * count;
    const uint32_t ncent = (uint32_t)((n + 99) / 100);
    s->h_prefix[0] = 0;
    for (uint32_t i = 0; i < count; i++) {
        FrameJob& J = s->h_jobs[i];
        memset(&J, 0, sizeof J);
        J.n = (uint32_t)n;
        job_set_filter(J, l[i], k[i], *sd);
        J.bits = s->d_bits + (size_t)i * s->mask_stride_w;
        J.witness = s->d_wit + (size_t)i * s->mask_stride_w;
        J.pass = s->d_pass + (size_t)i * s->pass_stride_w;
        s->h_prefix[i + 1] = s->h_prefix[i] + ncent;
    }
    CK(c, cudaMemcpyAsync(s->d_prefix, s->h_prefix, 4 * ((size_t)count + 1), cudaMemcpyHostToDevice, c->st));
    if (int r = stream_decode_slots(s, count, (uint32_t)max_l, wlen)) return r;
    CK(c, cudaMemcpy2DAsync(masks_little, mask_slot, s->d_dec, stride, mbytes, count, cudaMemcpyDeviceToHost, c->st));
    CK(c, cudaMemcpyAsync(s->h_wlen, s->d_wlen, 4 * (size_t)count, cudaMemcpyDeviceToHost, c->st));
    c->d2h += (int64_t)mbytes * count + 4 * (int64_t)count;
    CK(c, cudaStreamSynchronize(c->st));
    for (uint32_t i = 0; i < count; i++) consumed[i] = s->h_wlen[i];
    return RBF_OK;
}


// ------------------------------------------------------------------------------------------
// N1 / N2: changed-value gather and frame reconstruction on the device
// ------------------------------------------------------------------------------------------
extern "C" int rbf_stream_gather_changed(rbf_stream* s, uint32_t pairs, uint8_t* values_out, uint64_t capacity,
                                         uint64_t* offsets_out) {
    if (!s || !offsets_out) return set_err(s ? s->c : nullptr, RBF_ERR_INVALID, "rbf_stream_gather_changed: NULL");
    rbf_ctx* c = s->c;
    if (pairs == 0 || pairs > s->last_pairs) return set_err(c, RBF_ERR_INVALID, "only %u pairs were encoded", s->last_pairs);
    CK(c, cudaSetDevice(c->device));
    const uint64_t pb = (uint64_t)s->C * s->S;
    uint64_t total = 0;
    for (uint32_t i = 0; i < pairs; i++) { offsets_out[i] = total; total += s->last_infos[i].ones * pb; }
    offsets_out[pairs] = total;
    if (!values_out) return RBF_OK;                      // size query
    if (capacity < total) return set_err(c, RBF_ERR_INVALID, "values buffer too small: %llu < %llu", (unsigned long long)capacity, (unsigned long long)total);
    void *d_vals, *d_jobs, *d_gcnt;
    int rc;
    if ((rc = scratch_get(c, 8, (size_t)total + 256, &d_vals)) || (rc = scratch_get(c, 9, sizeof(GatherJob) * pairs, &d_jobs)) ||
        (rc = scratch_get(c, 13, 4 * (size_t)pairs * gather_chunks((uint32_t)s->npix) + 64, &d_gcnt)))
        return rc;
    std::vector<GatherJob> jobs(pairs);
    for (uint32_t i = 0; i < pairs; i++) {
        jobs[i].mask = s->d_mask + (size_t)i * s->mask_stride_w;
        jobs[i].frame = s->h_pairs[i].curr;
        jobs[i].values = (uint8_t*)d_vals + offsets_out[i];
        jobs[i].out_frame = nullptr;
        jobs[i].npix = (uint32_t)s->npix;
        jobs[i].pix_bytes = (uint32_t)pb;
    }
    CK(c, cudaMemcpyAsync(d_jobs, jobs.data(), sizeof(GatherJob) * pairs, cudaMemcpyHostToDevice, c->st));
    LAUNCH(c, launch_gather_scatter((const GatherJob*)d_jobs, (int)pairs, 0, (uint32_t)s->npix, (uint32_t)pb, (uint32_t*)d_gcnt, nullptr, c->st));
    c->launches++;
    if (total) { CK(c, cudaMemcpyAsync(values_out, d_vals, (size_t)total, cudaMemcpyDeviceToHost, c->st)); c->d2h += (int64_t)total; }
    CK(c, cudaStreamSynchronize(c->st));
    return RBF_OK;
}

extern "C" int rbf_stream_apply_diff(rbf_stream* s, uint32_t base_frame, uint32_t out_frame, const uint8_t* mask_packed_little,
                                     const uint8_t* values, uint64_t values_bytes, uint64_t* applied_pixels) {
    if (!s || !mask_packed_little || (!values && values_bytes)) return set_err(s ? s->c : nullptr, RBF_ERR_INVALID, "rbf_stream_apply_diff: NULL");
    rbf_ctx* c = s->c;
    if (base_frame >= s->max_frames || out_frame >= s->max_frames) return set_err(c, RBF_ERR_INVALID, "frame index outside the store");
    if (s->frame_bytes == 0) return set_err(c, RBF_ERR_STATE, "decode-only image stream (0 channels): it has no image store");
    CK(c, cudaSetDevice(c->device));
    const uint64_t pb = (uint64_t)s->C * s->S;
    const size_t mbytes = (size_t)((s->npix + 7) / 8), mwords = s->mask_stride_w;
    void *d_mask, *d_vals, *d_job, *d_gcnt;
    int rc;
    if ((rc = scratch_get(c, 10, mwords * 4, &d_mask)) || (rc = scratch_get(c, 8, (size_t)values_bytes + 256, &d_vals)) ||
        (rc = scratch_get(c, 9, sizeof(GatherJob) + 64, &d_job)) || (rc = scratch_get(c, 13, 4 * (size_t)gather_chunks((uint32_t)s->npix) + 64, &d_gcnt)))
        return rc;
    CK(c, cudaMemsetAsync(d_mask, 0, mwords * 4, c->st));
    CK(c, cudaMemcpyAsync(d_mask, mask_packed_little, mbytes, cudaMemcpyHostToDevice, c->st)); c->h2d += (int64_t)mbytes;
    if (values_bytes) { CK(c, cudaMemcpyAsync(d_vals, values, (size_t)values_bytes, cudaMemcpyHostToDevice, c->st)); c->h2d += (int64_t)values_bytes; }
    uint8_t* dst = s->d_frames + (size_t)out_frame * s->frame_stride;
    if (out_frame != base_frame)
        CK(c, cudaMemcpyAsync(dst, s->d_frames + (size_t)base_frame * s->frame_stride, s->frame_bytes, cudaMemcpyDeviceToDevice, c->st));
    GatherJob J;
    J.mask = (const uint32_t*)d_mask; J.frame = nullptr; J.values = (uint8_t*)d_vals; J.out_frame = dst;
    J.npix = (uint32_t)s->npix; J.pix_bytes = (uint32_t)pb;
    uint32_t* d_cnt = (uint32_t*)((uint8_t*)d_job + sizeof(GatherJob));
    // the reference applies the diff only when the value count matches the mask (ivc:882): count first
    CK(c, cudaMemsetAsync(d_cnt, 0, 4, c->st));
    LAUNCH(c, launch_popcount((const uint32_t*)d_mask, (s->npix + 31) / 32, d_cnt, c->st));
    uint32_t h_cnt = 0;
    CK(c, cudaMemcpyAsync(&h_cnt, d_cnt, 4, cudaMemcpyDeviceToHost, c->st));
    CK(c, cudaStreamSynchronize(c->st));
    if (applied_pixels) *applied_pixels = 0;
    if ((uint64_t)h_cnt * pb != values_bytes) return RBF_OK;       // ivc:882: mismatch -> the base frame is returned unchanged
    CK(c, cudaMemcpyAsync(d_job, &J, sizeof J, cudaMemcpyHostToDevice, c->st));
    LAUNCH(c, launch_gather_scatter((const GatherJob*)d_job, 1, 1, (uint32_t)s->npix, (uint32_t)pb, (uint32_t*)d_gcnt, nullptr, c->st));
    c->launches++;
    CK(c, cudaStreamSynchronize(c->st));
    if (applied_pixels) *applied_pixels = h_cnt;
    return RBF_OK;
}

extern "C" int rbf_stream_download(rbf_stream* s, uint32_t frame, void* host_out) {
    if (!s || !host_out || frame >= s->max_frames) return set_err(s ? s->c : nullptr, RBF_ERR_INVALID, "rbf_stream_download: bad argument");
    rbf_ctx* c = s->c;
    CK(c, cudaMemcpyAsync(host_out, s->d_frames + (size_t)frame * s->frame_stride, s->frame_bytes, cudaMemcpyDeviceToHost, c->st));
    c->d2h += (int64_t)s->frame_bytes;
    CK(c, cudaStreamSynchronize(c->st));
    return RBF_OK;
}


// ------------------------------------------------------------------------------------------
// N3: cv2.medianBlur(frame, 5) of VideoFrameCompressor._estimate_noise_level (ivc:738)
// ------------------------------------------------------------------------------------------
extern "C" int rbf_median_blur5(rbf_ctx* c, const void* plane_in, uint32_t H, uint32_t W, uint32_t sample_bytes, void* plane_out) {
    if (!c || !plane_in || !plane_out) return set_err(c, RBF_ERR_INVALID, "rbf_median_blur5: NULL");
    if (!(sample_bytes == 1 || sample_bytes == 2) || H == 0 || W == 0) return set_err(c, RBF_ERR_INVALID, "rbf_median_blur5: bad shape");
    CK(c, cudaSetDevice(c->device));
    const size_t bytes = (size_t)H * W * sample_bytes;
    void *d_in, *d_out;
    int rc;
    if ((rc = scratch_get(c, 11, bytes, &d_in)) || (rc = scratch_get(c, 12, bytes, &d_out))) return rc;
    CK(c, cudaMemcpyAsync(d_in, plane_in, bytes, cudaMemcpyHostToDevice, c->st)); c->h2d += (int64_t)bytes;
    LAUNCH(c, launch_median5(d_in, 1, H, W, (int)sample_bytes, d_out, c->st));
    CK(c, cudaMemcpyAsync(plane_out, d_out, bytes, cudaMemcpyDeviceToHost, c->st)); c->d2h += (int64_t)bytes;
    CK(c, cudaStreamSynchronize(c->st));
    return RBF_OK;
}

extern "C" int rbf_stream_median5(rbf_stream* s, uint32_t frame, void* plane_out) {
    if (!s || !plane_out || frame >= s->max_frames) return set_err(s ? s->c : nullptr, RBF_ERR_INVALID, "rbf_stream_median5: bad argument");
    rbf_ctx* c = s->c;
    if (s->frame_bytes == 0) return set_err(c, RBF_ERR_STATE, "decode-only image stream (0 channels): it has no image store");
    CK(c, cudaSetDevice(c->device));
    const size_t bytes = (size_t)s->npix * s->S;
    void* d_out;
    int rc;
    if ((rc = scratch_get(c, 12, bytes, &d_out))) return rc;
    LAUNCH(c, launch_median5(s->d_frames + (size_t)frame * s->frame_stride, s->C, s->H, s->W, (int)s->S, d_out, c->st));
    CK(c, cudaMemcpyAsync(plane_out, d_out, bytes, cudaMemcpyDeviceToHost, c->st)); c->d2h += (int64_t)bytes;
    CK(c, cudaStreamSynchronize(c->st));
    return RBF_OK;
}

// ------------------------------------------------------------------------------------------
// NCCL (dlopen'ed so that single-GPU use needs no NCCL at all)
// ------------------------------------------------------------------------------------------
typedef struct { char internal[128]; } nccl_uid;
typedef int (*fn_GetUniqueId)(nccl_uid*);
typedef int (*fn_CommInitRank)(void**, int, nccl_uid, int);
typedef int (*fn_AllGather)(const void*, void*, size_t, int, void*, cudaStream_t);
typedef int (*fn_CommDestroy)(void*);
typedef const char* (*fn_GetErrorString)(int);

static void* g_nccl = nullptr;
static void* nccl_handle() {
    if (!g_nccl) {
        g_nccl = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!g_nccl) g_nccl = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    }
    return g_nccl;
}
extern "C" int rbf_nccl_unique_id(uint8_t id_out[128]) {
    void* h = nccl_handle();
    if (!h) return set_err(nullptr, RBF_ERR_NCCL, "cannot dlopen libnccl.so.2: %s", dlerror());
    fn_GetUniqueId f = (fn_GetUniqueId)dlsym(h, "ncclGetUniqueId");
    if (!f) return set_err(nullptr, RBF_ERR_NCCL, "ncclGetUniqueId not found");
    nccl_uid u;
    int r = f(&u);
    if (r) return set_err(nullptr, RBF_ERR_NCCL, "ncclGetUniqueId failed: %d", r);
    memcpy(id_out, u.internal, 128);
    return RBF_OK;
}
extern "C" int rbf_nccl_init(rbf_ctx* c, const uint8_t id[128], int rank, int nranks) {
    if (!c || !id) return set_err(c, RBF_ERR_INVALID, "rbf_nccl_init: NULL");
    void* h = nccl_handle();
    if (!h) return set_err(c, RBF_ERR_NCCL, "cannot dlopen libnccl.so.2: %s", dlerror());
    fn_CommInitRank f = (fn_CommInitRank)dlsym(h, "ncclCommInitRank");
    if (!f) return set_err(c, RBF_ERR_NCCL, "ncclCommInitRank not found");
    CK(c, cudaSetDevice(c->device));
    nccl_uid u;
    memcpy(u.internal, id, 128);
    void* comm = nullptr;
    int r = f(&comm, nranks, u, rank);
    if (r) {
        fn_GetErrorString es = (fn_GetErrorString)dlsym(h, "ncclGetErrorString");
        return set_err(c, RBF_ERR_NCCL, "ncclCommInitRank failed: %s", es ? es(r) : "?");
    }
    c->nccl_lib = h; c->nccl_comm = comm; c->rank = rank; c->nranks = nranks;
    return RBF_OK;
}
static int nccl_allgather_on(rbf_ctx* c, const void* d_send, void* d_recv, uint64_t bytes_per_rank, cudaStream_t st) {
    if (!c || !c->nccl_comm) return set_err(c, RBF_ERR_STATE, "rbf_nccl_allgather: communicator not initialised");
    fn_AllGather f = (fn_AllGather)dlsym(c->nccl_lib, "ncclAllGather");
    if (!f) return set_err(c, RBF_ERR_NCCL, "ncclAllGather not found");
    int r = f(d_send, d_recv, (size_t)bytes_per_rank, /*ncclUint8*/ 1, c->nccl_comm, st);
    if (r) {
        fn_GetErrorString es = (fn_GetErrorString)dlsym(c->nccl_lib, "ncclGetErrorString");
        return set_err(c, RBF_ERR_NCCL, "ncclAllGather failed: %s", es ? es(r) : "?");
    }
    c->launches++;
    return RBF_OK;
}
extern "C" int rbf_nccl_allgather(rbf_ctx* c, const void* d_send, void* d_recv, uint64_t bytes_per_rank) {
    return nccl_allgather_on(c, d_send, d_recv, bytes_per_rank, c ? c->st : nullptr);
}
// Packs the bit arrays of the last encode into fixed-size slots and all-gathers them on the context's communication
// stream: the call returns once the work is enqueued, the next rbf_stream_encode overlaps it (it only waits for the
// packing before it clears the bit arrays).  d_recv is complete after rbf_sync, rbf_timer_stop_ms or rbf_memcpy_d2h.
static int ensure_comm_stream(rbf_ctx* c) {
    if (!c->st_comm) {
        CK(c, cudaStreamCreateWithFlags(&c->st_comm, cudaStreamNonBlocking));
        CK(c, cudaEventCreateWithFlags(&c->ev_enc, cudaEventDisableTiming));
        CK(c, cudaEventCreateWithFlags(&c->ev_pack, cudaEventDisableTiming));
        CK(c, cudaEventCreateWithFlags(&c->ev_comm, cudaEventDisableTiming));
    }
    return RBF_OK;
}
extern "C" int rbf_stream_allgather_bitmaps(rbf_stream* s, uint32_t pairs, uint64_t slot_bytes, void* d_send, void* d_recv) {
    if (!s || !d_recv) return set_err(s ? s->c : nullptr, RBF_ERR_INVALID, "rbf_stream_allgather_bitmaps: NULL");
    rbf_ctx* c = s->c;
    const size_t stride = s->mask_stride_w * 4;
    if (slot_bytes == 0 || slot_bytes > stride || (slot_bytes & 15) || pairs == 0 || pairs > s->max_pairs)
        return set_err(c, RBF_ERR_INVALID, "bad slot/pairs");
    if (c->peer_nranks > 0) {
        // peer-memory exchange: one kernel stores this rank's slots into every rank's receive buffer over NVLink
        if (d_recv != (void*)c->peer_recv[c->peer_rank]) return set_err(c, RBF_ERR_INVALID, "d_recv is not the buffer given to rbf_peer_gather_init");
        if (int r = ensure_comm_stream(c)) return r;
        CK(c, cudaEventRecord(c->ev_enc, c->st));                   // the encode that produced the bit arrays
        CK(c, cudaStreamWaitEvent(c->st_comm, c->ev_enc, 0));
        // every rank has signalled the previous exchange => it has consumed the one before it: that half is free everywhere
        if (c->peer_seq > 0)
            LAUNCH(c, launch_peer_wait(c->peer_flags[c->peer_rank], c->peer_nranks, c->peer_seq, kPeerTimeoutCycles, c->peer_err, c->st_comm));
        c->peer_seq++;
        const uint32_t slot_w = (uint32_t)(slot_bytes / 4);
        const size_t half_w = (size_t)c->peer_nranks * pairs * slot_w;
        const size_t dst_off_w = (size_t)(c->peer_seq & 1u) * half_w + (size_t)c->peer_rank * pairs * slot_w;
        LAUNCH(c, launch_push_slots(s->d_bits, s->mask_stride_w, slot_w, pairs, c->peer_recv, c->peer_flags, c->peer_nranks, c->peer_rank,
                                    dst_off_w, c->peer_seq, c->sm_count, c->st_comm));
        c->launches++;                                              // push + signal
        CK(c, cudaEventRecord(c->ev_pack, c->st_comm));
        CK(c, cudaEventRecord(c->ev_comm, c->st_comm));
        c->pack_pending = c->comm_pending = c->peer_wait_pending = true;
        return RBF_OK;
    }
    if (!d_send) return set_err(c, RBF_ERR_INVALID, "rbf_stream_allgather_bitmaps: d_send is NULL");
    if (!c->nccl_comm) return set_err(c, RBF_ERR_STATE, "rbf_stream_allgather_bitmaps: communicator not initialised");
    if (int r = ensure_comm_stream(c)) return r;
    CK(c, cudaEventRecord(c->ev_enc, c->st));                       // the encode that produced the bit arrays
    CK(c, cudaStreamWaitEvent(c->st_comm, c->ev_enc, 0));
    CK(c, cudaMemcpy2DAsync(d_send, slot_bytes, s->d_bits, stride, slot_bytes, pairs, cudaMemcpyDeviceToDevice, c->st_comm));
    CK(c, cudaEventRecord(c->ev_pack, c->st_comm));
    c->pack_pending = true;
    if (int r = nccl_allgather_on(c, d_send, d_recv, slot_bytes * pairs, c->st_comm)) return r;
    CK(c, cudaEventRecord(c->ev_comm, c->st_comm));
    c->comm_pending = true;
    return RBF_OK;
}

// ------------------------------------------------------------------------------------------
// exchange over NVLink peer memory: CUDA IPC handles travel over the caller's channel (like the NCCL id)
// ------------------------------------------------------------------------------------------
extern "C" int rbf_peer_export(rbf_ctx* c, const void* d_ptr, uint8_t handle_out[64]) {
    if (!c || !d_ptr || !handle_out) return set_err(c, RBF_ERR_INVALID, "rbf_peer_export: NULL");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    CK(c, cudaSetDevice(c->device));
    cudaIpcMemHandle_t h;
    CK(c, cudaIpcGetMemHandle(&h, const_cast<void*>(d_ptr)));
    memcpy(handle_out, &h, 64);
    return RBF_OK;
}
extern "C" int rbf_peer_open(rbf_ctx* c, const uint8_t handle[64], void** d_out) {
    if (!c || !handle || !d_out) return set_err(c, RBF_ERR_INVALID, "rbf_peer_open: NULL");
    CK(c, cudaSetDevice(c->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    CK(c, cudaIpcOpenMemHandle(d_out, h, cudaIpcMemLazyEnablePeerAccess));
    return RBF_OK;
}
extern "C" int rbf_peer_close(rbf_ctx* c, void* d_ptr) {
    if (!c) return RBF_ERR_INVALID;
    if (d_ptr) CK(c, cudaIpcCloseMemHandle(d_ptr));
    return RBF_OK;
}
extern "C" int rbf_peer_gather_init(rbf_ctx* c, int rank, int nranks, void* const* recv_ptrs, void* const* flag_ptrs) {
    if (!c || !recv_ptrs || !flag_ptrs) return set_err(c, RBF_ERR_INVALID, "rbf_peer_gather_init: NULL");
    if (nranks < 1 || nranks > 16 || rank < 0 || rank >= nranks) return set_err(c, RBF_ERR_INVALID, "rank %d of %d", rank, nranks);
    for (int r = 0; r < nranks; r++)
        if (!recv_ptrs[r] || !flag_ptrs[r]) return set_err(c, RBF_ERR_INVALID, "rbf_peer_gather_init: pointer of rank %d is NULL", r);
    CK(c, cudaSetDevice(c->device));
    if (!c->peer_err) {
        CK(c, cudaHostAlloc((void**)&c->peer_err, 64, cudaHostAllocMapped));
        *c->peer_err = 0;
    }
    for (int r = 0; r < 16; r++) {
        c->peer_recv[r] = r < nranks ? (uint32_t*)recv_ptrs[r] : nullptr;
        c->peer_flags[r] = r < nranks ? (uint32_t*)flag_ptrs[r] : nullptr;
    }
    c->peer_rank = rank; c->peer_nranks = nranks; c->peer_seq = 0; c->peer_wait_pending = false;
    return RBF_OK;
}
extern "C" int rbf_peer_gather_half(rbf_ctx* c, uint32_t* half_out) {
    if (!c || !half_out) return RBF_ERR_INVALID;
    if (c->peer_nranks == 0 || c->peer_seq == 0) return set_err(c, RBF_ERR_STATE, "no peer exchange has run");
    *half_out = c->peer_seq & 1u;
    return RBF_OK;
}
extern "C" int rbf_peer_gather_shutdown(rbf_ctx* c) {
    if (!c) return RBF_ERR_INVALID;
    if (c->st_comm) CK(c, cudaStreamSynchronize(c->st_comm));
    if (c->st) CK(c, cudaStreamSynchronize(c->st));
    c->peer_nranks = 0; c->peer_seq = 0; c->peer_wait_pending = false; c->comm_pending = c->pack_pending = false;
    return RBF_OK;
}
extern "C" int rbf_nccl_destroy(rbf_ctx* c) {
    if (!c) return RBF_ERR_INVALID;
    if (c->st_comm) cudaStreamSynchronize(c->st_comm);
    c->comm_pending = c->pack_pending = false;
    if (c->nccl_comm && c->nccl_lib) {
        fn_CommDestroy f = (fn_CommDestroy)dlsym(c->nccl_lib, "ncclCommDestroy");
        if (f) f(c->nccl_comm);
    }
    c->nccl_comm = nullptr;
    return RBF_OK;
}
