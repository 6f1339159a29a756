// rbf_k1_threshold.cuh -- K1: |Y_prev - Y_curr| > thr -> packed mask + counts (ivc:788-808, ivc:211).  Included by rbf_kernels.cu inside namespace rbf.
#pragma once

// ------------------------------------------------------------------------------------------
// K1: threshold + popcount.  One thread = 32 consecutive pixels = one mask word; the pixel
// bytes are read with 128-bit streaming loads (2*PB of them per frame, all issued up front).
// PB = bytes per pixel (channels * sample bytes), S = sample bytes; Y is the first sample.
// ------------------------------------------------------------------------------------------
template <int PB, int S>
__device__ __forceinline__ int absdiff_sample(uint32_t a, uint32_t b) {
    if (S == 1) {
        int d = (int)a - (int)b;
        return d < 0 ? -d : d;
    } else {                                           // numpy int16 wrap-around (ivc:801)
        int16_t x = (int16_t)(uint16_t)a, y = (int16_t)(uint16_t)b;
        int16_t d = (int16_t)(x - y);
        int16_t ad = (int16_t)(d < 0 ? -d : d);      // abs(-32768) stays -32768
        return (int)ad;
    }
}

// cv2.cvtColor(frame, cv2.COLOR_BGR2GRAY) of the reference's non-YUV colour branch (ivc:792-795): OpenCV's 15-bit
// fixed point, identical for 8- and 16-bit samples (checked against cv2 4.13 in tests/golden/make_golden.py)
__device__ __forceinline__ uint32_t bgr2gray_fixed(uint32_t b, uint32_t g, uint32_t r) {
    return (b * 3735u + g * 19235u + r * 9798u + 16384u) >> 15;
}

// 256-bit streaming load: one 32 B sector per thread per instruction (LDG.E.256 on sm_100a)
__device__ __forceinline__ void ldg256_stream(const void* p, uint32_t* r) {
    asm volatile("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "l"(p));
}

// Four consecutive 8-bit YUV444 pixels = three 32-bit words per frame.  Byte-SIMD:
//   nm = 4-bit mask of  |Ya - Yb| > thr  (VABSDIFF4 + per-byte compare),  nd = 4-bit "any byte differs".
// gt_or / gt_and fold the out-of-range thresholds (thr < 0: always, thr > 254: never) into the compare.
__device__ __forceinline__ void yuv8_group4(uint32_t a0, uint32_t a1, uint32_t a2, uint32_t b0, uint32_t b1, uint32_t b2,
                                            uint32_t thr4, uint32_t gt_or, uint32_t gt_and, uint32_t& nm, uint32_t& nd) {
    const uint32_t ya = __byte_perm(__byte_perm(a0, a1, 0x0630), a2, 0x5210);   // Y bytes of pixels 0..3
    const uint32_t yb = __byte_perm(__byte_perm(b0, b1, 0x0630), b2, 0x5210);
    const uint32_t gt = (__vcmpgtu4(__vabsdiffu4(ya, yb), thr4) & gt_and) | gt_or;
    nm = ((gt & 0x01010101u) * 0x01020408u) >> 24;
    const uint32_t x0 = a0 ^ b0, x1 = a1 ^ b1, x2 = a2 ^ b2;
    const uint32_t f0 = x0 & 0x00ffffffu, f1 = __funnelshift_r(x0, x1, 24) & 0x00ffffffu,
                   f2 = __funnelshift_r(x1, x2, 16) & 0x00ffffffu, f3 = x2 >> 8;
    nd = min(f0, 1u) | (min(f1, 1u) << 1) | (min(f2, 1u) << 2) | (min(f3, 1u) << 3);
}

template <int PB, int S, bool GRAY = false>
__global__ void __launch_bounds__(256) k_threshold(const PairJob* __restrict__ pairs, uint32_t npix, int thr, int any_mode,
                                                   uint32_t* __restrict__ ones, uint32_t* __restrict__ resid) {
    static_assert(!GRAY || PB == 3 * S, "BGR->gray needs three samples per pixel");
    const PairJob pj = pairs[blockIdx.y];
    const uint32_t nwords = (npix + 31u) >> 5;
    uint32_t cnt_ones = 0, cnt_res = 0;
    const uint32_t thr4 = (uint32_t)(thr < 0 ? 0 : (thr > 254 ? 254 : thr)) * 0x01010101u;
    const uint32_t gt_or = thr < 0 ? 0xffffffffu : 0u, gt_and = thr > 254 ? 0u : 0xffffffffu;
    const uint32_t any_mask = any_mode ? 0xfu : 0u;
    for (uint32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < nwords; w += gridDim.x * blockDim.x) {
        const uint32_t px0 = w << 5;
        uint32_t m = 0, r = 0;
        if (px0 + 32u <= npix) {
            if (PB == 3 && S == 1 && !GRAY) {
                uint32_t A[24], B[24];
                const uint8_t* pa = pj.prev + (size_t)px0 * 3;
                const uint8_t* pb = pj.curr + (size_t)px0 * 3;
#pragma unroll
                for (int j = 0; j < 3; j++) ldg256_stream(pa + 32 * j, A + 8 * j);
#pragma unroll
                for (int j = 0; j < 3; j++) ldg256_stream(pb + 32 * j, B + 8 * j);
#pragma unroll
                for (int g = 0; g < 8; g++) {
                    uint32_t nm, nd;
                    yuv8_group4(A[3 * g], A[3 * g + 1], A[3 * g + 2], B[3 * g], B[3 * g + 1], B[3 * g + 2], thr4, gt_or, gt_and, nm, nd);
                    nm |= nd & any_mask;
                    m |= nm << (4 * g);
                    r |= (nd & ~nm) << (4 * g);
                }
            } else {
                constexpr int NV = PB;                     // 256-bit loads per 32 pixels
                constexpr int HV = (NV > 3) ? NV / 2 : NV; // at most 3 in flight per frame
                constexpr int HALVES = NV / HV;
                constexpr int PXH = 32 / HALVES;
#pragma unroll
                for (int hf = 0; hf < HALVES; hf++) {
                    uint32_t A[8 * HV], B[8 * HV];
                    const uint8_t* pa = pj.prev + (size_t)(px0 + hf * PXH) * PB;
                    const uint8_t* pb = pj.curr + (size_t)(px0 + hf * PXH) * PB;
#pragma unroll
                    for (int j = 0; j < HV; j++) ldg256_stream(pa + 32 * j, A + 8 * j);
#pragma unroll
                    for (int j = 0; j < HV; j++) ldg256_stream(pb + 32 * j, B + 8 * j);
#pragma unroll
                    for (int k = 0; k < PXH; k++) {
                        const int o = k * PB;              // byte offset of the pixel (compile-time)
                        const uint32_t smask = (S == 1) ? 0xffu : 0xffffu;
                        uint32_t ya = (A[o >> 2] >> (8 * (o & 3))) & smask;
                        uint32_t yb = (B[o >> 2] >> (8 * (o & 3))) & smask;
                        if (GRAY) {                        // samples 1 and 2 of the pixel (compile-time offsets; S == 2 samples are 2-aligned)
                            const int p1 = o + S, p2 = o + 2 * S;
                            const uint32_t a1 = (A[p1 >> 2] >> (8 * (p1 & 3))) & smask, a2 = (A[p2 >> 2] >> (8 * (p2 & 3))) & smask;
                            const uint32_t b1 = (B[p1 >> 2] >> (8 * (p1 & 3))) & smask, b2 = (B[p2 >> 2] >> (8 * (p2 & 3))) & smask;
                            ya = bgr2gray_fixed(ya, a1, a2);
                            yb = bgr2gray_fixed(yb, b1, b2);
                        }
                        uint32_t anyd = 0;                 // any byte of the pixel differs
#pragma unroll
                        for (int q = 0; q < PB; q++) {
                            const int oq = o + q;
                            anyd |= ((A[oq >> 2] ^ B[oq >> 2]) >> (8 * (oq & 3))) & 0xffu;
                        }
                        const uint32_t bit = ((absdiff_sample<PB, S>(ya, yb) > thr) || (any_mode && anyd != 0u)) ? 1u : 0u;
                        m |= bit << (hf * PXH + k);
                        r |= ((anyd != 0u && bit == 0u) ? 1u : 0u) << (hf * PXH + k);
                    }
                }
            }
        } else {                                        // ragged last word: scalar loads
            for (uint32_t k = 0; k < 32u && px0 + k < npix; k++) {
                const uint8_t* a = pj.prev + (size_t)(px0 + k) * PB;
                const uint8_t* b = pj.curr + (size_t)(px0 + k) * PB;
                uint32_t ya = a[0], yb = b[0];
                if (S == 2) { ya |= (uint32_t)a[1] << 8; yb |= (uint32_t)b[1] << 8; }
                if (GRAY) {
                    uint32_t a1 = a[S], a2 = a[2 * S], b1 = b[S], b2 = b[2 * S];
                    if (S == 2) { a1 |= (uint32_t)a[3] << 8; a2 |= (uint32_t)a[5] << 8; b1 |= (uint32_t)b[3] << 8; b2 |= (uint32_t)b[5] << 8; }
                    ya = bgr2gray_fixed(ya, a1, a2);
                    yb = bgr2gray_fixed(yb, b1, b2);
                }
                uint32_t anyd = 0;
                for (int q = 0; q < PB; q++) anyd |= (uint32_t)(a[q] ^ b[q]);
                const uint32_t bit = ((absdiff_sample<PB, S>(ya, yb) > thr) || (any_mode && anyd != 0u)) ? 1u : 0u;
                m |= bit << k;
                r |= ((anyd != 0u && bit == 0u) ? 1u : 0u) << k;
            }
        }
        pj.mask[w] = m;
        cnt_ones += __popc(m);
        cnt_res += __popc(r);
    }
    // block reduction -> one atomic per block
    __shared__ uint32_t s_o[8], s_r[8];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        cnt_ones += __shfl_xor_sync(0xffffffffu, cnt_ones, d);
        cnt_res += __shfl_xor_sync(0xffffffffu, cnt_res, d);
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { s_o[warp] = cnt_ones; s_r[warp] = cnt_res; }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t to = 0, tr = 0;
        for (int i = 0; i < (int)(blockDim.x >> 5); i++) { to += s_o[i]; tr += s_r[i]; }
        if (to) atomicAdd(ones + blockIdx.y, to);
        if (tr) atomicAdd(resid + blockIdx.y, tr);
    }
}

// ------------------------------------------------------------------------------------------
// K1 (TMA variant): persistent CTAs, 4-stage mbarrier ring, one elected thread issues
// cp.async.bulk copies of a 2 x 12 KB tile (prev, curr); for 8-bit YUV444 each lane reads
// four pixels (three words, bank-conflict free) and runs the same byte-SIMD as above; the
// per-lane nibbles are OR-reduced over 8-lane groups (REDUX) into mask words.
// ------------------------------------------------------------------------------------------
constexpr int TMA_STAGES = 4;
constexpr int TMA_TILE_BYTES = 12288;                  // per frame per stage (4096 px at 3 B/px)
constexpr int TMA_THREADS = 256;

template <int PB, int S>
__global__ void __launch_bounds__(TMA_THREADS) k_threshold_tma(const PairJob* __restrict__ pairs, int F, uint32_t npix,
                                                               int thr, int any_mode, uint32_t* __restrict__ ones,
                                                               uint32_t* __restrict__ resid) {
    constexpr uint32_t TP = TMA_TILE_BYTES / PB;       // pixels per tile (multiple of 32*8)
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ __align__(8) uint64_t full[TMA_STAGES];
    uint8_t* bufA = smem;                               // [STAGES][TILE]
    uint8_t* bufB = smem + TMA_STAGES * TMA_TILE_BYTES;
    const uint32_t tiles_per_frame = npix / TP;         // full tiles only (bulk copies need 16 B multiples)
    const uint64_t total = (uint64_t)tiles_per_frame * (uint64_t)F;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int NWARP = TMA_THREADS / 32;
    constexpr uint32_t WPW = TP / 32 / NWARP;           // mask words per warp per tile
    const uint32_t thr4 = (uint32_t)(thr < 0 ? 0 : (thr > 254 ? 254 : thr)) * 0x01010101u;
    const uint32_t gt_or = thr < 0 ? 0xffffffffu : 0u, gt_and = thr > 254 ? 0u : 0xffffffffu;
    const uint32_t any_mask = any_mode ? 0xfu : 0u;

    if (threadIdx.x == 0) {
        for (int s = 0; s < TMA_STAGES; s++) mbar_init(&full[s], 1);
        fence_mbar_init();
    }
    __syncthreads();

    auto issue = [&](uint64_t t, int slot) {
        const uint32_t f = (uint32_t)(t / tiles_per_frame), ti = (uint32_t)(t % tiles_per_frame);
        const PairJob pj = pairs[f];
        mbar_expect_tx(&full[slot], 2 * TMA_TILE_BYTES);
        bulk_g2s(bufA + slot * TMA_TILE_BYTES, pj.prev + (size_t)ti * TMA_TILE_BYTES, TMA_TILE_BYTES, &full[slot]);
        bulk_g2s(bufB + slot * TMA_TILE_BYTES, pj.curr + (size_t)ti * TMA_TILE_BYTES, TMA_TILE_BYTES, &full[slot]);
    };

    // prologue
    uint64_t t0 = blockIdx.x;
    if (threadIdx.x == 0) {
        for (int s = 0; s < TMA_STAGES - 1; s++) {
            uint64_t t = t0 + (uint64_t)s * gridDim.x;
            if (t < total) issue(t, s);
        }
    }
    uint32_t it = 0, acc_o = 0, acc_r = 0, acc_f = 0xffffffffu;     // per-thread counts of the current frame
    auto flush_counts = [&]() {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            acc_o += __shfl_xor_sync(0xffffffffu, acc_o, d);
            acc_r += __shfl_xor_sync(0xffffffffu, acc_r, d);
        }
        if (lane == 0 && acc_f != 0xffffffffu) {
            if (acc_o) atomicAdd(ones + acc_f, acc_o);
            if (acc_r) atomicAdd(resid + acc_f, acc_r);
        }
        acc_o = 0; acc_r = 0;
    };
    for (uint64_t t = t0; t < total; t += gridDim.x, it++) {
        const int slot = it % TMA_STAGES;
        const uint32_t parity = (it / TMA_STAGES) & 1u;
        if (threadIdx.x == 0) {                         // refill the slot freed by the previous iteration
            uint64_t tn = t + (uint64_t)(TMA_STAGES - 1) * gridDim.x;
            if (tn < total) { fence_proxy_async(); issue(tn, (it + TMA_STAGES - 1) % TMA_STAGES); }
        }
        const uint32_t f = (uint32_t)(t / tiles_per_frame), ti = (uint32_t)(t % tiles_per_frame);
        if (f != acc_f) { flush_counts(); acc_f = f; }  // warp-uniform
        mbar_wait(&full[slot], parity);
        const uint8_t* a = bufA + slot * TMA_TILE_BYTES;
        const uint8_t* b = bufB + slot * TMA_TILE_BYTES;
        uint32_t* mask_out = pairs[f].mask + (size_t)ti * (TP / 32) + warp * WPW;
        if (PB == 3 && S == 1) {
            const uint32_t* a32 = reinterpret_cast<const uint32_t*>(a) + (size_t)warp * WPW * 24;   // 32 px = 24 words
            const uint32_t* b32 = reinterpret_cast<const uint32_t*>(b) + (size_t)warp * WPW * 24;
#pragma unroll 2
            for (uint32_t k = 0; k < WPW / 4; k++) {      // 128 pixels (4 mask words) per iteration
                const uint32_t o = (k * 32u + lane) * 3u;
                uint32_t nm, nd;
                yuv8_group4(a32[o], a32[o + 1], a32[o + 2], b32[o], b32[o + 1], b32[o + 2], thr4, gt_or, gt_and, nm, nd);
                nm |= nd & any_mask;
                const uint32_t nr = nd & ~nm;
                const uint32_t grp = 0xffu << (lane & 24);
                const uint32_t wm = __reduce_or_sync(grp, nm << (4 * (lane & 7)));
                const uint32_t wr = __reduce_or_sync(grp, nr << (4 * (lane & 7)));
                if ((lane & 7) == 0) { mask_out[k * 4 + (lane >> 3)] = wm; acc_o += __popc(wm); acc_r += __popc(wr); }
            }
        } else {
            uint32_t myword = 0;
#pragma unroll 4
            for (uint32_t k = 0; k < WPW; k++) {
                const uint32_t px = (warp * WPW + k) * 32u + lane;
                const uint8_t* pa = a + px * PB;
                const uint8_t* pb = b + px * PB;
                uint32_t ya, yb, anyd = 0;
                if (S == 1) { ya = pa[0]; yb = pb[0]; }
                else { ya = *reinterpret_cast<const uint16_t*>(pa); yb = *reinterpret_cast<const uint16_t*>(pb); }
#pragma unroll
                for (int q = 0; q < PB; q += S) {
                    if (S == 1) anyd |= (uint32_t)(pa[q] ^ pb[q]);
                    else anyd |= (uint32_t)(*reinterpret_cast<const uint16_t*>(pa + q) ^ *reinterpret_cast<const uint16_t*>(pb + q));
                }
                const bool bit = (absdiff_sample<PB, S>(ya, yb) > thr) || (any_mode && anyd != 0u);
                const uint32_t bm = __ballot_sync(0xffffffffu, bit);
                const uint32_t br = __ballot_sync(0xffffffffu, (!bit) && anyd != 0u);
                if (lane == (int)k) myword = bm;
                if (lane == 0) { acc_o += __popc(bm); acc_r += __popc(br); }
            }
            if (lane < (int)WPW) mask_out[lane] = myword;
        }
        __syncthreads();                                // slot may be refilled next iteration
    }
    flush_counts();
}

// remainder of each frame after the last full TMA tile: same maths with guarded scalar loads
template <int PB, int S>
__global__ void __launch_bounds__(256) k_threshold_tail(const PairJob* __restrict__ pairs, uint32_t npix, uint32_t px_begin,
                                                        int thr, int any_mode, uint32_t* __restrict__ ones, uint32_t* __restrict__ resid) {
    const PairJob pj = pairs[blockIdx.y];
    const uint32_t w0 = px_begin >> 5, nwords = (npix + 31u) >> 5;
    for (uint32_t w = w0 + blockIdx.x * blockDim.x + threadIdx.x; w < nwords; w += gridDim.x * blockDim.x) {
        uint32_t m = 0, r = 0;
        for (uint32_t k = 0; k < 32u && (w << 5) + k < npix; k++) {
            const uint8_t* a = pj.prev + (size_t)((w << 5) + k) * PB;
            const uint8_t* b = pj.curr + (size_t)((w << 5) + k) * PB;
            uint32_t ya = a[0], yb = b[0];
            if (S == 2) { ya |= (uint32_t)a[1] << 8; yb |= (uint32_t)b[1] << 8; }
            uint32_t anyd = 0;
            for (int q = 0; q < PB; q++) anyd |= (uint32_t)(a[q] ^ b[q]);
            const uint32_t bit = ((absdiff_sample<PB, S>(ya, yb) > thr) || (any_mode && anyd != 0u)) ? 1u : 0u;
            m |= bit << k;
            r |= ((anyd != 0u && bit == 0u) ? 1u : 0u) << k;
        }
        pj.mask[w] = m;
        if (m) atomicAdd(ones + blockIdx.y, __popc(m));
        if (r) atomicAdd(resid + blockIdx.y, __popc(r));
    }
}

#include "rbf_k1_binarize.cuh"                         // the single-image K1 shares ldg256_stream
