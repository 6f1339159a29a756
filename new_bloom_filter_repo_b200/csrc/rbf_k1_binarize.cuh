// rbf_k1_binarize.cuh -- single-frame K1: BloomFilterCompressor._binarize_image (bloom_compress.py:67-87) -> packed mask +
// ones count (bc:253), and its launcher.  Included by rbf_k1_threshold.cuh (so by rbf_kernels.cu) inside namespace rbf.
#pragma once

// ------------------------------------------------------------------------------------------
// One thread = 32 consecutive pixels = one mask word; the image (PairJob::curr) is read with C*S 256-bit streaming loads per
// word, all issued up front.  Images are batched over blockIdx.y.
//
// bc:79-84 is  (np.mean(img, axis=2).astype(np.uint8) if C > 1 else img) > threshold.  For uint8 samples the uint8 cast of the
// mean is floor(sum / C) for every sum (checked exhaustively for C = 2, 3, 4 with numpy 2.3), so with t = floor(threshold)
// clamped to [-1, sample max]:   pixel is 1  <=>  sum of its C samples >= C * (t + 1)  =: need   (no division; C = 1 is v > t).
// The host folds the threshold into `need` (launch_binarize).
// ------------------------------------------------------------------------------------------
template <int C, int S>
__device__ __forceinline__ uint32_t binarize_pixel_sum(const uint32_t* R, int k) {   // k: pixel of the word (compile-time)
    if (S == 2) return (R[k >> 1] >> (16 * (k & 1))) & 0xffffu;                      // C == 1
    if (C == 4) return __dp4a(R[k], 0x01010101u, 0u);                                // RGBA: one pixel per word
    if (C == 2) return __dp4a(R[k >> 1], (k & 1) ? 0x01010000u : 0x00000101u, 0u);
    uint32_t sum = 0;                                                                 // C == 3 (C == 1 takes the SIMD path)
#pragma unroll
    for (int q = 0; q < C; q++) {
        const int o = C * k + q;
        sum += (R[o >> 2] >> (8 * (o & 3))) & 0xffu;
    }
    return sum;
}

template <int C, int S>
__global__ void __launch_bounds__(256) k_binarize(const PairJob* __restrict__ images, uint32_t npix, uint32_t need,
                                                  uint32_t* __restrict__ ones) {
    static_assert(S == 1 || C == 1, "multi-channel images have 8-bit samples");
    constexpr int NV = C * S;                             // 256-bit loads per 32 pixels
    const PairJob pj = images[blockIdx.y];
    const uint32_t nwords = (npix + 31u) >> 5;
    // 8-bit grey: byte-SIMD compare against need (need == 256, i.e. threshold >= 255, can never hold)
    const uint32_t need4 = (need > 255u ? 255u : need) * 0x01010101u, ge_and = need > 255u ? 0u : 0xffffffffu;
    uint32_t cnt = 0;
    for (uint32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < nwords; w += gridDim.x * blockDim.x) {
        const uint32_t px0 = w << 5;
        uint32_t m = 0;
        if (px0 + 32u <= npix) {
            uint32_t R[8 * NV];
            const uint8_t* p = pj.curr + (size_t)px0 * NV;
#pragma unroll
            for (int j = 0; j < NV; j++) ldg256_stream(p + 32 * j, R + 8 * j);
            if (C == 1 && S == 1) {
#pragma unroll
                for (int g = 0; g < 8; g++) {
                    const uint32_t ge = __vcmpgeu4(R[g], need4) & ge_and;
                    m |= (((ge & 0x01010101u) * 0x01020408u) >> 24) << (4 * g);
                }
            } else {
#pragma unroll
                for (int k = 0; k < 32; k++) m |= (binarize_pixel_sum<C, S>(R, k) >= need ? 1u : 0u) << k;
            }
        } else {                                          // ragged last word: scalar loads
            for (uint32_t k = 0; k < 32u && px0 + k < npix; k++) {
                const uint8_t* a = pj.curr + (size_t)(px0 + k) * NV;
                uint32_t sum = 0;
                if (S == 2) sum = (uint32_t)a[0] | ((uint32_t)a[1] << 8);
                else for (int q = 0; q < C; q++) sum += a[q];
                m |= (sum >= need ? 1u : 0u) << k;
            }
        }
        pj.mask[w] = m;
        cnt += __popc(m);
    }
    // block reduction -> one atomic per block
    __shared__ uint32_t s_o[8];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, d);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) s_o[warp] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int i = 0; i < (int)(blockDim.x >> 5); i++) t += s_o[i];
        if (t) atomicAdd(ones + blockIdx.y, t);
    }
}

template <int C, int S>
static cudaError_t launch_binarize_t(const PairJob* d_images, int F, uint32_t npix, uint32_t need, uint32_t* d_ones, int sm_count,
                                     int ctas_per_sm, cudaStream_t st) {
    const uint32_t nwords = (npix + 31u) >> 5;
    uint32_t bx = (nwords + 255u) / 256u;
    const uint32_t cap = (uint32_t)(sm_count * (ctas_per_sm > 0 ? ctas_per_sm : 32));
    if ((uint64_t)bx * (uint64_t)F > cap) { bx = (cap + (uint32_t)F - 1u) / (uint32_t)F; if (bx < 1u) bx = 1u; }
    k_binarize<C, S><<<dim3(bx, (unsigned)F), 256, 0, st>>>(d_images, npix, need, d_ones);
    return cudaGetLastError();
}

cudaError_t launch_binarize(const PairJob* d_images, int F, uint32_t npix, int channels, int sample_bytes, int thr_int,
                            uint32_t* d_ones, int sm_count, int ctas_per_sm, cudaStream_t st) {
    if (F <= 0 || npix == 0) return cudaSuccess;
    const int vmax = sample_bytes == 1 ? 255 : 65535;
    const int t = thr_int < -1 ? -1 : (thr_int > vmax ? vmax : thr_int);   // v > t: t < 0 -> all ones, t >= max -> all zeros
    const uint32_t need = (uint32_t)channels * (uint32_t)(t + 1);
    if (sample_bytes == 1) {
        switch (channels) {
        case 1: return launch_binarize_t<1, 1>(d_images, F, npix, need, d_ones, sm_count, ctas_per_sm, st);
        case 2: return launch_binarize_t<2, 1>(d_images, F, npix, need, d_ones, sm_count, ctas_per_sm, st);
        case 3: return launch_binarize_t<3, 1>(d_images, F, npix, need, d_ones, sm_count, ctas_per_sm, st);
        case 4: return launch_binarize_t<4, 1>(d_images, F, npix, need, d_ones, sm_count, ctas_per_sm, st);
        default: return cudaErrorInvalidValue;
        }
    }
    if (sample_bytes == 2 && channels == 1) return launch_binarize_t<1, 2>(d_images, F, npix, need, d_ones, sm_count, ctas_per_sm, st);
    return cudaErrorInvalidValue;
}
