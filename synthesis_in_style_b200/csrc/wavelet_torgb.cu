// SWAGAN wavelet ToRGB in one pass (scf/networks/swagan/model.py:71-98):
//   out[B,12,H,W] = modconv1x1(x, style; no demod) + bias[12] + dwt( upsample( iwt(skip[B,12,H/2,W/2]) ) )
// iwt: upfirdn2d(band, k, up=2, pad=(1,0)) summed over the four bands; upsample: upfirdn2d(k*4, up=2, pad=(2,1));
// dwt: upfirdn2d(k, down=2) per band.  The skip chain is evaluated per output pixel from the skip's 2 x 4 neighbourhood
// (3 x 6 image-domain pixels, 2 x 8 up-sampled pixels per 4-pixel quad), with the taps of the module's own buffers.
// With `final_iwt_k` the last ToRGB of the generator also applies the generator's inverse Haar transform and writes the
// image [B,3,2H,2W]: each image pixel depends on exactly one 12-channel pixel, so the 12-channel map is never stored.
//   algorithmic bytes: B*C*H*W*4 + B*12*(H/2)*(W/2)*4 + B*12*H*W*4   (x is read once, 128-bit streaming loads)
#include "common.cuh"
#include "kernels.h"

namespace sis {

constexpr int WRGB_CH = 12;
constexpr int WRGB_TAPS = 64;   // [iwt 2x2 x4][upsample 4x4][dwt 2x2 x4][final iwt 2x2 x4]

// scale*W transposed to [C][12] (one channel's 12 weights = three 128-bit shared loads) and the taps
__device__ __forceinline__ void wrgb_load_smem(const WaveletToRgbArgs& a, float* swr, float* taps, int tid, int nthreads) {
    for (int i = tid; i < WRGB_CH * a.C; i += nthreads) {
        const int c = i / WRGB_CH, j = i - c * WRGB_CH;
        swr[i] = a.w[(int64_t)j * a.C + c];
    }
    if (tid < WRGB_TAPS) {
        const int t = tid / 16;
        const float* p = t == 0 ? a.iwt_k : t == 1 ? a.up_k : t == 2 ? a.dwt_k : a.final_iwt_k;
        taps[tid] = p ? p[tid % 16] : 0.0f;
    }
}

// acc[j][p] += scale*W[j,c] * s[b,c] * x[b,c,pix+p] for channel c; products w*s rounded first (as torgb_kernel)
__device__ __forceinline__ void wrgb_accumulate(float (&acc)[WRGB_CH][4], const float* swr, int c, float s, float4 v) {
    const float4* wr = reinterpret_cast<const float4*>(swr + WRGB_CH * c);
#pragma unroll
    for (int q = 0; q < 3; ++q) {
        const float4 w4 = wr[q];
        const float wj[4] = {__fmul_rn(w4.x, s), __fmul_rn(w4.y, s), __fmul_rn(w4.z, s), __fmul_rn(w4.w, s)};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float* o = acc[q * 4 + k];
            o[0] = fmaf(wj[k], v.x, o[0]); o[1] = fmaf(wj[k], v.y, o[1]);
            o[2] = fmaf(wj[k], v.z, o[2]); o[3] = fmaf(wj[k], v.w, o[3]);
        }
    }
}

// Bias, skip chain and store for the quad (y, x..x+3) of sample b.  x % 4 == 0.
__device__ __forceinline__ void wrgb_epilogue(const WaveletToRgbArgs& a, const float* taps, float (&acc)[WRGB_CH][4], int b, int y, int x) {
    const float* k_iwt = taps;        // [band][2][2]
    const float* k_up = taps + 16;    // [4][4]
    const float* k_dwt = taps + 32;   // [band][2][2]
    const float* k_fin = taps + 48;   // [band][2][2]
#pragma unroll
    for (int j = 0; j < WRGB_CH; ++j)
#pragma unroll
        for (int p = 0; p < 4; ++p) acc[j][p] = __fadd_rn(acc[j][p], __ldg(a.bias + j));
    if (a.skip) {
        const int SH = a.H / 2, SW = a.W / 2;
        const int64_t band_stride = (int64_t)3 * SH * SW;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            const float* sp = a.skip + ((int64_t)b * WRGB_CH + ch) * SH * SW;
            // image-domain skip (inverse Haar) at rows y-1..y+1, cols x-1..x+4; zero outside the map
            float I[3][6];
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                const int P = y - 1 + i;
                const bool row_ok = P >= 0 && P < a.H;
                const int pr = P & 1;
#pragma unroll
                for (int q = 0; q < 6; ++q) {
                    const int Q = x - 1 + q;          // Q & 1 == (q + 1) & 1 since x is even
                    float v = 0.0f;
                    if (row_ok && Q >= 0 && Q < a.W) {
                        const float* src = sp + (int64_t)(P >> 1) * SW + (Q >> 1);
#pragma unroll
                        for (int band = 0; band < 4; ++band) {
                            const float t = __fmul_rn(__ldg(src + band * band_stride), k_iwt[band * 4 + pr * 2 + ((q + 1) & 1)]);
                            v = band == 0 ? t : __fadd_rn(v, t);
                        }
                    }
                    I[i][q] = v;
                }
            }
            // Upsample at rows 2y+r, cols 2x..2x+7 (the 2x2 polyphase taps of torgb_skip_tap)
            float U[2][8];
#pragma unroll
            for (int r = 0; r < 2; ++r)
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const int p = c >> 1, cb = c & 1;
                    float u = 0.0f;
#pragma unroll
                    for (int yy = 0; yy < 2; ++yy)
#pragma unroll
                        for (int xx = 0; xx < 2; ++xx)
                            u = __fmaf_rn(I[r + yy][p + cb + xx], k_up[(3 - r - 2 * yy) * 4 + (3 - cb - 2 * xx)], u);
                    U[r][c] = u;
                }
            // Haar analysis (down 2, flipped 2x2 taps), added band by band
#pragma unroll
            for (int band = 0; band < 4; ++band)
#pragma unroll
                for (int p = 0; p < 4; ++p) {
                    float d = 0.0f;
#pragma unroll
                    for (int r = 0; r < 2; ++r)
#pragma unroll
                        for (int cb = 0; cb < 2; ++cb) d = __fmaf_rn(U[r][2 * p + cb], k_dwt[band * 4 + (1 - r) * 2 + (1 - cb)], d);
                    acc[band * 3 + ch][p] = __fadd_rn(acc[band * 3 + ch][p], d);
                }
        }
    }
    if (!a.final_iwt_k) {
        const int64_t hw = (int64_t)a.H * a.W;
#pragma unroll
        for (int j = 0; j < WRGB_CH; ++j)
            *reinterpret_cast<float4*>(a.out + ((int64_t)b * WRGB_CH + j) * hw + (int64_t)y * a.W + x) =
                make_float4(acc[j][0], acc[j][1], acc[j][2], acc[j][3]);
        return;
    }
    // generator's inverse Haar transform: image[ch][2y+r][2x'+cb] = sum_band out[band*3+ch][y][x'] * k[band][r][cb]
    const int OW = 2 * a.W;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch)
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            float o[8];
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const int p = c >> 1, cb = c & 1;
                float v = __fmul_rn(acc[ch][p], k_fin[r * 2 + cb]);
#pragma unroll
                for (int band = 1; band < 4; ++band) v = __fadd_rn(v, __fmul_rn(acc[band * 3 + ch][p], k_fin[band * 4 + r * 2 + cb]));
                o[c] = v;
            }
            float4* dst = reinterpret_cast<float4*>(a.out + (((int64_t)b * 3 + ch) * 2 * a.H + 2 * y + r) * OW + 2 * x);
            dst[0] = make_float4(o[0], o[1], o[2], o[3]);
            dst[1] = make_float4(o[4], o[5], o[6], o[7]);
        }
}

// Large maps: one thread = 4 consecutive pixels x all channels (as torgb_wide_kernel).
__global__ void __launch_bounds__(256) wavelet_torgb_wide_kernel(WaveletToRgbArgs a) {
    extern __shared__ float4 wrgb_smem4[];
    float* swr = reinterpret_cast<float*>(wrgb_smem4);
    float* taps = swr + WRGB_CH * a.C;
    const int tid = threadIdx.x;
    wrgb_load_smem(a, swr, taps, tid, 256);
    __syncthreads();
    const int64_t hw = (int64_t)a.H * a.W;
    const int64_t quads_per_sample = hw >> 2;
    const int64_t q = (int64_t)blockIdx.x * 256 + tid;
    if (q >= quads_per_sample * a.batch) return;
    const int b = (int)(q / quads_per_sample);
    const int64_t pix = (q - (int64_t)b * quads_per_sample) << 2;
    const float* xb = a.x + ((int64_t)b * a.C) * hw + pix;
    const float* sb = a.s + (int64_t)b * a.C;
    float acc[WRGB_CH][4] = {};
#pragma unroll 4
    for (int c = 0; c < a.C; ++c)
        wrgb_accumulate(acc, swr, c, __ldg(sb + c), ld_stream_f4(reinterpret_cast<const float4*>(xb + (int64_t)c * hw)));
    const int y = (int)(pix / a.W), x = (int)(pix - (int64_t)y * a.W);
    wrgb_epilogue(a, taps, acc, b, y, x);
}

// Smaller maps: blockDim = (32 quads, 8 slices); each slice sums a channel range, the slices are reduced through shared
// memory in fixed order, and one warp runs the epilogue (as torgb_kernel; 8 slices, not 32, for the small maps: with 12
// outputs per pixel a 512- or 1024-thread block cannot hold the epilogue's registers without spilling).
__global__ void __launch_bounds__(256) wavelet_torgb_kernel(WaveletToRgbArgs a) {
    extern __shared__ float4 wrgb_smem4[];
    float* swr = reinterpret_cast<float*>(wrgb_smem4);
    float* taps = swr + WRGB_CH * a.C;
    float* red = taps + WRGB_TAPS;                     // [slices][12*4][32]
    const int lane = threadIdx.x, slice = threadIdx.y, nsl = blockDim.y;
    const int tid = slice * 32 + lane, nthreads = 32 * nsl;
    wrgb_load_smem(a, swr, taps, tid, nthreads);
    __syncthreads();
    const int64_t hw = (int64_t)a.H * a.W;
    const int64_t quads_per_sample = hw / 4;
    const int64_t total_quads = quads_per_sample * a.batch;
    const int cps = (a.C + nsl - 1) / nsl;
    const int c_begin = slice * cps, c_end = min(a.C, c_begin + cps);
    constexpr int NV = WRGB_CH * 4;
    for (int64_t q0 = (int64_t)blockIdx.x * 32; q0 < total_quads; q0 += (int64_t)gridDim.x * 32) {
        const int64_t q = q0 + lane;
        const bool valid = q < total_quads;
        const int b = valid ? (int)(q / quads_per_sample) : 0;
        const int64_t pix = valid ? (q - (int64_t)b * quads_per_sample) * 4 : 0;
        float acc[WRGB_CH][4] = {};
        if (valid) {
            const float* xb = a.x + ((int64_t)b * a.C) * hw + pix;
            const float* sb = a.s + (int64_t)b * a.C;
#pragma unroll 4
            for (int c = c_begin; c < c_end; ++c)
                wrgb_accumulate(acc, swr, c, __ldg(sb + c), ld_stream_f4(reinterpret_cast<const float4*>(xb + (int64_t)c * hw)));
        }
#pragma unroll
        for (int j = 0; j < WRGB_CH; ++j)
#pragma unroll
            for (int p = 0; p < 4; ++p) red[((slice * NV) + j * 4 + p) * 32 + lane] = acc[j][p];
        __syncthreads();
        for (int e = tid; e < NV * 32; e += nthreads) {     // slot 0 receives the sum over the slices, in slice order
            float v = red[e];
            for (int s = 1; s < nsl; ++s) v += red[s * NV * 32 + e];
            red[e] = v;
        }
        __syncthreads();
        if (slice == 0 && valid) {
#pragma unroll
            for (int j = 0; j < WRGB_CH; ++j)
#pragma unroll
                for (int p = 0; p < 4; ++p) acc[j][p] = red[(j * 4 + p) * 32 + lane];
            const int y = (int)(pix / a.W), x = (int)(pix - (int64_t)y * a.W);
            wrgb_epilogue(a, taps, acc, b, y, x);
        }
        __syncthreads();
    }
}

int launch_wavelet_torgb(const WaveletToRgbArgs& a, cudaStream_t stream) {
    SIS_REQUIRE(a.W % 4 == 0 && a.H % 2 == 0, "wavelet_torgb: the map width must be a multiple of 4 and its height even (got %dx%d)", a.H, a.W);
    SIS_REQUIRE(!a.skip || (a.iwt_k && a.up_k && a.dwt_k), "wavelet_torgb: a skip needs the iwt, upsample and dwt taps");
    const int64_t quads = (int64_t)a.H * a.W / 4 * a.batch;
    const size_t base_smem = (size_t)(WRGB_CH * a.C + WRGB_TAPS) * sizeof(float);
    if (quads >= (int64_t)kNumSMs * 512 && base_smem <= 48 * 1024) {
        wavelet_torgb_wide_kernel<<<(unsigned)ceil_div64(quads, 256), 256, base_smem, stream>>>(a);
        SIS_CHECK_LAUNCH();
        return SIS_OK;
    }
    const int64_t blocks = ceil_div64(quads, 32);
    const int64_t cap = (int64_t)kNumSMs * 8;
    const int grid = (int)(blocks < cap ? blocks : cap);
    constexpr int slices = 8;
    const size_t smem = base_smem + (size_t)slices * WRGB_CH * 4 * 32 * sizeof(float);
    constexpr size_t kMaxSmem = 160 * 1024;
    SIS_REQUIRE(smem <= kMaxSmem, "wavelet_torgb: %d input channels need more shared memory than a block has", a.C);
    if (smem > 48 * 1024) {
        static bool configured = false;
        if (!configured) {
            SIS_CHECK_CUDA(cudaFuncSetAttribute(wavelet_torgb_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
            configured = true;
        }
    }
    wavelet_torgb_kernel<<<grid, dim3(32, slices), smem, stream>>>(a);
    SIS_CHECK_LAUNCH();
    return SIS_OK;
}

}  // namespace sis
