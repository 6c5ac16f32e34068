// DatasetGAN labeller (SURVEY.md §8(f) row 3): all captures -> per-pixel ensemble of MLP classifiers -> label image.
//   scf/data/dataset_gan_dataset.py:12-34            scale_activations (bilinear upsample of every capture to S x S, concat)
//   scf/networks/pixel_classifier/model.py:40-121    PixelClassifier (Linear F->128, ReLU, BN, Linear 128->32, ReLU, BN,
//                                                     Linear 32->n), PixelEnsembleClassifier.predict_classes (torch.mode)
//   scf/segmentation/dataset_gan_segmenter.py:34-60  predict_labels, label_images_to_color_images
//
// The reference materialises the upsampled feature tensor [B, S, S, F] (F = 5888 at 256^2: 1.5 GB per image) and runs
// three F -> 128 GEMMs over it (0.3 TFLOP per image).  Both the upsample and the first Linear are linear maps and the
// upsample acts per channel, so they commute:
//     Linear1(upsample(x_l))  =  upsample(W1[:, slice_l] x_l)
// Here the first layer runs at every capture's NATIVE resolution -- captures of one resolution stacked along K, the
// networks of the ensemble stacked along N (3 x 128 = 384) -- on the tcgen05 conv GEMM (one tap, bf16 hi/lo split,
// fp32 accumulation): 19 GFLOP per image instead of 297.  One tail kernel then, per output pixel, gathers the bilinear
// taps of the 6 low-resolution products and the full-resolution one, and runs the rest of every network in registers:
// ReLU, the two remaining Linears with the eval-mode BatchNorms folded into them, argmax, and the mode vote.
#include <map>
#include <string>
#include <vector>
#include <cmath>
#include "common.cuh"
#include "dataset_gan_common.cuh"
#include "kernels.h"
#include "modconv_tc.h"
#include "../../include/sis_b200.h"

namespace sis {

struct GanTailArgs {
    const float* y[GAN_MAX_GROUPS];     // first-layer products per resolution: fp32 [B][M*128][r][r] (NCHW) or, when
    int res[GAN_MAX_GROUPS];            // nhwc[g], [B][r][r][M*128]
    int nhwc[GAN_MAX_GROUPS];
    int n_groups;
    int batch, S, n_models, n_class;
    const float* b1;                    // [M][128]
    const float* w2t;                   // [M][128][32]   W2[j][i] * sc1[i], transposed
    const float* b2;                    // [M][32]        b2 + W2 sh1
    const float* w3;                    // [M][n][32]     W3[c][j] * sc2[j]
    const float* b3;                    // [M][n]         b3 + W3 sh2
    uint8_t* labels;                    // [B][S][S]
    uint8_t* votes;                     // [B][S][S][M] or null
    const uint8_t* colors;              // [n][3] or null
    uint8_t* color_image;               // [B][S][S][3] or null
};

// One thread per output pixel, 128 pixels per block.  Per network: z[128] in registers.
__global__ void __launch_bounds__(128) dataset_gan_tail_kernel(GanTailArgs a) {
    __shared__ __align__(16) float s_w2t[GAN_H1 * GAN_H2];
    __shared__ float s_b1[GAN_H1], s_b2[GAN_H2], s_w3[31 * GAN_H2], s_b3[32];
    const int tid = threadIdx.x;
    const int64_t total = (int64_t)a.batch * a.S * a.S;
    int64_t p = (int64_t)blockIdx.x * 128 + tid;
    const bool valid = p < total;
    if (!valid) p = total - 1;
    const int b = (int)(p / ((int64_t)a.S * a.S));
    const int rem = (int)(p - (int64_t)b * a.S * a.S);
    const int oy = rem / a.S, ox = rem - oy * a.S;
    int vote[GAN_MAX_MODELS];

    for (int m = 0; m < a.n_models; ++m) {
        __syncthreads();
        for (int i = tid; i < GAN_H1 * GAN_H2; i += 128) s_w2t[i] = a.w2t[(int64_t)m * GAN_H1 * GAN_H2 + i];
        s_b1[tid] = a.b1[m * GAN_H1 + tid];
        if (tid < GAN_H2) s_b2[tid] = a.b2[m * GAN_H2 + tid];
        for (int i = tid; i < a.n_class * GAN_H2; i += 128) s_w3[i] = a.w3[(int64_t)m * a.n_class * GAN_H2 + i];
        if (tid < a.n_class) s_b3[tid] = a.b3[m * a.n_class + tid];
        __syncthreads();

        float z[GAN_H1];
#pragma unroll
        for (int i = 0; i < GAN_H1; ++i) z[i] = s_b1[i];
        for (int g = 0; g < a.n_groups; ++g) {
            const int r = a.res[g];
            const int64_t plane = (int64_t)r * r;
            const float* base = a.y[g] + ((int64_t)b * a.n_models + m) * GAN_H1 * plane;
            if (r == a.S) {
                const float* q = base + (int64_t)oy * r + ox;
#pragma unroll
                for (int i = 0; i < GAN_H1; ++i) z[i] += __ldg(q + (int64_t)i * plane);
            } else {
                const GanBilinearTap tap = gan_bilinear_tap(oy, ox, r, a.S);
                const int y0 = tap.y0, y1 = tap.y1, x0 = tap.x0, x1 = tap.x1;
                const float w00 = tap.w00, w01 = tap.w01, w10 = tap.w10, w11 = tap.w11;
                const float* q00 = base + y0 * r + x0; const float* q01 = base + y0 * r + x1;
                const float* q10 = base + y1 * r + x0; const float* q11 = base + y1 * r + x1;
#pragma unroll
                for (int i = 0; i < GAN_H1; ++i) {
                    const int64_t o = (int64_t)i * plane;
                    float v = w00 * __ldg(q00 + o);
                    v = fmaf(w01, __ldg(q01 + o), v);
                    v = fmaf(w10, __ldg(q10 + o), v);
                    v = fmaf(w11, __ldg(q11 + o), v);
                    z[i] += v;
                }
            }
        }
        // Linear2 (BatchNorm1 folded in) over relu(z): 32 outputs as 16 packed pairs
        float2 u2[GAN_H2 / 2];
#pragma unroll
        for (int j = 0; j < GAN_H2 / 2; ++j) u2[j] = make_float2(s_b2[2 * j], s_b2[2 * j + 1]);
#pragma unroll
        for (int i = 0; i < GAN_H1; ++i) {
            const float h = fmaxf(z[i], 0.0f);
            const float2 hh = make_float2(h, h);
            const float4* wrow = reinterpret_cast<const float4*>(s_w2t + i * GAN_H2);
#pragma unroll
            for (int q = 0; q < GAN_H2 / 4; ++q) {
                const float4 w = wrow[q];
                u2[2 * q] = pk_fma(hh, make_float2(w.x, w.y), u2[2 * q]);
                u2[2 * q + 1] = pk_fma(hh, make_float2(w.z, w.w), u2[2 * q + 1]);
            }
        }
        float u[GAN_H2];
#pragma unroll
        for (int j = 0; j < GAN_H2 / 2; ++j) { u[2 * j] = fmaxf(u2[j].x, 0.0f); u[2 * j + 1] = fmaxf(u2[j].y, 0.0f); }
        // Linear3 (BatchNorm2 folded in) + argmax (first maximum, as torch.max)
        float best = -INFINITY;
        int arg = 0;
        for (int c = 0; c < a.n_class; ++c) {
            float acc = s_b3[c];
#pragma unroll
            for (int j = 0; j < GAN_H2; ++j) acc = fmaf(s_w3[c * GAN_H2 + j], u[j], acc);
            if (acc > best) { best = acc; arg = c; }
        }
        vote[m] = arg;
    }
    if (!valid) return;
    // torch.mode over the networks: the most frequent class, the smallest one on ties
    int label = 0, best_count = 0;
    for (int m = 0; m < a.n_models; ++m) {
        int count = 0;
        for (int q = 0; q < a.n_models; ++q) count += (vote[q] == vote[m]);
        if (count > best_count || (count == best_count && vote[m] < label)) { best_count = count; label = vote[m]; }
    }
    a.labels[p] = (uint8_t)label;
    if (a.votes)
        for (int m = 0; m < a.n_models; ++m) a.votes[p * a.n_models + m] = (uint8_t)vote[m];
    if (a.color_image && a.colors) {
        a.color_image[p * 3 + 0] = a.colors[label * 3 + 0];
        a.color_image[p * 3 + 1] = a.colors[label * 3 + 1];
        a.color_image[p * 3 + 2] = a.colors[label * 3 + 2];
    }
}

// Tiled variant (S a multiple of 16): a block is a 16 x 8 pixel tile.  The low-resolution products are NHWC; per network,
// 32-channel chunk and resolution the tile's source footprint (at most 6 x 10 pixels) is staged in shared memory with
// 128 B coalesced rows and every thread accumulates its four taps from there; the full-resolution product is NCHW and
// is read directly (consecutive lanes = consecutive pixels).  Working in 32-channel chunks keeps a thread at 32
// activations + 32 second-layer accumulators (the chunk is folded into Linear2 as soon as it is complete), so four
// blocks fit on an SM.
constexpr int GAN_TX = 16, GAN_TY = 8, GAN_CH = 32, GAN_SRC_STRIDE = GAN_CH + 4;
constexpr int GAN_SRC_PIX = 60 + 24 + 12 + 9 + 9 + 9 + 9;      // footprints of up to 7 low-resolution products, scales 2, 4, 8, >= 16

__device__ __forceinline__ void gan_src_range(int o0, int n, int r, int S, int& lo, int& hi) {
    const float sc = (float)r / (float)S;
    lo = (int)fmaxf(((float)o0 + 0.5f) * sc - 0.5f, 0.0f);
    hi = min((int)fmaxf(((float)(o0 + n - 1) + 0.5f) * sc - 0.5f, 0.0f) + 1, r - 1);
}

__global__ void __launch_bounds__(128, 4) dataset_gan_tail_tiled_kernel(GanTailArgs a) {
    __shared__ __align__(16) float s_src[GAN_SRC_PIX * GAN_SRC_STRIDE];
    __shared__ __align__(16) float s_w2t[GAN_H1 * GAN_H2];
    __shared__ float s_b1[GAN_H1], s_b2[GAN_H2], s_w3[31 * GAN_H2], s_b3[32];
    const int tid = threadIdx.x;
    const int tiles_x = a.S / GAN_TX, tiles_y = a.S / GAN_TY;
    const int tile = blockIdx.x;
    const int b = tile / (tiles_x * tiles_y);
    const int trem = tile - b * tiles_x * tiles_y;
    const int oy0 = (trem / tiles_x) * GAN_TY, ox0 = (trem % tiles_x) * GAN_TX;
    const int oy = oy0 + tid / GAN_TX, ox = ox0 + tid % GAN_TX;
    const int N = a.n_models * GAN_H1;
    int vote[GAN_MAX_MODELS];

    for (int m = 0; m < a.n_models; ++m) {
        __syncthreads();
        for (int i = tid; i < GAN_H1 * GAN_H2; i += 128) s_w2t[i] = a.w2t[(int64_t)m * GAN_H1 * GAN_H2 + i];
        s_b1[tid] = a.b1[m * GAN_H1 + tid];
        if (tid < GAN_H2) s_b2[tid] = a.b2[m * GAN_H2 + tid];
        for (int i = tid; i < a.n_class * GAN_H2; i += 128) s_w3[i] = a.w3[(int64_t)m * a.n_class * GAN_H2 + i];
        if (tid < a.n_class) s_b3[tid] = a.b3[m * a.n_class + tid];
        __syncthreads();

        float2 u2[GAN_H2 / 2];
#pragma unroll
        for (int j = 0; j < GAN_H2 / 2; ++j) u2[j] = make_float2(s_b2[2 * j], s_b2[2 * j + 1]);

#pragma unroll 1
        for (int ch0 = 0; ch0 < GAN_H1; ch0 += GAN_CH) {
            float z[GAN_CH];
#pragma unroll
            for (int i = 0; i < GAN_CH; ++i) z[i] = s_b1[ch0 + i];
            // stage the footprints of ALL low-resolution products for this chunk at once (at most 60 + 24 + 12 + 9 + 9 + 6
            // source pixels for scales 2 .. 64): two block barriers per chunk instead of two per product
            __syncthreads();                                     // the previous chunk's taps are consumed
            int base_px[GAN_MAX_GROUPS];
            {
                int acc_px = 0;
                for (int g = 0; g < a.n_groups; ++g) {
                    base_px[g] = acc_px;
                    if (!a.nhwc[g]) continue;
                    const int r = a.res[g];
                    int fy0, fy1, fx0, fx1;
                    gan_src_range(oy0, GAN_TY, r, a.S, fy0, fy1);
                    gan_src_range(ox0, GAN_TX, r, a.S, fx0, fx1);
                    const int fw = fx1 - fx0 + 1, fh = fy1 - fy0 + 1;
                    for (int q = tid; q < fh * fw * (GAN_CH / 4); q += 128) {
                        const int px = q / (GAN_CH / 4), c4 = q - px * (GAN_CH / 4);
                        const int py = px / fw, pxx = px - py * fw;
                        const float4 v = __ldg(reinterpret_cast<const float4*>(
                            a.y[g] + (((int64_t)b * r + fy0 + py) * r + fx0 + pxx) * N + m * GAN_H1 + ch0) + c4);
                        *reinterpret_cast<float4*>(s_src + (acc_px + px) * GAN_SRC_STRIDE + c4 * 4) = v;
                    }
                    acc_px += fh * fw;
                }
            }
            __syncthreads();
#pragma unroll 1
            for (int g = 0; g < a.n_groups; ++g) {
                const int r = a.res[g];
                if (!a.nhwc[g]) {
                    const int64_t plane = (int64_t)r * r;
                    const float* q = a.y[g] + (((int64_t)b * a.n_models + m) * GAN_H1 + ch0) * plane + (int64_t)oy * r + ox;
#pragma unroll
                    for (int i = 0; i < GAN_CH; ++i) z[i] += __ldg(q + (int64_t)i * plane);
                    continue;
                }
                int fy0, fy1, fx0, fx1;
                gan_src_range(oy0, GAN_TY, r, a.S, fy0, fy1);
                gan_src_range(ox0, GAN_TX, r, a.S, fx0, fx1);
                const int fw = fx1 - fx0 + 1;
                const float* src = s_src + base_px[g] * GAN_SRC_STRIDE;
                const GanBilinearTap tap = gan_bilinear_tap(oy, ox, r, a.S);
                const int y0 = tap.y0, y1 = tap.y1, x0 = tap.x0, x1 = tap.x1;
                const float w00 = tap.w00, w01 = tap.w01, w10 = tap.w10, w11 = tap.w11;
                const float4* q00 = reinterpret_cast<const float4*>(src + ((y0 - fy0) * fw + x0 - fx0) * GAN_SRC_STRIDE);
                const float4* q01 = reinterpret_cast<const float4*>(src + ((y0 - fy0) * fw + x1 - fx0) * GAN_SRC_STRIDE);
                const float4* q10 = reinterpret_cast<const float4*>(src + ((y1 - fy0) * fw + x0 - fx0) * GAN_SRC_STRIDE);
                const float4* q11 = reinterpret_cast<const float4*>(src + ((y1 - fy0) * fw + x1 - fx0) * GAN_SRC_STRIDE);
#pragma unroll
                for (int i4 = 0; i4 < GAN_CH / 4; ++i4) {
                    const float4 v00 = q00[i4], v01 = q01[i4], v10 = q10[i4], v11 = q11[i4];
                    z[4 * i4 + 0] += fmaf(w11, v11.x, fmaf(w10, v10.x, fmaf(w01, v01.x, w00 * v00.x)));
                    z[4 * i4 + 1] += fmaf(w11, v11.y, fmaf(w10, v10.y, fmaf(w01, v01.y, w00 * v00.y)));
                    z[4 * i4 + 2] += fmaf(w11, v11.z, fmaf(w10, v10.z, fmaf(w01, v01.z, w00 * v00.z)));
                    z[4 * i4 + 3] += fmaf(w11, v11.w, fmaf(w10, v10.w, fmaf(w01, v01.w, w00 * v00.w)));
                }
            }
            // fold the finished chunk into Linear2 (BatchNorm1 folded in)
#pragma unroll
            for (int i = 0; i < GAN_CH; ++i) {
                const float h = fmaxf(z[i], 0.0f);
                const float2 hh = make_float2(h, h);
                const float4* wrow = reinterpret_cast<const float4*>(s_w2t + (ch0 + i) * GAN_H2);
#pragma unroll
                for (int q = 0; q < GAN_H2 / 4; ++q) {
                    const float4 w = wrow[q];
                    u2[2 * q] = pk_fma(hh, make_float2(w.x, w.y), u2[2 * q]);
                    u2[2 * q + 1] = pk_fma(hh, make_float2(w.z, w.w), u2[2 * q + 1]);
                }
            }
        }
        float u[GAN_H2];
#pragma unroll
        for (int j = 0; j < GAN_H2 / 2; ++j) { u[2 * j] = fmaxf(u2[j].x, 0.0f); u[2 * j + 1] = fmaxf(u2[j].y, 0.0f); }
        float best = -INFINITY;
        int arg = 0;
        for (int c = 0; c < a.n_class; ++c) {
            float acc = s_b3[c];
#pragma unroll
            for (int j = 0; j < GAN_H2; ++j) acc = fmaf(s_w3[c * GAN_H2 + j], u[j], acc);
            if (acc > best) { best = acc; arg = c; }
        }
        vote[m] = arg;
    }
    int label = 0, best_count = 0;
    for (int m = 0; m < a.n_models; ++m) {
        int count = 0;
        for (int q = 0; q < a.n_models; ++q) count += (vote[q] == vote[m]);
        if (count > best_count || (count == best_count && vote[m] < label)) { best_count = count; label = vote[m]; }
    }
    const int64_t p = ((int64_t)b * a.S + oy) * a.S + ox;
    a.labels[p] = (uint8_t)label;
    if (a.votes)
        for (int m = 0; m < a.n_models; ++m) a.votes[p * a.n_models + m] = (uint8_t)vote[m];
    if (a.color_image && a.colors) {
        a.color_image[p * 3 + 0] = a.colors[label * 3 + 0];
        a.color_image[p * 3 + 1] = a.colors[label * 3 + 1];
        a.color_image[p * 3 + 2] = a.colors[label * 3 + 2];
    }
}

struct GanGroup {
    int res = 0, k = 0;
    std::vector<int> layers, feat_off, chan;
    void *a_hi = nullptr, *a_lo = nullptr, *w_hi = nullptr, *w_lo = nullptr;
    float* y = nullptr;
};

}  // namespace sis

struct sis_pixel_ensemble {
    int n_models = 0, feature_size = 0, n_class = 0;
    std::vector<std::map<std::string, std::vector<float>>> host;     // per network: reference state-dict key -> values
    bool prepared = false;
    float *d_w1 = nullptr, *d_b1 = nullptr, *d_w2t = nullptr, *d_b2 = nullptr, *d_w3 = nullptr, *d_b3 = nullptr;
    float* d_ones = nullptr; unsigned int* d_error = nullptr; uint8_t* d_colors = nullptr;
    std::vector<sis::GanGroup> groups;
    std::vector<int> sig;                                            // (batch, channels..., res...) the groups were built for
};

namespace sis {

static void free_groups(sis_pixel_ensemble* e) {
    for (auto& g : e->groups) {
        cudaFree(g.a_hi); cudaFree(g.a_lo); cudaFree(g.w_hi); cudaFree(g.w_lo); cudaFree(g.y);
    }
    e->groups.clear();
    e->sig.clear();
    if (e->d_ones) { cudaFree(e->d_ones); e->d_ones = nullptr; }
}

static int expect(const std::map<std::string, std::vector<float>>& sd, const char* key, size_t n) {
    auto it = sd.find(key);
    SIS_REQUIRE(it != sd.end(), "pixel ensemble: parameter '%s' was never set", key);
    SIS_REQUIRE(it->second.size() == n, "pixel ensemble: parameter '%s' has %zu values, expected %zu", key, it->second.size(), n);
    return SIS_OK;
}

}  // namespace sis

extern "C" int sis_pixel_ensemble_create(sis_pixel_ensemble** out, int n_models, int feature_size, int n_class) {
    using namespace sis;
    SIS_REQUIRE(out, "sis_pixel_ensemble_create: null output");
    SIS_REQUIRE(n_models >= 1 && n_models <= GAN_MAX_MODELS, "pixel ensemble: 1..%d networks (got %d)", GAN_MAX_MODELS, n_models);
    SIS_REQUIRE(n_class >= 1 && n_class < 32, "pixel ensemble: the 128/32 classifier is the reference's n_class < 32 variant (got %d)", n_class);
    SIS_REQUIRE(feature_size > 0 && feature_size % 32 == 0, "pixel ensemble: feature size must be a positive multiple of 32 (got %d)", feature_size);
    auto* e = new sis_pixel_ensemble();
    e->n_models = n_models; e->feature_size = feature_size; e->n_class = n_class;
    e->host.resize(n_models);
    *out = e;
    return SIS_OK;
}

extern "C" void sis_pixel_ensemble_destroy(sis_pixel_ensemble* e) {
    if (!e) return;
    sis::free_groups(e);
    cudaFree(e->d_w1); cudaFree(e->d_b1); cudaFree(e->d_w2t); cudaFree(e->d_b2); cudaFree(e->d_w3); cudaFree(e->d_b3);
    cudaFree(e->d_colors);
    delete e;
}

extern "C" int sis_pixel_ensemble_set_param(sis_pixel_ensemble* e, int model, const char* name, const float* host_data, int64_t numel) {
    using namespace sis;
    SIS_REQUIRE(e && name && host_data, "sis_pixel_ensemble_set_param: null argument");
    SIS_REQUIRE(model >= 0 && model < e->n_models, "pixel ensemble: network index %d out of range", model);
    e->host[model][name].assign(host_data, host_data + numel);
    e->prepared = false;
    return SIS_OK;
}

extern "C" int sis_pixel_ensemble_prepare(sis_pixel_ensemble* e, void* stream_) {
    using namespace sis;
    SIS_REQUIRE(e, "sis_pixel_ensemble_prepare: null ensemble");
    cudaStream_t stream = (cudaStream_t)stream_;
    const int M = e->n_models, F = e->feature_size, n = e->n_class;
    std::vector<float> w1((size_t)M * GAN_H1 * F), b1((size_t)M * GAN_H1), w2t((size_t)M * GAN_H1 * GAN_H2), b2((size_t)M * GAN_H2),
        w3((size_t)M * n * GAN_H2), b3((size_t)M * n);
    for (int m = 0; m < M; ++m) {
        const auto& sd = e->host[m];
        SIS_PROPAGATE(expect(sd, "layers.0.weight", (size_t)GAN_H1 * F)); SIS_PROPAGATE(expect(sd, "layers.0.bias", GAN_H1));
        SIS_PROPAGATE(expect(sd, "layers.3.weight", (size_t)GAN_H2 * GAN_H1)); SIS_PROPAGATE(expect(sd, "layers.3.bias", GAN_H2));
        SIS_PROPAGATE(expect(sd, "layers.6.weight", (size_t)n * GAN_H2)); SIS_PROPAGATE(expect(sd, "layers.6.bias", n));
        for (const char* bn : {"layers.2", "layers.5"}) {
            const size_t f = std::string(bn) == "layers.2" ? GAN_H1 : GAN_H2;
            for (const char* part : {".weight", ".bias", ".running_mean", ".running_var"})
                SIS_PROPAGATE(expect(sd, (std::string(bn) + part).c_str(), f));
        }
        std::copy(sd.at("layers.0.weight").begin(), sd.at("layers.0.weight").end(), w1.begin() + (size_t)m * GAN_H1 * F);
        std::copy(sd.at("layers.0.bias").begin(), sd.at("layers.0.bias").end(), b1.begin() + (size_t)m * GAN_H1);
        // eval-mode BatchNorm1d after the ReLU = h * sc + sh; fold it into the next Linear (double precision)
        auto fold = [&](const char* bn, int f, std::vector<double>& sc, std::vector<double>& sh) {
            const auto& g = sd.at(std::string(bn) + ".weight"); const auto& be = sd.at(std::string(bn) + ".bias");
            const auto& mu = sd.at(std::string(bn) + ".running_mean"); const auto& var = sd.at(std::string(bn) + ".running_var");
            sc.resize(f); sh.resize(f);
            for (int i = 0; i < f; ++i) { sc[i] = (double)g[i] / std::sqrt((double)var[i] + 1e-5); sh[i] = (double)be[i] - (double)mu[i] * sc[i]; }
        };
        std::vector<double> sc1, sh1, sc2, sh2;
        fold("layers.2", GAN_H1, sc1, sh1);
        fold("layers.5", GAN_H2, sc2, sh2);
        const auto& W2 = sd.at("layers.3.weight"); const auto& B2 = sd.at("layers.3.bias");
        for (int j = 0; j < GAN_H2; ++j) {
            double acc = B2[j];
            for (int i = 0; i < GAN_H1; ++i) {
                w2t[((size_t)m * GAN_H1 + i) * GAN_H2 + j] = (float)((double)W2[(size_t)j * GAN_H1 + i] * sc1[i]);
                acc += (double)W2[(size_t)j * GAN_H1 + i] * sh1[i];
            }
            b2[(size_t)m * GAN_H2 + j] = (float)acc;
        }
        const auto& W3 = sd.at("layers.6.weight"); const auto& B3 = sd.at("layers.6.bias");
        for (int c = 0; c < n; ++c) {
            double acc = B3[c];
            for (int j = 0; j < GAN_H2; ++j) {
                w3[((size_t)m * n + c) * GAN_H2 + j] = (float)((double)W3[(size_t)c * GAN_H2 + j] * sc2[j]);
                acc += (double)W3[(size_t)c * GAN_H2 + j] * sh2[j];
            }
            b3[(size_t)m * n + c] = (float)acc;
        }
    }
    auto upload = [&](float*& d, const std::vector<float>& h) -> int {
        if (d) cudaFree(d);
        d = nullptr;
        SIS_CHECK_CUDA(cudaMalloc(&d, h.size() * sizeof(float)));
        SIS_CHECK_CUDA(cudaMemcpyAsync(d, h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice, stream));
        return SIS_OK;
    };
    SIS_PROPAGATE(upload(e->d_w1, w1)); SIS_PROPAGATE(upload(e->d_b1, b1)); SIS_PROPAGATE(upload(e->d_w2t, w2t));
    SIS_PROPAGATE(upload(e->d_b2, b2)); SIS_PROPAGATE(upload(e->d_w3, w3)); SIS_PROPAGATE(upload(e->d_b3, b3));
    if (!e->d_error) e->d_error = watchdog_word();
    SIS_CHECK_CUDA(cudaStreamSynchronize(stream));      // the host vectors go out of scope
    free_groups(e);
    e->prepared = true;
    return SIS_OK;
}

extern "C" int sis_pixel_ensemble_label(sis_pixel_ensemble* e, int n_layers, const float* const* d_activations, const int* channels,
                                        const int* resolutions, int batch, int image_size, uint8_t* d_labels, uint8_t* d_votes,
                                        const uint8_t* host_colors, uint8_t* d_color_image, void* stream_) {
    using namespace sis;
    SIS_REQUIRE(e && e->prepared, "sis_pixel_ensemble_label: call sis_pixel_ensemble_prepare first");
    SIS_REQUIRE(n_layers > 0 && d_activations && channels && resolutions && d_labels, "sis_pixel_ensemble_label: null argument");
    SIS_REQUIRE(batch > 0 && image_size > 0, "sis_pixel_ensemble_label: bad batch / image size");
    cudaStream_t stream = (cudaStream_t)stream_;
    const int M = e->n_models, N = M * GAN_H1;
    std::vector<int> sig = {batch, image_size};
    int feat = 0;
    for (int l = 0; l < n_layers; ++l) {
        SIS_REQUIRE(d_activations[l], "sis_pixel_ensemble_label: activation %d is null", l);
        SIS_REQUIRE(channels[l] % 32 == 0, "pixel ensemble: capture %d has %d channels; multiples of 32 only", l, channels[l]);
        SIS_REQUIRE(resolutions[l] <= image_size, "pixel ensemble: capture %d is larger than the image", l);
        sig.push_back(channels[l]); sig.push_back(resolutions[l]);
        feat += channels[l];
    }
    SIS_REQUIRE(feat == e->feature_size, "pixel ensemble: captures carry %d features, the classifiers expect %d", feat, e->feature_size);
    if (sig != e->sig) {
        // (re)build the per-resolution groups: stacked A planes, packed weight slices, product buffers
        free_groups(e);
        int off = 0;
        for (int l = 0; l < n_layers; ++l) {
            GanGroup* g = nullptr;
            for (auto& cand : e->groups) if (cand.res == resolutions[l]) g = &cand;
            if (!g) { e->groups.emplace_back(); g = &e->groups.back(); g->res = resolutions[l]; }
            g->layers.push_back(l); g->feat_off.push_back(off); g->chan.push_back(channels[l]);
            g->k += channels[l];
            off += channels[l];
        }
        SIS_REQUIRE((int)e->groups.size() <= GAN_MAX_GROUPS, "pixel ensemble: more than %d distinct capture resolutions", GAN_MAX_GROUPS);
        for (auto& g : e->groups) {
            const size_t a_elems = (size_t)batch * g.res * g.res * g.k;
            SIS_CHECK_CUDA(cudaMalloc(&g.a_hi, a_elems * 2)); SIS_CHECK_CUDA(cudaMalloc(&g.a_lo, a_elems * 2));
            SIS_CHECK_CUDA(cudaMalloc(&g.w_hi, (size_t)N * g.k * 2)); SIS_CHECK_CUDA(cudaMalloc(&g.w_lo, (size_t)N * g.k * 2));
            SIS_CHECK_CUDA(cudaMalloc((void**)&g.y, (size_t)batch * N * g.res * g.res * sizeof(float)));
            int koff = 0;
            for (size_t i = 0; i < g.layers.size(); ++i) {
                SIS_PROPAGATE(tc_pack_matrix_split(g.w_hi, g.w_lo, e->d_w1, N, g.chan[i], e->feature_size, g.feat_off[i], g.k, koff, stream));
                koff += g.chan[i];
            }
        }
        std::vector<float> ones((size_t)batch * N, 1.0f);
        SIS_CHECK_CUDA(cudaMalloc((void**)&e->d_ones, ones.size() * sizeof(float)));
        SIS_CHECK_CUDA(cudaMemcpyAsync(e->d_ones, ones.data(), ones.size() * sizeof(float), cudaMemcpyHostToDevice, stream));
        SIS_CHECK_CUDA(cudaStreamSynchronize(stream));
        e->sig = sig;
    }
    if (host_colors) {
        if (!e->d_colors) SIS_CHECK_CUDA(cudaMalloc((void**)&e->d_colors, 32 * 3));
        SIS_CHECK_CUDA(cudaMemcpyAsync(e->d_colors, host_colors, (size_t)e->n_class * 3, cudaMemcpyHostToDevice, stream));
    }
    GanTailArgs t;
    memset(&t, 0, sizeof(t));
    // tiled tail: 16 x 8 pixel tiles, power-of-two integer scale factors (footprints of at most 6 x 10 source pixels)
    bool tiled = image_size % GAN_TX == 0 && image_size % GAN_TY == 0;
    int footprint_px = 0;                     // conservative bound of the staged source pixels of all low-resolution products
    for (auto& g : e->groups) {
        tiled = tiled && image_size % g.res == 0 && (g.res == image_size || image_size / g.res >= 2);
        if (g.res < image_size && image_size % g.res == 0) {
            const int scale = image_size / g.res;
            footprint_px += std::min(g.res, ceil_div(GAN_TY, scale) + 2) * std::min(g.res, ceil_div(GAN_TX, scale) + 2);
        }
    }
    tiled = tiled && footprint_px <= GAN_SRC_PIX;
    int gi = 0;
    for (auto& g : e->groups) {
        int koff = 0;
        for (size_t i = 0; i < g.layers.size(); ++i) {
            SIS_PROPAGATE(tc_nchw_to_nhwc_split(g.a_hi, g.a_lo, d_activations[g.layers[i]], batch, g.chan[i], (int64_t)g.res * g.res, g.k, koff, stream));
            koff += g.chan[i];
        }
        const bool nhwc = tiled && g.res < image_size;
        SIS_PROPAGATE(tc_conv1x1(g.a_hi, g.a_lo, g.w_hi, g.w_lo, batch, g.res, g.k, N, e->d_ones, g.y, nhwc, e->d_error, stream));
        t.y[gi] = g.y; t.res[gi] = g.res; t.nhwc[gi] = nhwc ? 1 : 0; ++gi;
    }
    t.n_groups = gi; t.batch = batch; t.S = image_size; t.n_models = M; t.n_class = e->n_class;
    t.b1 = e->d_b1; t.w2t = e->d_w2t; t.b2 = e->d_b2; t.w3 = e->d_w3; t.b3 = e->d_b3;
    t.labels = d_labels; t.votes = d_votes; t.colors = host_colors ? e->d_colors : nullptr; t.color_image = d_color_image;
    const int64_t total = (int64_t)batch * image_size * image_size;
    {
        ProfScope prof(PROF_LABEL, stream);
        if (tiled) {
            const unsigned tiles = (unsigned)((int64_t)batch * (image_size / GAN_TX) * (image_size / GAN_TY));
            dataset_gan_tail_tiled_kernel<<<tiles, 128, 0, stream>>>(t);
        } else {
            dataset_gan_tail_kernel<<<(unsigned)ceil_div64(total, 128), 128, 0, stream>>>(t);
        }
        SIS_CHECK_LAUNCH();
    }
    return SIS_OK;
}

extern "C" int sis_pixel_ensemble_check(sis_pixel_ensemble* e, void* stream_) {
    using namespace sis;
    SIS_REQUIRE(e, "sis_pixel_ensemble_check: null ensemble");
    const cudaError_t sync = cudaStreamSynchronize((cudaStream_t)stream_);
    const unsigned int h = e->d_error ? *(volatile unsigned int*)e->d_error : 0u;
    if (h) { set_error("tcgen05 conv watchdog fired: code 0x%x (%s)", h, cudaGetErrorString(sync)); return SIS_ERR_CUDA; }
    if (sync != cudaSuccess) { set_error("cudaStreamSynchronize failed: %s", cudaGetErrorString(sync)); return SIS_ERR_CUDA; }
    return SIS_OK;
}
