// Activation -> semantic-class labelling, fully on the device, one pass over the activation map per layer.
//   FactorCatalog.predict / pairwise_distance   scf/segmentation/gan_local_edit/factor_catalog.py:47-75
//   partial_flat                                scf/segmentation/gan_local_edit/ptutils.py:25-28
//   predict_clusters (class OR masks)           scf/segmentation/base_cluster_based_dataset_segmenter.py:119-138
//   resize_to_image_size (nearest)              scf/segmentation/base_dataset_segmenter.py:32-42
//   bilinear feature upsample (DatasetGAN path) scf/create_dataset_for_segmentation.py:39-44
// The reference ships every labelled map to the CPU, builds an [N,k,C] temporary, and ships ids back.
//
// HBM-bound (AI ~ k/2 FLOP/B): algorithmic bytes per layer = B*H*W*C*4 (activations, read once, 128-bit
// coalesced along W) + B*H*W (ids) + n_class*B*S*S (masks) + k*C*4.
// Thread = 4 consecutive pixels x one channel slice; the k partial distances of the SLICES slices are
// reduced through shared memory in fixed order (deterministic), then argmin (ties -> lowest k, as
// torch.argmin), class-bit LUT, nearest replication of the masks to SxS, and a warp-aggregated histogram.
#include "common.cuh"
#include "kernels.h"
#include "torgb_common.cuh"
#include <cstring>

namespace sis {

constexpr int LBL_SLICES = 8;

template <int KMAX, int PPT>
struct LabelSmem {
    // centroids transposed [C][KMAX] + reduction scratch [SLICES][KMAX][PPT][32]
    static size_t bytes(int C) { return ((size_t)C * KMAX + (size_t)LBL_SLICES * KMAX * PPT * 32) * sizeof(float) + 64 * sizeof(unsigned); }
};

__device__ __forceinline__ void write_label_outputs(const LabelArgs& a, int b, int y, int x, int id, float best,
                                                    float second) {
    const int64_t n = ((int64_t)b * a.H + y) * a.W + x;
    if (a.ids_u8) a.ids_u8[n] = (uint8_t)id;
    if (a.ids_i64) a.ids_i64[n] = id;
    if (a.margin) a.margin[n] = second - best;
}

// nearest source index as ATen's legacy `nearest`: min(floor(dst * (in/out)), in-1), scale in float.
__device__ __forceinline__ int nearest_src(int dst, float scale, int in_size) {
    int s = (int)floorf((float)dst * scale);
    return s < in_size - 1 ? s : in_size - 1;
}

template <int KMAX, int PPT>
__global__ void __launch_bounds__(32 * LBL_SLICES) label_native_kernel(LabelArgs a) {
    extern __shared__ float smem[];
    float* sc = smem;                                   // [C][KMAX]
    float* red = smem + (size_t)a.C * KMAX;             // [SLICES][KMAX][PPT][32]
    unsigned* shist = reinterpret_cast<unsigned*>(red + LBL_SLICES * KMAX * PPT * 32);  // [KMAX<=64]
    const int lane = threadIdx.x, slice = threadIdx.y;
    const int tid = slice * 32 + lane;
    for (int i = tid; i < a.C * KMAX; i += 32 * LBL_SLICES) {
        int c = i / KMAX, kk = i - c * KMAX;
        sc[i] = kk < a.k ? a.centroids[(int64_t)kk * a.C + c] : 0.0f;
    }
    if (tid < 64) shist[tid] = 0;
    __syncthreads();

    const int64_t hw = (int64_t)a.H * a.W;
    const int64_t groups_per_sample = hw / PPT;
    const int64_t total_groups = groups_per_sample * a.batch;
    const int cps = (a.C + LBL_SLICES - 1) / LBL_SLICES;
    const int c_begin = slice * cps, c_end = min(a.C, c_begin + cps);
    const int rep = a.S / a.H;   // integer replication factor when S % H == 0, else generic path below
    const bool int_ratio = (a.S % a.H == 0) && (a.S % a.W == 0) && (a.H == a.W);

    for (int64_t g0 = (int64_t)blockIdx.x * 32; g0 < total_groups; g0 += (int64_t)gridDim.x * 32) {
        const int64_t g = g0 + lane;
        const bool valid = g < total_groups;
        const int b = valid ? (int)(g / groups_per_sample) : 0;
        const int64_t pix = valid ? (g - (int64_t)b * groups_per_sample) * PPT : 0;
        float acc[KMAX][PPT];
#pragma unroll
        for (int kk = 0; kk < KMAX; ++kk)
#pragma unroll
            for (int p = 0; p < PPT; ++p) acc[kk][p] = 0.0f;
        if (valid) {
            const float* xb = a.act + ((int64_t)b * a.C) * hw + pix;
#pragma unroll 8
            for (int c = c_begin; c < c_end; ++c) {
                float xv[PPT];
                if (PPT == 4) {
                    const float4 v = ld_stream_f4(reinterpret_cast<const float4*>(xb + (int64_t)c * hw));
                    xv[0] = v.x; xv[1] = v.y; xv[2 % PPT] = v.z; xv[3 % PPT] = v.w;
                } else {
#pragma unroll
                    for (int p = 0; p < PPT; ++p) xv[p] = __ldg(xb + (int64_t)c * hw + p);
                }
                const float* cc = sc + (size_t)c * KMAX;
#pragma unroll
                for (int kk = 0; kk < KMAX; ++kk) {
                    const float m = cc[kk];
#pragma unroll
                    for (int p = 0; p < PPT; ++p) {
                        const float df = __fsub_rn(xv[p], m);      // (A - B) ** 2 summed over channels
                        acc[kk][p] = __fmaf_rn(df, df, acc[kk][p]);
                    }
                }
            }
        }
#pragma unroll
        for (int kk = 0; kk < KMAX; ++kk)
#pragma unroll
            for (int p = 0; p < PPT; ++p) red[((slice * KMAX + kk) * PPT + p) * 32 + lane] = acc[kk][p];
        __syncthreads();
        // finalisation: PPT*32 pixels, one thread each (threads 0 .. PPT*32-1)
        if (tid < PPT * 32) {
            const int ln = tid % 32, p = tid / 32;
            const int64_t gg = g0 + ln;
            int id = -1;
            if (gg < total_groups) {
                float best = INFINITY, second = INFINITY;
                id = 0;
                for (int kk = 0; kk < a.k; ++kk) {
                    float d = 0.0f;
#pragma unroll
                    for (int s = 0; s < LBL_SLICES; ++s) d += red[((s * KMAX + kk) * PPT + p) * 32 + ln];
                    if (d < best) { second = best; best = d; id = kk; }
                    else if (d < second) { second = d; }
                }
                const int bb = (int)(gg / groups_per_sample);
                const int64_t px = (gg - (int64_t)bb * groups_per_sample) * PPT + p;
                const int y = (int)(px / a.W), x = (int)(px % a.W);
                write_label_outputs(a, bb, y, x, id, best, second);
                if (a.masks) {
                    const uint32_t bits = __ldg(a.class_bits + id);
                    const int64_t plane = (int64_t)a.S * a.S;
                    if (int_ratio) {
                        for (int j = 0; j < a.n_class; ++j) {
                            const uint8_t m = (bits >> j) & 1u;
                            uint8_t* dst = a.masks + ((int64_t)j * a.batch + bb) * plane + (int64_t)y * rep * a.S + (int64_t)x * rep;
                            if ((rep & 3) == 0 && ((((uintptr_t)a.masks) & 3) == 0)) {
                                const uint32_t word = m * 0x01010101u;   // 4 replicated pixels per store
                                for (int ry = 0; ry < rep; ++ry)
                                    for (int rx = 0; rx < rep / 4; ++rx)
                                        reinterpret_cast<uint32_t*>(dst + (int64_t)ry * a.S)[rx] = word;
                            } else {
                                for (int ry = 0; ry < rep; ++ry)
                                    for (int rx = 0; rx < rep; ++rx) dst[(int64_t)ry * a.S + rx] = m;
                            }
                        }
                    }
                }
            }
            if (a.hist) {
                // warp-aggregated histogram: one shared atomic per (warp, cluster present)
                for (int kk = 0; kk < a.k; ++kk) {
                    const unsigned m = __ballot_sync(0xffffffffu, id == kk);
                    if (ln == 0 && m) atomicAdd(&shist[kk], __popc(m));
                }
            }
        }
        __syncthreads();
    }
    if (a.hist && tid < a.k && shist[tid]) atomicAdd(a.hist + tid, (unsigned long long)shist[tid]);
}

// Wide variant for large maps (>= ~150k pixel quads: enough threads without slicing the channels): one thread = 4
// consecutive pixels x ALL channels.  A block of 256 threads reads 4 KB contiguous per channel plane (DRAM-friendly),
// keeps 8 independent 128-bit loads in flight per thread, needs no shared-memory reduction and no barrier, and
// finalises in registers: packed 4-pixel stores for ids and masks (32-bit for rep 1, 128-bit rows for rep 4).
// RGB = true: the ToRGB of the same tensor (1x1 modulated conv, bias, upsampled skip; model.py:355-364) rides along in
// the same pass: the activation map is read once instead of twice.
// The inner loop is packed fp32x2 (FADD2 / FFMA2 on pixel pairs): the centroid table and the per-sample ToRGB weights
// sit in shared memory pre-splatted as (m, m) pairs, so a channel costs 1 LDG.128 + 2 LDS.128 + 4k packed ops per
// 4 pixels (+ 3 LDS.64 + 6 FFMA2 for RGB): the scalar version of the fused kernel was issue-bound at half the speed.
// KMAX > 8 switches to the expanded form d_k = |c_k|^2 - 2 x.c_k (+ |x|^2, common to all k and therefore dropped: ids and
// margins are unchanged): k packed FMAs per pixel pair per channel instead of 2k.  At k ~ 20 the direct form needs more
// fp32 FMA throughput than the SM has per HBM byte; SURVEY.md §7 measured <= 1 flip per 131 k pixels (never at margin
// > 1e-3) between the two forms.  k <= 8 keeps the reference's (A - B)^2 form, which is memory-bound anyway.
// SPLIT = 4 (maps with fewer than two blocks per SM, e.g. 64^2 at batch 32: 128 blocks on 148 SMs at 34-48 % of the DRAM
// peak): a block is 64 quads x 4 channel slices, each slice accumulates a quarter of the channels for the same pixels and
// slices 1..3 hand their partial sums to slice 0 through shared memory (added in slice order: deterministic), which
// finalises as before: four times the blocks and loads in flight for the same bytes.
template <int KMAX, bool RGB, int SPLIT = 1>
__global__ void __launch_bounds__(256, (KMAX > 8 ? 2 : 3)) label_wide_kernel(LabelArgs a, ToRgbArgs g) {
    constexpr bool EXPANDED = KMAX > 8;
    constexpr int QPB = 256 / SPLIT;                                            // quads per block
    extern __shared__ float smem[];
    float2* sc2 = reinterpret_cast<float2*>(smem);                              // [C][KMAX] splatted centroids
    float2* sw2 = sc2 + (size_t)a.C * KMAX;                                     // [C][3] splatted scale*W*s of this sample (RGB)
    // the tables and (SPLIT > 1) the partial sums of slices 1.. share one region: the sums are written after the channel loop
    constexpr int RED_FLOATS = (SPLIT - 1) * (256 / SPLIT) * (KMAX * 4 + (RGB ? 12 : 0));
    const int tab_floats = a.C * KMAX * 2 + (RGB ? 6 * a.C : 0);
    unsigned* shist = reinterpret_cast<unsigned*>(smem + (tab_floats > RED_FLOATS ? tab_floats : RED_FLOATS));  // [KMAX]
    float* scn = reinterpret_cast<float*>(shist + KMAX);                        // [KMAX] |c_k|^2 (expanded form)
    const int tid = threadIdx.x;
    const int64_t hw = (int64_t)a.H * a.W;
    const int64_t quads_per_sample = hw >> 2;                                   // a multiple of 256 (checked on the host):
    const int64_t total = quads_per_sample * a.batch;                           // a block never straddles two samples
    const int slice = tid / QPB;
    const int64_t q = (int64_t)blockIdx.x * QPB + (tid - slice * QPB);
    const int b_blk = (int)(((int64_t)blockIdx.x * QPB) / quads_per_sample);
    for (int i = tid; i < a.C * KMAX; i += 256) {
        int c = i / KMAX, kk = i - c * KMAX;
        const float m = kk < a.k ? a.centroids[(int64_t)kk * a.C + c] : 0.0f;
        if (EXPANDED) reinterpret_cast<float*>(sc2)[i] = m;     // [C][KMAX] floats: FFMA2 operands are (m_k, m_k+1) pairs
        else sc2[i] = make_float2(m, m);                          // [C][KMAX] pixel-pair splats
    }
    if (RGB) {
        const float* sb = g.s + (int64_t)b_blk * a.C;
        for (int i = tid; i < 3 * a.C; i += 256) {
            const int c = i / 3, j = i - c * 3;
            const float w = __fmul_rn(g.w[j * a.C + c], sb[c]);                 // (scale*W) * s, as the reference orders it
            sw2[i] = make_float2(w, w);
        }
    }
    if (tid < KMAX) {
        shist[tid] = 0;
        float cn = 0.0f;
        if (EXPANDED && tid < a.k)
            for (int c = 0; c < a.C; ++c) { const float m = a.centroids[(int64_t)tid * a.C + c]; cn = fmaf(m, m, cn); }
        scn[tid] = cn;
    }
    __syncthreads();
    const bool valid = q < total;
    int ids[4] = {-1, -1, -1, -1};
    if (valid) {
        const int b = b_blk;
        const int64_t pix = (q - (int64_t)b * quads_per_sample) << 2;
        const float* xb = a.act + ((int64_t)b * a.C) * hw + pix;
        // direct form: acc2[k][pixel pair];  expanded form: accK[k pair][pixel]
        float2 acc2[EXPANDED ? 1 : KMAX][2];
        float2 accK[EXPANDED ? KMAX / 2 : 1][4];
        float2 rgb2[3][2];
#pragma unroll
        for (int kk = 0; kk < (EXPANDED ? 1 : KMAX); ++kk) { acc2[kk][0] = make_float2(0.f, 0.f); acc2[kk][1] = make_float2(0.f, 0.f); }
#pragma unroll
        for (int kk = 0; kk < (EXPANDED ? KMAX / 2 : 1); ++kk)
#pragma unroll
            for (int p = 0; p < 4; ++p) accK[kk][p] = make_float2(0.f, 0.f);
#pragma unroll
        for (int j = 0; j < 3; ++j) { rgb2[j][0] = make_float2(0.f, 0.f); rgb2[j][1] = make_float2(0.f, 0.f); }
        const int c_per = a.C / SPLIT, c_begin = slice * c_per, c_end = c_begin + c_per;     // C % SPLIT == 0 (host-side check)
#pragma unroll 8
        for (int c = c_begin; c < c_end; ++c) {
            const float4 v = ld_stream_f4(reinterpret_cast<const float4*>(xb + (int64_t)c * hw));
            const float2 x01 = make_float2(v.x, v.y), x23 = make_float2(v.z, v.w);
            if (RGB) {
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    const float2 w = sw2[c * 3 + j];
                    rgb2[j][0] = pk_fma(w, x01, rgb2[j][0]);
                    rgb2[j][1] = pk_fma(w, x23, rgb2[j][1]);
                }
            }
            if (EXPANDED) {
                const float2* cc = reinterpret_cast<const float2*>(reinterpret_cast<const float*>(sc2) + (size_t)c * KMAX);
                const float2 xs[4] = {make_float2(v.x, v.x), make_float2(v.y, v.y), make_float2(v.z, v.z), make_float2(v.w, v.w)};
#pragma unroll
                for (int kk = 0; kk < KMAX / 2; ++kk) {
                    const float2 m = cc[kk];                                     // (c_2kk, c_2kk+1)
#pragma unroll
                    for (int p = 0; p < 4; ++p) accK[kk][p] = pk_fma(xs[p], m, accK[kk][p]);   // x . c_k
                }
            } else {
                const float2* cc = sc2 + (size_t)c * KMAX;
#pragma unroll
                for (int kk = 0; kk < KMAX; ++kk) {
                    const float2 m = cc[kk];
                    const float2 d0 = pk_sub(x01, m), d1 = pk_sub(x23, m);      // (A - B) ** 2 summed over channels
                    acc2[kk][0] = pk_fma(d0, d0, acc2[kk][0]);
                    acc2[kk][1] = pk_fma(d1, d1, acc2[kk][1]);
                }
            }
        }
        if (SPLIT > 1) {
            // every thread of the block is in range (quads per sample is a multiple of 256): the barrier is uniform
            constexpr int NACC = KMAX * 4 + (RGB ? 12 : 0);
            float* red = smem;                                                   // [SPLIT - 1][QPB][NACC], conflict-free by quad
            const int ql = tid - slice * QPB;
            __syncthreads();                                                     // every slice is done with the tables
            if (slice > 0) {
                float* r = red + ((size_t)(slice - 1) * NACC) * QPB + ql;
                if (EXPANDED) {
#pragma unroll
                    for (int kk = 0; kk < KMAX / 2; ++kk)
#pragma unroll
                        for (int p = 0; p < 4; ++p) { r[(kk * 8 + p * 2) * QPB] = accK[kk][p].x; r[(kk * 8 + p * 2 + 1) * QPB] = accK[kk][p].y; }
                } else {
#pragma unroll
                    for (int kk = 0; kk < KMAX; ++kk) {
                        r[(kk * 4 + 0) * QPB] = acc2[kk][0].x; r[(kk * 4 + 1) * QPB] = acc2[kk][0].y;
                        r[(kk * 4 + 2) * QPB] = acc2[kk][1].x; r[(kk * 4 + 3) * QPB] = acc2[kk][1].y;
                    }
                }
                if (RGB) {
#pragma unroll
                    for (int j = 0; j < 3; ++j) {
                        r[(KMAX * 4 + j * 4 + 0) * QPB] = rgb2[j][0].x; r[(KMAX * 4 + j * 4 + 1) * QPB] = rgb2[j][0].y;
                        r[(KMAX * 4 + j * 4 + 2) * QPB] = rgb2[j][1].x; r[(KMAX * 4 + j * 4 + 3) * QPB] = rgb2[j][1].y;
                    }
                }
            }
            __syncthreads();
            if (slice == 0) {
#pragma unroll
                for (int sl = 0; sl < SPLIT - 1; ++sl) {
                    const float* r = red + ((size_t)sl * NACC) * QPB + ql;
                    if (EXPANDED) {
#pragma unroll
                        for (int kk = 0; kk < KMAX / 2; ++kk)
#pragma unroll
                            for (int p = 0; p < 4; ++p) { accK[kk][p].x += r[(kk * 8 + p * 2) * QPB]; accK[kk][p].y += r[(kk * 8 + p * 2 + 1) * QPB]; }
                    } else {
#pragma unroll
                        for (int kk = 0; kk < KMAX; ++kk) {
                            acc2[kk][0].x += r[(kk * 4 + 0) * QPB]; acc2[kk][0].y += r[(kk * 4 + 1) * QPB];
                            acc2[kk][1].x += r[(kk * 4 + 2) * QPB]; acc2[kk][1].y += r[(kk * 4 + 3) * QPB];
                        }
                    }
                    if (RGB) {
#pragma unroll
                        for (int j = 0; j < 3; ++j) {
                            rgb2[j][0].x += r[(KMAX * 4 + j * 4 + 0) * QPB]; rgb2[j][0].y += r[(KMAX * 4 + j * 4 + 1) * QPB];
                            rgb2[j][1].x += r[(KMAX * 4 + j * 4 + 2) * QPB]; rgb2[j][1].y += r[(KMAX * 4 + j * 4 + 3) * QPB];
                        }
                    }
                }
            }
        }
        if (slice == 0) {
        float acc[KMAX][4];
        if (EXPANDED) {
#pragma unroll
            for (int kk = 0; kk < KMAX; ++kk) {
                const float cn = scn[kk];                                        // |c_k|^2
#pragma unroll
                for (int p = 0; p < 4; ++p) {
                    const float dot = (kk & 1) ? accK[kk / 2][p].y : accK[kk / 2][p].x;
                    acc[kk][p] = fmaf(-2.0f, dot, cn);
                }
            }
        } else {
#pragma unroll
            for (int kk = 0; kk < KMAX; ++kk) { acc[kk][0] = acc2[kk][0].x; acc[kk][1] = acc2[kk][0].y; acc[kk][2] = acc2[kk][1].x; acc[kk][3] = acc2[kk][1].y; }
        }
        float rgb[3][4];
#pragma unroll
        for (int j = 0; j < 3; ++j) { rgb[j][0] = rgb2[j][0].x; rgb[j][1] = rgb2[j][0].y; rgb[j][2] = rgb2[j][1].x; rgb[j][3] = rgb2[j][1].y; }
        float best[4], second[4];
#pragma unroll
        for (int p = 0; p < 4; ++p) { best[p] = INFINITY; second[p] = INFINITY; ids[p] = 0; }
#pragma unroll
        for (int kk = 0; kk < KMAX; ++kk) {
            if (kk < a.k) {
#pragma unroll
                for (int p = 0; p < 4; ++p) {
                    const float d = acc[kk][p];
                    if (d < best[p]) { second[p] = best[p]; best[p] = d; ids[p] = kk; }
                    else if (d < second[p]) { second[p] = d; }
                }
            }
        }
        if (RGB) {
            const int y = (int)(pix / a.W), x = (int)(pix - (int64_t)y * a.W);
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                float o[4];
#pragma unroll
                for (int p = 0; p < 4; ++p) {
                    float v = __fadd_rn(rgb[j][p], g.bias[j]);
                    if (g.skip) v = __fadd_rn(v, torgb_skip_tap(g, g.skip + ((int64_t)b * 3 + j) * (hw >> 2), y, x + p));
                    o[p] = v;
                }
                *reinterpret_cast<float4*>(g.out + ((int64_t)b * 3 + j) * hw + pix) = make_float4(o[0], o[1], o[2], o[3]);
            }
        }
        const int64_t n0 = (int64_t)b * hw + pix;       // flat [B,H,W] index of the first pixel
        if (a.ids_u8) *reinterpret_cast<uint32_t*>(a.ids_u8 + n0) = (uint32_t)ids[0] | ((uint32_t)ids[1] << 8) | ((uint32_t)ids[2] << 16) | ((uint32_t)ids[3] << 24);
        if (a.ids_i64) {
#pragma unroll
            for (int p = 0; p < 4; ++p) a.ids_i64[n0 + p] = ids[p];
        }
        if (a.margin) *reinterpret_cast<float4*>(a.margin + n0) = make_float4(second[0] - best[0], second[1] - best[1], second[2] - best[2], second[3] - best[3]);
        if (a.masks) {
            uint32_t bits[4];
#pragma unroll
            for (int p = 0; p < 4; ++p) bits[p] = __ldg(a.class_bits + ids[p]);
            const int rep = a.S / a.H;
            const int y = (int)(pix / a.W), x = (int)(pix - (int64_t)y * a.W);
            const int64_t plane = (int64_t)a.S * a.S;
            for (int j = 0; j < a.n_class; ++j) {
                uint8_t* dst = a.masks + ((int64_t)j * a.batch + b) * plane + (int64_t)y * rep * a.S + (int64_t)x * rep;
                const uint32_t m0 = (bits[0] >> j) & 1u, m1 = (bits[1] >> j) & 1u, m2 = (bits[2] >> j) & 1u, m3 = (bits[3] >> j) & 1u;
                if (rep == 1) {
                    *reinterpret_cast<uint32_t*>(dst) = m0 | (m1 << 8) | (m2 << 16) | (m3 << 24);
                } else if (rep == 4) {
                    const uint4 row = make_uint4(m0 * 0x01010101u, m1 * 0x01010101u, m2 * 0x01010101u, m3 * 0x01010101u);
#pragma unroll
                    for (int ry = 0; ry < 4; ++ry) *reinterpret_cast<uint4*>(dst + (int64_t)ry * a.S) = row;
                } else {
                    const uint32_t mm[4] = {m0, m1, m2, m3};
                    for (int ry = 0; ry < rep; ++ry)
                        for (int p = 0; p < 4; ++p)
                            for (int rx = 0; rx < rep; ++rx) dst[(int64_t)ry * a.S + p * rep + rx] = (uint8_t)mm[p];
                }
            }
        }
        }      // slice 0
    }
    if (a.hist) {
        for (int kk = 0; kk < a.k; ++kk) {
            const unsigned c = (unsigned)(ids[0] == kk) + (unsigned)(ids[1] == kk) + (unsigned)(ids[2] == kk) + (unsigned)(ids[3] == kk);
            const unsigned tot = __reduce_add_sync(0xffffffffu, c);
            if ((tid & 31) == 0 && tot) atomicAdd(&shist[kk], tot);
        }
        __syncthreads();
        if (tid < a.k && shist[tid]) atomicAdd(a.hist + tid, (unsigned long long)shist[tid]);
    }
}

// masks for a non-integer resize ratio: gather from the ids (rare; power-of-two sizes never take it)
__global__ void __launch_bounds__(256) masks_gather_kernel(uint8_t* __restrict__ masks, const uint8_t* __restrict__ ids,
                                                           const uint32_t* __restrict__ class_bits, int n_class,
                                                           int batch, int H, int W, int S) {
    const int64_t total = (int64_t)batch * S * S;
    const float sy = (float)H / (float)S, sx = (float)W / (float)S;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int x = (int)(i % S);
        const int y = (int)((i / S) % S);
        const int b = (int)(i / ((int64_t)S * S));
        const int id = ids[((int64_t)b * H + nearest_src(y, sy, H)) * W + nearest_src(x, sx, W)];
        const uint32_t bits = class_bits[id];
        for (int j = 0; j < n_class; ++j) masks[((int64_t)j * batch + b) * S * S + (int64_t)y * S + x] = (bits >> j) & 1u;
    }
}

// mode 1: bilinear upsample (align_corners=False, ATen's area_pixel_compute_source_index) of the features to
// SxS, then assign.  One thread per output pixel, centroids in shared memory; the 4 taps are gathered per
// channel (each source element is re-read ~ (S/H)^2 times but from L1/L2: DRAM traffic stays ~ one pass).
template <int KMAX>
__global__ void __launch_bounds__(256) label_bilinear_kernel(LabelArgs a) {
    extern __shared__ float smem[];
    float* sc = smem;  // [C][KMAX]
    for (int i = threadIdx.x; i < a.C * KMAX; i += blockDim.x) {
        int c = i / KMAX, kk = i - c * KMAX;
        sc[i] = kk < a.k ? a.centroids[(int64_t)kk * a.C + c] : 0.0f;
    }
    __syncthreads();
    const int S = a.S;
    const int64_t total = (int64_t)a.batch * S * S;
    const float scale_h = (float)a.H / (float)S, scale_w = (float)a.W / (float)S;  // 1/scale_factor
    const int64_t hw = (int64_t)a.H * a.W;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int x = (int)(i % S), y = (int)((i / S) % S), b = (int)(i / ((int64_t)S * S));
        float fy = fmaxf(scale_h * ((float)y + 0.5f) - 0.5f, 0.0f);
        float fx = fmaxf(scale_w * ((float)x + 0.5f) - 0.5f, 0.0f);
        const int y0 = (int)fy, x0 = (int)fx;
        const int y1 = y0 + (y0 < a.H - 1 ? 1 : 0), x1 = x0 + (x0 < a.W - 1 ? 1 : 0);
        const float ly = fy - (float)y0, lx = fx - (float)x0, hy = 1.0f - ly, hx = 1.0f - lx;
        const float* xb = a.act + (int64_t)b * a.C * hw;
        float acc[KMAX];
#pragma unroll
        for (int kk = 0; kk < KMAX; ++kk) acc[kk] = 0.0f;
        for (int c = 0; c < a.C; ++c) {
            const float* pc = xb + (int64_t)c * hw;
            const float v00 = __ldg(pc + (int64_t)y0 * a.W + x0), v01 = __ldg(pc + (int64_t)y0 * a.W + x1);
            const float v10 = __ldg(pc + (int64_t)y1 * a.W + x0), v11 = __ldg(pc + (int64_t)y1 * a.W + x1);
            // ATen upsample_bilinear2d: h0lambda*(w0lambda*v00 + w1lambda*v01) + h1lambda*(w0lambda*v10 + w1lambda*v11)
            const float v = __fadd_rn(__fmul_rn(hy, __fadd_rn(__fmul_rn(hx, v00), __fmul_rn(lx, v01))),
                                      __fmul_rn(ly, __fadd_rn(__fmul_rn(hx, v10), __fmul_rn(lx, v11))));
            const float* cc = sc + (size_t)c * KMAX;
#pragma unroll
            for (int kk = 0; kk < KMAX; ++kk) {
                const float df = __fsub_rn(v, cc[kk]);
                acc[kk] = __fmaf_rn(df, df, acc[kk]);
            }
        }
        float best = INFINITY, second = INFINITY;
        int id = 0;
        for (int kk = 0; kk < a.k; ++kk) {
            const float d = acc[kk];
            if (d < best) { second = best; best = d; id = kk; }
            else if (d < second) { second = d; }
        }
        if (a.ids_u8) a.ids_u8[i] = (uint8_t)id;
        if (a.ids_i64) a.ids_i64[i] = id;
        if (a.margin) a.margin[i] = second - best;
        if (a.masks) {
            const uint32_t bits = __ldg(a.class_bits + id);
            for (int j = 0; j < a.n_class; ++j)
                a.masks[((int64_t)j * a.batch + b) * S * S + (int64_t)y * S + x] = (bits >> j) & 1u;
        }
        if (a.hist) atomicAdd(a.hist + id, 1ull);
    }
}

__global__ void __launch_bounds__(256) class_masks_from_ids_kernel(uint8_t* __restrict__ masks, const int64_t* __restrict__ ids,
                                                                   const uint32_t* __restrict__ class_bits, int k,
                                                                   int n_class, int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t id = ids[i];
        const uint32_t bits = (id >= 0 && id < k) ? class_bits[id] : 0u;
        for (int j = 0; j < n_class; ++j) masks[(int64_t)j * n + i] = (bits >> j) & 1u;
    }
}

__global__ void __launch_bounds__(256) nearest_resize_u8_kernel(uint8_t* __restrict__ out, const uint8_t* __restrict__ in,
                                                                int64_t planes, int h, int w, int oh, int ow) {
    const float sy = (float)h / (float)oh, sx = (float)w / (float)ow;
    const int64_t total = planes * oh * ow;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int x = (int)(i % ow), y = (int)((i / ow) % oh);
        const int64_t p = i / ((int64_t)ow * oh);
        out[i] = in[(p * h + nearest_src(y, sy, h)) * w + nearest_src(x, sx, w)];
    }
}

__global__ void __launch_bounds__(256) or_u8_kernel(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        dst[i] = dst[i] | src[i];
}

static int flat_grid(int64_t n, int per_block = 256) {
    int64_t b = ceil_div64(n, per_block);
    int64_t cap = (int64_t)kNumSMs * 8;
    return (int)(b < 1 ? 1 : (b < cap ? b : cap));
}

template <int KMAX, int PPT>
static int launch_native(const LabelArgs& a, cudaStream_t stream) {
    size_t smem = LabelSmem<KMAX, PPT>::bytes(a.C);
    auto kern = label_native_kernel<KMAX, PPT>;
    if (smem > 48 * 1024) SIS_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t groups = (int64_t)a.H * a.W / PPT * a.batch;
    int64_t blocks = ceil_div64(groups, 32);
    int64_t cap = (int64_t)kNumSMs * 4;
    int grid = (int)(blocks < cap ? blocks : cap);
    kern<<<grid, dim3(32, LBL_SLICES), smem, stream>>>(a);
    SIS_CHECK_LAUNCH();
    return SIS_OK;
}

template <int KMAX, bool RGB, int SPLIT>
static int launch_wide_split(const LabelArgs& a, const ToRgbArgs& g, cudaStream_t stream) {
    constexpr int QPB = 256 / SPLIT, NACC = KMAX * 4 + (RGB ? 12 : 0);
    const size_t tab = (size_t)a.C * KMAX * 2 + (RGB ? 6 * a.C : 0), red = (size_t)(SPLIT - 1) * QPB * NACC;   // share one region
    size_t smem = ((tab > red ? tab : red) + 2 * KMAX) * sizeof(float);
    auto kern = label_wide_kernel<KMAX, RGB, SPLIT>;
    if (smem > 48 * 1024) SIS_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t quads = (int64_t)a.H * a.W / 4 * a.batch;
    kern<<<(unsigned)ceil_div64(quads, QPB), 256, smem, stream>>>(a, g);
    SIS_CHECK_LAUNCH();
    return SIS_OK;
}

template <int KMAX, bool RGB>
static int launch_wide_impl(const LabelArgs& a, const ToRgbArgs& g, cudaStream_t stream) {
    // fewer than two blocks per SM: split the channels over four thread groups (measured, 64^2 maps at batch 32:
    // 68 -> 59 us, 99 -> 80 us with the ToRGB fused)
    const int64_t quads = (int64_t)a.H * a.W / 4 * a.batch;
    if (quads / 256 < 2 * kNumSMs && a.C % 4 == 0) return launch_wide_split<KMAX, RGB, 4>(a, g, stream);
    return launch_wide_split<KMAX, RGB, 1>(a, g, stream);
}
template <int KMAX>
static int launch_wide(const LabelArgs& a, const ToRgbArgs* g, cudaStream_t stream) {
    if (g) return launch_wide_impl<KMAX, true>(a, *g, stream);
    ToRgbArgs none;
    memset(&none, 0, sizeof(none));
    return launch_wide_impl<KMAX, false>(a, none, stream);
}

template <int KMAX>
static int launch_bilinear(const LabelArgs& a, cudaStream_t stream) {
    size_t smem = (size_t)a.C * KMAX * sizeof(float);
    auto kern = label_bilinear_kernel<KMAX>;
    if (smem > 48 * 1024) SIS_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<flat_grid((int64_t)a.batch * a.S * a.S), 256, smem, stream>>>(a);
    SIS_CHECK_LAUNCH();
    return SIS_OK;
}

}  // namespace sis

using namespace sis;

namespace sis {

// pixel quads from which the wide kernel is used; measured: it wins from ~24 k quads (64^2 maps at batch 32: 80 -> 67 us)
constexpr int64_t kWideMinQuads = (int64_t)kNumSMs * 160;

int launch_label(const LabelArgs& a_in, int mode, const ToRgbArgs* fuse_rgb, bool* fused, cudaStream_t stream) {
    LabelArgs a = a_in;
    if (fused) *fused = false;
    const int batch = a.batch, channels = a.C, h = a.H, w = a.W, k = a.k, n_class = a.n_class, image_size = a.S;
    SIS_REQUIRE(batch >= 0 && channels >= 1 && h >= 0 && w >= 0, "label_assign: bad shape");
    SIS_REQUIRE(k >= 1 && k <= 64, "label_assign: k must be in [1, 64] (got %d)", k);
    SIS_REQUIRE(n_class >= 0 && n_class <= 32, "label_assign: n_class must be <= 32");
    SIS_REQUIRE(mode == 0 || mode == 1, "label_assign: mode must be 0 or 1");
    SIS_REQUIRE(!a.masks || (a.class_bits && image_size >= h && image_size >= w),
                "label_assign: masks need class bits and image_size >= map size");
    SIS_REQUIRE((size_t)channels * 64 * 4 <= 200 * 1024 || k <= 32, "label_assign: centroid table does not fit shared memory");
    if ((int64_t)batch * h * w == 0) return SIS_OK;
    SIS_REQUIRE(a.act && a.centroids, "label_assign: activations / centroids must be CUDA tensors (null pointer)");
    ProfScope prof(PROF_LABEL, stream);
    if (mode == 1) {
        SIS_REQUIRE(image_size >= 1, "label_assign: image_size required for mode 1");
        if (k <= 4) return launch_bilinear<4>(a, stream);
        if (k <= 8) return launch_bilinear<8>(a, stream);
        if (k <= 16) return launch_bilinear<16>(a, stream);
        if (k <= 32) return launch_bilinear<32>(a, stream);
        return launch_bilinear<64>(a, stream);
    }
    const bool vec4 = ((h * w) % 4 == 0) && ((((uintptr_t)a.act) & 15) == 0);
    const bool int_ratio = a.masks && (image_size % h == 0) && (image_size % w == 0) && (h == w);
    uint8_t* d_masks = a.masks;
    bool gather = a.masks && !int_ratio;
    if (gather) {
        // non-integer ratio: masks are gathered from the ids afterwards
        SIS_REQUIRE(a.ids_u8 != nullptr, "label_assign: non-integer resize ratio needs d_ids_u8");
        a.masks = nullptr;
    }
    int st;
    // wide path: enough pixel quads to fill the GPU without slicing channels, integer (or no) mask replication,
    // rows that are a multiple of 4 pixels, k small enough for 4 x k register accumulators
    const int64_t quads = (int64_t)h * w / 4 * batch;
    const bool wide_ok = vec4 && k <= 24 && (size_t)channels * 24 * 8 <= 160 * 1024 && w % 4 == 0 && quads >= kWideMinQuads && ((int64_t)h * w / 4) % 256 == 0 &&
                         (!a.masks || (int_ratio && ((((uintptr_t)a.masks) & 15) == 0))) &&
                         (!a.ids_u8 || ((((uintptr_t)a.ids_u8) & 3) == 0)) && (!a.margin || ((((uintptr_t)a.margin) & 15) == 0));
    if (wide_ok) {
        const ToRgbArgs* g = (fuse_rgb && fuse_rgb->x == a.act && fuse_rgb->C == channels && fuse_rgb->H == h && fuse_rgb->W == w &&
                              fuse_rgb->batch == batch) ? fuse_rgb : nullptr;
        if (k <= 4) st = launch_wide<4>(a, g, stream);
        else if (k <= 8) st = launch_wide<8>(a, g, stream);
        else if (k <= 16) st = launch_wide<16>(a, g, stream);
        else st = launch_wide<24>(a, g, stream);
        if (g && fused && st == SIS_OK) *fused = true;
    } else if (vec4) {
        if (k <= 4) st = launch_native<4, 4>(a, stream);
        else if (k <= 8) st = launch_native<8, 4>(a, stream);
        else if (k <= 16) st = launch_native<16, 4>(a, stream);
        else if (k <= 32) st = launch_native<32, 2>(a, stream);
        else st = launch_native<64, 1>(a, stream);
    } else {
        if (k <= 8) st = launch_native<8, 1>(a, stream);
        else if (k <= 32) st = launch_native<32, 1>(a, stream);
        else st = launch_native<64, 1>(a, stream);
    }
    SIS_PROPAGATE(st);
    if (gather) {
        masks_gather_kernel<<<flat_grid((int64_t)batch * image_size * image_size), 256, 0, stream>>>(
            d_masks, a.ids_u8, a.class_bits, n_class, batch, h, w, image_size);
        SIS_CHECK_LAUNCH();
    }
    return SIS_OK;
}

}  // namespace sis

extern "C" int sis_label_assign(const float* d_act, int batch, int channels, int h, int w, const float* d_centroids,
                                int k, const uint32_t* d_cluster_class_bits, int n_class, int image_size, int mode,
                                uint8_t* d_ids_u8, int64_t* d_ids_i64, uint8_t* d_masks, float* d_margin,
                                unsigned long long* d_hist, void* stream_) {
    LabelArgs a;
    a.act = d_act; a.batch = batch; a.C = channels; a.H = h; a.W = w; a.centroids = d_centroids; a.k = k;
    a.class_bits = d_cluster_class_bits; a.n_class = n_class; a.S = image_size;
    a.ids_u8 = d_ids_u8; a.ids_i64 = d_ids_i64; a.masks = d_masks; a.margin = d_margin; a.hist = d_hist;
    return launch_label(a, mode, nullptr, nullptr, (cudaStream_t)stream_);
}

extern "C" int sis_class_masks_from_ids(const int64_t* d_ids, int64_t n, const uint32_t* d_cluster_class_bits, int k,
                                        int n_class, uint8_t* d_masks, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    SIS_REQUIRE(n >= 0 && k >= 0 && n_class >= 0 && n_class <= 32, "class_masks_from_ids: bad arguments");
    if (n == 0 || n_class == 0) return SIS_OK;
    SIS_REQUIRE(d_ids && d_cluster_class_bits && d_masks, "class_masks_from_ids: null pointer");
    class_masks_from_ids_kernel<<<flat_grid(n), 256, 0, stream>>>(d_masks, d_ids, d_cluster_class_bits, k, n_class, n);
    SIS_CHECK_LAUNCH();
    return SIS_OK;
}

extern "C" int sis_nearest_resize_u8(const uint8_t* d_in, int64_t planes, int h, int w, int out_h, int out_w,
                                     uint8_t* d_out, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    SIS_REQUIRE(planes >= 0 && h >= 1 && w >= 1 && out_h >= 0 && out_w >= 0, "nearest_resize_u8: bad shape");
    if (planes * out_h * out_w == 0) return SIS_OK;
    SIS_REQUIRE(d_in && d_out, "nearest_resize_u8: null pointer");
    nearest_resize_u8_kernel<<<flat_grid(planes * out_h * out_w), 256, 0, stream>>>(d_out, d_in, planes, h, w, out_h, out_w);
    SIS_CHECK_LAUNCH();
    return SIS_OK;
}

extern "C" int sis_or_u8(uint8_t* d_dst, const uint8_t* d_src, int64_t n, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    SIS_REQUIRE(n >= 0, "or_u8: negative size");
    if (n == 0) return SIS_OK;
    SIS_REQUIRE(d_dst && d_src, "or_u8: null pointer");
    or_u8_kernel<<<flat_grid(n), 256, 0, stream>>>(d_dst, d_src, n);
    SIS_CHECK_LAUNCH();
    return SIS_OK;
}
