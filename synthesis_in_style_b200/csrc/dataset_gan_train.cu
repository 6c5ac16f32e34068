// Training of DatasetGAN pixel-classifier ensembles (sis_pixel_train_*): every network of the ensemble advances in the
// same three launches per step, and the host enqueues a chunk of steps without synchronising.
//
// One step of network m (the recipe of DatasetGAN's train_interpreter.py, restated by oracle/dataset_gan_train_oracle.py):
//   (a) pt_forward_kernel, grid (K slices, networks): draw the step's B pixels from the network's epoch permutation,
//       gather their F features (every capture bilinearly upsampled to S x S at that pixel, as the labeller's tail kernel
//       does) for a 128-channel slice of F, keep the rows, and write the slice's partial first-layer product.
//   (b) pt_tail_kernel, one CTA per network: sum the partials in slice order, then ReLU -> BatchNorm(train) -> Linear ->
//       ReLU -> BatchNorm(train) -> Linear -> mean softmax cross-entropy, the backward pass through all of it (batch
//       statistics terms included), the running statistics, the loss and the stop rule.
//   (c) pt_update_kernel, grid (K slices, networks): dW1 = dh1^T f for the slice and Adam on W1; slice 0 also runs Adam
//       on the small tensors.
// All arithmetic is fp32 FFMA and every sum has a fixed order, so a network's result depends neither on the networks
// it shares a launch with nor on how its steps are split into calls.
#include <cmath>
#include <map>
#include <string>
#include <vector>
#include "common.cuh"
#include "dataset_gan_common.cuh"
#include "../../include/sis_b200.h"

namespace sis {
namespace {

constexpr int kPtMaxBatch = 64;
constexpr int kPtMaxLayers = 20;
constexpr int kPtKSlice = 128;                 // channels of F per CTA in (a) and (c): a function of F only
constexpr int kPtThreads = 256;
constexpr int kPtFStride = kPtMaxBatch + 4;    // s_fT[kk][p]
constexpr int kPtWStride = GAN_H1 + 4;         // s_wT[kk][j]
constexpr double kPtLr = 1e-3;
constexpr double kPtBeta1Exact = 0.9, kPtBeta2Exact = 0.999;
constexpr float kPtBeta2 = 0.999f, kPtEps = 1e-8f;
constexpr float kPtBnEps = 1e-5f, kPtBnMomentum = 0.1f;
constexpr int kPtFirstRuleEpoch = 4;           // DatasetGAN: `if epoch > 3`
constexpr int kPtPatience = 50;                // DatasetGAN: `if break_count > 50`

// Offsets of the small trainable tensors in a network's packed vector (torch layouts: Linear weights [out][in]).
constexpr int kOffB1 = 0, kOffG1 = 128, kOffBe1 = 256, kOffW2 = 384, kOffB2 = kOffW2 + GAN_H2 * GAN_H1, kOffG2 = kOffB2 + 32,
              kOffBe2 = kOffG2 + 32, kOffW3 = kOffBe2 + 32;
__host__ __device__ constexpr int off_b3(int n_class) { return kOffW3 + GAN_H2 * n_class; }
__host__ __device__ constexpr int small_size(int n_class) { return off_b3(n_class) + n_class; }
constexpr int kRstat = 2 * GAN_H1 + 2 * GAN_H2;     // running_mean1, running_var1, running_mean2, running_var2

struct PtState {
    uint64_t key;              // the network's draw key
    int64_t steps_done;        // optimiser steps applied (= num_batches_tracked)
    int64_t max_steps;         // epochs * steps per epoch
    int32_t done;              // 0 training, 1 stopped: the word the host polls
    int32_t ran;               // the tail ran the current step: the update applies it
    int32_t break_count;
    float best_loss;
};

struct PtArgs {
    const float* act[kPtMaxLayers];
    int chan[kPtMaxLayers], res[kPtMaxLayers], coff[kPtMaxLayers + 1];
    int n_layers;
    const uint8_t* labels;     // [A][S][S]
    int S, F, n_class, B, n_split, half_bits;
    int64_t n_pix, steps_per_epoch;
    float* w1;                 // [M][128][F]
    float* m1; float* v1;
    float* small; float* msmall; float* vsmall; float* gsmall;   // [M][P]
    float* rstat;              // [M][kRstat]
    float* feat;               // [M][B][F]
    float* part;               // [M][n_split][B][128]
    float* dh1;                // [M][B][128]
    int32_t* pix;              // [M][B]
    float* loss;               // [M][max_steps]
    PtState* st;               // [M]
};

__host__ __device__ __forceinline__ uint64_t pt_mix(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

// Position i of an epoch's permutation of [0, n): a 4-round Feistel network over 2 * half bits keyed by the epoch key,
// cycle-walked back into [0, n).  A bijection of [0, n), a pure function of (key, epoch, i).
__device__ __forceinline__ int64_t pt_permute(uint64_t key, uint64_t epoch, uint64_t i, uint64_t n, int half) {
    const uint64_t ekey = pt_mix(key ^ pt_mix(epoch));
    const uint64_t mask = (1ull << half) - 1ull;
    uint64_t x = i;
    do {
        uint64_t l = x >> half, r = x & mask;
        for (uint64_t round = 0; round < 4; ++round) {
            const uint64_t f = pt_mix(ekey ^ (round << 56) ^ r) & mask;
            const uint64_t nl = r;
            r = l ^ f;
            l = nl;
        }
        x = (l << half) | r;
    } while (x >= n);
    return (int64_t)x;
}

__global__ void __launch_bounds__(kPtThreads) pt_forward_kernel(PtArgs a) {
    extern __shared__ __align__(16) float smem[];
    float* s_fT = smem;                                  // [kPtKSlice][kPtFStride]
    float* s_wT = s_fT + kPtKSlice * kPtFStride;         // [kPtKSlice][kPtWStride]
    __shared__ int s_pix[kPtMaxBatch];
    const int m = blockIdx.y, split = blockIdx.x, tid = threadIdx.x;
    const PtState st = a.st[m];
    if (st.done) return;
    const int B = a.B, F = a.F, S = a.S;
    const int k0 = split * kPtKSlice, kc = min(kPtKSlice, F - k0);
    if (tid < B) {
        const int64_t t = st.steps_done;
        const int64_t epoch = t / a.steps_per_epoch, pos = t - epoch * a.steps_per_epoch;
        const int px = (int)pt_permute(st.key, (uint64_t)epoch, (uint64_t)(pos * B + tid), (uint64_t)a.n_pix, a.half_bits);
        s_pix[tid] = px;
        if (split == 0) a.pix[m * B + tid] = px;
    }
    const float* w1 = a.w1 + (size_t)m * GAN_H1 * F;
    for (int idx = tid; idx < GAN_H1 * kc; idx += kPtThreads) {
        const int j = idx / kc, kk = idx - j * kc;
        s_wT[kk * kPtWStride + j] = w1[(size_t)j * F + k0 + kk];
    }
    __syncthreads();
    // gather: feature k0 + kk of pixel p
    float* feat = a.feat + (size_t)m * B * F;
    for (int idx = tid; idx < B * kc; idx += kPtThreads) {
        const int kk = idx / B, p = idx - kk * B;
        const int k = k0 + kk;
        int l = 0;
        while (k >= a.coff[l + 1]) ++l;
        const int c = k - a.coff[l], r = a.res[l];
        const int px = s_pix[p];
        const int img = px / (S * S), rem = px - img * S * S;
        const int oy = rem / S, ox = rem - oy * S;
        const float* q = a.act[l] + ((size_t)img * a.chan[l] + c) * r * r;
        float v;
        if (r == S) {
            v = __ldg(q + oy * r + ox);
        } else {
            const GanBilinearTap tp = gan_bilinear_tap(oy, ox, r, S);
            v = tp.w00 * __ldg(q + tp.y0 * r + tp.x0);
            v = fmaf(tp.w01, __ldg(q + tp.y0 * r + tp.x1), v);
            v = fmaf(tp.w10, __ldg(q + tp.y1 * r + tp.x0), v);
            v = fmaf(tp.w11, __ldg(q + tp.y1 * r + tp.x1), v);
        }
        s_fT[kk * kPtFStride + p] = v;
        feat[(size_t)p * F + k] = v;
    }
    __syncthreads();
    // partial h1[p][j] over the slice: thread (tp, tj) owns pixels 4 tp .. 4 tp + 3 and outputs 8 tj .. 8 tj + 7
    const int tp = tid & 15, tj = tid >> 4;
    float acc[4][8];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[i][q] = 0.f;
    for (int kk = 0; kk < kc; ++kk) {
        const float4 f = *reinterpret_cast<const float4*>(s_fT + kk * kPtFStride + 4 * tp);
        const float4 wa = *reinterpret_cast<const float4*>(s_wT + kk * kPtWStride + 8 * tj);
        const float4 wb = *reinterpret_cast<const float4*>(s_wT + kk * kPtWStride + 8 * tj + 4);
        const float fv[4] = {f.x, f.y, f.z, f.w};
        const float wv[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int q = 0; q < 8; ++q) acc[i][q] = fmaf(fv[i], wv[q], acc[i][q]);
    }
    float* part = a.part + ((size_t)m * a.n_split + split) * B * GAN_H1;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int p = 4 * tp + i;
        if (p < B)
#pragma unroll
            for (int q = 0; q < 8; ++q) part[p * GAN_H1 + 8 * tj + q] = acc[i][q];
    }
}

// BatchNorm1d in training mode over the batch for features [0, nf) of x[B][nf]: batch mean, biased variance; the running
// statistics take the unbiased variance with momentum 0.1.  Writes xhat and the inverse standard deviations.
__device__ void pt_bn_forward(const float* x, float* xhat, float* istd, int B, int nf, float* rmean, float* rvar) {
    for (int j = threadIdx.x; j < nf; j += kPtThreads) {
        float sum = 0.f;
        for (int p = 0; p < B; ++p) sum += x[p * nf + j];
        const float mean = sum / (float)B;
        float ss = 0.f;
        for (int p = 0; p < B; ++p) { const float d = x[p * nf + j] - mean; ss = fmaf(d, d, ss); }
        const float var = ss / (float)B;
        const float is = 1.0f / sqrtf(var + kPtBnEps);
        istd[j] = is;
        for (int p = 0; p < B; ++p) xhat[p * nf + j] = (x[p * nf + j] - mean) * is;
        rmean[j] = fmaf(kPtBnMomentum, mean - rmean[j], rmean[j]);
        rvar[j] = fmaf(kPtBnMomentum, ss / (float)(B - 1) - rvar[j], rvar[j]);
    }
}

// Backward of y = gamma * xhat + beta followed by the ReLU that produced x (mask x > 0): dy[B][nf] in, dx (masked) out in
// place; d gamma and d beta to grads.
__device__ void pt_bn_backward(float* d, const float* xhat, const float* x, const float* istd, const float* gamma, int B, int nf,
                               float* dgamma, float* dbeta) {
    for (int j = threadIdx.x; j < nf; j += kPtThreads) {
        float sdy = 0.f, sdyx = 0.f;
        for (int p = 0; p < B; ++p) { sdy += d[p * nf + j]; sdyx = fmaf(d[p * nf + j], xhat[p * nf + j], sdyx); }
        dgamma[j] = sdyx;
        dbeta[j] = sdy;
        const float g = gamma[j], is = istd[j];
        const float mdy = sdy / (float)B, mdyx = sdyx / (float)B;
        for (int p = 0; p < B; ++p) {
            const float dx = (d[p * nf + j] - mdy - xhat[p * nf + j] * mdyx) * is * g;
            d[p * nf + j] = x[p * nf + j] > 0.f ? dx : 0.f;
        }
    }
}

__global__ void __launch_bounds__(kPtThreads) pt_tail_kernel(PtArgs a) {
    extern __shared__ __align__(16) float smem[];
    const int m = blockIdx.x, tid = threadIdx.x;
    PtState* stp = a.st + m;
    if (stp->done) {
        if (tid == 0) stp->ran = 0;
        return;
    }
    const int B = a.B, n = a.n_class, P = small_size(n);
    float* s_a1 = smem;                         // [B][128] relu(h1)
    float* s_xh1 = s_a1 + kPtMaxBatch * GAN_H1;  // [B][128]
    float* s_d1 = s_xh1 + kPtMaxBatch * GAN_H1;  // [B][128] dy1, then dh1
    float* s_a2 = s_d1 + kPtMaxBatch * GAN_H1;   // [B][32]
    float* s_xh2 = s_a2 + kPtMaxBatch * GAN_H2;
    float* s_d2 = s_xh2 + kPtMaxBatch * GAN_H2;
    float* s_lg = s_d2 + kPtMaxBatch * GAN_H2;   // [B][32] logits, then d logits
    float* s_istd1 = s_lg + kPtMaxBatch * GAN_H2;
    float* s_istd2 = s_istd1 + GAN_H1;
    float* s_lossp = s_istd2 + GAN_H2;
    float* s_p = s_lossp + kPtMaxBatch;          // [P] parameters
    __shared__ int s_y[kPtMaxBatch];

    const float* prm = a.small + (size_t)m * P;
    for (int i = tid; i < P; i += kPtThreads) s_p[i] = prm[i];
    if (tid < B) s_y[tid] = a.labels[a.pix[m * B + tid]];
    const float* part = a.part + (size_t)m * a.n_split * B * GAN_H1;
    for (int e = tid; e < B * GAN_H1; e += kPtThreads) {
        float sum = 0.f;
        for (int s = 0; s < a.n_split; ++s) sum += part[(size_t)s * B * GAN_H1 + e];
        s_a1[e] = fmaxf(sum + prm[kOffB1 + (e & (GAN_H1 - 1))], 0.f);
    }
    __syncthreads();
    float* rs = a.rstat + (size_t)m * kRstat;
    pt_bn_forward(s_a1, s_xh1, s_istd1, B, GAN_H1, rs, rs + GAN_H1);
    __syncthreads();
    // h2 = W2 y1 + b2, y1 = gamma1 xhat1 + beta1
    for (int e = tid; e < B * GAN_H2; e += kPtThreads) {
        const int p = e / GAN_H2, o = e - p * GAN_H2;
        float acc = s_p[kOffB2 + o];
        for (int j = 0; j < GAN_H1; ++j)
            acc = fmaf(s_p[kOffW2 + o * GAN_H1 + j], fmaf(s_p[kOffG1 + j], s_xh1[p * GAN_H1 + j], s_p[kOffBe1 + j]), acc);
        s_a2[e] = fmaxf(acc, 0.f);
    }
    __syncthreads();
    pt_bn_forward(s_a2, s_xh2, s_istd2, B, GAN_H2, rs + 2 * GAN_H1, rs + 2 * GAN_H1 + GAN_H2);
    __syncthreads();
    for (int e = tid; e < B * n; e += kPtThreads) {
        const int p = e / n, c = e - p * n;
        float acc = s_p[off_b3(n) + c];
        for (int o = 0; o < GAN_H2; ++o)
            acc = fmaf(s_p[kOffW3 + c * GAN_H2 + o], fmaf(s_p[kOffG2 + o], s_xh2[p * GAN_H2 + o], s_p[kOffBe2 + o]), acc);
        s_lg[p * GAN_H2 + c] = acc;
    }
    __syncthreads();
    // softmax cross-entropy, mean over the batch: d logits = (softmax - onehot) / B
    if (tid < B) {
        float* l = s_lg + tid * GAN_H2;
        float mx = -INFINITY;
        for (int c = 0; c < n; ++c) mx = fmaxf(mx, l[c]);
        float se = 0.f;
        for (int c = 0; c < n; ++c) se += expf(l[c] - mx);
        const float lse = mx + logf(se);
        float ly = 0.f;
        for (int c = 0; c < n; ++c) ly = c == s_y[tid] ? l[c] : ly;
        s_lossp[tid] = lse - ly;
        for (int c = 0; c < n; ++c) l[c] = (expf(l[c] - lse) - (c == s_y[tid] ? 1.f : 0.f)) / (float)B;
    }
    __syncthreads();
    float* g = a.gsmall + (size_t)m * P;
    // Linear 3: d b3, d W3, d y2
    for (int e = tid; e < n * (GAN_H2 + 1); e += kPtThreads) {
        if (e < n * GAN_H2) {
            const int c = e / GAN_H2, o = e - c * GAN_H2;
            float acc = 0.f;
            for (int p = 0; p < B; ++p)
                acc = fmaf(s_lg[p * GAN_H2 + c], fmaf(s_p[kOffG2 + o], s_xh2[p * GAN_H2 + o], s_p[kOffBe2 + o]), acc);
            g[kOffW3 + e] = acc;
        } else {
            const int c = e - n * GAN_H2;
            float acc = 0.f;
            for (int p = 0; p < B; ++p) acc += s_lg[p * GAN_H2 + c];
            g[off_b3(n) + c] = acc;
        }
    }
    for (int e = tid; e < B * GAN_H2; e += kPtThreads) {
        const int p = e / GAN_H2, o = e - p * GAN_H2;
        float acc = 0.f;
        for (int c = 0; c < n; ++c) acc = fmaf(s_lg[p * GAN_H2 + c], s_p[kOffW3 + c * GAN_H2 + o], acc);
        s_d2[e] = acc;
    }
    __syncthreads();
    pt_bn_backward(s_d2, s_xh2, s_a2, s_istd2, s_p + kOffG2, B, GAN_H2, g + kOffG2, g + kOffBe2);
    __syncthreads();
    // Linear 2: d b2, d W2, d y1
    for (int e = tid; e < GAN_H2 * (GAN_H1 + 1); e += kPtThreads) {
        if (e < GAN_H2 * GAN_H1) {
            const int o = e / GAN_H1, j = e - o * GAN_H1;
            float acc = 0.f;
            for (int p = 0; p < B; ++p)
                acc = fmaf(s_d2[p * GAN_H2 + o], fmaf(s_p[kOffG1 + j], s_xh1[p * GAN_H1 + j], s_p[kOffBe1 + j]), acc);
            g[kOffW2 + e] = acc;
        } else {
            const int o = e - GAN_H2 * GAN_H1;
            float acc = 0.f;
            for (int p = 0; p < B; ++p) acc += s_d2[p * GAN_H2 + o];
            g[kOffB2 + o] = acc;
        }
    }
    for (int e = tid; e < B * GAN_H1; e += kPtThreads) {
        const int p = e / GAN_H1, j = e - p * GAN_H1;
        float acc = 0.f;
        for (int o = 0; o < GAN_H2; ++o) acc = fmaf(s_d2[p * GAN_H2 + o], s_p[kOffW2 + o * GAN_H1 + j], acc);
        s_d1[e] = acc;
    }
    __syncthreads();
    pt_bn_backward(s_d1, s_xh1, s_a1, s_istd1, s_p + kOffG1, B, GAN_H1, g + kOffG1, g + kOffBe1);
    __syncthreads();
    float* dh1 = a.dh1 + (size_t)m * B * GAN_H1;
    for (int e = tid; e < B * GAN_H1; e += kPtThreads) dh1[e] = s_d1[e];
    for (int j = tid; j < GAN_H1; j += kPtThreads) {
        float acc = 0.f;
        for (int p = 0; p < B; ++p) acc += s_d1[p * GAN_H1 + j];
        g[kOffB1 + j] = acc;
    }
    if (tid == 0) {
        float sum = 0.f;
        for (int p = 0; p < B; ++p) sum += s_lossp[p];
        const float loss = sum / (float)B;
        PtState st = *stp;
        a.loss[(size_t)m * st.max_steps + st.steps_done] = loss;
        // DatasetGAN's rule: from epoch 4 on, stop after more than 50 consecutive steps without a new best loss
        if (st.steps_done / a.steps_per_epoch >= kPtFirstRuleEpoch) {
            if (loss < st.best_loss) { st.best_loss = loss; st.break_count = 0; }
            else st.break_count += 1;
        }
        st.steps_done += 1;
        st.done = st.break_count > kPtPatience || st.steps_done >= st.max_steps;
        st.ran = 1;
        *stp = st;
    }
}

// torch.optim.Adam (no weight decay, no amsgrad) on one element
__device__ __forceinline__ void pt_adam(float& p, float& mo, float& ve, float g, float step_size, float bc2_sqrt) {
    // 1 - beta in double, as torch's Python scalars (1.f - 0.999f is 1.3e-5 away from 0.001f)
    mo = fmaf((float)(1.0 - kPtBeta1Exact), g - mo, mo);
    ve = fmaf((float)(1.0 - kPtBeta2Exact), g * g, kPtBeta2 * ve);
    const float denom = sqrtf(ve) / bc2_sqrt + kPtEps;
    p = fmaf(-step_size, mo / denom, p);
}

__global__ void __launch_bounds__(kPtThreads) pt_update_kernel(PtArgs a) {
    extern __shared__ __align__(16) float smem[];
    const int m = blockIdx.y, split = blockIdx.x, tid = threadIdx.x;
    const PtState st = a.st[m];
    if (!st.ran) return;
    const int B = a.B, F = a.F;
    const int k0 = split * kPtKSlice, kc = min(kPtKSlice, F - k0);
    const double t = (double)st.steps_done;
    const float step_size = (float)(kPtLr / (1.0 - pow(0.9, t)));     // in double, as torch's Python scalars
    const float bc2_sqrt = (float)sqrt(1.0 - pow(0.999, t));
    float* s_f = smem;                           // [B][kPtKSlice]
    float* s_dh = s_f + kPtMaxBatch * kPtKSlice;  // [B][128]
    const float* feat = a.feat + (size_t)m * B * F;
    const float* dh1 = a.dh1 + (size_t)m * B * GAN_H1;
    for (int idx = tid; idx < B * kc; idx += kPtThreads) {
        const int p = idx / kc, kk = idx - p * kc;
        s_f[p * kPtKSlice + kk] = feat[(size_t)p * F + k0 + kk];
    }
    for (int idx = tid; idx < B * GAN_H1; idx += kPtThreads) s_dh[idx] = dh1[idx];
    __syncthreads();
    const int kk = tid & (kPtKSlice - 1);
    if (kk < kc) {
        const size_t base = (size_t)m * GAN_H1 * F + k0 + kk;
        for (int j = tid >> 7; j < GAN_H1; j += kPtThreads / kPtKSlice) {
            float gr = 0.f;
            for (int p = 0; p < B; ++p) gr = fmaf(s_dh[p * GAN_H1 + j], s_f[p * kPtKSlice + kk], gr);
            const size_t o = base + (size_t)j * F;
            float p = a.w1[o], mo = a.m1[o], ve = a.v1[o];
            pt_adam(p, mo, ve, gr, step_size, bc2_sqrt);
            a.w1[o] = p; a.m1[o] = mo; a.v1[o] = ve;
        }
    }
    if (split == 0) {
        const int P = small_size(a.n_class);
        const size_t base = (size_t)m * P;
        for (int i = tid; i < P; i += kPtThreads) {
            float p = a.small[base + i], mo = a.msmall[base + i], ve = a.vsmall[base + i];
            pt_adam(p, mo, ve, a.gsmall[base + i], step_size, bc2_sqrt);
            a.small[base + i] = p; a.msmall[base + i] = mo; a.vsmall[base + i] = ve;
        }
    }
}

size_t pt_forward_smem() { return sizeof(float) * (size_t)kPtKSlice * (kPtFStride + kPtWStride); }
size_t pt_tail_smem(int n_class) {
    return sizeof(float) * ((size_t)3 * kPtMaxBatch * GAN_H1 + 4 * kPtMaxBatch * GAN_H2 + GAN_H1 + GAN_H2 + kPtMaxBatch + small_size(n_class));
}
size_t pt_update_smem() { return sizeof(float) * (size_t)kPtMaxBatch * (kPtKSlice + GAN_H1); }

int expect_param(const std::map<std::string, std::vector<float>>& sd, const std::string& key, size_t n) {
    auto it = sd.find(key);
    SIS_REQUIRE(it != sd.end(), "pixel train: parameter '%s' was never set", key.c_str());
    SIS_REQUIRE(it->second.size() == n, "pixel train: parameter '%s' has %zu values, expected %zu", key.c_str(), it->second.size(), n);
    return SIS_OK;
}

// (state-dict key, offset in the packed small vector or -1, offset in the running statistics or -1, element count)
struct PtKey { const char* name; int small_off; int rstat_off; int count; };
std::vector<PtKey> pt_keys(int n) {
    return {{"layers.0.bias", kOffB1, -1, GAN_H1},         {"layers.2.weight", kOffG1, -1, GAN_H1},
            {"layers.2.bias", kOffBe1, -1, GAN_H1},        {"layers.2.running_mean", -1, 0, GAN_H1},
            {"layers.2.running_var", -1, GAN_H1, GAN_H1},  {"layers.3.weight", kOffW2, -1, GAN_H2 * GAN_H1},
            {"layers.3.bias", kOffB2, -1, GAN_H2},         {"layers.5.weight", kOffG2, -1, GAN_H2},
            {"layers.5.bias", kOffBe2, -1, GAN_H2},        {"layers.5.running_mean", -1, 2 * GAN_H1, GAN_H2},
            {"layers.5.running_var", -1, 2 * GAN_H1 + GAN_H2, GAN_H2}, {"layers.6.weight", kOffW3, -1, n * GAN_H2},
            {"layers.6.bias", off_b3(n), -1, n}};
}

}  // namespace
}  // namespace sis

struct sis_pixel_train {
    int n_models = 0, feature_size = 0, n_class = 0, batch = 0;
    std::vector<std::map<std::string, std::vector<float>>> host;
    bool has_data = false, prepared = false;
    sis::PtArgs args{};
    void* buffers[14] = {};
};

namespace {
void pt_free(sis_pixel_train* t) {
    for (void*& b : t->buffers) { cudaFree(b); b = nullptr; }
    t->prepared = false;
}
}  // namespace

extern "C" int sis_pixel_train_create(sis_pixel_train** out, int n_models, int feature_size, int n_class, int batch_pixels) {
    using namespace sis;
    SIS_REQUIRE(out, "sis_pixel_train_create: null output");
    SIS_REQUIRE(n_models >= 1 && n_models <= GAN_MAX_MODELS, "pixel train: 1..%d networks (got %d)", GAN_MAX_MODELS, n_models);
    SIS_REQUIRE(n_class >= 2 && n_class < 32, "pixel train: the 128/32 classifier takes 2 <= n_class < 32 (got %d)", n_class);
    SIS_REQUIRE(feature_size > 0 && feature_size % 32 == 0, "pixel train: feature size must be a positive multiple of 32 (got %d)", feature_size);
    SIS_REQUIRE(batch_pixels >= 2 && batch_pixels <= kPtMaxBatch, "pixel train: batch of 2..%d pixels (got %d)", kPtMaxBatch, batch_pixels);
    auto* t = new sis_pixel_train();
    t->n_models = n_models; t->feature_size = feature_size; t->n_class = n_class; t->batch = batch_pixels;
    t->host.resize(n_models);
    *out = t;
    return SIS_OK;
}

extern "C" void sis_pixel_train_destroy(sis_pixel_train* t) {
    if (!t) return;
    pt_free(t);
    delete t;
}

extern "C" int sis_pixel_train_set_param(sis_pixel_train* t, int model, const char* name, const float* host_data, int64_t numel) {
    using namespace sis;
    SIS_REQUIRE(t && name && host_data && numel >= 0, "sis_pixel_train_set_param: null argument");
    SIS_REQUIRE(model >= 0 && model < t->n_models, "pixel train: network index %d out of range", model);
    t->host[model][name].assign(host_data, host_data + numel);
    t->prepared = false;
    return SIS_OK;
}

extern "C" int sis_pixel_train_set_data(sis_pixel_train* t, int n_layers, const float* const* d_activations, const int* channels,
                                        const int* resolutions, int n_images, int image_size, const uint8_t* d_labels) {
    using namespace sis;
    SIS_REQUIRE(t && d_activations && channels && resolutions && d_labels, "sis_pixel_train_set_data: null argument");
    SIS_REQUIRE(n_layers >= 1 && n_layers <= kPtMaxLayers, "pixel train: 1..%d captures (got %d)", kPtMaxLayers, n_layers);
    SIS_REQUIRE(n_images >= 1 && image_size >= 1, "pixel train: bad image count / size");
    const int64_t n_pix = (int64_t)n_images * image_size * image_size;
    SIS_REQUIRE(n_pix >= t->batch, "pixel train: %lld annotated pixels, fewer than one batch of %d", (long long)n_pix, t->batch);
    SIS_REQUIRE(n_pix <= INT32_MAX, "pixel train: %lld annotated pixels exceed 2^31 - 1", (long long)n_pix);
    PtArgs& a = t->args;
    int off = 0;
    for (int l = 0; l < n_layers; ++l) {
        SIS_REQUIRE(d_activations[l], "pixel train: capture %d is null", l);
        SIS_REQUIRE(channels[l] >= 1 && resolutions[l] >= 1 && resolutions[l] <= image_size,
                    "pixel train: capture %d has %d channels at %d^2 (image %d^2)", l, channels[l], resolutions[l], image_size);
        a.act[l] = d_activations[l]; a.chan[l] = channels[l]; a.res[l] = resolutions[l]; a.coff[l] = off;
        off += channels[l];
    }
    SIS_REQUIRE(off == t->feature_size, "pixel train: captures carry %d features, the classifiers expect %d", off, t->feature_size);
    a.coff[n_layers] = off;
    a.n_layers = n_layers;
    a.labels = d_labels;
    a.S = image_size;
    a.n_pix = n_pix;
    int bits = 2;
    while (bits < 62 && (1ll << bits) < n_pix) bits += 2;
    a.half_bits = bits / 2;
    t->has_data = true;
    t->prepared = false;
    return SIS_OK;
}

extern "C" int sis_pixel_train_prepare(sis_pixel_train* t, const uint64_t* keys, int epochs, void* stream_) {
    using namespace sis;
    SIS_REQUIRE(t && keys, "sis_pixel_train_prepare: null argument");
    SIS_REQUIRE(t->has_data, "sis_pixel_train_prepare: call sis_pixel_train_set_data first");
    SIS_REQUIRE(epochs >= 1, "pixel train: epochs must be >= 1 (got %d)", epochs);
    cudaStream_t stream = (cudaStream_t)stream_;
    const int M = t->n_models, F = t->feature_size, n = t->n_class, B = t->batch, P = small_size(n);
    PtArgs& a = t->args;
    a.F = F; a.n_class = n; a.B = B;
    a.n_split = ceil_div(F, kPtKSlice);
    a.steps_per_epoch = a.n_pix / B;
    const int64_t max_steps = (int64_t)epochs * a.steps_per_epoch;
    std::vector<float> w1((size_t)M * GAN_H1 * F), small((size_t)M * P), rstat((size_t)M * kRstat);
    const auto keys_n = pt_keys(n);
    for (int m = 0; m < M; ++m) {
        const auto& sd = t->host[m];
        SIS_PROPAGATE(expect_param(sd, "layers.0.weight", (size_t)GAN_H1 * F));
        std::copy(sd.at("layers.0.weight").begin(), sd.at("layers.0.weight").end(), w1.begin() + (size_t)m * GAN_H1 * F);
        for (const PtKey& k : keys_n) {
            SIS_PROPAGATE(expect_param(sd, k.name, (size_t)k.count));
            const auto& v = sd.at(k.name);
            if (k.small_off >= 0) std::copy(v.begin(), v.end(), small.begin() + (size_t)m * P + k.small_off);
            else std::copy(v.begin(), v.end(), rstat.begin() + (size_t)m * kRstat + k.rstat_off);
        }
    }
    pt_free(t);
    const size_t sizes[14] = {sizeof(float) * w1.size(), sizeof(float) * w1.size(), sizeof(float) * w1.size(),
                              sizeof(float) * small.size(), sizeof(float) * small.size(), sizeof(float) * small.size(),
                              sizeof(float) * small.size(), sizeof(float) * rstat.size(), sizeof(float) * M * B * F,
                              sizeof(float) * M * a.n_split * B * GAN_H1, sizeof(float) * M * B * GAN_H1, sizeof(int32_t) * M * B,
                              sizeof(float) * M * max_steps, sizeof(PtState) * M};
    for (int i = 0; i < 14; ++i) SIS_CHECK_CUDA(cudaMalloc(&t->buffers[i], sizes[i]));
    for (int i : {1, 2, 4, 5, 6, 8, 9, 10, 11, 12}) SIS_CHECK_CUDA(cudaMemsetAsync(t->buffers[i], 0, sizes[i], stream));
    a.w1 = (float*)t->buffers[0]; a.m1 = (float*)t->buffers[1]; a.v1 = (float*)t->buffers[2];
    a.small = (float*)t->buffers[3]; a.msmall = (float*)t->buffers[4]; a.vsmall = (float*)t->buffers[5]; a.gsmall = (float*)t->buffers[6];
    a.rstat = (float*)t->buffers[7]; a.feat = (float*)t->buffers[8]; a.part = (float*)t->buffers[9]; a.dh1 = (float*)t->buffers[10];
    a.pix = (int32_t*)t->buffers[11]; a.loss = (float*)t->buffers[12]; a.st = (PtState*)t->buffers[13];
    std::vector<PtState> st(M);
    for (int m = 0; m < M; ++m) {
        st[m] = PtState{};
        st[m].key = keys[m];
        st[m].max_steps = max_steps;
        st[m].best_loss = 10000000.f;                   // DatasetGAN's initial best_loss
    }
    SIS_CHECK_CUDA(cudaMemcpyAsync(a.w1, w1.data(), sizes[0], cudaMemcpyHostToDevice, stream));
    SIS_CHECK_CUDA(cudaMemcpyAsync(a.small, small.data(), sizes[3], cudaMemcpyHostToDevice, stream));
    SIS_CHECK_CUDA(cudaMemcpyAsync(a.rstat, rstat.data(), sizes[7], cudaMemcpyHostToDevice, stream));
    SIS_CHECK_CUDA(cudaMemcpyAsync(a.st, st.data(), sizes[13], cudaMemcpyHostToDevice, stream));
    SIS_CHECK_CUDA(cudaStreamSynchronize(stream));      // the host vectors go out of scope
    int dev = 0;
    SIS_CHECK_CUDA(cudaGetDevice(&dev));
    static bool attr_set[64] = {};                      // the shared-memory limit is a per-device attribute
    if (dev >= 64 || !attr_set[dev]) {
        SIS_CHECK_CUDA(cudaFuncSetAttribute(pt_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pt_forward_smem()));
        SIS_CHECK_CUDA(cudaFuncSetAttribute(pt_tail_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pt_tail_smem(31)));
        SIS_CHECK_CUDA(cudaFuncSetAttribute(pt_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pt_update_smem()));
        if (dev < 64) attr_set[dev] = true;
    }
    t->prepared = true;
    return SIS_OK;
}

extern "C" int sis_pixel_train_steps(sis_pixel_train* t, int steps, void* stream_) {
    using namespace sis;
    SIS_REQUIRE(t && t->prepared, "sis_pixel_train_steps: call sis_pixel_train_prepare first");
    SIS_REQUIRE(steps >= 1, "sis_pixel_train_steps: steps must be >= 1");
    cudaStream_t stream = (cudaStream_t)stream_;
    const PtArgs& a = t->args;
    const dim3 wide((unsigned)a.n_split, (unsigned)t->n_models);
    ProfScope prof(PROF_OTHER, stream);
    for (int s = 0; s < steps; ++s) {
        pt_forward_kernel<<<wide, kPtThreads, pt_forward_smem(), stream>>>(a);
        SIS_CHECK_LAUNCH();
        pt_tail_kernel<<<t->n_models, kPtThreads, pt_tail_smem(t->n_class), stream>>>(a);
        SIS_CHECK_LAUNCH();
        pt_update_kernel<<<wide, kPtThreads, pt_update_smem(), stream>>>(a);
        SIS_CHECK_LAUNCH();
    }
    return SIS_OK;
}

extern "C" int sis_pixel_train_status(sis_pixel_train* t, int32_t* done, int64_t* steps_done, void* stream_) {
    using namespace sis;
    SIS_REQUIRE(t && t->prepared && done && steps_done, "sis_pixel_train_status: null argument or not prepared");
    std::vector<PtState> st(t->n_models);
    SIS_CHECK_CUDA(cudaMemcpyAsync(st.data(), t->args.st, sizeof(PtState) * st.size(), cudaMemcpyDeviceToHost, (cudaStream_t)stream_));
    SIS_CHECK_CUDA(cudaStreamSynchronize((cudaStream_t)stream_));
    for (int m = 0; m < t->n_models; ++m) { done[m] = st[m].done; steps_done[m] = st[m].steps_done; }
    return SIS_OK;
}

extern "C" int sis_pixel_train_read_param(sis_pixel_train* t, int model, const char* name, float* host_out, int64_t numel, void* stream_) {
    using namespace sis;
    SIS_REQUIRE(t && t->prepared && name && host_out, "sis_pixel_train_read_param: null argument or not prepared");
    SIS_REQUIRE(model >= 0 && model < t->n_models, "pixel train: network index %d out of range", model);
    const PtArgs& a = t->args;
    const int P = small_size(t->n_class);
    const float* src = nullptr;
    int64_t count = 0;
    if (std::string(name) == "layers.0.weight") {
        src = a.w1 + (size_t)model * GAN_H1 * a.F; count = (int64_t)GAN_H1 * a.F;
    } else {
        for (const PtKey& k : pt_keys(t->n_class))
            if (std::string(name) == k.name) {
                src = k.small_off >= 0 ? a.small + (size_t)model * P + k.small_off : a.rstat + (size_t)model * kRstat + k.rstat_off;
                count = k.count;
            }
    }
    SIS_REQUIRE(src, "pixel train: no trained tensor '%s'", name);
    SIS_REQUIRE(numel == count, "pixel train: '%s' has %lld values, asked for %lld", name, (long long)count, (long long)numel);
    SIS_CHECK_CUDA(cudaMemcpyAsync(host_out, src, sizeof(float) * count, cudaMemcpyDeviceToHost, (cudaStream_t)stream_));
    SIS_CHECK_CUDA(cudaStreamSynchronize((cudaStream_t)stream_));
    return SIS_OK;
}

extern "C" int sis_pixel_train_read_losses(sis_pixel_train* t, int model, float* host_out, int64_t count, void* stream_) {
    using namespace sis;
    SIS_REQUIRE(t && t->prepared && host_out, "sis_pixel_train_read_losses: null argument or not prepared");
    SIS_REQUIRE(model >= 0 && model < t->n_models, "pixel train: network index %d out of range", model);
    SIS_REQUIRE(count >= 0, "pixel train: negative loss count");
    if (count == 0) return SIS_OK;
    std::vector<PtState> st(t->n_models);
    SIS_CHECK_CUDA(cudaMemcpyAsync(st.data(), t->args.st, sizeof(PtState) * st.size(), cudaMemcpyDeviceToHost, (cudaStream_t)stream_));
    SIS_CHECK_CUDA(cudaStreamSynchronize((cudaStream_t)stream_));
    SIS_REQUIRE(count <= st[model].steps_done, "pixel train: %lld losses asked, network %d ran %lld steps", (long long)count, model,
                (long long)st[model].steps_done);
    SIS_CHECK_CUDA(cudaMemcpyAsync(host_out, t->args.loss + (size_t)model * st[model].max_steps, sizeof(float) * count,
                                   cudaMemcpyDeviceToHost, (cudaStream_t)stream_));
    SIS_CHECK_CUDA(cudaStreamSynchronize((cudaStream_t)stream_));
    return SIS_OK;
}
