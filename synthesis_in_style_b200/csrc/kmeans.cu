// Spherical mini-batch k-means steps for catalog creation (sis_kmeans_steps): one CTA per fit, a fixed number of steps
// per launch.  Each step is the loop body of scf/segmentation/gan_local_edit/spherical_kmeans.py's fit (sklearn 0.24's
// MiniBatchKMeans._mini_batch_step on unit rows): renormalise, nearest centre of every batch row, random reassignment of
// starved centres, count-weighted update, renormalise, EWA-inertia early stopping.  oracle/kmeans_oracle.py restates it.
//
// The batch rows stay in global memory (up to 1024 x 512 fp32 would not fit on chip); a CTA keeps its centres, the drawn
// row indices, labels and distances in shared memory.  Every sum has a fixed order, so a fit's result does not depend on
// which other fits share the launch or on how many steps each launch runs.
#include <float.h>
#include "common.cuh"

namespace sis {
namespace {

constexpr int kKmThreads = 256;
constexpr int kKmWarps = kKmThreads / 32;
constexpr int kKmMaxK = 32;         // one lane per centre in the assignment and the reassignment
constexpr int kKmMaxChannels = 512;
constexpr int kKmMaxBatch = 1024;

__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

// Draw `stream` of row j at step t: stream 0 picks batch rows (u mod n), stream 1 orders the rows that replace starved
// centres.  A pure function of its arguments, so the oracle restates it and batching cannot change it.
__device__ __forceinline__ uint64_t km_draw(uint64_t seed_mix, uint64_t t, uint64_t j, uint64_t stream) {
    return splitmix64(splitmix64(seed_mix ^ t) ^ ((j << 1) | stream));
}

// Centre rows are stored with an odd stride so that lane i reading centre i, channel c hits bank (i * stride + c) % 32:
// all 32 lanes distinct.
__host__ __device__ __forceinline__ int centre_stride(int channels) { return channels | 1; }

size_t km_smem_bytes(int k, int channels) {
    return sizeof(float) * ((size_t)k * centre_stride(channels) + (size_t)kKmWarps * channels)
         + kKmMaxBatch * (sizeof(int) + sizeof(int) + sizeof(float) + sizeof(uint64_t));
}

__global__ void kmeans_init_state_kernel(sis_kmeans_state* st, sis_kmeans_state v) { *st = v; }

// Each warp renormalises centres w, w + kKmWarps, ...: x / max(||x||, 1e-12) as the reference's normalisation.
__device__ void normalise_centres(float* cent, int k, int channels, int stride) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = warp; i < k; i += kKmWarps) {
        float* row = cent + (size_t)i * stride;
        float ss = 0.f;
        for (int c = lane; c < channels; c += 32) ss = fmaf(row[c], row[c], ss);
        for (int o = 16; o; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
        const float nrm = fmaxf(sqrtf(ss), 1e-12f);
        for (int c = lane; c < channels; c += 32) row[c] = __fdiv_rn(row[c], nrm);
    }
}

__global__ void __launch_bounds__(kKmThreads) kmeans_steps_kernel(const sis_kmeans_fit* __restrict__ fits, int steps,
                                                                  const int32_t* __restrict__ indices, int n_indices,
                                                                  float* __restrict__ batch_inertia) {
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ float s_counts[kKmMaxK];
    __shared__ int s_nin[kKmMaxK];
    __shared__ int s_pick[kKmMaxK];
    __shared__ int s_run, s_reassign, s_n_re;
    __shared__ unsigned s_starved;
    __shared__ float s_new_count;

    const sis_kmeans_fit f = fits[blockIdx.x];
    const int k = f.k, channels = f.channels, stride = centre_stride(channels);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool explicit_rows = indices != nullptr;
    // the 8-byte keys come first: the centre rows have an odd stride, so what follows them is only 4-byte aligned
    uint64_t* s_key = reinterpret_cast<uint64_t*>(smem);
    int* s_idx = reinterpret_cast<int*>(s_key + kKmMaxBatch);
    int* s_lab = s_idx + kKmMaxBatch;
    float* s_dist = reinterpret_cast<float*>(s_lab + kKmMaxBatch);
    float* cent = s_dist + kKmMaxBatch;
    float* stage = cent + (size_t)k * stride;

    sis_kmeans_state st{};
    if (!explicit_rows) st = *f.d_state;          // every thread keeps a copy; thread 0's is written back
    if (!explicit_rows && st.done) return;
    const int bs = explicit_rows ? n_indices : st.batch_size;
    const uint64_t seed_mix = splitmix64(st.seed);
    const double alpha = fmin(1.0, (double)bs * 2.0 / (double)(f.n + 1));

    for (int i = threadIdx.x; i < k * channels; i += kKmThreads)
        cent[(i / channels) * stride + i % channels] = f.d_centers[i];
    if (threadIdx.x < k) s_counts[threadIdx.x] = f.d_counts[threadIdx.x];
    __syncthreads();

    const uint64_t t0 = (uint64_t)st.steps_done;      // only thread 0 advances its copy of the state
    for (int s = 0; s < steps; ++s) {
        const uint64_t t = t0 + s;
        for (int j = threadIdx.x; j < bs; j += kKmThreads)
            s_idx[j] = explicit_rows ? indices[j] : (int)(km_draw(seed_mix, t, j, 0) % (uint64_t)f.n);
        normalise_centres(cent, k, channels, stride);
        if (threadIdx.x == 0) {
            float cmin = FLT_MAX;
            for (int i = 0; i < k; ++i) cmin = fminf(cmin, s_counts[i]);
            s_reassign = !explicit_rows && st.reassignment_ratio > 0.f && (t + 1) % (uint64_t)(10 + (int64_t)cmin) == 0;
        }
        if (threadIdx.x < kKmMaxK) s_nin[threadIdx.x] = 0;
        __syncthreads();

        // nearest centre of every batch row: one warp per row, lane i against centre i, ties to the lower index
        for (int j = warp; j < bs; j += kKmWarps) {
            const float* x = f.d_points + (int64_t)s_idx[j] * channels;
            float* xr = stage + warp * channels;
            for (int c = lane; c < channels; c += 32) xr[c] = x[c];
            __syncwarp();
            float d = FLT_MAX;
            if (lane < k) {
                const float* m = cent + lane * stride;
                float acc = 0.f;
#pragma unroll 4
                for (int c = 0; c < channels; ++c) {
                    const float e = xr[c] - m[c];
                    acc = fmaf(e, e, acc);
                }
                d = acc;
            }
            int best = lane;
            for (int o = 16; o; o >>= 1) {
                const float od = __shfl_xor_sync(0xffffffffu, d, o);
                const int ob = __shfl_xor_sync(0xffffffffu, best, o);
                if (od < d || (od == d && ob < best)) { d = od; best = ob; }
            }
            if (lane == 0) { s_lab[j] = best; s_dist[j] = d; atomicAdd(&s_nin[best], 1); }
            __syncwarp();
        }
        __syncthreads();

        if (s_reassign) {
            // sklearn 0.24: centres with count < ratio * max count are starved; at most half the batch is reassigned (the
            // lowest counts, ties to the lower index); they take rows of the batch and the smallest remaining count
            for (int j = threadIdx.x; j < bs; j += kKmThreads) s_key[j] = km_draw(seed_mix, t, j, 1);
            if (warp == 0) {
                const float cnt = lane < k ? s_counts[lane] : 0.f;
                float cmax = lane < k ? cnt : -FLT_MAX;
                for (int o = 16; o; o >>= 1) cmax = fmaxf(cmax, __shfl_xor_sync(0xffffffffu, cmax, o));
                bool starved = lane < k && cnt < __fmul_rn(st.reassignment_ratio, cmax);
                if (2 * __popc(__ballot_sync(0xffffffffu, starved)) > bs) {
                    int rank = 0;
                    for (int i = 0; i < k; ++i) {
                        const float ci = __shfl_sync(0xffffffffu, cnt, i);
                        rank += (ci < cnt || (ci == cnt && i < lane));
                    }
                    starved = starved && rank < bs / 2;
                }
                const unsigned mask = __ballot_sync(0xffffffffu, starved);
                float keep_min = (lane < k && !starved) ? cnt : FLT_MAX;
                for (int o = 16; o; o >>= 1) keep_min = fminf(keep_min, __shfl_xor_sync(0xffffffffu, keep_min, o));
                if (lane == 0) {
                    s_starved = mask;
                    s_n_re = __popc(mask);
                    s_new_count = keep_min == FLT_MAX ? 0.f : keep_min;
                }
            }
            __syncthreads();
            const int n_re = s_n_re;
            if (n_re) {
                for (int j = threadIdx.x; j < bs; j += kKmThreads) {          // the n_re rows of smallest key, in key order
                    const uint64_t key = s_key[j];
                    int rank = 0;
                    for (int i = 0; i < bs && rank < n_re; ++i) rank += (s_key[i] < key || (s_key[i] == key && i < j));
                    if (rank < n_re) s_pick[rank] = j;
                }
                __syncthreads();
                unsigned mask = s_starved;
                for (int q = 0; q < n_re; ++q) {
                    const int ci = __ffs((int)mask) - 1;
                    mask &= mask - 1;
                    const float* x = f.d_points + (int64_t)s_idx[s_pick[q]] * channels;
                    for (int c = threadIdx.x; c < channels; c += kKmThreads) cent[ci * stride + c] = x[c];
                    if (threadIdx.x == 0) s_counts[ci] = s_new_count;
                }
            }
            __syncthreads();
        }

        // count-weighted update of the centres that received rows: (m * count + sum of rows) / (count + rows)
        for (int c = threadIdx.x; c < channels; c += kKmThreads) {
            for (int i = 0; i < k; ++i)
                if (s_nin[i]) cent[i * stride + c] *= s_counts[i];
            for (int j = 0; j < bs; ++j) cent[s_lab[j] * stride + c] += f.d_points[(int64_t)s_idx[j] * channels + c];
            for (int i = 0; i < k; ++i)
                if (s_nin[i]) cent[i * stride + c] = __fdiv_rn(cent[i * stride + c], s_counts[i] + (float)s_nin[i]);
        }
        __syncthreads();
        if (threadIdx.x < k) s_counts[threadIdx.x] += (float)s_nin[threadIdx.x];
        normalise_centres(cent, k, channels, stride);

        if (warp == 0) {
            double sum = 0.0;
            for (int j = lane; j < bs; j += 32) sum += (double)s_dist[j];
            for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
            const float inertia = (float)(sum / bs);
            if (lane == 0 && batch_inertia) batch_inertia[(size_t)blockIdx.x * steps + s] = inertia;
            if (lane == 0 && !explicit_rows) {
                // EWA of the batch inertia in fp64, as the reference's Python floats (no FMA contraction)
                const double bi = (double)inertia;
                if (st.steps_done == 0) st.ewa = bi;
                else st.ewa = __dadd_rn(__dmul_rn(st.ewa, 1.0 - alpha), __dmul_rn(bi, alpha));
                if (st.steps_done == 0 || st.ewa < st.ewa_min) { st.ewa_min = st.ewa; st.no_improvement = 0; }
                else st.no_improvement += 1;
                st.steps_done += 1;
                st.done = st.steps_done >= st.max_steps ||
                          (st.max_no_improvement >= 0 && st.no_improvement >= st.max_no_improvement);
                s_run = !st.done;
            }
        }
        __syncthreads();
        if (explicit_rows) break;                  // one step per explicit index list
        if (!s_run) break;
    }

    for (int i = threadIdx.x; i < k * channels; i += kKmThreads)
        f.d_centers[i] = cent[(i / channels) * stride + i % channels];
    if (threadIdx.x < k) f.d_counts[threadIdx.x] = s_counts[threadIdx.x];
    if (threadIdx.x == 0 && !explicit_rows) *f.d_state = st;
}

}  // namespace
}  // namespace sis

extern "C" int sis_kmeans_state_bytes(void) { return (int)sizeof(sis_kmeans_state); }

extern "C" int sis_kmeans_init_state(void* d_state, uint64_t seed, int batch_size, int64_t max_steps, int max_no_improvement,
                                     float reassignment_ratio, void* stream) {
    using namespace sis;
    SIS_REQUIRE(d_state, "kmeans_init_state: d_state is NULL");
    SIS_REQUIRE(batch_size >= 1 && batch_size <= kKmMaxBatch, "kmeans_init_state: batch_size %d outside [1, %d]", batch_size, kKmMaxBatch);
    SIS_REQUIRE(max_steps >= 1, "kmeans_init_state: max_steps must be >= 1");
    SIS_REQUIRE(reassignment_ratio >= 0.f && reassignment_ratio <= 1.f, "kmeans_init_state: reassignment_ratio must be in [0, 1]");
    sis_kmeans_state v{};
    v.seed = seed;
    v.max_steps = max_steps;
    v.batch_size = batch_size;
    v.max_no_improvement = max_no_improvement < 0 ? -1 : max_no_improvement;
    v.reassignment_ratio = reassignment_ratio;
    kmeans_init_state_kernel<<<1, 1, 0, (cudaStream_t)stream>>>((sis_kmeans_state*)d_state, v);
    SIS_CHECK_LAUNCH();
    return SIS_OK;
}

extern "C" int sis_kmeans_steps(const sis_kmeans_fit* fits, int n_fits, int steps, const int32_t* d_indices, int n_indices,
                                float* d_batch_inertia, void* stream) {
    using namespace sis;
    SIS_REQUIRE(fits && n_fits >= 1, "kmeans_steps: no fits");
    SIS_REQUIRE(steps >= 1, "kmeans_steps: steps must be >= 1");
    if (d_indices) {
        SIS_REQUIRE(steps == 1, "kmeans_steps: an explicit index list runs exactly one step");
        SIS_REQUIRE(n_indices >= 1 && n_indices <= kKmMaxBatch, "kmeans_steps: n_indices %d outside [1, %d]", n_indices, kKmMaxBatch);
    }
    size_t smem = 0;
    for (int i = 0; i < n_fits; ++i) {
        const sis_kmeans_fit& f = fits[i];
        SIS_REQUIRE(f.k >= 2 && f.k <= kKmMaxK, "kmeans_steps: fit %d: k = %d outside [2, %d]", i, f.k, kKmMaxK);
        SIS_REQUIRE(f.channels >= 1 && f.channels <= kKmMaxChannels, "kmeans_steps: fit %d: channels = %d outside [1, %d]", i,
                    f.channels, kKmMaxChannels);
        SIS_REQUIRE(f.n >= f.k, "kmeans_steps: fit %d: n = %lld < k = %d", i, (long long)f.n, f.k);
        SIS_REQUIRE(f.n <= INT32_MAX, "kmeans_steps: fit %d: n = %lld exceeds 2^31 - 1 rows", i, (long long)f.n);
        SIS_REQUIRE(f.d_points && f.d_centers && f.d_counts, "kmeans_steps: fit %d: NULL points, centers or counts", i);
        SIS_REQUIRE(d_indices || f.d_state, "kmeans_steps: fit %d: NULL state", i);
        const size_t b = km_smem_bytes(f.k, f.channels);
        smem = b > smem ? b : smem;
    }
    cudaStream_t s = (cudaStream_t)stream;
    int dev = 0;
    SIS_CHECK_CUDA(cudaGetDevice(&dev));
    static bool attr_set[64] = {};                 // the shared-memory limit is a per-device attribute
    if (dev >= 64 || !attr_set[dev]) {
        SIS_CHECK_CUDA(cudaFuncSetAttribute(kmeans_steps_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            (int)km_smem_bytes(kKmMaxK, kKmMaxChannels)));
        if (dev < 64) attr_set[dev] = true;
    }
    // the descriptors go to a stream-ordered device buffer: freed after the launch, no host synchronisation
    sis_kmeans_fit* d_fits = nullptr;
    const size_t bytes = sizeof(sis_kmeans_fit) * (size_t)n_fits;
    SIS_CHECK_CUDA(cudaMallocAsync((void**)&d_fits, bytes, s));
    SIS_CHECK_CUDA(cudaMemcpyAsync(d_fits, fits, bytes, cudaMemcpyHostToDevice, s));
    {
        ProfScope prof(PROF_OTHER, s);
        kmeans_steps_kernel<<<n_fits, kKmThreads, smem, s>>>(d_fits, steps, d_indices, n_indices, d_batch_inertia);
        cudaError_t e = cudaGetLastError();
        cudaFreeAsync(d_fits, s);
        if (e != cudaSuccess) {
            set_error("kmeans_steps: launch failed: %s", cudaGetErrorString(e));
            return SIS_ERR_CUDA;
        }
        count_launch();
    }
    return SIS_OK;
}
