// Stand-alone layer entry points, so that the reference's module-level forwards work outside the fused plan:
//   ModulatedConv2d.forward / StyledConv.forward   scf/networks/stylegan2/model.py:237-278, 336-342
//   ToRGB.forward                                  model.py:355-364
//   EqualLinear.forward, PixelNorm.forward         model.py:152-162, 19-20
//   NoiseInjection.forward                         model.py:287-292
// They run the same kernels as sis_generator_forward (tcgen05 or fp32 conv, blur, ToRGB, linear), one layer per
// call, with the weight repacking done per call (the fused plan does it once at prepare time and is the fast path).
// Scratch buffers are process-global and grow-only: like the reference, these entry points are not re-entrant.
#include <cmath>
#include <cstring>
#include <map>
#include "common.cuh"
#include "kernels.h"
#include "modconv_tc.h"

namespace sis {

struct Scratch {
    void* p = nullptr; size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return SIS_OK;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        SIS_CHECK_CUDA(cudaMalloc(&p, bytes));
        cap = bytes;
        return SIS_OK;
    }
    template <typename T> T* as() const { return (T*)p; }
};

struct LayerScratch {
    Scratch mod_w, s, wsq, d, w_scaled, jobs, tmp, lin_w, lin_b;
    TcConvWeights tcw;
    TcWorkspace tcws;
    size_t tc_plane_bytes = 0;
};
static LayerScratch g_ls;

__global__ void noise_injection_kernel(float* __restrict__ out, const float* __restrict__ x, const float* __restrict__ noise,
                                       const float* __restrict__ weight, int64_t hw, int64_t chw, int64_t noise_bstride, int64_t total) {
    const float w = weight[0];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = i / chw, p = i % hw;
        out[i] = __fadd_rn(x[i], __fmul_rn(w, noise[b * noise_bstride + p]));   // image + weight * noise
    }
}
__global__ void fill_kernel(float* p, float v, int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = v;
}

static int run_linear(const float* A, int lda, const float* W, const float* bias, float* C, int ldc, int M, int N, int K, int square_a,
                      int epilogue, cudaStream_t stream) {
    LinearJob j;
    j.A = A; j.lda = lda; j.W = W; j.bias = bias; j.C = C; j.ldc = ldc; j.M = M; j.N = N; j.K = K; j.square_a = square_a; j.epilogue = epilogue;
    SIS_PROPAGATE(g_ls.jobs.reserve(sizeof(LinearJob)));
    SIS_CHECK_CUDA(cudaMemcpyAsync(g_ls.jobs.p, &j, sizeof(j), cudaMemcpyHostToDevice, stream));
    return launch_linear_jobs(g_ls.jobs.as<LinearJob>(), 1, M, N, K, K % 4 == 0 && (((uintptr_t)A | (uintptr_t)W) & 15) == 0 && lda % 4 == 0, stream);
}

static int flat_grid(int64_t n) {
    int64_t b = ceil_div64(n, 256), cap = (int64_t)kNumSMs * 8;
    return (int)(b < 1 ? 1 : (b < cap ? b : cap));
}

}  // namespace sis

using namespace sis;

extern "C" int sis_pixel_norm(const float* d_x, float* d_out, int64_t rows, int dim, void* stream) {
    SIS_REQUIRE(rows >= 0 && dim >= 1, "pixel_norm: bad shape");
    if (rows == 0) return SIS_OK;
    SIS_REQUIRE(d_x && d_out, "pixel_norm: input must be a CUDA tensor (null pointer)");
    return launch_pixel_norm(d_out, d_x, rows, dim, (cudaStream_t)stream);
}

extern "C" int sis_equal_linear(const float* d_x, int64_t rows, int in_dim, const float* d_weight, const float* d_bias, int out_dim,
                                float lr_mul, int fused_lrelu, float* d_out, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    SIS_REQUIRE(rows >= 0 && rows < (1ll << 31) && in_dim >= 1 && out_dim >= 1, "equal_linear: bad shape");
    if (rows == 0) return SIS_OK;
    SIS_REQUIRE(d_x && d_weight && d_out, "equal_linear: input must be a CUDA tensor (null pointer)");
    const float scale = (float)((1.0 / std::sqrt((double)in_dim)) * (double)lr_mul);     // model.py:149
    SIS_PROPAGATE(g_ls.lin_w.reserve((size_t)in_dim * out_dim * sizeof(float)));
    SIS_PROPAGATE(launch_scale_copy(g_ls.lin_w.as<float>(), d_weight, scale, (int64_t)in_dim * out_dim, stream));
    const float* bias = nullptr;
    if (d_bias) {
        SIS_PROPAGATE(g_ls.lin_b.reserve((size_t)out_dim * sizeof(float)));
        SIS_PROPAGATE(launch_scale_copy(g_ls.lin_b.as<float>(), d_bias, lr_mul, out_dim, stream));
        bias = g_ls.lin_b.as<float>();
    }
    return run_linear(d_x, in_dim, g_ls.lin_w.as<float>(), bias, d_out, out_dim, (int)rows, out_dim, in_dim, 0,
                      fused_lrelu ? LINEAR_EPI_BIAS_LRELU : LINEAR_EPI_BIAS, stream);
}

extern "C" int sis_noise_injection(const float* d_x, const float* d_noise, int64_t noise_batch_stride, const float* d_weight, int batch,
                                   int channels, int h, int w, float* d_out, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    const int64_t hw = (int64_t)h * w, total = hw * channels * batch;
    SIS_REQUIRE(total >= 0, "noise_injection: bad shape");
    if (total == 0) return SIS_OK;
    SIS_REQUIRE(d_x && d_noise && d_weight && d_out, "noise_injection: input must be a CUDA tensor (null pointer)");
    noise_injection_kernel<<<flat_grid(total), 256, 0, stream>>>(d_out, d_x, d_noise, d_weight, hw, hw * channels, noise_batch_stride, total);
    SIS_CHECK_LAUNCH();
    return SIS_OK;
}

extern "C" int sis_to_rgb(const float* d_x, int batch, int cin, int res, const float* d_weight, const float* d_mod_weight,
                          const float* d_mod_bias, int style_dim, const float* d_style, const float* d_bias, const float* d_skip,
                          const float* d_up_kernel, float* d_out, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    SIS_REQUIRE(batch >= 0 && cin >= 1 && res >= 1 && style_dim >= 1, "to_rgb: bad shape");
    if (batch == 0) return SIS_OK;
    SIS_REQUIRE(d_x && d_weight && d_mod_weight && d_mod_bias && d_style && d_bias && d_out, "to_rgb: input must be a CUDA tensor (null pointer)");
    SIS_REQUIRE(!d_skip || d_up_kernel, "to_rgb: a skip image needs the upsample kernel");
    SIS_REQUIRE((res * res) % 4 == 0, "to_rgb: resolution must be even");
    LayerScratch& L = g_ls;
    SIS_PROPAGATE(L.mod_w.reserve((size_t)cin * style_dim * sizeof(float)));
    SIS_PROPAGATE(launch_scale_copy(L.mod_w.as<float>(), d_mod_weight, (float)(1.0 / std::sqrt((double)style_dim)), (int64_t)cin * style_dim, stream));
    SIS_PROPAGATE(L.s.reserve((size_t)batch * cin * sizeof(float)));
    SIS_PROPAGATE(run_linear(d_style, style_dim, L.mod_w.as<float>(), d_mod_bias, L.s.as<float>(), cin, batch, cin, style_dim, 0, LINEAR_EPI_BIAS, stream));
    SIS_PROPAGATE(L.w_scaled.reserve((size_t)3 * cin * sizeof(float)));
    SIS_PROPAGATE(launch_scale_copy(L.w_scaled.as<float>(), d_weight, (float)(1.0 / std::sqrt((double)cin)), (int64_t)3 * cin, stream));
    ToRgbArgs t;
    t.x = d_x; t.s = L.s.as<float>(); t.w = L.w_scaled.as<float>(); t.bias = d_bias; t.skip = d_skip; t.up_k = d_up_kernel;
    t.out = d_out; t.batch = batch; t.C = cin; t.H = res; t.W = res;
    return launch_torgb(t, stream);
}

extern "C" int sis_wavelet_to_rgb(const float* d_x, int batch, int cin, int res, const float* d_weight, const float* d_mod_weight,
                                  const float* d_mod_bias, int style_dim, const float* d_style, const float* d_bias, const float* d_skip,
                                  const float* d_iwt, const float* d_up_kernel, const float* d_dwt, float* d_out, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    SIS_REQUIRE(batch >= 0 && cin >= 1 && res >= 1 && style_dim >= 1, "wavelet_to_rgb: bad shape");
    if (batch == 0) return SIS_OK;
    SIS_REQUIRE(d_x && d_weight && d_mod_weight && d_mod_bias && d_style && d_bias && d_out, "wavelet_to_rgb: input must be a CUDA tensor (null pointer)");
    SIS_REQUIRE(!d_skip || (d_iwt && d_up_kernel && d_dwt), "wavelet_to_rgb: a skip needs the iwt, upsample and dwt taps");
    SIS_REQUIRE(res % 4 == 0, "wavelet_to_rgb: resolution must be a multiple of 4 (got %d)", res);
    LayerScratch& L = g_ls;
    SIS_PROPAGATE(L.mod_w.reserve((size_t)cin * style_dim * sizeof(float)));
    SIS_PROPAGATE(launch_scale_copy(L.mod_w.as<float>(), d_mod_weight, (float)(1.0 / std::sqrt((double)style_dim)), (int64_t)cin * style_dim, stream));
    SIS_PROPAGATE(L.s.reserve((size_t)batch * cin * sizeof(float)));
    SIS_PROPAGATE(run_linear(d_style, style_dim, L.mod_w.as<float>(), d_mod_bias, L.s.as<float>(), cin, batch, cin, style_dim, 0, LINEAR_EPI_BIAS, stream));
    SIS_PROPAGATE(L.w_scaled.reserve((size_t)12 * cin * sizeof(float)));
    SIS_PROPAGATE(launch_scale_copy(L.w_scaled.as<float>(), d_weight, (float)(1.0 / std::sqrt((double)cin)), (int64_t)12 * cin, stream));
    WaveletToRgbArgs t;
    t.x = d_x; t.s = L.s.as<float>(); t.w = L.w_scaled.as<float>(); t.bias = d_bias; t.skip = d_skip;
    t.iwt_k = d_iwt; t.up_k = d_up_kernel; t.dwt_k = d_dwt; t.final_iwt_k = nullptr;
    t.out = d_out; t.batch = batch; t.C = cin; t.H = res; t.W = res;
    ProfScope prof(PROF_TORGB, stream);
    return launch_wavelet_torgb(t, stream);
}

extern "C" int sis_modulated_conv2d(const float* d_x, int batch, int cin, int res, const float* d_weight, int cout,
                                    const float* d_mod_weight, const float* d_mod_bias, int style_dim, const float* d_style,
                                    int demodulate, int upsample, const float* d_blur_kernel, const float* d_noise,
                                    int64_t noise_batch_stride, const float* d_noise_weight, const float* d_act_bias, int activate,
                                    float* d_out, int precision, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    SIS_REQUIRE(batch >= 0 && cin >= 1 && cout >= 1 && res >= 1 && style_dim >= 1, "modulated_conv2d: bad shape");
    if (batch == 0) return SIS_OK;
    SIS_REQUIRE(d_x && d_weight && d_mod_weight && d_mod_bias && d_style && d_out, "modulated_conv2d: input must be a CUDA tensor (null pointer)");
    SIS_REQUIRE(!upsample || d_blur_kernel, "modulated_conv2d: upsample needs the blur kernel");
    SIS_REQUIRE(!d_noise || d_noise_weight, "modulated_conv2d: noise needs its weight");
    SIS_REQUIRE(precision == SIS_PRECISION_FP32 || precision == SIS_PRECISION_BF16X3, "modulated_conv2d: unknown precision %d", precision);
    LayerScratch& L = g_ls;
    const int64_t n_oi = (int64_t)cout * cin;
    const float scale = (float)(1.0 / std::sqrt((double)cin * 9.0));
    const int res_out = upsample ? 2 * res : res;
    // s = modulation(style); d = rsqrt(sum (scale*W*s)^2 + 1e-8) or 1
    SIS_PROPAGATE(L.mod_w.reserve((size_t)cin * style_dim * sizeof(float)));
    SIS_PROPAGATE(launch_scale_copy(L.mod_w.as<float>(), d_mod_weight, (float)(1.0 / std::sqrt((double)style_dim)), (int64_t)cin * style_dim, stream));
    SIS_PROPAGATE(L.s.reserve((size_t)batch * cin * sizeof(float)));
    SIS_PROPAGATE(run_linear(d_style, style_dim, L.mod_w.as<float>(), d_mod_bias, L.s.as<float>(), cin, batch, cin, style_dim, 0, LINEAR_EPI_BIAS, stream));
    SIS_PROPAGATE(L.d.reserve((size_t)batch * cout * sizeof(float)));
    if (demodulate) {
        SIS_PROPAGATE(L.wsq.reserve((size_t)n_oi * sizeof(float)));
        SIS_PROPAGATE(launch_weight_sq(L.wsq.as<float>(), d_weight, scale, n_oi, 9, stream));
        SIS_PROPAGATE(run_linear(L.s.as<float>(), cin, L.wsq.as<float>(), nullptr, L.d.as<float>(), cout, batch, cout, cin, 1, LINEAR_EPI_RSQRT_EPS, stream));
    } else {
        fill_kernel<<<flat_grid((int64_t)batch * cout), 256, 0, stream>>>(L.d.as<float>(), 1.0f, (int64_t)batch * cout);
        SIS_CHECK_LAUNCH();
    }
    float noise_w = 0.0f;
    if (d_noise) {
        SIS_CHECK_CUDA(cudaMemcpyAsync(&noise_w, d_noise_weight, sizeof(float), cudaMemcpyDeviceToHost, stream));
        SIS_CHECK_CUDA(cudaStreamSynchronize(stream));
    }
    if (upsample) SIS_PROPAGATE(L.tmp.reserve((size_t)batch * cout * (res_out + 1) * (res_out + 1) * sizeof(float)));
    const bool tc_ok = precision == SIS_PRECISION_BF16X3 && cin % 32 == 0 && cout % 32 == 0;
    if (tc_ok) {
        SIS_PROPAGATE(tc_pack_weights(L.tcw, d_weight, cin, cout, upsample != 0, scale, stream));
        // operand planes for this one layer: slot 0 in, slot 1 unused
        std::map<int, int> chan = {{res, cin}};
        const size_t need = (size_t)batch * cin * res * res * 2;
        if (need > L.tc_plane_bytes || L.tcws.batch != batch) {
            tc_free_workspace(L.tcws);
            int res_p2 = 4;                       // the workspace is sized per power-of-two resolution; round odd sizes up
            while (res_p2 < res) res_p2 *= 2;
            SIS_PROPAGATE(tc_ensure_workspace(L.tcws, batch, res_p2, cin, std::map<int, int>{{4, cin}, {8, cin}, {16, cin}, {32, cin}, {64, cin},
                                                                                          {128, cin}, {256, cin}, {512, cin}, {1024, cin}}));
            L.tc_plane_bytes = L.tcws.a_bytes;
        }
        SIS_PROPAGATE(tc_prescale_split(L.tcws, 0, d_x, L.s.as<float>(), batch, cin, res, res, stream));
        bool sep = false;
        if (upsample) {
            float k[16];
            SIS_CHECK_CUDA(cudaMemcpyAsync(k, d_blur_kernel, sizeof(k), cudaMemcpyDeviceToHost, stream));
            SIS_CHECK_CUDA(cudaStreamSynchronize(stream));
            float mx = 0.0f;
            for (int i = 0; i < 16; ++i) mx = std::max(mx, std::fabs(k[i]));
            sep = k[15] != 0.0f;
            for (int i = 0; i < 4 && sep; ++i)
                for (int j = 0; j < 4; ++j)
                    if (std::fabs(k[i * 4 + j] - k[i * 4 + 3] * k[12 + j] / k[15]) > 1e-6f * mx) sep = false;
        }
        TcConvCall call;
        call.batch = batch; call.cin = cin; call.cout = cout; call.res_in = res; call.res_out = res_out; call.up = upsample != 0;
        call.demod = L.d.as<float>(); call.noise = d_noise; call.noise_bstride = noise_batch_stride; call.noise_w = noise_w;
        call.bias = d_act_bias; call.act = activate != 0; call.blur_k = d_blur_kernel; call.blur_separable = sep;
        call.out_f32 = d_out; call.s_next = nullptr; call.in_slot = 0; call.out_slot = 1; call.upconv_tmp = L.tmp.as<float>();
        return tc_modconv(L.tcws, L.tcw, call, stream);
    }
    // fp32 CUDA-core path
    SIS_PROPAGATE(L.w_scaled.reserve((size_t)n_oi * 9 * sizeof(float)));
    if (upsample) SIS_PROPAGATE(launch_scale_flip3x3(L.w_scaled.as<float>(), d_weight, scale, n_oi, stream));
    else SIS_PROPAGATE(launch_scale_copy(L.w_scaled.as<float>(), d_weight, scale, n_oi * 9, stream));
    ModConvSimtArgs m;
    m.x = d_x; m.w = L.w_scaled.as<float>(); m.s = L.s.as<float>(); m.d = L.d.as<float>(); m.Cin = cin; m.Cout = cout; m.H = res; m.W = res;
    m.noise = d_noise; m.noise_bstride = noise_batch_stride; m.noise_w = noise_w; m.bias = d_act_bias;
    if (!upsample) {
        m.out = d_out; m.OH = res; m.OW = res; m.pad = 1; m.zero_insert = 0; m.fuse_act = activate ? 1 : 0;
        if (!activate && (d_noise || d_act_bias)) { set_error("modulated_conv2d: noise / bias without activation is not a reference layer"); return SIS_ERR_UNSUPPORTED; }
        return launch_modconv3x3_simt(m, batch, stream);
    }
    const int th = res_out + 1;
    m.out = L.tmp.as<float>(); m.OH = th; m.OW = th; m.pad = 2; m.zero_insert = 1; m.fuse_act = 0;
    SIS_PROPAGATE(launch_modconv3x3_simt(m, batch, stream));
    BlurActArgs bl;
    bl.in = L.tmp.as<float>(); bl.out = d_out; bl.planes = (int64_t)batch * cout; bl.C = cout; bl.IH = th; bl.IW = th; bl.OH = res_out; bl.OW = res_out;
    bl.blur_k = d_blur_kernel; bl.noise = d_noise; bl.noise_bstride = noise_batch_stride; bl.noise_w = noise_w; bl.bias = d_act_bias; bl.act = activate ? 1 : 0;
    return launch_blur_noise_act(bl, stream);
}
