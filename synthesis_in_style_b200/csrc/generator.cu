// Host-side plan of the StyleGAN2 generator forward (Generator.forward, scf/networks/stylegan2/model.py:479-561) and of
// the SWAGAN generator forward (scf/networks/swagan/model.py:200-286: the same conv trunk stopped at size / 2, 12-channel
// wavelet ToRGBs, and the image as the inverse Haar transform of the last skip).
// Owns repacked weights and grow-only device workspaces; every forward is a fixed sequence of launches on the
// caller's stream.  See DESIGN.md for the layer schedule and the data layout in HBM.
#include <map>
#include <string>
#include <vector>
#include <cmath>
#include <cstring>
#include "common.cuh"
#include "kernels.h"
#include "modconv_tc.h"

namespace sis {

struct DevBuf {
    void* p = nullptr; size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return SIS_OK;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        SIS_CHECK_CUDA(cudaMalloc(&p, bytes));
        cap = bytes;
        return SIS_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <typename T> T* as() const { return (T*)p; }
};

struct ConvLayer {
    int cin = 0, cout = 0, res_in = 0, res_out = 0; bool up = false;
    std::string prefix;
    DevBuf w_scaled, wsq, mod_w, mod_b, act_bias, blur_k;
    float noise_w = 0.0f;
    float blur_host[16] = {0};
    bool blur_separable = false;
    TcConvWeights tc;        // bf16 hi/lo packs for the tcgen05 path
    float* s = nullptr;      // [B, cin]  (workspace slices)
    float* d = nullptr;      // [B, cout]
};
struct RgbLayer {
    int cin = 0, res = 0; bool up = false;
    std::string prefix;
    DevBuf w_scaled, mod_w, mod_b, bias, up_k;
    DevBuf iwt_k, dwt_k;     // SWAGAN: [4 bands][2][2] Haar taps of the skip path
    float* s = nullptr;      // [B, cin]
};

}  // namespace sis

using namespace sis;

struct sis_generator {
    int size = 0, style_dim = 0, n_mlp = 0, channel_multiplier = 2;
    // variant: StyleGAN2 = 3-channel ToRGBs, trunk at the image size; SWAGAN = 12-channel wavelet ToRGBs, trunk at
    // size / 2 and the image written by the last ToRGB through the generator's inverse Haar transform (`iwt_k`)
    int rgb_channels = 3, trunk_size = 0;
    DevBuf iwt_k;
    int log_size = 0, num_layers = 0, n_latent = 0;
    std::map<int, int> channels;
    std::map<std::string, std::pair<const float*, int64_t>> params;
    bool prepared = false;
    std::vector<DevBuf> mlp_w, mlp_b;
    DevBuf const_input;
    std::vector<ConvLayer> convs;
    std::vector<RgbLayer> rgbs;
    // workspaces
    int ws_batch = -1;
    DevBuf latent, wbuf[2], mlp_tmp[2], styles, demods, jobs_dev, act_pp[2], upconv_tmp, skip_pp[2];
    DevBuf style_tmp[2], style_jobs;
    int64_t style_rows_cap = 0;
    std::vector<LinearJob> host_jobs;  // [mlp*2 styles][mod jobs][demod jobs]
    int n_mod_jobs = 0, n_demod_jobs = 0, max_mod_n = 0, max_demod_n = 0, max_demod_k = 0;
    TcWorkspace tc_ws;
};

static int act_channels(const sis_generator* g, int idx, int* res) {
    // capture idx: 0 const input (4x4), 1 conv1 (4x4), then two per resolution
    int r = idx <= 1 ? 4 : (1 << ((idx - 2) / 2 + 3));
    if (res) *res = r;
    return g->channels.at(r);
}

static sis_generator* new_plan(int size, int trunk_size, int rgb_channels, int style_dim, int n_mlp, int channel_multiplier) {
    sis_generator* g = new sis_generator();
    g->size = size; g->style_dim = style_dim; g->n_mlp = n_mlp; g->channel_multiplier = channel_multiplier;
    g->rgb_channels = rgb_channels; g->trunk_size = trunk_size;
    g->log_size = (int)std::lround(std::log2((double)trunk_size));
    g->num_layers = (g->log_size - 2) * 2 + 1;
    g->n_latent = g->log_size * 2 - 2;
    // Generator.get_channels, model.py:443-455
    g->channels = {{4, 512}, {8, 512}, {16, 512}, {32, 512}, {64, 256 * channel_multiplier}, {128, 128 * channel_multiplier},
                   {256, 64 * channel_multiplier}, {512, 32 * channel_multiplier}, {1024, 16 * channel_multiplier}};
    g->mlp_w.resize(n_mlp); g->mlp_b.resize(n_mlp);
    // StyledConv layers in execution order: conv1, then (up, plain) per resolution; ToRGB per resolution
    int cin = g->channels[4];
    ConvLayer c1; c1.cin = cin; c1.cout = cin; c1.res_in = 4; c1.res_out = 4; c1.up = false; c1.prefix = "conv1";
    g->convs.push_back(std::move(c1));
    RgbLayer r1; r1.cin = cin; r1.res = 4; r1.up = false; r1.prefix = "to_rgb1";
    g->rgbs.push_back(std::move(r1));
    for (int i = 3, j = 0; i <= g->log_size; ++i, ++j) {
        int res = 1 << i, cout = g->channels[res];
        ConvLayer a; a.cin = cin; a.cout = cout; a.res_in = res / 2; a.res_out = res; a.up = true;
        a.prefix = "convs." + std::to_string(2 * j);
        ConvLayer b; b.cin = cout; b.cout = cout; b.res_in = res; b.res_out = res; b.up = false;
        b.prefix = "convs." + std::to_string(2 * j + 1);
        g->convs.push_back(std::move(a)); g->convs.push_back(std::move(b));
        RgbLayer r; r.cin = cout; r.res = res; r.up = true; r.prefix = "to_rgbs." + std::to_string(j);
        g->rgbs.push_back(std::move(r));
        cin = cout;
    }
    return g;
}

extern "C" int sis_generator_create(int size, int style_dim, int n_mlp, int channel_multiplier, sis_generator** out) {
    SIS_REQUIRE(out != nullptr, "generator_create: out is null");
    SIS_REQUIRE(size >= 8 && size <= 1024 && (size & (size - 1)) == 0, "generator_create: size must be a power of two in [8, 1024] (got %d)", size);
    SIS_REQUIRE(style_dim >= 1 && n_mlp >= 0 && channel_multiplier >= 1, "generator_create: bad style_dim / n_mlp / channel_multiplier");
    *out = new_plan(size, size, 3, style_dim, n_mlp, channel_multiplier);
    return SIS_OK;
}

extern "C" int sis_generator_create_swagan(int size, int style_dim, int n_mlp, int channel_multiplier, sis_generator** out) {
    SIS_REQUIRE(out != nullptr, "generator_create_swagan: out is null");
    SIS_REQUIRE(size >= 16 && size <= 1024 && (size & (size - 1)) == 0, "generator_create_swagan: size must be a power of two in [16, 1024] (got %d)", size);
    SIS_REQUIRE(style_dim >= 1 && n_mlp >= 0 && channel_multiplier >= 1, "generator_create_swagan: bad style_dim / n_mlp / channel_multiplier");
    *out = new_plan(size, size / 2, 12, style_dim, n_mlp, channel_multiplier);
    return SIS_OK;
}

extern "C" int sis_generator_destroy(sis_generator* g) {
    if (!g) return SIS_OK;
    for (auto& b : g->mlp_w) b.release();
    for (auto& b : g->mlp_b) b.release();
    g->const_input.release();
    for (auto& c : g->convs) {
        c.w_scaled.release(); c.wsq.release(); c.mod_w.release(); c.mod_b.release(); c.act_bias.release(); c.blur_k.release();
        tc_free_weights(c.tc);
    }
    for (auto& r : g->rgbs) {
        r.w_scaled.release(); r.mod_w.release(); r.mod_b.release(); r.bias.release(); r.up_k.release(); r.iwt_k.release(); r.dwt_k.release();
    }
    g->iwt_k.release();
    DevBuf* bufs[] = {&g->latent, &g->wbuf[0], &g->wbuf[1], &g->mlp_tmp[0], &g->mlp_tmp[1], &g->styles, &g->demods, &g->jobs_dev,
                      &g->act_pp[0], &g->act_pp[1], &g->upconv_tmp, &g->skip_pp[0], &g->skip_pp[1], &g->style_tmp[0],
                      &g->style_tmp[1], &g->style_jobs};
    for (DevBuf* b : bufs) b->release();
    tc_free_workspace(g->tc_ws);
    delete g;
    return SIS_OK;
}

extern "C" int sis_generator_set_param(sis_generator* g, const char* key, const float* d_ptr, int64_t numel) {
    SIS_REQUIRE(g && key, "generator_set_param: null generator / key");
    SIS_REQUIRE(d_ptr != nullptr || numel == 0, "generator_set_param: %s must be a CUDA tensor (null pointer)", key);
    g->params[key] = {d_ptr, numel};
    g->prepared = false;
    return SIS_OK;
}

extern "C" int sis_generator_n_latent(const sis_generator* g) { return g ? g->n_latent : -1; }
extern "C" int sis_generator_num_layers(const sis_generator* g) { return g ? g->num_layers : -1; }
extern "C" int sis_generator_activation_shape(const sis_generator* g, int idx, int* channels, int* res) {
    SIS_REQUIRE(g && idx >= 0 && idx < g->n_latent, "generator_activation_shape: bad index");
    int r; int c = act_channels(g, idx, &r);
    if (channels) *channels = c;
    if (res) *res = r;
    return SIS_OK;
}

static int get_param(sis_generator* g, const std::string& key, int64_t expect, const float** out) {
    auto it = g->params.find(key);
    if (it == g->params.end()) { set_error("generator: missing parameter '%s'", key.c_str()); return SIS_ERR_STATE; }
    if (it->second.second != expect) {
        set_error("generator: parameter '%s' has %lld elements, expected %lld", key.c_str(), (long long)it->second.second, (long long)expect);
        return SIS_ERR_INVALID;
    }
    *out = it->second.first;
    return SIS_OK;
}

static int copy_param(sis_generator* g, const std::string& key, int64_t n, DevBuf& dst, float scale, cudaStream_t stream) {
    const float* src;
    SIS_PROPAGATE(get_param(g, key, n, &src));
    SIS_PROPAGATE(dst.reserve((size_t)n * sizeof(float)));
    if (scale == 1.0f) SIS_CHECK_CUDA(cudaMemcpyAsync(dst.p, src, (size_t)n * sizeof(float), cudaMemcpyDeviceToDevice, stream));
    else SIS_PROPAGATE(launch_scale_copy(dst.as<float>(), src, scale, n, stream));
    return SIS_OK;
}

// `<prefix>.{ll,lh,hl,hh}` (2x2 each, swagan/model.py:28-68) -> dst [4 bands][2][2]
static int copy_haar_taps(sis_generator* g, const std::string& prefix, DevBuf& dst, cudaStream_t stream) {
    SIS_PROPAGATE(dst.reserve(16 * sizeof(float)));
    const char* bands[4] = {"ll", "lh", "hl", "hh"};
    for (int i = 0; i < 4; ++i) {
        const float* src;
        SIS_PROPAGATE(get_param(g, prefix + "." + bands[i], 4, &src));
        SIS_CHECK_CUDA(cudaMemcpyAsync(dst.as<float>() + 4 * i, src, 4 * sizeof(float), cudaMemcpyDeviceToDevice, stream));
    }
    return SIS_OK;
}

extern "C" int sis_generator_prepare(sis_generator* g, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    SIS_REQUIRE(g != nullptr, "generator_prepare: null generator");
    const int sd = g->style_dim;
    const float lr_mlp = 0.01f;
    // EqualLinear (model.py:149): scale = lr_mul / sqrt(in_dim); bias * lr_mul
    const float mlp_scale = (float)((1.0 / std::sqrt((double)sd)) * (double)lr_mlp);
    for (int i = 0; i < g->n_mlp; ++i) {
        std::string p = "style." + std::to_string(i + 1);
        SIS_PROPAGATE(copy_param(g, p + ".weight", (int64_t)sd * sd, g->mlp_w[i], mlp_scale, stream));
        SIS_PROPAGATE(copy_param(g, p + ".bias", sd, g->mlp_b[i], lr_mlp, stream));
    }
    const int c4 = g->channels[4];
    SIS_PROPAGATE(copy_param(g, "input.input", (int64_t)c4 * 16, g->const_input, 1.0f, stream));
    const float mod_scale = (float)(1.0 / std::sqrt((double)sd));
    std::vector<float*> noise_w_dst;
    for (auto& c : g->convs) {
        const int64_t n_oi = (int64_t)c.cout * c.cin;
        const float scale = (float)(1.0 / std::sqrt((double)c.cin * 9.0));   // model.py:213-214
        const float* w;
        SIS_PROPAGATE(get_param(g, c.prefix + ".conv.weight", n_oi * 9, &w));
        SIS_PROPAGATE(c.w_scaled.reserve((size_t)n_oi * 9 * sizeof(float)));
        if (c.up) SIS_PROPAGATE(launch_scale_flip3x3(c.w_scaled.as<float>(), w, scale, n_oi, stream));
        else SIS_PROPAGATE(launch_scale_copy(c.w_scaled.as<float>(), w, scale, n_oi * 9, stream));
        SIS_PROPAGATE(c.wsq.reserve((size_t)n_oi * sizeof(float)));
        SIS_PROPAGATE(launch_weight_sq(c.wsq.as<float>(), w, scale, n_oi, 9, stream));
        SIS_PROPAGATE(copy_param(g, c.prefix + ".conv.modulation.weight", (int64_t)c.cin * sd, c.mod_w, mod_scale, stream));
        SIS_PROPAGATE(copy_param(g, c.prefix + ".conv.modulation.bias", c.cin, c.mod_b, 1.0f, stream));
        SIS_PROPAGATE(copy_param(g, c.prefix + ".activate.bias", c.cout, c.act_bias, 1.0f, stream));
        if (c.up) {
            SIS_PROPAGATE(copy_param(g, c.prefix + ".conv.blur.kernel", 16, c.blur_k, 1.0f, stream));
            SIS_CHECK_CUDA(cudaMemcpyAsync(c.blur_host, c.blur_k.p, 16 * sizeof(float), cudaMemcpyDeviceToHost, stream));
        }
        const float* nw;
        SIS_PROPAGATE(get_param(g, c.prefix + ".noise.weight", 1, &nw));
        SIS_CHECK_CUDA(cudaMemcpyAsync(&c.noise_w, nw, sizeof(float), cudaMemcpyDeviceToHost, stream));
        SIS_PROPAGATE(tc_pack_weights(c.tc, w, c.cin, c.cout, c.up, scale, stream));
    }
    const int rc = g->rgb_channels;
    for (auto& r : g->rgbs) {
        const float scale = (float)(1.0 / std::sqrt((double)r.cin));          // 1x1 kernel: fan_in = cin
        SIS_PROPAGATE(copy_param(g, r.prefix + ".conv.weight", (int64_t)rc * r.cin, r.w_scaled, scale, stream));
        SIS_PROPAGATE(copy_param(g, r.prefix + ".conv.modulation.weight", (int64_t)r.cin * sd, r.mod_w, mod_scale, stream));
        SIS_PROPAGATE(copy_param(g, r.prefix + ".conv.modulation.bias", r.cin, r.mod_b, 1.0f, stream));
        SIS_PROPAGATE(copy_param(g, r.prefix + ".bias", rc, r.bias, 1.0f, stream));
        if (r.up) SIS_PROPAGATE(copy_param(g, r.prefix + ".upsample.kernel", 16, r.up_k, 1.0f, stream));
        if (r.up && rc == 12) {
            SIS_PROPAGATE(copy_haar_taps(g, r.prefix + ".iwt", r.iwt_k, stream));
            SIS_PROPAGATE(copy_haar_taps(g, r.prefix + ".dwt", r.dwt_k, stream));
        }
    }
    if (rc == 12) SIS_PROPAGATE(copy_haar_taps(g, "iwt", g->iwt_k, stream));
    SIS_CHECK_CUDA(cudaStreamSynchronize(stream));  // noise weights and blur taps are read on the host
    for (auto& c : g->convs) {
        if (!c.up) continue;
        // rank-1 test k[i][j] == k[i][0]*k[0][j]/k[0][0]: the reference's make_kernel([1,3,3,1]) always passes
        const float* k = c.blur_host;
        float mx = 0.0f;
        for (int i = 0; i < 16; ++i) mx = std::max(mx, std::fabs(k[i]));
        bool sep = k[15] != 0.0f;   // flipped taps: element [0][0] of the flipped kernel is k[3][3]
        for (int i = 0; i < 4 && sep; ++i)
            for (int j = 0; j < 4; ++j)
                if (std::fabs(k[i * 4 + j] - k[i * 4 + 3] * k[12 + j] / k[15]) > 1e-6f * mx) sep = false;
        c.blur_separable = sep;
    }
    g->prepared = true;
    g->ws_batch = -1;
    return SIS_OK;
}

// ---- style MLP ------------------------------------------------------------------------------------------------
static int run_style_mlp(sis_generator* g, const float* z, float* w_out, int64_t n, float* tmp0, float* tmp1,
                         LinearJob* d_jobs, LinearJob* h_jobs, cudaStream_t stream) {
    // PixelNorm + n_mlp x (EqualLinear + fused lrelu), model.py:383-392
    const int sd = g->style_dim;
    SIS_PROPAGATE(launch_pixel_norm(g->n_mlp ? tmp0 : w_out, z, n, sd, stream));
    float* cur = tmp0;
    for (int i = 0; i < g->n_mlp; ++i) {
        LinearJob& j = h_jobs[i];
        float* dst = (i == g->n_mlp - 1) ? w_out : (cur == tmp0 ? tmp1 : tmp0);
        j.A = cur; j.lda = sd; j.W = g->mlp_w[i].as<float>(); j.bias = g->mlp_b[i].as<float>(); j.C = dst; j.ldc = sd;
        j.M = (int)n; j.N = sd; j.K = sd; j.square_a = 0; j.epilogue = LINEAR_EPI_BIAS_LRELU;
        cur = dst;
    }
    if (g->n_mlp) {
        SIS_CHECK_CUDA(cudaMemcpyAsync(d_jobs, h_jobs, sizeof(LinearJob) * g->n_mlp, cudaMemcpyHostToDevice, stream));
        for (int i = 0; i < g->n_mlp; ++i) SIS_PROPAGATE(launch_linear_jobs(d_jobs + i, 1, (int)n, sd, sd, sd % 4 == 0, stream));
    }
    return SIS_OK;
}

extern "C" int sis_generator_style(sis_generator* g, const float* d_z, float* d_w, int64_t n, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    SIS_REQUIRE(g && g->prepared, "generator_style: generator not prepared");
    if (n == 0) return SIS_OK;
    SIS_REQUIRE(d_z && d_w && n > 0 && n < (1ll << 31), "generator_style: bad arguments");
    const size_t bytes = (size_t)n * g->style_dim * sizeof(float);
    SIS_PROPAGATE(g->style_tmp[0].reserve(bytes));
    SIS_PROPAGATE(g->style_tmp[1].reserve(bytes));
    SIS_PROPAGATE(g->style_jobs.reserve(sizeof(LinearJob) * (g->n_mlp + 1)));
    std::vector<LinearJob> jobs(g->n_mlp + 1);
    SIS_PROPAGATE(run_style_mlp(g, d_z, d_w, n, g->style_tmp[0].as<float>(), g->style_tmp[1].as<float>(),
                                g->style_jobs.as<LinearJob>(), jobs.data(), stream));
    // jobs vector is pageable host memory: cudaMemcpyAsync from pageable memory returns after staging, safe to free.
    return SIS_OK;
}

// ---- workspace ------------------------------------------------------------------------------------------------
static int ensure_workspace(sis_generator* g, int B) {
    if (g->ws_batch == B) return SIS_OK;
    const int sd = g->style_dim;
    SIS_PROPAGATE(g->latent.reserve((size_t)B * g->n_latent * sd * sizeof(float)));
    for (int i = 0; i < 2; ++i) {
        SIS_PROPAGATE(g->wbuf[i].reserve((size_t)B * sd * sizeof(float)));
        SIS_PROPAGATE(g->mlp_tmp[i].reserve((size_t)B * sd * sizeof(float)));
    }
    size_t s_total = 0, d_total = 0;
    for (auto& c : g->convs) { s_total += (size_t)B * c.cin; d_total += (size_t)B * c.cout; }
    for (auto& r : g->rgbs) s_total += (size_t)B * r.cin;
    SIS_PROPAGATE(g->styles.reserve(s_total * sizeof(float)));
    SIS_PROPAGATE(g->demods.reserve(d_total * sizeof(float)));
    float* sp = g->styles.as<float>(); float* dp = g->demods.as<float>();
    for (auto& c : g->convs) { c.s = sp; sp += (size_t)B * c.cin; c.d = dp; dp += (size_t)B * c.cout; }
    for (auto& r : g->rgbs) { r.s = sp; sp += (size_t)B * r.cin; }
    size_t max_act = 0, max_up = 0;
    for (auto& c : g->convs) {
        max_act = std::max(max_act, (size_t)B * c.cout * c.res_out * c.res_out);
        if (c.up) max_up = std::max(max_up, (size_t)B * c.cout * (c.res_out + 1) * (c.res_out + 1));
    }
    for (int i = 0; i < 2; ++i) {
        SIS_PROPAGATE(g->act_pp[i].reserve(max_act * sizeof(float)));
        SIS_PROPAGATE(g->skip_pp[i].reserve((size_t)B * 3 * g->size * g->size * sizeof(float)));
    }
    SIS_PROPAGATE(g->upconv_tmp.reserve(max_up * sizeof(float)));

    // linear jobs: [2*n_mlp style-MLP jobs][modulation jobs][demod jobs]
    const int n_mlp_jobs = 2 * g->n_mlp;
    g->n_mod_jobs = (int)(g->convs.size() + g->rgbs.size());
    g->n_demod_jobs = (int)g->convs.size();
    g->host_jobs.assign(n_mlp_jobs + g->n_mod_jobs + g->n_demod_jobs, LinearJob());
    SIS_PROPAGATE(g->jobs_dev.reserve(g->host_jobs.size() * sizeof(LinearJob)));
    g->max_mod_n = 0; g->max_demod_n = 0; g->max_demod_k = 0;
    int ji = n_mlp_jobs;
    const float* lat = g->latent.as<float>();
    const int ldl = g->n_latent * sd;
    auto mod_job = [&](const float* mod_w, const float* mod_b, float* s, int cin, int latent_idx) {
        LinearJob& j = g->host_jobs[ji++];
        j.A = lat + (size_t)latent_idx * sd; j.lda = ldl; j.W = mod_w; j.bias = mod_b; j.C = s; j.ldc = cin;
        j.M = B; j.N = cin; j.K = sd; j.square_a = 0; j.epilogue = LINEAR_EPI_BIAS;
        g->max_mod_n = std::max(g->max_mod_n, cin);
    };
    // StyledConv layer L uses latent[:, L]; ToRGB r uses latent[:, 2r+1]  (model.py:534-552)
    for (size_t L = 0; L < g->convs.size(); ++L) mod_job(g->convs[L].mod_w.as<float>(), g->convs[L].mod_b.as<float>(), g->convs[L].s, g->convs[L].cin, (int)L);
    for (size_t r = 0; r < g->rgbs.size(); ++r) mod_job(g->rgbs[r].mod_w.as<float>(), g->rgbs[r].mod_b.as<float>(), g->rgbs[r].s, g->rgbs[r].cin, (int)(2 * r + 1));
    for (auto& c : g->convs) {
        LinearJob& j = g->host_jobs[ji++];
        j.A = c.s; j.lda = c.cin; j.W = c.wsq.as<float>(); j.bias = nullptr; j.C = c.d; j.ldc = c.cout;
        j.M = B; j.N = c.cout; j.K = c.cin; j.square_a = 1; j.epilogue = LINEAR_EPI_RSQRT_EPS;
        g->max_demod_n = std::max(g->max_demod_n, c.cout);
        g->max_demod_k = std::max(g->max_demod_k, c.cin);
    }
    g->ws_batch = B;
    return SIS_OK;
}

// label jobs attached to activation `idx`; `rgb` = the ToRGB reading the same tensor (fused when possible)
static int run_label_jobs(const sis_forward_args* a, int idx, const float* act, int batch, int C, int res, const ToRgbArgs* rgb,
                          bool* rgb_done, cudaStream_t stream) {
    if (rgb_done) *rgb_done = false;
    for (int j = 0; j < a->n_label_jobs; ++j) {
        const sis_label_job& job = a->label_jobs[j];
        if (job.activation_idx != idx) continue;
        LabelArgs la;
        la.act = act; la.batch = batch; la.C = C; la.H = res; la.W = res; la.centroids = job.d_centroids; la.k = job.k;
        la.class_bits = job.d_cluster_class_bits; la.n_class = job.n_class; la.S = job.image_size;
        la.ids_u8 = job.d_ids_u8; la.ids_i64 = job.d_ids_i64; la.masks = job.d_masks; la.margin = job.d_margin; la.hist = job.d_hist;
        bool fused = false;
        const bool try_fuse = rgb && rgb_done && !*rgb_done;
        SIS_PROPAGATE(launch_label(la, 0, try_fuse ? rgb : nullptr, &fused, stream));
        if (fused) *rgb_done = true;
    }
    return SIS_OK;
}

extern "C" int sis_generator_check(sis_generator* g, void* stream_) {
    SIS_REQUIRE(g != nullptr, "generator_check: null generator");
    return tc_check_error(g->tc_ws, (cudaStream_t)stream_);
}

extern "C" int sis_generator_forward(sis_generator* g, const sis_forward_args* a, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    SIS_REQUIRE(g && a, "generator_forward: null argument");
    if (!g->prepared) { set_error("generator_forward: sis_generator_prepare has not been called since the last set_param"); return SIS_ERR_STATE; }
    const int B = a->batch;
    SIS_REQUIRE(B >= 0, "generator_forward: negative batch");
    if (B == 0) return SIS_OK;
    SIS_REQUIRE(a->n_styles == 1 || a->n_styles == 2, "generator_forward: n_styles must be 1 or 2");
    SIS_REQUIRE(a->d_styles[0] && (a->n_styles == 1 || a->d_styles[1]), "generator_forward: styles must be CUDA tensors (null pointer)");
    SIS_REQUIRE(!(a->styles_are_wplus && a->n_styles != 1), "generator_forward: a W+ latent cannot be mixed with a second style");
    SIS_REQUIRE(!(a->styles_are_wplus && !a->input_is_latent), "generator_forward: W+ input requires input_is_latent");
    SIS_REQUIRE(a->n_styles == 1 || (a->inject_index >= 0 && a->inject_index <= g->n_latent), "generator_forward: inject_index out of range");
    SIS_REQUIRE(!(a->truncation < 1.0f) || a->d_truncation_latent, "generator_forward: truncation < 1 needs truncation_latent");
    SIS_REQUIRE(a->d_noise && a->noise_batch_stride, "generator_forward: noise list is null");
    SIS_REQUIRE(a->d_image, "generator_forward: image output is null");
    SIS_REQUIRE(a->precision == SIS_PRECISION_FP32 || a->precision == SIS_PRECISION_BF16X3, "generator_forward: unknown precision %d", a->precision);
    for (int l = 0; l < g->num_layers; ++l) SIS_REQUIRE(a->d_noise[l] != nullptr, "generator_forward: noise[%d] is null", l);
    SIS_REQUIRE(a->n_label_jobs >= 0 && (a->n_label_jobs == 0 || a->label_jobs), "generator_forward: label_jobs is null");
    for (int j = 0; j < a->n_label_jobs; ++j)
        SIS_REQUIRE(a->label_jobs[j].activation_idx >= 0 && a->label_jobs[j].activation_idx < g->n_latent,
                    "generator_forward: label job %d names activation %d", j, a->label_jobs[j].activation_idx);
    SIS_PROPAGATE(ensure_workspace(g, B));
    const int sd = g->style_dim;
    const bool tc = a->precision == SIS_PRECISION_BF16X3;

    // 1. styles -> w
    ProfScope* prof_map = new ProfScope(PROF_MAPPING, stream);
    struct ProfGuard { ProfScope** p; ~ProfGuard() { if (*p) { delete *p; *p = nullptr; } } } prof_guard{&prof_map};
    const float* w[2] = {a->d_styles[0], a->n_styles == 2 ? a->d_styles[1] : nullptr};
    LinearJob* d_jobs = g->jobs_dev.as<LinearJob>();
    if (!a->input_is_latent) {
        for (int j = 0; j < a->n_styles; ++j) {
            SIS_PROPAGATE(run_style_mlp(g, a->d_styles[j], g->wbuf[j].as<float>(), B, g->mlp_tmp[0].as<float>(), g->mlp_tmp[1].as<float>(),
                                        d_jobs + j * g->n_mlp, g->host_jobs.data() + j * g->n_mlp, stream));
            w[j] = g->wbuf[j].as<float>();
        }
    }
    // 2. latent [B, n_latent, sd]
    SIS_PROPAGATE(launch_assemble_latent(g->latent.as<float>(), w[0], w[1], a->styles_are_wplus, a->n_styles == 2 ? a->inject_index : g->n_latent,
                                         a->truncation, a->d_truncation_latent, a->truncation_latent_rows, B, g->n_latent, sd, stream));
    if (a->d_latent_out)
        SIS_CHECK_CUDA(cudaMemcpyAsync(a->d_latent_out, g->latent.p, (size_t)B * g->n_latent * sd * sizeof(float), cudaMemcpyDeviceToDevice, stream));
    // 3. modulation + demodulation for every layer (two batched launches)
    const int n_mlp_jobs = 2 * g->n_mlp;
    SIS_CHECK_CUDA(cudaMemcpyAsync(d_jobs + n_mlp_jobs, g->host_jobs.data() + n_mlp_jobs, sizeof(LinearJob) * (g->n_mod_jobs + g->n_demod_jobs),
                                   cudaMemcpyHostToDevice, stream));
    SIS_PROPAGATE(launch_linear_jobs(d_jobs + n_mlp_jobs, g->n_mod_jobs, B, g->max_mod_n, sd, sd % 4 == 0, stream));
    SIS_PROPAGATE(launch_linear_jobs(d_jobs + n_mlp_jobs + g->n_mod_jobs, g->n_demod_jobs, B, g->max_demod_n, g->max_demod_k, true, stream));

    delete prof_map; prof_map = nullptr;

    // 4. layers
    auto act_dst = [&](int idx, int pp) -> float* {
        if (a->d_activations && a->d_activations[idx]) return a->d_activations[idx];
        return g->act_pp[pp].as<float>();
    };
    if (tc) SIS_PROPAGATE(tc_ensure_workspace(g->tc_ws, B, g->trunk_size, g->channels[4], g->channels));

    float* x = act_dst(0, 0);
    SIS_PROPAGATE(launch_const_input(x, g->const_input.as<float>(), (int64_t)g->channels[4] * 16, B, stream));
    if (tc) SIS_PROPAGATE(tc_prescale_split(g->tc_ws, 0, x, g->convs[0].s, B, g->convs[0].cin, 4, 4, stream));
    SIS_PROPAGATE(run_label_jobs(a, 0, x, B, g->channels[4], 4, nullptr, nullptr, stream));
    int pp = 1;
    const float* skip = nullptr;
    int rgb_i = 0;
    for (size_t L = 0; L < g->convs.size(); ++L) {
        ConvLayer& c = g->convs[L];
        float* y = act_dst((int)L + 1, pp);
        const float* noise = a->d_noise[L];
        const int64_t nstride = a->noise_batch_stride[L];
        const float* s_next = (L + 1 < g->convs.size()) ? g->convs[L + 1].s : nullptr;
        if (tc) {
            TcConvCall call;
            call.batch = B; call.cin = c.cin; call.cout = c.cout; call.res_in = c.res_in; call.res_out = c.res_out; call.up = c.up;
            call.demod = c.d; call.noise = noise; call.noise_bstride = nstride; call.noise_w = c.noise_w; call.bias = c.act_bias.as<float>();
            call.blur_k = c.up ? c.blur_k.as<float>() : nullptr; call.blur_separable = c.blur_separable; call.out_f32 = y; call.s_next = s_next;
            call.in_slot = (int)(L & 1); call.out_slot = (int)((L + 1) & 1);
            call.upconv_tmp = g->upconv_tmp.as<float>();
            SIS_PROPAGATE(tc_modconv(g->tc_ws, c.tc, call, stream));
        } else {
            ModConvSimtArgs m;
            m.x = x; m.w = c.w_scaled.as<float>(); m.s = c.s; m.d = c.d; m.Cin = c.cin; m.Cout = c.cout;
            m.H = c.res_in; m.W = c.res_in; m.noise = noise; m.noise_bstride = nstride; m.noise_w = c.noise_w; m.bias = c.act_bias.as<float>();
            if (!c.up) {
                m.out = y; m.OH = c.res_out; m.OW = c.res_out; m.pad = 1; m.zero_insert = 0; m.fuse_act = 1;
                ProfScope prof(PROF_CONV_SIMT, stream);
                SIS_PROPAGATE(launch_modconv3x3_simt(m, B, stream));
            } else {
                const int th = c.res_out + 1;
                m.out = g->upconv_tmp.as<float>(); m.OH = th; m.OW = th; m.pad = 2; m.zero_insert = 1; m.fuse_act = 0;
                {
                    ProfScope prof(PROF_CONV_SIMT, stream);
                    SIS_PROPAGATE(launch_modconv3x3_simt(m, B, stream));
                }
                BlurActArgs bl;
                bl.in = g->upconv_tmp.as<float>(); bl.out = y; bl.planes = (int64_t)B * c.cout; bl.C = c.cout; bl.IH = th; bl.IW = th;
                bl.OH = c.res_out; bl.OW = c.res_out; bl.blur_k = c.blur_k.as<float>(); bl.noise = noise; bl.noise_bstride = nstride;
                bl.noise_w = c.noise_w; bl.bias = c.act_bias.as<float>(); bl.act = 1;
                ProfScope prof(PROF_BLUR_SIMT, stream);
                SIS_PROPAGATE(launch_blur_noise_act(bl, stream));
            }
        }
        x = y; pp ^= 1;
        if (L % 2 == 0 && g->rgb_channels == 12) {   // SWAGAN ToRGB (swagan/model.py:253-284); labelling runs unfused
            RgbLayer& r = g->rgbs[rgb_i];
            const bool last = rgb_i + 1 == (int)g->rgbs.size();
            SIS_PROPAGATE(run_label_jobs(a, (int)L + 1, x, B, c.cout, c.res_out, nullptr, nullptr, stream));
            WaveletToRgbArgs t;
            t.x = x; t.s = r.s; t.w = r.w_scaled.as<float>(); t.bias = r.bias.as<float>(); t.skip = skip;
            t.iwt_k = r.iwt_k.as<float>(); t.up_k = r.up_k.as<float>(); t.dwt_k = r.dwt_k.as<float>();
            t.final_iwt_k = last ? g->iwt_k.as<float>() : nullptr;     // the last one writes the image (:285)
            t.out = last ? a->d_image : g->skip_pp[rgb_i & 1].as<float>();
            t.batch = B; t.C = r.cin; t.H = r.res; t.W = r.res;
            {
                ProfScope prof(PROF_TORGB, stream);
                SIS_PROPAGATE(launch_wavelet_torgb(t, stream));
            }
            skip = t.out;
            ++rgb_i;
        } else if (L % 2 == 0) {  // ToRGB after conv1 and after the second conv of every block (model.py:538,550)
            RgbLayer& r = g->rgbs[rgb_i];
            const bool last = rgb_i + 1 == (int)g->rgbs.size();
            float* out = last ? a->d_image : g->skip_pp[rgb_i & 1].as<float>();
            ToRgbArgs t;
            t.x = x; t.s = r.s; t.w = r.w_scaled.as<float>(); t.bias = r.bias.as<float>(); t.skip = skip; t.up_k = r.up ? r.up_k.as<float>() : nullptr;
            t.out = out; t.batch = B; t.C = r.cin; t.H = r.res; t.W = r.res;
            bool rgb_done = false;
            SIS_PROPAGATE(run_label_jobs(a, (int)L + 1, x, B, c.cout, c.res_out, &t, &rgb_done, stream));
            if (!rgb_done) {
                ProfScope prof(PROF_TORGB, stream);
                SIS_PROPAGATE(launch_torgb(t, stream));
            }
            skip = out;
            ++rgb_i;
        } else {
            SIS_PROPAGATE(run_label_jobs(a, (int)L + 1, x, B, c.cout, c.res_out, nullptr, nullptr, stream));
        }
    }
    return SIS_OK;
}
