// tcgen05 / TMA implicit-GEMM modulated convolution (sis_precision BF16X3) — internal interface.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <map>

namespace sis {

// bf16 hi/lo split of scale*W, layout [tap = ky*3+kx][Cout][Cin] (K-major rows of Cin), shared by the plain
// conv and the transposed conv (which indexes taps directly, without the flip).
struct TcConvWeights {
    void* hi = nullptr; void* lo = nullptr;
    int cin = 0, cout = 0;
};

struct TcWorkspace {
    // A-operand planes: NHWC bf16, pre-multiplied by the consuming conv's style.  Two slots (ping-pong).
    void* a_hi[2] = {nullptr, nullptr};
    void* a_lo[2] = {nullptr, nullptr};
    size_t a_bytes = 0;
    int batch = -1;
    unsigned int* d_error = nullptr;              // device-side watchdog / error word
};

struct TcConvCall {
    int batch, cin, cout, res_in, res_out; bool up;
    const float* demod;        // [B, cout]
    const float* noise; int64_t noise_bstride; float noise_w;   // noise may be null (= no noise)
    const float* bias;         // [cout] or null
    bool act = true;           // lrelu(0.2)*sqrt2 after noise + bias (StyledConv); false = bare ModulatedConv2d
    const float* blur_k;       // [4,4] (up only)
    bool blur_separable;       // blur_k is an outer product (checked on the host at prepare time)
    float* out_f32;            // [B, cout, res_out, res_out] NCHW (the captured activation)
    const float* s_next;       // [B, cout] style of the next conv (null for the last layer)
    int in_slot, out_slot;
    float* upconv_tmp;         // [B, 2H+1, 2H+1, cout] fp32 NHWC scratch (up only)
};

int tc_pack_weights(TcConvWeights& w, const float* d_weight, int cin, int cout, bool up, float scale, cudaStream_t stream);
void tc_free_weights(TcConvWeights& w);
int tc_ensure_workspace(TcWorkspace& ws, int batch, int size, int c4, const std::map<int, int>& channels);
void tc_free_workspace(TcWorkspace& ws);
// x [B,C,H,W] fp32 NCHW, s [B,C] -> slot planes (NHWC bf16 hi/lo of s*x)
int tc_prescale_split(TcWorkspace& ws, int slot, const float* x, const float* s, int batch, int c, int h, int w, cudaStream_t stream);
int tc_modconv(TcWorkspace& ws, const TcConvWeights& w, const TcConvCall& call, cudaStream_t stream);
// 0 if no device-side watchdog fired since the last call (synchronises the stream).
int tc_check_error(TcWorkspace& ws, cudaStream_t stream);

// DatasetGAN labeller building blocks: capture -> channel slice of an NHWC bf16 hi/lo pair, weight matrix slice -> hi/lo,
// and the single-tap GEMM out[b,n,y,x] = sum_k W[n,k] A[b,y,x,k] (fp32 NCHW, or NHWC, out).
int tc_nchw_to_nhwc_split(void* hi, void* lo, const float* x, int batch, int c, int64_t hw, int c_total, int c_off, cudaStream_t stream);
int tc_pack_matrix_split(void* hi, void* lo, const float* w, int n, int k, int k_total, int k_off, int out_total, int out_off, cudaStream_t stream);
int tc_conv1x1(const void* a_hi, const void* a_lo, const void* w_hi, const void* w_lo, int batch, int res, int cin, int cout,
               const float* ones, float* out, bool out_nhwc, unsigned int* d_error, cudaStream_t stream);

}  // namespace sis
