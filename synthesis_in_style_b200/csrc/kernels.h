// Internal launch interfaces between the translation units of libsis_b200 (not part of the C-ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace sis {

enum { LINEAR_EPI_BIAS = 0, LINEAR_EPI_BIAS_LRELU = 1, LINEAR_EPI_RSQRT_EPS = 2 };

struct LinearJob {
    const float* A; int lda;      // [M, K] (row stride lda)
    const float* W;               // [N, K]
    const float* bias;            // [N] or null
    float* C; int ldc;            // [M, N]
    int M, N, K;
    int square_a;                 // use A*A
    int epilogue;
};

struct ModConvSimtArgs {
    const float* x;   // [B, Cin, H, W]
    const float* w;   // [Cout, Cin, 3, 3] pre-scaled (pre-flipped for the transposed conv)
    const float* s;   // [B, Cin]
    const float* d;   // [B, Cout] or null
    float* out;       // [B, Cout, OH, OW]
    int Cin, Cout, H, W, OH, OW, pad, zero_insert;
    const float* noise; int64_t noise_bstride; float noise_w; const float* bias; int fuse_act;
};

struct BlurActArgs {
    const float* in; float* out; int64_t planes; int C, IH, IW, OH, OW;
    const float* blur_k; const float* noise; int64_t noise_bstride; float noise_w; const float* bias;
    int act;   // 1: + noise + bias, lrelu*sqrt2 (StyledConv); 0: blur only
};

struct ToRgbArgs {
    const float* x;     // [B, C, H, W]
    const float* s;     // [B, C]
    const float* w;     // [3, C] pre-scaled
    const float* bias;  // [3]
    const float* skip;  // [B, 3, H/2, W/2] or null
    const float* up_k;  // [4,4]
    float* out;         // [B, 3, H, W]
    int batch, C, H, W;
};

// SWAGAN ToRGB (wavelet_torgb.cu): 12 output channels = 4 Haar bands x RGB
struct WaveletToRgbArgs {
    const float* x;            // [B, C, H, W]
    const float* s;            // [B, C]
    const float* w;            // [12, C] pre-scaled
    const float* bias;         // [12]
    const float* skip;         // [B, 12, H/2, W/2] or null
    const float* iwt_k;        // [4 bands][2][2] inverse Haar taps applied to the skip
    const float* up_k;         // [4][4]
    const float* dwt_k;        // [4 bands][2][2]
    const float* final_iwt_k;  // [4 bands][2][2] or null: write the image [B, 3, 2H, 2W] instead of [B, 12, H, W]
    float* out;
    int batch, C, H, W;
};

struct LabelArgs {
    const float* act; int batch, C, H, W;
    const float* centroids; int k;
    const uint32_t* class_bits; int n_class; int S;
    uint8_t* ids_u8; int64_t* ids_i64; uint8_t* masks; float* margin; unsigned long long* hist;
};

// Labelling of one activation map (mode 0 native + nearest resize, mode 1 bilinear-then-assign).  When `fuse_rgb` is
// given (a ToRGB over the SAME tensor) and the shapes allow the wide kernel, both are done in one pass over the
// activations and *fused is set; otherwise only the labelling runs and the caller launches ToRGB itself.
int launch_label(const LabelArgs& a, int mode, const ToRgbArgs* fuse_rgb, bool* fused, cudaStream_t stream);

int launch_pixel_norm(float* out, const float* z, int64_t rows, int dim, cudaStream_t stream);
// small_m_ok: every job has K % 4 == 0, 16-byte aligned A rows / W rows (then the weight-streaming kernel is used)
int launch_linear_jobs(const LinearJob* d_jobs, int n_jobs, int max_m, int max_n, int max_k, bool small_m_ok, cudaStream_t stream);
int launch_assemble_latent(float* latent, const float* w0, const float* w1, int wplus, int inject_index,
                           float truncation, const float* tlat, int tlat_rows, int batch, int n_latent, int dim,
                           cudaStream_t stream);
int launch_scale_copy(float* out, const float* in, float scale, int64_t n, cudaStream_t stream);
int launch_weight_sq(float* wsq, const float* w, float scale, int64_t n_oi, int taps, cudaStream_t stream);
int launch_scale_flip3x3(float* out, const float* in, float scale, int64_t n_oi, cudaStream_t stream);
int launch_modconv3x3_simt(const ModConvSimtArgs& a, int batch, cudaStream_t stream);
int launch_const_input(float* out, const float* inp, int64_t per_sample, int batch, cudaStream_t stream);
int launch_blur_noise_act(const BlurActArgs& a, cudaStream_t stream);
int launch_torgb(const ToRgbArgs& a, cudaStream_t stream);
int launch_wavelet_torgb(const WaveletToRgbArgs& a, cudaStream_t stream);

}  // namespace sis
