/*
 * sis_b200.h — C-ABI of the B200-native Synthesis-in-Style hot path (libsis_b200.so).
 *
 * Plain pointers and sizes only; no torch types.  Every pointer named `d_*` / documented as "device" is a
 * CUDA device pointer on the current device; `stream` is a `cudaStream_t` passed as `void*` (0 = legacy
 * default stream).  All launches are asynchronous on `stream`; nothing synchronises unless stated.
 * Every function returns 0 on success and a non-zero `sis_status` otherwise; `sis_last_error()` gives the
 * message of the last failure on the calling thread.  Paths are relative to /root/reference
 * (`scf/` = `stylegan_code_finder/`).
 *
 * The library is sm_100a only and has no CPU fallback.
 */
#ifndef SIS_B200_H
#define SIS_B200_H

#include <stdint.h>

#if defined(__GNUC__)
#define SIS_API __attribute__((visibility("default")))
#else
#define SIS_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    SIS_OK = 0,
    SIS_ERR_INVALID = 1,   /* bad argument (the reference would TORCH_CHECK / produce garbage) */
    SIS_ERR_CUDA = 2,      /* a CUDA runtime / driver call failed */
    SIS_ERR_UNSUPPORTED = 3,
    SIS_ERR_STATE = 4      /* object used before it was prepared, missing weights, ... */
} sis_status;

typedef enum { SIS_F32 = 0, SIS_F16 = 1, SIS_F64 = 2 } sis_dtype;

SIS_API const char* sis_last_error(void);
SIS_API int sis_version(void);
/* Every device-side wait of the tcgen05 kernels is bounded (~2 s); a wait that gives up writes its code (0x100.. producer,
 * 0x200.. MMA issuer, 0x300.. operand ring, 0x400.. epilogue, 0x500/0x600 halo ring) to a word of mapped host memory and
 * traps.  The trap poisons the CUDA context (every later call fails with a sticky launch error); this word is still
 * readable.  0 = no watchdog fired since load / the last clear. */
SIS_API unsigned int sis_watchdog_code(void);
SIS_API void sis_watchdog_clear(void);
/* Number of kernel launches issued by this library on the calling process since load (all threads). */
SIS_API uint64_t sis_launch_count(void);

/* Optional timing of the library's own launches with CUDA events recorded on the launching stream, by kernel
 * category (0 mapping/modulation, 1 tcgen05 conv GEMM, 2 blur+act+split, 3 ToRGB, 4 fp32 conv, 5 labelling,
 * 6 fp32 blur+act, 7 other, 8 tcgen05 conv GEMM of layers with Cout <= 64).  Used by bench.py for the roofline figures; off by default (no events recorded).
 * sis_profile_collect synchronises on the recorded events, sums per category and clears the log. */
SIS_API int sis_profile_enable(int on);
SIS_API int sis_profile_collect(double* ms_by_category, uint64_t* count_by_category, int n_categories);

/* ---------------------------------------------------------------------------------------------------------
 * Op 1 — replaces pybind `fused.fused_bias_act(input, bias, refer, act, grad, alpha, scale)`
 *   scf/networks/stylegan2/op/fused_bias_act.cpp:11-20 -> fused_bias_act_kernel.cu:18-98.
 * y[i] = act(x[i] + b[(i / step_b) % size_b]) * scale;  act*10+grad: 30 lrelu, 31 lrelu gated by ref,
 * 12/32 zero, everything else linear.  size_b == 0 => no bias; d_ref == NULL => no ref.
 * x/out/ref: `size_x` elements of `dtype`; bias: `size_b` elements of `dtype`.
 * ------------------------------------------------------------------------------------------------------- */
SIS_API int sis_fused_bias_act(void* d_out, const void* d_x, const void* d_bias, const void* d_ref, int dtype,
                       int64_t size_x, int64_t step_b, int64_t size_b, int act, int grad, float alpha,
                       float scale, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Op 2 — replaces pybind `upfirdn2d.upfirdn2d(input[major,H,W,minor], kernel[kh,kw], up_x, up_y, down_x,
 * down_y, pad_x0, pad_x1, pad_y0, pad_y1)`  scf/networks/stylegan2/op/upfirdn2d.cpp:12-23 ->
 * upfirdn2d_kernel.cu:52-272.  Output is [major, out_h, out_w, minor] with
 * out = (in*up + pad0 + pad1 - k + down) / down  (upfirdn2d_kernel.cu:168-169); compute it with
 * sis_upfirdn2d_out_size.  Unlike the reference (which silently returns uninitialised memory when no
 * mode matches, upfirdn2d_kernel.cu:172-226) every (up, down, kernel<=32x32) combination is computed.
 * The reference dispatches on the input dtype and reads the taps as that dtype; `d_kernel` is `dtype` too.
 * ------------------------------------------------------------------------------------------------------- */
SIS_API int sis_upfirdn2d_out_size(int in_size, int up, int down, int pad0, int pad1, int ksize);
SIS_API int sis_upfirdn2d(void* d_out, const void* d_x, const void* d_kernel, int dtype, int64_t major, int in_h,
                  int in_w, int minor, int kernel_h, int kernel_w, int up_x, int up_y, int down_x, int down_y,
                  int pad_x0, int pad_x1, int pad_y0, int pad_y1, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Generator — replaces `Generator.forward` scf/networks/stylegan2/model.py:479-561 and everything it calls
 * (PixelNorm :15-20, EqualLinear :133-162, ModulatedConv2d :237-278, Blur :76-92, NoiseInjection :287-292,
 * StyledConv :336-342, ToRGB :355-364, ConstantInput :295-305), `mean_latent` :468-474.
 *
 * Lifecycle: create -> set_param for every state-dict tensor (keys of SURVEY.md §8b, fp32 device
 * pointers; the library COPIES / repacks them at prepare time, so the caller's tensors may change
 * afterwards — call prepare again to pick the changes up) -> prepare -> forward*.
 * ------------------------------------------------------------------------------------------------------- */
typedef struct sis_generator sis_generator;

typedef enum {
    SIS_PRECISION_FP32 = 0,    /* fp32 FMA implicit GEMM on CUDA cores (bit-closest to the reference) */
    SIS_PRECISION_BF16X3 = 1   /* tcgen05 bf16 split precision: hi*hi + hi*lo + lo*hi, fp32 TMEM accumulate */
} sis_precision;

SIS_API int sis_generator_create(int size, int style_dim, int n_mlp, int channel_multiplier, sis_generator** out);
/* SWAGAN generator (scf/networks/swagan/model.py:101-286), size a power of two in [16, 1024]: the StyleGAN2 conv trunk of
 * size / 2 (log_size = log2(size) - 1, num_layers = 2*log_size - 3, n_latent = 2*log_size - 2, same channel table, noise maps
 * and activation indices), 12-channel wavelet ToRGBs (keys to_rgb*.conv.weight [1,12,Cin,1,1], to_rgb*.bias [1,12,1,1],
 * and on the up-sampling ones upsample.kernel, iwt.{ll,lh,hl,hh}, dwt.{ll,lh,hl,hh}) and the generator's own iwt.* for the
 * final inverse Haar transform.  Every other sis_generator_* function works on the handle unchanged; d_image is
 * [batch,3,size,size].  Label jobs on an activation that also feeds a ToRGB run as a separate pass. */
SIS_API int sis_generator_create_swagan(int size, int style_dim, int n_mlp, int channel_multiplier, sis_generator** out);
SIS_API int sis_generator_destroy(sis_generator* g);
/* `key` is the reference state-dict key, e.g. "convs.3.conv.modulation.weight". */
SIS_API int sis_generator_set_param(sis_generator* g, const char* key, const float* d_ptr, int64_t numel);
SIS_API int sis_generator_prepare(sis_generator* g, void* stream);
SIS_API int sis_generator_n_latent(const sis_generator* g);
SIS_API int sis_generator_num_layers(const sis_generator* g);
/* channels of captured activation `idx` (0..n_latent-1) and its resolution */
SIS_API int sis_generator_activation_shape(const sis_generator* g, int idx, int* channels, int* res);

/* style MLP: `Generator.style` / `get_latent`, model.py:383-392,476-477.  z,w: [n, style_dim] fp32 device. */
SIS_API int sis_generator_style(sis_generator* g, const float* d_z, float* d_w, int64_t n, void* stream);

/* A labelling job executed inside the forward, right after activation `activation_idx` has been produced (same
 * semantics and outputs as sis_label_assign, mode 0).  When the activation also feeds a ToRGB and the map is large,
 * labelling and ToRGB run as ONE pass over the activation tensor. */
typedef struct {
    int activation_idx;
    const float* d_centroids; int k;
    const uint32_t* d_cluster_class_bits; int n_class; int image_size;
    uint8_t* d_ids_u8; int64_t* d_ids_i64; uint8_t* d_masks; float* d_margin; unsigned long long* d_hist;
} sis_label_job;

typedef struct {
    int batch;
    /* --- styles (model.py:491-528) ---
     * d_styles[j]: [batch, style_dim] (z if !input_is_latent, else w), or [batch, n_latent, style_dim]
     * when styles_are_wplus (single style only, model.py:515-519). n_styles is 1 or 2. */
    int n_styles;
    const float* d_styles[2];
    int input_is_latent;
    int styles_are_wplus;
    int inject_index;            /* used when n_styles == 2; the caller resolves the random default */
    float truncation;            /* < 1 => w = t_latent + truncation*(w - t_latent), model.py:502-510 */
    const float* d_truncation_latent; /* [1 or batch, style_dim] */
    int truncation_latent_rows;  /* 1 or batch */
    /* --- noise (model.py:494-500, 287-292) ---
     * d_noise[l]: noise map of layer l (num_layers entries), [1,1,H,W] (noise_batch_stride[l] = 0) or
     * [batch,1,H,W] (stride = H*W).  All must be non-NULL: the caller draws `randomize_noise` maps. */
    const float* const* d_noise;
    const int64_t* noise_batch_stride;
    /* --- outputs --- */
    float* d_image;              /* [batch, 3, size, size] fp32 */
    float* d_latent_out;         /* optional [batch, n_latent, style_dim] (return_latents) or NULL */
    float* const* d_activations; /* optional: n_latent pointers, entry idx = [batch, C_idx, H_idx, H_idx] fp32
                                    NCHW or NULL to skip that capture (model.py:530-549) */
    int precision;               /* sis_precision */
    /* --- optional fused labelling (NULL / 0 = none) --- */
    int n_label_jobs;
    const sis_label_job* label_jobs;
} sis_forward_args;

SIS_API int sis_generator_forward(sis_generator* g, const sis_forward_args* args, void* stream);
/* Synchronises `stream` and reports a fired tcgen05 watchdog ("... watchdog fired: code 0x...") or the stream's error. */
SIS_API int sis_generator_check(sis_generator* g, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Stand-alone layers — the reference's module-level forwards outside the fused plan (same kernels, one layer per call,
 * weights repacked per call; NOT re-entrant, like the reference's single-threaded use).  All tensors fp32 on device.
 *   sis_modulated_conv2d   ModulatedConv2d.forward (model.py:237-278, 3x3 only) and, with noise / act_bias /
 *                          activate, StyledConv.forward (model.py:336-342).  x [B,Cin,res,res]; weight [1,Cout,Cin,3,3];
 *                          mod_weight [Cin,style_dim]; style [B,style_dim]; upsample needs blur_kernel [4,4] and
 *                          writes [B,Cout,2res,2res]; noise [1 or B,1,R,R] (stride 0 or R*R) with its scalar weight.
 *   sis_to_rgb             ToRGB.forward (model.py:355-364): 1x1 modulated conv (no demod) + bias [3] + upsampled skip
 *                          [B,3,res/2,res/2] (up_kernel [4,4]) -> [B,3,res,res].
 *   sis_wavelet_to_rgb     SWAGAN ToRGB.forward (swagan/model.py:84-98), one pass: 1x1 modulated conv (no demod) to 12
 *                          channels (weight [12,Cin]) + bias [12] + dwt(upsample(iwt(skip))) of the skip [B,12,res/2,res/2]
 *                          (iwt / dwt taps [4,2,2] in ll, lh, hl, hh order, up_kernel [4,4]) -> [B,12,res,res];
 *                          res a multiple of 4.
 *   sis_equal_linear       EqualLinear.forward (model.py:152-162), optional fused leaky ReLU.
 *   sis_pixel_norm         PixelNorm.forward (model.py:19-20) over rows of `dim`.
 *   sis_noise_injection    NoiseInjection.forward (model.py:287-292): x + weight * noise.
 * ------------------------------------------------------------------------------------------------------- */
SIS_API int sis_modulated_conv2d(const float* d_x, int batch, int cin, int res, const float* d_weight, int cout,
                                 const float* d_mod_weight, const float* d_mod_bias, int style_dim, const float* d_style,
                                 int demodulate, int upsample, const float* d_blur_kernel, const float* d_noise,
                                 int64_t noise_batch_stride, const float* d_noise_weight, const float* d_act_bias, int activate,
                                 float* d_out, int precision, void* stream);
SIS_API int sis_to_rgb(const float* d_x, int batch, int cin, int res, const float* d_weight, const float* d_mod_weight,
                       const float* d_mod_bias, int style_dim, const float* d_style, const float* d_bias, const float* d_skip,
                       const float* d_up_kernel, float* d_out, void* stream);
SIS_API int sis_wavelet_to_rgb(const float* d_x, int batch, int cin, int res, const float* d_weight, const float* d_mod_weight,
                               const float* d_mod_bias, int style_dim, const float* d_style, const float* d_bias, const float* d_skip,
                               const float* d_iwt, const float* d_up_kernel, const float* d_dwt, float* d_out, void* stream);
SIS_API int sis_equal_linear(const float* d_x, int64_t rows, int in_dim, const float* d_weight, const float* d_bias, int out_dim,
                             float lr_mul, int fused_lrelu, float* d_out, void* stream);
SIS_API int sis_pixel_norm(const float* d_x, float* d_out, int64_t rows, int dim, void* stream);
SIS_API int sis_noise_injection(const float* d_x, const float* d_noise, int64_t noise_batch_stride, const float* d_weight, int batch,
                                int channels, int h, int w, float* d_out, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Labelling — replaces, on the device and in one pass per layer,
 *   FactorCatalog.predict / pairwise_distance  scf/segmentation/gan_local_edit/factor_catalog.py:47-75
 *   predict_clusters                           scf/segmentation/base_cluster_based_dataset_segmenter.py:119-138
 *   resize_to_image_size                       scf/segmentation/base_dataset_segmenter.py:32-42
 * d_act: [batch, C, H, W] fp32 NCHW.  d_centroids: [k, C] fp32.  ids = argmin_k sum_c (x_c - m_kc)^2, ties ->
 * lowest k.  d_cluster_class_bits[k]: bit j set <=> cluster belongs to class j (n_class <= 32).
 * Outputs (each optional / NULL):
 *   d_ids_u8  [batch,H,W] uint8, d_ids_i64 [batch,H,W] int64 (the reference's dtype),
 *   d_masks   [n_class, batch, S, S] uint8 0/1, nearest-resized to S (src = floor(dst*H/S)); S >= H,
 *   d_margin  [batch,H,W] fp32 second-best minus best distance,
 *   d_hist    [k] uint64, cluster pixel counts ACCUMULATED (atomicAdd) at native resolution.
 * mode 0: assign at native resolution then nearest-resize (reference cluster path).
 * mode 1: bilinear-upsample features to SxS (align_corners=False) then assign; ids/margin are [batch,S,S].
 * ------------------------------------------------------------------------------------------------------- */
SIS_API int sis_label_assign(const float* d_act, int batch, int channels, int h, int w, const float* d_centroids, int k,
                     const uint32_t* d_cluster_class_bits, int n_class, int image_size, int mode,
                     uint8_t* d_ids_u8, int64_t* d_ids_i64, uint8_t* d_masks, float* d_margin,
                     unsigned long long* d_hist, void* stream);

/* predict_clusters' mask step alone: ids(int64)[n] -> masks [n_class, n] uint8
 * (base_cluster_based_dataset_segmenter.py:131-135). */
SIS_API int sis_class_masks_from_ids(const int64_t* d_ids, int64_t n, const uint32_t* d_cluster_class_bits, int k,
                             int n_class, uint8_t* d_masks, void* stream);

/* resize_to_image_size alone: nearest resize of uint8/bool planes [planes, h, w] -> [planes, S, S]
 * (base_dataset_segmenter.py:38, F.interpolate default mode). */
SIS_API int sis_nearest_resize_u8(const uint8_t* d_in, int64_t planes, int h, int w, int out_h, int out_w, uint8_t* d_out,
                          void* stream);

/* merge_sub_images: dst |= src over n bytes (black_white_handwritten_printed_text_segmenter.py:31-40). */
SIS_API int sis_or_u8(uint8_t* d_dst, const uint8_t* d_src, int64_t n, void* stream);

/* make_image (pytorch_training.images.make_image, call site scf/create_dataset_for_segmentation.py:135):
 * [batch,3,S,S] fp32 -> [batch,S,S,3] uint8, clamp(-1,1), (x+1)/2*255 truncated. */
SIS_API int sis_make_image_u8(const float* d_image, int batch, int size, uint8_t* d_out, void* stream);

/* -----------------------------------------------------------------------------------------------------------
 * Contour stage on the device: class masks -> colour label images + drop decision (SURVEY.md 8(f) row 1).
 * Replaces the host loop of BlackWhiteHandwrittenPrintedTextDatasetSegmenter.create_segmentation_image
 *   scf/segmentation/black_white_handwritten_printed_text_segmenter.py:42-99   (extract_text_regions, drop rule, driver)
 *   scf/segmentation/base_cluster_based_dataset_segmenter.py:148-450           (cluster_image_to_contours, contour_overlap,
 *       merge_contours*, merge_finegrained_segmentation, classify_fine_grained_contours, drop_too_small_contours,
 *       render_segmentation_image)
 *   scf/segmentation/base_dataset_segmenter.py:52-57                           (dilate_image)
 * from the merged, image-size uint8 masks on (what prepare_image_segmentation + merge_sub_images produce).
 *
 * d_det_masks  : HOST array of n_det_keys*n_classes device pointers, entry [k*n_classes + c] = mask [batch,S,S] of class c
 *                (classes = class_to_color_map without 'background', in its order) under keys_for_class_determination[k]
 * d_fine_masks : HOST array of n_fine_keys device pointers: mask [batch,S,S] of the fine-grained class
 *                ('printed_text') under keys_for_finegrained_segmentation[k]; the last one is also the ink mask of the
 *                rendering step
 * colors_rgb   : HOST, (1 + n_classes) * 3 bytes: background colour, then the classes
 * render_rank  : HOST, n_classes ints: position of each class in the mask dict the reference's renderer iterates
 *                (a later class overwrites an earlier one)
 * S <= 1024.
 * d_label_rgb  : uint8 [batch,S,S,3];  d_flags: int32 [batch]: 0 keep, 1 drop, 2 = take this image through the host path
 *                (the reference's drop rule reads the FIRST contour of a class; the device does not order contours and
 *                only decides when the order cannot matter; also set for the whole batch when a capacity is exceeded)
 * d_info       : DEVICE, 3 ints or NULL: shapes found, fixpoint rounds that did work, reason the batch was handed to the
 *                host (0 none, 1 capacity, 3 fixpoint still moving after the enqueued rounds)
 * Fully asynchronous: the merge fixpoint is controlled on the device (a fixed number of rounds is enqueued, kernels with
 * nothing left to do return at once); the call never synchronises the stream. */
SIS_API int sis_contour_stage_workspace_bytes(int batch, int size, int n_classes, int n_det_keys, int n_fine_keys, int64_t* bytes);
SIS_API int sis_contour_stage(const uint8_t* const* d_det_masks, const uint8_t* const* d_fine_masks, int batch, int size,
                      int n_classes, int n_det_keys, int n_fine_keys, int fine_class, int only_keep_overlapping,
                      double min_class_contour_area, const uint8_t* colors_rgb, const int* render_rank,
                      void* d_workspace, int64_t workspace_bytes, uint8_t* d_label_rgb, int32_t* d_flags, int32_t* d_info,
                      void* stream);

/* -----------------------------------------------------------------------------------------------------------
 * Host-side writer of the dataset's PNG files (no device work; HOST pointers): file i holds, side by side, row rows[i]
 * of `h_left` [n, height, width_left, channels] and of `h_right` [n, height, width_right, channels] (either side may be
 * absent: width 0).  Replaces scf/create_dataset_for_segmentation.py:84-99 (save_image / save_generated_images:
 * numpy.concatenate + PIL.Image.save per file) with native threads: filter 'Up', zlib `level` (0 = stored), one IDAT.
 * The parent directories must exist.  Blocks until every file is written; call it off the thread that drives the GPU. */
SIS_API int sis_png_write_pairs(const uint8_t* h_left, const uint8_t* h_right, int height, int width_left, int width_right,
                        int channels, const int32_t* rows, const char* const* paths, int n_files, int level, int n_threads);

/* -----------------------------------------------------------------------------------------------------------
 * DatasetGAN labeller (the other `segmenter_type`): every capture -> ensemble of per-pixel MLP classifiers -> labels.
 * Replaces DatasetGANSegmenter.create_segmentation_image's device work
 *   scf/segmentation/dataset_gan_segmenter.py:34-60  (predict_labels, label_images_to_color_images)
 *   scf/data/dataset_gan_dataset.py:12-34            (scale_activations: bilinear upsample to S x S + concat)
 *   scf/networks/pixel_classifier/model.py:40-121    (PixelClassifier n_class < 32: Linear F->128, ReLU, BatchNorm1d,
 *                                                     Linear 128->32, ReLU, BatchNorm1d, Linear 32->n; ensemble mode vote)
 * Networks are in eval mode.  Parameters are set per network under the reference's state-dict keys
 * ("layers.0.weight" [128,F], "layers.0.bias", "layers.2.{weight,bias,running_mean,running_var}", "layers.3.*",
 * "layers.5.*", "layers.6.weight" [n,32], "layers.6.bias") from HOST memory, then `prepare` uploads them.
 * `label`: captures in the generator's dict order (their channels must sum to feature_size), fp32 NCHW on the device;
 *   d_labels [batch,S,S] uint8 (required), d_votes [batch,S,S,n_models] uint8 (optional),
 *   host_colors [n_class*3] uint8 in HOST memory + d_color_image [batch,S,S,3] uint8 (optional, both or neither).
 * Asynchronous on `stream`; `check` synchronises it and reports a fired GEMM watchdog.
 * ----------------------------------------------------------------------------------------------------------- */
typedef struct sis_pixel_ensemble sis_pixel_ensemble;
SIS_API int sis_pixel_ensemble_create(sis_pixel_ensemble** out, int n_models, int feature_size, int n_class);
SIS_API void sis_pixel_ensemble_destroy(sis_pixel_ensemble* e);
SIS_API int sis_pixel_ensemble_set_param(sis_pixel_ensemble* e, int model, const char* name, const float* host_data, int64_t numel);
SIS_API int sis_pixel_ensemble_prepare(sis_pixel_ensemble* e, void* stream);
SIS_API int sis_pixel_ensemble_label(sis_pixel_ensemble* e, int n_layers, const float* const* d_activations, const int* channels,
                             const int* resolutions, int batch, int image_size, uint8_t* d_labels, uint8_t* d_votes,
                             const uint8_t* host_colors, uint8_t* d_color_image, void* stream);
SIS_API int sis_pixel_ensemble_check(sis_pixel_ensemble* e, void* stream);

/* -----------------------------------------------------------------------------------------------------------
 * Catalog creation: steps of spherical mini-batch k-means, many independent fits per launch (one CTA per fit).
 * Replaces the loop of MiniBatchSphericalKMeans.fit, scf/segmentation/gan_local_edit/spherical_kmeans.py:159-312
 * (sklearn 0.24's MiniBatchKMeans on unit rows, centres renormalised after every step).  One step: renormalise the
 * centres; reassign iff (t+1) % (10 + int(min counts)) == 0; nearest centre of each batch row; starved centres (count <
 * ratio * max count, at most half the batch, lowest counts first) take batch rows and the smallest other count;
 * count-weighted update; renormalise; batch inertia (mean squared distance), its EWA with alpha = min(1, 2 bs / (n+1)) in
 * fp64, the no-improvement counter and the stop test (steps_done == max_steps, or no_improvement >= max_no_improvement
 * when that is >= 0).
 *
 * Draws are counter based: h(t, j, s) = splitmix64(splitmix64(splitmix64(seed) ^ t) ^ (j << 1 | s)).  Batch row j of
 * step t is h(t, j, 0) mod n; when centres are reassigned, the rows of the n_re smallest h(t, j, 1) (ties to the lower
 * j) replace the starved centres in index order.  A fit's result does not depend on the other fits of a launch, nor on
 * how its steps are split across calls.
 *
 * fits          : HOST array of n_fits descriptors (device pointers inside).  k in [2, 32], channels <= 512, n >= k.
 *                 Fits may differ in n, channels and k.  Points are unit rows; centres are updated in place.
 * d_indices     : NULL: each fit runs up to `steps` drawn steps and a fit that is done returns at once.  Otherwise
 *                 steps must be 1 and every fit runs one step on these n_indices (<= 1024) rows: no draw, no
 *                 reassignment, no EWA, the state is neither read nor written (d_state may be NULL).
 * d_batch_inertia: optional [n_fits, steps] fp32, the batch inertia of each step run (entries of steps not run are
 *                 left as they are).
 * Asynchronous on `stream`; never synchronises.  sis_kmeans_init_state fills one fit's state (batch_size in
 * [1, 1024], max_steps >= 1, max_no_improvement < 0 = never stop early).
 * ----------------------------------------------------------------------------------------------------------- */
typedef struct {
    uint64_t seed;
    int64_t steps_done;          /* the fit's n_iter_ */
    int64_t max_steps;
    int64_t done;                /* 0 running, 1 finished: the word the host polls */
    double ewa, ewa_min;
    int32_t batch_size, max_no_improvement, no_improvement;
    float reassignment_ratio;
} sis_kmeans_state;

typedef struct {
    const float* d_points; int64_t n; int channels;   /* unit rows, [n, channels] row-major */
    int k; float* d_centers; float* d_counts;          /* [k, channels] unit rows, [k] */
    sis_kmeans_state* d_state;                         /* per-fit state, sis_kmeans_state_bytes() */
} sis_kmeans_fit;

SIS_API int sis_kmeans_state_bytes(void);
SIS_API int sis_kmeans_init_state(void* d_state, uint64_t seed, int batch_size, int64_t max_steps, int max_no_improvement,
                                  float reassignment_ratio, void* stream);
SIS_API int sis_kmeans_steps(const sis_kmeans_fit* fits, int n_fits, int steps, const int32_t* d_indices, int n_indices,
                             float* d_batch_inertia, void* stream);

/* -----------------------------------------------------------------------------------------------------------
 * Training of a DatasetGAN pixel-classifier ensemble (the networks sis_pixel_ensemble_* evaluates), on the annotated
 * pixels of generated images.  The recipe is this project's own, after DatasetGAN's train_interpreter.py:
 *   - batches of `batch_pixels` (2..64) annotated pixels; each network draws its own order per epoch, a bijective
 *     counter permutation of the A*S*S pixels (4-round Feistel network with cycle walking, keyed by the network's key
 *     and the epoch: oracle/dataset_gan_train_oracle.py restates it); the trailing partial batch is dropped;
 *   - features: every capture bilinearly upsampled to S x S at the pixel (align_corners = False), concatenated in
 *     capture order, as the labeller; the networks run Linear, ReLU, BatchNorm1d in training mode (batch mean, biased
 *     variance; running statistics with momentum 0.1 and the unbiased variance), ..., mean softmax cross-entropy;
 *   - torch.optim.Adam on the 10 trainable tensors: lr 1e-3, betas (0.9, 0.999), eps 1e-8, bias correction;
 *   - stopping: after `epochs` epochs, or, from epoch 4 on, after 51 consecutive steps whose loss is not below the
 *     network's best.  fp32 arithmetic with fixed summation orders: a network's result depends neither on the other
 *     networks of the trainer nor on how its steps are split into calls.
 * create       : 1..8 networks, 2 <= n_class < 32, feature_size a positive multiple of 32.
 * set_param    : initial values per network under the state-dict keys of sis_pixel_ensemble_set_param (HOST memory).
 * set_data     : captures fp32 NCHW [n_images, C_l, r_l, r_l] and labels uint8 [n_images, S, S] (ids < n_class) on
 *                the device; they must stay alive and unchanged while the trainer runs.  n_images * S * S <= 2^31 - 1.
 * prepare      : uploads the parameters, zeroes the optimiser state; keys[m] is network m's draw key.
 * steps        : enqueues `steps` steps for every network that has not stopped; never synchronises.
 * status       : synchronises `stream`; done[m] (0/1) and steps_done[m] (= num_batches_tracked) per network.
 * read_param   : the current value of a state-dict key (running statistics included) into HOST memory.
 * read_losses  : the first `count` (<= steps_done) per-step losses of a network into HOST memory.
 * ----------------------------------------------------------------------------------------------------------- */
typedef struct sis_pixel_train sis_pixel_train;
SIS_API int sis_pixel_train_create(sis_pixel_train** out, int n_models, int feature_size, int n_class, int batch_pixels);
SIS_API void sis_pixel_train_destroy(sis_pixel_train* t);
SIS_API int sis_pixel_train_set_param(sis_pixel_train* t, int model, const char* name, const float* host_data, int64_t numel);
SIS_API int sis_pixel_train_set_data(sis_pixel_train* t, int n_layers, const float* const* d_activations, const int* channels,
                                     const int* resolutions, int n_images, int image_size, const uint8_t* d_labels);
SIS_API int sis_pixel_train_prepare(sis_pixel_train* t, const uint64_t* keys, int epochs, void* stream);
SIS_API int sis_pixel_train_steps(sis_pixel_train* t, int steps, void* stream);
SIS_API int sis_pixel_train_status(sis_pixel_train* t, int32_t* done, int64_t* steps_done, void* stream);
SIS_API int sis_pixel_train_read_param(sis_pixel_train* t, int model, const char* name, float* host_out, int64_t numel, void* stream);
SIS_API int sis_pixel_train_read_losses(sis_pixel_train* t, int model, float* host_out, int64_t count, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SIS_B200_H */
