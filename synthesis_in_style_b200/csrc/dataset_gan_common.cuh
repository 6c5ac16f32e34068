// Shared by the DatasetGAN labeller (dataset_gan.cu) and its trainer (dataset_gan_train.cu): the classifier's sizes and
// the source taps of one output pixel of a capture's bilinear upsample.
#pragma once
#include <cuda_runtime.h>

namespace sis {

constexpr int GAN_H1 = 128, GAN_H2 = 32, GAN_MAX_GROUPS = 8, GAN_MAX_MODELS = 8;

struct GanBilinearTap {
    int y0, y1, x0, x1;
    float w00, w01, w10, w11;
};

// nn.Upsample(scale_factor = S / r, mode='bilinear'), align_corners = False (ATen's area_pixel_compute_source_index):
// src = max((dst + 0.5) * r / S - 0.5, 0), i0 = floor(src), i1 = min(i0 + 1, r - 1).  A value is
// w00 q[y0][x0] + w01 q[y0][x1] + w10 q[y1][x0] + w11 q[y1][x1], accumulated in that order.
__device__ __forceinline__ GanBilinearTap gan_bilinear_tap(int oy, int ox, int r, int S) {
    const float sc = (float)r / (float)S;
    const float fy = fmaxf(((float)oy + 0.5f) * sc - 0.5f, 0.0f), fx = fmaxf(((float)ox + 0.5f) * sc - 0.5f, 0.0f);
    GanBilinearTap t;
    t.y0 = (int)fy; t.x0 = (int)fx;
    t.y1 = min(t.y0 + 1, r - 1); t.x1 = min(t.x0 + 1, r - 1);
    const float ly = fy - (float)t.y0, lx = fx - (float)t.x0;
    t.w00 = (1.0f - ly) * (1.0f - lx); t.w01 = (1.0f - ly) * lx; t.w10 = ly * (1.0f - lx); t.w11 = ly * lx;
    return t;
}

}  // namespace sis
