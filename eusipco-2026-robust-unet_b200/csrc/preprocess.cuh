// The per-pixel arithmetic of rbu_preprocess, shared by every kernel that writes normalised network input
// (preprocess.cu, patches.cu), so the bit-exact contract with the numpy oracle is stated once.
#pragma once
#include "rbu_common.cuh"

// One uint8 RGB pixel -> o[k * plane] for k < nc.  Channels 0-2 are torchvision's ToTensor + Normalize with the
// ImageNet constants (Main_Final.py:697-701): (x/255 - mean)/std.  The reference has no HSV code (SURVEY.md §8c): the
// optional extra planes are build-defined and pinned to OpenCV float semantics -- nc == 4 appends S; nc == 6 appends
// H/360, S, V.  Every operation is an explicitly rounded IEEE fp32 op (no FMA contraction).
__device__ __forceinline__ void preprocess_pixel(const uint8_t (&rgb)[3], int nc, float* o, long long plane) {
  const float mean[3] = {0.485f, 0.456f, 0.406f};
  const float stdv[3] = {0.229f, 0.224f, 0.225f};
  float c[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) c[k] = __fdiv_rn((float)rgb[k], 255.0f);
#pragma unroll
  for (int k = 0; k < 3; ++k) o[k * plane] = __fdiv_rn(__fsub_rn(c[k], mean[k]), stdv[k]);
  if (nc > 3) {
    const float r = c[0], g = c[1], b = c[2];
    const float v = fmaxf(fmaxf(r, g), b);
    const float mn = fminf(fminf(r, g), b);
    const float diff = __fsub_rn(v, mn);
    const float s = v > 0.f ? __fdiv_rn(diff, v) : 0.f;
    if (nc == 4) {
      o[3 * plane] = s;
    } else {
      float h = 0.f;
      if (diff > 0.f) {
        if (v == r) h = __fdiv_rn(__fsub_rn(g, b), diff);
        else if (v == g) h = __fadd_rn(2.0f, __fdiv_rn(__fsub_rn(b, r), diff));
        else h = __fadd_rn(4.0f, __fdiv_rn(__fsub_rn(r, g), diff));
        h = __fmul_rn(h, 60.0f);
        if (h < 0.f) h = __fadd_rn(h, 360.0f);
      }
      o[3 * plane] = __fdiv_rn(h, 360.0f);
      o[4 * plane] = s;
      o[5 * plane] = v;
    }
  }
}
