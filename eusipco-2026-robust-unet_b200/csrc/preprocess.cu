// Input preprocessing: uint8 RGB [B,H,W,3] -> fp32 NCHW planes, the arithmetic of preprocess_pixel (preprocess.cuh):
// Normalize in channels 0-2, the build-defined HSV planes beyond, bit-identical to the numpy oracle.
#include "preprocess.cuh"

namespace {

__global__ void __launch_bounds__(256)
preprocess_kernel(const uint8_t* __restrict__ img, long P, int HW, int nc, float* __restrict__ out) {
  for (long p = blockIdx.x * (long)blockDim.x + threadIdx.x; p < P; p += (long)gridDim.x * blockDim.x) {
    const long n = p / HW;
    const long pl = p - n * HW;
    const uint8_t rgb[3] = {img[p * 3], img[p * 3 + 1], img[p * 3 + 2]};
    preprocess_pixel(rgb, nc, out + n * (long)nc * HW + pl, HW);
  }
}

}  // namespace

extern "C" int rbu_preprocess(const uint8_t* img, int B, int H, int W, int n_channels, float* out, void* stream) {
  RBU_CHECK_ARG(img && out && B > 0 && H > 0 && W > 0, "rbu_preprocess: bad arguments");
  RBU_CHECK_ARG(n_channels == 3 || n_channels == 4 || n_channels == 6, "rbu_preprocess: n_channels must be 3, 4 or 6");
  const long P = (long)B * H * W;
  long blocks = (P + 255) / 256;
  const long cap = (long)rbu_num_sms() * 16;
  if (blocks > cap) blocks = cap;
  preprocess_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(img, P, H * W, n_channels, out);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}
