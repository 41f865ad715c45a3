// GPU side of the steps either side of the hot path (SURVEY.md 8f3):
//   up_pack_input_u8_s2d   uint8 HWC camera / decoder images -> (x - mean) / std -> the 2x2 space-to-depth NHWC 16-bit
//                          tensor the stem convolution reads (utils/mpii_data.py:184-185 + Mytransforms.normalize :10-25
//                          + to_tensor :27-43), skipping the fp32 NCHW staging copy (4x fewer host->device bytes)
//   up_gaussian_labels     ground-truth heat-maps from key-points: K Gaussians + background channel, bit-for-bit the
//                          arithmetic of utils/mpii_data.py:62-65,165-181 (float64 exp, > 1 -> 1, < 0.0099 -> 0, fp32
//                          store, background = 1 - max)
#include "up_internal.h"

namespace up {

// one thread per space-to-depth pixel: reads two rows x 6 bytes (2 pixels x 3 channels), writes 16 channels (12 real,
// order (ph, pw, c) as up_pack_input_s2d)
template <int kMode>
__global__ void pack_input_u8_s2d_kernel(const uint8_t* __restrict__ x, uint16_t* __restrict__ y, int n, int h, int w,
                                         long long plane, int wpitch, int wpad, float mean, float inv_std) {
  const int hq = h / 2, wq = w / 2;
  const long long total = static_cast<long long>(n) * hq * wq;
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (i >= total) return;
  const int xq = static_cast<int>(i % wq);
  long long t = i / wq;
  const int yq = static_cast<int>(t % hq);
  const int b = static_cast<int>(t / hq);
  float v0[8], v1[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    v0[e] = 0.f;
    v1[e] = 0.f;
  }
#pragma unroll
  for (int ph = 0; ph < 2; ++ph) {
    const uint8_t* src = x + ((static_cast<long long>(b) * h + (2 * yq + ph)) * w + 2 * xq) * 3;   // 6 bytes, 2-aligned
    const uint16_t* s2 = reinterpret_cast<const uint16_t*>(src);
    const uint32_t a = __ldg(s2), bb = __ldg(s2 + 1), c = __ldg(s2 + 2);
    const uint8_t px[6] = {static_cast<uint8_t>(a & 0xFF), static_cast<uint8_t>(a >> 8), static_cast<uint8_t>(bb & 0xFF),
                           static_cast<uint8_t>(bb >> 8), static_cast<uint8_t>(c & 0xFF), static_cast<uint8_t>(c >> 8)};
#pragma unroll
    for (int pw = 0; pw < 2; ++pw) {
#pragma unroll
      for (int ch = 0; ch < 3; ++ch) {
        const int idx = (ph * 2 + pw) * 3 + ch;
        const float f = (static_cast<float>(px[pw * 3 + ch]) - mean) * inv_std;   // Mytransforms.normalize: sub_(m).div_(s)
        if (idx < 8) v0[idx] = f; else v1[idx - 8] = f;
      }
    }
  }
  uint16_t* o = y + ((static_cast<long long>(b) * hq + yq) * wpitch + xq + wpad) * 16;
  store8_16<kMode>(o, plane, v0);
  store8_16<kMode>(o + 8, plane, v1);
}

// one thread per (image, pixel): all K joints + the background channel
__global__ void gaussian_labels_kernel(const float* __restrict__ kpts, float* __restrict__ heat, int n, int k, int h, int w,
                                       double stride, double sigma, int background, int truncate) {
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  const long long total = static_cast<long long>(n) * h * w;
  if (i >= total) return;
  const int xx = static_cast<int>(i % w);
  const int yy = static_cast<int>((i / w) % h);
  const int b = static_cast<int>(i / (static_cast<long long>(w) * h));
  const int c0 = background ? 1 : 0;
  float* out = heat + (static_cast<long long>(b) * (k + c0)) * h * w + static_cast<long long>(yy) * w + xx;
  float mx = -INFINITY;
  for (int j = 0; j < k; ++j) {
    const float kx = kpts[(static_cast<long long>(b) * k + j) * 2 + 0];
    const float ky = kpts[(static_cast<long long>(b) * k + j) * 2 + 1];
    // x = int(kpt[i][0]) * 1.0 / stride (mpii_data.py:168-169); the centre map passes int(center / stride): truncate = 2
    double cx, cy;
    if (truncate == 2) {
      // center is a float32 torch tensor: center[0] / stride is an fp32 division, int() truncates it
      cx = static_cast<double>(static_cast<long long>(kx / static_cast<float>(stride)));
      cy = static_cast<double>(static_cast<long long>(ky / static_cast<float>(stride)));
    } else {
      cx = static_cast<double>(static_cast<long long>(kx)) * 1.0 / stride;
      cy = static_cast<double>(static_cast<long long>(ky)) * 1.0 / stride;
    }
    const double dx = static_cast<double>(xx) - cx, dy = static_cast<double>(yy) - cy;
    const double d2 = dx * dx + dy * dy;
    double g = exp(-d2 / 2.0 / sigma / sigma);     // guassian_kernel, mpii_data.py:62-65
    if (g > 1.0) g = 1.0;
    if (g < 0.0099) g = 0.0;
    const float gf = static_cast<float>(g);
    out[static_cast<long long>(j + c0) * h * w] = gf;
    mx = fmaxf(mx, gf);
  }
  if (background) out[0] = 1.0f - mx;             // heatmap[:, :, 0] = 1.0 - max over joints (fp32)
}

}  // namespace up

using namespace up;

extern "C" int up_pack_input_u8_s2d(const uint8_t* x_nhwc, void* y, int n, int h, int w, int dtype,
                                    int64_t y_plane_stride, int y_wpitch, int y_wpad_left, float mean, float std_,
                                    void* stream) {
  UP_CHECK_ARG(x_nhwc && y, "up_pack_input_u8_s2d: null argument");
  UP_CHECK_ARG(n > 0 && h > 0 && w > 0 && h % 2 == 0 && w % 2 == 0, "up_pack_input_u8_s2d: h, w must be even");
  UP_CHECK_ARG((reinterpret_cast<uintptr_t>(y) & 15) == 0 && (reinterpret_cast<uintptr_t>(x_nhwc) & 1) == 0,
               "up_pack_input_u8_s2d: alignment");
  UP_CHECK_ARG(std_ != 0.f, "up_pack_input_u8_s2d: std must be non-zero");
  if (y_wpitch <= 0) y_wpitch = w / 2;
  UP_CHECK_ARG(y_wpad_left >= 0 && y_wpad_left + w / 2 <= y_wpitch, "up_pack_input_u8_s2d: bad row pitch / padding");
  const long long total = static_cast<long long>(n) * (h / 2) * (w / 2);
  const int grid = static_cast<int>((total + 255) / 256);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const float inv = 1.0f / std_;
  // (x - m) / s with s a power of two (256: mpii_data.py:184) is exact either way; for other s this is x * (1/s)
  if (dtype == UP_FP16) pack_input_u8_s2d_kernel<0><<<grid, 256, 0, st>>>(x_nhwc, static_cast<uint16_t*>(y), n, h, w, y_plane_stride, y_wpitch, y_wpad_left, mean, inv);
  else if (dtype == UP_BF16) pack_input_u8_s2d_kernel<1><<<grid, 256, 0, st>>>(x_nhwc, static_cast<uint16_t*>(y), n, h, w, y_plane_stride, y_wpitch, y_wpad_left, mean, inv);
  else if (dtype == UP_SPLIT) pack_input_u8_s2d_kernel<2><<<grid, 256, 0, st>>>(x_nhwc, static_cast<uint16_t*>(y), n, h, w, y_plane_stride, y_wpitch, y_wpad_left, mean, inv);
  else return fail(UP_ERR_INVALID, "up_pack_input_u8_s2d: bad dtype %d", dtype);
  UP_CHECK_LAUNCH("pack_input_u8_s2d_kernel");
  return 0;
}

extern "C" int up_gaussian_labels(const float* kpts, float* heat, int n, int k, int h, int w, float stride, float sigma,
                                  int background, int truncate_mode, void* stream) {
  UP_CHECK_ARG(kpts && heat && n > 0 && k > 0 && h > 0 && w > 0, "up_gaussian_labels: bad argument");
  UP_CHECK_ARG(stride > 0.f && sigma > 0.f, "up_gaussian_labels: stride and sigma must be positive");
  UP_CHECK_ARG(truncate_mode == 1 || truncate_mode == 2, "up_gaussian_labels: truncate_mode is 1 (joints) or 2 (centre map)");
  const long long total = static_cast<long long>(n) * h * w;
  gaussian_labels_kernel<<<static_cast<int>((total + 127) / 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
      kpts, heat, n, k, h, w, static_cast<double>(stride), static_cast<double>(sigma), background ? 1 : 0, truncate_mode);
  UP_CHECK_LAUNCH("gaussian_labels_kernel");
  return 0;
}
