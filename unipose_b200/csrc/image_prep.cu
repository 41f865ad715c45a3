// up_resize_pack_u8: a ragged batch of decoded uint8 HWC images -> the network input, in one launch.
//
// Per image: cv2.resize(img, (out_w, out_h)) (utils/mpii_data.py:159-162, utils/lsp_lspet_data.py:211), bit for bit
// OpenCV's 8-bit INTER_LINEAR path, then the optional mirror of Mytransforms.hflip (utils/Mytransforms.py:501-505),
// then one of three stores: the stem's normalised space-to-depth tensor (same layout and bits as
// up_pack_input_u8_s2d, so the resized image never exists in memory), uint8 HWC, or normalised fp32 NCHW.
//
// OpenCV's arithmetic (oracle/image_prep_oracle.py restates it in numpy and checks it against cv2):
//   f = float((d + 0.5) * (1 / (dst / src)) - 0.5) in double then float32, s = floor(f), f -= s
//   weights c0 = round((1 - f) * 2048), c1 = round(f * 2048)
//   columns: s < 0 -> (0, 0); s >= w - 1 -> (w - 1, 0).  Rows keep their fraction, only the row indices are clamped.
//   horizontal: r = S[s] * a0 + S[s + 1] * a1 (int32); vertical (SIMD rounding): ((r0 >> 4) * b0 >> 16) +
//   ((r1 >> 4) * b1 >> 16), then (v + 2) >> 2 saturated to uint8.  A source exactly twice the target in both
//   dimensions takes cv2's INTER_AREA fast path instead: (2x2 sum + 2) >> 2.
// The double / float steps use explicit _rn intrinsics so that nvcc cannot contract them into FMAs: the bits of f
// decide the weights.
//
// Work split: one thread block per (image, output row pair), i.e. one row of space-to-depth pixels.  The block
// computes the column coefficients of its image into shared memory (the flip is folded in there: output column x
// reads the coefficients of resized column out_w - 1 - x), stages the (at most four) source rows it needs into shared
// memory with 16-byte loads when the row start is 16-byte aligned and byte loads otherwise, then each thread makes one
// 2x2 output block (one space-to-depth pixel: 12 values) from shared memory with int32 accumulators.
#include "up_internal.h"

namespace up {
namespace {

constexpr int kCoefOne = 2048;   // INTER_RESIZE_COEF_SCALE

// cv2's source index and fixed-point weights of destination index d along one axis.
__device__ __forceinline__ void axis_coef(int d, double scale, int src, bool clamp_fraction, int& s, int& c0, int& c1) {
  const float f0 = static_cast<float>(__dadd_rn(__dmul_rn(__dadd_rn(static_cast<double>(d), 0.5), scale), -0.5));
  int si = static_cast<int>(floorf(f0));
  float f = __fsub_rn(f0, static_cast<float>(si));
  if (clamp_fraction) {
    if (si < 0) { f = 0.f; si = 0; }
    if (si >= src - 1) { f = 0.f; si = src - 1; }
  }
  c0 = __float2int_rn(__fmul_rn(__fsub_rn(1.f, f), static_cast<float>(kCoefOne)));
  c1 = __float2int_rn(__fmul_rn(f, static_cast<float>(kCoefOne)));
  s = si;
}

__device__ __forceinline__ double inv_ratio(int dst, int src) {
  return __ddiv_rn(1.0, __ddiv_rn(static_cast<double>(dst), static_cast<double>(src)));
}

// Copy `bytes` bytes of one source row to shared memory.
__device__ __forceinline__ void stage_row(const uint8_t* __restrict__ p, uint8_t* dst, int bytes) {
  int done = 0;
  if ((reinterpret_cast<uintptr_t>(p) & 15) == 0) {
    const int nv = bytes >> 4;
    for (int i = threadIdx.x; i < nv; i += blockDim.x)
      reinterpret_cast<uint4*>(dst)[i] = __ldg(reinterpret_cast<const uint4*>(p) + i);
    done = nv << 4;
  }
  for (int i = done + threadIdx.x; i < bytes; i += blockDim.x) dst[i] = __ldg(p + i);
}

// kOut: 0 fp16 / 1 bf16 / 2 split space-to-depth, 3 uint8 HWC, 4 fp32 NCHW.
template <int kOut>
__global__ void __launch_bounds__(256) resize_pack_u8_kernel(const UpImageJob* __restrict__ jobs, int out_h, int out_w,
                                                             void* __restrict__ y, long long plane, int wpitch, int wpad,
                                                             int row_bytes, float mean, float inv_std, float std_) {
  extern __shared__ __align__(16) uint8_t smem[];
  const int b = blockIdx.y, yq = blockIdx.x;
  const UpImageJob job = jobs[b];
  const int h = job.h, w = job.w;
  const bool area = (h == 2 * out_h && w == 2 * out_w);
  int* xo0 = reinterpret_cast<int*>(smem);        // byte offset of the left source pixel, per output column
  int* xo1 = xo0 + out_w;                          // ... of the right one
  uint32_t* xab = reinterpret_cast<uint32_t*>(xo1 + out_w);   // a0 | a1 << 16
  uint8_t* rows = smem + ((12 * out_w + 15) & ~15);

  const double sx_scale = inv_ratio(out_w, w);
  for (int ox = threadIdx.x; ox < out_w; ox += blockDim.x) {
    const int rx = job.flip ? out_w - 1 - ox : ox;
    if (area) {
      xo0[ox] = 6 * rx;
      xo1[ox] = 6 * rx + 3;
      xab[ox] = 0;
    } else {
      int s, a0, a1;
      axis_coef(rx, sx_scale, w, true, s, a0, a1);
      xo0[ox] = 3 * s;
      xo1[ox] = 3 * min(s + 1, w - 1);     // a1 == 0 wherever s + 1 would leave the image
      xab[ox] = static_cast<uint32_t>(a0) | (static_cast<uint32_t>(a1) << 16);
    }
  }
  // source rows of output rows 2yq (slots 0, 1) and 2yq + 1 (slots 2, 3), with their weights
  int srow[4], beta[4];
  const double sy_scale = inv_ratio(out_h, h);
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int oy = 2 * yq + r;
    if (area) {
      srow[2 * r] = 2 * oy;
      srow[2 * r + 1] = 2 * oy + 1;
      beta[2 * r] = beta[2 * r + 1] = 0;
    } else {
      int s, b0, b1;
      axis_coef(oy, sy_scale, h, false, s, b0, b1);
      srow[2 * r] = min(max(s, 0), h - 1);
      srow[2 * r + 1] = min(max(s + 1, 0), h - 1);
      beta[2 * r] = b0;
      beta[2 * r + 1] = b1;
    }
  }
  // stage each distinct source row once (an upscale repeats rows)
  int slot[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    slot[k] = k;
#pragma unroll
    for (int j = 0; j < k; ++j)
      if (slot[k] == k && srow[j] == srow[k]) slot[k] = slot[j];
    if (slot[k] == k) stage_row(job.src + static_cast<long long>(srow[k]) * job.pitch, rows + k * row_bytes, 3 * w);
  }
  __syncthreads();

  const int wq = out_w / 2;
  for (int xq = threadIdx.x; xq < wq; xq += blockDim.x) {
    uint8_t px[2][2][3];   // [row][column][channel]
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const uint8_t* r0 = rows + slot[2 * r] * row_bytes;
      const uint8_t* r1 = rows + slot[2 * r + 1] * row_bytes;
#pragma unroll
      for (int pw = 0; pw < 2; ++pw) {
        const int ox = 2 * xq + pw;
        const int o0 = xo0[ox], o1 = xo1[ox];
        const uint32_t ab = xab[ox];
        const int a0 = static_cast<int>(ab & 0xFFFF), a1 = static_cast<int>(ab >> 16);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          int u;
          if (area) {
            u = (r0[o0 + c] + r0[o1 + c] + r1[o0 + c] + r1[o1 + c] + 2) >> 2;
          } else {
            const int h0 = r0[o0 + c] * a0 + r0[o1 + c] * a1;
            const int h1 = r1[o0 + c] * a0 + r1[o1 + c] * a1;
            const int v = (((h0 >> 4) * beta[2 * r]) >> 16) + (((h1 >> 4) * beta[2 * r + 1]) >> 16);
            u = min(max((v + 2) >> 2, 0), 255);
          }
          px[r][pw][c] = static_cast<uint8_t>(u);
        }
      }
    }
    if constexpr (kOut <= 2) {
      // space-to-depth pixel: 16 channels, order (ph, pw, c), 12 real (as pack_input_u8_s2d_kernel)
      float v0[8], v1[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) v0[e] = v1[e] = 0.f;
#pragma unroll
      for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int pw = 0; pw < 2; ++pw)
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            const int idx = (r * 2 + pw) * 3 + c;
            const float f = (static_cast<float>(px[r][pw][c]) - mean) * inv_std;
            if (idx < 8) v0[idx] = f; else v1[idx - 8] = f;
          }
      uint16_t* o = static_cast<uint16_t*>(y) + ((static_cast<long long>(b) * (out_h / 2) + yq) * wpitch + xq + wpad) * 16;
      store8_16<kOut>(o, plane, v0);
      store8_16<kOut>(o + 8, plane, v1);
    } else if constexpr (kOut == 3) {
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        uint16_t* o = reinterpret_cast<uint16_t*>(static_cast<uint8_t*>(y) +
                                                  ((static_cast<long long>(b) * out_h + 2 * yq + r) * out_w + 2 * xq) * 3);
        o[0] = px[r][0][0] | (px[r][0][1] << 8);
        o[1] = px[r][0][2] | (px[r][1][0] << 8);
        o[2] = px[r][1][1] | (px[r][1][2] << 8);
      }
    } else {
#pragma unroll
      for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int r = 0; r < 2; ++r) {
          float2* o = reinterpret_cast<float2*>(static_cast<float*>(y) +
                                                ((static_cast<long long>(b) * 3 + c) * out_h + 2 * yq + r) * out_w + 2 * xq);
          *o = make_float2(__fdiv_rn(static_cast<float>(px[r][0][c]) - mean, std_),
                           __fdiv_rn(static_cast<float>(px[r][1][c]) - mean, std_));
        }
    }
  }
}

}  // namespace
}  // namespace up

using namespace up;

extern "C" int up_resize_pack_u8(const UpImageJob* jobs, const UpImageJob* jobs_dev, int n, int out_h, int out_w,
                                 int out_format, void* y, int64_t y_plane_stride, int y_wpitch, int y_wpad_left,
                                 float mean, float std_, void* stream) {
  UP_CHECK_ARG(jobs && jobs_dev && y, "up_resize_pack_u8: null argument (jobs, jobs_dev and y are required)");
  UP_CHECK_ARG(n > 0 && n <= 65535, "up_resize_pack_u8: batch size %d outside [1, 65535]", n);
  UP_CHECK_ARG(out_h > 0 && out_w > 0 && out_h % 16 == 0 && out_w % 16 == 0,
               "up_resize_pack_u8: output size %dx%d must be positive multiples of 16", out_h, out_w);
  int max_w = 0;
  for (int i = 0; i < n; ++i) {
    const UpImageJob& j = jobs[i];
    UP_CHECK_ARG(j.src != nullptr, "up_resize_pack_u8: image %d has a null source pointer", i);
    UP_CHECK_ARG(j.h > 0 && j.w > 0, "up_resize_pack_u8: image %d is empty (%d x %d)", i, j.h, j.w);
    UP_CHECK_ARG(j.w <= (1 << 28) / 3 && j.pitch >= 3 * j.w,
                 "up_resize_pack_u8: image %d: row pitch %d bytes is less than 3 * width (%d)", i, j.pitch, j.w);
    UP_CHECK_ARG(j.flip == 0 || j.flip == 1, "up_resize_pack_u8: image %d: flip must be 0 or 1", i);
    max_w = j.w > max_w ? j.w : max_w;
  }
  const bool s2d = out_format == UP_BF16 || out_format == UP_FP16 || out_format == UP_SPLIT;
  UP_CHECK_ARG(s2d || out_format == UP_RESIZE_OUT_U8 || out_format == UP_RESIZE_OUT_F32,
               "up_resize_pack_u8: bad out_format %d", out_format);
  UP_CHECK_ARG(std_ != 0.f, "up_resize_pack_u8: std must be non-zero");
  if (s2d) {
    UP_CHECK_ARG((reinterpret_cast<uintptr_t>(y) & 15) == 0, "up_resize_pack_u8: y must be 16-byte aligned");
    if (y_wpitch <= 0) y_wpitch = out_w / 2;
    UP_CHECK_ARG(y_wpad_left >= 0 && y_wpad_left + out_w / 2 <= y_wpitch, "up_resize_pack_u8: bad row pitch / padding");
  } else {
    UP_CHECK_ARG((reinterpret_cast<uintptr_t>(y) & 7) == 0, "up_resize_pack_u8: y must be 8-byte aligned");
  }
  DeviceInfo* di = device_info();
  if (!di) return UP_ERR_UNSUPPORTED;
  const int row_bytes = (3 * max_w + 15) & ~15;
  const size_t smem = static_cast<size_t>((12 * out_w + 15) & ~15) + 4 * static_cast<size_t>(row_bytes);
  UP_CHECK_ARG(smem <= di->max_smem, "up_resize_pack_u8: an image %d pixels wide needs %zu bytes of shared memory "
               "(device limit %zu)", max_w, smem, di->max_smem);
  int threads = ((out_w / 2 + 31) / 32) * 32;
  threads = threads < 64 ? 64 : (threads > 256 ? 256 : threads);
  const dim3 grid(out_h / 2, n);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const float inv = 1.0f / std_;
  // (x - m) / s with s a power of two (256: mpii_data.py:184) is exact either way; for other s the space-to-depth
  // output is x * (1/s) as in up_pack_input_u8_s2d, the fp32 output a true division as Mytransforms.normalize
#define UP_RESIZE_LAUNCH(K)                                                                                            \
  do {                                                                                                                 \
    if (smem > 48 * 1024 &&                                                                                            \
        check_cuda(cudaFuncSetAttribute(resize_pack_u8_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize,         \
                                        static_cast<int>(smem)), "cudaFuncSetAttribute(resize_pack_u8_kernel)"))       \
      return UP_ERR_CUDA;                                                                                              \
    resize_pack_u8_kernel<K><<<grid, threads, smem, st>>>(jobs_dev, out_h, out_w, y, y_plane_stride, y_wpitch,         \
                                                         y_wpad_left, row_bytes, mean, inv, std_);                     \
  } while (0)
  switch (out_format) {
    case UP_FP16: UP_RESIZE_LAUNCH(0); break;
    case UP_BF16: UP_RESIZE_LAUNCH(1); break;
    case UP_SPLIT: UP_RESIZE_LAUNCH(2); break;
    case UP_RESIZE_OUT_U8: UP_RESIZE_LAUNCH(3); break;
    default: UP_RESIZE_LAUNCH(4); break;
  }
#undef UP_RESIZE_LAUNCH
  UP_CHECK_LAUNCH("resize_pack_u8_kernel");
  return 0;
}
