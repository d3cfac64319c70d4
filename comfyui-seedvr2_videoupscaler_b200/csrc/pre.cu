// Clip pre-processing (SURVEY.md §8(f) rank 3): the reference's prepare_video_transforms
// (src/core/generation_utils.py:72-84) as one pass over the output:
//   side resize, antialiased bicubic  (SideResize -> torchvision resize -> torch _upsample_bicubic2d_aa:
//                                      separable Keys cubic a = -0.5, support widened by the down-scale factor,
//                                      weights normalised, fp32 accumulation, horizontal taps first)
//   -> bf16 -> clamp(0,1) -> pad to multiples of 16 with zeros (DivisiblePad, divisible_crop.py:43-80)
//   -> Normalize(0.5, 0.5) -> t c h w -> c t h w
// The tap tables (first tap, tap count, weights per output column / row) are built on the device by a tiny kernel
// so that the call needs no host arrays and no synchronisation.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "svr2_internal.h"

namespace svr2 {
namespace {

constexpr int kMaxTaps = kAaMaxTaps;

__device__ __forceinline__ float rn(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }

__device__ __forceinline__ double cubic_aa(double x) {
  const double a = -0.5;
  x = fabs(x);
  if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1.0;
  if (x < 2.0) return (((x - 5.0) * x + 8.0) * x - 4.0) * a;
  return 0.0;
}

// table layout per axis: first[out], count[out], weights[out][K]
__global__ void aa_table_kernel(int in_size, int out_size, int K, int* __restrict__ first, int* __restrict__ count,
                                float* __restrict__ weights) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= out_size) return;
  const float scale = (float)in_size / (float)out_size;
  const float support = scale >= 1.0f ? 2.0f * scale : 2.0f;
  const float invscale = scale >= 1.0f ? 1.0f / scale : 1.0f;
  const float center = (float)((double)scale * ((double)i + 0.5));
  int lo = (int)(float)((double)center - (double)support + 0.5);
  if (lo < 0) lo = 0;
  int hi = (int)(float)((double)center + (double)support + 0.5);
  if (hi > in_size) hi = in_size;
  int n = hi - lo;
  if (n > K) n = K;
  const float lo_m_center = (float)((double)lo - (double)center);
  float tot = 0.f;
  float* w = weights + (long long)i * K;
  for (int j = 0; j < n; ++j) {
    const float arg = (float)(((double)j + (double)lo_m_center + 0.5) * (double)invscale);
    const float v = (float)cubic_aa((double)arg);
    w[j] = v;
    tot += v;
  }
  for (int j = 0; j < n; ++j)
    if (tot != 0.f) w[j] /= tot;
  for (int j = n; j < K; ++j) w[j] = 0.f;
  first[i] = lo;
  count[i] = n;
}

template <typename T>
__device__ __forceinline__ float load_bf16_rounded(const T* p);
template <>
__device__ __forceinline__ float load_bf16_rounded<float>(const float* p) { return rn(*p); }
template <>
__device__ __forceinline__ float load_bf16_rounded<__nv_bfloat16>(const __nv_bfloat16* p) { return __bfloat162float(*p); }
template <>
__device__ __forceinline__ float load_bf16_rounded<__half>(const __half* p) { return rn(__half2float(*p)); }

// One thread per output pixel, all three channels.
//   in : channels_last ? [T, h, w, Cin] : [T, 3, h, w]   (values rounded to bf16 on load = the compute dtype)
//   out: finish ? [3, T, Hp, Wp] clamp/pad/normalise : [T, 3, H, W] plain resize (Hp = H, Wp = W)
template <typename T>
__global__ void __launch_bounds__(256) resize_kernel(const T* __restrict__ in, __nv_bfloat16* __restrict__ out,
                                                     int frames, int h, int w, int cin, int channels_last, int H,
                                                     int W, int Hp, int Wp, int finish, int K,
                                                     const int* __restrict__ xfirst, const int* __restrict__ xcount,
                                                     const float* __restrict__ xw, const int* __restrict__ yfirst,
                                                     const int* __restrict__ ycount, const float* __restrict__ yw) {
  const int ox = blockIdx.x * 64 + (threadIdx.x & 63);
  const int oy = blockIdx.y * 4 + (threadIdx.x >> 6);
  const int t = blockIdx.z;
  if (ox >= Wp || oy >= Hp) return;
  const long long plane = (long long)Hp * Wp;
  float res[3];
  if (ox >= W || oy >= H) {
    res[0] = res[1] = res[2] = 0.f;                       // DivisiblePad: zeros before normalisation
  } else {
    const int x0 = xfirst[ox], nx = xcount[ox], y0 = yfirst[oy], ny = ycount[oy];
    const float* wx = xw + (long long)ox * K;
    const float* wy = yw + (long long)oy * K;
    // one pass over the taps for all three channels: each weight is fetched once, the per-channel accumulation
    // order (horizontal taps left to right, then rows top to bottom) is that of torch's kernel
    const long long cstride = channels_last ? 1 : (long long)h * w;
    const long long pstride = channels_last ? cin : 1;
    const T* base = in + (channels_last ? ((long long)t * h * w) * cin : ((long long)t * 3) * h * w);
    float acc[3] = {0.f, 0.f, 0.f};
    for (int j = 0; j < ny; ++j) {
      const T* row = base + ((long long)(y0 + j) * w + x0) * pstride;
      const float w0 = wx[0];
      float r[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) r[c] = load_bf16_rounded<T>(row + c * cstride) * w0;
      for (int i = 1; i < nx; ++i) {
        const float wi = wx[i];
#pragma unroll
        for (int c = 0; c < 3; ++c) r[c] += load_bf16_rounded<T>(row + i * pstride + c * cstride) * wi;
      }
      const float wj = wy[j];
#pragma unroll
      for (int c = 0; c < 3; ++c) acc[c] = (j == 0) ? r[c] * wj : acc[c] + r[c] * wj;
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) res[c] = rn(acc[c]);
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    if (finish) {
      const float v = fminf(fmaxf(res[c], 0.f), 1.f);
      out[((long long)c * frames + t) * plane + (long long)oy * Wp + ox] = __float2bfloat16_rn(rn(v - 0.5f) / 0.5f);
    } else {
      out[((long long)t * 3 + c) * plane + (long long)oy * Wp + ox] = __float2bfloat16_rn(res[c]);
    }
  }
}

inline size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

}  // namespace

int aa_taps(int in_size, int out_size) {
  const float scale = (float)in_size / (float)out_size;
  const float support = scale >= 1.0f ? 2.0f * scale : 2.0f;
  return (int)ceilf(support) * 2 + 1;
}

void aa_tables(int in_size, int out_size, int K, int* first, int* count, float* weights, cudaStream_t s) {
  aa_table_kernel<<<(out_size + 127) / 128, 128, 0, s>>>(in_size, out_size, K, first, count, weights);
}

}  // namespace svr2

using namespace svr2;

extern "C" int64_t svr2_resize_scratch_bytes(int h, int w, int H, int W) {
  if (h <= 0 || w <= 0 || H <= 0 || W <= 0) return 0;
  const int K = aa_taps(h, H) > aa_taps(w, W) ? aa_taps(h, H) : aa_taps(w, W);
  return (int64_t)(2 * align256((size_t)(H > W ? H : W) * 2 * sizeof(int)) +
                   2 * align256((size_t)(H > W ? H : W) * K * sizeof(float)));
}

extern "C" int svr2_resize_bicubic_aa_bf16(const void* in, int in_dtype, int channels_last, int cin, int frames, int h,
                                           int w, void* out, int H, int W, int finish, void* scratch,
                                           int64_t scratch_bytes, void* stream) {
  if (frames <= 0 || h <= 0 || w <= 0 || H <= 0 || W <= 0) return set_error(SVR2_ERR_ARG, "svr2_resize: empty image");
  if (frames > 65535) return set_error(SVR2_ERR_ARG, "svr2_resize: at most 65535 frames per call");
  if (cin < 3 || (!channels_last && cin != 3)) return set_error(SVR2_ERR_ARG, "svr2_resize: need >= 3 channels");
  const int K = aa_taps(h, H) > aa_taps(w, W) ? aa_taps(h, H) : aa_taps(w, W);
  if (K > kMaxTaps) return set_error(SVR2_ERR_ARG, "svr2_resize: down-scale factor too large (> 7x)");
  if (!scratch || scratch_bytes < svr2_resize_scratch_bytes(h, w, H, W))
    return set_error(SVR2_ERR_ARG, "svr2_resize: scratch too small (svr2_resize_scratch_bytes)");
  cudaStream_t s = (cudaStream_t)stream;
  const int L = H > W ? H : W;
  uint8_t* base = (uint8_t*)scratch;
  const size_t seg_i = align256((size_t)L * 2 * sizeof(int)), seg_w = align256((size_t)L * K * sizeof(float));
  int* xfirst = (int*)base;
  int* xcount = xfirst + L;
  int* yfirst = (int*)(base + seg_i);
  int* ycount = yfirst + L;
  float* xw = (float*)(base + 2 * seg_i);
  float* yw = (float*)(base + 2 * seg_i + seg_w);
  aa_tables(w, W, K, xfirst, xcount, xw, s);
  aa_tables(h, H, K, yfirst, ycount, yw, s);
  int rc = check_launch("aa_table");
  if (rc) return rc;
  const int Hp = finish ? (H + 15) / 16 * 16 : H, Wp = finish ? (W + 15) / 16 * 16 : W;
  dim3 grid((Wp + 63) / 64, (Hp + 3) / 4, frames);
#define SVR2_RESIZE(T)                                                                                             \
  resize_kernel<T><<<grid, 256, 0, s>>>((const T*)in, (__nv_bfloat16*)out, frames, h, w, cin, channels_last, H, W, \
                                        Hp, Wp, finish, K, xfirst, xcount, xw, yfirst, ycount, yw)
  if (in_dtype == 0) SVR2_RESIZE(float);
  else if (in_dtype == 1) SVR2_RESIZE(__nv_bfloat16);
  else if (in_dtype == 2) SVR2_RESIZE(__half);
  else return set_error(SVR2_ERR_ARG, "svr2_resize: in_dtype 0 fp32 | 1 bf16 | 2 fp16");
#undef SVR2_RESIZE
  return check_launch("resize_bicubic_aa");
}
