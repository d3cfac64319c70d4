// Edge-guided alpha upscaling of RGBA clips: the reference's edge_guided_alpha_upscale
// (src/core/alpha_upscaling.py:289-438) on the device.
//   svr2_alpha_resize_f32  source alpha -> antialiased bicubic to (H, W), clamp(0,1); counts the binary-mask test
//   svr2_alpha_edges_u8    upscaled RGB -> normalisation flags + per-frame Sobel maxima, then the edge map
//                          (cv2 RGB2GRAY + Sobel 3x3 BORDER_REFLECT_101, integer-exact, one maximum per frame)
//   svr2_alpha_refine      guided filter (eps 0.002, r = 2 binary / 3 gradient) with the binary-mask refinement fused
//                          into its second box pass
// The three batch-wide decisions (binary mask, first and second [-1,1] -> [0,1] normalisation) live in the caller's
// scratch as device counters / flags that the later kernels read: nothing synchronises with the host, and a captured
// CUDA graph stays correct when a replay's data flips a decision.
//
// The elementwise steps round every intermediate the way torch's separate CUDA kernels do (__f*_rn: no FMA
// contraction), and the box means sum their window row by row in avg_pool2d's order, so the device path reproduces
// the torch restatement (oracle/alpha_oracle.py) on the GPU up to the order of the 3-channel mean.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "svr2_internal.h"

namespace svr2 {
namespace {

constexpr int kMaxRadius = 3;
constexpr float kEps = 0.002f;

// ctrl block at the head of the scratch
struct AlphaCtrl {
  unsigned long long near_zero, near_one;  // source alpha < 0.1 / > 0.9
  unsigned int norm;                       // bit 0: min(rgb) < 0; bit 1: min((rgb + 1) / 2) < 0
  unsigned int pad;
};

inline size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

struct Layout {
  size_t ctrl, maxima, xi, yi, xw, yw, ab, total;
  int K;
};

Layout layout(int frames, int h, int w, int H, int W) {
  Layout l;
  l.K = aa_taps(h, H) > aa_taps(w, W) ? aa_taps(h, H) : aa_taps(w, W);
  l.ctrl = 0;
  l.maxima = align256(sizeof(AlphaCtrl));
  l.xi = l.maxima + align256((size_t)frames * 3 * sizeof(unsigned int));
  l.yi = l.xi + align256((size_t)W * 2 * sizeof(int));
  l.xw = l.yi + align256((size_t)H * 2 * sizeof(int));
  l.yw = l.xw + align256((size_t)W * l.K * sizeof(float));
  l.ab = l.yw + align256((size_t)H * l.K * sizeof(float));
  l.total = l.ab + align256((size_t)frames * H * W * sizeof(float2));
  return l;
}

__device__ __forceinline__ float rn_bf16(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }
template <typename T>
__device__ __forceinline__ float load_bf16_rounded(const T* p);
template <>
__device__ __forceinline__ float load_bf16_rounded<float>(const float* p) { return rn_bf16(*p); }
template <>
__device__ __forceinline__ float load_bf16_rounded<__nv_bfloat16>(const __nv_bfloat16* p) { return __bfloat162float(*p); }
template <>
__device__ __forceinline__ float load_bf16_rounded<__half>(const __half* p) { return rn_bf16(__half2float(*p)); }

__device__ __forceinline__ float ldf(const float* p) { return *p; }
__device__ __forceinline__ float ldf(const __nv_bfloat16* p) { return __bfloat162float(*p); }

__device__ __forceinline__ float norm1(float x) { return __fmul_rn(__fadd_rn(x, 1.f), 0.5f); }   // (x + 1) / 2

__device__ __forceinline__ bool is_binary(const AlphaCtrl* c, long long numel) {
  // (fp32(nz) + fp32(no)) / numel > 0.95, with torch CUDA's division by a scalar (multiply by the reciprocal)
  const float sum = __fadd_rn(__ull2float_rn(c->near_zero), __ull2float_rn(c->near_one));
  return __fmul_rn(sum, __fdiv_rn(1.f, (float)numel)) > 0.95f;
}

// ---------------------------------------------------------------- source alpha: binary-mask counts
// alpha element i of frame-major [T, h, w] sits at in[i * cstride + coff]
template <typename T>
__global__ void __launch_bounds__(256) alpha_count_kernel(const T* __restrict__ in, long long n, int cstride, int coff,
                                                          AlphaCtrl* __restrict__ ctrl) {
  unsigned int nz = 0, no = 0;
  for (long long i = blockIdx.x * 256ll + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const float a = load_bf16_rounded<T>(in + i * cstride + coff);
    nz += a < 0.1f;
    no += a > 0.9f;
  }
  nz = __reduce_add_sync(0xffffffffu, nz);
  no = __reduce_add_sync(0xffffffffu, no);
  if ((threadIdx.x & 31) == 0) {
    if (nz) atomicAdd(&ctrl->near_zero, (unsigned long long)nz);
    if (no) atomicAdd(&ctrl->near_one, (unsigned long long)no);
  }
}

// ---------------------------------------------------------------- source alpha: antialiased bicubic, fp32 result
// torch _upsample_bicubic2d_aa order: per tap row the horizontal taps left to right, then the rows top to bottom
template <typename T>
__global__ void __launch_bounds__(256) alpha_resize_kernel(const T* __restrict__ in, int cstride, int coff, int h, int w,
                                                           float* __restrict__ out, int H, int W, int K,
                                                           const int* __restrict__ xfirst, const int* __restrict__ xcount,
                                                           const float* __restrict__ xw, const int* __restrict__ yfirst,
                                                           const int* __restrict__ ycount, const float* __restrict__ yw) {
  const int ox = blockIdx.x * 64 + (threadIdx.x & 63);
  const int oy = blockIdx.y * 4 + (threadIdx.x >> 6);
  const int t = blockIdx.z;
  if (ox >= W || oy >= H) return;
  const int x0 = xfirst[ox], nx = xcount[ox], y0 = yfirst[oy], ny = ycount[oy];
  const float* wx = xw + (long long)ox * K;
  const float* wy = yw + (long long)oy * K;
  const T* base = in + (long long)t * h * w * cstride + coff;
  float acc = 0.f;
  for (int j = 0; j < ny; ++j) {
    const T* row = base + ((long long)(y0 + j) * w + x0) * cstride;
    float r = load_bf16_rounded<T>(row) * wx[0];
    for (int i = 1; i < nx; ++i) r += load_bf16_rounded<T>(row + (long long)i * cstride) * wx[i];
    acc = (j == 0) ? r * wy[j] : acc + r * wy[j];
  }
  out[((long long)t * H + oy) * W + ox] = fminf(fmaxf(acc, 0.f), 1.f);
}

// ---------------------------------------------------------------- edge map
constexpr int kEdgeTx = 32, kEdgeTy = 8;

__device__ __forceinline__ int reflect101(int i, int n) {
  if (n == 1) return 0;
  i = i < 0 ? -i : i;
  return i >= n ? 2 * n - 2 - i : i;
}
// numpy (x * 255).clip(0, 255).astype(uint8)
__device__ __forceinline__ int to_u8(float x) { return (int)fminf(fmaxf(__fmul_rn(x, 255.f), 0.f), 255.f); }
// OpenCV COLOR_RGB2GRAY on 8-bit input
__device__ __forceinline__ unsigned int gray8(int r, int g, int b) { return (9798 * r + 19235 * g + 3735 * b + 16384) >> 15; }

struct RgbView {
  long long cs, ts, rs;   // channel, frame, row strides in elements (pixels are contiguous)
};

// Loads the (kEdgeTx + 2) x (kEdgeTy + 2) gray tile around the block's outputs with the gray of all three
// normalisation variants packed per pixel (byte v = variant v: raw, normalised once, twice); returns the OR of
// this thread's normalisation flag bits.
template <typename TR>
__device__ unsigned int load_gray_tile(const TR* __restrict__ rgb, RgbView v, int t, int H, int W, int x0, int y0,
                                       unsigned int (*tile)[kEdgeTx + 2]) {
  unsigned int flags = 0;
  const TR* f = rgb + (long long)t * v.ts;
  for (int k = threadIdx.x; k < (kEdgeTx + 2) * (kEdgeTy + 2); k += blockDim.x) {
    const int ty = k / (kEdgeTx + 2), tx = k % (kEdgeTx + 2);
    const int y = reflect101(min(y0 + ty - 1, H), H), x = reflect101(min(x0 + tx - 1, W), W);
    const TR* p = f + (long long)y * v.rs + x;
    float c[3];
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) c[ch] = ldf(p + ch * v.cs);
    unsigned int packed = 0;
    int u[3][3];
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
      const float n1 = norm1(c[ch]), n2 = norm1(n1);
      flags |= (c[ch] < 0.f ? 1u : 0u) | (n1 < 0.f ? 2u : 0u);
      u[0][ch] = to_u8(c[ch]);
      u[1][ch] = to_u8(n1);
      u[2][ch] = to_u8(n2);
    }
#pragma unroll
    for (int var = 0; var < 3; ++var) packed |= gray8(u[var][0], u[var][1], u[var][2]) << (8 * var);
    tile[ty][tx] = packed;
  }
  return flags;
}

// gx^2 + gy^2 of cv2.Sobel(ksize=3) at tile position (ty, tx) (the output pixel's tile coordinates + 1)
__device__ __forceinline__ int sobel_sq(unsigned int (*tile)[kEdgeTx + 2], int ty, int tx, int var) {
  auto g = [&](int dy, int dx) { return (int)((tile[ty + dy][tx + dx] >> (8 * var)) & 0xff); };
  const int gx = (g(-1, 1) - g(-1, -1)) + 2 * (g(0, 1) - g(0, -1)) + (g(1, 1) - g(1, -1));
  const int gy = (g(1, -1) - g(-1, -1)) + 2 * (g(1, 0) - g(-1, 0)) + (g(1, 1) - g(-1, 1));
  return gx * gx + gy * gy;
}

// pass 1: normalisation flags (ctrl->norm) and per-frame maxima of gx^2 + gy^2 for every variant
template <typename TR>
__global__ void __launch_bounds__(256) edge_stats_kernel(const TR* __restrict__ rgb, RgbView v, int H, int W,
                                                         AlphaCtrl* __restrict__ ctrl, unsigned int* __restrict__ maxima) {
  __shared__ unsigned int tile[kEdgeTy + 2][kEdgeTx + 2];
  const int t = blockIdx.z, x0 = blockIdx.x * kEdgeTx, y0 = blockIdx.y * kEdgeTy;
  unsigned int flags = load_gray_tile(rgb, v, t, H, W, x0, y0, tile);
  __syncthreads();
  const int tx = threadIdx.x % kEdgeTx, ty = threadIdx.x / kEdgeTx;
  const bool in = x0 + tx < W && y0 + ty < H;
  // every block of a frame targets the same few words: read them (L2) first and only issue the atomics that can
  // change them, or the same-address atomics serialise the whole pass
  flags = __reduce_or_sync(0xffffffffu, flags);
  if ((threadIdx.x & 31) == 0 && (__ldcg(&ctrl->norm) | flags) != __ldcg(&ctrl->norm)) atomicOr(&ctrl->norm, flags);
#pragma unroll
  for (int var = 0; var < 3; ++var) {
    const unsigned int s = __reduce_max_sync(0xffffffffu, in ? (unsigned int)sobel_sq(tile, ty + 1, tx + 1, var) : 0u);
    if ((threadIdx.x & 31) == 0 && s > __ldcg(&maxima[t * 3 + var])) atomicMax(&maxima[t * 3 + var], s);
  }
}

// pass 2: edge_u8 = trunc(sqrt(s) / sqrt(max_frame) * 255) in fp64 (numpy's order); 0 for a frame without edges
template <typename TR>
__global__ void __launch_bounds__(256) edge_kernel(const TR* __restrict__ rgb, RgbView v, int H, int W,
                                                   const AlphaCtrl* __restrict__ ctrl,
                                                   const unsigned int* __restrict__ maxima, uint8_t* __restrict__ edges) {
  __shared__ unsigned int tile[kEdgeTy + 2][kEdgeTx + 2];
  const int t = blockIdx.z, x0 = blockIdx.x * kEdgeTx, y0 = blockIdx.y * kEdgeTy;
  load_gray_tile(rgb, v, t, H, W, x0, y0, tile);
  __syncthreads();
  const int tx = threadIdx.x % kEdgeTx, ty = threadIdx.x / kEdgeTx;
  if (x0 + tx >= W || y0 + ty >= H) return;
  const unsigned int norm = ctrl->norm;
  const int var = (norm & 1u) ? ((norm & 2u) ? 2 : 1) : 0;
  const unsigned int m = maxima[t * 3 + var];
  int e = 0;
  if (m) e = (int)(sqrt((double)sobel_sq(tile, ty + 1, tx + 1, var)) / sqrt((double)m) * 255.0);
  edges[((long long)t * H + y0 + ty) * W + x0 + tx] = (uint8_t)e;
}

// ---------------------------------------------------------------- guided filter
// Output tile 32 x 32 per block of 32 x 8 threads (4 rows each), inputs with a halo of r <= kMaxRadius.
constexpr int kGfT = 32, kGfS = kGfT + 2 * kMaxRadius;

// the guide: mean of the three channels of rgb_n, as torch's CUDA mean reduces them ((r + g) + b) * (1/3)
template <typename TR>
__device__ __forceinline__ float guide_at(const TR* __restrict__ rgb, RgbView v, int t, int y, int x, bool norm) {
  const TR* p = rgb + t * v.ts + y * v.rs + x;
  float c[3];
#pragma unroll
  for (int ch = 0; ch < 3; ++ch) {
    c[ch] = ldf(p + ch * v.cs);
    if (norm) c[ch] = norm1(c[ch]);
  }
  return __fmul_rn(__fadd_rn(__fadd_rn(c[0], c[1]), c[2]), 1.f / 3.f);
}

// stage 1: per pixel a = cov(I, p) / (var(I) + eps), b = mean(p) - a mean(I) over the (2r+1)^2 box
template <typename TR>
__global__ void __launch_bounds__(256) guided_ab_kernel(const TR* __restrict__ rgb, RgbView v,
                                                        const float* __restrict__ alpha, int H, int W, long long numel,
                                                        const AlphaCtrl* __restrict__ ctrl, float2* __restrict__ ab) {
  __shared__ float sI[kGfS][kGfS], sP[kGfS][kGfS];
  const int t = blockIdx.z, x0 = blockIdx.x * kGfT, y0 = blockIdx.y * kGfT;
  const bool norm = ctrl->norm & 1u;
  const int r = is_binary(ctrl, numel) ? 2 : 3;
  const int span = kGfT + 2 * r;
  for (int k = threadIdx.x; k < span * span; k += blockDim.x) {
    const int ty = k / span, tx = k % span;
    const int y = y0 + ty - r, x = x0 + tx - r;
    const bool in = y >= 0 && y < H && x >= 0 && x < W;     // avg_pool2d's zero padding
    sI[ty][tx] = in ? guide_at(rgb, v, t, y, x, norm) : 0.f;
    sP[ty][tx] = in ? alpha[((long long)t * H + y) * W + x] : 0.f;
  }
  __syncthreads();
  const float pool = (float)((2 * r + 1) * (2 * r + 1));
  const int tx = threadIdx.x % kGfT;
  for (int ty = threadIdx.x / kGfT; ty < kGfT; ty += blockDim.x / kGfT) {
    if (x0 + tx >= W || y0 + ty >= H) continue;
    float sI1 = 0.f, sP1 = 0.f, sII = 0.f, sIP = 0.f;
    for (int dy = 0; dy <= 2 * r; ++dy)
      for (int dx = 0; dx <= 2 * r; ++dx) {
        const float i = sI[ty + dy][tx + dx], p = sP[ty + dy][tx + dx];
        sI1 = __fadd_rn(sI1, i);
        sP1 = __fadd_rn(sP1, p);
        sII = __fadd_rn(sII, __fmul_rn(i, i));
        sIP = __fadd_rn(sIP, __fmul_rn(i, p));
      }
    const float mI = __fdiv_rn(sI1, pool), mP = __fdiv_rn(sP1, pool);
    const float var = __fsub_rn(__fdiv_rn(sII, pool), __fmul_rn(mI, mI));
    const float cov = __fsub_rn(__fdiv_rn(sIP, pool), __fmul_rn(mI, mP));
    const float a = __fdiv_rn(cov, __fadd_rn(var, kEps));
    ab[((long long)t * H + y0 + ty) * W + x0 + tx] = make_float2(a, __fsub_rn(mP, __fmul_rn(a, mI)));
  }
}

__device__ __forceinline__ float step05(float x) { return x > 0.5f ? 1.f : 0.f; }

// stage 2: q = box(a) I + box(b); binary masks then get the edge-aware refinement (alpha_upscaling.py:358-408);
// clamp(0, 1) and store
template <typename TR, typename TO>
__global__ void __launch_bounds__(256) guided_out_kernel(const TR* __restrict__ rgb, RgbView v,
                                                         const float2* __restrict__ ab, const uint8_t* __restrict__ edges,
                                                         int H, int W, long long numel, const AlphaCtrl* __restrict__ ctrl,
                                                         TO* __restrict__ out, int out_stride) {
  __shared__ float2 sAB[kGfS][kGfS];
  const int t = blockIdx.z, x0 = blockIdx.x * kGfT, y0 = blockIdx.y * kGfT;
  const bool norm = ctrl->norm & 1u;
  const bool binary = is_binary(ctrl, numel);
  const int r = binary ? 2 : 3;
  const int span = kGfT + 2 * r;
  for (int k = threadIdx.x; k < span * span; k += blockDim.x) {
    const int ty = k / span, tx = k % span;
    const int y = y0 + ty - r, x = x0 + tx - r;
    const bool in = y >= 0 && y < H && x >= 0 && x < W;
    sAB[ty][tx] = in ? ab[((long long)t * H + y) * W + x] : make_float2(0.f, 0.f);
  }
  __syncthreads();
  const float pool = (float)((2 * r + 1) * (2 * r + 1));
  const int tx = threadIdx.x % kGfT;
  for (int ty = threadIdx.x / kGfT; ty < kGfT; ty += blockDim.x / kGfT) {
    const int y = y0 + ty, x = x0 + tx;
    if (x >= W || y >= H) continue;
    float sa = 0.f, sb = 0.f;
    for (int dy = 0; dy <= 2 * r; ++dy)
      for (int dx = 0; dx <= 2 * r; ++dx) {
        const float2 e = sAB[ty + dy][tx + dx];
        sa = __fadd_rn(sa, e.x);
        sb = __fadd_rn(sb, e.y);
      }
    const float I = guide_at(rgb, v, t, y, x, norm);
    const float q = __fadd_rn(__fmul_rn(__fdiv_rn(sa, pool), I), __fdiv_rn(sb, pool));
    float res = q;
    if (binary) {
      const uint8_t* ef = edges + (long long)t * H * W;
      int tmax = 0;                                          // max_pool2d(3, 1, 1): -inf padding
      for (int dy = -1; dy <= 1; ++dy)
        for (int dx = -1; dx <= 1; ++dx) {
          const int yy = y + dy, xx = x + dx;
          if (yy >= 0 && yy < H && xx >= 0 && xx < W) tmax = max(tmax, (int)ef[(long long)yy * W + xx]);
        }
      const float edge = __fdiv_rn((float)ef[(long long)y * W + x], 255.f);
      const float transition = __fdiv_rn((float)tmax, 255.f);
      float comb;
      if (transition < 0.05f) {
        comb = step05(q);
      } else {
        const float ce = 1.f / (1.f + expf(-__fmul_rn(__fsub_rn(q, 0.5f), 12.f)));
        const float s = fminf(fmaxf(__fmul_rn(edge, 4.f), 0.f), 1.f);
        comb = __fadd_rn(__fmul_rn(q, __fsub_rn(1.f, s)), __fmul_rn(ce, s));
      }
      if (transition < 0.03f) comb = step05(comb);
      if (comb > 0.3f && comb < 0.7f && !(edge > 0.15f)) comb = step05(comb);
      res = comb;
    }
    res = fminf(fmaxf(res, 0.f), 1.f);
    const long long o = (((long long)t * H + y) * W + x) * out_stride;
    if constexpr (sizeof(TO) == 4) out[o] = res;
    else out[o] = __float2bfloat16_rn(res);
  }
}

int check_sizes(const char* what, int frames, int h, int w, int H, int W) {
  if (frames <= 0 || h <= 0 || w <= 0 || H <= 0 || W <= 0) return set_error(SVR2_ERR_ARG, what);
  if (frames > 65535) return set_error(SVR2_ERR_ARG, "svr2_alpha: at most 65535 frames per call");
  if (aa_taps(h, H) > kAaMaxTaps || aa_taps(w, W) > kAaMaxTaps)
    return set_error(SVR2_ERR_ARG, "svr2_alpha: alpha down-scale factor too large (> 7x)");
  return SVR2_OK;
}

int check_scratch(const char* what, const void* scratch, int64_t bytes, int frames, int h, int w, int H, int W) {
  if (!scratch || bytes < (int64_t)layout(frames, h, w, H, W).total) return set_error(SVR2_ERR_ARG, what);
  return SVR2_OK;
}

}  // namespace
}  // namespace svr2

using namespace svr2;

extern "C" int64_t svr2_alpha_scratch_bytes(int frames, int h, int w, int H, int W) {
  if (frames <= 0 || h <= 0 || w <= 0 || H <= 0 || W <= 0) return 0;
  return (int64_t)layout(frames, h, w, H, W).total;
}

extern "C" int svr2_alpha_resize_f32(const void* alpha, int dtype, int channels, int channel, int frames, int h, int w,
                                     float* out, int H, int W, void* scratch, int64_t scratch_bytes, void* stream) {
  int rc = check_sizes("svr2_alpha_resize_f32: empty image", frames, h, w, H, W);
  if (rc) return rc;
  if (!alpha || !out) return set_error(SVR2_ERR_ARG, "svr2_alpha_resize_f32: null tensor");
  if (channels < 0 || (channels > 0 && (channel < 0 || channel >= channels)) || (channels == 0 && channel != 0))
    return set_error(SVR2_ERR_ARG, "svr2_alpha_resize_f32: channel outside [0, channels)");
  rc = check_scratch("svr2_alpha_resize_f32: scratch too small (svr2_alpha_scratch_bytes)", scratch, scratch_bytes,
                     frames, h, w, H, W);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  const Layout l = layout(frames, h, w, H, W);
  uint8_t* base = (uint8_t*)scratch;
  AlphaCtrl* ctrl = (AlphaCtrl*)(base + l.ctrl);
  int* xi = (int*)(base + l.xi);
  int* yi = (int*)(base + l.yi);
  float* xw = (float*)(base + l.xw);
  float* yw = (float*)(base + l.yw);
  if (cudaMemsetAsync(ctrl, 0, 2 * sizeof(unsigned long long), s) != cudaSuccess)
    return check_launch("svr2_alpha_resize_f32: memset");
  aa_tables(w, W, l.K, xi, xi + W, xw, s);
  aa_tables(h, H, l.K, yi, yi + H, yw, s);
  const int cs = channels > 0 ? channels : 1;
  const long long n = (long long)frames * h * w;
  const int cblocks = (int)((n + 255) / 256 < 4096 ? (n + 255) / 256 : 4096);
  dim3 grid((W + 63) / 64, (H + 3) / 4, frames);
#define SVR2_ALPHA_RESIZE(T)                                                                                        \
  alpha_count_kernel<T><<<cblocks, 256, 0, s>>>((const T*)alpha, n, cs, channel, ctrl);                             \
  alpha_resize_kernel<T><<<grid, 256, 0, s>>>((const T*)alpha, cs, channel, h, w, out, H, W, l.K, xi, xi + W, xw, yi, \
                                              yi + H, yw)
  if (dtype == 0) { SVR2_ALPHA_RESIZE(float); }
  else if (dtype == 1) { SVR2_ALPHA_RESIZE(__nv_bfloat16); }
  else if (dtype == 2) { SVR2_ALPHA_RESIZE(__half); }
  else return set_error(SVR2_ERR_ARG, "svr2_alpha_resize_f32: dtype 0 fp32 | 1 bf16 | 2 fp16");
#undef SVR2_ALPHA_RESIZE
  return check_launch("svr2_alpha_resize_f32");
}

extern "C" int svr2_alpha_edges_u8(const void* rgb, int rgb_dtype, int64_t chan_stride, int64_t frame_stride,
                                   int64_t row_stride, int frames, int h, int w, int H, int W, uint8_t* edges,
                                   void* scratch, int64_t scratch_bytes, void* stream) {
  int rc = check_sizes("svr2_alpha_edges_u8: empty image", frames, h, w, H, W);
  if (rc) return rc;
  if (!rgb || !edges) return set_error(SVR2_ERR_ARG, "svr2_alpha_edges_u8: null tensor");
  if (row_stride < W) return set_error(SVR2_ERR_ARG, "svr2_alpha_edges_u8: row stride shorter than a row");
  rc = check_scratch("svr2_alpha_edges_u8: scratch too small (svr2_alpha_scratch_bytes)", scratch, scratch_bytes, frames,
                     h, w, H, W);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  const Layout l = layout(frames, h, w, H, W);
  uint8_t* base = (uint8_t*)scratch;
  AlphaCtrl* ctrl = (AlphaCtrl*)(base + l.ctrl);
  unsigned int* maxima = (unsigned int*)(base + l.maxima);
  if (cudaMemsetAsync(&ctrl->norm, 0, sizeof(unsigned int), s) != cudaSuccess ||
      cudaMemsetAsync(maxima, 0, (size_t)frames * 3 * sizeof(unsigned int), s) != cudaSuccess)
    return check_launch("svr2_alpha_edges_u8: memset");
  const RgbView v{chan_stride, frame_stride, row_stride};
  dim3 grid((W + kEdgeTx - 1) / kEdgeTx, (H + kEdgeTy - 1) / kEdgeTy, frames);
#define SVR2_ALPHA_EDGES(T)                                                                            \
  edge_stats_kernel<T><<<grid, 256, 0, s>>>((const T*)rgb, v, H, W, ctrl, maxima);                     \
  edge_kernel<T><<<grid, 256, 0, s>>>((const T*)rgb, v, H, W, ctrl, maxima, edges)
  if (rgb_dtype == 0) { SVR2_ALPHA_EDGES(float); }
  else if (rgb_dtype == 1) { SVR2_ALPHA_EDGES(__nv_bfloat16); }
  else return set_error(SVR2_ERR_ARG, "svr2_alpha_edges_u8: rgb_dtype 0 fp32 | 1 bf16");
#undef SVR2_ALPHA_EDGES
  return check_launch("svr2_alpha_edges_u8");
}

extern "C" int svr2_alpha_refine(const void* rgb, int rgb_dtype, int64_t chan_stride, int64_t frame_stride,
                                 int64_t row_stride, const float* alpha_up, const uint8_t* edges, int frames, int h,
                                 int w, int H, int W, void* out, int out_dtype, int out_stride, void* scratch,
                                 int64_t scratch_bytes, void* stream) {
  int rc = check_sizes("svr2_alpha_refine: empty image", frames, h, w, H, W);
  if (rc) return rc;
  if (!rgb || !alpha_up || !edges || !out) return set_error(SVR2_ERR_ARG, "svr2_alpha_refine: null tensor");
  if (row_stride < W || out_stride < 1) return set_error(SVR2_ERR_ARG, "svr2_alpha_refine: bad stride");
  rc = check_scratch("svr2_alpha_refine: scratch too small (svr2_alpha_scratch_bytes)", scratch, scratch_bytes, frames, h,
                     w, H, W);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  const Layout l = layout(frames, h, w, H, W);
  uint8_t* base = (uint8_t*)scratch;
  const AlphaCtrl* ctrl = (const AlphaCtrl*)(base + l.ctrl);
  float2* ab = (float2*)(base + l.ab);
  const long long numel = (long long)frames * h * w;
  const RgbView v{chan_stride, frame_stride, row_stride};
  dim3 grid((W + kGfT - 1) / kGfT, (H + kGfT - 1) / kGfT, frames);
#define SVR2_ALPHA_REFINE(TR, TO)                                                                                 \
  guided_ab_kernel<TR><<<grid, 256, 0, s>>>((const TR*)rgb, v, alpha_up, H, W, numel, ctrl, ab);                  \
  guided_out_kernel<TR, TO><<<grid, 256, 0, s>>>((const TR*)rgb, v, ab, edges, H, W, numel, ctrl, (TO*)out, out_stride)
  if (rgb_dtype != 0 && rgb_dtype != 1) return set_error(SVR2_ERR_ARG, "svr2_alpha_refine: rgb_dtype 0 fp32 | 1 bf16");
  if (out_dtype != 0 && out_dtype != 1) return set_error(SVR2_ERR_ARG, "svr2_alpha_refine: out_dtype 0 fp32 | 1 bf16");
  if (rgb_dtype == 0 && out_dtype == 0) { SVR2_ALPHA_REFINE(float, float); }
  else if (rgb_dtype == 0) { SVR2_ALPHA_REFINE(float, __nv_bfloat16); }
  else if (out_dtype == 0) { SVR2_ALPHA_REFINE(__nv_bfloat16, float); }
  else { SVR2_ALPHA_REFINE(__nv_bfloat16, __nv_bfloat16); }
#undef SVR2_ALPHA_REFINE
  return check_launch("svr2_alpha_refine");
}
