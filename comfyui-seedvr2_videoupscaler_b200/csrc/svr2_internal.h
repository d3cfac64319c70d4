// Internal (non-ABI) declarations shared by the .cu files of libsvr2.so.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/svr2.h"

namespace svr2 {
int set_error(int code, const char* msg);  // records the message for svr2_last_error(), returns code
int num_sms();          // of the current device
int current_device();   // cudaGetDevice, clamped to the per-device cache size
int make_tmap_bf16(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                   const uint32_t* box);
// elementwise.cu: layout converters / conv_out gather with an explicit NCDHW channel stride (temporal slices of a clip)
int ncdhw_to_ndhwc_strided(const void* in, int in_dtype, int C, int T, int H, int W, int64_t chan_stride, void* out,
                           int C_pad, int out_t_pad, float div, void* stream);
int ndhwc_to_ncdhw_strided(const void* in, int ld_in, int C, int T, int H, int W, void* out, int out_dtype,
                           int64_t chan_stride, void* stream);
int conv_tap_gather_strided(const float* z, int64_t ldz, int co_n, const void* bias, int T, int H, int W, void* out,
                            int out_dtype, int64_t chan_stride, void* stream);
// pre.cu: tap tables of torch's antialiased bicubic resize (_upsample_bicubic2d_aa) along one axis, laid out as
// first[out], count[out], weights[out][K]; K = the larger aa_taps() of the two axes, at most kAaMaxTaps
constexpr int kAaMaxTaps = 32;
int aa_taps(int in_size, int out_size);
void aa_tables(int in_size, int out_size, int K, int* first, int* count, float* weights, cudaStream_t s);
inline int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    char buf[256];
    snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(e));
    return set_error(SVR2_ERR_CUDA, buf);
  }
  return SVR2_OK;
}
}  // namespace svr2
