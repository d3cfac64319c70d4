/* libsvr2.so — C ABI of the B200-native SeedVR2 hot path (DiT forward + video-VAE).
 *
 * Every entry point is `extern "C"`, takes plain device pointers / sizes and a
 * CUDA stream handle (`void*` = cudaStream_t, 0 = default stream); no torch types.
 * All work is stream-ordered, no hidden synchronisation, no CPU fallback.
 * Return value: SVR2_OK (0) or a negative svr2_status; the message is available
 * from svr2_last_error() (thread-local).  Caller owns every buffer.
 *
 * bf16 = __nv_bfloat16 (torch.bfloat16) unless stated.  "Reference" citations are
 * file:line under numz/ComfyUI-SeedVR2_VideoUpscaler @ 4490bd1 — the Python
 * call each entry point replaces (the reference has no FFI of its own; see
 * INTEGRATION.md for the ctypes binding a maintainer would add).
 */
#ifndef SVR2_H_
#define SVR2_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum svr2_status {
  SVR2_OK = 0,
  SVR2_ERR_ARG = -1,   /* invalid argument / unsupported shape */
  SVR2_ERR_CUDA = -2,  /* CUDA runtime / driver error */
  SVR2_ERR_ARCH = -3,  /* device is not sm_100 */
};

/* epilogue flags of svr2_linear_bf16 / svr2_conv3d_bf16 (applied in this order,
 * each step rounded to bf16 where the reference's bf16 path rounds) */
enum svr2_epilogue {
  SVR2_EPI_BIAS = 1,      /* + bias[n]                                   nn.Linear / Conv3d bias              */
  SVR2_EPI_GATE = 2,      /* * gate[n] (fp32)                            AdaSingle "out", modulation.py:109-116 */
  SVR2_EPI_RESIDUAL = 4,  /* + residual[m,n]                             mmsr_block.py:113-114,125-126         */
  SVR2_EPI_SWIGLU = 8,    /* silu(acc[:, j]) * acc[:, j+128] per 256-col tile (weights interleaved) mlp.py:60-62 */
  SVR2_EPI_GELU = 16,     /* gelu_tanh                                   dit_7b/mlp.py:35-43                   */
  SVR2_EPI_F32 = 32,      /* fp32 output = acc * out_scale (attention scores)                                  */
  SVR2_EPI_SILU = 128,    /* silu                                        embedding.py:56-60                    */
  SVR2_EPI_ROWSTAT = 256, /* attention pass 1: out[m][slot] = (max, sum exp2) of acc*out_scale over the slot's columns   */
  SVR2_EPI_PEXP = 512,    /* attention pass 2: out = bf16(exp2(acc*out_scale - gate[m])), gate = per-row log2-sum-exp     */
  SVR2_EPI_ROWSCALE = 1024, /* acc * rowscale[m] first (svr2_linear_ex_bf16): un-normalised probabilities x V / row sum   */
};

const char* svr2_last_error(void);
/* 1: GEMM/conv tiles are executed by CTA pairs (tcgen05 cta_group::2, 256-row tiles); 0: single-CTA tiles.
 * Default from the environment variable SVR2_CTA_PAIR (unset = library default). */
void svr2_set_cta_pair(int on);
/* Stride-1 3x3 convs: 0 = generic tiles (32 x 8 / 16 x 8 pixels), 1 (default) = the W-reuse kernel for Cout <= 128 (tiles of
 * one 256-pixel row segment, the three horizontal taps read one activation stage) where rows split into segments with <= 4 %
 * waste, 2 = wherever a row holds a segment and also in the CTA-pair kernels (Cout >= 256, 128-pixel segments), 3 = 1 + the
 * CTA-pair kernels under the waste rule.  Default from SVR2_CONV_WR.  Changes svr2_conv_stat_slots(). */
void svr2_set_conv_wreuse(int mode);
int svr2_version(void);
/* fills sm count / major / minor of the current device; SVR2_ERR_ARCH unless sm_100 */
int svr2_device_check(int* sm_count, int* cc_major, int* cc_minor);

/* ---- Handle-based engine API (SURVEY.md §8(b)): one svr2_t per (process, device); not thread-safe; all work is
 * stream-ordered on the passed stream.  Ownership: the caller owns every I/O buffer; the engine owns its workspace and
 * the weights it copied (or borrows device pointers that must outlive the handle).  Errors: 0 = ok, negative svr2_status,
 * message from svr2_engine_last_error(); nothing throws across the ABI; there is no CPU fallback.
 *
 * The handle runs the whole NaDiT forward natively (C++ host runtime, csrc/engine.cu): window / RoPE geometry
 * (window.py:28-83, na.py:320-424,583-641, rope.py:130-176), workspace plan and the kernel sequence of
 * NaDiT.forward (dit_3b/nadit.py:190-248, dit_7b/nadit.py:152-190) for b = 1 at the folded timestep. */
typedef struct svr2_engine svr2_t;
typedef struct svr2_model_desc {
  int variant;        /* 0 = SeedVR2-3B structure, 1 = 7B structure (RoPE kind, window-size tables); 2 = the video VAE
                       * (s8_c16_t4 causal 3-D conv autoencoder; the remaining fields are ignored) */
  int dim, heads;     /* dim == heads * 128 */
  int layers, mm_layers;
  int txt_in_dim, in_ch, out_ch;
  int mlp_kind;       /* 0 = SwiGLU (mlp.py:46-62), 1 = GELU-tanh with biases (dit_7b/mlp.py:28-43) */
  int mlp_hidden;     /* 6912 (3B) / 12288 (7B) */
  int out_norm;       /* vid_out_norm + vid_out_ada present (3B) */
  int last_vid_only;  /* last block: text stream skips ada / mlp (mmsr_block.py:73-82) */
  float eps;
  float timestep;     /* the t folded into the AdaSingle vectors at load (informational) */
} svr2_model_desc;
typedef struct svr2_tensor_desc {
  const char* name;   /* engine-layout name, e.g. "12.vid.qkv.w", "12.vid.attn_scale", "12.rope_freqs", "vid_in.w" */
  const void* data;   /* host or device pointer */
  int dtype;          /* 0 fp32, 1 bf16, 2 fp16 */
  int rank;
  int64_t shape[5];
} svr2_tensor_desc;
int svr2_create(svr2_t** out, int device, const svr2_model_desc* desc);
void svr2_destroy(svr2_t* engine);
const char* svr2_engine_last_error(svr2_t* engine);
/* Weights in the engine layout (what weights.py / B200NaDiT._load produce: K-major bf16 matrices, SwiGLU gate / in rows
 * interleaved per 128, AdaSingle vectors E[:,layer,g] + P folded to fp32, "<i>.rope_freqs" in the checkpoint dtype).
 * copy != 0: the engine copies (caller keeps ownership of the source); copy == 0: device pointers are borrowed. */
int svr2_load_weights(svr2_t* engine, const svr2_tensor_desc* tensors, size_t n, int copy);
/* bytes of engine-owned workspace one forward of this geometry uses (T, H, W = latent frames / rows / columns) */
size_t svr2_workspace_bytes(svr2_t* engine, int T, int H, int W, int txt_len);
/* vid [T*H*W, in_ch] bf16, txt [txt_len, txt_in_dim] bf16 -> out [T*H*W, out_ch] bf16 (NaDiTOutput.vid_sample).  The
 * first call for a geometry builds its index tables (synchronous uploads) and may grow the workspace. */
int svr2_dit_forward(svr2_t* engine, const void* vid, const void* txt, int T, int H, int W, int txt_len, void* out,
                     void* stream);
/* the same forward in a caller-provided workspace (>= svr2_workspace_bytes, 256-byte aligned): the engine allocates and
 * retains nothing, so hosts that pool device memory (PyTorch's allocator, a CUDA-graph capture) keep control of it */
int svr2_dit_forward_ws(svr2_t* engine, const void* vid, const void* txt, int T, int H, int W, int txt_len, void* out,
                        void* workspace, size_t workspace_bytes, void* stream);

/* ---- Video VAE on a handle created with svr2_model_desc.variant == 2 (native host runtime csrc/vae_engine.cu).
 * Replaces VideoAutoencoderKLWrapper.encode / .decode (video_vae_v3/modules/attn_video_vae.py:1680-1698) incl. the
 * temporal slicing with the causal convs' memories (slicing_encode / slicing_decode :1254-1300,
 * causal_inflation_lib.py:306-352).  Weights (svr2_load_weights) carry the checkpoint's key names in the kernels'
 * layout: conv weights [Cout, kt, kh, kw, Cin] bf16 (rank 5, channels padded to a multiple of 64), "<resnet>.conv2+shortcut.
 * weight / .bias" = [W2 ; Wsc] rows and summed biases for resnets with a channel change, "upscale_conv.weight" [r*C, C],
 * "encoder.conv_in.weight" [128, 128] (im2col, K = 81 padded), "decoder.conv_out.weight" [81, 128] (tap-major), vectors bf16.
 *
 * All activations live in ONE workspace: svr2_vae_workspace_bytes() is exact (a dry run of the same sequence over a
 * first-fit arena), for direction 0 = encode (T sample frames of H x W pixels, H and W multiples of 8) or 1 = decode
 * (T latent frames of H x W latent pixels) cut into temporal slices of `slice_frames` (encode: sample frames, a multiple
 * of 4; decode: latent frames; 0 = un-sliced; the first slice additionally holds frame 0, like the reference's).  The
 * sliced result is bit-identical to the un-sliced one.  workspace == NULL: the engine owns (and grows) the workspace.
 *   encode: x [3, T, H, W] (x_dtype 0 f32 | 1 bf16 | 2 f16, values in [-1, 1]) -> latent [16, (T-1)/4+1, H/8, W/8] bf16
 *           (posterior mode; multiply by the scaling factor outside);
 *   decode: z [16, T, h, w] -> sample [3, 4T-3, 8h, 8w] bf16. */
size_t svr2_vae_workspace_bytes(svr2_t* engine, int direction, int T, int H, int W, int slice_frames);
int svr2_vae_encode(svr2_t* engine, const void* x, int x_dtype, int T, int H, int W, int slice_frames, void* latent,
                    void* workspace, size_t workspace_bytes, void* stream);
int svr2_vae_decode(svr2_t* engine, const void* z, int z_dtype, int T, int h, int w, int slice_frames, void* sample,
                    void* workspace, size_t workspace_bytes, void* stream);
/* kernels launched by the handle's last svr2_vae_encode / svr2_vae_decode */
int64_t svr2_vae_last_launches(svr2_t* engine);

/* ---- K1: Linear.  out[M,N] = epi(a[M,K] @ w[N,K]^T).  Replaces nn.Linear at
 * dit_3b/nablocks/attention/mmattn.py:56-59,173,269; dit_3b/mlp.py:56-61; dit_7b/mlp.py:35-43;
 * dit_3b/patch/patch_v1.py:37,62; dit_3b/embedding.py:38-40; diffusers Attention to_q/k/v/out
 * (attn_video_vae.py:612-632).  lda/ldw/ldc in elements, multiples of 8. */
int svr2_linear_bf16(const void* a, int64_t lda, const void* w, int64_t ldw, int M, int N, int K, int epi_flags,
                     const void* bias, const float* gate, const void* residual, void* out, int64_t ldc,
                     float out_scale, void* stream);

/* ---- K6: causal Conv3d (implicit GEMM).  Replaces InflatedCausalConv3d.forward
 * (video_vae_v3/modules/causal_inflation_lib.py:213-305) incl. Downsample3D's (0,1,0,1) pad
 * (attn_video_vae.py:242-244).  x: [T_in_total,H,W,Cin] NDHWC, the causal halo frames are real
 * frames at the front of x; w: [Cout][kt][kh][kw][Cin]; y: [out_t_pad+T_out,Ho,Wo,ldc]. */
int svr2_conv3d_bf16(const void* x, int T_in_total, int H, int W, int Cin, const void* w, int Cout, int kt, int kh,
                     int kw, int stride_t, int stride_hw, int pad_hw, int T_out, int epi_flags, const void* bias,
                     const void* residual, void* y, int out_t_pad, int out_dup_head, int ldc, void* stream);

/* Same conv, additionally emitting per-tile GroupNorm partial sums (fp32, deterministic order) of the stored
 * output so that the following causal_norm_wrapper needs no statistics pass.  stat_partial: [T_out][slots][Cout/8]
 * float4; pass NULL to query *stat_slots (bytes needed = T_out * slots * Cout/8 * 16). */
int svr2_conv3d_stats_bf16(const void* x, int T_in_total, int H, int W, int Cin, const void* w, int Cout, int kt, int kh,
                           int kw, int stride_t, int stride_hw, int pad_hw, int T_out, int epi_flags, const void* bias,
                           const void* residual, void* y, int out_t_pad, int out_dup_head, int ldc, void* stat_partial,
                           int64_t stat_bytes, int* stat_slots, void* stream);

/* slots per frame of the statistics output for an output of H_out x W_out pixels (pure function of the tile shape:
 * lets a caller plan memory without the NULL query) */
int svr2_conv_stat_slots(int Cout, int H_out, int W_out);

/* Stride-1 causal conv with the ResnetBlock3D 1x1x1 conv_shortcut fused in as extra K-blocks (attn_video_vae.py:311-362:
 * `x = conv_shortcut(x); return x + hidden`): y = conv(x; w[:, :kt*kh*kw*Cin]) + x2 . w[:, kt*kh*kw*Cin:]^T + bias,
 * x2 = [T_out, H, W, C2] bf16 (the block input, no halo, C2 % 64 == 0), w = [Cout][kt*kh*kw*Cin + C2] (conv2 weight rows
 * followed by the shortcut weight rows), bias = conv bias + shortcut bias.  One fp32 accumulation and one bf16 rounding
 * replace the reference's two roundings + add; saves the shortcut launch, its output write and the residual re-read.
 * Statistics output as svr2_conv3d_stats_bf16 (stat_partial == NULL: size query). */
int svr2_conv3d_shortcut_stats_bf16(const void* x, int T_in_total, int H, int W, int Cin, const void* w, int Cout, int kt,
                                    int kh, int kw, int T_out, const void* bias, const void* x2, int C2, void* y,
                                    int out_t_pad, int out_dup_head, void* stat_partial, int64_t stat_bytes,
                                    int* stat_slots, void* stream);

/* ---- Upsample3D: 1x1x1 conv + 'b (x y z c) f h w -> b c (f z) (h x) (w y)' + remove_head
 * (attn_video_vae.py:135-153, causal_inflation_lib.py:412-419) in one GEMM. */
int svr2_upsample_shuffle_bf16(const void* x, int F, int H, int W, int C, const void* w, const void* bias,
                               int temporal, int drop_head, void* y, int out_t_pad, int out_dup_head, void* stream);

/* ---- K4: varlen (windowed) self-attention, head_dim 128, non-causal, scale 1/sqrt(128).
 * Drop-in for FlashAttentionVarlen.forward / pytorch_varlen_attention (dit_3b/attention.py:27-64,
 * 114-148): q,k,v,out [total, heads, 128] bf16, cu_seqlens int32 [n_seq+1] (device).
 * out_row_map (optional, device int32 [total]): output row r is written to row out_row_map[r]
 * (fuses window_reverse, mmattn.py:264). */
int svr2_attn_varlen_bf16(const void* q, const void* k, const void* v, void* out, const int32_t* cu_seqlens,
                          int n_seq, int total, int heads, int max_seqlen, const int32_t* out_row_map,
                          void* stream);

/* ---- K2: RMSNorm (+optional affine) + AdaSingle "in".  CustomRMSNorm.forward
 * (dit_3b/normalization.py:88-109) + AdaSingle.forward (modulation.py:109-111).
 * mode 0: y = bf16((rms(x)*w) * scale + shift)          (attention branch / output head)
 * mode 1: y = bf16(bf16(bf16(rms(x)) * scale) + shift)  (MLP branch, mmsr_block.py:117-122) */
int svr2_rmsnorm_ada_bf16(const void* x, void* y, int rows, int dim, float eps, const float* weight,
                          const float* scale, const float* shift, int mode, void* stream);

/* ---- q/k RMSNorm(128, affine) + 3-axis RoPE + window partition + per-window text concat
 * (mmattn.py:199-248, rope.py:116-176, na.py:320-424).  qkv_vid [L,3*heads*128], qkv_txt [l,...];
 * row_src[total]: >=0 video token index, <0: -(text index+1); row_rope[total*3]: rows of the
 * cos/sin tables per axis (or -1 = no rotation); tables [R][nfreq] fp32. */
int svr2_qk_norm_rope_window_bf16(const void* qkv_vid, const void* qkv_txt, const int32_t* row_src,
                                  const int32_t* row_rope, const float* cos_tab, const float* sin_tab, int nfreq,
                                  const float* wq_vid, const float* wk_vid, const float* wq_txt, const float* wk_txt,
                                  float eps, int total, int heads, void* q, void* k, void* v, void* stream);
/* the same kernel on the subset of output rows in row_list[n_rows] (window-order row ids) */
int svr2_qk_norm_rope_rows_bf16(const void* qkv_vid, const void* qkv_txt, const int32_t* row_src, const int32_t* row_rope,
                                const float* cos_tab, const float* sin_tab, int nfreq, const float* wq_vid,
                                const float* wk_vid, const float* wq_txt, const float* wk_txt, float eps,
                                const int32_t* row_list, int n_rows, int heads, void* q, void* k, void* v, void* stream);
/* QKV projection (nn.Linear, mmattn.py:173) with everything NaSwinAttention does before the attention call fused into the
 * GEMM epilogue: bf16 rounding of the projection, per-head q/k RMSNorm (fp32, affine [128]), 3-axis RoPE on interleaved
 * pairs from cos/sin tables [R, nfreq] (nfreq = 21: 3B, 10: 7B), window partition (mmattn.py:199-248, rope.py:116-176).
 * a [M, K] (row stride lda), w [3*heads*128, K]; token m goes to row tok_dst[m] of q / k / v ([rows, heads*128]);
 * tok_rope [M, 3] = table rows per axis or -1; qk_weight [2][128] = q-norm, k-norm weights (fp32).  heads even. */
int svr2_linear_qkv_rope_bf16(const void* a, int64_t lda, const void* w, int64_t ldw, int M, int heads, int K,
                              const int32_t* tok_dst, const int32_t* tok_rope, const float* cos_tab, const float* sin_tab,
                              int nfreq, const float* qk_weight, float eps, void* q, void* k, void* v, void* stream);


/* mean over windows of the text rows (na.py:396-417): in [n_win, l, dim] -> out [l, dim] */
int svr2_txt_window_mean_bf16(const void* in, void* out, int n_win, int l, int dim, void* stream);

/* NaPatchIn / NaPatchOut rearranges (patch_v1.py:76-127), patch (1,2,2) */
int svr2_patchify_bf16(const void* vid, void* out, int T, int H, int W, int C, int ld_out, void* stream);
int svr2_unpatchify_bf16(const void* in, int ld_in, void* out, int T, int H, int W, int C, void* stream);

/* ---- K7: per-frame GroupNorm(32) (+SiLU).  causal_norm_wrapper
 * (causal_inflation_lib.py:354-409) + nn.SiLU.  x,y: [F,HW,C] NDHWC.  Deterministic (no float atomics):
 * block partials -> fixed-order finalize -> apply.  scratch: svr2_groupnorm_scratch_bytes() bytes, 8-aligned. */
int svr2_groupnorm_bf16(const void* x, void* y, int frames, int hw, int C, const void* gamma, const void* beta,
                        float eps, int silu, int out_t_pad, int out_dup_head, double* scratch,
                        int64_t scratch_bytes, void* stream);
int64_t svr2_groupnorm_scratch_bytes(int frames, int hw, int C);
/* GroupNorm(+SiLU) from the partial sums of svr2_conv3d_stats_bf16 (finalize + apply; coef_scratch: frames*C*8 B) */
int svr2_groupnorm_from_stats_bf16(const void* x, void* y, int frames, int hw, int C, const void* gamma,
                                   const void* beta, float eps, int silu, int out_t_pad, int out_dup_head,
                                   const void* stat_partial, int stat_slots, void* coef_scratch, void* stream);

/* VAE mid-block attention (1 head, d = 512; attn_video_vae.py:656-668) as two GEMM passes that never
 * materialise the fp32 score matrix: pass 1 = svr2_linear_bf16(..., SVR2_EPI_ROWSTAT) + svr2_rowstat_combine,
 * pass 2 = svr2_linear_bf16(..., SVR2_EPI_PEXP) writing normalised bf16 probabilities, then P @ V. */
int svr2_rowstat_slots(int N);
int svr2_rowstat_combine(const void* partial, int slots, int64_t ld, float* lse, int rows, void* stream);
/* Single-pass variant without the duplicated Q K^T (default for n >= 256 keys):
 *   1. reference exponent m^[m]: svr2_linear_bf16(q, every 16th key, SVR2_EPI_ROWSTAT) + svr2_rowstat_max — a 1/16-cost GEMM;
 *      any m^ within ~96 powers of two of the true row maximum is as good as the maximum itself;
 *   2. svr2_linear_ex_bf16(q, k, SVR2_EPI_PEXP, gate = m^, stat_out): un-normalised bf16(exp2(s - m^)) plus per-slot
 *      (max score, fp32 sum of the exponentials); svr2_pexp_stat_combine -> rowscale = 1 / sum and a device flag if some
 *      row's true maximum exceeded m^ by more than the safe margin (or the sum is not a positive finite number);
 *   3. svr2_linear_ex_bf16(P~, V^T, SVR2_EPI_ROWSCALE, rowscale) = softmax(q k^T) v;
 *   4. the exact two-pass launches above with run_if = flag: no-ops unless step 2 raised it (never observed). */
int svr2_linear_ex_bf16(const void* a, int64_t lda, const void* w, int64_t ldw, int M, int N, int K, int epi_flags,
                        const void* bias, const float* gate, const void* residual, void* out, int64_t ldc, float out_scale,
                        const float* rowscale, void* stat_out, int64_t ld_stat, const int* run_if, void* stream);
int svr2_rowstat_max(const void* partial, int slots, int64_t ld, float* mhat, int rows, int* flag_reset, void* stream);
int svr2_pexp_stat_combine(const void* partial, int slots, int64_t ld, const float* mhat, float* rowscale, int rows,
                           int* flag, void* stream);
/* row softmax fp32 -> bf16 (materialised-score variant, kept for small problems / tests) */
int svr2_softmax_rows_bf16(const float* s, int64_t lds, void* p, int64_t ldp, int rows, int cols, void* stream);
int svr2_transpose_bf16(const void* in, int64_t ld_in, void* out, int64_t ld_out, int rows, int cols, void* stream);

/* layout glue (optimization/performance.py:12-166): NCDHW any-float <-> NDHWC bf16 with halo / channel pad */
int svr2_ncdhw_to_ndhwc_bf16(const void* in, int in_dtype, int C, int T, int H, int W, void* out, int C_pad,
                             int out_t_pad, float div, void* stream);
int svr2_ndhwc_to_ncdhw(const void* in, int ld_in, int C, int T, int H, int W, void* out, int out_dtype,
                        void* stream);
/* Decoder conv_out (128 -> 3; attn_video_vae.py:1031-1033) second half: z[tap*co_n+co][pixel] (fp32, from one
 * svr2_linear_bf16(weights-as-A, activations-as-B, SVR2_EPI_F32) over all input pixels incl. the halo frames)
 * -> out[co][t][h][w] = bf16(bias + sum over the 27 taps), NCDHW. */
int svr2_conv_tap_gather(const float* z, int64_t ldz, int co_n, const void* bias, int T, int H, int W, void* out,
                         int out_dtype, void* stream);
/* 3x3x3 im2col for the 3-channel encoder conv_in: x [2+T,H,W,Cpad] -> out [T*H*W, ld_out] (81 real cols) */
int svr2_im2col3_bf16(const void* x, int T, int H, int W, int C, int ld_in, void* out, int ld_out, void* stream);

/* ---- Post-decode colour correction + image formatting (phase 4 of the reference pipeline,
 * generation_phases.py:1236-1345; SURVEY.md §8(f) rank 2).  Planar bf16 images [planes = T*3][H][W] in [-1,1].
 *
 * One level of the wavelet pyramid of wavelet_decomposition (src/utils/color_fix.py:122-184):
 *   low = bf16(blur_r(img)), 3x3 (1,2,1)x(1,2,1)/16, dilation r = min(radius, max(1, min(H,W)/8)), replicate pad;
 *   high (optional, in place) = bf16(bf16(high + img) - low)   [first != 0: high starts at zero];
 *   add_to/out (optional, replaces the `low` store) : out = clamp(bf16(add_to + low), -1, 1) — the recombination
 *   of wavelet_reconstruction (color_fix.py:187-246) fused into the last level of the style pass. */
int svr2_wavelet_level_bf16(const void* img, void* low, void* high, const void* add_to, void* out, int planes, int H,
                            int W, int radius, int first, void* stream);
/* adaptive_instance_normalization (color_fix.py:72-119): per plane, out = (c - mean_c) / std_c * std_s + mean_s with
 * unbiased variance, eps 1e-5 and the reference's bf16 rounding points.  stats_scratch: planes * 4 floats. */
int svr2_adain_bf16(const void* content, const void* style, void* out, int planes, int64_t hw, float* stats_scratch,
                    void* stream);
/* _rgb_to_lab_batch (color_fix.py:299-321, 368-413): rgb [frames,3,hw] bf16 in [-1,1] -> lab [3][frames*hw] fp32 */
int svr2_rgb_to_lab_f32(const void* rgb, float* lab, int frames, int64_t hw, void* stream);
/* luminance blend + _lab_to_rgb_batch (color_fix.py:333-357, 416-474): L = L_content * w + L_matched * (1 - w)
 * (L_matched may be NULL: L = L_content), a, b [frames*hw] fp32 -> rgb [frames,3,hw] bf16 in [-1,1] */
int svr2_lab_to_rgb_bf16(const float* L_content, const float* L_matched, const float* a, const float* b,
                         float luminance_weight, void* rgb, int frames, int64_t hw, void* stream);
/* _histogram_matching_channel (color_fix.py:477-521) for equally sized inputs: the r-th smallest source element is
 * replaced by the r-th smallest reference value (radix sorts + scatter). */
int64_t svr2_histogram_match_scratch_bytes(int64_t n);
int svr2_histogram_match_f32(const float* source, const float* reference, float* out, int64_t n, void* scratch,
                             int64_t scratch_bytes, void* stream);
/* final formatting (generation_phases.py:1322-1345): sample [frames,3,hw] bf16 -> image [frames,hw,3] bf16,
 * clamp(-1,1) * 0.5 + 0.5 */
int svr2_sample_to_image_bf16(const void* sample, void* image, int frames, int64_t hw, void* stream);

/* Temporal-overlap cross-fade of two neighbouring frame ranges (blend_overlapping_frames,
 * src/core/generation_utils.py:284-312): out[f] = bf16(bf16(prev[f] * w_prev[f]) + bf16(cur[f] * w_cur[f])); the
 * per-frame weights (Hann window for overlap >= 3, linear below) are passed as device fp32 arrays of bf16 values. */
int svr2_blend_overlap_bf16(const void* prev_tail, const void* cur_head, void* out, const float* w_prev,
                            const float* w_cur, int overlap, int64_t frame_elems, void* stream);

/* The same cross-fade on fp32 frames — the merge of per-GPU results (inference_cli.py:1241-1270): out = prev * w_prev +
 * cur * w_cur with three separately rounded fp32 operations. */
int svr2_blend_overlap_f32(const float* prev_tail, const float* cur_head, float* out, const float* w_prev,
                           const float* w_cur, int overlap, int64_t frame_elems, void* stream);

/* ---- Spatially tiled VAE seams (VideoAutoencoderKL.tiled_encode / tiled_decode, attn_video_vae.py:1302-1630; optional,
 * off in every BASELINE config).  Accumulate one tile [planes, eff_h, eff_w] (plane / row strides in elements) into
 * result [planes, H, W] at (y0, x0) with separable bf16 edge weights, and its weight into count [H, W]; rounding points
 * are torch's: tile.mul_(wh).mul_(ww); result += tile; count.addcmul_(wh, ww).  Then result.div_(count.clamp(1e-6)). */
int svr2_tile_accumulate_bf16(const void* tile, int64_t tile_plane_stride, int tile_row_stride, int planes, int eff_h,
                              int eff_w, const void* weight_h, const void* weight_w, void* result, void* count, int H,
                              int W, int y0, int x0, void* stream);
int svr2_tile_normalize_bf16(void* result, const void* count, int planes, int64_t hw, void* stream);

/* ---- Clip pre-processing (prepare_video_transforms, src/core/generation_utils.py:72-84; SURVEY.md §8(f) rank 3).
 * Antialiased bicubic resize (torchvision resize -> torch _upsample_bicubic2d_aa semantics, fp32 accumulation, result
 * rounded to bf16) of frames given as [T,h,w,cin] (channels_last != 0, first 3 channels) or [T,3,h,w]; in_dtype
 * 0 fp32 | 1 bf16 | 2 fp16, values rounded to bf16 on load (the pipeline's compute dtype).
 *   finish == 0: out [T,3,H,W] bf16 (plain resize);
 *   finish != 0: out [3,T,Hp,Wp] bf16 = clamp(0,1) -> zero pad to multiples of 16 -> (x - 0.5) / 0.5 -> c t h w,
 *                Hp = ceil16(H), Wp = ceil16(W)  (what VideoDiffusionInfer.vae_encode consumes). */
int64_t svr2_resize_scratch_bytes(int h, int w, int H, int W);
int svr2_resize_bicubic_aa_bf16(const void* in, int in_dtype, int channels_last, int cin, int frames, int h, int w,
                                void* out, int H, int W, int finish, void* scratch, int64_t scratch_bytes, void* stream);

/* ---- Alpha of RGBA clips (edge_guided_alpha_upscale, src/core/alpha_upscaling.py:289-438).
 * Three stages over one caller-owned scratch of svr2_alpha_scratch_bytes(T, h, w, H, W) bytes: the stages leave the
 * batch-wide decisions (binary mask; [-1,1] -> [0,1] normalisation of the RGB, once or twice) there as device flags,
 * so svr2_alpha_refine must run after svr2_alpha_resize_f32 and svr2_alpha_edges_u8 on the same scratch and stream.
 * No stage synchronises with the host.  The RGB is the decoded sample [T,3,H,W] before colour correction, fp32 or
 * bf16 (rgb_dtype 0 | 1) with element strides between channels, frames and rows (pixels contiguous).
 *   svr2_alpha_resize_f32: source alpha = channel `channel` of [T,h,w,channels] (channels > 0) or [T,1,h,w]
 *     (channels == 0), dtype 0 fp32 | 1 bf16 | 2 fp16, rounded to bf16 on load -> out [T,H,W] fp32 = antialiased
 *     bicubic (torch _upsample_bicubic2d_aa) then clamp(0,1); also counts the source alpha < 0.1 and > 0.9.
 *   svr2_alpha_edges_u8: edges [T,H,W] u8 = the reference's Sobel edge map (cv2 RGB2GRAY, Sobel 3x3 with
 *     BORDER_REFLECT_101, magnitude / per-frame maximum * 255 truncated, 0 for a frame without edges), bit-exact.
 *   svr2_alpha_refine: guided filter of the resized alpha by the mean of the normalised RGB (eps 0.002, radius 2 for
 *     a binary mask, else 3), the binary-mask refinement, clamp(0,1) -> out element ((t*H + y)*W + x) * out_stride,
 *     out_dtype 0 fp32 | 1 bf16 (out_stride 1: [T,1,H,W]; 4 with out at channel 3: the alpha of [T,H,W,4]). */
int64_t svr2_alpha_scratch_bytes(int frames, int h, int w, int H, int W);
int svr2_alpha_resize_f32(const void* alpha, int dtype, int channels, int channel, int frames, int h, int w, float* out,
                          int H, int W, void* scratch, int64_t scratch_bytes, void* stream);
int svr2_alpha_edges_u8(const void* rgb, int rgb_dtype, int64_t chan_stride, int64_t frame_stride, int64_t row_stride,
                        int frames, int h, int w, int H, int W, uint8_t* edges, void* scratch, int64_t scratch_bytes,
                        void* stream);
int svr2_alpha_refine(const void* rgb, int rgb_dtype, int64_t chan_stride, int64_t frame_stride, int64_t row_stride,
                      const float* alpha_up, const uint8_t* edges, int frames, int h, int w, int H, int W, void* out,
                      int out_dtype, int out_stride, void* scratch, int64_t scratch_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SVR2_H_ */
