/* flowhigh_b200 -- C ABI of the B200-native FLowHigh inference kernels (sm_100a).
 *
 * The reference (resemble-ai/flowhigh) has no FFI / plugin interface: its hot path is pure
 * PyTorch.  The drop-in boundary is therefore the Python class API (flowhigh_b200.FlowHighSR
 * mirrors src/flowhigh/flowhighsr.py:21-149); THIS header is the boundary underneath it, the
 * set of entry points the Python host code binds with ctypes (flowhigh_b200/_lib.py), and the
 * ones a maintainer of the reference would bind to replace the cited torch/scipy calls
 * (INTEGRATION.md shows the ctypes stubs).
 *
 * Conventions
 *   - every pointer is a raw DEVICE address (tensor.data_ptr()); the caller owns every buffer,
 *     including workspaces; no entry point allocates or synchronises.
 *   - `stream` is a cudaStream_t passed as void* (torch.cuda.current_stream().cuda_stream).
 *   - return value: 0 = ok, negative = FH_ERR_*; fh_last_error_string() gives the reason
 *     (thread-local).  There is no CPU fallback anywhere.
 *   - fp32 tensors use the reference's layouts; "chunked" tensors are [rows-of-8-channels]:
 *     element (t, c) of a [L, C] activation lives at ((c/8) * Lp + t) * 8 + c%8, i.e. the
 *     tcgen05 no-swizzle K-major core-matrix layout, so an implicit-GEMM tap is a row shift.
 */
#ifndef FLOWHIGH_B200_H
#define FLOWHIGH_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FH_OK 0
#define FH_ERR_BAD_SHAPE (-1)
#define FH_ERR_BAD_ALIGN (-2)
#define FH_ERR_UNSUPPORTED_CFG (-3)
#define FH_ERR_CUDA (-4)

int fh_version(void);
const char* fh_last_error_string(void);
/* number of kernel launches issued through this library by the calling process */
int64_t fh_launch_count(void);
/* Overflow / NaN guard of the 16-bit tensor path.  `status` is a DEVICE uint32 the caller owns and zeroes (NULL turns
 * the guard off); it is remembered per host thread and handed to every later launch from that thread of a kernel that
 * writes 16-bit operands (fh_tc_conv, fh_snake_aa_chunked[_h], fh_to_chunked_16, fh_rmsnorm_f32, fh_layernorm_f32,
 * fh_qknorm_rope_tiles, fh_attention_tc5, fh_cast_f32_16, fh_sum_cast_f32).  fp16 conversions
 * saturate at +-65504; a saturated, infinite or NaN operand ORs bit 0 into *status.  The host reads the word once per
 * generate() -- the device-side replacement of the reference's per-NFE `torch.isnan(x).any()` prints
 * (models/flow.py:256-267), without their four host syncs per NFE. */
int fh_set_status_word(uint32_t* status);
/* Debug aid: `word` is a uint32 in PINNED HOST memory (or NULL).  The tcgen05 kernels bound every mbarrier wait; a wait
 * that times out (a protocol bug) writes (wait code | block << 8 | warp << 24) there before trapping -- host memory
 * survives the resulting launch failure.  Thread-local like the status word. */
int fh_set_debug_word(uint32_t* word);

/* ---------------------------------------------------------------- resampler + peak normalise
 * replaces scipy.signal.resample_poly + `cond /= max|cond|`   flowhighsr.py:68-69
 *   y[b,m] = sum_i x[b,i] * h[(m + n_pre_remove)*down - n_pre_pad - i*up]
 * absmax[b] (may be NULL) receives max|y[b,:]| via atomicMax on the fp32 bit pattern; it must be
 * zeroed by the caller (fh_fill_f32). */
int fh_resample_poly_f32(const float* x, float* y, const float* h, uint32_t* absmax_bits,
                         int B, int T_in, int T_out, int ntaps, int up, int down,
                         int n_pre_pad, int n_pre_remove, void* stream);
/* y[b,:] = x[b,:] / absmax[b] * scale   (true division, like numpy / torch) */
int fh_scale_by_absmax_f32(const float* x, float* y, const uint32_t* absmax_bits, float scale,
                           int B, int T, void* stream);
int fh_absmax_f32(const float* x, uint32_t* absmax_bits, int B, int T, void* stream);
int fh_fill_u32(uint32_t* p, uint32_t v, int64_t n, void* stream);

/* ---------------------------------------------------------------- log-mel front end
 * replaces MelVoco.encode   models/melvoco.py:56-86  (+ librosa.filters.mel, modules.py:31-36)
 *   audio [B,T] fp32 -> mel [B,N,256] fp32,  N = T/480 (T >= 785)
 * window [2048] fp32; twiddle [1024] float2 = exp(-2 pi i k / 2048); sparse mel filterbank:
 * mel_start[256] (first bin), mel_len[256], mel_w [256*mel_stride] fp32.
 * precise != 0 runs the FFT in fp64 (fp32-parity path: the reference's own fp32 noise floor in
 * the empty bands is at the tolerance, SURVEY.md F11). */
int fh_stft_logmel_f32(const float* audio, float* mel, const float* window, const float* twiddle,
                       const int* mel_start, const int* mel_len, const float* mel_w, int mel_stride,
                       int B, int T, int N, int precise, void* stream);

/* ---------------------------------------------------------------- post-processing
 * replaces PostProcessing.post_processing   postprocessing.py:18-41
 * STFT: n_fft = win = 2048, hop 480, periodic Hann, center, ZERO pad; NT = 1 + T/480 frames.
 * No spectrogram reaches HBM: two real frames share one complex FFT.
 * fh_pp_src_energy: energy[B,1025] = sum_t |STFT(src)| (workspace of fh_pp_energy_ws_bytes(B, NT) bytes, 8-byte aligned);
 * fh_pp_fused: per frame STFT(pred), STFT(src) -> splice at cutoff[b] -> inverse FFT -> windowed frames [B,NT,2048]
 * for fh_pp_overlap_add_f32.  pred [B,Tp] and src [B,T] must span the same NT = 1 + T/480 frames. */
int fh_pp_energy_ws_bytes(int B, int NT);
int fh_pp_src_energy_f32(const float* src, float* energy, void* workspace, const float* window, const float* twiddle,
                         int B, int T, int NT, void* stream);
int fh_pp_fused_f32(const float* pred, const float* src, const int* cutoff, float* frames, const float* window,
                    const float* twiddle, int B, int Tp, int T, int NT, void* stream);
/* cutoff[b] = postprocessing.py:10-16 applied to energy[b,:] (cumsum, 0.99 threshold) */
int fh_pp_cutoff(const float* energy, int* cutoff, int B, float threshold, void* stream);
/* y[b,t] = OLA(frames)[t+1024] / OLA(window^2)[t+1024] for t < length (torch.istft semantics) */
int fh_pp_overlap_add_f32(const float* frames, float* y, const float* window, uint32_t* absmax_bits,
                          int B, int NT, int length, void* stream);

/* long-form stitch (engine capability, SURVEY.md 8e): K uniform chunks [K, clen] whose starts are
 * `step` apart (clen/2 <= step <= clen) -> out[total]; overlaps are linearly cross-faded. */
int fh_ola_crossfade_f32(const float* chunks, float* out, int K, int clen, int step, int64_t total,
                         void* stream);

/* ---------------------------------------------------------------- backbone, fp32 path
 * out[M,N] (ldc) = alpha * (A[M,K](lda) . W[N,K](ldw)^T + bias[N]) + beta_res * res[M,N](ldr)
 * replaces nn.Linear at flow.py:239,261; attend.py:176,189; transformer.py:100-103.
 * With alpha = dt, res = y this is the fused Euler / midpoint CFM update of
 * torchdiffeq.odeint (cfm_superresolution.py:243). */
int fh_sgemm_nt_f32(const float* A, int lda, const float* W, int ldw, const float* bias,
                    const float* res, int ldr, float beta_res, float alpha,
                    float* out, int ldc, int M, int N, int K, void* stream);
/* out[N] = act(W[N,K] . x[K] + b[N]);  act: 0 none, 1 SiLU  (flow.py:92-96, transformer.py:85) */
int fh_gemv_f32(const float* W, const float* x, const float* b, float* out, int N, int K, int act,
                void* stream);
/* out[2*half] = [sin(2 pi t w), cos(2 pi t w)]     pos_emb.py:22-26 */
int fh_sincos_embed_f32(const float* w, float t, float* out, int half, void* stream);
/* out = E + gelu(dwconv_k(E) + b) over time, E [B,N,C], w [C,k]   transformer.py:33-46, flow.py:240 */
int fh_dwconv_gelu_res_f32(const float* E, const float* w, const float* b, float* out,
                           int B, int N, int C, int k, void* stream);
/* ConvNeXt variant of the vector field (models/convnext.py:9-93, flow.py:124-139,247-253):
 * fh_dwconv_f32: depthwise Conv1d over time, odd k (7 in ConvNeXtBlock), zero padding, + bias; [B,N,C] fp32, out of place.
 * fh_layernorm_f32: F.layer_norm(x, eps) * w + b per row (AdaLayerNorm with w = scale(t), b = shift(t); b may be NULL);
 *   out_mode as in fh_rmsnorm_f32.
 * fh_gelu_f32: exact-erf GELU, fp32 row-major in and out. */
int fh_dwconv_f32(const float* x, const float* w, const float* b, float* out, int B, int N, int C, int k, void* stream);
int fh_layernorm_f32(const float* x, const float* w, const float* b, void* out, int out_mode, int64_t out_rows,
                     int M, int C, float eps, void* stream);
int fh_gelu_f32(const float* x, float* out, int M, int C, void* stream);

/* out = x / max(||x||,1e-12) * sqrt(C) * gamma + beta (beta may be NULL)   transformer.py:49-59,82-88
 * out_mode 0: fp32 row-major [M,C];  1: bf16 chunked [C/8][Mp][8] (row pitch out_rows);  2: fp16 chunked. */
int fh_rmsnorm_f32(const float* x, const float* gamma, const float* beta, void* out, int out_mode,
                   int64_t out_rows, int M, int C, void* stream);
/* qkv [B*N, 3*H*D] -> q,k,v [B,H,N,D]; q,k: l2norm * gamma[h,d] * sqrt(D), rotary (halves)
 * attend.py:144-151,179-184; pos_emb.py:45-60 */
int fh_qknorm_rope_f32(const float* qkv, const float* qg, const float* kg, const float* inv_freq,
                       float* q, float* k, float* v, int B, int N, int H, int D, void* stream);
/* out[B*N, H*D] fp32 row-major = softmax(scale q k^T) v   attend.py:123-137 (no mask) */
int fh_attention_f32(const float* q, const float* k, const float* v, float* out, int B, int H, int N, int D, float scale,
                     void* stream);
/* 16-bit tensor path of the two calls above (attention_tc5.cu): the logits reach +-640, so q (pre-multiplied by `scale`)
 * and k are hi + lo 16-bit pairs and the logits are S = qh.kh + ql.kh + qh.kl in fp32; v and P are 16-bit.
 * fh_qknorm_rope_tiles writes the operands as ready-made shared-memory images of the MMAs (no-swizzle K-major core
 * matrices), one contiguous tile per 128-query tile / 64-key block:
 *   q5 [B*H][ceil(N/128)][hi | lo][D/8][128][8]   k5 [B*H][ceil(N/64)][hi | lo][D/8][64][8]   v5 [B*H][ceil(N/64)][8][D][8]
 * (v5 = V^T, keys past N zero-filled); fh_attention_tc5_operand_elems(which = 0 / 1 / 2, ...) gives their sizes in 16-bit
 * elements.  fh_attention_tc5: S and P.V as tcgen05.mma into TMEM, softmax by one thread per query row, running output
 * in registers; out [B*N, H*D], out_mode / out_rows as in fh_rmsnorm_f32. */
int64_t fh_attention_tc5_operand_elems(int which, int B, int H, int N);
int fh_qknorm_rope_tiles(const float* qkv, const float* qg, const float* kg, const float* inv_freq,
                         void* q5, void* k5, void* v5, int B, int N, int H, int D, float scale, int fp16, void* stream);
int fh_attention_tc5(const void* q5, const void* k5, const void* v5, void* out, int out_mode, int64_t out_rows,
                     int B, int H, int N, int D, int fp16, void* stream);
/* g[M,inner] = gelu(u[M, inner + i]) * u[M, i]    transformer.py:92-95 */
int fh_geglu_f32(const float* u, float* g, int M, int inner, void* stream);
/* y = a*x + b*z  elementwise (prior: y0 = cond + sigma*eps, cfm_superresolution.py:222-230) */
int fh_axpby_f32(const float* x, const float* z, float a, float b, float* y, int64_t n, void* stream);

/* Adaptive-step solver helpers (use_torchode=True: torchode.Tsit5 / Dopri5 + IntegralController,
 * cfm_superresolution.py:259-276).
 *   fh_rk_lincomb_f32:      out = (base ? base : 0) + sum_{j<nk} coef_host[j] * k[j*kstride + i]   (nk <= 8; coef_host is a
 *                           HOST array, passed to the kernel by value) -- stage states, the solution and the error estimate
 *   fh_rk_scaled_sumsq_f32: out[b] = sum_i (e[b,i] / (atol + rtol * max(|y0[b,i]|, |y1[b,i]|)))^2  in fp64, one block per
 *                           problem instance (fixed summation order); y1 may be NULL.  The controller's error ratio is
 *                           sqrt(out[b] / n). */
int fh_rk_lincomb_f32(const float* base, const float* k, int64_t kstride, int nk, const float* coef_host, float* out,
                      int64_t n, void* stream);
int fh_rk_scaled_sumsq_f32(const float* e, const float* y0, const float* y1, float atol, float rtol, int B, int64_t n,
                           double* out, void* stream);

/* out[m, :] = row[:]  (null_cond broadcast for classifier-free guidance, flow.py:224-230) */
int fh_broadcast_row_f32(const float* row, float* out, int64_t M, int C, void* stream);
/* cutoff[b] = locate_cutoff_freq(exp(mel[b]))  cfm_superresolution.py:134-144,154-159 (percentile 0.9995) */
int fh_mel_cutoff_f32(const float* mel, int* cutoff, int B, int N, int F, float percentile, void* stream);
/* out[b,n,f] = f < cutoff[b] ? lo : hi   (mel_replace_ops, cfm_superresolution.py:146-152) */
int fh_mel_splice_f32(const float* lo, const float* hi, const int* cutoff, float* out, int B, int N, int F,
                      void* stream);

/* ---------------------------------------------------------------- vocoder, fp32 path  [B,C,L]
 * Generic tapped convolution: for phase p in [0,P):
 *   out[b, co, P*t + p] = alpha * ( bias[co] + sum_m sum_ci w[p][co][ci][m] * x[b, ci, t + off[p][m]] )
 *                         + beta_res * res[b,co,P*t+p] + (accumulate ? out : 0)
 * P = 1: Conv1d with dilation (bigvgan/models.py:27-43) ; P = stride: ConvTranspose1d polyphase
 * (models.py:140-146).  x is zero outside [0,L).  w [P][Cout][Cin][ntaps], off [P][ntaps]. */
int fh_conv1d_taps_f32(const float* x, const float* w, const float* bias, const int* off,
                       const float* res, float beta_res, float alpha, int accumulate, float* out,
                       int B, int Cin, int Cout, int L, int ntaps, int P, void* stream);
/* anti-aliased Snake / SnakeBeta: Activation1d.forward  alias_free_torch/act.py:23-28
 * x [B,C,L] -> y [B,C,L]; a = alpha (exp'd if logscale), inv_b = 1/(beta+1e-9) per channel. */
int fh_snake_aa_f32(const float* x, float* y, const float* a, const float* inv_b, const float* filt,
                    int B, int C, int L, void* stream);
/* y[b,t] = tanh(bias + sum_ci sum_j w[ci,j] x[b,ci,t+j-3])   models.py:190-192 */
int fh_convpost_tanh_f32(const float* x, const float* w, float bias, float* y, int B, int C, int L,
                         void* stream);
/* [B,R,C] -> [B,C,R]  (the `b n d -> b d n` rearrange at melvoco.py:115) */
int fh_transpose_f32(const float* src, float* dst, int B, int R, int C, void* stream);
/* elementwise fp32 -> bf16 / fp16 (whole chunked buffers, halos included) */
int fh_cast_f32_16(const float* src, void* dst, int64_t n, int fp16, void* stream);
/* precision "fp16x2" (activation operands kept as hi + lo fp16 pairs against duplicated weights: ~22-bit activations at
 * twice the MMAs; meets the LSD <= 0.05 dB bar on high-dynamic-range clips where 11-bit operands leave 0.08 dB):
 * chunked fp32 [B][nchunk][rows][8] -> chunked 16-bit [B][2 nchunk][rows][8] = [round(x) | round(x - hi)], halos included. */
int fh_cast_f32_16_split(const float* src, void* dst, int64_t chunk_elems, int nchunk, int64_t src_batch,
                         int64_t dst_batch, int B, int fp16, void* stream);
/* out = a + b + c + d (b, c, d optional): the mean over the AMP branches of a BigVGAN stage (bigvgan/models.py:181-187, each
 * branch pre-scaled by 1/num_kernels), as fp32 (out32) and / or 16-bit (out16); same flat geometry for all buffers. */
int fh_sum_cast_f32(const float* a, const float* b, const float* c, const float* d, float* out32, void* out16,
                    int64_t n, int fp16, void* stream);

/* ---------------------------------------------------------------- tensor-core path (tcgen05)
 * Implicit-GEMM tapped convolution on chunked 16-bit operands (bf16 or fp16) -> fp32 in TMEM.
 *   A: activations, chunked 16-bit [B][Cin/8][Lp_a][8] with >= halo zero rows each side of [0,L)
 *   W: packed by fh_tc_pack_* (host side, flowhigh_b200/packing.py) into the smem image
 *   out(t, n) at out + b*out_batch + (n/8)*out_chunk + (P*t+p)*out_row + n%8, fp32 or 16-bit
 * A Linear layer is the k = 1 case with L = number of tokens. */
typedef struct {
  const void* a;          /* chunked 16-bit activations */
  int64_t a_batch;        /* elements between batches */
  int64_t a_chunk;        /* elements between 8-channel chunks (= Lp_a * 8) */
  int a_row0;             /* row index of t = 0 inside a chunk (left halo) */
  const void* w;          /* packed weights */
  const float* bias;      /* [Cout] or NULL */
  const void* res;        /* residual, addressed like out (res_is_16 selects the width) or NULL */
  void* out;
  int64_t out_batch, out_chunk, out_row;
  int64_t res_batch, res_chunk, res_row;
  int out_is_16, res_is_16; /* output / residual stored as 16-bit (type given by `fp16`) instead of fp32 */
  float alpha, beta_res;
  int accumulate;         /* out += ... (fp32 out only) */
  int geglu;              /* epilogue pairs columns (2i, 2i+1) -> gelu(col 2i+1) * col 2i */
  int B, L, Cin, Cout;    /* Cin and Cout multiples of 8 (whole 8-channel chunks) */
  int ntaps, P;           /* taps per phase, phases (output stride) */
  const int* tap_off;     /* HOST pointer [P][ntaps] row offsets */
  int bn;                 /* N tile, multiple of 16, <= 256 */
  int fp16;               /* 16-bit operand format: 0 = bfloat16, 1 = IEEE half (same rate, 3 more mantissa bits) */
  int act;                /* 0 none, 1 exact-erf GELU on (acc + bias) * alpha, before the residual (convnext.py:56-57) */
  const float* acc_src;   /* accumulate != 0: rows to add, fp32 with the output geometry; NULL = the output itself.
                           * Lets the last AMP branch of a stage (bigvgan/models.py:181-187, xs / num_kernels) write the
                           * mean directly as the 16-bit operand of the next upsampler (out_is_16 = 1). */
  int two_cta;            /* CTA-pair kernel (tcgen05 cta_group::2, M = 256): `w` must be packed per CTA rank
                           * ([p][nt][ci-pair][rank][tap][2][bn/2][8], packing.pack_tc(two_cta=True)) */
} fh_tc_conv_args;
int fh_tc_conv(const fh_tc_conv_args* args, void* stream);
/* bytes of the packed weight image for given shape (host helper, no GPU work) */
int64_t fh_tc_packed_weight_bytes(int Cin, int Cout, int ntaps, int P, int bn);

/* fp32 [B,C,L] planar or [M,C] row-major -> chunked 16-bit (bf16, or half when fp16 != 0); src strides in elements */
int fh_to_chunked_16(const float* src, int64_t src_batch, int64_t src_c, int64_t src_t,
                     void* dst, int64_t dst_batch, int64_t dst_chunk, int dst_row0,
                     int B, int C, int L, int fp16, void* stream);
/* fh_to_chunked_16 with the hi + lo split: channels [0, C) = round(x), [Cpad, Cpad + C) = round(x - hi), Cpad = 8 ceil(C / 8) */
int fh_to_chunked_16_split(const float* src, int64_t src_batch, int64_t src_c, int64_t src_t,
                           void* dst, int64_t dst_batch, int64_t dst_chunk, int dst_row0,
                           int B, int C, int L, int fp16, void* stream);
/* chunked anti-aliased snake: x chunked fp32 -> y chunked (same geometry); out_kind 0 fp32, 1 bf16, 2 fp16 */
int fh_snake_aa_chunked(const float* x, void* y, const float* a, const float* inv_b, const float* filt,
                        int64_t batch_stride, int64_t chunk_stride, int row0, int B, int C, int L,
                        int out_kind, void* stream);
/* same op with an fp16 chunked input (written by fh_tc_conv with out_is_16) and fp16 output: Activation1d.forward
 * (alias_free_torch/act.py:23-28) between the two convolutions of an AMPBlock1 unit (bigvgan/models.py:63-72) */
int fh_snake_aa_chunked_h(const void* x16, void* y, const float* a, const float* inv_b, const float* filt,
                          int64_t batch_stride, int64_t chunk_stride, int row0, int B, int C, int L, void* stream);
/* Activation1d.forward with fp32 rows in and fp16 hi + lo rows out (precision "fp16x2"): y has 2 C channels per batch
 * ([hi chunks | lo chunks], batch stride y_batch_stride); the input is split hi + lo inside the kernel as well. */
int fh_snake_aa_chunked_split(const float* x, void* y, const float* a, const float* inv_b, const float* filt,
                              int64_t x_batch_stride, int64_t y_batch_stride, int64_t chunk_stride, int row0,
                              int B, int C, int L, void* stream);
int fh_convpost_tanh_chunked(const float* x, int64_t batch_stride, int64_t chunk_stride, int row0,
                             const float* w, float bias, float* y, int B, int C, int L, void* stream);

/* The tail of BigVGAN.forward in one kernel (bigvgan/models.py:189-192): activation_post (Activation1d, fp32) ->
 * conv_post (C -> 1, k = 7) -> tanh; x chunked fp32, y [B, L].  The activated tensor stays in shared memory. */
int fh_snakepost_convpost_tanh(const float* x, int64_t batch_stride, int64_t chunk_stride, int row0,
                               const float* a, const float* inv_b, const float* filt, const float* w, float bias,
                               float* y, int B, int C, int L, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FLOWHIGH_B200_H */
