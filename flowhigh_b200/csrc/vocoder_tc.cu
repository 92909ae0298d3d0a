// Memory-bound vocoder kernels of the tensor-core path, on the chunked [C/8][Lp][8] layout that
// fh_tc_conv consumes: fused anti-aliased Snake/SnakeBeta (alias_free_torch/act.py:23-28,
// resample.py:25-33, filter.py:86-94, activations.py:48-59,107-119) and conv_post + tanh
// (bigvgan/models.py:189-192).  The residual stream stays fp32; only MMA operands are 16-bit.
#include "common.cuh"
#include "snake_worker.cuh"
#include "snake_mma.cuh"

namespace {

// ------------------------------------------------------------------------------ anti-aliased snake
// The kernel body lives in snake_worker.cuh: persistent CTAs of one 128-thread worker each, 17 outputs per thread.
constexpr int PR = 17;

template <int OUT_KIND, bool BULK_OUT>
__global__ void __launch_bounds__(128, 4) snake_aa_chunked_tma_kernel(const __grid_constant__ fh::SnakeParams S) {
  extern __shared__ __align__(128) unsigned char snake_smem[];
  fh::snake_worker<OUT_KIND, BULK_OUT, PR>(S, snake_smem, threadIdx.x, blockIdx.x, gridDim.x, 0);
}

// fp16 output mode: both FIR filters as Toeplitz MMAs (snake_mma.cuh).  SPLIT_X: hi/lo split of the input.
template <bool SPLIT_X, int NB, int MINB, bool IN16, bool SPLIT_OUT>
__global__ void __launch_bounds__(128, MINB) snake_aa_mma_kernel(const __grid_constant__ fh::SnakeParams S) {
  extern __shared__ __align__(128) unsigned char snake_smem[];
  fh::snake_mma_cta<SPLIT_X, NB, IN16, SPLIT_OUT>(S, snake_smem, threadIdx.x, blockIdx.x, gridDim.x);
}

template <bool SPLIT_X, int NB, int MINB, bool IN16 = false, bool SPLIT_OUT = false>
void launch_snake_mma(fh::SnakeParams sp, int B, int C, int L, int sms, cudaStream_t stream) {
  using G = fh::SnakeMmaGeom<NB>;
  static int smem_set[64] = {0};
  fh::ensure_dyn_smem(snake_aa_mma_kernel<SPLIT_X, NB, MINB, IN16, SPLIT_OUT>, G::smem_bytes(IN16, SPLIT_OUT), smem_set);
  sp.ntile = (L + G::kRows - 1) / G::kRows;
  const long long total = (long long)sp.ntile * (C / 8) * B;
  sp.total = (int)total;
  const int grid = (int)(total < (long long)sms * MINB ? total : (long long)sms * MINB);
  snake_aa_mma_kernel<SPLIT_X, NB, MINB, IN16, SPLIT_OUT><<<grid, 128, G::smem_bytes(IN16, SPLIT_OUT), stream>>>(sp);
}

// conv_post (C -> 1, k = 7, zero padding) + tanh on the chunked fp32 layout (bigvgan/models.py:190-192).  HBM-bound:
// 4 (C + 1) bytes per output sample.  A CTA stages the (256 + 6)-row window of every 8-channel chunk in shared memory with
// coalesced 16-byte loads (each input row is read from HBM once; the first version re-read it 7 times through L1 and
// reached 1.6 TB/s), then one thread per output sample walks the 7 taps x C channels from shared memory; the 7 C weights
// are broadcast reads of a shared table.
constexpr int kCpT = 256;  // outputs per CTA
__global__ void __launch_bounds__(kCpT) convpost_tanh_chunked_kernel(const float* __restrict__ x, long long batch_stride,
                                                                     long long chunk_stride, int row0,
                                                                     const float* __restrict__ w, float bias,
                                                                     float* __restrict__ y, int C, int L) {
  extern __shared__ __align__(16) float cp_smem[];
  const int nchunk = C >> 3;
  float* s_w = cp_smem;                              // [C][7] padded to a multiple of 4 floats
  float* tile = cp_smem + ((C * 7 + 3) & ~3);        // [nchunk][kCpT + 6][8]
  const int b = blockIdx.y, t0 = blockIdx.x * kCpT;
  for (int i = threadIdx.x; i < C * 7; i += kCpT) s_w[i] = __ldg(w + i);
  const float* xb = x + (long long)b * batch_stride;
  const int rows = kCpT + 6;
  for (int i = threadIdx.x; i < nchunk * rows * 2; i += kCpT) {
    const int h = i & 1, r = (i >> 1) % rows, ch = (i >> 1) / rows;
    const int t = t0 - 3 + r;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (t >= 0 && t < L) v = __ldg(reinterpret_cast<const float4*>(xb + (long long)ch * chunk_stride + (long long)(row0 + t) * 8) + h);
    reinterpret_cast<float4*>(tile)[i] = v;  // same (chunk, row, half) order as the flat index
  }
  __syncthreads();
  const int t = t0 + threadIdx.x;
  if (t >= L) return;
  float acc = bias;
  for (int ch = 0; ch < nchunk; ++ch) {
    const float* tp = tile + ((size_t)ch * rows + threadIdx.x) * 8;
    const float* wp = s_w + ch * 56;
#pragma unroll
    for (int j = 0; j < 7; ++j) {
      const float4 v0 = *reinterpret_cast<const float4*>(tp + j * 8), v1 = *reinterpret_cast<const float4*>(tp + j * 8 + 4);
      acc = fmaf(wp[j], v0.x, acc);
      acc = fmaf(wp[7 + j], v0.y, acc);
      acc = fmaf(wp[14 + j], v0.z, acc);
      acc = fmaf(wp[21 + j], v0.w, acc);
      acc = fmaf(wp[28 + j], v1.x, acc);
      acc = fmaf(wp[35 + j], v1.y, acc);
      acc = fmaf(wp[42 + j], v1.z, acc);
      acc = fmaf(wp[49 + j], v1.w, acc);
    }
  }
  y[(long long)b * L + t] = tanhf(acc);
}

// ------------------------------------------------------------------------------ activation_post + conv_post + tanh
// The tail of BigVGAN.forward in ONE kernel (bigvgan/models.py:189-192): Activation1d(SnakeBeta) on the last stage's
// fp32 rows, Conv1d(C -> 1, k = 7, zero padding) and tanh.  The activated tensor (4 C bytes per sample written and read
// back by the two-kernel form) never leaves shared memory: HBM traffic is 4 C bytes in + 4 bytes out per sample.
// A CTA of 128 threads owns 512 output samples.  Per 8-channel chunk it stages the (544 + 10)-row fp32 window
// (replicate-clamped rows: the snake's own padding), runs the register-blocked scalar snake of snake_worker.cuh (one
// thread = 2 channels x 17 rows, all taps packed FFMA2) and writes the activated rows, zeroed outside [0, L) (the conv's
// zero padding), into a shared tile.  Then one thread = 4 consecutive outputs: it walks its 10 tile rows ONCE with the 56
// weights of the chunk in registers (the two-kernel form re-read every row 7 times from L1).  Tile rows carry a 16-byte
// pad every 4 rows so that the 128-byte row stride between neighbouring threads does not land on one bank group.
constexpr int kSpR = 17, kSpRows = 32 * kSpR, kSpT = 512, kSpXRows = kSpRows + 10;
constexpr int kSpTileBytes = kSpRows * 32 + (kSpRows / 4) * 16;  // one chunk's activated rows, padded
__device__ __forceinline__ int sp_row_off(int a) { return a * 32 + (a >> 2) * 16; }

__global__ void __launch_bounds__(128) snakepost_convpost_tanh_kernel(const float* __restrict__ x, long long batch_stride,
                                                                      long long chunk_stride, int row0,
                                                                      const float* __restrict__ sn_a,
                                                                      const float* __restrict__ sn_inv_b,
                                                                      const float* __restrict__ filt,
                                                                      const float* __restrict__ w, float bias,
                                                                      float* __restrict__ y, int C, int L) {
  extern __shared__ __align__(16) unsigned char sp_smem[];
  const int nchunk = C >> 3;
  float* s_w = reinterpret_cast<float*>(sp_smem);                                    // [C][7]
  float* xs = reinterpret_cast<float*>(sp_smem + (((C * 7 + 3) & ~3) * 4));          // [kSpXRows][8]
  unsigned char* tile = reinterpret_cast<unsigned char*>(xs) + kSpXRows * 32;        // [nchunk][kSpTileBytes]
  const int tid = threadIdx.x, b = blockIdx.y, t0 = blockIdx.x * kSpT;
  const int tA0 = t0 - 3;  // time of tile row 0
  for (int i = tid; i < C * 7; i += 128) s_w[i] = __ldg(w + i);
  float2 fu[12], fd[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) {
    const float fk = __ldg(filt + k);
    fu[k] = make_float2(2.0f * fk, 2.0f * fk);
    fd[k] = make_float2(fk, fk);
  }
  const int e2 = tid & 3, g = tid >> 2;
  const float* xb = x + (long long)b * batch_stride;
  for (int ch = 0; ch < nchunk; ++ch) {
    __syncthreads();  // the previous chunk's window has been consumed
    for (int i = tid; i < kSpXRows * 2; i += 128) {
      const int r = i >> 1, h = i & 1;
      const int t = min(max(tA0 - 5 + r, 0), L - 1);  // replicate clamp (resample.py:27, filter.py:88)
      reinterpret_cast<float4*>(xs)[i] = __ldg(reinterpret_cast<const float4*>(xb + (long long)ch * chunk_stride + (long long)(row0 + t) * 8) + h);
    }
    __syncthreads();
    const int q0 = tA0 + g * kSpR;  // time of this thread's first row
    unsigned char* tp = tile + (size_t)ch * kSpTileBytes;
    if (q0 < L && q0 + kSpR > 0) {
      const int c0 = ch * 8 + 2 * e2;
      const float2 al2 = make_float2(2.0f * __ldg(sn_a + c0), 2.0f * __ldg(sn_a + c0 + 1));
      const float2 hib = make_float2(0.5f * __ldg(sn_inv_b + c0), 0.5f * __ldg(sn_inv_b + c0 + 1));
      const float2 nhib = make_float2(-hib.x, -hib.y);
      float2 xv[kSpR + 10];
      const float* xp = xs + g * (kSpR * 8) + 2 * e2;
#pragma unroll
      for (int j = 0; j < kSpR + 10; ++j) xv[j] = *reinterpret_cast<const float2*>(xp + j * 8);
      float2 sv[2 * kSpR + 10];
#pragma unroll
      for (int i = 0; i < 2 * kSpR + 10; ++i) {
        const int qq = (i - 5) >> 1;
        float2 u = make_float2(0.f, 0.f);
        if ((i & 1) == 0) {
#pragma unroll
          for (int d = -2; d <= 3; ++d) u = fh::sw_ffma2(xv[qq + d + 5], fu[6 - 2 * d], u);
        } else {
#pragma unroll
          for (int d = -3; d <= 2; ++d) u = fh::sw_ffma2(xv[qq + d + 5], fu[5 - 2 * d], u);
        }
        const float2 z = fh::sw_fmul2(u, al2);
        const float2 cz = make_float2(__cosf(z.x), __cosf(z.y));
        sv[i] = fh::sw_ffma2(cz, nhib, u);
      }
      // replicate clamp of the 2x-rate signal: local index i holds s'[2 q0 - 5 + i]; s'[m < 0] = s'[0], s'[m > 2L-1] = s'[2L-1]
      const int i_lo = 5 - 2 * q0, i_hi = 2 * (L - q0) + 4;
      if (i_lo > 0 || i_hi < 2 * kSpR + 9) {
        float2 lo_v = sv[0], hi_v = sv[2 * kSpR + 9];
#pragma unroll
        for (int i = 0; i < 2 * kSpR + 10; ++i) {
          if (i == i_lo) lo_v = sv[i];
          if (i == i_hi) hi_v = sv[i];
        }
#pragma unroll
        for (int i = 0; i < 2 * kSpR + 10; ++i) {
          if (i < i_lo) sv[i] = lo_v;
          if (i > i_hi) sv[i] = hi_v;
        }
      }
#pragma unroll
      for (int j = 0; j < kSpR; ++j) {
        float2 acc = hib;
#pragma unroll
        for (int k = 0; k < 12; ++k) acc = fh::sw_ffma2(fd[k], sv[2 * j + k], acc);
        const int t = q0 + j;
        if (t < 0 || t >= L) acc = make_float2(0.f, 0.f);  // conv_post zero padding
        *reinterpret_cast<float2*>(tp + sp_row_off(g * kSpR + j) + 8 * e2) = acc;
      }
    } else {
#pragma unroll
      for (int j = 0; j < kSpR; ++j) *reinterpret_cast<float2*>(tp + sp_row_off(g * kSpR + j) + 8 * e2) = make_float2(0.f, 0.f);
    }
  }
  __syncthreads();
  // ---- conv_post + tanh: outputs t0 + 4 tid + {0..3} from tile rows 4 tid .. 4 tid + 9
  const int o = 4 * tid;
  if (t0 + o >= L) return;
  float acc[4] = {bias, bias, bias, bias};
  for (int ch = 0; ch < nchunk; ++ch) {
    float wr[56];
#pragma unroll
    for (int i = 0; i < 56; ++i) wr[i] = s_w[ch * 56 + i];  // [c][7]
    const unsigned char* tp = tile + (size_t)ch * kSpTileBytes;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      const float4 v0 = *reinterpret_cast<const float4*>(tp + sp_row_off(o + r));
      const float4 v1 = *reinterpret_cast<const float4*>(tp + sp_row_off(o + r) + 16);
      const float v[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
#pragma unroll
      for (int oo = 0; oo < 4; ++oo) {
        const int j = r - oo;  // tap
        if (j >= 0 && j < 7) {
#pragma unroll
          for (int c = 0; c < 8; ++c) acc[oo] = fmaf(wr[c * 7 + j], v[c], acc[oo]);
        }
      }
    }
  }
  float* yp = y + (long long)b * L + t0 + o;
  if (t0 + o + 3 < L && ((((long long)b * L + t0 + o) & 3) == 0)) {
    *reinterpret_cast<float4*>(yp) = make_float4(tanhf(acc[0]), tanhf(acc[1]), tanhf(acc[2]), tanhf(acc[3]));
  } else {
#pragma unroll
    for (int oo = 0; oo < 4; ++oo)
      if (t0 + o + oo < L) yp[oo] = tanhf(acc[oo]);
  }
}

}  // namespace

extern "C" __attribute__((visibility("default"))) int fh_snake_aa_chunked(
    const float* x, void* y, const float* a, const float* inv_b, const float* filt, int64_t batch_stride,
    int64_t chunk_stride, int row0, int B, int C, int L, int out_kind, void* stream) {
  FH_REQUIRE(B > 0 && C > 0 && (C % 8) == 0 && L > 0, FH_ERR_BAD_SHAPE, "fh_snake_aa_chunked: C must be a multiple of 8");
  FH_REQUIRE(out_kind >= 0 && out_kind <= 2, FH_ERR_BAD_SHAPE, "fh_snake_aa_chunked: out_kind must be 0 (fp32), 1 (bf16), 2 (fp16)");
  FH_REQUIRE(((uintptr_t)x % 16) == 0 && (batch_stride % 8) == 0 && (chunk_stride % 8) == 0, FH_ERR_BAD_ALIGN,
             "fh_snake_aa_chunked: x must be 16-byte aligned and strides multiples of 8");
  // fp16 output: the Toeplitz-MMA kernel.  Its hi/lo split of the input (as in fh_snake_aa_chunked_split) buys < 0.3 dB
  // of end-to-end SNR for 15 % more kernel time; neither it nor the hi/lo split of the filter taps was ever the default,
  // and both were removed.  A left halo shorter than the MMA kernel's window falls back to the scalar kernel.
  const bool use_mma = out_kind == 2 && row0 >= fh::SnakeMmaGeom<8>::kHalo;
  constexpr int kTileRows = fh::SnakeGeom<PR>::kRows;
  const int ntile = (L + kTileRows - 1) / kTileRows;
  const long long total = (long long)ntile * (C / 8) * B;
  FH_REQUIRE(total <= 2147483647LL && row0 >= 5, FH_ERR_BAD_SHAPE, "fh_snake_aa_chunked: needs a left halo of >= 5 rows");
  const int sms = fh::dev_sms();
  constexpr int kPerSm = 4;  // persistent CTAs per SM of the scalar kernel (4 fill the SM)
  const int grid = (int)(total < (long long)sms * kPerSm ? total : (long long)sms * kPerSm);
  fh::SnakeParams sp;
  sp.x = x, sp.y = y, sp.a = a, sp.inv_b = inv_b, sp.filt = filt;
  sp.batch_stride = batch_stride, sp.chunk_stride = chunk_stride, sp.y_batch_stride = batch_stride, sp.lo_offset = 0;
  sp.row0 = row0, sp.nchunk = C / 8, sp.L = L, sp.ntile = ntile, sp.total = (int)total, sp.fp16 = out_kind == 2;
  sp.status = fh::status_word();
  if (use_mma) {
    FH_REQUIRE((long long)((L + 511) / 512) * (C / 8) * B <= 2147483647LL, FH_ERR_BAD_SHAPE, "fh_snake_aa_chunked: too many work items");
    // 8 blocks of 8 outputs per half-segment, 4 CTAs per SM (4-block segments at 6 CTAs per SM: 142 vs 118 ms per step)
    // 128-output segments at 2 CTAs per SM against 64-output segments at 4: 6 % less halo work (MUFU, MMAs)
    // and half the warps -- 87.0 vs 93.3 ms per step.  A single input window per CTA (3 CTAs per SM) measured no better
    // and was removed.
    launch_snake_mma<false, 16, 2>(sp, B, C, L, sms, (cudaStream_t)stream);
    return fh::check_launch("fh_snake_aa_chunked");
  }
  // scalar kernel; 16-bit outputs go to HBM through a bulk store of the output tile
  constexpr int kSmem = fh::SnakeGeom<PR>::kSmemBytes;
#define FH_SNAKE_LAUNCH(KIND, BULK) snake_aa_chunked_tma_kernel<KIND, BULK><<<grid, 128, kSmem, (cudaStream_t)stream>>>(sp)
  if (out_kind == 0) FH_SNAKE_LAUNCH(0, false);
  else if (out_kind == 1) FH_SNAKE_LAUNCH(1, true);
  else FH_SNAKE_LAUNCH(2, true);
#undef FH_SNAKE_LAUNCH
  return fh::check_launch("fh_snake_aa_chunked");
}

// fp32 in -> fp16 hi + lo out (precision "fp16x2"): y holds 2 C channels per batch, [hi chunks | lo chunks]; the input is
// split hi + lo as well (two MMAs per up-filter block), so the activation keeps ~22 bits into the following convolution,
// whose weights are duplicated over the doubled input channels.
extern "C" __attribute__((visibility("default"))) int fh_snake_aa_chunked_split(
    const float* x, void* y, const float* a, const float* inv_b, const float* filt, int64_t x_batch_stride,
    int64_t y_batch_stride, int64_t chunk_stride, int row0, int B, int C, int L, void* stream) {
  FH_REQUIRE(B > 0 && C > 0 && (C % 8) == 0 && L > 0, FH_ERR_BAD_SHAPE, "fh_snake_aa_chunked_split: C must be a multiple of 8");
  FH_REQUIRE(((uintptr_t)x % 16) == 0 && ((uintptr_t)y % 16) == 0 && (x_batch_stride % 8) == 0 && (y_batch_stride % 8) == 0 &&
                 (chunk_stride % 8) == 0,
             FH_ERR_BAD_ALIGN, "fh_snake_aa_chunked_split: buffers must be 16-byte aligned and strides multiples of 8");
  FH_REQUIRE(row0 >= fh::SnakeMmaGeom<8>::kHalo, FH_ERR_BAD_SHAPE, "fh_snake_aa_chunked_split: needs a left halo of >= 8 rows");
  FH_REQUIRE((long long)((L + 511) / 512) * (C / 8) * B <= 2147483647LL, FH_ERR_BAD_SHAPE,
             "fh_snake_aa_chunked_split: too many work items");
  fh::SnakeParams sp;
  sp.x = x, sp.y = y, sp.a = a, sp.inv_b = inv_b, sp.filt = filt;
  sp.batch_stride = x_batch_stride, sp.chunk_stride = chunk_stride, sp.y_batch_stride = y_batch_stride;
  sp.lo_offset = (int64_t)(C / 8) * chunk_stride;
  sp.row0 = row0, sp.nchunk = C / 8, sp.L = L, sp.ntile = 0, sp.total = 0, sp.fp16 = 1;
  sp.status = fh::status_word();
  launch_snake_mma<true, 8, 3, false, true>(sp, B, C, L, fh::dev_sms(), (cudaStream_t)stream);
  return fh::check_launch("fh_snake_aa_chunked_split");
}

// fp16 in -> fp16 out on the same chunked geometry: the input was written by the 16-bit epilogue of the first
// convolution of an AMP unit (fh_tc_conv with out_is_16), so the fp32 round trip of that tensor disappears.
extern "C" __attribute__((visibility("default"))) int fh_snake_aa_chunked_h(
    const void* x16, void* y, const float* a, const float* inv_b, const float* filt, int64_t batch_stride,
    int64_t chunk_stride, int row0, int B, int C, int L, void* stream) {
  FH_REQUIRE(B > 0 && C > 0 && (C % 8) == 0 && L > 0, FH_ERR_BAD_SHAPE, "fh_snake_aa_chunked_h: C must be a multiple of 8");
  FH_REQUIRE(((uintptr_t)x16 % 16) == 0 && ((uintptr_t)y % 16) == 0 && (batch_stride % 8) == 0 && (chunk_stride % 8) == 0,
             FH_ERR_BAD_ALIGN, "fh_snake_aa_chunked_h: buffers must be 16-byte aligned and strides multiples of 8");
  FH_REQUIRE(row0 >= fh::SnakeMmaGeom<8>::kHalo, FH_ERR_BAD_SHAPE, "fh_snake_aa_chunked_h: needs a left halo of >= 8 rows");
  FH_REQUIRE((long long)((L + 511) / 512) * (C / 8) * B <= 2147483647LL, FH_ERR_BAD_SHAPE,
             "fh_snake_aa_chunked_h: too many work items");
  const int sms = fh::dev_sms();
  fh::SnakeParams sp;
  sp.x = (const float*)x16, sp.y = y, sp.a = a, sp.inv_b = inv_b, sp.filt = filt;
  sp.batch_stride = batch_stride, sp.chunk_stride = chunk_stride, sp.y_batch_stride = batch_stride, sp.lo_offset = 0;
  sp.row0 = row0, sp.nchunk = C / 8, sp.L = L, sp.ntile = 0, sp.total = 0, sp.fp16 = 1;
  sp.status = fh::status_word();
  // 128-output segments at 3 CTAs per SM.  Five CTAs per SM fit with 64-output segments and the half-size fp16 windows
  // (33 KB, 90 registers) -- measured SLOWER (101.5 vs 98.3 ms per step, like every other occupancy increase of this
  // kernel: it is not latency-bound); a single input window per CTA (4 CTAs per SM) measured no better.  Both were removed.
  launch_snake_mma<false, 16, 3, true>(sp, B, C, L, sms, (cudaStream_t)stream);
  return fh::check_launch("fh_snake_aa_chunked_h");
}

extern "C" __attribute__((visibility("default"))) int fh_convpost_tanh_chunked(
    const float* x, int64_t batch_stride, int64_t chunk_stride, int row0, const float* w, float bias, float* y, int B,
    int C, int L, void* stream) {
  FH_REQUIRE(B > 0 && C > 0 && (C % 8) == 0 && L > 0 && B <= 65535, FH_ERR_BAD_SHAPE,
             "fh_convpost_tanh_chunked: bad shape");
  const int smem = (((C * 7 + 3) & ~3) + (C / 8) * (kCpT + 6) * 8) * (int)sizeof(float);
  FH_REQUIRE(smem <= 200 * 1024, FH_ERR_UNSUPPORTED_CFG, "fh_convpost_tanh_chunked: C=%d too wide for the shared-memory tile", C);
  static int smem_set[64] = {0};
  if (smem > 48 * 1024) fh::ensure_dyn_smem(convpost_tanh_chunked_kernel, smem, smem_set);
  convpost_tanh_chunked_kernel<<<dim3((L + kCpT - 1) / kCpT, B), kCpT, smem, (cudaStream_t)stream>>>(x, batch_stride, chunk_stride,
                                                                                               row0, w, bias, y, C, L);
  return fh::check_launch("fh_convpost_tanh_chunked");
}

// activation_post + conv_post + tanh fused (bigvgan/models.py:189-192): x chunked fp32 [B][C/8][Lp][8] -> y [B, L]
extern "C" __attribute__((visibility("default"))) int fh_snakepost_convpost_tanh(
    const float* x, int64_t batch_stride, int64_t chunk_stride, int row0, const float* a, const float* inv_b,
    const float* filt, const float* w, float bias, float* y, int B, int C, int L, void* stream) {
  FH_REQUIRE(B > 0 && C > 0 && (C % 8) == 0 && C <= 64 && L > 0 && B <= 65535, FH_ERR_BAD_SHAPE,
             "fh_snakepost_convpost_tanh: C must be a multiple of 8, <= 64");
  FH_REQUIRE(((uintptr_t)x % 16) == 0 && (batch_stride % 8) == 0 && (chunk_stride % 8) == 0, FH_ERR_BAD_ALIGN,
             "fh_snakepost_convpost_tanh: alignment");
  const int smem = ((C * 7 + 3) & ~3) * 4 + kSpXRows * 32 + (C / 8) * kSpTileBytes;
  static int smem_set[64] = {0};
  cudaError_t e = fh::ensure_dyn_smem(snakepost_convpost_tanh_kernel, smem, smem_set);
  FH_REQUIRE(e == cudaSuccess, FH_ERR_CUDA, "fh_snakepost_convpost_tanh: cannot opt in to %d bytes of smem", smem);
  snakepost_convpost_tanh_kernel<<<dim3((L + kSpT - 1) / kSpT, B), 128, smem, (cudaStream_t)stream>>>(
      x, batch_stride, chunk_stride, row0, a, inv_b, filt, w, bias, y, C, L);
  return fh::check_launch("fh_snakepost_convpost_tanh");
}
