// fp32 CUDA-core kernels of the FLowHigh vector-field network (models/flow.py:180-274,
// models/transformer.py, models/attend.py, models/pos_emb.py).  This is the fp32 parity path
// and the home of the memory-bound pieces (norms, rotary, depthwise conv, GEGLU) that the
// tensor-core path reuses with chunked-bf16 outputs.
#include "common.cuh"

namespace {

// ------------------------------------------------------------------------------ SGEMM (NT)
// out = alpha * (A . W^T + bias) + beta_res * res.   64x64 tile, BK 16, 256 threads, 4x4 micro-tile.
constexpr int GT = 64, GK = 16;
__global__ void __launch_bounds__(256) sgemm_nt_kernel(const float* __restrict__ A, int lda, const float* __restrict__ W,
                                                       int ldw, const float* __restrict__ bias,
                                                       const float* __restrict__ res, int ldr, float beta_res,
                                                       float alpha, float* __restrict__ out, int ldc, int M, int N,
                                                       int K) {
  __shared__ float As[GK][GT + 4];
  __shared__ float Ws[GK][GT + 4];
  const int m0 = blockIdx.y * GT, n0 = blockIdx.x * GT;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;  // tx -> n, ty -> m
  const int lr = threadIdx.x >> 2, lc = (threadIdx.x & 3) * 4;  // loader: row 0..63, k 0,4,8,12
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += GK) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int k = k0 + lc + i;
      const int m = m0 + lr, n = n0 + lr;
      As[lc + i][lr] = (m < M && k < K) ? __ldg(A + (size_t)m * lda + k) : 0.f;
      Ws[lc + i][lr] = (n < N && k < K) ? __ldg(W + (size_t)n * ldw + k) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < GK; ++k) {
      float a[4], w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[k][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) w[j] = Ws[k][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= N) continue;
      float v = acc[i][j];
      if (bias) v += bias[n];
      v *= alpha;
      if (res) v = fmaf(beta_res, res[(size_t)m * ldr + n], v);
      out[(size_t)m * ldc + n] = v;
    }
  }
}

// ------------------------------------------------------------------------------ GEMV / time MLP
__global__ void gemv_kernel(const float* __restrict__ W, const float* __restrict__ x, const float* __restrict__ b,
                            float* __restrict__ out, int N, int K, int act) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= N) return;
  float acc = 0.f;
  for (int k = lane; k < K; k += 32) acc = fmaf(W[(size_t)row * K + k], x[k], acc);
  acc = fh::warp_sum(acc);
  if (lane == 0) {
    if (b) acc += b[row];
    if (act == 1) acc = acc / (1.0f + expf(-acc));  // SiLU
    out[row] = acc;
  }
}

__global__ void sincos_embed_kernel(const float* __restrict__ w, float t, float* __restrict__ out, int half) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= half) return;
  const float f = t * w[i] * 2.0f * 3.14159265358979323846f;  // x * w * 2 * pi (pos_emb.py:24)
  out[i] = sinf(f);
  out[half + i] = cosf(f);
}

// ------------------------------------------------------------------------------ conv pos embed
// out[n, c] = E[n, c] + gelu(b[c] + sum_j w[c, j] E[n + j - k/2, c])   (transformer.py:28-46, flow.py:240)
// HBM-bound (one fp32 read + one write per element).  A thread owns one channel and kDwT consecutive time steps:
// the kDwT + K - 1 inputs it needs are loaded once into registers (coalesced over the 128 channels of the block,
// halo re-reads between neighbouring tiles are L2 hits) and all K taps run from registers, fully unrolled.
// GELU_RES = false: plain depthwise Conv1d + bias (ConvNeXtBlock.dwconv, convnext.py:29,47).
constexpr int kDwT = 32;
template <int K, bool GELU_RES>
__global__ void __launch_bounds__(128) dwconv_gelu_res_kernel(const float* __restrict__ E, const float* __restrict__ w,
                                                              const float* __restrict__ b, float* __restrict__ out, int N,
                                                              int C) {
  const int c = blockIdx.x * 128 + threadIdx.x;
  const int n0 = blockIdx.y * kDwT, bi = blockIdx.z;
  if (c >= C) return;
  const float* e = E + (size_t)bi * N * C + c;
  constexpr int half = K >> 1;
  float wr[K];
#pragma unroll
  for (int j = 0; j < K; ++j) wr[j] = __ldg(w + (size_t)c * K + j);
  float x[kDwT + K - 1];
#pragma unroll
  for (int i = 0; i < kDwT + K - 1; ++i) {
    const int nn = n0 + i - half;
    x[i] = (nn >= 0 && nn < N) ? __ldg(e + (size_t)nn * C) : 0.f;  // Conv1d zero padding
  }
  const float bias = __ldg(b + c);
  float* o = out + ((size_t)bi * N + n0) * C + c;
#pragma unroll
  for (int t = 0; t < kDwT; ++t) {
    if (n0 + t < N) {
      float acc = bias;
#pragma unroll
      for (int j = 0; j < K; ++j) acc = fmaf(wr[j], x[t + j], acc);
      o[(size_t)t * C] = GELU_RES ? x[t + half] + fh::gelu_erf(acc) : acc;
    }
  }
}

// any odd kernel size (the checkpoint uses 31)
__global__ void dwconv_gelu_res_generic_kernel(const float* __restrict__ E, const float* __restrict__ w,
                                               const float* __restrict__ b, float* __restrict__ out, int N, int C, int k,
                                               int gelu_res) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = blockIdx.y, bi = blockIdx.z;
  if (c >= C) return;
  const float* e = E + (size_t)bi * N * C;
  const int half = k >> 1;
  float acc = b[c];
  for (int j = 0; j < k; ++j) {
    const int nn = n + j - half;
    if (nn >= 0 && nn < N) acc = fmaf(__ldg(w + (size_t)c * k + j), __ldg(e + (size_t)nn * C + c), acc);
  }
  out[((size_t)bi * N + n) * C + c] = gelu_res ? e[(size_t)n * C + c] + fh::gelu_erf(acc) : acc;
}

// ------------------------------------------------------------------------------ LayerNorm / AdaLayerNorm
// y = (x - mean) / sqrt(var + eps) * w + b  (F.layer_norm, biased variance).  AdaLayerNorm (convnext.py:86-93) is the
// same kernel with w = scale(t), b = shift(t).  One warp per row, the row lives in registers (C <= 1024);
// out_mode 0 -> fp32 row-major, 1 / 2 -> bf16 / fp16 chunked [C/8][rows][8].
__global__ void layernorm_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ b,
                                 void* __restrict__ out, int out_mode, int64_t out_rows, int M, int C, float eps,
                                 unsigned int* status) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= M) return;
  const float* xr = x + (size_t)row * C;
  float v[32];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const int c = lane + 32 * i;
    v[i] = c < C ? xr[c] : 0.f;
    s += v[i];
  }
  const float mean = fh::warp_sum(s) / (float)C;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const int c = lane + 32 * i;
    const float d = c < C ? v[i] - mean : 0.f;
    q = fmaf(d, d, q);
  }
  const float inv = rsqrtf(fh::warp_sum(q) / (float)C + eps);
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const int c = lane + 32 * i;
    if (c >= C) break;
    float y = (v[i] - mean) * inv * w[c];
    if (b) y += b[c];
    if (out_mode == 0) ((float*)out)[(size_t)row * C + c] = y;
    else ((unsigned short*)out)[fh::chunked_index(out_rows * 8, row, c)] = fh::cvt16_guard(y, out_mode == 2, status);
  }
}

// exact-erf GELU, fp32 row-major (nn.GELU, convnext.py:36)
__global__ void gelu_kernel(const float* __restrict__ x, float* __restrict__ out, int M, int C) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)M * C) return;
  out[i] = fh::gelu_erf(x[i]);
}

// ------------------------------------------------------------------------------ (adaptive) RMS norm
// one warp per row; out_mode 0 -> fp32 row-major, 1 -> bf16 chunked [C/8][rows][8]
__global__ void rmsnorm_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                               const float* __restrict__ beta, void* __restrict__ out, int out_mode, int64_t out_rows,
                               int M, int C, unsigned int* status) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= M) return;
  const float* xr = x + (size_t)row * C;
  float ss = 0.f;
  for (int c = lane; c < C; c += 32) {
    const float v = xr[c];
    ss = fmaf(v, v, ss);
  }
  ss = fh::warp_sum(ss);
  const float inv = sqrtf((float)C) / fmaxf(sqrtf(ss), 1e-12f);  // F.normalize eps, * dim**0.5
  if (out_mode == 0) {
    float* o = (float*)out + (size_t)row * C;
    for (int c = lane; c < C; c += 32) {
      float v = xr[c] * inv * gamma[c];
      if (beta) v += beta[c];
      o[c] = v;
    }
  } else {
    unsigned short* o = (unsigned short*)out;
    for (int c = lane; c < C; c += 32) {
      float v = xr[c] * inv * gamma[c];
      if (beta) v += beta[c];
      o[fh::chunked_index(out_rows * 8, row, c)] = fh::cvt16_guard(v, out_mode == 2, status);
    }
  }
}

// ------------------------------------------------------------------------------ q/k norm + rotary
// one warp per (token, head); D = 64: lane handles d = lane and lane + 32 (the rotary pair).
__global__ void qknorm_rope_kernel(const float* __restrict__ qkv, const float* __restrict__ qg,
                                   const float* __restrict__ kg, const float* __restrict__ inv_freq,
                                   float* __restrict__ q, float* __restrict__ k, float* __restrict__ v, int B, int N,
                                   int H) {
  constexpr int D = 64;
  const int gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (gw >= B * N * H) return;
  const int h = gw % H, tok = gw / H, n = tok % N, bi = tok / N;
  const float* src = qkv + (size_t)tok * 3 * H * D + h * D;
  const size_t dst = (((size_t)bi * H + h) * N + n) * D;
  const float fr = (float)n * inv_freq[lane];  // freqs = cat(f, f): both halves share it
  const float cs = cosf(fr), sn = sinf(fr);
#pragma unroll
  for (int which = 0; which < 2; ++which) {
    const float* s = src + which * H * D;
    const float* g = (which == 0 ? qg : kg) + h * D;
    float x1 = s[lane], x2 = s[lane + 32];
    float ss = fh::warp_sum(x1 * x1 + x2 * x2);
    const float inv = 8.0f / fmaxf(sqrtf(ss), 1e-12f);  // dim_head ** 0.5 = 8 (attend.py:147)
    x1 = x1 * inv * g[lane];  // F.normalize(x) * gamma * scale -- product order differs by <= 1 ulp
    x2 = x2 * inv * g[lane + 32];
    float* o = (which == 0 ? q : k) + dst;
    o[lane] = x1 * cs - x2 * sn;  // t*cos + rotate_half(t)*sin, rotate_half = (-x2, x1)
    o[lane + 32] = x2 * cs + x1 * sn;
  }
  const float* s = src + 2 * H * D;
  v[dst + lane] = s[lane];
  v[dst + lane + 32] = s[lane + 32];
}

// ------------------------------------------------------------------------------ attention (fp32)
// softmax(scale q k^T) v, no mask.  One CTA per (64 queries, b*h); keys streamed in blocks of 64;
// online softmax.  256 threads: thread (ty, tx) owns S/O rows 4*ty..+3, cols 4*tx..+3.
__global__ void __launch_bounds__(256) attention_f32_kernel(const float* __restrict__ Q, const float* __restrict__ Kt,
                                                            const float* __restrict__ V, float* __restrict__ out, int H,
                                                            int N, float scale) {
  constexpr int D = 64, BQ = 64, BK = 64;
  extern __shared__ __align__(16) float att_smem[];
  float (*Qs)[BQ + 1] = reinterpret_cast<float (*)[BQ + 1]>(att_smem);                      // [d][q]
  float (*Ks)[BK + 1] = reinterpret_cast<float (*)[BK + 1]>(att_smem + D * (BQ + 1));       // [d][key]
  float (*Ps)[BK + 1] = reinterpret_cast<float (*)[BK + 1]>(att_smem + 2 * D * (BQ + 1));   // [q][key]
  float (*Vs)[D + 4] = reinterpret_cast<float (*)[D + 4]>(att_smem + 3 * D * (BQ + 1));     // [key][d]
  const int bh = blockIdx.y, q0 = blockIdx.x * BQ;
  const int bi = bh / H, h = bh % H;
  const float* qb = Q + (size_t)bh * N * D;
  const float* kb = Kt + (size_t)bh * N * D;
  const float* vb = V + (size_t)bh * N * D;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  for (int i = threadIdx.x; i < BQ * D; i += 256) {
    const int r = i / D, d = i % D;
    Qs[d][r] = (q0 + r < N) ? qb[(size_t)(q0 + r) * D + d] * scale : 0.f;
  }
  float o[4][4] = {};
  float mrow[4], lrow[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) mrow[i] = -INFINITY, lrow[i] = 0.f;
  for (int k0 = 0; k0 < N; k0 += BK) {
    __syncthreads();
    for (int i = threadIdx.x; i < BK * D; i += 256) {
      const int r = i / D, d = i % D;
      const bool ok = k0 + r < N;
      Ks[d][r] = ok ? kb[(size_t)(k0 + r) * D + d] : 0.f;
      Vs[r][d] = ok ? vb[(size_t)(k0 + r) * D + d] : 0.f;
    }
    __syncthreads();
    float s[4][4] = {};
#pragma unroll 8
    for (int d = 0; d < D; ++d) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = Qs[d][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Ks[d][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) s[i][j] = fmaf(a[i], b[j], s[i][j]);
    }
    // row max over the 64 keys of this block: 16 tx-lanes of the same ty are contiguous lanes
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (k0 + tx * 4 + j >= N) s[i][j] = -INFINITY;
        mx = fmaxf(mx, s[i][j]);
      }
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
      const float mnew = fmaxf(mrow[i], mx);
      const float corr = expf(mrow[i] - mnew);
      float psum = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float p = expf(s[i][j] - mnew);
        Ps[ty * 4 + i][tx * 4 + j] = p;
        psum += p;
      }
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) psum += __shfl_xor_sync(0xffffffffu, psum, off);
      lrow[i] = lrow[i] * corr + psum;
      mrow[i] = mnew;
#pragma unroll
      for (int j = 0; j < 4; ++j) o[i][j] *= corr;
    }
    __syncthreads();
#pragma unroll 8
    for (int kk = 0; kk < BK; ++kk) {
      float p[4], vv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) p[i] = Ps[ty * 4 + i][kk];
#pragma unroll
      for (int j = 0; j < 4; ++j) vv[j] = Vs[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) o[i][j] = fmaf(p[i], vv[j], o[i][j]);
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int qi = q0 + ty * 4 + i;
    if (qi >= N) continue;
    const float inv = 1.0f / lrow[i];
    const int64_t row = (int64_t)bi * N + qi;
#pragma unroll
    for (int j = 0; j < 4; ++j) out[row * (H * D) + h * D + tx * 4 + j] = o[i][j] * inv;
  }
}

// ------------------------------------------------------------------------------ GEGLU / axpby
__global__ void geglu_kernel(const float* __restrict__ u, float* __restrict__ g, int inner) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int m = blockIdx.y;
  if (i >= inner) return;
  const float* ur = u + (size_t)m * 2 * inner;
  g[(size_t)m * inner + i] = fh::gelu_erf(ur[inner + i]) * ur[i];
}

__global__ void axpby_kernel(const float* __restrict__ x, const float* __restrict__ z, float a, float b,
                             float* __restrict__ y, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] = z ? a * x[i] + b * z[i] : a * x[i];
}

__global__ void broadcast_row_kernel(const float* __restrict__ row, float* __restrict__ out, int64_t M, int C) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < M * C) out[i] = row[i % C];
}

// ------------------------------------------------------------------------------ adaptive Runge-Kutta helpers
// (torchode path, cfm_superresolution.py:259-276: stage combination and the controller's scaled error norm)
struct RkCoefs { float c[8]; };

__global__ void rk_lincomb_kernel(const float* __restrict__ base, const float* __restrict__ k, int64_t kstride, int nk,
                                  RkCoefs cf, float* __restrict__ out, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float acc = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j)
    if (j < nk && cf.c[j] != 0.f) acc = fmaf(cf.c[j], k[(size_t)j * kstride + i], acc);
  out[i] = base ? base[i] + acc : acc;
}

// one block per problem instance: a fixed summation order, so accept / reject decisions are reproducible
__global__ void rk_scaled_sumsq_kernel(const float* __restrict__ e, const float* __restrict__ y0,
                                       const float* __restrict__ y1, float atol, float rtol, int64_t n,
                                       double* __restrict__ out) {
  __shared__ double part[32];
  const int64_t off = (int64_t)blockIdx.x * n;
  double acc = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    float m = fabsf(y0[off + i]);
    if (y1) m = fmaxf(m, fabsf(y1[off + i]));
    const float r = e[off + i] / fmaf(rtol, m, atol);
    acc += (double)r * (double)r;
  }
  for (int s = 16; s > 0; s >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, s);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    acc = threadIdx.x < (blockDim.x >> 5) ? part[threadIdx.x] : 0.0;
    for (int s = 16; s > 0; s >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, s);
    if (threadIdx.x == 0) out[blockIdx.x] = acc;
  }
}

// cfm_superresolution.py:134-144 on exp(mel) of one clip [N, F]: e[f] = sum_n exp(mel[n,f]); cumsum;
// scan from the top for the first bin whose cumulative energy is below percentile * total (bin 0 never tested)
__global__ void mel_cutoff_kernel(const float* __restrict__ mel, int* __restrict__ cutoff, int N, int F,
                                  float percentile) {
  extern __shared__ float e_sm[];
  const int b = blockIdx.x;
  const float* m = mel + (size_t)b * N * F;
  for (int f = threadIdx.x; f < F; f += blockDim.x) {
    float acc = 0.f;
    for (int n = 0; n < N; ++n) acc += fabsf(expf(m[(size_t)n * F + f]));
    e_sm[f] = acc;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float acc = 0.f;
    for (int f = 0; f < F; ++f) {
      acc += e_sm[f];
      e_sm[f] = acc;
    }
    const float thr = e_sm[F - 1] * percentile;
    int c = 0;
    for (int idx = F - 1; idx >= 1; --idx)
      if (e_sm[idx] < thr) {
        c = idx;
        break;
      }
    cutoff[b] = c;
  }
}

__global__ void mel_splice_kernel(const float* __restrict__ lo, const float* __restrict__ hi,
                                  const int* __restrict__ cutoff, float* __restrict__ out, int64_t per_clip, int F,
                                  int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int b = (int)(i / per_clip), f = (int)(i % F);
  out[i] = f < cutoff[b] ? lo[i] : hi[i];
}

}  // namespace

// ================================================================================ C ABI
extern "C" __attribute__((visibility("default"))) int fh_sgemm_nt_f32(const float* A, int lda, const float* W, int ldw, const float* bias, const float* res,
                               int ldr, float beta_res, float alpha, float* out, int ldc, int M, int N, int K,
                               void* stream) {
  FH_REQUIRE(M > 0 && N > 0 && K > 0 && lda >= K && ldw >= K && ldc >= N, FH_ERR_BAD_SHAPE,
             "fh_sgemm_nt_f32: bad shape M=%d N=%d K=%d", M, N, K);
  dim3 grid((N + GT - 1) / GT, (M + GT - 1) / GT);
  sgemm_nt_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(A, lda, W, ldw, bias, res, ldr, beta_res, alpha, out, ldc, M,
                                                          N, K);
  return fh::check_launch("fh_sgemm_nt_f32");
}

extern "C" __attribute__((visibility("default"))) int fh_gemv_f32(const float* W, const float* x, const float* b, float* out, int N, int K, int act,
                           void* stream) {
  FH_REQUIRE(N > 0 && K > 0, FH_ERR_BAD_SHAPE, "fh_gemv_f32: bad shape");
  gemv_kernel<<<(N + 7) / 8, 256, 0, (cudaStream_t)stream>>>(W, x, b, out, N, K, act);
  return fh::check_launch("fh_gemv_f32");
}

extern "C" __attribute__((visibility("default"))) int fh_sincos_embed_f32(const float* w, float t, float* out, int half, void* stream) {
  FH_REQUIRE(half > 0, FH_ERR_BAD_SHAPE, "fh_sincos_embed_f32: bad shape");
  sincos_embed_kernel<<<(half + 255) / 256, 256, 0, (cudaStream_t)stream>>>(w, t, out, half);
  return fh::check_launch("fh_sincos_embed_f32");
}

extern "C" __attribute__((visibility("default"))) int fh_dwconv_gelu_res_f32(const float* E, const float* w, const float* b, float* out, int B, int N, int C,
                                      int k, void* stream) {
  FH_REQUIRE(B > 0 && N > 0 && C > 0 && (k & 1), FH_ERR_BAD_SHAPE, "fh_dwconv_gelu_res_f32: kernel size must be odd");
  FH_REQUIRE(N <= 65535 && B <= 65535, FH_ERR_BAD_SHAPE, "fh_dwconv_gelu_res_f32: N, B must be <= 65535");
  if (k == 31)
    dwconv_gelu_res_kernel<31, true><<<dim3((C + 127) / 128, (N + kDwT - 1) / kDwT, B), 128, 0, (cudaStream_t)stream>>>(E, w, b, out, N, C);
  else
    dwconv_gelu_res_generic_kernel<<<dim3((C + 255) / 256, N, B), 256, 0, (cudaStream_t)stream>>>(E, w, b, out, N, C, k, 1);
  return fh::check_launch("fh_dwconv_gelu_res_f32");
}

extern "C" __attribute__((visibility("default"))) int fh_dwconv_f32(const float* x, const float* w, const float* b, float* out, int B, int N, int C,
                             int k, void* stream) {
  FH_REQUIRE(B > 0 && N > 0 && C > 0 && (k & 1), FH_ERR_BAD_SHAPE, "fh_dwconv_f32: kernel size must be odd");
  FH_REQUIRE(N <= 65535 && B <= 65535 && x != out, FH_ERR_BAD_SHAPE, "fh_dwconv_f32: N, B must be <= 65535, out of place");
  if (k == 7)
    dwconv_gelu_res_kernel<7, false><<<dim3((C + 127) / 128, (N + kDwT - 1) / kDwT, B), 128, 0, (cudaStream_t)stream>>>(x, w, b, out, N, C);
  else
    dwconv_gelu_res_generic_kernel<<<dim3((C + 255) / 256, N, B), 256, 0, (cudaStream_t)stream>>>(x, w, b, out, N, C, k, 0);
  return fh::check_launch("fh_dwconv_f32");
}

extern "C" __attribute__((visibility("default"))) int fh_layernorm_f32(const float* x, const float* w, const float* b, void* out, int out_mode,
                                int64_t out_rows, int M, int C, float eps, void* stream) {
  FH_REQUIRE(M > 0 && C > 0 && C <= 1024 && w != nullptr && (out_mode == 0 || (C % 8 == 0 && out_rows >= M)), FH_ERR_BAD_SHAPE,
             "fh_layernorm_f32: bad shape (C <= 1024)");
  layernorm_kernel<<<(M + 7) / 8, 256, 0, (cudaStream_t)stream>>>(x, w, b, out, out_mode, out_rows, M, C, eps,
                                                                  fh::status_word());
  return fh::check_launch("fh_layernorm_f32");
}

extern "C" __attribute__((visibility("default"))) int fh_gelu_f32(const float* x, float* out, int M, int C, void* stream) {
  FH_REQUIRE(M > 0 && C > 0, FH_ERR_BAD_SHAPE, "fh_gelu_f32: bad shape");
  const long long n = (long long)M * C;
  gelu_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, out, M, C);
  return fh::check_launch("fh_gelu_f32");
}

extern "C" __attribute__((visibility("default"))) int fh_rmsnorm_f32(const float* x, const float* gamma, const float* beta, void* out, int out_mode,
                              int64_t out_rows, int M, int C, void* stream) {
  FH_REQUIRE(M > 0 && C > 0 && (out_mode == 0 || (C % 8 == 0 && out_rows >= M)), FH_ERR_BAD_SHAPE,
             "fh_rmsnorm_f32: bad shape");
  rmsnorm_kernel<<<(M + 7) / 8, 256, 0, (cudaStream_t)stream>>>(x, gamma, beta, out, out_mode, out_rows, M, C,
                                                                fh::status_word());
  return fh::check_launch("fh_rmsnorm_f32");
}

extern "C" __attribute__((visibility("default"))) int fh_qknorm_rope_f32(const float* qkv, const float* qg, const float* kg, const float* inv_freq, float* q,
                                  float* k, float* v, int B, int N, int H, int D, void* stream) {
  FH_REQUIRE(D == 64, FH_ERR_UNSUPPORTED_CFG, "fh_qknorm_rope_f32: dim_head must be 64 (got %d)", D);
  const int64_t warps = (int64_t)B * N * H;
  qknorm_rope_kernel<<<(unsigned)((warps + 7) / 8), 256, 0, (cudaStream_t)stream>>>(qkv, qg, kg, inv_freq, q, k, v, B, N,
                                                                                   H);
  return fh::check_launch("fh_qknorm_rope_f32");
}

extern "C" __attribute__((visibility("default"))) int fh_attention_f32(const float* q, const float* k, const float* v, float* out, int B,
                                int H, int N, int D, float scale, void* stream) {
  FH_REQUIRE(D == 64, FH_ERR_UNSUPPORTED_CFG, "fh_attention_f32: dim_head must be 64 (got %d)", D);
  FH_REQUIRE(B * H <= 65535, FH_ERR_BAD_SHAPE, "fh_attention_f32: B*H must be <= 65535");
  constexpr int kAttSmem = (3 * 64 * 65 + 64 * 68) * (int)sizeof(float);
  static int smem_set[64] = {0};
  fh::ensure_dyn_smem(attention_f32_kernel, kAttSmem, smem_set);
  attention_f32_kernel<<<dim3((N + 63) / 64, B * H), 256, kAttSmem, (cudaStream_t)stream>>>(q, k, v, out, H, N, scale);
  return fh::check_launch("fh_attention_f32");
}

extern "C" __attribute__((visibility("default"))) int fh_geglu_f32(const float* u, float* g, int M, int inner, void* stream) {
  FH_REQUIRE(M > 0 && inner > 0, FH_ERR_BAD_SHAPE, "fh_geglu_f32: bad shape");
  FH_REQUIRE(M <= 65535 * 1024, FH_ERR_BAD_SHAPE, "fh_geglu_f32: M too large");
  // grid.y is limited to 65535: rows beyond it go to further launches
  for (int done = 0; done < M; done += 65535) {
    const int cnt = M - done > 65535 ? 65535 : M - done;
    geglu_kernel<<<dim3((inner + 255) / 256, cnt), 256, 0, (cudaStream_t)stream>>>(u + (size_t)done * 2 * inner,
                                                                                  g + (size_t)done * inner, inner);
    const int rc = fh::check_launch("fh_geglu_f32");
    if (rc) return rc;
  }
  return FH_OK;
}

extern "C" __attribute__((visibility("default"))) int fh_axpby_f32(const float* x, const float* z, float a, float b, float* y, int64_t n, void* stream) {
  if (n <= 0) return FH_OK;
  axpby_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, z, a, b, y, n);
  return fh::check_launch("fh_axpby_f32");
}

extern "C" __attribute__((visibility("default"))) int fh_rk_lincomb_f32(const float* base, const float* k, int64_t kstride,
                                                                       int nk, const float* coef_host, float* out,
                                                                       int64_t n, void* stream) {
  FH_REQUIRE(nk >= 1 && nk <= 8 && coef_host != nullptr && n > 0, FH_ERR_BAD_SHAPE, "fh_rk_lincomb_f32: 1 <= nk <= 8");
  RkCoefs cf;
  for (int j = 0; j < 8; ++j) cf.c[j] = j < nk ? coef_host[j] : 0.f;
  rk_lincomb_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(base, k, kstride, nk, cf, out, n);
  return fh::check_launch("fh_rk_lincomb_f32");
}

extern "C" __attribute__((visibility("default"))) int fh_rk_scaled_sumsq_f32(const float* e, const float* y0,
                                                                            const float* y1, float atol, float rtol,
                                                                            int B, int64_t n, double* out, void* stream) {
  FH_REQUIRE(B > 0 && n > 0 && e && y0 && out, FH_ERR_BAD_SHAPE, "fh_rk_scaled_sumsq_f32: bad arguments");
  rk_scaled_sumsq_kernel<<<B, 1024, 0, (cudaStream_t)stream>>>(e, y0, y1, atol, rtol, n, out);
  return fh::check_launch("fh_rk_scaled_sumsq_f32");
}

extern "C" __attribute__((visibility("default"))) int fh_broadcast_row_f32(const float* row, float* out, int64_t M, int C,
                                                                          void* stream) {
  FH_REQUIRE(M > 0 && C > 0, FH_ERR_BAD_SHAPE, "fh_broadcast_row_f32: bad shape");
  broadcast_row_kernel<<<(unsigned)((M * C + 255) / 256), 256, 0, (cudaStream_t)stream>>>(row, out, M, C);
  return fh::check_launch("fh_broadcast_row_f32");
}

extern "C" __attribute__((visibility("default"))) int fh_mel_cutoff_f32(const float* mel, int* cutoff, int B, int N, int F,
                                                                       float percentile, void* stream) {
  FH_REQUIRE(B > 0 && N > 0 && F > 0 && F <= 4096, FH_ERR_BAD_SHAPE, "fh_mel_cutoff_f32: bad shape");
  mel_cutoff_kernel<<<B, 256, F * sizeof(float), (cudaStream_t)stream>>>(mel, cutoff, N, F, percentile);
  return fh::check_launch("fh_mel_cutoff_f32");
}

extern "C" __attribute__((visibility("default"))) int fh_mel_splice_f32(const float* lo, const float* hi, const int* cutoff,
                                                                       float* out, int B, int N, int F, void* stream) {
  FH_REQUIRE(B > 0 && N > 0 && F > 0, FH_ERR_BAD_SHAPE, "fh_mel_splice_f32: bad shape");
  const int64_t n = (int64_t)B * N * F;
  mel_splice_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(lo, hi, cutoff, out, (int64_t)N * F, F,
                                                                                 n);
  return fh::check_launch("fh_mel_splice_f32");
}
