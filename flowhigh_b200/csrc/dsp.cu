// DSP stages of FlowHighSR.generate as CUDA kernels: polyphase resampler + peak normalise
// (flowhighsr.py:68-69), log-mel front end (melvoco.py:56-86) and the STFT-domain
// post-processing (postprocessing.py:18-41).  All HBM-bound; one CTA per STFT frame with the
// 2048-point FFT staged in shared memory.
#include <stdarg.h>
#include <atomic>
#include "common.cuh"

namespace fh {
static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches += n; }
static thread_local unsigned int* g_status = nullptr;
unsigned int* status_word() { return g_status; }
static thread_local unsigned int* g_errword = nullptr;
unsigned int* err_word() { return g_errword; }
}  // namespace fh

extern "C" __attribute__((visibility("default"))) int fh_version(void) { return 1; }
extern "C" __attribute__((visibility("default"))) const char* fh_last_error_string(void) { return fh::g_err; }
extern "C" __attribute__((visibility("default"))) int64_t fh_launch_count(void) { return (int64_t)fh::g_launches.load(); }
extern "C" __attribute__((visibility("default"))) int fh_set_status_word(uint32_t* status) {
  fh::g_status = status;
  return FH_OK;
}
extern "C" __attribute__((visibility("default"))) int fh_set_debug_word(uint32_t* word) {
  fh::g_errword = word;
  return FH_OK;
}

namespace {

// ------------------------------------------------------------------------------ utilities
__global__ void fill_u32_kernel(uint32_t* p, uint32_t v, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

__device__ __forceinline__ void block_absmax_atomic(float v, uint32_t* dst) {
  __shared__ float red[32];
  v = fh::warp_max(v);
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) red[w] = v;
  __syncthreads();
  if (w == 0) {
    int nw = (blockDim.x + 31) >> 5;
    float m = lane < nw ? red[lane] : 0.f;
    m = fh::warp_max(m);
    if (lane == 0) atomicMax(dst, __float_as_uint(m));
  }
}

// ------------------------------------------------------------------------------ resampler
// One thread per output sample:  y[m] = sum_i x[i] h[n(m) - i up],  n(m) = (m + n_pre_remove) down - n_pre_pad.
// IDX is the type of the tap index n: int when (T_out + n_pre_remove) * down fits 31 bits (every clip up to ~40 minutes
// at 48 kHz for the integer ratios), else long long.  The two divisions are done once per output in IDX arithmetic and
// the tap walk is pure 32-bit (ncu of the first version: issue-bound on 64-bit divisions and 64-bit tap indices, 0.04 of HBM).
template <typename IDX>
__global__ void __launch_bounds__(256) resample_poly_kernel(const float* __restrict__ x, float* __restrict__ y,
                                                            const float* __restrict__ h, uint32_t* absmax, int T_in, int T_out,
                                                            int ntaps, int up, int down, int n_pre_pad, int n_pre_remove) {
  const int b = blockIdx.y;
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  float acc = 0.f;
  if (m < T_out) {
    const IDX n = (IDX)(m + n_pre_remove) * down - n_pre_pad;  // tap index for i = 0
    if (n >= 0) {
      const IDX lo = n - ntaps + 1;
      const int i_lo = lo > 0 ? (int)((lo + up - 1) / up) : 0;
      int i_hi = (int)(n / up);
      int tap = (int)(n - (IDX)i_hi * up);  // tap of x[i_hi]; grows by `up` per step down in i
      if (i_hi > T_in - 1) {
        tap += (i_hi - (T_in - 1)) * up;
        i_hi = T_in - 1;
      }
      const float* xp = x + (size_t)b * T_in + i_hi;
      for (int k = i_hi - i_lo; k >= 0; --k, --xp, tap += up) acc = fmaf(__ldg(xp), __ldg(h + tap), acc);
    }
    y[(size_t)b * T_out + m] = acc;
  }
  if (absmax) block_absmax_atomic(fabsf(acc), absmax + b);
}

__global__ void absmax_kernel(const float* __restrict__ x, uint32_t* absmax, int T) {
  const int b = blockIdx.y;
  float m = 0.f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < T; i += gridDim.x * blockDim.x)
    m = fmaxf(m, fabsf(x[(size_t)b * T + i]));
  block_absmax_atomic(m, absmax + b);
}

__global__ void scale_by_absmax_kernel(const float* __restrict__ x, float* __restrict__ y,
                                       const uint32_t* __restrict__ absmax, float scale, int T) {
  const int b = blockIdx.y;
  const float mx = __uint_as_float(absmax[b]);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < T; i += gridDim.x * blockDim.x) {
    float v = x[(size_t)b * T + i] / mx;  // IEEE division, as numpy / torch
    y[(size_t)b * T + i] = scale == 1.0f ? v : v * scale;
  }
}

// ------------------------------------------------------------------------------ 2048-point FFT
// 2048 = 16 x 16 x 8 in three register-blocked passes by 128 threads (16 complex values per thread), two shared-memory
// exchanges between them (the first version was a radix-2 Stockham: 11 passes, 11 block barriers, ~5x the instructions).
//   pass 1: thread t     : DFT16 over j of x[t + 128 j],            twiddle W2048^(t k1)   -> b[k1][t]        (row 136)
//   pass 2: thread(k1,ta): DFT16 over tb of b[k1][ta + 8 tb],       twiddle W128^(ta k2)   -> a[ta][16 k2+k1] (row 258)
//   pass 3: thread c (x2): DFT8 over ta of a[ta][c]                                        -> out[c + 256 k3]
// Row strides 136 / 258 make every 64-bit shared-memory access of a half-warp conflict free.  Buffers hold kFftBuf
// complex values each; input in `a` (natural order), result in `b` (natural order).  Forward: exp(-2 pi i jk/n);
// inverse: conjugate in, conjugate out, unscaled.  blockDim.x must be 128.
constexpr int kFftBuf = 16 * 136;  // 2176 >= 8 * 258, >= 2048
template <typename T>
struct Cplx {
  T x, y;
};
template <typename T>
__device__ __forceinline__ Cplx<T> cmul(Cplx<T> a, Cplx<T> b) {
  return {a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x};
}

template <typename T>
__device__ __forceinline__ Cplx<T> twiddle(const float2* __restrict__ tw, int idx);  // exp(-2 pi i idx / 2048)
template <>
__device__ __forceinline__ Cplx<float> twiddle<float>(const float2* __restrict__ tw, int idx) {
  // the table holds the upper half circle, idx in [0, 1024): W^(idx + 1024) = -W^idx
  const float2 w = __ldg(tw + (idx & 1023));
  return (idx & 1024) ? Cplx<float>{-w.x, -w.y} : Cplx<float>{w.x, w.y};
}
template <>
__device__ __forceinline__ Cplx<double> twiddle<double>(const float2* __restrict__, int idx) {
  double s, c;
  sincospi(-(double)idx / 1024.0, &s, &c);
  return {c, s};
}

// forward 4-point DFT in place: (a, b, c, d) -> (X0, X1, X2, X3), W4 = -i
template <typename T>
__device__ __forceinline__ void dft4(Cplx<T>& a, Cplx<T>& b, Cplx<T>& c, Cplx<T>& d) {
  const Cplx<T> s0 = {a.x + c.x, a.y + c.y}, d0 = {a.x - c.x, a.y - c.y};
  const Cplx<T> s1 = {b.x + d.x, b.y + d.y}, d1 = {b.x - d.x, b.y - d.y};
  a = {s0.x + s1.x, s0.y + s1.y};
  c = {s0.x - s1.x, s0.y - s1.y};
  b = {d0.x + d1.y, d0.y - d1.x};  // d0 - i d1
  d = {d0.x - d1.y, d0.y + d1.x};  // d0 + i d1
}
// multiply by exp(-2 pi i m / 16), m a compile-time constant
template <int M, typename T>
__device__ __forceinline__ Cplx<T> mul_w16(Cplx<T> v) {
  constexpr int m = M & 15;
  if (m == 0) return v;
  if (m == 4) return {v.y, -v.x};
  if (m == 8) return {-v.x, -v.y};
  if (m == 12) return {-v.y, v.x};
  // cos / -sin of 2 pi m / 16
  const T c1 = (T)0.92387953251128675613, s1 = (T)0.38268343236508977173, r2 = (T)0.70710678118654752440;
  T c, sn;  // w = c - i sn
  switch (m) {
    case 1: c = c1, sn = s1; break;
    case 2: c = r2, sn = r2; break;
    case 3: c = s1, sn = c1; break;
    case 5: c = -s1, sn = c1; break;
    case 6: c = -r2, sn = r2; break;
    case 7: c = -c1, sn = s1; break;
    case 9: c = -c1, sn = -s1; break;
    case 10: c = -r2, sn = -r2; break;
    case 11: c = -s1, sn = -c1; break;
    case 13: c = s1, sn = -c1; break;
    case 14: c = r2, sn = -r2; break;
    default: c = c1, sn = -s1; break;  // 15
  }
  return {v.x * c + v.y * sn, v.y * c - v.x * sn};
}
// forward 16-point DFT in registers: v[n] -> v[k]  (n = 4 n1 + n2, k = k1 + 4 k2)
template <typename T>
__device__ __forceinline__ void dft16(Cplx<T> (&v)[16]) {
#pragma unroll
  for (int n2 = 0; n2 < 4; ++n2) dft4(v[n2], v[4 + n2], v[8 + n2], v[12 + n2]);  // v[4 k1 + n2] = a[n2][k1]
  v[5] = mul_w16<1>(v[5]), v[9] = mul_w16<2>(v[9]), v[13] = mul_w16<3>(v[13]);    // n2 = 1
  v[6] = mul_w16<2>(v[6]), v[10] = mul_w16<4>(v[10]), v[14] = mul_w16<6>(v[14]);  // n2 = 2
  v[7] = mul_w16<3>(v[7]), v[11] = mul_w16<6>(v[11]), v[15] = mul_w16<9>(v[15]);  // n2 = 3
#pragma unroll
  for (int k1 = 0; k1 < 4; ++k1) dft4(v[4 * k1], v[4 * k1 + 1], v[4 * k1 + 2], v[4 * k1 + 3]);  // v[4 k1 + k2] = X[k1 + 4 k2]
  // to natural order: X[k] with k = k1 + 4 k2 sits at 4 k1 + k2 -> transpose the 4 x 4 index
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = i + 1; j < 4; ++j) {
      const Cplx<T> t = v[4 * i + j];
      v[4 * i + j] = v[4 * j + i];
      v[4 * j + i] = t;
    }
}
// forward 8-point DFT in registers (n = 2 n1 + n2, k = k1 + 4 k2), natural order out
template <typename T>
__device__ __forceinline__ void dft8(Cplx<T> (&v)[8]) {
  dft4(v[0], v[2], v[4], v[6]);  // n2 = 0: v[2 k1]     = a[0][k1]
  dft4(v[1], v[3], v[5], v[7]);  // n2 = 1: v[2 k1 + 1] = a[1][k1]
  v[3] = mul_w16<2>(v[3]), v[5] = mul_w16<4>(v[5]), v[7] = mul_w16<6>(v[7]);  // W8^k1
  Cplx<T> o[8];
#pragma unroll
  for (int k1 = 0; k1 < 4; ++k1) {
    o[k1] = {v[2 * k1].x + v[2 * k1 + 1].x, v[2 * k1].y + v[2 * k1 + 1].y};
    o[k1 + 4] = {v[2 * k1].x - v[2 * k1 + 1].x, v[2 * k1].y - v[2 * k1 + 1].y};
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) v[k] = o[k];
}

template <typename T, bool INVERSE>
__device__ Cplx<T>* fft2048(Cplx<T>* a, Cplx<T>* b, const float2* __restrict__ tw) {
  const int t = threadIdx.x;  // 0..127
  Cplx<T> v[16];
  // ---- pass 1
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    v[j] = a[t + 128 * j];
    if (INVERSE) v[j].y = -v[j].y;
  }
  dft16(v);
#pragma unroll
  for (int k1 = 0; k1 < 16; ++k1) b[k1 * 136 + t] = k1 ? cmul(v[k1], twiddle<T>(tw, (t * k1) & 2047)) : v[0];
  __syncthreads();
  // ---- pass 2
  {
    const int k1 = t >> 3, ta = t & 7;
#pragma unroll
    for (int tb = 0; tb < 16; ++tb) v[tb] = b[k1 * 136 + ta + 8 * tb];
    dft16(v);
#pragma unroll
    for (int k2 = 0; k2 < 16; ++k2) a[ta * 258 + k2 * 16 + k1] = k2 ? cmul(v[k2], twiddle<T>(tw, (16 * ta * k2) & 2047)) : v[0];
  }
  __syncthreads();
  // ---- pass 3 (two 8-point transforms per thread)
  Cplx<T> z[2][8];
#pragma unroll
  for (int h = 0; h < 2; ++h) {
#pragma unroll
    for (int ta = 0; ta < 8; ++ta) z[h][ta] = a[ta * 258 + t + 128 * h];
    dft8(z[h]);
  }
  __syncthreads();  // every thread has read `a`; the caller may reuse it (and `b` below is a different buffer)
#pragma unroll
  for (int h = 0; h < 2; ++h)
#pragma unroll
    for (int k3 = 0; k3 < 8; ++k3) {
      Cplx<T> o = z[h][k3];
      if (INVERSE) o.y = -o.y;
      b[t + 128 * h + 256 * k3] = o;
    }
  __syncthreads();
  return b;
}

// ------------------------------------------------------------------------------ log-mel
template <typename T>
__global__ void __launch_bounds__(128) stft_logmel_kernel(const float* __restrict__ audio, float* __restrict__ mel,
                                                          const float* __restrict__ window,
                                                          const float2* __restrict__ tw,
                                                          const int* __restrict__ mel_start,
                                                          const int* __restrict__ mel_len,
                                                          const float* __restrict__ mel_w, int mel_stride, int Tlen,
                                                          int N) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Cplx<T>* a = reinterpret_cast<Cplx<T>*>(smem_raw);
  Cplx<T>* b = a + kFftBuf;
  const int n = blockIdx.x, bi = blockIdx.y;
  const float* x = audio + (size_t)bi * Tlen;
  for (int i = threadIdx.x; i < 2048; i += blockDim.x) {
    int pos = n * 480 + i - 784;  // reflect pad 784 (melvoco.py:74)
    if (pos < 0) pos = -pos;
    if (pos >= Tlen) pos = 2 * (Tlen - 1) - pos;
    const T v = (T)__ldg(x + pos) * (T)__ldg(window + i);  // fp32 product in the fp32 kernel, as torch.stft
    a[i] = {v, (T)0};
  }
  __syncthreads();
  Cplx<T>* r = fft2048<T, false>(a, b, tw);
  float* mag = reinterpret_cast<float*>(r == a ? b : a);
  for (int f = threadIdx.x; f <= 1024; f += blockDim.x) {
    const float re = (float)r[f].x, im = (float)r[f].y;
    mag[f] = sqrtf(re * re + im * im + 1e-9f);
  }
  __syncthreads();
  for (int m = threadIdx.x; m < 256; m += blockDim.x) {
    const int s = mel_start[m], len = mel_len[m];
    const float* w = mel_w + (size_t)m * mel_stride;
    float acc = 0.f;
    for (int i = 0; i < len; ++i) acc = fmaf(__ldg(w + i), mag[s + i], acc);
    mel[((size_t)bi * N + n) * 256 + m] = logf(fmaxf(acc, 1e-5f));
  }
}

// ------------------------------------------------------------------------------ post-processing
__global__ void pp_cutoff_kernel(const float* __restrict__ energy, int* __restrict__ cutoff, float threshold) {
  // sequential fp32 cumsum like torch.cumsum on CPU; scan from the top, never testing bin 0
  __shared__ float cum[1025];
  const int bi = blockIdx.x;
  if (threadIdx.x == 0) {
    float acc = 0.f;
    for (int f = 0; f <= 1024; ++f) {
      acc += energy[(size_t)bi * 1025 + f];
      cum[f] = acc;
    }
    const float thr = cum[1024] * threshold;
    int cr = 0;
    for (int idx = 1024; idx >= 1; --idx)
      if (cum[idx] < thr) {
        cr = idx;
        break;
      }
    cutoff[bi] = cr;
  }
}

// ---- fused post-processing: no spectrogram ever reaches HBM ------------------------------------------------------
// Two REAL frames share one complex FFT: X = FFT(p + i s)  =>  P[f] = (X[f] + conj X[-f]) / 2,  S[f] = (X[f] - conj X[-f]) / 2i.
__device__ __forceinline__ void split_two_real(const Cplx<float>* r, int f, float2& P, float2& S) {
  const Cplx<float> a = r[f], c = r[(2048 - f) & 2047];
  P = make_float2(0.5f * (a.x + c.x), 0.5f * (a.y - c.y));
  S = make_float2(0.5f * (a.y + c.y), -0.5f * (a.x - c.x));
}
__device__ __forceinline__ float frame_sample(const float* __restrict__ x, int Tlen, int n, int i, const float* __restrict__ window) {
  const int pos = n * 480 + i - 1024;  // center=True, pad_mode='constant' (postprocessing.py:7)
  return (pos >= 0 && pos < Tlen) ? __ldg(x + pos) * __ldg(window + i) : 0.f;
}

// energy partials of the SOURCE spectrum (postprocessing.py:10-16 needs sum_t |S[f,t]|): one block = 8 consecutive
// frames as 4 two-for-one FFTs, per-bin sums kept in double registers, one partial row per block (fixed order ->
// deterministic cutoff), reduced by pp_energy_reduce_kernel.
constexpr int kEnergyFrames = 8;
__global__ void __launch_bounds__(128) pp_src_energy_kernel(const float* __restrict__ src, double* __restrict__ partial,
                                                            const float* __restrict__ window,
                                                            const float2* __restrict__ tw, int Tlen, int NT, int G) {
  __shared__ __align__(16) Cplx<float> sa[kFftBuf];
  __shared__ __align__(16) Cplx<float> sb[kFftBuf];
  const int g = blockIdx.x, bi = blockIdx.y, t = threadIdx.x;
  const float* x = src + (size_t)bi * Tlen;
  double acc[9];
#pragma unroll
  for (int j = 0; j < 9; ++j) acc[j] = 0.0;
  for (int pair = 0; pair < kEnergyFrames / 2; ++pair) {
    const int n0 = g * kEnergyFrames + 2 * pair, n1 = n0 + 1;
    if (n0 >= NT) break;  // block-uniform
    for (int i = t; i < 2048; i += 128)
      sa[i] = {frame_sample(x, Tlen, n0, i, window), n1 < NT ? frame_sample(x, Tlen, n1, i, window) : 0.f};
    __syncthreads();
    const Cplx<float>* r = fft2048<float, false>(sa, sb, tw);
#pragma unroll
    for (int j = 0; j < 9; ++j) {
      const int f = t + 128 * j;
      if (f <= 1024) {
        float2 P, S;
        split_two_real(r, f, P, S);
        acc[j] += (double)hypotf(P.x, P.y);
        if (n1 < NT) acc[j] += (double)hypotf(S.x, S.y);
      }
    }
  }
  double* out = partial + ((size_t)bi * G + g) * 1025;
#pragma unroll
  for (int j = 0; j < 9; ++j) {
    const int f = t + 128 * j;
    if (f <= 1024) out[f] = acc[j];
  }
}
__global__ void pp_energy_reduce_kernel(const double* __restrict__ partial, float* __restrict__ energy, int G) {
  const int bi = blockIdx.y;
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f > 1024) return;
  double acc = 0.0;
  for (int g = 0; g < G; ++g) acc += partial[((size_t)bi * G + g) * 1025 + f];
  energy[(size_t)bi * 1025 + f] = (float)acc;
}

// per frame: FFT(pred + i src) -> split -> splice (src below the cutoff bin, pred from it on) -> Hermitian spectrum ->
// inverse FFT -> windowed frame for the overlap-add (postprocessing.py:22-39, torch.istft)
__global__ void __launch_bounds__(128) pp_fused_kernel(const float* __restrict__ pred, const float* __restrict__ src,
                                                       const int* __restrict__ cutoff, float* __restrict__ frames,
                                                       const float* __restrict__ window, const float2* __restrict__ tw,
                                                       int Tp, int Tlen, int NT) {
  __shared__ __align__(16) Cplx<float> sa[kFftBuf];
  __shared__ __align__(16) Cplx<float> sb[kFftBuf];
  const int n = blockIdx.x, bi = blockIdx.y, t = threadIdx.x;
  const float* xp = pred + (size_t)bi * Tp;
  const float* xs = src + (size_t)bi * Tlen;
  for (int i = t; i < 2048; i += 128) sa[i] = {frame_sample(xp, Tp, n, i, window), frame_sample(xs, Tlen, n, i, window)};
  __syncthreads();
  const Cplx<float>* r = fft2048<float, false>(sa, sb, tw);
  const int cr = cutoff[bi];
  for (int k = t; k < 2048; k += 128) {
    const int f = k <= 1024 ? k : 2048 - k;
    float2 P, S;
    split_two_real(r, f, P, S);
    float2 v = f < cr ? S : P;
    if (f == 0 || f == 1024) v.y = 0.f;  // c2r ignores the imaginary part of DC / Nyquist
    if (k > 1024) v.y = -v.y;
    sa[k] = {v.x, v.y};
  }
  __syncthreads();
  const Cplx<float>* y = fft2048<float, true>(sa, sb, tw);
  float* out = frames + ((size_t)bi * NT + n) * 2048;
  for (int i = t; i < 2048; i += 128) out[i] = y[i].x * (1.0f / 2048.0f) * __ldg(window + i);
}

__global__ void pp_overlap_add_kernel(const float* __restrict__ frames, float* __restrict__ y,
                                      const float* __restrict__ window, uint32_t* absmax, int NT, int length) {
  const int bi = blockIdx.y;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  float v = 0.f;
  if (t < length) {
    const int p = t + 1024;
    int n_hi = p / 480;
    if (n_hi > NT - 1) n_hi = NT - 1;
    int n_lo = p - 2047 > 0 ? (p - 2047 + 479) / 480 : 0;
    float acc = 0.f, env = 0.f;
    for (int n = n_lo; n <= n_hi; ++n) {
      const int i = p - 480 * n;
      acc += frames[((size_t)bi * NT + n) * 2048 + i];
      const float w = __ldg(window + i);
      env = fmaf(w, w, env);
    }
    v = env > 1e-11f ? acc / env : 0.f;
    y[(size_t)bi * length + t] = v;
  }
  if (absmax) block_absmax_atomic(fabsf(v), absmax + bi);
}

// long-form stitch: uniform chunks k = 0..K-1 spanning [k*step, k*step + clen); linear cross-fade in overlaps
__global__ void ola_crossfade_kernel(const float* __restrict__ chunks, float* __restrict__ out, int K, int clen,
                                     int step, long long total) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const int ov = clen - step;
  int k = (int)(t / step);
  if (k > K - 1) k = K - 1;
  const int o = (int)(t - (long long)k * step);  // offset inside chunk k
  float v = chunks[(long long)k * clen + o];
  if (k > 0 && o < ov) {  // also covered by the tail of chunk k-1
    const float w = ((float)o + 0.5f) / (float)ov;
    const float prev = chunks[(long long)(k - 1) * clen + (o + step)];
    v = w * v + (1.0f - w) * prev;
  }
  out[t] = v;
}

}  // namespace

// ================================================================================ C ABI
extern "C" __attribute__((visibility("default"))) int fh_fill_u32(uint32_t* p, uint32_t v, int64_t n, void* stream) {
  if (n <= 0) return FH_OK;
  fill_u32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(p, v, n);
  return fh::check_launch("fh_fill_u32");
}

extern "C" __attribute__((visibility("default"))) int fh_resample_poly_f32(const float* x, float* y, const float* h, uint32_t* absmax_bits, int B, int T_in,
                                    int T_out, int ntaps, int up, int down, int n_pre_pad, int n_pre_remove,
                                    void* stream) {
  FH_REQUIRE(B > 0 && T_in > 0 && T_out > 0 && ntaps > 0 && up > 0 && down > 0, FH_ERR_BAD_SHAPE,
             "fh_resample_poly_f32: bad shape B=%d T_in=%d T_out=%d", B, T_in, T_out);
  dim3 grid((T_out + 255) / 256, B);
  if (((long long)T_out + n_pre_remove) * down < (1ll << 31))
    resample_poly_kernel<int><<<grid, 256, 0, (cudaStream_t)stream>>>(x, y, h, absmax_bits, T_in, T_out, ntaps, up, down,
                                                                     n_pre_pad, n_pre_remove);
  else
    resample_poly_kernel<long long><<<grid, 256, 0, (cudaStream_t)stream>>>(x, y, h, absmax_bits, T_in, T_out, ntaps, up, down,
                                                                           n_pre_pad, n_pre_remove);
  return fh::check_launch("fh_resample_poly_f32");
}

extern "C" __attribute__((visibility("default"))) int fh_absmax_f32(const float* x, uint32_t* absmax_bits, int B, int T, void* stream) {
  FH_REQUIRE(B > 0 && T > 0, FH_ERR_BAD_SHAPE, "fh_absmax_f32: bad shape");
  int bx = (T + 256 * 8 - 1) / (256 * 8);
  if (bx > 1024) bx = 1024;
  absmax_kernel<<<dim3(bx, B), 256, 0, (cudaStream_t)stream>>>(x, absmax_bits, T);
  return fh::check_launch("fh_absmax_f32");
}

extern "C" __attribute__((visibility("default"))) int fh_scale_by_absmax_f32(const float* x, float* y, const uint32_t* absmax_bits, float scale, int B, int T,
                                      void* stream) {
  FH_REQUIRE(B > 0 && T > 0, FH_ERR_BAD_SHAPE, "fh_scale_by_absmax_f32: bad shape");
  int bx = (T + 256 * 4 - 1) / (256 * 4);
  if (bx > 2048) bx = 2048;
  scale_by_absmax_kernel<<<dim3(bx, B), 256, 0, (cudaStream_t)stream>>>(x, y, absmax_bits, scale, T);
  return fh::check_launch("fh_scale_by_absmax_f32");
}

extern "C" __attribute__((visibility("default"))) int fh_stft_logmel_f32(const float* audio, float* mel, const float* window, const float* twiddle,
                                  const int* mel_start, const int* mel_len, const float* mel_w, int mel_stride, int B,
                                  int T, int N, int precise, void* stream) {
  FH_REQUIRE(B > 0 && N > 0 && T >= 785, FH_ERR_BAD_SHAPE,
             "fh_stft_logmel_f32: need T >= 785 for the 784-sample reflect pad (got T=%d)", T);
  FH_REQUIRE(N == (T + 1568 - 2048) / 480 + 1, FH_ERR_BAD_SHAPE, "fh_stft_logmel_f32: N=%d does not match T=%d", N, T);
  dim3 grid(N, B);
  if (precise) {
    const int smem = 2 * kFftBuf * sizeof(double) * 2;
    static int smem_set[64] = {0};
    fh::ensure_dyn_smem(stft_logmel_kernel<double>, smem, smem_set);
    stft_logmel_kernel<double><<<grid, 128, smem, (cudaStream_t)stream>>>(
        audio, mel, window, (const float2*)twiddle, mel_start, mel_len, mel_w, mel_stride, T, N);
  } else {
    const int smem = 2 * kFftBuf * sizeof(float) * 2;
    stft_logmel_kernel<float><<<grid, 128, smem, (cudaStream_t)stream>>>(
        audio, mel, window, (const float2*)twiddle, mel_start, mel_len, mel_w, mel_stride, T, N);
  }
  return fh::check_launch("fh_stft_logmel_f32");
}

extern "C" __attribute__((visibility("default"))) int fh_pp_cutoff(const float* energy, int* cutoff, int B, float threshold, void* stream) {
  FH_REQUIRE(B > 0, FH_ERR_BAD_SHAPE, "fh_pp_cutoff: bad shape");
  pp_cutoff_kernel<<<B, 32, 0, (cudaStream_t)stream>>>(energy, cutoff, threshold);
  return fh::check_launch("fh_pp_cutoff");
}

extern "C" __attribute__((visibility("default"))) int fh_pp_energy_ws_bytes(int B, int NT) {
  if (B <= 0 || NT <= 0) return -1;
  const long long b = (long long)B * ((NT + kEnergyFrames - 1) / kEnergyFrames) * 1025 * 8;
  return b > 2147483647LL ? -1 : (int)b;
}

extern "C" __attribute__((visibility("default"))) int fh_pp_src_energy_f32(const float* src, float* energy, void* workspace,
                                                                           const float* window, const float* twiddle, int B,
                                                                           int T, int NT, void* stream) {
  FH_REQUIRE(B > 0 && T > 0 && NT == 1 + T / 480 && B <= 65535, FH_ERR_BAD_SHAPE, "fh_pp_src_energy_f32: NT=%d does not match T=%d",
             NT, T);
  FH_REQUIRE(workspace != nullptr && ((uintptr_t)workspace % 8) == 0, FH_ERR_BAD_ALIGN, "fh_pp_src_energy_f32: workspace");
  const int G = (NT + kEnergyFrames - 1) / kEnergyFrames;
  pp_src_energy_kernel<<<dim3(G, B), 128, 0, (cudaStream_t)stream>>>(src, (double*)workspace, window, (const float2*)twiddle, T,
                                                                   NT, G);
  int rc = fh::check_launch("fh_pp_src_energy_f32");
  if (rc != FH_OK) return rc;
  pp_energy_reduce_kernel<<<dim3((1025 + 127) / 128, B), 128, 0, (cudaStream_t)stream>>>((const double*)workspace, energy, G);
  return fh::check_launch("fh_pp_src_energy_f32(reduce)");
}

extern "C" __attribute__((visibility("default"))) int fh_pp_fused_f32(const float* pred, const float* src, const int* cutoff,
                                                                      float* frames, const float* window, const float* twiddle,
                                                                      int B, int Tp, int T, int NT, void* stream) {
  FH_REQUIRE(B > 0 && T > 0 && Tp > 0 && NT == 1 + T / 480 && NT == 1 + Tp / 480 && B <= 65535, FH_ERR_BAD_SHAPE,
             "fh_pp_fused_f32: pred (%d) and src (%d samples) must span the same %d frames", Tp, T, NT);
  pp_fused_kernel<<<dim3(NT, B), 128, 0, (cudaStream_t)stream>>>(pred, src, cutoff, frames, window, (const float2*)twiddle, Tp,
                                                                T, NT);
  return fh::check_launch("fh_pp_fused_f32");
}

extern "C" __attribute__((visibility("default"))) int fh_pp_overlap_add_f32(const float* frames, float* y, const float* window, uint32_t* absmax_bits, int B,
                                     int NT, int length, void* stream) {
  FH_REQUIRE(B > 0 && NT > 0 && length > 0, FH_ERR_BAD_SHAPE, "fh_pp_overlap_add_f32: bad shape");
  pp_overlap_add_kernel<<<dim3((length + 255) / 256, B), 256, 0, (cudaStream_t)stream>>>(frames, y, window, absmax_bits,
                                                                                       NT, length);
  return fh::check_launch("fh_pp_overlap_add_f32");
}

extern "C" __attribute__((visibility("default"))) int fh_ola_crossfade_f32(const float* chunks, float* out, int K,
                                                                          int clen, int step, int64_t total,
                                                                          void* stream) {
  FH_REQUIRE(K > 0 && clen > 0 && step > 0 && step <= clen && 2 * step >= clen && total > 0 &&
                 total <= (int64_t)(K - 1) * step + clen,
             FH_ERR_BAD_SHAPE, "fh_ola_crossfade_f32: need clen/2 <= step <= clen and total within the chunks");
  ola_crossfade_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(chunks, out, K, clen, step,
                                                                                         total);
  return fh::check_launch("fh_ola_crossfade_f32");
}
