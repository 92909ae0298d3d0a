// Anti-aliased Snake / SnakeBeta on the chunked [C/8][Lp][8] layout as a *worker*: a group of 128 threads that walks
// (batch, chunk, time-tile) work items with its own shared-memory buffers and named barrier.  The standalone kernel
// (vocoder_tc.cu) is one worker per CTA.
//
// y[q] = sum_k f[k] s~[2q+k-5];  s[m] = u[m] + inv_b sin^2(a u[m]);  u[m] = 2 sum_i x~[i] f[m+5-2i]
// (x~ / s~ = replicate-clamped; closed form of up2x -> snake -> down2x, SURVEY.md A.5; reference:
// alias_free_torch/act.py:23-28, resample.py:25-33, filter.py:86-94, activations.py:48-59,107-119).
//
// Register-blocked and 2-wide: one thread owns TWO adjacent channels and R consecutive outputs; every filter tap is
// one packed FFMA2 (fma.rn.f32x2, sm_100; measured 1.55x the scalar FFMA rate, tools/ffma2_bench.cu) on a channel
// pair, applied from registers.  sin^2(z) is evaluated as (1 - cos 2z)/2 so that
//     s' = u - (inv_b/2) cos(2 a u),   y = sum_k f[k] s'~[.] + inv_b/2      (sum_k f[k] = 1)
// costs one packed multiply, two MUFU.COS and one packed FMA per pair.  cos.approx's absolute error (~1e-6 for
// |arg| < 1e2) is far below the 16-bit operand rounding that follows.
//
// The (32 R + 10) x 8-channel fp32 input window of the NEXT item is fetched with one cp.async.bulk (UBLKCP) into the
// other shared-memory buffer while the current item is computed; R odd makes the un-padded 32-byte-row window bank-
// conflict free for the (4 pairs x 8 groups) 64-bit reads of a warp; replicate clamps are patched in shared memory
// and in registers on the first / last tile of a sequence only (group-uniform branch).  16-bit outputs go through a
// shared-memory image of the output tile (32 R rows x 16 B, contiguous in HBM) written by one bulk store.
#pragma once
#include "common.cuh"

namespace fh {

struct SnakeParams {
  const float* x;
  void* y;
  const float* a;
  const float* inv_b;
  const float* filt;
  long long batch_stride, chunk_stride;
  long long y_batch_stride;  // batch stride of y (elements; the hi + lo output of the split mode has twice the chunks)
  long long lo_offset;       // split mode: element offset of the "lo" chunks behind the "hi" chunks of y, else 0
  int row0, nchunk, L, ntile, total;
  int fp16;  // 16-bit output format when OUT_KIND == 3 (chosen at run time): 0 bfloat16, 1 IEEE half
  unsigned int* status;  // overflow / NaN status word of the caller (common.cuh Guard16) or nullptr
};

template <int R>
struct SnakeGeom {
  static constexpr int kRows = R * 32;       // time steps per tile
  static constexpr int kXRows = kRows + 10;  // rows per staged window
  static constexpr int kXBytes = kXRows * 32;
  static constexpr int kYBytes = kRows * 16;
  // shared memory of one worker: two input windows, one 16-bit output image, two mbarriers
  static constexpr int kSmemBytes = ((2 * kXBytes + kYBytes + 16 + 127) / 128) * 128;
};

__device__ __forceinline__ float2 sw_ffma2(float2 a, float2 b, float2 c) {
  unsigned long long ra = *reinterpret_cast<unsigned long long*>(&a), rb = *reinterpret_cast<unsigned long long*>(&b),
                     rc = *reinterpret_cast<unsigned long long*>(&c), rd;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
  return *reinterpret_cast<float2*>(&rd);
}
__device__ __forceinline__ float2 sw_fmul2(float2 a, float2 b) {
  unsigned long long ra = *reinterpret_cast<unsigned long long*>(&a), rb = *reinterpret_cast<unsigned long long*>(&b), rd;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
  return *reinterpret_cast<float2*>(&rd);
}
__device__ __forceinline__ uint32_t sw_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void sw_mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0;
  const long long t0 = clock64();
  while (!ok) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity), "r"(2000u)  // suspend-time hint (ns): a waiting warp sleeps instead of taking issue slots
        : "memory");
    if (!ok && clock64() - t0 > 4000000000LL) __trap();
  }
}
__device__ __forceinline__ void sw_group_sync(int bar_id) {
  asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
}

// `smem` points to SnakeGeom<R>::kSmemBytes bytes (128-byte aligned) owned by this worker; `tid` in [0, 128);
// work items worker, worker + nworkers, ... ; bar_id is the named barrier of this group of 128 threads.
// OUT_KIND: 0 fp32, 1 bf16, 2 fp16, 3 = 16-bit with the format taken from S.fp16 (one instantiation for both).
template <int OUT_KIND, bool BULK_OUT, int R>
__device__ __forceinline__ void snake_worker(const SnakeParams& S, unsigned char* smem, int tid, int worker, int nworkers,
                                             int bar_id) {
  const int out_fp16 = OUT_KIND == 3 ? S.fp16 : (OUT_KIND == 2);
  using G = SnakeGeom<R>;
  float* xs0 = reinterpret_cast<float*>(smem);
  float* xs1 = reinterpret_cast<float*>(smem + G::kXBytes);
  unsigned char* ys = smem + 2 * G::kXBytes;
  const uint32_t bar0 = sw_u32(smem + 2 * G::kXBytes + G::kYBytes);
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0) : "memory");
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0 + 8) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  sw_group_sync(bar_id);
  const int rows_per_chunk = (int)(S.chunk_stride >> 3);
  auto issue = [&](int item, int buf) {
    const int tile = item % S.ntile;
    const int rest = item / S.ntile;
    const int ch = rest % S.nchunk, b = rest / S.nchunk;
    const int r_first = S.row0 + tile * G::kRows - 5;  // >= row0 - 5 >= 0 (left halo)
    int nrows = rows_per_chunk - r_first;              // stay inside this chunk's rows
    nrows = nrows < G::kXRows ? nrows : G::kXRows;
    const float* src = S.x + (long long)b * S.batch_stride + (long long)ch * S.chunk_stride + (long long)r_first * 8;
    const uint32_t bar = bar0 + 8 * buf;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t)nrows * 32u) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     sw_u32(buf ? xs1 : xs0)),
                 "l"(src), "r"((uint32_t)nrows * 32u), "r"(bar)
                 : "memory");
  };
  float2 fu[12], fd[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) {
    const float fk = __ldg(S.filt + k);
    fu[k] = make_float2(2.0f * fk, 2.0f * fk);
    fd[k] = make_float2(fk, fk);
  }
  const int e2 = tid & 3, g = tid >> 2;
  Guard16 guard;
  int item = worker;
  if (item < S.total && tid == 0) issue(item, 0);
  int buf = 0;
  uint32_t ph0 = 0, ph1 = 0;
  for (; item < S.total; item += nworkers) {
    const int tile = item % S.ntile;
    const int rest = item / S.ntile;
    const int ch = rest % S.nchunk, b = rest / S.nchunk;
    const int qt = tile * G::kRows;
    const bool edge = (tile == 0) || (qt + G::kRows + 5 > S.L);
    sw_mbar_wait(bar0 + 8 * buf, buf ? ph1 : ph0);
    if (buf) ph1 ^= 1; else ph0 ^= 1;
    float* xt = buf ? xs1 : xs0;
    if (edge) {  // replicate-pad the window in shared memory: rows t < 0 <- x[0], rows t >= L <- x[L-1]
      for (int i = tid; i < G::kXRows * 2; i += 128) {
        const int r = i >> 1, h = i & 1;
        const int t = qt - 5 + r;
        const int tc = min(max(t, 0), S.L - 1);
        if (tc != t) {
          const int rc = tc - (qt - 5);
          if (rc >= 0 && rc < G::kXRows)
            *reinterpret_cast<float4*>(&xt[r * 8 + h * 4]) = *reinterpret_cast<const float4*>(&xt[rc * 8 + h * 4]);
        }
      }
      sw_group_sync(bar_id);
    }
    const int c0 = ch * 8 + 2 * e2;
    const float2 al2 = make_float2(2.0f * __ldg(S.a + c0), 2.0f * __ldg(S.a + c0 + 1));
    const float2 hib = make_float2(0.5f * __ldg(S.inv_b + c0), 0.5f * __ldg(S.inv_b + c0 + 1));
    const float2 nhib = make_float2(-hib.x, -hib.y);
    const int q0 = qt + g * R;
    float2 xv[R + 10];
    const float* xp = xt + g * (R * 8) + 2 * e2;
#pragma unroll
    for (int j = 0; j < R + 10; ++j) xv[j] = *reinterpret_cast<const float2*>(xp + j * 8);
    if (BULK_OUT && tid == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // ys is free again
    sw_group_sync(bar_id);  // every thread has read this buffer's window
    if (tid == 0 && item + nworkers < S.total) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      issue(item + nworkers, buf ^ 1);  // that buffer was fully read one iteration ago
    }
    if (q0 < S.L) {
      float2 s[2 * R + 10];
#pragma unroll
      for (int i = 0; i < 2 * R + 10; ++i) {
        const int qq = (i - 5) >> 1;
        float2 u = make_float2(0.f, 0.f);
        if ((i & 1) == 0) {
#pragma unroll
          for (int d = -2; d <= 3; ++d) u = sw_ffma2(xv[qq + d + 5], fu[6 - 2 * d], u);
        } else {
#pragma unroll
          for (int d = -3; d <= 2; ++d) u = sw_ffma2(xv[qq + d + 5], fu[5 - 2 * d], u);
        }
        const float2 z = sw_fmul2(u, al2);
        const float2 c = make_float2(__cosf(z.x), __cosf(z.y));
        s[i] = sw_ffma2(c, nhib, u);
      }
      if (edge && (q0 == 0 || q0 + R + 3 >= S.L)) {
        const int ic = 2 * (S.L - q0) + 5;
        float2 prev = s[5];
#pragma unroll
        for (int i = 0; i < 2 * R + 10; ++i) {
          if (q0 == 0 && i < 5) s[i] = prev;
          if (i < ic) prev = s[i];
          else s[i] = prev;
        }
      }
      const long long obase =
          (long long)b * S.y_batch_stride + (long long)ch * S.chunk_stride + (long long)(S.row0 + q0) * 8 + 2 * e2;
#pragma unroll
      for (int j = 0; j < R; ++j) {
        // the bulk-store path writes into the shared-memory image (rows past L are never stored to HBM): no
        // per-output predicate there, so the 17 tap chains are one basic block and get interleaved by the scheduler
        if (BULK_OUT || !edge || q0 + j < S.L) {
          float2 acc = hib;
#pragma unroll
          for (int k = 0; k < 12; ++k) acc = sw_ffma2(fd[k], s[2 * j + k], acc);
          if (OUT_KIND) {
            const uint32_t hv = pack16(acc.x, acc.y, out_fp16);
            guard.see(hv, out_fp16);
            if (BULK_OUT) *reinterpret_cast<uint32_t*>(ys + (size_t)(g * R + j) * 16 + 4 * e2) = hv;
            else *reinterpret_cast<uint32_t*>((unsigned short*)S.y + obase + j * 8) = hv;
          } else
            *reinterpret_cast<float2*>((float*)S.y + obase + j * 8) = acc;
        }
      }
    }
    if (BULK_OUT) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      sw_group_sync(bar_id);
      if (tid == 0) {
        const int nrows = min(G::kRows, S.L - qt);
        const unsigned short* dst = (const unsigned short*)S.y + (long long)b * S.y_batch_stride +
                                    (long long)ch * S.chunk_stride + (long long)(S.row0 + qt) * 8;
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(sw_u32(ys)),
                     "r"((uint32_t)nrows * 16u)
                     : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
    }
    buf ^= 1;
  }
  if (BULK_OUT && tid == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
  if (OUT_KIND) guard.commit(S.status, out_fp16);
}

}  // namespace fh
