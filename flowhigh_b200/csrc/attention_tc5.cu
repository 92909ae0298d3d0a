// tcgen05 / TMEM attention for the 16-bit path: softmax(10 q k^T) v, no mask (attend.py:123-137), head dim 64.
//
// The logits reach +-640, so q (pre-scaled) and k are hi + lo 16-bit pairs and S = qh.kh + ql.kh + qh.kl accumulates in
// fp32; P is rounded to 16 bits for P.V.  An mma.sync kernel with the same arithmetic measured 2.9 x slower (DESIGN.md §4).
// Where the work runs:
//   * one CTA = 128 queries of one (batch, head); keys in blocks of 64.  S (128 x 64) is ONE accumulator in TMEM built by
//     12 tcgen05.mma (three operand pairings x four K = 16 steps), P.V (128 x 64) by four more; both issued by one thread.
//   * operands arrive as ready-made shared-memory images: fh_qknorm_rope_tiles writes q / k / v^T directly in the
//     no-swizzle K-major core-matrix layout ([8-element K group][row][8]), one contiguous tile per query tile / key
//     block, so the producer is one elected lane issuing cp.async.bulk copies against mbarriers.
//   * softmax: 128 threads, one query row each (a thread's TMEM lane), two passes over the S accumulator with
//     tcgen05.ld (row maximum, then exp2 + pack + store of the P row into the shared-memory A image of the P.V MMA) --
//     no shuffles, no cross-thread reductions.
//   * the running output stays in REGISTERS: every P.V product lands in a fresh TMEM buffer and is folded in one block
//     later as O = O * corr + PV, so nothing in TMEM is ever rescaled and the fold overlaps the next block's MMAs.
//   * S and PV buffers are double-buffered in TMEM (4 x 64 = 256 columns), K and V stages double-buffered in shared
//     memory with separate barriers (K is released when S is done, V when P.V is done); 97 KB + 256 columns per CTA,
//     so two CTAs share an SM and one's softmax overlaps the other's MMAs.
// Warps 0-3: softmax (TMEM lane groups 0-3), warp 4: producer, warp 5: MMA issuer + TMEM allocator.
#include <type_traits>
#include "common.cuh"
#include "tc_ptx.cuh"

namespace {

constexpr int QT = 128, KB = 64, DH = 64;
constexpr uint32_t kQBytes = 2u * 8u * QT * 16u;  // [hi | lo][d/8][128 q][8]     32 KB
constexpr uint32_t kKBytes = 2u * 8u * KB * 16u;  // [hi | lo][d/8][64 keys][8]   16 KB
constexpr uint32_t kVBytes = 8u * DH * 16u;       // [key/8][64 d][8 keys]         8 KB
constexpr uint32_t kPBytes = 8u * QT * 16u;       // [key/8][128 q][8 keys]       16 KB
constexpr uint32_t kOffQ = 1024, kOffK = kOffQ + kQBytes, kOffV = kOffK + 2 * kKBytes, kOffP = kOffV + 2 * kVBytes;
constexpr uint32_t kSmem5 = kOffP + kPBytes;      // 99 328 B
constexpr int kThreads5 = 192;
constexpr float kLog2e = 1.4426950408889634f;

enum Bar { Q_FULL = 0, K_FULL = 1, K_EMPTY = 3, V_FULL = 5, V_EMPTY = 7, S_FULL = 9, S_FREE = 11, P_FULL = 13, O_FULL = 14,
           O_FREE = 16, N_BARS = 18 };

struct At5Params {
  const unsigned short* q5;
  const unsigned short* k5;
  const unsigned short* v5;
  void* out;
  long long out_rows;
  int out_mode, H, N, nqt, nkb, fp16;
  unsigned int* status;
  unsigned int* err_flag;
};

__device__ __forceinline__ float max3f(float a, float b, float c) {
  float y;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(y) : "f"(a), "f"(b), "f"(c));
  return y;
}
__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__global__ void __launch_bounds__(kThreads5, 2) attention_tc5_kernel(const __grid_constant__ At5Params P) {
  extern __shared__ __align__(1024) unsigned char smem[];
  const uint32_t bar0 = smem_u32(smem);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 256);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int qt = blockIdx.x, bh = blockIdx.y;
  const int nkb = P.nkb;
  auto bar = [&](int which, int idx = 0) { return bar0 + 8u * (uint32_t)(which + idx); };

  if (threadIdx.x == 0) {
    mbar_init(bar(Q_FULL), 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(bar(K_FULL, s), 1);
      mbar_init(bar(K_EMPTY, s), 1);
      mbar_init(bar(V_FULL, s), 1);
      mbar_init(bar(V_EMPTY, s), 1);
      mbar_init(bar(S_FULL, s), 1);
      mbar_init(bar(S_FREE, s), 128);
      mbar_init(bar(O_FULL, s), 1);
      mbar_init(bar(O_FREE, s), 128);
    }
    mbar_init(bar(P_FULL), 128);
    fence_barrier_init();
  }
  if (warp == 5) tmem_alloc(smem_u32(tmem_slot), 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t sQ = bar0 + kOffQ, sK = bar0 + kOffK, sV = bar0 + kOffV, sP = bar0 + kOffP;

  if (warp == 4) {
    // ===================================================================== producer
    if (lane == 0) {
      const unsigned short* qsrc = P.q5 + ((size_t)bh * P.nqt + qt) * (kQBytes / 2);
      const unsigned short* ksrc = P.k5 + (size_t)bh * nkb * (kKBytes / 2);
      const unsigned short* vsrc = P.v5 + (size_t)bh * nkb * (kVBytes / 2);
      mbar_expect_tx(bar(Q_FULL), kQBytes);
      bulk_g2s(sQ, qsrc, kQBytes, bar(Q_FULL));
      for (int i = 0; i < nkb; ++i) {
        const int s = i & 1;
        const uint32_t par = (uint32_t)((i >> 1) & 1);
        mbar_wait(bar(K_EMPTY, s), par ^ 1, P.err_flag, 11);
        mbar_expect_tx(bar(K_FULL, s), kKBytes);
        bulk_g2s(sK + (uint32_t)s * kKBytes, ksrc + (size_t)i * (kKBytes / 2), kKBytes, bar(K_FULL, s));
        mbar_wait(bar(V_EMPTY, s), par ^ 1, P.err_flag, 12);
        mbar_expect_tx(bar(V_FULL, s), kVBytes);
        bulk_g2s(sV + (uint32_t)s * kVBytes, vsrc + (size_t)i * (kVBytes / 2), kVBytes, bar(V_FULL, s));
      }
    }
  } else if (warp == 5) {
    // ===================================================================== MMA issuer
    const bool leader = elect_one();
    const uint32_t idesc = make_idesc(64, P.fp16);
    const uint32_t hi = (128u >> 4) | (1u << 14);  // SBO = 128 B, descriptor version 1
    const uint32_t lbo_q = ((QT * 16u) >> 4) << 16, lbo_k = ((KB * 16u) >> 4) << 16;  // stride between 8-element K groups
    auto issue_S = [&](int i) {
      const int s = i & 1;
      const uint32_t par = (uint32_t)((i >> 1) & 1);
      mbar_wait(bar(K_FULL, s), par, P.err_flag, 21);
      mbar_wait(bar(S_FREE, s), par ^ 1, P.err_flag, 22);
      tc_fence_after();
      if (leader) {
        const uint32_t d = tmem_base + (uint32_t)s * 64u;
        const uint32_t kb = sK + (uint32_t)s * kKBytes;
        uint32_t acc = 0;
#pragma unroll
        for (int pass = 0; pass < 3; ++pass) {  // qh.kh, ql.kh, qh.kl
          const uint32_t qa = sQ + (pass == 1 ? kQBytes / 2 : 0u);
          const uint32_t ka = kb + (pass == 2 ? kKBytes / 2 : 0u);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {
            umma_f16_split(d, lbo_q | ((qa + (uint32_t)kk * 2u * QT * 16u) >> 4), hi,
                           lbo_k | ((ka + (uint32_t)kk * 2u * KB * 16u) >> 4), hi, idesc, acc);
            acc = 1;
          }
        }
        umma_commit(bar(S_FULL, s));
        umma_commit(bar(K_EMPTY, s));
      }
      __syncwarp();
    };
    auto issue_PV = [&](int i) {
      const int s = i & 1;
      const uint32_t par = (uint32_t)((i >> 1) & 1);
      mbar_wait(bar(V_FULL, s), par, P.err_flag, 23);
      mbar_wait(bar(O_FREE, s), par ^ 1, P.err_flag, 24);
      mbar_wait(bar(P_FULL), (uint32_t)(i & 1), P.err_flag, 25);
      tc_fence_after();
      if (leader) {
        const uint32_t d = tmem_base + 128u + (uint32_t)s * 64u;
        const uint32_t vb = sV + (uint32_t)s * kVBytes;
#pragma unroll
        for (int kt = 0; kt < 4; ++kt)  // 16 keys per step: A = P [128 q][keys], B = V^T [64 d][keys]
          umma_f16_split(d, lbo_q | ((sP + (uint32_t)kt * 2u * QT * 16u) >> 4), hi,
                         lbo_k | ((vb + (uint32_t)kt * 2u * DH * 16u) >> 4), hi, idesc, kt > 0 ? 1u : 0u);
        umma_commit(bar(O_FULL, s));
        umma_commit(bar(V_EMPTY, s));
      }
      __syncwarp();
    };
    mbar_wait(bar(Q_FULL), 0, P.err_flag, 20);
    issue_S(0);
    for (int i = 0; i < nkb; ++i) {
      if (i + 1 < nkb) issue_S(i + 1);
      issue_PV(i);
    }
  } else {
    // ===================================================================== softmax + output (warps 0..3)
    const int r = warp * 32 + lane;  // query row of the tile = TMEM lane
    const uint32_t tlane = tmem_base + ((uint32_t)(warp * 32) << 16);
    const uint32_t prow = sP + (uint32_t)r * 16u;
    const int fp16 = P.fp16;
    float O[64];
#pragma unroll
    for (int j = 0; j < 64; ++j) O[j] = 0.f;
    float m2 = -INFINITY, l = 0.f, corr_pend = 0.f;
    auto fold = [&](int j) {  // O = O * corr_pend + PV_j
      const uint32_t t = tlane + 128u + (uint32_t)(j & 1) * 64u;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint32_t v[16];
        tmem_ld16(t + (uint32_t)c * 16u, v);
        tmem_ld_wait();
#pragma unroll
        for (int e = 0; e < 16; ++e) O[c * 16 + e] = fmaf(O[c * 16 + e], corr_pend, __uint_as_float(v[e]));
      }
      tc_fence_before();
      mbar_arrive(bar(O_FREE, j & 1));
    };
    // one key block; MASKED only for a last block with fewer than 64 keys (the index tests cost as much as the softmax)
    auto block = [&](int i, auto masked_tag) {
      constexpr bool MASKED = decltype(masked_tag)::value;
      const int s = i & 1;
      const uint32_t tS = tlane + (uint32_t)s * 64u;
      const int nvalid = P.N - i * KB;  // keys of this block that exist (>= 64 unless MASKED)
      mbar_wait(bar(S_FULL, s), (uint32_t)((i >> 1) & 1), P.err_flag, 31);
      tc_fence_after();
      // ---- pass 1: row maximum
      float mx = -INFINITY;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint32_t v[16];
        tmem_ld16(tS + (uint32_t)c * 16u, v);
        tmem_ld_wait();
        if (MASKED) {
#pragma unroll
          for (int e = 0; e < 16; ++e)
            if (c * 16 + e < nvalid) mx = fmaxf(mx, __uint_as_float(v[e]));
        } else {
#pragma unroll
          for (int e = 0; e < 16; e += 2) mx = max3f(mx, __uint_as_float(v[e]), __uint_as_float(v[e + 1]));
        }
      }
      const float m_new = fmaxf(m2, mx * kLog2e);
      const float corr = ex2f(m2 - m_new);
      m2 = m_new;
      // the P image is single-buffered: P.V of the previous block must have retired before it is overwritten
      if (i > 0) {
        mbar_wait(bar(O_FULL, (i - 1) & 1), (uint32_t)(((i - 1) >> 1) & 1), P.err_flag, 32);
        tc_fence_after();
      }
      // ---- pass 2: p = 2^(s log2e - m), packed into the A image of the P.V MMA
      float psum0 = 0.f, psum1 = 0.f;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint32_t v[16];
        tmem_ld16(tS + (uint32_t)c * 16u, v);
        tmem_ld_wait();
        uint32_t pk[8];
#pragma unroll
        for (int e = 0; e < 16; e += 2) {
          float p0 = ex2f(fmaf(__uint_as_float(v[e]), kLog2e, -m_new));
          float p1 = ex2f(fmaf(__uint_as_float(v[e + 1]), kLog2e, -m_new));
          if (MASKED) {
            if (c * 16 + e >= nvalid) p0 = 0.f;
            if (c * 16 + e + 1 >= nvalid) p1 = 0.f;
          }
          psum0 += p0;
          psum1 += p1;
          pk[e >> 1] = fh::pack16(p0, p1, fp16);
        }
        asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(prow + (uint32_t)(2 * c) * (QT * 16u)), "r"(pk[0]),
                     "r"(pk[1]), "r"(pk[2]), "r"(pk[3])
                     : "memory");
        asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(prow + (uint32_t)(2 * c + 1) * (QT * 16u)), "r"(pk[4]),
                     "r"(pk[5]), "r"(pk[6]), "r"(pk[7])
                     : "memory");
      }
      tc_fence_before();
      mbar_arrive(bar(S_FREE, s));
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy P stores before the MMA's async reads
      mbar_arrive(bar(P_FULL));
      l = fmaf(l, corr, psum0 + psum1);
      if (i > 0) fold(i - 1);
      corr_pend = corr;
    };
    const int nfull = P.N / KB;  // blocks with all 64 keys
    for (int i = 0; i < nfull; ++i) block(i, std::false_type{});
    if (nfull < nkb) block(nfull, std::true_type{});
    mbar_wait(bar(O_FULL, (nkb - 1) & 1), (uint32_t)(((nkb - 1) >> 1) & 1), P.err_flag, 33);
    tc_fence_after();
    fold(nkb - 1);
    // ---- normalise and store
    const int qi = qt * QT + r;
    if (qi < P.N) {
      const float inv = 1.0f / l;
      const int bi = bh / P.H, h = bh % P.H;
      const long long row = (long long)bi * P.N + qi;
      if (P.out_mode == 0) {
        float4* dst = reinterpret_cast<float4*>((float*)P.out + row * (P.H * DH) + h * DH);
#pragma unroll
        for (int j = 0; j < 16; ++j) dst[j] = make_float4(O[4 * j] * inv, O[4 * j + 1] * inv, O[4 * j + 2] * inv, O[4 * j + 3] * inv);
      } else {
        fh::Guard16 guard;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          uint4 w;
          w.x = fh::pack16(O[8 * c] * inv, O[8 * c + 1] * inv, fp16);
          w.y = fh::pack16(O[8 * c + 2] * inv, O[8 * c + 3] * inv, fp16);
          w.z = fh::pack16(O[8 * c + 4] * inv, O[8 * c + 5] * inv, fp16);
          w.w = fh::pack16(O[8 * c + 6] * inv, O[8 * c + 7] * inv, fp16);
          guard.see(w.x, fp16), guard.see(w.y, fp16), guard.see(w.z, fp16), guard.see(w.w, fp16);
          *reinterpret_cast<uint4*>((unsigned short*)P.out + fh::chunked_index(P.out_rows * 8, row, h * DH + 8 * c)) = w;
        }
        guard.commit(P.status, fp16);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}

// q/k-norm + rotary (attend.py:144-151,179-184; pos_emb.py:45-60) emitting the operand images of attention_tc5_kernel:
//   q5 [B*H][ceil(N/128)][hi | lo][d/8][128][8]   (q pre-multiplied by `scale`)
//   k5 [B*H][ceil(N/64)][hi | lo][d/8][64][8]
// One warp per (token, head), lane = d and d + 32.
__global__ void qknorm_rope_tiles_kernel(const float* __restrict__ qkv, const float* __restrict__ qg,
                                         const float* __restrict__ kg, const float* __restrict__ inv_freq,
                                         unsigned short* __restrict__ q5, unsigned short* __restrict__ k5, int B, int N, int H,
                                         int nqt, int nkb, float scale, int fp16, unsigned int* status) {
  constexpr int D = 64;
  const int gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (gw >= B * N * H) return;
  const int h = gw % H, tok = gw / H, n = tok % N, bi = tok / N;
  const int bh = bi * H + h;
  const float* src = qkv + (size_t)tok * 3 * H * D + h * D;
  const float fr = (float)n * inv_freq[lane];
  const float cs = cosf(fr), sn = sinf(fr);
#pragma unroll
  for (int which = 0; which < 2; ++which) {
    const float* s = src + which * H * D;
    const float* gm = (which == 0 ? qg : kg) + h * D;
    float x1 = s[lane], x2 = s[lane + 32];
    const float ss = fh::warp_sum(x1 * x1 + x2 * x2);
    const float inv = 8.0f / fmaxf(sqrtf(ss), 1e-12f);
    x1 = x1 * inv * gm[lane];
    x2 = x2 * inv * gm[lane + 32];
    float y1 = x1 * cs - x2 * sn, y2 = x2 * cs + x1 * sn;
    if (which == 0) y1 *= scale, y2 *= scale;
    const int rows = which == 0 ? QT : KB;
    const int tile = n / rows, r = n % rows;
    unsigned short* base = (which == 0 ? q5 + ((size_t)bh * nqt + tile) * (kQBytes / 2)
                                       : k5 + ((size_t)bh * nkb + tile) * (kKBytes / 2));
    const size_t lo_off = (size_t)8 * rows * 8;
    const size_t e1 = (size_t)(lane >> 3) * rows * 8 + (size_t)r * 8 + (lane & 7);  // d = lane
    const size_t e2 = e1 + (size_t)4 * rows * 8;                                     // d = lane + 32
    const unsigned short h1 = fh::cvt16_guard(y1, fp16, status), h2 = fh::cvt16_guard(y2, fp16, status);
    const float f1 = fp16 ? __half2float(*reinterpret_cast<const __half*>(&h1)) : __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(&h1));
    const float f2 = fp16 ? __half2float(*reinterpret_cast<const __half*>(&h2)) : __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(&h2));
    base[e1] = h1;
    base[e2] = h2;
    base[lo_off + e1] = fh::cvt16(y1 - f1, fp16);
    base[lo_off + e2] = fh::cvt16(y2 - f2, fp16);
  }
}

// v5 [B*H][ceil(N/64)][key/8][64 d][8 keys] = V^T in K-major core matrices; keys past N are written as zeros (P is zero
// there, and 0 x stale-NaN would not be).  One thread per (b, h, group of 8 keys, d): 8 coalesced reads, one 16-byte store.
__global__ void v_tiles_kernel(const float* __restrict__ qkv, unsigned short* __restrict__ v5, int B, int N, int H, int nkb,
                               int fp16, unsigned int* status) {
  constexpr int D = 64;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = (long long)B * H * nkb * 8 * D;
  if (idx >= total) return;
  const int d = (int)(idx % D);
  long long t = idx / D;
  const int g = (int)(t % (nkb * 8));  // key group
  t /= (nkb * 8);
  const int h = (int)(t % H), bi = (int)(t / H);
  float v[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int n = g * 8 + j;
    v[j] = n < N ? __ldg(qkv + ((size_t)bi * N + n) * 3 * H * D + 2 * H * D + h * D + d) : 0.f;
  }
  uint4 w;
  w.x = fh::pack16_guard(v[0], v[1], fp16, status);
  w.y = fh::pack16_guard(v[2], v[3], fp16, status);
  w.z = fh::pack16_guard(v[4], v[5], fp16, status);
  w.w = fh::pack16_guard(v[6], v[7], fp16, status);
  // [bh][kb = g / 8][g % 8][d][8]
  *reinterpret_cast<uint4*>(v5 + ((((size_t)(bi * H + h) * nkb * 8 + g) * D) + d) * 8) = w;
}

}  // namespace

extern "C" __attribute__((visibility("default"))) int64_t fh_attention_tc5_operand_elems(int which, int B, int H, int N) {
  const int64_t nqt = (N + QT - 1) / QT, nkb = (N + KB - 1) / KB;
  if (which == 0) return (int64_t)B * H * nqt * (kQBytes / 2);
  if (which == 1) return (int64_t)B * H * nkb * (kKBytes / 2);
  return (int64_t)B * H * nkb * (kVBytes / 2);
}

extern "C" __attribute__((visibility("default"))) int fh_qknorm_rope_tiles(
    const float* qkv, const float* qg, const float* kg, const float* inv_freq, void* q5, void* k5, void* v5, int B, int N,
    int H, int D, float scale, int fp16, void* stream) {
  FH_REQUIRE(D == 64, FH_ERR_UNSUPPORTED_CFG, "fh_qknorm_rope_tiles: dim_head must be 64 (got %d)", D);
  FH_REQUIRE(B > 0 && N > 0 && H > 0, FH_ERR_BAD_SHAPE, "fh_qknorm_rope_tiles: bad shape");
  const int nqt = (N + QT - 1) / QT, nkb = (N + KB - 1) / KB;
  const int64_t warps = (int64_t)B * N * H;
  qknorm_rope_tiles_kernel<<<(unsigned)((warps + 7) / 8), 256, 0, (cudaStream_t)stream>>>(
      qkv, qg, kg, inv_freq, (unsigned short*)q5, (unsigned short*)k5, B, N, H, nqt, nkb, scale, fp16, fh::status_word());
  int rc = fh::check_launch("fh_qknorm_rope_tiles");
  if (rc != FH_OK) return rc;
  const int64_t total = (int64_t)B * H * nkb * 8 * 64;
  v_tiles_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(qkv, (unsigned short*)v5, B, N, H, nkb, fp16,
                                                                                  fh::status_word());
  return fh::check_launch("fh_qknorm_rope_tiles(v)");
}

extern "C" __attribute__((visibility("default"))) int fh_attention_tc5(const void* q5, const void* k5, const void* v5, void* out,
                                                                      int out_mode, int64_t out_rows, int B, int H, int N,
                                                                      int D, int fp16, void* stream) {
  FH_REQUIRE(D == 64, FH_ERR_UNSUPPORTED_CFG, "fh_attention_tc5: dim_head must be 64 (got %d)", D);
  FH_REQUIRE(B > 0 && H > 0 && B * H <= 65535 && N > 0, FH_ERR_BAD_SHAPE, "fh_attention_tc5: B*H must be <= 65535");
  static int set5[64] = {0};
  FH_REQUIRE(fh::ensure_dyn_smem(attention_tc5_kernel, (int)kSmem5, set5) == cudaSuccess, FH_ERR_CUDA,
             "fh_attention_tc5: cannot opt in to %u bytes of shared memory", kSmem5);
  At5Params P;
  P.q5 = (const unsigned short*)q5;
  P.k5 = (const unsigned short*)k5;
  P.v5 = (const unsigned short*)v5;
  P.out = out;
  P.out_rows = out_rows;
  P.out_mode = out_mode;
  P.H = H;
  P.N = N;
  P.nqt = (N + QT - 1) / QT;
  P.nkb = (N + KB - 1) / KB;
  P.fp16 = fp16;
  P.status = fh::status_word();
  P.err_flag = fh::err_word();
  attention_tc5_kernel<<<dim3(P.nqt, B * H), kThreads5, kSmem5, (cudaStream_t)stream>>>(P);
  return fh::check_launch("fh_attention_tc5");
}
