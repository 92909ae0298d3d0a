// Anti-aliased Snake / SnakeBeta with both FIR filters on the tensor pipe (fp16 output mode of the chunked layout).
//
// Same closed form as snake_worker.cuh (SURVEY.md A.5; reference alias_free_torch/act.py:23-28, resample.py:25-33,
// filter.py:86-94, activations.py:48-59,107-119):
//   u[m] = 2 sum_i x~[i] f[m+5-2i]      s'[m] = u[m] - (inv_b/2) cos(2 a u[m])      y[q] = inv_b/2 + sum_k f[k] s'~[2q+k-5]
// The scalar kernel spends 24 of its ~34 issue slots per element on the 6 + 6 + 12 filter taps.  Here the two filters
// are banded Toeplitz matrices applied with mma.sync.m16n8k16 (fp16 operands, fp32 accumulate):
//   * M = 16 independent sequences = 8 channels of one chunk x 2 time segments ("halves") of the tile, so a thread
//     (g = lane / 4, q = lane % 4) only ever needs the snake parameters of channel g;
//   * up stage:  D[seq][8 up-samples] = X[seq][16 input steps] . Tup[16][8]; the fp32 input is rounded to fp16
//     (SPLIT_X: split x = hi + lo, two MMAs -- measured to buy < 0.3 dB end to end); the k-slot -> time map inside an
//     8-step block is permuted (slot 2q -> row q, slot 2q+1 -> row q+4) so that the fragment loads from the
//     [time][8 ch] fp32 window are bank-conflict free; the Toeplitz fragment is built with the same permutation;
//   * snake on the accumulator registers (packed FMUL2 / FFMA2, MUFU.COS);
//   * two adjacent accumulator tiles of the up stage ARE the A fragment of the down stage (16 up-samples), so
//     nothing is shuffled or staged:  Y[seq][8 outputs] = sum_{d=-1,0,1} S_{i+d}[seq][16] . Tdn_d[16][8];
//   * the filter taps are fp16, chosen by error feedback inside each polyphase branch (exact DC gains);
//   * the output tile goes to shared memory with stmatrix.trans ([time][8 ch] rows) and to HBM with one bulk store.
// Replicate clamps: x~ is patched in the shared-memory window (first / last segments); the s~ clamp only changes the
// first and last three outputs of a sequence, which the warp recomputes in scalar fp32 on those segments.
// Pipeline: one shared double-buffered input window per CTA tile (cp.async.bulk against an mbarrier), everything
// else per warp -- see snake_mma_cta below.
#pragma once
#include <cuda_fp16.h>
#include "snake_worker.cuh"

namespace fh {

template <int NB>  // 8-output blocks per half-segment
struct SnakeMmaGeom {
  static constexpr int kWarps = 4;
  static constexpr int kSeg = 8 * NB;           // outputs per half-segment
  static constexpr int kWarpRows = 2 * kSeg;    // outputs per warp and tile (two halves, adjacent in time)
  static constexpr int kRows = kWarps * kWarpRows;
  static constexpr int kHalo = 8;               // window rows before / after the tile
  static constexpr int kXRows = kRows + 2 * kHalo;
  static constexpr int kXBytes = kXRows * 32;  // fp32 rows; fp16 input rows take half of it
  static constexpr int kWarpYBytes = kWarpRows * 16;
  // two input windows, per warp two output images, 128 control bytes: two mbarriers, two release counters, 2 x 12 taps
  static constexpr int smem_bytes(bool in16, bool split_out = false) {
    return 2 * (in16 ? kXBytes / 2 : kXBytes) + (split_out ? 4 : 2) * kWarps * kWarpYBytes + 128;
  }
};

__device__ __forceinline__ uint32_t sm_pack(float lo, float hi) {
  __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ void sm_split(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  __half2 h = __floats2half2_rn(x0, x1);
  const float2 hf = __half22float2(h);
  hi = *reinterpret_cast<uint32_t*>(&h);
  lo = sm_pack(x0 - hf.x, x1 - hf.y);
}
__device__ __forceinline__ void sm_mma(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                       uint32_t b1, float c0, float c1, float c2, float c3) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%11,%12,%13};"
      : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1), "f"(c0), "f"(c1), "f"(c2), "f"(c3));
}

// K = 8 form (A fragment = one 16 x 8 half of a 16 x 16 fragment: registers {a0, a1} = k 0..7, {a2, a3} = k 8..15)
__device__ __forceinline__ void sm_mma_k8(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t b0, float c0, float c1, float c2,
                                          float c3) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%7,%8,%9,%10};"
               : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
               : "r"(a0), "r"(a1), "r"(b0), "f"(c0), "f"(c1), "f"(c2), "f"(c3));
}

// ---- pieces of snake_mma_cta -------------------------------------------------------------------------------------------

// fp16 taps by ERROR FEEDBACK instead of round-to-nearest (one thread): within each polyphase branch (even / odd taps)
// the taps are rounded in order of decreasing magnitude and every rounding error is carried into the next, finer-grained
// tap, so the branch sums (the DC gains) stay exact to ~2^-20.  On low-pass signals the response error of the rounded
// filters drops from -66 dB (round-to-nearest) to -83 dB (CPU experiment, DESIGN.md section 4).
// s_taps[0, 12): up-filter taps (2 f), [12, 24): down-filter taps (f).
// Four independent (filter, polyphase branch) chains: called by threads 0..3 with part = thread index (the serial form cost
// ~3 us at the start of every launch -- a tenth of a B = 1 snake launch).
__device__ __forceinline__ void snake_mma_make_taps(const float* __restrict__ filt, float* s_taps, int part) {
  const int w = part >> 1, ph = part & 1;
  const float scale = w ? 1.0f : 2.0f;
  float f[6];
#pragma unroll
  for (int c = 0; c < 6; ++c) f[c] = __ldg(filt + 2 * c + ph);
  unsigned done = 0;
  float carry = 0.f;
#pragma unroll
  for (int n = 0; n < 6; ++n) {
    int best = 0;
    float bm = -1.f;
#pragma unroll
    for (int c = 0; c < 6; ++c) {
      const float m = fabsf(f[c]);
      if (!((done >> c) & 1u) && m > bm) bm = m, best = c;
    }
    done |= 1u << best;
    float fb = f[0];
#pragma unroll
    for (int c = 1; c < 6; ++c) fb = best == c ? f[c] : fb;
    const float v = scale * fb + carry;
    const float h = __half2float(__float2half_rn(v));
    carry = v - h;
    s_taps[12 * w + 2 * best + ph] = h;
  }
}

// Toeplitz B fragments (k16 x n8, "col") of one thread: reg r holds k-slots 2q + 8r, 2q + 8r + 1 of column n = g
struct SnakeFrags {
  uint32_t bu[2][2], bd[3][2];
};
template <bool IN16>
__device__ __forceinline__ void snake_mma_frags(const float* s_taps, int lane, SnakeFrags& F) {
  const int g = lane >> 2, q = lane & 3;
  auto tap = [&](int idx, float scale) -> float {  // scale 2 = up filter, 1 = down filter
    return (idx >= 0 && idx < 12) ? s_taps[(scale == 2.0f ? 0 : 12) + idx] : 0.f;
  };
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    // up n-block e of a 16-up-sample block starting at input step T: up-sample m = 2T + 8e + n from the input steps
    // T - 8 + ko (e = 0) or T + ko (e = 1), ko = q + 8r (slot 2q + 8r) and q + 4 + 8r (slot 2q + 8r + 1); ko = slot
    // for the ldmatrix-fed fp16 input
    const int base = e ? 13 : 21;
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int ko0 = IN16 ? 2 * q + 8 * r : q + 8 * r, ko1 = IN16 ? ko0 + 1 : ko0 + 4;
      const float v0 = tap(g + base - 2 * ko0, 2.0f), v1 = tap(g + base - 2 * ko1, 2.0f);
      F.bu[e][r] = sm_pack(v0, v1);
    }
  }
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    // down block: output Q + n from the up-samples 2Q + 16 (d - 1) + c, c = k-slot (identity map)
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int c0 = 2 * q + 8 * r;
      const float v0 = tap(16 * (d - 1) + c0 - 2 * g + 5, 1.0f), v1 = tap(16 * (d - 1) + c0 + 1 - 2 * g + 5, 1.0f);
      F.bd[d][r] = sm_pack(v0, v1);
    }
  }
}

// One warp, one unit: the 2 x (8 NB) outputs q0 .. q0 + 16 NB - 1 of the 8 channels of chunk `ch`.
//   xw : shared-memory window of the unit, row 0 = time q0 - kHalo, 16 NB + 2 kHalo rows of 8 channels
//        (fp32 rows of 32 bytes, or fp16 rows of 16 bytes when IN16); rows [lo, hi) relative to xw exist (the replicate
//        patch may read a clamped row from a neighbour's part of a shared window)
//   yt : shared-memory output image, row 0 = time q0, 16-byte rows [time][8 ch] fp16
// edge: the unit touches t < 0 or t >= L (replicate clamps apply).  Rows of the image with t >= L are computed from the
// clamped signal (finite) and must be ignored / overwritten by the caller.
// SPLIT_OUT: the fp32 result is written as hi + lo fp16 pairs (yt_lo: second image, same geometry) -- the operand of a
// convolution whose input channels are doubled [hi | lo] against duplicated weights keeps ~22 bits of the activation.
template <bool SPLIT_X, int NB, bool IN16, bool SPLIT_OUT = false>
__device__ __forceinline__ void snake_mma_unit(const SnakeFrags& F, float* xw, unsigned char* yt, int q0, int L, int ch,
                                               const float* __restrict__ sn_a, const float* __restrict__ sn_inv_b,
                                               const float* __restrict__ sn_filt, bool edge, int lo, int hi, int lane,
                                               Guard16& guard, unsigned char* yt_lo = nullptr) {
  using G = SnakeMmaGeom<NB>;
  const int g = lane >> 2, q = lane & 3;
  if (edge) {
    // replicate-pad the rows this warp reads: t < 0 <- x[0], t >= L <- x[L-1] (a neighbour warp may write the same
    // values into the shared halo rows)
    for (int i = lane; i < (G::kWarpRows + 2 * G::kHalo) * 2; i += 32) {
      const int r = i >> 1, h = i & 1;
      const int t = q0 - G::kHalo + r;
      const int tc = min(max(t, 0), L - 1);
      if (tc != t) {
        const int rc = tc - (q0 - G::kHalo);
        if (rc >= lo && rc < hi) {
          if (IN16) {  // 16-byte rows: two 8-byte halves
            const uint2* w16 = reinterpret_cast<const uint2*>(xw);
            reinterpret_cast<uint2*>(xw)[r * 2 + h] = w16[rc * 2 + h];
          } else {
            *reinterpret_cast<float4*>(&xw[r * 8 + h * 4]) = *reinterpret_cast<const float4*>(&xw[rc * 8 + h * 4]);
          }
        }
      }
    }
    __syncwarp();
  }
  {
    const int cg = ch * 8 + g;
    const float alv = 2.0f * __ldg(sn_a + cg), hib = 0.5f * __ldg(sn_inv_b + cg);
    const float2 al2 = make_float2(alv, alv), nhib2 = make_float2(-hib, -hib);
    // window row of unit row r is r + kHalo; input block jx of half h covers window rows h kSeg + 8 jx + 8 ...
    const float* xp = xw + q * 8 + g;
    // stmatrix row addresses: lanes 0-7 = rows of half A, lanes 8-15 = rows of half B (others ignored by .x2)
    const uint32_t st_base = sw_u32(yt) + (uint32_t)((lane & 7) + ((lane >> 3) & 1) * G::kSeg) * 16u;
    uint32_t xh[NB + 2][2], xl[NB + 2][2];  // input blocks jx = -1 .. NB at index jx + 1
    auto load_x = [&](int jx) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const float x0 = xp[(8 * jx + 8) * 8 + h * G::kSeg * 8], x1 = xp[(8 * jx + 12) * 8 + h * G::kSeg * 8];
        if (SPLIT_X) sm_split(x0, x1, xh[jx + 1][h], xl[jx + 1][h]);
        else xh[jx + 1][h] = sm_pack(x0, x1);
      }
    };
    // up n-block (j, e): the 8 up-samples 2 (q0 + 8 j) + 8 e + n, both halves, into dd
    // fp16 input: lane l addresses row (l & 7) of matrix l >> 3: {half A, half B} x {first, second 8 input steps}
    const uint32_t lm_base = sw_u32(xw) + (uint32_t)((lane & 7) + ((lane >> 3) & 1) * G::kSeg + (lane >> 4) * 8) * 16u;
    auto up_mma = [&](int j, int e, float (&dd)[4]) {
      if (IN16) {
        const int k0 = (e ? 8 * j : 8 * j - 8) + G::kHalo;  // first window row (relative to this unit's half A)
        uint32_t a0, a1, a2, a3;
        asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                     : "=r"(a0), "=r"(a1), "=r"(a2), "=r"(a3)
                     : "r"(lm_base + (uint32_t)(k0 * 16)));
        sm_mma(dd, a0, a1, a2, a3, F.bu[e][0], F.bu[e][1], 0.f, 0.f, 0.f, 0.f);
        return;
      }
      const int p = (e ? j : j - 1) + 1, n = p + 1;
      sm_mma(dd, xh[p][0], xh[p][1], xh[n][0], xh[n][1], F.bu[e][0], F.bu[e][1], 0.f, 0.f, 0.f, 0.f);
      if (SPLIT_X) sm_mma(dd, xl[p][0], xl[p][1], xl[n][0], xl[n][1], F.bu[e][0], F.bu[e][1], dd[0], dd[1], dd[2], dd[3]);
    };
    auto snake2 = [&](float u0, float u1) -> uint32_t {
      const float2 u = make_float2(u0, u1);
      const float2 z = sw_fmul2(u, al2);
      const float2 c = make_float2(__cosf(z.x), __cosf(z.y));
      const float2 s = sw_ffma2(c, nhib2, u);
      return sm_pack(s.x, s.y);
    };
    // Software pipeline, in-order issue in mind (mma.sync are volatile asm, i.e. issued in source order): in step j
    //   1. the up-stage MMAs of step j + 1 are issued,
    //   2. the snake of step j runs on accumulators issued one step earlier        -> A fragment U_j,
    //   3. U_j is scattered into the three down blocks it touches (j - 1: last term, j: middle, j + 1: first), three
    //      independent MMAs; every down accumulator is next touched one whole step later.
    float dd[2][2][4];  // [step parity][e][acc]
    float y[3][4];      // down accumulators of blocks i, at index i % 3
    if (!IN16) {
      load_x(-1);
      load_x(0);
      if (NB >= 1) load_x(1);
    }
    up_mma(-1, 1, dd[0][1]);
#pragma unroll
    for (int j = -1; j <= NB; ++j) {
      const int cur = (j + 1) & 1, nxt = cur ^ 1;
      if (!IN16 && j + 3 <= NB) load_x(j + 3);  // consumed by the MMAs issued in the next step
      if (j + 1 <= NB) {
        up_mma(j + 1, 0, dd[nxt][0]);
        if (j + 1 < NB) up_mma(j + 1, 1, dd[nxt][1]);
      }
      uint32_t U[4];  // A fragment of the 16 up-samples of step j
      if (j >= 0) U[0] = snake2(dd[cur][0][0], dd[cur][0][1]), U[1] = snake2(dd[cur][0][2], dd[cur][0][3]);
      else U[0] = U[1] = 0u;  // up-samples below 2 q0 - 8 only meet zero weights
      if (j < NB) U[2] = snake2(dd[cur][1][0], dd[cur][1][1]), U[3] = snake2(dd[cur][1][2], dd[cur][1][3]);
      else U[2] = U[3] = 0u;
      // The 12-tap down filter reaches 5 up-samples back and 6 forward of an output block's own 16: of the previous
      // block only the LAST 8 up-samples carry non-zero weights and of the next block only the FIRST 8, so those two
      // terms are K = 8 MMAs on half of the A fragment (the other half of the Toeplitz fragment is identically zero).
      if (j >= 1) {  // last term of down block j - 1 (first 8 up-samples of step j), then store it
        float (&yy)[4] = y[(j - 1) % 3];
        sm_mma_k8(yy, U[0], U[1], F.bd[2][0], yy[0], yy[1], yy[2], yy[3]);
      }
      if (j >= 0 && j < NB) {
        float (&yy)[4] = y[j % 3];
        sm_mma(yy, U[0], U[1], U[2], U[3], F.bd[1][0], F.bd[1][1], yy[0], yy[1], yy[2], yy[3]);
      }
      if (j + 1 < NB) {  // first term of down block j + 1 (last 8 up-samples of step j)
        float (&yy)[4] = y[(j + 1) % 3];
        sm_mma_k8(yy, U[2], U[3], F.bd[0][1], hib, hib, hib, hib);
      }
      if (j >= 1) {
        // outputs q0 + 8 i + {2 q, 2 q + 1} of channel g, both halves: the accumulator tile is an 8 x 8 [seq][time]
        // fragment per half, stored TRANSPOSED ([time][8 ch] rows of 16 bytes) by one stmatrix
        const int i = j - 1;
        const float (&yy)[4] = y[i % 3];
        const uint32_t r0 = pack16(yy[0], yy[1], 1), r1 = pack16(yy[2], yy[3], 1);
        guard.see(r0, 1);
        guard.see(r1, 1);
        asm volatile("stmatrix.sync.aligned.m8n8.x2.trans.shared.b16 [%0], {%1, %2};" ::"r"(st_base + (uint32_t)(8 * i * 16)),
                     "r"(r0), "r"(r1)
                     : "memory");
        if (SPLIT_OUT) {
          const float2 h0 = __half22float2(*reinterpret_cast<const __half2*>(&r0));
          const float2 h1 = __half22float2(*reinterpret_cast<const __half2*>(&r1));
          const uint32_t l0 = pack16(yy[0] - h0.x, yy[1] - h0.y, 1), l1 = pack16(yy[2] - h1.x, yy[3] - h1.y, 1);
          asm volatile("stmatrix.sync.aligned.m8n8.x2.trans.shared.b16 [%0], {%1, %2};" ::"r"(
                           st_base + (uint32_t)(yt_lo - yt) + (uint32_t)(8 * i * 16)),
                       "r"(l0), "r"(l1)
                       : "memory");
        }
      }
    }
  }
  if (edge) {  // the s~ clamp changes outputs 0..2 and L-3..L-1 only: recompute those in scalar fp32
    __syncwarp();
    for (int w = lane; w < 48; w += 32) {
      const int c = w & 7, o = w >> 3;
      const int qq = o < 3 ? o : L - 6 + o;
      if (qq >= q0 && qq < q0 + G::kWarpRows && qq < L && (o < 3 || qq >= 3)) {
        const int cc = ch * 8 + c;
        const float alv = 2.0f * __ldg(sn_a + cc), hib = 0.5f * __ldg(sn_inv_b + cc);
        float acc = hib;
        for (int k = 0; k < 12; ++k) {
          const int m = min(max(2 * qq + k - 5, 0), 2 * L - 1);
          const int ihi = (m + 5) >> 1;
          float u = 0.f;
          for (int t6 = 0; t6 < 6; ++t6) {
            const int i = ihi - t6;
            const int ic = min(max(i, 0), L - 1);
            const int xi = (ic - q0 + G::kHalo) * 8 + c;
            const float xv = IN16 ? __half2float(reinterpret_cast<const __half*>(xw)[xi]) : xw[xi];
            u = fmaf(2.0f * __ldg(sn_filt + (m + 5 - 2 * i)), xv, u);
          }
          acc = fmaf(__ldg(sn_filt + k), u - hib * __cosf(alv * u), acc);
        }
        const __half hv = __float2half_rn(acc);
        *reinterpret_cast<__half*>(yt + (size_t)(qq - q0) * 16 + 2 * c) = hv;
        if (SPLIT_OUT) *reinterpret_cast<__half*>(yt_lo + (size_t)(qq - q0) * 16 + 2 * c) = __float2half_rn(acc - __half2float(hv));
      }
    }
  }
}

// One CTA of 4 warps walks tiles (batch, chunk, kRows outputs) cta, cta + nctas, ...  The input window of a tile is
// shared (one cp.async.bulk against a "full" mbarrier); everything else is per warp: each warp computes its own
// 2 x kSeg rows, stores them with its own bulk store and releases the window through a shared-memory counter -- the
// last warp to release a window refills it with the tile after next.  There is no CTA-wide barrier in the loop (ncu
// on a bar.sync version: 16 % of the warp stalls).
// IN16: the input is already fp16 on the same chunked layout (16-byte rows, written by the 16-bit epilogue of the
// preceding convolution): the A fragments of the up stage come straight from the window with one ldmatrix.x4.trans
// per 8 up-samples (identity k-slot -> time map), no conversion instructions at all.
template <bool SPLIT_X, int NB, bool IN16 = false, bool SPLIT_OUT = false>
__device__ __forceinline__ void snake_mma_cta(const SnakeParams& S, unsigned char* smem, int tid, int cta, int nctas) {
  using G = SnakeMmaGeom<NB>;
  const int lane = tid & 31, warp = tid >> 5;
  constexpr int kXB = IN16 ? G::kXBytes / 2 : G::kXBytes;  // bytes of one input window
  float* xs0 = reinterpret_cast<float*>(smem);
  float* xs1 = reinterpret_cast<float*>(smem + kXB);
  constexpr int kImg = SPLIT_OUT ? 2 : 1;  // images per buffer (hi, lo)
  unsigned char* ys0 = smem + 2 * kXB + warp * 2 * kImg * G::kWarpYBytes;  // this warp's two output buffers
  unsigned char* ctl = smem + 2 * kXB + 2 * kImg * G::kWarps * G::kWarpYBytes;
  const uint32_t bar0 = sw_u32(ctl);
  int* released = reinterpret_cast<int*>(ctl + 16);  // warps done with window 0 / 1
  float* s_taps = reinterpret_cast<float*>(ctl + 32);  // [0, 12): up-filter taps (2 f), [12, 24): down-filter taps (f)
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0) : "memory");
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0 + 8) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    released[0] = released[1] = 0;
  }
  if (tid < 4) snake_mma_make_taps(S.filt, s_taps, tid);
  // rows a clipped copy does not fill must hold finite values (they only ever meet zero filter weights)
  for (int i = tid; i < 2 * kXB / 16; i += 32 * G::kWarps) reinterpret_cast<float4*>(smem)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  __syncthreads();
  const int rows_per_chunk = (int)(S.chunk_stride >> 3);
  // (tile, chunk, batch) of an item advance by running coordinates: item -> item + nctas adds (d_tile, d_ch, d_b) with
  // carries (the ncu source page showed the two divisions per tile and warp as ~6 % of all instructions)
  const int d_tile = nctas % S.ntile, d_rest = nctas / S.ntile;
  const int d_ch = d_rest % S.nchunk, d_b = d_rest / S.nchunk;
  auto advance = [&](int& tile, int& ch, int& b) {
    tile += d_tile;
    ch += d_ch;
    b += d_b;
    if (tile >= S.ntile) tile -= S.ntile, ++ch;
    if (ch >= S.nchunk) ch -= S.nchunk, ++b;
  };
  auto issue = [&](int tile, int ch, int b, int buf) {
    const int r_first = S.row0 + tile * G::kRows - G::kHalo;  // >= 0: the launcher requires row0 >= kHalo
    int nrows = rows_per_chunk - r_first;                     // stay inside this chunk's rows
    nrows = nrows < G::kXRows ? nrows : G::kXRows;
    const long long eoff = (long long)b * S.batch_stride + (long long)ch * S.chunk_stride + (long long)r_first * 8;
    const void* src = IN16 ? (const void*)((const unsigned short*)S.x + eoff) : (const void*)(S.x + eoff);
    const uint32_t bytes = (uint32_t)nrows * (IN16 ? 16u : 32u);
    const uint32_t bar = bar0 + 8 * buf;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     sw_u32(buf ? xs1 : xs0)),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
  };

  SnakeFrags F;
  snake_mma_frags<IN16>(s_taps, lane, F);
  // Overflow guard: the fp16 roundings of the input and of the snake samples do NOT saturate, so an out-of-range value
  // becomes inf, turns the outputs it reaches into inf / NaN, and is caught where the outputs are packed (saturating).
  Guard16 guard;
  int item = cta;
  int tile = item % S.ntile, ch = (item / S.ntile) % S.nchunk, b = (item / S.ntile) / S.nchunk;
  int tile_f = tile, ch_f = ch, b_f = b;  // coordinates of the item two steps ahead (the one a release refills)
  if (tid == 0 && item < S.total) issue(tile, ch, b, 0);
  advance(tile_f, ch_f, b_f);
  if (tid == 0 && item + nctas < S.total) issue(tile_f, ch_f, b_f, 1);
  advance(tile_f, ch_f, b_f);
  int buf = 0, ybuf = 0;
  uint32_t ph0 = 0, ph1 = 0;
  const int ssA = warp * G::kWarpRows;  // first tile row of this warp's half A; half B starts kSeg rows later
  for (; item < S.total; item += nctas, advance(tile, ch, b), advance(tile_f, ch_f, b_f)) {
    const int qt = tile * G::kRows;
    const bool edge = (tile == 0) || (qt + G::kRows + G::kHalo > S.L);
    const bool active = qt + ssA < S.L;  // warp-uniform
    sw_mbar_wait(bar0 + 8 * buf, buf ? ph1 : ph0);
    if (buf) ph1 ^= 1; else ph0 ^= 1;
    float* xt = buf ? xs1 : xs0;
    unsigned char* yt = ys0 + (size_t)ybuf * kImg * G::kWarpYBytes;
    if (active) {
      float* xw = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(xt) + (size_t)ssA * (IN16 ? 16 : 32));
      snake_mma_unit<SPLIT_X, NB, IN16, SPLIT_OUT>(F, xw, yt, qt + ssA, S.L, ch, S.a, S.inv_b, S.filt, edge, -ssA,
                                                   G::kXRows - ssA, lane, guard, yt + G::kWarpYBytes);
    }
    // generic-proxy accesses of this warp (window reads / patches, output image writes) before the async proxy's
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    // the bulk store of the previous tile reads this warp's other image, which the next tile rewrites
    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncwarp();
    if (lane == 0) {
      if (active) {
        const int nrows = min(G::kWarpRows, S.L - qt - ssA);
        const unsigned short* dst = (const unsigned short*)S.y + (long long)b * S.y_batch_stride +
                                    (long long)ch * S.chunk_stride + (long long)(S.row0 + qt + ssA) * 8;
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(sw_u32(yt)),
                     "r"((uint32_t)nrows * 16u)
                     : "memory");
        if (SPLIT_OUT)
          asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst + S.lo_offset),
                       "r"(sw_u32(yt + G::kWarpYBytes)), "r"((uint32_t)nrows * 16u)
                       : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
      // release the window; the last of the four warps refills it with the tile after next
      __threadfence_block();
      if (atomicAdd(&released[buf], 1) == G::kWarps - 1) {
        released[buf] = 0;  // next touched after the refill below has landed and been consumed
        __threadfence_block();
        if (item + 2 * nctas < S.total) {
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          issue(tile_f, ch_f, b_f, buf);
        }
      }
    }
    buf ^= 1;
    ybuf ^= 1;
  }
  if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
  guard.commit(S.status, 1);
}

}  // namespace fh
