// tcgen05 / TMEM implicit-GEMM tapped convolution for sm_100a.
//
// One kernel serves every GEMM-shaped op of the hot path: the BigVGAN Conv1d / dilated Conv1d
// (bigvgan/models.py:27-43), the ConvTranspose1d upsamplers in polyphase form (models.py:140-146)
// and the backbone Linear layers (k = 1; flow.py:239,261, attend.py:176,189, transformer.py:100-103).
//
// Data layout ("chunked"): an activation [L, C] is stored as [C/8][Lp][8] bf16, so the 8 channels
// of one time step are one 16-byte row and 8 consecutive time steps x 8 channels are one
// contiguous 128-byte tcgen05 core matrix (no-swizzle, K-major canonical layout
// ((8,m),(8,2)):((16B,SBO=128B),(1,LBO))).  Consequences:
//   * a (128 + halo)-row window of one chunk is ONE cp.async.bulk (UBLKCP) of contiguous bytes;
//   * every convolution tap reads the SAME shared-memory window through a descriptor whose start
//     address is shifted by tap_offset*16 B -- the activation tile is fetched once per k taps;
//   * the two 8-channel halves of a K=16 MMA step are addressed by LBO, so no im2col, no swizzle.
// Weights are pre-packed on the host into the exact shared-memory image (packing.py), one bulk
// copy per stage.  Accumulators live in TMEM (2 x bn columns, double buffered across tiles);
// the epilogue (bias, alpha, residual, accumulate, GEGLU, bf16/fp32, chunked or row-major output)
// reads them with tcgen05.ld.  Warp roles: warp 0 = bulk-copy producer, warp 1 = MMA issuer +
// TMEM allocator, warps 2.. = epilogue (8 by default; 12 / 16 for the narrow HBM-bound shapes, whose
// residual rows additionally stream through a per-warp cp.async ring).  Persistent CTAs, static tile striding.
#include "common.cuh"
#include "tc_ptx.cuh"

namespace {

constexpr int kMaxTapOff = 64;
constexpr int kMaxSpan = 64;                   // max (max_off - min_off) of the taps of one phase
constexpr int kMaxStages = 8;
constexpr int kThreads = 320;                  // 10 warps: producer, MMA, 8 epilogue

struct TcParams {
  const __nv_bfloat16* a;
  const __nv_bfloat16* w;
  const float* bias;
  const void* res;
  void* out;
  long long a_batch, a_chunk;
  long long out_batch, out_chunk, out_row;
  long long res_batch, res_chunk, res_row;
  int a_row0;
  int out_is_16, res_is_16, fp16, accumulate, geglu;
  const float* acc_src;  // accumulate source when it is not the output itself (fp32, output geometry); else nullptr
  int act_gelu;        // exact-erf GELU on (acc + bias) * alpha before the residual (ConvNeXt pwconv1)
  float alpha, beta_res;
  int B, L, Cin, Cout, ntaps, P, bn;
  int m_tiles, n_tiles, total_tiles;
  int ci_pairs;        // ceil(Cin / 16)
  int ci_odd;          // Cin % 16 == 8: the last pair has one real 8-channel chunk; its partner is a zeroed smem window
  int tap_pair;        // ci_odd: the odd chunk's taps are issued two per MMA (K halves = two taps; mma_role)
  int tg, n_groups;    // taps per smem stage, groups per ci-pair
  int kc;              // ci-pairs per smem stage (> 1 only when a stage holds all taps: few-tap convs, Linear)
  int msub;            // 128-row sub-tiles per CTA tile (1, 2, 4 or 8): B operand reuse + epilogue MLP
  int acc_stages;      // TMEM accumulator stages: 2 (epilogue overlaps the next tile) or 1 (msub*bn > 256)
  int wrows;           // rows fetched per chunk window: 128*msub + (max_off - min_off)
  int arows_pad;       // rows reserved per chunk window in an A slot
  int stages, stage_bytes;
  // empty_ring, m_stride and m_valid are always stages, 128 msub and 128 msub.  They stay fields: folding them into the
  // kernels moves the spills of tc_conv_kernel<16> and the register count of tc_conv2_kernel.
  int empty_ring;       // number of "stage consumed" barriers the MMA issuer cycles through
  int min_off[16];
  int tap_rel0[16];     // (offset of tap 0) - min_off of the phase
  int tap_step[16];     // offset(tap j+1) - offset(tap j) when the taps of a phase form an arithmetic sequence
  int fast_epi;         // epilogue_fast applies (bias table in shared memory behind the stages)
  int res_async;        // residual rows through the per-warp cp.async ring at ring_off (epilogue_fast<.., RES_ASYNC>)
  int ring_off;
  int epi_warps;        // 8 or 16 (tc_conv_kernel<EW>)
  int v8;               // fp32 output / residual rows are 32-byte aligned: 256-bit epilogue accesses
  int tap_arith;        // all phases arithmetic: the MMA issuer strides descriptors instead of reading the offset table
  int tap_off[kMaxTapOff];
  unsigned int* err_flag;
  unsigned int* status;  // overflow / NaN status word of the caller (common.cuh Guard16) or nullptr
  int two_cta;            // tc_conv2_kernel: CTA pairs share every weight slot (cta_group::2 MMA, M = 256)
  int m_stride, m_valid;  // output rows a tile advances by / keeps
};


struct TileCoord {
  int b, p, mt, nt;
};
__device__ __forceinline__ TileCoord decode_tile(const TcParams& P, int id) {
  TileCoord c;
  if (P.two_cta) {
    // ids 2k / 2k + 1 = the two M tiles of one CTA pair (same batch, phase and N tile): a CTA steps by an even grid,
    // so the parity of its ids is its rank in the pair.  m_tiles counts PAIRS here; mt may point past L (void tile).
    const int r = id & 1;
    id >>= 1;
    c.nt = id % P.n_tiles;
    id /= P.n_tiles;
    c.mt = 2 * (id % P.m_tiles) + r;
    id /= P.m_tiles;
    c.p = id % P.P;
    c.b = id / P.P;
    return c;
  }
  c.nt = id % P.n_tiles;
  id /= P.n_tiles;
  c.mt = id % P.m_tiles;
  id /= P.m_tiles;
  c.p = id % P.P;
  c.b = id / P.P;
  return c;
}

__device__ __forceinline__ float gelu_f(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }

// ------------------------------------------------------------------------------ the kernel
// residual rows for one 16-column group (two 8-channel chunks) of one output row
__device__ __forceinline__ void load_res16(const TcParams& P, long long rbase, int n0, bool ok, float (&r)[16]) {
#pragma unroll
  for (int hh = 0; hh < 2; ++hh) {
    const int n = n0 + hh * 8;
    if (!ok || n >= P.Cout) {
#pragma unroll
      for (int i = 0; i < 8; ++i) r[hh * 8 + i] = 0.f;
      continue;
    }
    const long long ridx = rbase + (long long)(n >> 3) * P.res_chunk;
    if (P.res_is_16) {
      const uint4 raw = *reinterpret_cast<const uint4*>((const unsigned short*)P.res + ridx);
      const uint32_t* h = reinterpret_cast<const uint32_t*>(&raw);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 f = fh::unpack16(h[i], P.fp16);
        r[hh * 8 + 2 * i] = f.x;
        r[hh * 8 + 2 * i + 1] = f.y;
      }
    } else if (P.v8) {
      float t[8];
      ldg_v8((const float*)P.res + ridx, t);
#pragma unroll
      for (int i = 0; i < 8; ++i) r[hh * 8 + i] = t[i];
    } else {
      const float4* rp = reinterpret_cast<const float4*>((const float*)P.res + ridx);
      const float4 r0 = rp[0], r1 = rp[1];
      r[hh * 8 + 0] = r0.x, r[hh * 8 + 1] = r0.y, r[hh * 8 + 2] = r0.z, r[hh * 8 + 3] = r0.w;
      r[hh * 8 + 4] = r1.x, r[hh * 8 + 5] = r1.y, r[hh * 8 + 6] = r1.z, r[hh * 8 + 7] = r1.w;
    }
  }
}

struct GroupIter {  // (sub-tile, 16-column group) of the groups one epilogue warp owns, in consumption order
  int sub, g;
  __device__ __forceinline__ void start(int first, int gps) {
    sub = 0;
    g = first;
    norm(gps);
  }
  __device__ __forceinline__ void norm(int gps) {
    while (g >= gps) {
      g -= gps;
      ++sub;
    }
  }
  __device__ __forceinline__ void step(int by, int gps) {
    g += by;
    norm(gps);
  }
};

// Epilogue role, shared by both kernels.  `gstep` warps share one TMEM lane group (a warp may only touch lanes
// 32*(warp%4)..+31) and split the 16-column groups of a tile round-robin (`half` = index within the share).
// Per warp the groups are software-pipelined: tcgen05.ld and the residual loads of the next group are in flight
// while the current group is scaled, added and stored.
__device__ __forceinline__ void epilogue_role(const TcParams& P, uint32_t tmem_base, uint32_t tfull0, uint32_t tempty0,
                                              int lane_grp, int half, int gstep, int lane, int tile_rows,
                                              uint32_t acc_cols) {
  const int r = lane_grp * 32 + lane;
  int as = 0, aphase = 0;
  const int groups_per_sub = P.bn >> 4;
  const bool use_res = P.res != nullptr && !P.geglu;
  fh::Guard16 guard;
  for (int tile = blockIdx.x; tile < P.total_tiles; tile += gridDim.x) {
    const TileCoord tc = decode_tile(P, tile);
    const int n_base = tc.nt * P.bn;
    const int t_base = tc.mt * tile_rows + r;
    const int t_lim = min(P.L, tc.mt * tile_rows + P.m_valid);  // rows this tile keeps
    const long long res_b = (long long)tc.b * P.res_batch;
    const long long out_b = (long long)tc.b * P.out_batch;
    const uint32_t taddr = tmem_base + ((uint32_t)(lane_grp * 32) << 16) + (uint32_t)as * acc_cols;

    // a group is a running (sub-tile, 16-column group) pair: no division per group (see epilogue_fast)
    auto fetch_res = [&](const GroupIter& it, float (&rr)[16]) {
      if (!use_res || it.sub >= P.msub) return;
      const int t = t_base + (it.sub << 7);
      load_res16(P, res_b + ((long long)t * P.P + tc.p) * P.res_row, n_base + (it.g << 4), t < t_lim, rr);
    };
    auto issue_ld = [&](const GroupIter& it, uint32_t (&v)[16]) {
      if (it.sub >= P.msub) return;
      const int c0 = it.g << 4;
      if (n_base + c0 < P.Cout) tmem_ld16(taddr + (uint32_t)(it.sub * P.bn + c0), v);  // warp-uniform
    };
    auto finish = [&](const GroupIter& it, const uint32_t (&v)[16], const float (&rr)[16]) {
      const int c0 = it.g << 4, t = t_base + (it.sub << 7);
      if (it.sub >= P.msub || n_base + c0 >= P.Cout || t >= t_lim) return;
      const long long orow = (long long)t * P.P + tc.p;
      if (P.geglu) {
        // columns (2i, 2i+1) = (x_i, gate_i) -> gelu(gate) * x ; 16 columns -> one 8-channel chunk
        const int n_out = (n_base + c0) >> 1;
        float o[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int n = n_base + c0 + 2 * i;
          float xv = __uint_as_float(v[2 * i]), gv = __uint_as_float(v[2 * i + 1]);
          if (P.bias) {
            xv += __ldg(P.bias + n);
            gv += __ldg(P.bias + n + 1);
          }
          o[i] = gelu_f(gv) * xv;
        }
        const long long idx = out_b + (long long)(n_out >> 3) * P.out_chunk + orow * P.out_row;
        if (P.out_is_16) {
          uint32_t h[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            h[i] = fh::pack16(o[2 * i], o[2 * i + 1], P.fp16);
            guard.see(h[i], P.fp16);
          }
          *reinterpret_cast<uint4*>((unsigned short*)P.out + idx) = *reinterpret_cast<uint4*>(h);
        } else {
          float4* dst = reinterpret_cast<float4*>((float*)P.out + idx);
          dst[0] = make_float4(o[0], o[1], o[2], o[3]);
          dst[1] = make_float4(o[4], o[5], o[6], o[7]);
        }
        return;
      }
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        const int n0 = n_base + c0 + hh * 8;
        if (n0 >= P.Cout) break;
        float o[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          float acc = __uint_as_float(v[hh * 8 + i]);
          if (P.bias) acc += __ldg(P.bias + n0 + i);
          o[i] = acc * P.alpha;
          if (P.act_gelu) o[i] = gelu_f(o[i]);
          if (use_res) o[i] = fmaf(P.beta_res, rr[hh * 8 + i], o[i]);
        }
        const long long idx = out_b + (long long)(n0 >> 3) * P.out_chunk + orow * P.out_row;
        if (P.out_is_16) {
          uint32_t h[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            h[i] = fh::pack16(o[2 * i], o[2 * i + 1], P.fp16);
            guard.see(h[i], P.fp16);
          }
          *reinterpret_cast<uint4*>((unsigned short*)P.out + idx) = *reinterpret_cast<uint4*>(h);
        } else if (P.v8) {
          float* dst = (float*)P.out + idx;
          if (P.accumulate) {
            float t[8];
            ldg_v8(dst, t);
#pragma unroll
            for (int i = 0; i < 8; ++i) o[i] += t[i];
          }
          stg_v8(dst, o);
        } else {
          float4* dst = reinterpret_cast<float4*>((float*)P.out + idx);
          if (P.accumulate) {
            const float4 p0 = dst[0], p1 = dst[1];
            o[0] += p0.x, o[1] += p0.y, o[2] += p0.z, o[3] += p0.w;
            o[4] += p1.x, o[5] += p1.y, o[6] += p1.z, o[7] += p1.w;
          }
          dst[0] = make_float4(o[0], o[1], o[2], o[3]);
          dst[1] = make_float4(o[4], o[5], o[6], o[7]);
        }
      }
    };

    uint32_t va[16], vb[16];
    float ra[16], rb[16];
    GroupIter ia, ib;
    ia.start(half, groups_per_sub);
    fetch_res(ia, ra);  // residual of the first group is requested BEFORE waiting for the accumulator
    mbar_wait(tfull0 + 8 * as, aphase, P.err_flag, 4);
    tc_fence_after();
    issue_ld(ia, va);
    while (ia.sub < P.msub) {
      tmem_ld_wait();
      ib = ia;
      ib.step(gstep, groups_per_sub);
      issue_ld(ib, vb);
      fetch_res(ib, rb);
      finish(ia, va, ra);
      if (ib.sub >= P.msub) break;
      tmem_ld_wait();
      ia = ib;
      ia.step(gstep, groups_per_sub);
      issue_ld(ia, va);
      fetch_res(ia, ra);
      finish(ib, vb, rb);
    }
    // all TMEM reads of this warp are complete (wait::ld above) -> release the accumulator
    tmem_ld_wait();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) {
      if (P.two_cta) mbar_arrive_cluster(mapa_u32(tempty0 + 8 * as, 0));  // the pair's MMA issuer lives in CTA 0
      else mbar_arrive(tempty0 + 8 * as);
    }
    if (++as == P.acc_stages) {
      as = 0;
      aphase ^= 1;
    }
  }
  if (P.out_is_16) guard.commit(P.status, P.fp16);
}

// Specialised epilogue for the hot vocoder / backbone shapes: fp32 output and residual in 32-byte-aligned rows, no GEGLU.
// The generic role above spends ~210 instructions per 16-column group (per-element __ldg of the bias, runtime flag tests);
// ncu showed the eight epilogue warps -- not HBM -- pacing the HBM-bound C <= 96 stages.  Here the bias (pre-multiplied by
// alpha) comes from a shared-memory table with broadcast 128-bit loads, the flags are template parameters, and a group
// costs ~45 instructions:  o = fma(acc, alpha, alpha * bias) [+ beta * residual] [+ previous output].
// OUT16: 16-bit output rows (16 bytes per chunk row, no residual / accumulate) -- the snake that follows a first AMP
// convolution reads them as MMA operands directly.
//
// Round 2, second pass (ncu source page of the C = 24 / 48 launches at B = 64, profiles/r2_ncu_hbm_convs.txt):
//  * two thirds of the ~125 instructions a group still cost were index arithmetic -- three integer divisions
//    (group -> sub-tile, column) and 64-bit address chains rebuilt from scratch for every group.  A group is now a
//    running (sub, g) pair (GroupIter) and every address is tile base + sub * sub_stride + g * group_stride.
//  * the residual launches sat on the first FFMA that consumes the residual row (39 % of all samples): with one group of
//    LDGs in flight per warp the residual stream is latency-bound (12 KB in flight per SM against ~1 us of DRAM latency).
//    RES_ASYNC: the residual rows of the next kResDepth groups are in flight as cp.async (LDGSTS) copies into a private
//    per-warp ring in shared memory, across tile boundaries; depth is set by cp.async.wait_group, not by the compiler's
//    scoreboard assignment (a register ring two groups deep measured no gain in round 2).  A warp's 32 rows of one
//    8-channel chunk are 1 KB of contiguous global memory: lane i copies 16-byte pieces i and i + 32, the owner of row r
//    reads pieces 2 r and 2 r + 1 back after wait_group + __syncwarp.
constexpr int kResLevelBytes = 2048;          // one group: 2 chunks x 32 rows x 32 bytes
// RD residual groups in flight per epilogue warp, RD + 1 ring levels (the level read in step k - 1 is refilled in step k):
// 3 with eight epilogue warps, 2 with twelve or sixteen (48 - 64 KB in flight per SM either way)
__host__ __device__ constexpr int res_depth(int epi_warps) { return epi_warps > 8 ? 2 : 3; }
__host__ __device__ constexpr int res_ring_bytes(int epi_warps) { return epi_warps * (res_depth(epi_warps) + 1) * kResLevelBytes; }

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// residual copy stream of one epilogue warp: runs kResDepth groups ahead of the consumer, across tiles
struct ResStream {
  int tile, sub, g;
  int t0, t_lim, n_base;
  long long base;  // element index of (row t0, chunk n_base / 8) of this tile's batch item
  bool live;
  __device__ __forceinline__ void open(const TcParams& P, int tile_, int tile_rows, int lane_grp, int half, int gps) {
    tile = tile_;
    live = tile < P.total_tiles;
    if (!live) return;
    const TileCoord tc = decode_tile(P, tile);
    n_base = tc.nt * P.bn;
    t0 = tc.mt * tile_rows + lane_grp * 32;
    t_lim = min(P.L, tc.mt * tile_rows + P.m_valid);
    base = (long long)tc.b * P.res_batch + (long long)t0 * 8 + (long long)(n_base >> 3) * P.res_chunk;
    sub = 0;
    g = half;
    while (g >= gps) {
      g -= gps;
      ++sub;
    }
  }
  // copies the rows of group (sub, g) into ring level `dst` (shared address) and commits one cp.async group
  __device__ __forceinline__ void issue(const TcParams& P, uint32_t dst, int lane) {
    if (live) {
      const int n0 = n_base + (g << 4);
      if (n0 < P.Cout) {
        const float* src = (const float*)P.res + base + (long long)sub * (128 * 8) + (long long)(2 * g) * P.res_chunk;
        const int row = t0 + sub * 128 + (lane >> 1);
        const bool two = n0 + 8 < P.Cout;
        if (row < t_lim) {
          cp_async16(dst + lane * 16, src + lane * 4);
          if (two) cp_async16(dst + 1024 + lane * 16, src + P.res_chunk + lane * 4);
        }
        if (row + 16 < t_lim) {
          cp_async16(dst + 512 + lane * 16, src + 128 + lane * 4);
          if (two) cp_async16(dst + 1536 + lane * 16, src + P.res_chunk + 128 + lane * 4);
        }
      }
    }
    cp_async_commit();
  }
  __device__ __forceinline__ void next(const TcParams& P, int tile_rows, int lane_grp, int half, int gstep, int gps) {
    if (!live) return;
    g += gstep;
    while (g >= gps) {
      g -= gps;
      ++sub;
    }
    if (sub >= P.msub) open(P, tile + gridDim.x, tile_rows, lane_grp, half, gps);
  }
};

template <bool HAS_RES, bool ACCUM, bool OUT16 = false, int RD = 0>
__device__ __forceinline__ void epilogue_fast(const TcParams& P, uint32_t tmem_base, uint32_t tfull0, uint32_t tempty0,
                                              int lane_grp, int half, int gstep, int lane, int tile_rows, uint32_t acc_cols,
                                              const float* s_bias, uint32_t ring) {
  const int r = lane_grp * 32 + lane;
  int as = 0, aphase = 0;
  const int gps = P.bn >> 4;  // 16-column groups per sub-tile
  const int msub = P.msub;
  const float alpha = P.alpha, beta = P.beta_res;
  const int bmask = P.bias ? ~0 : 0;  // no bias: every group reads the 16 zeros at the head of the table
  const float* resp = (const float*)P.res;
  float* outp = (float*)P.out;
  const float* accp = P.acc_src ? P.acc_src : (const float*)P.out;  // "previous output" rows of the accumulate form
  const long long res_rs = (long long)P.P * P.res_row, out_rs = (long long)P.P * P.out_row;
  const long long res_sub = 128 * res_rs, out_sub = 128 * out_rs;       // one sub-tile down
  const long long res_grp = 2 * P.res_chunk, out_grp = 2 * P.out_chunk;  // one 16-column group to the right
  const int fp16 = P.fp16;
  fh::Guard16 guard;
  constexpr bool RES_ASYNC = RD > 0;
  constexpr int kResDepth = RD, kResLevels = RD + 1;

  ResStream rs;
  int lvl = 0;  // ring level the consumer reads next
  if (RES_ASYNC) {
    ring += (uint32_t)((lane_grp * gstep + half) * (kResLevels * kResLevelBytes));
    rs.open(P, blockIdx.x, tile_rows, lane_grp, half, gps);
#pragma unroll
    for (int d = 0; d < kResDepth; ++d) {
      rs.issue(P, ring + d * kResLevelBytes, lane);
      rs.next(P, tile_rows, lane_grp, half, gstep, gps);
    }
  }

  for (int tile = blockIdx.x; tile < P.total_tiles; tile += gridDim.x) {
    const TileCoord tc = decode_tile(P, tile);
    const int n_base = tc.nt * P.bn;
    const int t_base = tc.mt * tile_rows + r;
    const int t_lim = min(P.L, tc.mt * tile_rows + P.m_valid);  // rows this tile keeps
    // element indices of (row t_base, chunk n_base / 8) in the residual and the output
    const long long res_0 = (long long)tc.b * P.res_batch + (long long)tc.p * P.res_row + (long long)t_base * res_rs +
                            (long long)(n_base >> 3) * P.res_chunk;
    const long long out_0 = (long long)tc.b * P.out_batch + (long long)tc.p * P.out_row + (long long)t_base * out_rs +
                            (long long)(n_base >> 3) * P.out_chunk;
    const uint32_t taddr = tmem_base + ((uint32_t)(lane_grp * 32) << 16) + (uint32_t)as * acc_cols;

    // a group is live for this thread when its columns exist and its row is kept
    auto live = [&](const GroupIter& it) { return n_base + (it.g << 4) < P.Cout && t_base + (it.sub << 7) < t_lim; };
    auto prefetch = [&](const GroupIter& it, float (&rr)[16], float (&pp)[16]) {
      if (it.sub >= msub || !live(it)) return;
      const bool two = n_base + (it.g << 4) + 8 < P.Cout;
      if (HAS_RES && !RES_ASYNC) {
        const float* q = resp + res_0 + it.sub * res_sub + it.g * res_grp;
        ldg_v8(q, *reinterpret_cast<float(*)[8]>(&rr[0]));
        if (two) ldg_v8(q + P.res_chunk, *reinterpret_cast<float(*)[8]>(&rr[8]));
      }
      if (ACCUM) {
        const float* q = accp + out_0 + it.sub * out_sub + it.g * out_grp;
        ldg_v8(q, *reinterpret_cast<float(*)[8]>(&pp[0]));
        if (two) ldg_v8(q + P.out_chunk, *reinterpret_cast<float(*)[8]>(&pp[8]));
      }
    };
    auto issue_ld = [&](const GroupIter& it, uint32_t (&v)[16]) {
      if (it.sub >= msub) return;
      if (n_base + (it.g << 4) < P.Cout) tmem_ld16(taddr + (uint32_t)(it.sub * P.bn + (it.g << 4)), v);  // warp-uniform
    };
    // RES_ASYNC: residual rows of the group consumed now -> registers; the freed level is refilled kResDepth groups ahead
    auto ring_step = [&](float (&rr)[16]) {
      cp_async_wait<(RD > 0 ? RD - 1 : 0)>();
      __syncwarp();
      const int fill = lvl == 0 ? kResLevels - 1 : lvl - 1;
      rs.issue(P, ring + (uint32_t)fill * kResLevelBytes, lane);
      rs.next(P, tile_rows, lane_grp, half, gstep, gps);
      const uint32_t src = ring + (uint32_t)lvl * kResLevelBytes + (uint32_t)lane * 32u;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const uint32_t a = src + (uint32_t)(q >> 1) * 1024u + (uint32_t)(q & 1) * 16u;
        asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];"
                     : "=f"(rr[4 * q]), "=f"(rr[4 * q + 1]), "=f"(rr[4 * q + 2]), "=f"(rr[4 * q + 3])
                     : "r"(a));
      }
      lvl = lvl == kResLevels - 1 ? 0 : lvl + 1;
    };
    auto finish = [&](const GroupIter& it, const uint32_t (&v)[16], const float (&rr)[16], const float (&pp)[16]) {
      if (!live(it)) return;
      const int n0 = n_base + (it.g << 4);
      const long long oidx = out_0 + it.sub * out_sub + it.g * out_grp;
      float* dst = outp + oidx;
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        if (hh == 1 && n0 + 8 >= P.Cout) break;
        const float4 b0 = *reinterpret_cast<const float4*>(s_bias + ((n0 + hh * 8) & bmask));
        const float4 b1 = *reinterpret_cast<const float4*>(s_bias + ((n0 + hh * 8) & bmask) + 4);
        const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
        float o[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          o[i] = fmaf(__uint_as_float(v[hh * 8 + i]), alpha, bb[i]);
          if (HAS_RES) o[i] = fmaf(beta, rr[hh * 8 + i], o[i]);
          if (ACCUM) o[i] += pp[hh * 8 + i];
        }
        if (OUT16) {
          uint32_t h[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            h[i] = fh::pack16(o[2 * i], o[2 * i + 1], fp16);
            guard.see(h[i], fp16);
          }
          *reinterpret_cast<uint4*>((unsigned short*)P.out + oidx + (long long)hh * P.out_chunk) = *reinterpret_cast<uint4*>(h);
        } else {
          stg_v8(dst + (long long)hh * P.out_chunk, o);
        }
      }
    };

    uint32_t va[16], vb[16];
    float ra[16], rb[16], pa[16], pb[16];
    GroupIter ia, ib;
    ia.start(half, gps);
    prefetch(ia, ra, pa);  // requested BEFORE waiting for the accumulator
    mbar_wait(tfull0 + 8 * as, aphase, P.err_flag, 4);
    tc_fence_after();
    issue_ld(ia, va);
    while (true) {
      tmem_ld_wait();
      ib = ia;
      ib.step(gstep, gps);
      issue_ld(ib, vb);
      prefetch(ib, rb, pb);
      if (RES_ASYNC) ring_step(ra);
      finish(ia, va, ra, pa);
      if (ib.sub >= msub) break;
      tmem_ld_wait();
      ia = ib;
      ia.step(gstep, gps);
      issue_ld(ia, va);
      prefetch(ia, ra, pa);
      if (RES_ASYNC) ring_step(rb);
      finish(ib, vb, rb, pb);
      if (ia.sub >= msub) break;
    }
    tmem_ld_wait();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) {
      if (P.two_cta) mbar_arrive_cluster(mapa_u32(tempty0 + 8 * as, 0));  // the pair's MMA issuer lives in CTA 0
      else mbar_arrive(tempty0 + 8 * as);
    }
    if (++as == P.acc_stages) {
      as = 0;
      aphase ^= 1;
    }
  }
  if (RES_ASYNC) cp_async_wait<0>();
  if (OUT16) guard.commit(P.status, fp16);
}

// MMA issuer role, shared by both kernels.  The ncu source page of the first version showed this warp, not the tensor
// pipe, pacing every shape but the widest (~300 cycles of uniform-datapath work per MMA: an integer modulo per stage,
// a shared-memory load + R2UR per tap, 64-bit descriptor arithmetic per MMA).  Here every per-stage and per-tap
// quantity is a running 32-bit value: stage base, tap stride (taps of a phase are an arithmetic sequence for Conv1d,
// dilated Conv1d and polyphase ConvTranspose1d), weight stride; the sub-tile loop is specialised outside the tap loop.
template <int MSUB, bool TWO = false>
__device__ __forceinline__ void issue_taps(uint32_t d_tmem, uint32_t bn, uint32_t a_lo, uint32_t a_step, uint32_t b_lo,
                                           uint32_t b_step, uint32_t hi, uint32_t idesc, uint32_t accum, int ntap) {
#pragma unroll 1
  for (int j = 0; j < ntap; ++j) {
#pragma unroll
    for (int sub = 0; sub < MSUB; ++sub) {
      if (TWO) umma2_f16_split(d_tmem + (uint32_t)sub * bn, a_lo + (uint32_t)sub * 128u, hi, b_lo, hi, idesc, accum);
      else umma_f16_split(d_tmem + (uint32_t)sub * bn, a_lo + (uint32_t)sub * 128u, hi, b_lo, hi, idesc, accum);
    }
    accum = 1;
    a_lo += a_step;
    b_lo += b_step;
  }
}

__device__ __forceinline__ void mma_role(const TcParams& P, uint32_t tmem_base, uint32_t full0, uint32_t empty0,
                                         uint32_t tfull0, uint32_t tempty0, uint32_t stage0, uint32_t a_chunk_bytes,
                                         const int* s_off) {
  const bool leader = elect_one();
  int stage = 0, phase = 0, as = 0, aphase = 0, estage = 0;
  const int EB = P.empty_ring;
  const int S = P.stages, msub = P.msub, ntaps = P.ntaps, tg = P.tg, n_groups = P.n_groups, ci_pairs = P.ci_pairs;
  const int kc = P.kc;
  const uint32_t bn = (uint32_t)P.bn;
  const uint32_t idesc = make_idesc(P.bn, P.fp16);
  const uint32_t hi = (128u >> 4) | (1u << 14);                 // SBO = 128 B, descriptor version 1 (bit 46)
  const uint32_t a_lbo = (a_chunk_bytes >> 4) << 16;            // LBO fields (bits 16..29 of the low word)
  const uint32_t b_lbo = ((bn * 16u) >> 4) << 16;
  const uint32_t b_step = (bn * 32u) >> 4;                      // one tap of weights
  const uint32_t a_slot_u = (2u * a_chunk_bytes) >> 4;
  const uint32_t stage_u = (uint32_t)P.stage_bytes >> 4, stage0_u = stage0 >> 4;
  const uint32_t acc_cols = (uint32_t)(P.msub * P.bn);
  const bool one_phase = P.P == 1;
  uint32_t rel0 = (uint32_t)P.tap_rel0[0], a_step = (uint32_t)P.tap_step[0];
  for (int tile = blockIdx.x; tile < P.total_tiles; tile += gridDim.x) {
    int ph = 0;
    if (!one_phase) {
      ph = decode_tile(P, tile).p;
      rel0 = (uint32_t)P.tap_rel0[ph];
      a_step = (uint32_t)P.tap_step[ph];
    }
    mbar_wait(tempty0 + 8 * as, aphase ^ 1, P.err_flag, 2);
    tc_fence_after();
    const uint32_t d_tmem = tmem_base + (uint32_t)as * acc_cols;
    uint32_t accum = 0;
    for (int cp = 0; cp < ci_pairs; cp += kc) {
      const int nkc = min(kc, ci_pairs - cp);
      int tap0 = 0;
      for (int g = 0; g < n_groups; ++g, tap0 += tg) {
        const int nt_g = min(tg, ntaps - tap0);
        mbar_wait(full0 + 8 * stage, phase, P.err_flag, 3);
        tc_fence_after();
        const uint32_t sa_u = stage0_u + (uint32_t)stage * stage_u;
        if (leader) {
          uint32_t b_lo = b_lbo | (sa_u + (uint32_t)kc * a_slot_u);  // weights sit behind the kc activation slots
          uint32_t a_base_lo = a_lbo | sa_u;
          for (int c = 0; c < nkc; ++c) {
            if (P.tap_pair && cp + c == ci_pairs - 1) {
              // Odd chunk count (24 channels): the last ci-pair has ONE real 8-channel chunk.  Instead of K = 16 MMAs whose
              // second K half is a zeroed partner window against zero weights, two TAPS share an MMA: K halves = (chunk @
              // tap 2j, chunk @ tap 2j + 1).  Both are descriptor choices on the data already in shared memory -- A: LBO =
              // one tap step on the same window, B: LBO = one tap slot (the first halves of two consecutive slots) -- so
              // neither the weight image nor the producer changes.  ceil(k / 2) instead of k MMAs for this pair (k = 11,
              // 24 channels: 17 instead of 22 per sub-tile; these launches are bound by MMA operand reads).  An odd last tap
              // keeps the old form (zero partner window, zero second half).
              const uint32_t a_pair = (a_step << 16) | ((a_base_lo & 0x3FFFu) + rel0 + (uint32_t)tap0 * a_step);
              const uint32_t b_pair = ((2u * bn) << 16) | (b_lo & 0x3FFFu);
              const int npair = nt_g >> 1;
              if (msub == 2) issue_taps<2>(d_tmem, bn, a_pair, 2u * a_step, b_pair, 2u * b_step, hi, idesc, accum, npair);
              else if (msub == 4) issue_taps<4>(d_tmem, bn, a_pair, 2u * a_step, b_pair, 2u * b_step, hi, idesc, accum, npair);
              else if (msub == 8) issue_taps<8>(d_tmem, bn, a_pair, 2u * a_step, b_pair, 2u * b_step, hi, idesc, accum, npair);
              else issue_taps<1>(d_tmem, bn, a_pair, 2u * a_step, b_pair, 2u * b_step, hi, idesc, accum, npair);
              if (nt_g & 1) {
                const uint32_t acc1 = npair > 0 ? 1u : accum;
                const uint32_t a_lo = a_base_lo + rel0 + (uint32_t)(tap0 + nt_g - 1) * a_step;
                const uint32_t b_1 = b_lo + (uint32_t)(nt_g - 1) * b_step;
                if (msub == 2) issue_taps<2>(d_tmem, bn, a_lo, a_step, b_1, b_step, hi, idesc, acc1, 1);
                else if (msub == 4) issue_taps<4>(d_tmem, bn, a_lo, a_step, b_1, b_step, hi, idesc, acc1, 1);
                else if (msub == 8) issue_taps<8>(d_tmem, bn, a_lo, a_step, b_1, b_step, hi, idesc, acc1, 1);
                else issue_taps<1>(d_tmem, bn, a_lo, a_step, b_1, b_step, hi, idesc, acc1, 1);
              }
            } else if (P.tap_arith) {
              const uint32_t a_lo = a_base_lo + rel0 + (uint32_t)tap0 * a_step;
              if (msub == 2) issue_taps<2>(d_tmem, bn, a_lo, a_step, b_lo, b_step, hi, idesc, accum, nt_g);
              else if (msub == 4) issue_taps<4>(d_tmem, bn, a_lo, a_step, b_lo, b_step, hi, idesc, accum, nt_g);
              else if (msub == 8) issue_taps<8>(d_tmem, bn, a_lo, a_step, b_lo, b_step, hi, idesc, accum, nt_g);
              else issue_taps<1>(d_tmem, bn, a_lo, a_step, b_lo, b_step, hi, idesc, accum, nt_g);
            } else {  // irregular tap offsets: table in shared memory
              const int* offs = s_off + ph * ntaps + tap0;
              uint32_t bl = b_lo, acc = accum;
              for (int j = 0; j < nt_g; ++j) {
                const uint32_t a_lo = a_base_lo + (uint32_t)offs[j];
                for (int sub = 0; sub < msub; ++sub)
                  umma_f16_split(d_tmem + (uint32_t)sub * bn, a_lo + (uint32_t)sub * 128u, hi, bl, hi, idesc, acc);
                acc = 1;
                bl += b_step;
              }
            }
            accum = 1;
            a_base_lo += a_slot_u;
            b_lo += (uint32_t)nt_g * b_step;
          }
          umma_commit(empty0 + 8 * estage);  // frees the smem stage when these MMAs retire
        }
        accum = 1;
        __syncwarp();
        if (++estage == EB) estage = 0;
        if (++stage == S) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
    if (leader) umma_commit(tfull0 + 8 * as);  // accumulator complete -> epilogue
    __syncwarp();
    if (++as == P.acc_stages) {
      as = 0;
      aphase ^= 1;
    }
  }
}

// Bulk-copy producer role (one elected lane): per stage, the (rows + span)-row window of each 8-channel chunk and the
// packed weights of the stage's taps, all signalled on the stage's full barrier.
__device__ __forceinline__ void producer_role(const TcParams& P, uint32_t full0, uint32_t empty0, uint32_t stage0,
                                              uint32_t a_chunk_bytes, int tile_rows) {
  const int S = P.stages;
  const uint32_t b_tap_bytes = (uint32_t)P.bn * 32u;
  const uint32_t a_slot_bytes = 2u * a_chunk_bytes;
  int stage = 0, phase = 0;
  for (int tile = blockIdx.x; tile < P.total_tiles; tile += gridDim.x) {
    const TileCoord tc = decode_tile(P, tile);
    const long long row = (long long)P.a_row0 + (long long)tc.mt * tile_rows + P.min_off[tc.p];
    const __nv_bfloat16* a_base = P.a + (long long)tc.b * P.a_batch + row * 8;
    // packed weights: [p][nt][cp][tap][2][bn][8]
    const __nv_bfloat16* w_base =
        P.w + ((long long)(tc.p * P.n_tiles + tc.nt) * P.ci_pairs) * ((long long)P.ntaps * P.bn * 16);
    for (int cp = 0; cp < P.ci_pairs; cp += P.kc) {
      const int nkc = min(P.kc, P.ci_pairs - cp);
      for (int g = 0; g < P.n_groups; ++g) {
        const int tap0 = g * P.tg;
        const int nt_g = min(P.tg, P.ntaps - tap0);
        mbar_wait(empty0 + 8 * stage, phase ^ 1, P.err_flag, 1);
        const uint32_t sa = stage0 + (uint32_t)stage * (uint32_t)P.stage_bytes;
        const uint32_t fb = full0 + 8 * stage;
        const uint32_t a_bytes = (uint32_t)P.wrows * 16u;
        const int nchunk = 2 * nkc - ((P.ci_odd && cp + nkc == P.ci_pairs) ? 1 : 0);
        const uint32_t w_bytes = (uint32_t)(nkc * nt_g) * b_tap_bytes;  // kc > 1 only with n_groups == 1: contiguous
        mbar_expect_tx(fb, (uint32_t)nchunk * a_bytes + w_bytes);
        for (int c = 0; c < nchunk; ++c)
          bulk_g2s(sa + (uint32_t)c * a_chunk_bytes, a_base + (long long)(2 * cp + c) * P.a_chunk, a_bytes, fb);
        bulk_g2s(sa + (uint32_t)P.kc * a_slot_bytes, w_base + ((long long)cp * P.ntaps + tap0) * ((long long)P.bn * 16),
                 w_bytes, fb);
        if (++stage == S) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  }
}

template <int EW = 8>
__device__ __forceinline__ void epilogue_dispatch(const TcParams& P, uint32_t tmem_base, uint32_t tfull0, uint32_t tempty0,
                                                  int lg, int hf, int lane, int tile_rows, uint32_t acc_cols,
                                                  const float* s_bias, int gstep = 2, uint32_t ring = 0) {
#define FH_EPI(...) epilogue_fast<__VA_ARGS__>(P, tmem_base, tfull0, tempty0, lg, hf, gstep, lane, tile_rows, acc_cols, s_bias, ring)
  constexpr int RD = res_depth(EW);
  if (P.fast_epi) {
    if (P.res_async && ring != 0) {  // residual rows through the cp.async ring (plain kernel, P == 1, fp32 residual)
      if (P.out_is_16 && P.accumulate) FH_EPI(true, true, true, RD);
      else if (P.accumulate) FH_EPI(true, true, false, RD);
      else FH_EPI(true, false, false, RD);
    } else if (P.out_is_16 && P.accumulate)  // last AMP branch of a stage: mean of the branches written as the next stage's operand
      FH_EPI(true, true, true);
    else if (P.out_is_16) FH_EPI(false, false, true);
    else if (P.res != nullptr && P.accumulate) FH_EPI(true, true);
    else if (P.res != nullptr) FH_EPI(true, false);
    else if (P.accumulate) FH_EPI(false, true);
    else FH_EPI(false, false);
  } else if (EW == 8) {
    epilogue_role(P, tmem_base, tfull0, tempty0, lg, hf, gstep, lane, tile_rows, acc_cols);
  } else {
    __trap();  // the 16-epilogue-warp kernel is only planned with the specialised epilogue
  }
#undef FH_EPI
}

// Per-CTA setup shared by the conv kernels: mbarriers, tap-offset table, alpha * bias table, zeroed partner windows.
// The caller allocates TMEM and issues the __syncthreads that publishes all of it.
__device__ __forceinline__ void conv_cta_setup(const TcParams& P, unsigned char* smem, int nthreads, int epi_warps) {
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem);
  const uint32_t full0 = smem_u32(bars), empty0 = full0 + 8 * kMaxStages;
  const uint32_t tfull0 = empty0 + 8 * kMaxStages, tempty0 = tfull0 + 16;
  const int S = P.stages;
  if (threadIdx.x == 0) {
    for (int i = 0; i < S; ++i) mbar_init(full0 + 8 * i, 1);
    for (int i = 0; i < P.empty_ring; ++i) mbar_init(empty0 + 8 * i, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(tfull0 + 8 * i, 1);
      mbar_init(tempty0 + 8 * i, epi_warps);
    }
    fence_barrier_init();
  }
  if (threadIdx.x >= 64 && threadIdx.x < 64 + P.P * P.ntaps) {
    const int i = threadIdx.x - 64;
    reinterpret_cast<int*>(smem + 512)[i] = P.tap_off[i] - P.min_off[i / P.ntaps];
  }
  if (P.fast_epi) {  // alpha * bias for every output channel of this launch (16 zeros when there is no bias)
    float* sb = reinterpret_cast<float*>(smem + 1024 + (size_t)S * P.stage_bytes);
    const int n = P.bias ? ((P.n_tiles * P.bn + 15) & ~15) : 16;
    for (int i = threadIdx.x; i < n; i += nthreads) sb[i] = (P.bias && i < P.Cout) ? P.alpha * __ldg(P.bias + i) : 0.f;
  }
  if (P.ci_odd) {
    // Odd chunk count (e.g. 24 channels): the partner window of the last chunk is never fetched.  Its weights are
    // zero, so it only has to hold finite values: zero every stage's second windows once (stale activations of other
    // pairs that land there later are finite as well).
    const uint32_t cb = (uint32_t)P.arows_pad * 16u;
    for (int st = 0; st < S * P.kc; ++st) {
      uint4* z = reinterpret_cast<uint4*>(smem + 1024 + (size_t)(st / P.kc) * P.stage_bytes + (size_t)(2 * (st % P.kc) + 1) * cb);
      for (uint32_t i = threadIdx.x; i < cb / 16u; i += nthreads) z[i] = make_uint4(0u, 0u, 0u, 0u);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
}

// EW = epilogue warps: 8 (default), or 16 for the HBM-bound narrow shapes whose epilogue -- two warps per scheduler,
// each issuing once every ~5 cycles (ncu: issue-active 40 %, stalls = fixed-latency dependencies) -- paced the launch.
template <int EW>
__global__ void __launch_bounds__(64 + 32 * EW, 1) tc_conv_kernel(const __grid_constant__ TcParams P) {
  extern __shared__ __align__(1024) unsigned char smem[];
  // [0,256): barriers; [256,260): tmem base; [512,768): tap offsets; stages from 1024; bias table behind the stages
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem);
  const uint32_t full0 = smem_u32(bars), empty0 = full0 + 8 * kMaxStages;
  const uint32_t tfull0 = empty0 + 8 * kMaxStages, tempty0 = tfull0 + 16;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 8 * (2 * kMaxStages + 4));
  const uint32_t stage0 = smem_u32(smem + 1024);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  conv_cta_setup(P, smem, 64 + 32 * EW, EW);
  if (warp == 1) tmem_alloc(smem_u32(tmem_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  int* s_off = reinterpret_cast<int*>(smem + 512);  // [P][ntaps] tap offsets relative to the phase minimum

  const uint32_t a_chunk_bytes = (uint32_t)P.arows_pad * 16u;  // one chunk window slot
  const int tile_rows = 128 * P.msub;
  const uint32_t acc_cols = (uint32_t)(P.msub * P.bn);   // TMEM columns of one accumulator stage

  if (warp == 0) {
    // ===================================================================== producer
    if (lane == 0) producer_role(P, full0, empty0, stage0, a_chunk_bytes, tile_rows);
  } else if (warp == 1) {
    // ===================================================================== MMA issuer
    mma_role(P, tmem_base, full0, empty0, tfull0, tempty0, stage0, a_chunk_bytes, s_off);
  } else {
    // ===================================================================== epilogue (warps 2..9)
    epilogue_dispatch<EW>(P, tmem_base, tfull0, tempty0, warp & 3, (warp - 2) >> 2, lane, tile_rows, acc_cols,
                          reinterpret_cast<const float*>(smem + 1024 + (size_t)P.stages * P.stage_bytes), EW / 4,
                      P.res_async ? smem_u32(smem + P.ring_off) : 0u);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------ CTA-pair variant (cta_group::2)
// Same implicit GEMM with the two SMs of a TPC as one MMA unit: the pair owns two adjacent 128 msub-row M tiles (one per
// CTA: own activation windows, own TMEM accumulators, own epilogue) and ONE weight stream -- each CTA fetches half of
// every weight slot (bn / 2 rows) and `tcgen05.mma.cta_group::2` (M = 256), issued by CTA 0's MMA thread, reads the A
// windows and the B halves of both CTAs.  Per SM the L2 -> SM weight traffic and the number of MMA instructions halve
// (ncu: the 192 / 384-channel shapes and the Linear layers are paced by the weight stream, the <= 48-channel shapes by the
// ~32-cycle fixed cost of an MMA).  Protocol on top of tc_conv_kernel's:
//   * "stage full": CTA 0 waits for its own loads AND for the peer's -- a relay warp in CTA 1 waits on CTA 1's local full
//     barrier and arrives remotely on CTA 0's `peerfull` barrier (bulk copies can only signal a barrier of their own CTA);
//   * "stage consumed" and "accumulator complete": tcgen05.commit multicast to the same barrier offset in both CTAs;
//   * "accumulator drained": the epilogue warps of both CTAs arrive on CTA 0's barrier (count 16);
//   * cluster barrier after the mbarrier inits and before TMEM dealloc / exit.
// Weights are packed per CTA rank ([p][nt][cp][rank][tap][2][bn / 2][8], packing.py two_cta).
constexpr int kThreads2 = 352;  // + relay warp

__device__ __forceinline__ uint32_t make_idesc2(int n, int fp16) {
  const uint32_t fmt = fp16 ? 0u : 1u;
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(n >> 3) << 17) | ((256u >> 4) << 24);
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads2, 1) tc_conv2_kernel(const __grid_constant__ TcParams P) {
  extern __shared__ __align__(1024) unsigned char smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem);
  const uint32_t full0 = smem_u32(bars), empty0 = full0 + 8 * kMaxStages;
  const uint32_t tfull0 = empty0 + 8 * kMaxStages, tempty0 = tfull0 + 16;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 8 * (2 * kMaxStages + 4));
  const uint32_t peerfull0 = smem_u32(smem + 192);
  const uint32_t stage0 = smem_u32(smem + 1024);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int S = P.stages;

  conv_cta_setup(P, smem, kThreads2, 16);  // tempty: 8 epilogue warps of each CTA arrive on CTA 0's barrier
  if (threadIdx.x == 0) {
    for (int i = 0; i < S; ++i) mbar_init(peerfull0 + 8 * i, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc2(smem_u32(tmem_slot), 512);
  tc_fence_before();
  cluster_sync_all();  // both CTAs' barriers exist before any remote arrive / multicast commit
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const uint32_t a_chunk_bytes = (uint32_t)P.arows_pad * 16u;
  const uint32_t a_slot_bytes = 2u * a_chunk_bytes;
  const int tile_rows = 128 * P.msub;
  const uint32_t acc_cols = (uint32_t)(P.msub * P.bn);
  const uint32_t hbn = (uint32_t)P.bn >> 1;             // weight rows per CTA
  const uint32_t b_tap_bytes = hbn * 32u;
  const int steps_per_tile = ((P.ci_pairs + P.kc - 1) / P.kc) * P.n_groups;

  if (warp == 0) {
    // ===================================================================== producer: own A windows + own half of the weights
    if (lane == 0) {
      int stage = 0, phase = 0;
      for (int tile = blockIdx.x; tile < P.total_tiles; tile += gridDim.x) {
        const TileCoord tc = decode_tile(P, tile);
        const long long row = (long long)P.a_row0 + (long long)tc.mt * tile_rows + P.min_off[tc.p];
        const bool has_a = (long long)tc.mt * tile_rows < P.L;  // void tile of an odd tail: weights only
        const __nv_bfloat16* a_base = P.a + (long long)tc.b * P.a_batch + row * 8;
        // packed weights: [p][nt][cp][rank][tap][2][bn / 2][8]
        const __nv_bfloat16* w_base = P.w + ((long long)(tc.p * P.n_tiles + tc.nt) * P.ci_pairs) * ((long long)P.ntaps * P.bn * 16);
        for (int cp = 0; cp < P.ci_pairs; cp += P.kc) {
          const int nkc = min(P.kc, P.ci_pairs - cp);
          for (int g = 0; g < P.n_groups; ++g) {
            const int tap0 = g * P.tg;
            const int nt_g = min(P.tg, P.ntaps - tap0);
            mbar_wait(empty0 + 8 * stage, phase ^ 1, P.err_flag, 1);
            const uint32_t sa = stage0 + (uint32_t)stage * (uint32_t)P.stage_bytes;
            const uint32_t fb = full0 + 8 * stage;
            const uint32_t a_bytes = (uint32_t)P.wrows * 16u;
            const int nchunk = has_a ? 2 * nkc - ((P.ci_odd && cp + nkc == P.ci_pairs) ? 1 : 0) : 0;
            const uint32_t w_bytes = (uint32_t)nt_g * b_tap_bytes;  // per ci-pair
            mbar_expect_tx(fb, (uint32_t)nchunk * a_bytes + (uint32_t)nkc * w_bytes);
            for (int c = 0; c < nchunk; ++c)
              bulk_g2s(sa + (uint32_t)c * a_chunk_bytes, a_base + (long long)(2 * cp + c) * P.a_chunk, a_bytes, fb);
            for (int c = 0; c < nkc; ++c)
              bulk_g2s(sa + (uint32_t)P.kc * a_slot_bytes + (uint32_t)c * w_bytes,
                       w_base + ((long long)((cp + c) * 2 + (int)rank) * P.ntaps + tap0) * ((long long)hbn * 16), w_bytes, fb);
            if (++stage == S) {
              stage = 0;
              phase ^= 1;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================================================================== MMA issuer: CTA 0 only
    if (rank == 0) {
      const bool leader = elect_one();
      int stage = 0, phase = 0, as = 0, aphase = 0;
      const int msub = P.msub, ntaps = P.ntaps, tg = P.tg, n_groups = P.n_groups, ci_pairs = P.ci_pairs, kc = P.kc;
      const uint32_t bn = (uint32_t)P.bn;
      const uint32_t idesc = make_idesc2(P.bn, P.fp16);
      const uint32_t hi = (128u >> 4) | (1u << 14);
      const uint32_t a_lbo = (a_chunk_bytes >> 4) << 16;
      const uint32_t b_lbo = ((hbn * 16u) >> 4) << 16;
      const uint32_t b_step = (hbn * 32u) >> 4;
      const uint32_t a_slot_u = (2u * a_chunk_bytes) >> 4;
      const uint32_t stage_u = (uint32_t)P.stage_bytes >> 4, stage0_u = stage0 >> 4;
      const int* s_off = reinterpret_cast<const int*>(smem + 512);
      for (int tile = blockIdx.x; tile < P.total_tiles; tile += gridDim.x) {
        const int ph = decode_tile(P, tile).p;
        const uint32_t rel0 = (uint32_t)P.tap_rel0[ph], a_step = (uint32_t)P.tap_step[ph];
        mbar_wait(tempty0 + 8 * as, aphase ^ 1, P.err_flag, 2);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)as * acc_cols;
        uint32_t accum = 0;
        for (int cp = 0; cp < ci_pairs; cp += kc) {
          const int nkc = min(kc, ci_pairs - cp);
          int tap0 = 0;
          for (int g = 0; g < n_groups; ++g, tap0 += tg) {
            const int nt_g = min(tg, ntaps - tap0);
            mbar_wait(full0 + 8 * stage, phase, P.err_flag, 3);
            mbar_wait(peerfull0 + 8 * stage, phase, P.err_flag, 8);
            tc_fence_after();
            const uint32_t sa_u = stage0_u + (uint32_t)stage * stage_u;
            if (leader) {
              uint32_t b_lo = b_lbo | (sa_u + (uint32_t)kc * a_slot_u);
              uint32_t a_base_lo = a_lbo | sa_u;
              for (int c = 0; c < nkc; ++c) {
                if (P.tap_arith) {  // same lean issue loop as the single-CTA kernel: running 32-bit descriptor words
                  const uint32_t a_lo = a_base_lo + rel0 + (uint32_t)tap0 * a_step;
                  if (msub == 2) issue_taps<2, true>(d_tmem, bn, a_lo, a_step, b_lo, b_step, hi, idesc, accum, nt_g);
                  else if (msub == 4) issue_taps<4, true>(d_tmem, bn, a_lo, a_step, b_lo, b_step, hi, idesc, accum, nt_g);
                  else if (msub == 8) issue_taps<8, true>(d_tmem, bn, a_lo, a_step, b_lo, b_step, hi, idesc, accum, nt_g);
                  else issue_taps<1, true>(d_tmem, bn, a_lo, a_step, b_lo, b_step, hi, idesc, accum, nt_g);
                } else {
                  const int* offs = s_off + ph * ntaps + tap0;
                  uint32_t bl = b_lo, acc = accum;
                  for (int j = 0; j < nt_g; ++j) {
                    const uint32_t a_lo = a_base_lo + (uint32_t)offs[j];
                    for (int sub = 0; sub < msub; ++sub)
                      umma2_f16_split(d_tmem + (uint32_t)sub * bn, a_lo + (uint32_t)sub * 128u, hi, bl, hi, idesc, acc);
                    acc = 1;
                    bl += b_step;
                  }
                }
                accum = 1;
                a_base_lo += a_slot_u;
                b_lo += (uint32_t)nt_g * b_step;
              }
              umma2_commit(empty0 + 8 * stage);  // frees the stage in BOTH CTAs when these MMAs retire
            }
            accum = 1;
            __syncwarp();
            if (++stage == S) {
              stage = 0;
              phase ^= 1;
            }
          }
        }
        if (leader) umma2_commit(tfull0 + 8 * as);  // both CTAs' epilogues
        __syncwarp();
        if (++as == P.acc_stages) {
          as = 0;
          aphase ^= 1;
        }
      }
    }
  } else if (warp == 10) {
    // ===================================================================== relay (CTA 1): local "stage full" -> CTA 0
    // one LANE per stage slot, each walking the generations of its own slot: a single relaying thread (wait, remote
    // arrive, next stage) was as slow as a 14-MMA stage and paced every shape with fewer than ~20 MMAs per stage
    if (rank == 1 && lane < S) {
      int my_tiles = 0;
      for (int tile = blockIdx.x; tile < P.total_tiles; tile += gridDim.x) ++my_tiles;
      const int total_steps = my_tiles * steps_per_tile;
      const uint32_t remote = mapa_u32(peerfull0 + 8 * lane, 0);
      for (int i = lane; i < total_steps; i += S) {
        mbar_wait(full0 + 8 * lane, (uint32_t)((i / S) & 1), P.err_flag, 9);
        mbar_arrive_cluster(remote);
      }
    }
  } else {
    // ===================================================================== epilogue (warps 2..9), own 128 msub rows
    epilogue_dispatch(P, tmem_base, tfull0, tempty0, warp & 3, (warp - 2) >> 2, lane, tile_rows, acc_cols,
                      reinterpret_cast<const float*>(smem + 1024 + (size_t)P.stages * P.stage_bytes));
  }
  tc_fence_before();
  cluster_sync_all();  // no CTA leaves (or frees TMEM) while its peer may still read its smem / signal its barriers
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc2(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------ layout helpers
__global__ void to_chunked_bf16_kernel(const float* __restrict__ src, long long src_batch, long long src_c,
                                       long long src_t, __nv_bfloat16* __restrict__ dst, long long dst_batch,
                                       long long dst_chunk, int dst_row0, int C, int L, int fp16, unsigned int* status,
                                       long long lo_offset) {
  // one thread per (t, chunk): gathers 8 channels, writes one 16-byte row
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int nch = (C + 7) >> 3;
  const int b = blockIdx.y;
  if (i >= (long long)nch * L) return;
  int t, ch;
  if (src_t == 1) {  // planar source: adjacent threads walk along t
    t = (int)(i % L);
    ch = (int)(i / L);
  } else {  // row-major source: adjacent threads walk along channels
    ch = (int)(i % nch);
    t = (int)(i / nch);
  }
  const float* s = src + (long long)b * src_batch + (long long)t * src_t;
  uint32_t h[4], l[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int c0 = ch * 8 + 2 * k;
    const float f0 = c0 < C ? s[(long long)c0 * src_c] : 0.f;
    const float f1 = c0 + 1 < C ? s[(long long)(c0 + 1) * src_c] : 0.f;
    h[k] = fh::pack16_guard(f0, f1, fp16, status);
    const float2 hf = fh::unpack16(h[k], fp16);
    l[k] = fh::pack16(f0 - hf.x, f1 - hf.y, fp16);
  }
  __nv_bfloat16* o = dst + (long long)b * dst_batch + (long long)ch * dst_chunk + (long long)(dst_row0 + t) * 8;
  *reinterpret_cast<uint4*>(o) = *reinterpret_cast<uint4*>(h);
  if (lo_offset) *reinterpret_cast<uint4*>(o + lo_offset) = *reinterpret_cast<uint4*>(l);  // hi + lo split (fp16x2)
}

}  // namespace

// ================================================================================ C ABI
extern "C" __attribute__((visibility("default"))) int64_t fh_tc_packed_weight_bytes(int Cin, int Cout, int ntaps, int P, int bn) {
  if (Cin <= 0 || Cout <= 0 || ntaps <= 0 || P <= 0 || bn <= 0 || (Cin % 8) || (bn % 16)) return -1;
  const int64_t n_tiles = (Cout + bn - 1) / bn;
  return (int64_t)P * n_tiles * ((Cin + 15) / 16) * ntaps * bn * 32;
}

// Validates the arguments and derives the launch plan (tile shape, stages, shared-memory carve-up).  Returns FH_OK or < 0.
static int tc_plan(const fh_tc_conv_args* a, TcParams& p, int* smem_out) {
  FH_REQUIRE(a != nullptr, FH_ERR_BAD_SHAPE, "fh_tc_conv: null args");
  FH_REQUIRE(a->B > 0 && a->L > 0 && a->Cin > 0 && a->Cout > 0, FH_ERR_BAD_SHAPE, "fh_tc_conv: bad shape");
  FH_REQUIRE(a->Cin % 8 == 0, FH_ERR_BAD_SHAPE, "fh_tc_conv: Cin=%d must be a multiple of 8", a->Cin);
  FH_REQUIRE(a->Cout % 8 == 0, FH_ERR_BAD_SHAPE, "fh_tc_conv: Cout=%d must be a multiple of 8", a->Cout);
  FH_REQUIRE(a->bn % 16 == 0 && a->bn >= 16 && a->bn <= 256, FH_ERR_UNSUPPORTED_CFG,
             "fh_tc_conv: bn=%d must be a multiple of 16 in [16,256]", a->bn);
  FH_REQUIRE(a->P >= 1 && a->P <= 16 && a->ntaps >= 1 && a->P * a->ntaps <= kMaxTapOff, FH_ERR_UNSUPPORTED_CFG,
             "fh_tc_conv: P=%d ntaps=%d unsupported", a->P, a->ntaps);
  FH_REQUIRE(!(a->geglu && (a->res || a->accumulate || (a->Cout % 16))), FH_ERR_UNSUPPORTED_CFG,
             "fh_tc_conv: geglu epilogue excludes residual/accumulate and needs Cout %% 16 == 0");
  FH_REQUIRE(!(a->accumulate && a->out_is_16) || (a->acc_src && a->res && !a->res_is_16), FH_ERR_UNSUPPORTED_CFG,
             "fh_tc_conv: accumulate into a 16-bit output needs acc_src (fp32) and an fp32 residual");
  FH_REQUIRE(((uintptr_t)a->a % 16) == 0 && ((uintptr_t)a->w % 16) == 0 && ((uintptr_t)a->out % 16) == 0 &&
                 ((uintptr_t)a->res % 16) == 0,
             FH_ERR_BAD_ALIGN, "fh_tc_conv: pointers must be 16-byte aligned");
  FH_REQUIRE(a->a_chunk % 8 == 0 && a->a_batch % 8 == 0, FH_ERR_BAD_ALIGN, "fh_tc_conv: A strides must be x8");
  const int esz_shift = a->out_is_16 ? 3 : 2;  // 16-byte alignment in elements
  FH_REQUIRE((a->out_batch % (1 << esz_shift)) == 0 && (a->out_chunk % (1 << esz_shift)) == 0 &&
                 (a->out_row % (1 << esz_shift)) == 0,
             FH_ERR_BAD_ALIGN, "fh_tc_conv: output strides break 16-byte alignment");

  memset(&p, 0, sizeof(p));
  p.a = (const __nv_bfloat16*)a->a;
  p.w = (const __nv_bfloat16*)a->w;
  p.bias = a->bias;
  p.res = a->res;
  p.out = a->out;
  p.a_batch = a->a_batch, p.a_chunk = a->a_chunk, p.a_row0 = a->a_row0;
  p.out_batch = a->out_batch, p.out_chunk = a->out_chunk, p.out_row = a->out_row;
  p.res_batch = a->res_batch, p.res_chunk = a->res_chunk, p.res_row = a->res_row;
  p.out_is_16 = a->out_is_16, p.res_is_16 = a->res_is_16, p.fp16 = a->fp16;
  p.accumulate = a->accumulate, p.geglu = a->geglu;
  p.acc_src = a->accumulate ? a->acc_src : nullptr;
  p.act_gelu = a->act == 1;
  FH_REQUIRE(a->act == 0 || (a->act == 1 && !a->geglu), FH_ERR_UNSUPPORTED_CFG, "fh_tc_conv: act must be 0 (none) or 1 (GELU, not with geglu)");
  p.alpha = a->alpha, p.beta_res = a->beta_res;
  p.status = fh::status_word();
  p.B = a->B, p.L = a->L, p.Cin = a->Cin, p.Cout = a->Cout, p.ntaps = a->ntaps, p.P = a->P, p.bn = a->bn;
  p.n_tiles = (a->Cout + a->bn - 1) / a->bn;
  const bool two = a->two_cta != 0;
  p.two_cta = two ? 1 : 0;
  // sub-tiles: reuse each weight slot for up to 4 x 128 rows when the accumulators fit TMEM twice over
  int msub = 256 / a->bn;
  msub = msub >= 8 ? 8 : (msub >= 4 ? 4 : (msub >= 2 ? 2 : 1));  // 8 x 128 rows for bn <= 32 (24-channel last stage)
  // Wide tiles (bn > 128): the weight stream from L2 (bn*32 B per MMA) is the limiter, so two 128-row
  // sub-tiles share every weight slot even though the accumulators (2*bn columns) then fill TMEM and
  // the epilogue no longer overlaps the next tile -- worth it once a tile carries enough MMAs.
  constexpr int kWideMsub = 2, kWideMinMmas = 96;
  // (Linear layers with many N tiles -- qkv, FF-in: 64 MMAs per tile -- gain 10 % from the shared weight slot as well;
  // the 4-tile output projection loses 15 % and keeps one sub-tile)
  const long long mmas_per_sub = (long long)a->ntaps * ((a->Cin + 15) / 16);
  if (a->bn > 128 && (mmas_per_sub >= kWideMinMmas || (mmas_per_sub >= 64 && p.n_tiles >= 8))) msub = kWideMsub;
  while (msub > 1 && (long long)a->B * a->P * ((a->L + 128 * msub - 1) / (128 * msub)) * p.n_tiles < 2 * 148)
    msub >>= 1;
  p.msub = msub;
  p.acc_stages = (2 * msub * a->bn <= 512) ? 2 : 1;
  p.m_stride = p.m_valid = 128 * msub;
  p.m_tiles = (a->L + 128 * msub - 1) / (128 * msub);
  p.ci_pairs = (a->Cin + 15) / 16;
  p.ci_odd = (a->Cin % 16) != 0;
  int span = 0, arith = 1;
  for (int ph = 0; ph < a->P; ++ph) {
    int mn = a->tap_off[ph * a->ntaps], mx = mn;
    for (int m = 0; m < a->ntaps; ++m) {
      const int o = a->tap_off[ph * a->ntaps + m];
      p.tap_off[ph * a->ntaps + m] = o;
      mn = o < mn ? o : mn;
      mx = o > mx ? o : mx;
    }
    p.min_off[ph] = mn;
    p.tap_rel0[ph] = a->tap_off[ph * a->ntaps] - mn;
    p.tap_step[ph] = a->ntaps > 1 ? a->tap_off[ph * a->ntaps + 1] - a->tap_off[ph * a->ntaps] : 0;
    for (int m = 1; m < a->ntaps; ++m)
      if (a->tap_off[ph * a->ntaps + m] - a->tap_off[ph * a->ntaps + m - 1] != p.tap_step[ph]) arith = 0;
    span = (mx - mn) > span ? (mx - mn) : span;
    FH_REQUIRE(a->a_row0 + mn >= 0, FH_ERR_BAD_SHAPE, "fh_tc_conv: left halo %d too small for tap offset %d",
               a->a_row0, mn);
  }
  FH_REQUIRE(span <= kMaxSpan, FH_ERR_UNSUPPORTED_CFG, "fh_tc_conv: tap span %d exceeds %d rows", span, kMaxSpan);
  p.tap_arith = arith;
  p.tap_pair = (p.ci_odd && arith && a->P == 1 && a->ntaps >= 2 && p.tap_step[0] > 0 && !two) ? 1 : 0;
  if (two) p.m_tiles = (p.m_tiles + 1) / 2;  // CTA PAIRS along M (decode_tile); an odd tail leaves one void tile
  const long long total = (long long)p.B * p.P * p.m_tiles * p.n_tiles * (two ? 2 : 1);
  FH_REQUIRE(total < (1ll << 31), FH_ERR_BAD_SHAPE, "fh_tc_conv: too many tiles");
  p.total_tiles = (int)total;
  {
    const bool out_ok = a->out_is_16 || (((uintptr_t)a->out % 32) == 0 && a->out_batch % 8 == 0 && a->out_chunk % 8 == 0 &&
                                         a->out_row % 8 == 0);
    const bool res_ok = a->res == nullptr || a->res_is_16 ||
                        (((uintptr_t)a->res % 32) == 0 && a->res_batch % 8 == 0 && a->res_chunk % 8 == 0 && a->res_row % 8 == 0);
    const bool acc_ok = !(a->accumulate && a->acc_src) ||
                        (((uintptr_t)a->acc_src % 32) == 0 && a->out_batch % 8 == 0 && a->out_chunk % 8 == 0 && a->out_row % 8 == 0);
    p.v8 = (out_ok && res_ok && acc_ok) ? 1 : 0;
  }
  p.wrows = 128 * msub + span;
  p.arows_pad = 128 * msub + kMaxSpan;
  // taps per stage: a weight slot of <= 48 KB for narrow and wide tiles alike (for narrow tiles all taps of a ci-pair
  // then share one activation window fetch), with the taps spread evenly over the groups (11 taps -> 6+5, not 10+1)
  constexpr int kSlotBytes = 48 * 1024;
  int tg = kSlotBytes / (a->bn * 32);
  if (tg < 1) tg = 1;
  if (tg > a->ntaps) tg = a->ntaps;
  p.n_groups = (a->ntaps + tg - 1) / tg;
  tg = (a->ntaps + p.n_groups - 1) / p.n_groups;
  p.tg = tg;
  // ci-pairs per stage: a stage should carry >= ~12 MMAs so that its barrier round trip is amortised (Linear layers are
  // one tap per ci-pair, k = 3 convs three), as long as at least 3-4 stages still fit
  constexpr int kKcMmas = 12;
  constexpr int kKcMmas2 = 24;  // CTA pairs: a stage costs two barrier round trips more (relay, multicast commit)
  constexpr int kSmemBudget = 200 * 1024;  // shared memory of the stages and the bias table without a residual ring
  int kc = 1;
  if (p.n_groups == 1) {
    const int pair_bytes = 2 * p.arows_pad * 16 + a->ntaps * (two ? a->bn / 2 : a->bn) * 32;
    const int kct = two ? kKcMmas2 : kKcMmas;
    kc = (kct + a->ntaps * msub - 1) / (a->ntaps * msub);
    if (kc > 4) kc = 4;
    if (kc > p.ci_pairs) kc = p.ci_pairs;
    while (kc > 1 && (kSmemBudget - 1024 - 8192) / (kc * pair_bytes) < 4) --kc;
  }
  p.kc = kc;
  p.stage_bytes = kc * (2 * p.arows_pad * 16 + tg * (two ? a->bn / 2 : a->bn) * 32);  // a CTA of a pair holds half of every weight slot
  p.stage_bytes = (p.stage_bytes + 127) & ~127;
  const int bias_tab = a->bias ? ((p.n_tiles * a->bn + 15) & ~15) * 4 : 64;
  p.fast_epi = (p.v8 && !a->geglu && !p.act_gelu && !(a->res && a->res_is_16) && bias_tab <= 8192 &&
                (!a->out_is_16 || (a->res == nullptr && !a->accumulate) || (a->accumulate && a->acc_src && a->res))) ? 1 : 0;
  FH_REQUIRE(p.fast_epi || !(a->accumulate && a->out_is_16), FH_ERR_UNSUPPORTED_CFG,
             "fh_tc_conv: accumulate into a 16-bit output is only implemented by the specialised epilogue");
  const int tail = p.fast_epi ? bias_tab : 0;
  // residual rows through the cp.async ring (epilogue_fast<.., RES_ASYNC>): the HBM-bound launches (<= 96 output channels in
  // one N tile, fp32 residual rows of 8 floats, P == 1) whose residual stream was latency-bound; the ring (64 KB) comes
  // out of the stage budget, which these launches do not need (a tile is 2 - 6 stages)
  constexpr int kResAsyncMaxCout = 192;
  constexpr int kEpiWideMaxBn = 96;  // widest N tile that runs with more than eight epilogue warps
  constexpr int kEw16Mmas = 64;      // sixteen epilogue warps up to this many MMAs per tile, twelve above
  // Epilogue warps.  The narrow (HBM-bound) shapes were paced by their eight epilogue warps: two per scheduler, each
  // issuing once every ~5 cycles (fixed-latency dependencies), so more warps are more throughput -- sixteen reach the
  // HBM roofline on the k = 3 shapes.  With many MMAs per tile (k >= 7) sixteen starve the single MMA-issuing warp of
  // issue slots on its scheduler (measured 20 - 30 % slower than twelve), so those run with twelve.
  p.epi_warps = 8;
  if (p.fast_epi && !two && a->bn <= kEpiWideMaxBn)
    p.epi_warps = (a->ntaps * p.ci_pairs * p.msub <= kEw16Mmas) ? 16 : 12;
  int ring = 0;
  if (p.fast_epi && !two && a->res != nullptr && !a->res_is_16 && a->P == 1 && a->res_row == 8 &&
      a->Cout <= kResAsyncMaxCout && p.msub * (a->bn >> 4) >= (p.epi_warps + 3) / 4 &&
      (216 * 1024 - 1024 - tail - 128 - res_ring_bytes(p.epi_warps)) / p.stage_bytes >= 2)
    ring = res_ring_bytes(p.epi_warps);
  int stages = ((ring ? 216 * 1024 - 128 - ring : kSmemBudget) - 1024 - tail) / p.stage_bytes;
  if (stages > kMaxStages) stages = kMaxStages;
  FH_REQUIRE(stages >= 2, FH_ERR_UNSUPPORTED_CFG, "fh_tc_conv: stage of %d bytes does not fit twice", p.stage_bytes);
  p.stages = stages;
  p.empty_ring = stages;
  p.err_flag = fh::err_word();
  p.res_async = ring ? 1 : 0;
  p.ring_off = (1024 + stages * p.stage_bytes + tail + 127) & ~127;
  *smem_out = ring ? p.ring_off + ring : 1024 + stages * p.stage_bytes + tail;
  return FH_OK;
}

extern "C" __attribute__((visibility("default"))) int fh_tc_conv(const fh_tc_conv_args* a, void* stream) {
  TcParams p;
  int smem = 0;
  const int rc = tc_plan(a, p, &smem);
  if (rc != FH_OK) return rc;
  const int num_sms = fh::dev_sms();
  const int grid = p.total_tiles < num_sms ? p.total_tiles : num_sms;
  if (p.two_cta) {
    static int smem_set2[64] = {0};
    cudaError_t e = fh::ensure_dyn_smem(tc_conv2_kernel, smem, smem_set2);
    FH_REQUIRE(e == cudaSuccess, FH_ERR_CUDA, "fh_tc_conv: cannot opt in to %d bytes of smem: %s", smem, cudaGetErrorString(e));
    int g2 = (p.total_tiles < (num_sms & ~1) ? p.total_tiles : (num_sms & ~1));  // total_tiles is even
    tc_conv2_kernel<<<g2, kThreads2, smem, (cudaStream_t)stream>>>(p);
    return fh::check_launch("fh_tc_conv(cta pair)");
  }
  static int smem_set[64] = {0}, smem_set12[64] = {0}, smem_set16[64] = {0};
  {
    cudaError_t e = p.epi_warps == 16   ? fh::ensure_dyn_smem(tc_conv_kernel<16>, smem, smem_set16)
                    : p.epi_warps == 12 ? fh::ensure_dyn_smem(tc_conv_kernel<12>, smem, smem_set12)
                                        : fh::ensure_dyn_smem(tc_conv_kernel<8>, smem, smem_set);
    FH_REQUIRE(e == cudaSuccess, FH_ERR_CUDA, "fh_tc_conv: cannot opt in to %d bytes of smem: %s", smem,
               cudaGetErrorString(e));
  }
  if (p.epi_warps == 16) tc_conv_kernel<16><<<grid, 64 + 32 * 16, smem, (cudaStream_t)stream>>>(p);
  else if (p.epi_warps == 12) tc_conv_kernel<12><<<grid, 64 + 32 * 12, smem, (cudaStream_t)stream>>>(p);
  else tc_conv_kernel<8><<<grid, kThreads, smem, (cudaStream_t)stream>>>(p);
  return fh::check_launch("fh_tc_conv");
}

extern "C" __attribute__((visibility("default"))) int fh_to_chunked_16(const float* src, int64_t src_batch, int64_t src_c, int64_t src_t, void* dst,
                                  int64_t dst_batch, int64_t dst_chunk, int dst_row0, int B, int C, int L,
                                  int fp16, void* stream) {
  FH_REQUIRE(B > 0 && C > 0 && L > 0 && B <= 65535, FH_ERR_BAD_SHAPE, "fh_to_chunked_16: bad shape");
  const long long n = (long long)((C + 7) / 8) * L;
  to_chunked_bf16_kernel<<<dim3((unsigned)((n + 255) / 256), B), 256, 0, (cudaStream_t)stream>>>(
      src, src_batch, src_c, src_t, (__nv_bfloat16*)dst, dst_batch, dst_chunk, dst_row0, C, L, fp16, fh::status_word(), 0);
  return fh::check_launch("fh_to_chunked_16");
}

// same, written as hi + lo 16-bit pairs: channels [0, C) = round(x), channels [Cpad, Cpad + C) = round(x - hi)
// (Cpad = C rounded up to 8); the operand of a convolution with duplicated weights (precision "fp16x2")
extern "C" __attribute__((visibility("default"))) int fh_to_chunked_16_split(const float* src, int64_t src_batch, int64_t src_c, int64_t src_t,
                                  void* dst, int64_t dst_batch, int64_t dst_chunk, int dst_row0, int B, int C, int L,
                                  int fp16, void* stream) {
  FH_REQUIRE(B > 0 && C > 0 && L > 0 && B <= 65535, FH_ERR_BAD_SHAPE, "fh_to_chunked_16_split: bad shape");
  const long long n = (long long)((C + 7) / 8) * L;
  to_chunked_bf16_kernel<<<dim3((unsigned)((n + 255) / 256), B), 256, 0, (cudaStream_t)stream>>>(
      src, src_batch, src_c, src_t, (__nv_bfloat16*)dst, dst_batch, dst_chunk, dst_row0, C, L, fp16, fh::status_word(),
      (long long)((C + 7) / 8) * dst_chunk);
  return fh::check_launch("fh_to_chunked_16_split");
}
