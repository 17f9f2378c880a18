// K2-K6, "wide" tcgen05 form: one 128-row tile (64 windows x 2 directions) per CTA, for the model shapes
// the two-tile kernel of forward_tc.cu has no room for:
//   * GRU with 65..128 units (BASELINE config 5b: T = 512, U = 128): the accumulator of one tile is
//     3*128 + 16 = 400 TMEM columns (two tiles do not fit 512) and the fp16 x2 pieces of [R | K/2]^T are
//     230 kB, more than one SM's shared memory.  Two CTAs of a cluster therefore work as a PAIR
//     (tcgen05.mma.cta_group::2, M = 256): each CTA keeps its own tile's state pieces (A, 128 rows) and HALF
//     of the weight rows (B, N/2), the tensor cores of both SMs read both halves, and every CTA's TMEM
//     receives all N columns of its own 128 rows -- no exchange of h over DSMEM.  The MMAs are issued by
//     one thread of the pair's leader CTA; the gate warps of both CTAs arrive on the leader's "ready"
//     mbarrier (remote arrive, release at cluster scope) and the commit is multicast to both CTAs' "done".
//   * LSTM (model.py:217-221; gates i, f, c, o, no attention): 4*U + 16 columns, single CTA for U <= 64.
// An MMA writes at most 256 columns, so the N columns are issued as column blocks of UB units
// (GRU 64: z|r|h of the block [+ 16 projection columns in block 0] = 208 / 192; LSTM 32: 144 / 128).
//
// Everything else follows forward_tc.cu: two fp16 pieces per operand and three products per K chunk
// (fp32-faithful, see there), the input projection and the biases folded into 16 extra K columns
// (one_hot(x_t) * 2^8 in A), gate columns pre-scaled so that the accumulator feeds ex2 directly, the FF
// kernel as 16 extra N columns, 16 gate warps (TMEM lane quadrant x unit quarter) + one issuer warp, the
// second phase (attention_vote_sum_tile) per tile.  Reference: deepgrp/model.py:217-230 (the RNN layer),
// :293-336 (the graph).
#include <algorithm>
#include <cmath>
#include <cstring>

#include "forward_tc_common.cuh"

namespace dgrp {

template <int UP_, int RNN_, bool PAIR_>
struct WCfg {
  static constexpr int UP = UP_, RNN = RNN_;
  static constexpr bool PAIR = PAIR_;
  static constexpr int G = RNN ? 4 : 3;             // gates: GRU z, r, h; LSTM i, f, c, o
  // units per column block, G * UB + 16 <= 256: GRU 64, LSTM 32.  (32-unit GRU blocks measured the same: 144 against
  // 147 Mbp/s at 128 units.)
  static constexpr int UB = UP < (RNN ? 32 : 64) ? UP : (RNN ? 32 : 64);
  static constexpr int NBLK = UP / UB;
  // several column blocks: the MMAs of one block overlap the gate work on another (see rnn_tcw_kernel; one round of
  // MMAs between two steps measured 117-125 against 134 Mbp/s at 128 units, 356 against 428 Mbp/s for LSTM, 60 units)
  static constexpr bool OVL = NBLK >= 2;
  static_assert(G * UB + 16 <= 256, "a column block is one MMA: at most 256 columns");
  static constexpr int NW0 = G * UB + 16, NW = G * UB;   // columns of block 0 (with the projection) / of the others
  static constexpr int N = G * UP + 16;
  static constexpr int KP = UP + 16, KC = KP / 8, SBO = KC * 128;
  static constexpr int ROWS = 128, WT = 64;
  static constexpr int NCTA = PAIR ? 2 : 1;
  static constexpr int A_BYTES = ROWS * KP * 2;     // one piece of the tile's state
  static constexpr int B_ROWS = N / NCTA;           // weight rows (= accumulator columns) held by one CTA
  static constexpr int B_BYTES = B_ROWS * KP * 2;   // one piece
  static constexpr int UBT = UB / 4, CB = UBT / 8;  // units / 8-unit chunks per gate thread and block
  static constexpr int UPT = UP / 4;
  static constexpr int PSTRIDE = UP + 4;            // GRU: floats per row of the h-gate input table
  static constexpr int TCOLS = N <= 128 ? 128 : (N <= 256 ? 256 : 512);
  static_assert(N <= 512, "accumulator exceeds the tensor memory");
  static_assert(UP % UB == 0 && UBT % 8 == 0, "block shape");
  __host__ __device__ static constexpr int coff(int b) { return b == 0 ? 0 : NW0 + (b - 1) * NW; }
  __host__ __device__ static constexpr int cw(int b) { return b == 0 ? NW0 : NW; }
};

// ---- cluster / pair primitives -----------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// address of `local` (a shared::cta address) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_rank(uint32_t local, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local), "r"(rank));
  return r;
}
// Remote arrive with the default semantics (release at CTA scope), as CUTLASS' ClusterBarrier::arrive(cta_id) does
// for the same hand-over in its 2-SM kernels: the data handed over is shared memory written by this thread and
// already made visible to the async proxy by fence.proxy.async, and TMEM reads ordered by
// tcgen05.fence::before_thread_sync.  (.release.cluster compiles to MEMBAR.ALL.GPU + ERRBAR + CGAERRBAR, which
// waits for every outstanding global scratch store of the warp: 13 % of the kernel's stall samples.)
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster_backoff(uint32_t bar, uint32_t parity) {
  uint32_t done;
  for (;;) {
    asm volatile(
        "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        " selp.u32 %0, 1, 0, p;\n}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) break;
    __nanosleep(32);
  }
}
__device__ __forceinline__ void umma_f16_pair(uint32_t d_tmem, uint64_t a, uint64_t b, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n"
      " tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n}"
      ::"r"(d_tmem), "l"(a), "l"(b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {   // arrives on `bar` of BOTH CTAs of the pair
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
      "h"((uint16_t)3)
      : "memory");
}

// LSTM cell for four units (Keras gate order i, f, c, o; one bias, already inside the accumulator through
// the one-hot K columns).  The accumulators arrive scaled by 1/us and pre-multiplied by -log2 e (i, f, o) or
// 2 log2 e (c~):  sigma = 1/(1 + 2^s),  tanh = 1 - 2/(2^a + 1);  c' = f c + i c~,  h' = o tanh(c').
// The four denominators of a unit share one reciprocal (each <= 2^30 + 1, so the product is finite).
__device__ __forceinline__ void lstm_cell4(const float *ai, const float *af, const float *ac, const float *ao,
                                           float *cst, float us, float2 &h01, float2 &h23) {
  float h[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float di = ex2_approx(fminf(ai[j] * us, 28.85f)) + 1.0f;
    const float df = ex2_approx(fminf(af[j] * us, 28.85f)) + 1.0f;
    const float dq = ex2_approx(fminf(ao[j] * us, 28.85f)) + 1.0f;
    const float dc = ex2_approx(fminf(ac[j] * us, 30.0f)) + 1.0f;
    const float m1 = di * df, m2 = dq * dc;
    const float inv = rcp_approx(m1 * m2);
    const float i1 = inv * m2, i2 = inv * m1;      // 1/(di df), 1/(dq dc)
    const float gi = i1 * df, gf = i1 * di, go = i2 * dc;
    const float ct = fmaf(-2.0f, i2 * dq, 1.0f);   // tanh(c~) = 1 - 2/dc
    const float c = fmaf(gf, cst[j], gi * ct);
    cst[j] = c;
    const float dn = ex2_approx(fminf(c * kTwoLog2e, 30.0f)) + 1.0f;
    h[j] = go * fmaf(-2.0f, rcp_approx(dn), 1.0f);
  }
  h01 = make_float2(h[0], h[1]);
  h23 = make_float2(h[2], h[3]);
}

// OVL (several column blocks): the MMAs of a round are issued block by block, as soon as the state columns they
// read have been written, so that the tensor core works while the gate warps do.  With blocks 0..n-1 (the gate warps
// go through them in this order, all 16 warps on one block at a time) and P(i, j) = "columns of block i from the
// state units of block j":
//   issuer, round t+1:  wait ready[j](t) -> P(i, j) for i < j and P(j, i) for i <= j      (j = 0 .. n-2)
//                       wait ready[n-1](t) -> P(i, n-1), commit done[i]                    (i = 0 .. n-2)
//                                             P(n-1, i), commit free[i] (i < n-1), commit done[n-1]
//   gates,  step  t+1:  wait done[j] -> gates of block j, the new state pieces kept in registers -> wait free[j] (the
//                       MMAs that read block j's old columns of A are done) -> write them, arrive ready[j]
// Only P(0, n-1) -- 1/n^2 of the products -- is exposed between two steps; a D block is overwritten (first product,
// no accumulate) only after the gate warps have read it (ready[j] is arrived on after the TMEM loads of block j).
template <int UP, int RNN, bool PAIR>
__global__ void __launch_bounds__(TC_THREADS, 1) rnn_tcw_kernel(const FwdParams p) {
  using K = WCfg<UP, RNN, PAIR>;
  constexpr int G = K::G;
  constexpr int NB = K::NBLK;
  constexpr bool OVL = K::OVL;
  static_assert(NB <= 4, "one ready / done / free barrier per column block: at most 4");
  constexpr int NBAR = OVL ? NB : 1;     // ready / done barriers: one per column block when overlapped
  extern __shared__ __align__(128) unsigned char smem_raw[];
  unsigned char *s_B = smem_raw;                                        // [2 pieces][B_BYTES]  this CTA's weight rows
  unsigned char *s_A = s_B + 2 * K::B_BYTES;                            // [2 pieces][A_BYTES]  this CTA's tile
  float *s_P = reinterpret_cast<float *>(s_A + 2 * K::A_BYTES);         // GRU: [10][PSTRIDE] h-gate rows of the input table
  float *s_scale = s_P + (RNN ? 0 : 10 * K::PSTRIDE);                   // [UP] attention scale
  float *s_score = s_scale + UP;                                        // [wpp][T]
  uint8_t *s_codes = reinterpret_cast<uint8_t *>(s_score + (size_t)p.wpp * p.T);   // [fwd | rc][code_span]
  __shared__ __align__(8) unsigned long long s_ready[4], s_done[4], s_free[4];
  __shared__ uint32_t s_tmem;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int T = p.T;
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;

  // ---- one-time setup -------------------------------------------------------------------------
  {
    const uint4 *src = reinterpret_cast<const uint4 *>(p.Bsplit) + (size_t)rank * (2 * K::B_BYTES / 16);
    uint4 *dst = reinterpret_cast<uint4 *>(s_B);
    for (int i = tid; i < 2 * K::B_BYTES / 16; i += TC_THREADS) dst[i] = src[i];
    if (!RNN)
      for (int i = tid; i < 10 * K::PSTRIDE; i += TC_THREADS) {
        const int row = i / K::PSTRIDE, j = i % K::PSTRIDE;
        const int c = row >= 8 ? 4 : (row >= 4 ? 7 - row : row);   // reverse complement: [3,2,1,0,4] (model.py:277)
        s_P[i] = j < UP ? p.P[((size_t)c * G + 2) * UP + j] * kTwoLog2e : 0.f;   // x.W_h + b_in (stays outside r * (.))
      }
    for (int i = tid; i < UP; i += TC_THREADS) s_scale[i] = (p.attention && i < p.U) ? p.scale[i] : 0.f;
    // the A operand starts all-zero (h[-1] = 0; the one-hot chunk's unused half stays zero for good)
    uint4 *a4 = reinterpret_cast<uint4 *>(s_A);
    for (int i = tid; i < 2 * K::A_BYTES / 16; i += TC_THREADS) a4[i] = make_uint4(0u, 0u, 0u, 0u);
  }
  if (warp == 0) {
    if (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem)),
                   "r"(K::TCOLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem)),
                   "r"(K::TCOLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  if (tid == 0) {
    // "ready": one arrival per gate warp of every CTA of the pair (lane 0, after the warp's fences);
    // "done" / "free": one arrival, an MMA commit
    for (int i = 0; i < 4; ++i) {
      mbar_init(smem_u32(&s_ready[i]), TC_GATE_WARPS * K::NCTA);
      mbar_init(smem_u32(&s_done[i]), 1);
      mbar_init(smem_u32(&s_free[i]), 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  fence_async_smem();
  tc_fence_before();
  if (PAIR) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = s_tmem;

  const bool is_gate = warp < TC_GATE_WARPS;
  const uint32_t bar_ready = smem_u32(&s_ready[0]), bar_done = smem_u32(&s_done[0]), bar_free = smem_u32(&s_free[0]);
  const int64_t n_tiles = launch_tiles(p, K::WT);
  // a unit of work = NCTA tiles (one per CTA of the pair); the pair owns a contiguous range of units
  const int64_t n_units = (n_tiles + K::NCTA - 1) / K::NCTA;
  const int64_t n_groups = gridDim.x / K::NCTA, grp = blockIdx.x / K::NCTA;
  const int64_t unit_lo = n_units * grp / n_groups, unit_hi = n_units * (grp + 1) / n_groups;

  if (!is_gate) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(TC_AUX_REGS));
    if (warp != TC_GATE_WARPS) return;   // the three idle warps of the issuer's warpgroup
    if (rank == 0) {
      // ===================== MMA issuer (leader CTA): T + 1 rounds per unit (round 0 = priming on h = 0) =====
      const uint32_t a0 = smem_u32(s_A), b0 = smem_u32(s_B);
      // the products of column block nb with the state units of block kb (all of them when kb < 0):
      // (A piece, B piece), smallest first: lo.hi, hi.lo, hi.hi; the one-hot K chunk (only in A's hi piece)
      // belongs to unit block 0
      auto issue = [&](int nb, int kb, uint32_t acc) {
        const uint32_t idesc = (1u << 4) | ((uint32_t)(K::cw(nb) >> 3) << 17) |
                               ((uint32_t)((K::ROWS * K::NCTA) >> 4) << 24);   // D fp32, A/B fp16 K-major, N, M
        const uint32_t d = tmem_base + (uint32_t)K::coff(nb);
        const uint32_t brow = b0 + (uint32_t)((K::coff(nb) / K::NCTA) / 8) * K::SBO;   // this block's rows of B
        const int pa[3] = {1, 0, 0}, pb[3] = {0, 1, 0};
        const int kc0 = kb < 0 ? 0 : kb * (K::UB / 16), kc1 = kb < 0 ? UP / 16 : (kb + 1) * (K::UB / 16);
#pragma unroll
        for (int q = 0; q < 3; ++q) {
#pragma unroll
          for (int kc = 0; kc < UP / 16 + 1; ++kc) {
            const bool onehot = kc == UP / 16;
            if (onehot ? !(pa[q] == 0 && kb <= 0) : (kc < kc0 || kc >= kc1)) continue;
            const uint64_t ad = umma_desc(a0 + pa[q] * K::A_BYTES + kc * 256, 128, K::SBO);
            const uint64_t bd = umma_desc(brow + pb[q] * K::B_BYTES + kc * 256, 128, K::SBO);
            if (PAIR) umma_f16_pair(d, ad, bd, idesc, acc);
            else umma_f16(d, ad, bd, idesc, acc);
            acc = 1;
          }
        }
      };
      auto commit = [&](uint32_t bar) {
        if (PAIR) umma_commit_pair(bar);
        else umma_commit(bar);
      };
      auto wait_ready = [&](int b, uint32_t parity) {
        if (PAIR) mbar_wait_cluster_backoff(bar_ready + 8 * b, parity);
        else mbar_wait_backoff(bar_ready + 8 * b, parity);
        tc_fence_after();
      };
      uint32_t rnd = 0;
      for (int64_t unit = unit_lo; unit < unit_hi; ++unit) {
        for (int k = 0; k <= T; ++k, ++rnd) {
          if (OVL) {
#pragma unroll
            for (int j = 0; j < NB; ++j) {
              wait_ready(j, rnd & 1u);
              if (lane == 0) {
                if (j < NB - 1) {
#pragma unroll
                  for (int i = 0; i < j; ++i) issue(i, j, 1u);
#pragma unroll
                  for (int i = 0; i <= j; ++i) issue(j, i, i > 0 ? 1u : 0u);
                } else {
#pragma unroll
                  for (int i = 0; i < NB - 1; ++i) { issue(i, j, 1u); commit(bar_done + 8 * i); }
#pragma unroll
                  for (int i = 0; i < NB; ++i) {
                    issue(j, i, i > 0 ? 1u : 0u);
                    if (i < NB - 1) commit(bar_free + 8 * i);
                  }
                  commit(bar_done + 8 * j);
                }
              }
              __syncwarp();
            }
          } else {
            wait_ready(0, rnd & 1u);
            if (lane == 0) {
#pragma unroll
              for (int b = 0; b < K::NBLK; ++b) issue(b, -1, 0u);
              commit(bar_done);
            }
            __syncwarp();
          }
        }
      }
    }
    if (PAIR) cluster_sync_all();   // teardown barrier of the pair (see the end of the kernel)
    return;
  }

  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(TC_GATE_REGS));
  __half *sum0 = reinterpret_cast<__half *>(p.scratch) + (size_t)blockIdx.x * K::WT * T * UP;   // [passes][T][UP/8][wpp][8]
  float *proj0 = p.ff2 + (size_t)blockIdx.x * K::WT * T * 16;                           // [WT][T][16]
  float *q0 = p.qbuf + (size_t)blockIdx.x * K::WT * UP;                                 // [WT][UP]
  const float2 us = make_float2(p.b_unscale, p.b_unscale);
  const int quad = warp & 3, uq = warp >> 2;
  const int row = quad * 32 + lane;        // row of the tile = TMEM lane
  const int wl = row >> 1, dir = row & 1;  // window in tile, direction
  const uint32_t a_row = (uint32_t)((row >> 3) * K::SBO + (row & 7) * 16);
  const uint32_t oh_off = a_row + (uint32_t)(UP / 8) * 128;   // the one-hot K chunk
  const uint32_t t_lane = tmem_base + ((uint32_t)(quad * 32) << 16);
  const size_t sum_thr = ((size_t)(wl / p.wpp) * T * (UP / 8) * p.wpp + (size_t)(wl % p.wpp)) * 8 + (dir ? 4 : 0);
  const int full_span = (K::WT - 1) * p.step + T;
  const int cbase = dir * p.code_span + (dir ? full_span - wl * p.step - T : wl * p.step);
  // every gate warp's lane 0 arrives on the leader's "ready" barriers
  const uint32_t ready_remote = PAIR ? map_to_rank(bar_ready, 0u) : bar_ready;
  auto arrive_ready = [&](int b) {
    tc_fence_before();
    fence_async_smem();
    __syncwarp();
    if (lane == 0) { if (PAIR) mbar_arrive_cluster(ready_remote + 8 * b); else mbar_arrive(bar_ready + 8 * b); }
  };
  uint32_t rnd = 0;   // rounds waited for

  for (int64_t unit = unit_lo; unit < unit_hi; ++unit) {
    const int64_t tile = unit * K::NCTA + rank;
    const bool live = tile < n_tiles;   // an odd tile count leaves the pair's second CTA a dead tile ('N' bases)
    // The bases of the tile (one contiguous span of 63 * step + T codes), translated to input-table rows:
    // a forward copy (rows 0..3, 8 for 'N') and a reversed + complemented one (rows 4..7, 9)
    {
      const TileRange tr = tile_range(p, tile, K::WT);
      const int64_t w_first = tr.w0;
      int64_t w_last = w_first + K::WT - 1;
      w_last = w_last < tr.hi ? w_last : tr.hi - 1;
      const int span = live ? (int)((w_last - w_first) * p.step) + T : 0;
      const uint8_t *src = p.codes + (w_first * (int64_t)p.step - p.codes_base);
      uint8_t *fwd_copy = s_codes, *rc_copy = s_codes + p.code_span;
      for (int i = tid; i < full_span; i += TC_GATE_WARPS * 32) {
        const int c = i < span ? src[i] : 4;
        fwd_copy[i] = (uint8_t)(c < 4 ? c : 8);
        rc_copy[full_span - 1 - i] = (uint8_t)(c < 4 ? c + 4 : 9);
      }
      gate_bar_sync();
    }
    float st[K::UPT];   // GRU: h[t-1] of this thread's units; LSTM: the cell state
#pragma unroll
    for (int j = 0; j < K::UPT; ++j) st[j] = 0.f;
    // h[-1] = 0: zero this thread's slots of A, put one_hot(x_0) into the extra K chunk and let the issuer
    // prime the accumulator (round 0), so that every step reads its pre-activations from TMEM
#pragma unroll
    for (int b = 0; b < K::NBLK; ++b)
#pragma unroll
      for (int cc = 0; cc < K::CB; ++cc) {
        const uint32_t off = a_row + (uint32_t)((b * K::UB + uq * K::UBT + cc * 8) >> 3) * 128;
        *reinterpret_cast<uint4 *>(s_A + off) = make_uint4(0u, 0u, 0u, 0u);
        *reinterpret_cast<uint4 *>(s_A + K::A_BYTES + off) = make_uint4(0u, 0u, 0u, 0u);
      }
    if (uq == 0) {
      *reinterpret_cast<uint4 *>(s_A + oh_off) = onehot_row(s_codes[cbase]);
      *reinterpret_cast<uint4 *>(s_A + oh_off + 128) = make_uint4(0u, 0u, 0u, 0u);   // (A doubles as the vote buffer)
    }
    arrive_ready(0);
    if (OVL) {
#pragma unroll
      for (int b = 1; b < NB; ++b) arrive_ready(b);
    }

#pragma unroll 1
    for (int t = 0; t < T; ++t) {
      const int trow = s_codes[cbase + t];   // input-table row of this step's base
      float pj[4];   // projection of h[t-1] (4 of the 16 extra columns per unit quarter; they sit in block 0)
#pragma unroll
      for (int b = 0; b < K::NBLK; ++b) {
        if (b < NBAR) {
          mbar_wait(bar_done + 8 * b, rnd & 1u);
          tc_fence_after();
        }
        if (b == 0) tmem_ld4(t_lane + (uint32_t)(G * K::UB + 4 * uq), pj);
        uint32_t hi[K::CB][4], lo[K::CB][4];   // the block's new state as operand pieces
#pragma unroll
        for (int cc = 0; cc < K::CB; ++cc) {
          const int ci = b * K::CB + cc;                       // this thread's chunk number
          const int ub = uq * K::UBT + cc * 8;                 // first unit of the chunk within the block
          const uint32_t taddr = t_lane + (uint32_t)(K::coff(b) + ub);
          float a0[8], a1[8], a2[8], a3[8];
          float2 hn2[4];   // the new state of the chunk's units
          tmem_ld8(taddr, a0);
          tmem_ld8(taddr + K::UB, a1);
          tmem_ld8(taddr + 2 * K::UB, a2);
          if (RNN) tmem_ld8(taddr + 3 * K::UB, a3);
          tmem_ld_wait();
#pragma unroll
          for (int j4 = 0; j4 < 2; ++j4) {
            if (RNN) {
              lstm_cell4(a0 + 4 * j4, a1 + 4 * j4, a2 + 4 * j4, a3 + 4 * j4, &st[ci * 8 + 4 * j4], us.x,
                         hn2[2 * j4], hn2[2 * j4 + 1]);
            } else {
              const float4 xh = *reinterpret_cast<const float4 *>(s_P + trow * K::PSTRIDE + b * K::UB + ub + 4 * j4);
              gru_cell4(xh, a0 + 4 * j4, a1 + 4 * j4, a2 + 4 * j4, &st[ci * 8 + 4 * j4], us, hn2[2 * j4],
                        hn2[2 * j4 + 1]);
            }
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) split2h(hn2[j], hi[cc][j], lo[cc][j]);
        }
        // new state -> operand pieces in A (one 16-byte core-matrix row per piece and chunk).  Overlapped: the MMAs
        // that still read block X's old columns (YX of this round) must have completed first.
        if (OVL && b < NB - 1) mbar_wait(bar_free + 8 * b, rnd & 1u);
#pragma unroll
        for (int cc = 0; cc < K::CB; ++cc) {
          const uint32_t off = a_row + (uint32_t)((b * K::UB + uq * K::UBT + cc * 8) >> 3) * 128;
          *reinterpret_cast<uint4 *>(s_A + off) = make_uint4(hi[cc][0], hi[cc][1], hi[cc][2], hi[cc][3]);
          *reinterpret_cast<uint4 *>(s_A + K::A_BYTES + off) = make_uint4(lo[cc][0], lo[cc][1], lo[cc][2], lo[cc][3]);
        }
        if (b == 0 && uq == 0 && t + 1 < T)   // the next step's base for the MMA's one-hot K columns
          *reinterpret_cast<uint4 *>(s_A + oh_off) = onehot_row(s_codes[cbase + t + 1]);
        // hand the block's new columns of A to the tensor core (the last step's MMA only feeds the projection);
        // the scratch stores of this step come after the release
        if (OVL || b == K::NBLK - 1) arrive_ready(OVL ? b : 0);
      }
      ++rnd;
      {
        // avg[t-1].K = h_fwd.(K/2) + h_rc.(K/2), stored by the fwd lane
        float4 o;
        o.x = (pj[0] + __shfl_xor_sync(0xffffffffu, pj[0], 1)) * us.x;
        o.y = (pj[1] + __shfl_xor_sync(0xffffffffu, pj[1], 1)) * us.x;
        o.z = (pj[2] + __shfl_xor_sync(0xffffffffu, pj[2], 1)) * us.x;
        o.w = (pj[3] + __shfl_xor_sync(0xffffffffu, pj[3], 1)) * us.x;
        if (dir == 0 && t > 0) *reinterpret_cast<float4 *>(proj0 + ((size_t)wl * T + t - 1) * 16 + 4 * uq) = o;
      }
      if (!RNN && p.attention) {   // (the LSTM graph has no attention, model.py:308)
#pragma unroll
        for (int ci = 0; ci < K::NBLK * K::CB; ++ci) {
          // h_fwd[t] + h_rc[t] (the GRU's state registers hold h[t] now): the partner row is the neighbouring
          // lane; the fwd lane stores units u0..u0+3 of the chunk, the rc lane u0+4..u0+7
          float2 sm2[2];
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const float2 lo2 = make_float2(st[ci * 8 + 2 * j], st[ci * 8 + 2 * j + 1]);
            const float2 hi2 = make_float2(st[ci * 8 + 4 + 2 * j], st[ci * 8 + 4 + 2 * j + 1]);
            const float2 send = dir ? lo2 : hi2;
            const float2 mine = dir ? hi2 : lo2;
            const float2 recv = make_float2(__shfl_xor_sync(0xffffffffu, send.x, 1),
                                            __shfl_xor_sync(0xffffffffu, send.y, 1));
            sm2[j] = __fadd2_rn(mine, recv);
          }
          const int u0 = (ci / K::CB) * K::UB + uq * K::UBT + (ci % K::CB) * 8;   // first unit of the chunk
          __half *dst = sum0 + sum_thr + ((size_t)t * (UP / 8) + (u0 >> 3)) * p.wpp * 8;
          const __half2 h0 = __floats2half2_rn(sm2[0].x, sm2[0].y), h1 = __floats2half2_rn(sm2[1].x, sm2[1].y);
          *reinterpret_cast<uint2 *>(dst) =
              make_uint2(*reinterpret_cast<const uint32_t *>(&h0), *reinterpret_cast<const uint32_t *>(&h1));
          if (t == T - 1)   // the query avg[T-1] in full precision
            *reinterpret_cast<float4 *>(q0 + (size_t)wl * UP + u0 + (dir ? 4 : 0)) =
                make_float4(0.5f * sm2[0].x, 0.5f * sm2[0].y, 0.5f * sm2[1].x, 0.5f * sm2[1].y);
        }
      }
    }
    // projection of the last state h[T-1] (round T; every barrier of the round is waited for, so that the
    // parities stay in step)
    {
      mbar_wait(bar_done, rnd & 1u);
      tc_fence_after();
      float pj[4];
      tmem_ld4(t_lane + (uint32_t)(G * K::UB + 4 * uq), pj);
      tmem_ld_wait();
      float4 o;
      o.x = (pj[0] + __shfl_xor_sync(0xffffffffu, pj[0], 1)) * us.x;
      o.y = (pj[1] + __shfl_xor_sync(0xffffffffu, pj[1], 1)) * us.x;
      o.z = (pj[2] + __shfl_xor_sync(0xffffffffu, pj[2], 1)) * us.x;
      o.w = (pj[3] + __shfl_xor_sync(0xffffffffu, pj[3], 1)) * us.x;
      if (dir == 0) *reinterpret_cast<float4 *>(proj0 + ((size_t)wl * T + (T - 1)) * 16 + 4 * uq) = o;
      if (OVL) {
#pragma unroll
        for (int b = 0; b < NB - 1; ++b) mbar_wait(bar_free + 8 * b, rnd & 1u);
#pragma unroll
        for (int b = 1; b < NB; ++b) mbar_wait(bar_done + 8 * b, rnd & 1u);
      }
      ++rnd;
      tc_fence_before();
    }
    // ---- attention + FF + softmax + vote for the CTA's tile ---------------------------------------
    __threadfence_block();
    gate_bar_sync();
    if (live)
      attention_vote_sum_tile<UP, K::WT, TC_GATE_WARPS>(p, sum0, q0, proj0, tile_range(p, tile, K::WT), p.wpp,
                                                        s_scale, s_score,
                                                        p.smem_vote == 1 ? reinterpret_cast<float *>(s_A)
                                                        : (p.smem_vote == 2 ? reinterpret_cast<float *>(s_codes + 2 * (size_t)p.code_span) : nullptr));
  }

  // ---- teardown: every MMA of the pair has completed (each CTA saw its last "done"); the pair's CTAs
  // leave together, the peer's shared memory and TMEM are operands of the leader's MMAs ----------------
  tc_fence_before();
  if (PAIR) cluster_sync_all(); else gate_bar_sync();
  if (warp == 0) {
    if (PAIR)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(K::TCOLS) : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(K::TCOLS) : "memory");
  }
}

template <int UP, int RNN, bool PAIR>
static size_t tcw_smem_bytes(int T, int wpp, int code_span) {
  using K = WCfg<UP, RNN, PAIR>;
  return (size_t)2 * K::B_BYTES + 2 * K::A_BYTES +
         sizeof(float) * ((size_t)(RNN ? 0 : 10 * K::PSTRIDE) + UP + (size_t)wpp * T) + 2 * (size_t)code_span + 128;
}

template <int UP, int RNN, bool PAIR>
static int launch_tcw_t(dgrp_ctx *c, dgrp_model *m, FwdParams &p) {
  using K = WCfg<UP, RNN, PAIR>;
  const int64_t n_windows = p.w_end - p.w_begin;
  if (n_windows <= 0 && p.w2_end <= p.w2_begin) return DGRP_OK;
  const int64_t span = (int64_t)(K::WT - 1) * p.step + p.T;
  if (span > 16384) return DGRP_E_UNSUPPORTED;
  p.code_span = (int)((span + 15) & ~(int64_t)15);
  int wpp = K::WT;
  while (wpp > 8 && tcw_smem_bytes<UP, RNN, PAIR>(p.T, wpp, p.code_span) > 227 * 1024) wpp >>= 1;
  const size_t smem = tcw_smem_bytes<UP, RNN, PAIR>(p.T, wpp, p.code_span);
  if (smem > 227 * 1024) return DGRP_E_UNSUPPORTED;   // caller falls back to the fp32 kernel
  p.wpp = wpp;
  const size_t vote_bytes = (size_t)span * p.C * sizeof(float);
  size_t smem_total = smem;
  p.smem_vote = 0;
  if (c->forward_smem_vote) {
    if (vote_bytes <= (size_t)2 * K::A_BYTES) p.smem_vote = 1;          // in the A operand, idle in the second phase
    else if (smem + vote_bytes <= 227 * 1024) { p.smem_vote = 2; smem_total = smem + vote_bytes; }   // a region of its own
  }
  if (p.query) return DGRP_OK;
  if (p.smem_vote) p.win_probs = nullptr;
  auto kern = rnn_tcw_kernel<UP, RNN, PAIR>;
  DGRP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_total));
  const int64_t n_tiles = (n_windows > 0 ? (n_windows + K::WT - 1) / K::WT : 0) +
                          (p.w2_end > p.w2_begin ? (p.w2_end - p.w2_begin + K::WT - 1) / K::WT : 0);
  const int64_t n_units = (n_tiles + K::NCTA - 1) / K::NCTA;
  const int64_t max_groups = c->sm_count / K::NCTA;
  const int grid = (int)(n_units < max_groups ? n_units : max_groups) * K::NCTA;
  const size_t rows = (size_t)grid * K::WT;   // window slots in flight
  DGRP_CHECK(c->avg.reserve(rows * p.T * UP * sizeof(__half) + rows * UP * sizeof(float)));
  DGRP_CHECK(c->io_c.reserve(rows * p.T * 16 * sizeof(float)));
  p.scratch = c->avg.as<float>();
  p.qbuf = reinterpret_cast<float *>(c->avg.as<unsigned char>() + rows * p.T * UP * sizeof(__half));
  p.ff2 = c->io_c.as<float>();
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(TC_THREADS);
  cfg.dynamicSmemBytes = smem_total;
  cfg.stream = c->stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = K::NCTA;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = PAIR ? 1 : 0;
  DGRP_CUDA(cudaLaunchKernelEx(&cfg, kern, p));
  c->launches++;
  return DGRP_OK;
}

// which = 1: single CTA, 2: CTA pair.  Returns DGRP_E_UNSUPPORTED when the shape has no wide form.
int launch_forward_tcw(dgrp_ctx *c, dgrp_model *m, FwdParams &p, int which) {
  const bool pair = which == 2;
  p.Bsplit = m->d_Bw[pair ? 1 : 0];
  if (!p.Bsplit) return DGRP_E_UNSUPPORTED;
  p.b_unscale = ldexpf(1.0f, -(8 + m->bw_shift));
  if (m->rnn == 0) {
    if (m->UP == 32) return pair ? DGRP_E_UNSUPPORTED : launch_tcw_t<32, 0, false>(c, m, p);
    if (m->UP == 64) return pair ? launch_tcw_t<64, 0, true>(c, m, p) : launch_tcw_t<64, 0, false>(c, m, p);
    if (m->UP == 128 && pair) return launch_tcw_t<128, 0, true>(c, m, p);
  } else {
    if (m->UP == 32) return pair ? DGRP_E_UNSUPPORTED : launch_tcw_t<32, 1, false>(c, m, p);
    if (m->UP == 64) return pair ? launch_tcw_t<64, 1, true>(c, m, p) : launch_tcw_t<64, 1, false>(c, m, p);
  }
  return DGRP_E_UNSUPPORTED;
}

// ---- host: the weight operand of the wide kernel -------------------------------------------------
// Column n of the accumulator (block b, then gate, then unit within the block; 16 projection columns at the
// end of block 0) against K row k (units, then 16 rows for the one-hot input columns).  Gate columns are
// pre-scaled (sigmoid gates by -log2 e, tanh gates by 2 log2 e), projection columns are the halved FF kernel.
// Rp [UP][G][UP], P [5][G][UP] (kernel + input bias), b1 [G][UP] (GRU recurrent bias; zero for LSTM).
template <int UP, int RNN>
static void tcw_fill(int U, int C, bool att, const float *Rp, const float *P, const float *b1, const float *ffk,
                     std::vector<float> &dense) {
  using K = WCfg<UP, RNN, false>;
  constexpr int G = K::G;
  dense.assign((size_t)K::N * K::KP, 0.f);
  for (int b = 0; b < K::NBLK; ++b)
    for (int x = 0; x < K::cw(b); ++x) {
      const int n = K::coff(b) + x;
      for (int k = 0; k < K::KP; ++k) {
        float v = 0.f;
        if (x < G * K::UB) {
          const int g = x / K::UB, u = b * K::UB + x % K::UB;
          const bool tanh_gate = g == 2;   // GRU: h; LSTM: c~
          const float sc = tanh_gate ? 2.8853900817779268f : -1.4426950408889634f;
          if (k < UP) v = Rp[((size_t)k * G + g) * UP + u] * sc;
          else if (k - UP < 5) {
            const int cc = k - UP;
            if (RNN) v = P[((size_t)cc * G + g) * UP + u] * sc;                        // x.W + b (the LSTM's only bias)
            else if (g < 2) v = (P[((size_t)cc * G + g) * UP + u] + b1[(size_t)g * UP + u]) * sc;   // z, r: both biases
            else v = b1[(size_t)g * UP + u] * sc;                                      // h: recurrent bias (inside r * (.))
          }
        } else if (k < U) {
          const int j = x - G * K::UB;   // 0..4: ctx half (attention only), 8..12: avg half
          if (j < 5 && j < C && att) v = 0.5f * ffk[(size_t)k * C + j];
          else if (j >= 8 && j - 8 < C && j < 13) v = 0.5f * ffk[(size_t)((att ? U : 0) + k) * C + (j - 8)];
        }
        dense[(size_t)n * K::KP + k] = v;
      }
    }
}

template <int UP, int RNN, bool PAIR>
static void tcw_pack(const std::vector<float> &dense, int shift, std::vector<uint16_t> &out) {
  using K = WCfg<UP, RNN, PAIR>;
  // [rank][piece][B_ROWS x KP] in the UMMA K-major core-matrix layout; CTA `rank` holds, for every column
  // block, rows [rank * cw/NCTA, (rank + 1) * cw/NCTA) of the block at local rows coff/NCTA ...
  out.assign((size_t)K::NCTA * 2 * K::B_ROWS * K::KP, 0);
  for (int r = 0; r < K::NCTA; ++r)
    for (int b = 0; b < K::NBLK; ++b) {
      const int w = K::cw(b) / K::NCTA;
      for (int i = 0; i < w; ++i) {
        const int n = K::coff(b) + r * w + i, nl = K::coff(b) / K::NCTA + i;
        for (int k = 0; k < K::KP; ++k) {
          const float x = std::ldexp(dense[(size_t)n * K::KP + k], shift);
          const __half hi = __float2half_rn(x);
          const __half lo = __float2half_rn(x - __half2float(hi));
          const size_t off = ((size_t)(nl / 8) * K::SBO + (size_t)(k / 8) * 128 + (nl % 8) * 16 + (k % 8) * 2) / 2;
          const size_t base = (size_t)r * 2 * K::B_ROWS * K::KP;
          memcpy(&out[base + off], &hi, 2);
          memcpy(&out[base + (size_t)K::B_ROWS * K::KP + off], &lo, 2);
        }
      }
    }
}

template <int UP, int RNN>
static void tcw_build_t(int U, int C, bool att, const float *Rp, const float *P, const float *b1, const float *ffk,
                        bool want_single, bool want_pair, std::vector<uint16_t> &single, std::vector<uint16_t> &pair,
                        int *shift) {
  std::vector<float> dense;
  tcw_fill<UP, RNN>(U, C, att, Rp, P, b1, ffk, dense);
  float bmax = 0.f;
  for (float v : dense) bmax = std::fmax(bmax, std::fabs(v));
  int s = 0;
  if (bmax > 0.f && std::isfinite(bmax)) {
    int e = 0;
    std::frexp(bmax, &e);   // the largest entry lands just below 2^14: the low pieces stay normal numbers
    s = std::min(24, std::max(-24, 14 - e));
  }
  *shift = s;
  if (want_single) tcw_pack<UP, RNN, false>(dense, s, single);
  if (want_pair) tcw_pack<UP, RNN, true>(dense, s, pair);
}

// Builds the operands for the shapes launch_forward_tcw serves (empty vectors otherwise): out[0] single CTA,
// out[1] CTA pair.
void build_tcw_operands(int rnn, int U, int UP, int C, bool att, const float *Rp, const float *P, const float *b1,
                        const float *ffk, std::vector<uint16_t> (&out)[2], int *shift) {
  for (auto &v : out) v.clear();
  *shift = 0;
  if (rnn == 0) {
    if (UP == 32) tcw_build_t<32, 0>(U, C, att, Rp, P, b1, ffk, true, false, out[0], out[1], shift);
    else if (UP == 64) tcw_build_t<64, 0>(U, C, att, Rp, P, b1, ffk, true, true, out[0], out[1], shift);
    else if (UP == 128) tcw_build_t<128, 0>(U, C, att, Rp, P, b1, ffk, false, true, out[0], out[1], shift);
  } else {
    if (UP == 32) tcw_build_t<32, 1>(U, C, att, Rp, P, b1, ffk, true, false, out[0], out[1], shift);
    else if (UP == 64) tcw_build_t<64, 1>(U, C, att, Rp, P, b1, ffk, true, true, out[0], out[1], shift);
  }
}

}  // namespace dgrp
