// K2-K6, tcgen05 form: the recurrent product h.R of both GRU passes on the 5th-generation tensor
// cores, attention + FF + softmax in a second phase of the same persistent kernel, the max-vote as
// plain stores + a gather pass (vote.cu).  forward.cu holds the fp32 FFMA form of the same math.
//
// Precision.  The parity bar (>= 99.99 % identical labels against a float32 CPU run, on random-init
// weights whose class margins are ~1e-4) needs fp32-faithful pre-activations through a 150..512 step
// recurrence (SURVEY.md section 7 H1); plain bf16 misses it by orders of magnitude.  Both operands are
// therefore split into two fp16 pieces of the scaled value (state x 2^8, weights x 2^shift so that the
// low pieces stay normal) and the product is formed from three piece products, each a kind::f16
// tcgen05.mma accumulating in fp32 into the same TMEM tile, smallest terms first: lo.hi + hi.lo + hi.hi,
// relative error ~2^-21 per product.  This measures the same distance from the float64 oracle as the fp32
// kernel (tools/accuracy_study.py); three bf16 pieces (six products) measured no closer at twice the
// tensor work.  The gates, sigmoid/tanh and the state update stay in fp32 registers.
//
// One CTA = 20 warps, persistent, one per SM; a unit of work = two tiles of 64 windows x 2 directions
// (M = 128 rows; row r = window r/2, direction r%2) in flight:
//   warps 0..15  gate warps: TMEM lane quadrant w % 4 (rows 32*(w%4) ..+31, one row per lane), unit
//                quarter w / 4; they wait for the tile's "done" mbarrier, read the accumulator
//                (tcgen05.ld), add the input projection (a table row: x_t is one-hot), apply the gates,
//                write the new state as operand pieces into A (shared memory), fence, arrive on the
//                tile's "ready" mbarrier, and only then store the step's scratch;
//   warp 16      MMA issuer: waits for "ready" (with back-off), issues the step's 3 x UP/16 + 2
//                tcgen05.mma (M128, N = 3*UP + 16, K16) and commits them to "done".
//                (Letting the last-arriving gate warp issue instead was measured 14 % slower.)
//   warps 17..19 exit after setmaxnreg: the CTA launches with 96 registers per thread, the issuer's
//                warpgroup drops to 24 and the gate warps rise to 112 (their loop spills at 96).
// While the tensor core multiplies tile X's new state by R, the gate warps work on tile Y.  A unit starts
// with a priming MMA round on an all-zero A operand (h[-1] = 0; two rounds when T is even), so the step
// loop has no special case and every unit runs an even number of rounds (barrier parities are a
// function of the step).  The z, r (h) columns of R, the input table and the biases are pre-scaled by
// -log2(e) (2 log2(e)) so that the accumulator feeds ex2 directly; reciprocals are shared four ways.
//   TMEM   2 x [128 lanes x (3*UP + 16) columns] fp32 accumulators: z | r | h gate blocks, then 16
//          projection columns h.(K/2) (the FF layer's two halves): avg[t].K = h_fwd[t].K/2 + h_rc[t].K/2
//          comes out of the same MMA and the second phase needs no FFMA over the units
//   smem   B = [R | K/2]^T pieces, [2][(3*UP+16) x (UP+16)], K-major core matrices, resident
//          A = state pieces, [2 tiles][2][128 x (UP+16)], rewritten every step by the gate warps
//          input table [10 rows][3*UP + 4] (A,C,G,T of either direction 4 banks apart, then 'N')
//          staged bases of the unit's tiles as table rows, [2 tiles][forward | reversed+complemented]
//          scores of one pass of the second phase, [wpp windows][T]
// Operand layout (no swizzle, K-major): 8-row x 16-byte core matrices, 128 B each; core matrices
// adjacent along K are 128 B apart (leading byte offset), along M/N they are UP/8 * 128 B apart
// (stride byte offset); one MMA consumes K = 16 = two core matrices.
//
// Scratch in HBM (per CTA, rewritten by every unit; the attention query avg[T-1] is only known after
// the last step, so the scores need a second pass over all avg[t]):
//   sum    f16[2][64/wpp][T][UP/8][wpp][8]  h_fwd[t] + h_rc[t] (= 2 avg[t], one lane shuffle) -- feeds ONLY the
//                                 additive-attention scores, so half precision suffices (|sum| < 2; a
//                                 probability moves by ~1e-7 on random-init weights, <= 3e-5 on sharp
//                                 ones); float32 measured 8 % slower
//   q      f32[2][64][UP]         avg[T-1] in full precision (the query)
//   proj   f32[2][64][T][16]      avg[t].K, both FF halves (the logits come from these, full precision)
// = 192 B per (window, t), written once and read once.  All CTAs run the same amount of work, so without
// care their second phases coincide and saturate HBM while the recurrence phases leave it idle: CTA b
// starts with (b mod 4) single-tile units, which shifts its phase by ~3/4 of a period each.  By the time
// the scratch is read back it has left the L2, and one SM's demand loads sustain only ~17 B/clk against
// HBM latency, so the second phase asks the L2 for it a few rows ahead (cp.async.bulk.prefetch.L2).
// The window probabilities go to [window][T][C] with plain stores; vote_gather_kernel max-merges them.
#include "forward_tc_common.cuh"

namespace dgrp {

template <int UP>
struct TCfg {
  static constexpr int NG = 3 * UP;            // gate columns (z | r | h)
  static constexpr int N = 3 * UP + 16;        // + 16 projection columns: h.[FF ctx half(5) pad(3) | FF avg half(5) pad(3)]
  static constexpr int ROWS = 128, WT = 64;
  static constexpr int UPT = UP / 4;           // units per gate thread
  // The z / r input projection is folded into the MMA: 16 more K columns hold one_hot(x_t) * 2^8 in A
  // (5 used) and, in B, the z / r rows of the input table plus the h gate's recurrent bias, so the gate
  // warps read only the h-gate row of the table (a quarter of their former shared-memory loads).
  static constexpr int KP = UP + 16;           // K of the operands
  static constexpr int KC = KP / 8;            // core matrices along K
  static constexpr int SBO = KC * 128;         // bytes between 8-row groups
  static constexpr int A_BYTES = ROWS * KP * 2;  // one piece of one tile
  static constexpr int B_BYTES = N * KP * 2;     // one piece
  static constexpr int PSTRIDE = 3 * UP + 4;     // floats per code row of the input table
  static constexpr int TCOLS = N <= 64 ? 64 : (N <= 128 ? 128 : 256);  // TMEM columns per tile
};


template <int UP>
__global__ void __launch_bounds__(TC_THREADS, 1) gru_tc_attention_vote_kernel(const FwdParams p) {
  using K = TCfg<UP>;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  unsigned char *s_B = smem_raw;                               // [2][B_BYTES]
  unsigned char *s_A = s_B + 2 * K::B_BYTES;                   // [2][2][A_BYTES]
  float *s_P = reinterpret_cast<float *>(s_A + 2 * 2 * K::A_BYTES);  // [10][PSTRIDE]: rows 0..3 A,C,G,T of the forward
                                                               // pass, 4..7 of the rc pass (complemented), 8, 9
                                                               // 'N' of either: the eight common rows start 4
                                                               // banks apart, so a warp's mixed reads do not conflict
                                                               // (only the h-gate columns are read)
  float *s_bh = s_P + 10 * K::PSTRIDE;                         // [UP] recurrent bias of the h gate (unread: B's
                                                               // one-hot K rows carry it)
  float *s_scale = s_bh + UP;                                  // [UP] attention scale
  float *s_score = s_scale + UP;                               // [wpp][T]
  uint8_t *s_codes = reinterpret_cast<uint8_t *>(s_score + (size_t)p.wpp * p.T);   // [2 tiles][fwd | rc][code_span] staged bases
  __shared__ __align__(8) unsigned long long s_ready[2], s_done[2];
  __shared__ uint32_t s_tmem;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int T = p.T;

  // ---- one-time setup -------------------------------------------------------------------------
  {
    const uint4 *src = reinterpret_cast<const uint4 *>(p.Bsplit);
    uint4 *dst = reinterpret_cast<uint4 *>(s_B);
    for (int i = tid; i < 2 * K::B_BYTES / 16; i += TC_THREADS) dst[i] = src[i];
    for (int i = tid; i < 10 * K::PSTRIDE; i += TC_THREADS) {
      const int row = i / K::PSTRIDE, j = i % K::PSTRIDE;
      // reverse complement: [3,2,1,0,4] (model.py:277)
      const int c = row >= 8 ? 4 : (row >= 4 ? 7 - row : row);
      // (x.W + b_in) + b_rec for z and r; the h gate keeps b_rec inside r * (h.R + b_rec)
      float v = 0.f;
      if (j < 2 * UP) v = (p.P[c * 3 * UP + j] + p.b1[j]) * kNegLog2e;
      else if (j < 3 * UP) v = p.P[c * 3 * UP + j] * kTwoLog2e;
      s_P[i] = v;
    }
    for (int i = tid; i < UP; i += TC_THREADS) {
      s_bh[i] = p.b1[2 * UP + i] * kTwoLog2e;
      s_scale[i] = (p.attention && i < p.U) ? p.scale[i] : 0.f;
    }
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(&s_tmem)),
                 "r"(2 * K::TCOLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
#ifdef DGRP_TC_TRACE
  for (int i = tid; i < 17 * 2 * 8; i += TC_THREADS) (&s_tc_trace[0][0][0])[i] = 0u;
  for (int i = tid; i < 16 * 8; i += TC_THREADS) (&s_tc_trace2[0][0])[i] = 0u;
#endif
  if (tid == 0) {
    mbar_init(smem_u32(&s_ready[0]), TC_GATE_WARPS * 32);
    mbar_init(smem_u32(&s_ready[1]), TC_GATE_WARPS * 32);
    mbar_init(smem_u32(&s_done[0]), 1);
    mbar_init(smem_u32(&s_done[1]), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = s_tmem;
  // 20 warps launch with 96 registers each; the issuer's warpgroup hands most of its share to the gate
  // warps, whose loop otherwise spills.  ptxas budgets registers per role only when each role's whole
  // code sits inside the setmaxnreg branch, so the two roles have their own copy of the unit loop and
  // meet only through the mbarriers; the gate warps synchronise among themselves on named barrier 1.
  const bool is_gate = warp < TC_GATE_WARPS;
  // Rounds per unit and tile slot: 1 priming round (2 when T is even) + T steps = an EVEN number, so that
  // every unit starts with both mbarriers of a slot at phase parity 0 and the parity of a wait is a
  // function of the step alone (a per-slot parity register was spilled and reloaded inside the step loop).
  const int extra = (T & 1) ? 0 : 1;
  const uint32_t bar_ready = smem_u32(&s_ready[0]), bar_done = smem_u32(&s_done[0]);
  const int64_t n_tiles = launch_tiles(p, K::WT);
  // this CTA's contiguous tile range; the first `lead` units are single tiles (phase shift, see top)
  const int64_t tile_lo = n_tiles * blockIdx.x / gridDim.x, tile_hi = n_tiles * (blockIdx.x + 1) / gridDim.x;
  const int64_t my_tiles = tile_hi - tile_lo;   // a single-tile unit costs ~3/4 of a period for half the work
  const int lead = my_tiles >= 32 ? (int)(blockIdx.x & 3) : (my_tiles >= 16 ? (int)(blockIdx.x & 1) : 0);
  // instruction descriptor: D fp32, A/B fp16, both K-major, N = 3*UP + 16, M = 128
  const uint32_t idesc = (1u << 4) | ((uint32_t)(K::N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);

  if (!is_gate) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(TC_AUX_REGS));
    if (warp != TC_GATE_WARPS) return;   // the three idle warps of the issuer's warpgroup
    int unit = 0;
    for (int64_t tile = tile_lo; tile < tile_hi; ++unit) {
      const int nt = (unit < lead || tile + 1 >= tile_hi) ? 1 : 2;
      const bool live1 = nt == 2;
      // ===================== MMA issuer: T + 1 rounds per tile (round 0 = priming on h = 0) =====
      TC_TRACE_DECL;
      for (int k = 0; k <= T + extra; ++k) {
#pragma unroll
        for (int s = 0; s < 2; ++s) {
          if (s == 1 && !live1) continue;
          TC_TRACE(6);
          mbar_wait_backoff(bar_ready + 8 * s, (uint32_t)(k & 1));
          tc_fence_after();
          TC_TRACE(5);
          if (lane == 0) {
            const uint32_t a0 = smem_u32(s_A + (size_t)s * 2 * K::A_BYTES), b0 = smem_u32(s_B);
            const uint32_t d = tmem_base + (uint32_t)(s * K::TCOLS);
            // (A piece, B piece), smallest products first: lo.hi, hi.lo, hi.hi
            const int pa[3] = {1, 0, 0};
            const int pb[3] = {0, 1, 0};
            uint32_t acc = 0;
#pragma unroll
            for (int q = 0; q < 3; ++q) {
              // the one-hot K chunk only exists in the hi piece of A (its lo piece is zero)
              const int nkc = UP / 16 + (pa[q] == 0 ? 1 : 0);
#pragma unroll
              for (int kc = 0; kc < UP / 16 + 1; ++kc) {
                if (kc >= nkc) break;
                const uint64_t ad = umma_desc(a0 + pa[q] * K::A_BYTES + kc * 256, 128, K::SBO);
                const uint64_t bd = umma_desc(b0 + pb[q] * K::B_BYTES + kc * 256, 128, K::SBO);
                umma_f16(d, ad, bd, idesc, acc);
                acc = 1;
              }
            }
            umma_commit(bar_done + 8 * s);
          }
          __syncwarp();
        }
      }
      tile += nt;
    }
#ifdef DGRP_TC_TRACE
    __syncwarp();
    if (blockIdx.x == 0 && lane < 16) g_tc_trace[16][lane >> 3][lane & 7] += s_tc_trace[16][lane >> 3][lane & 7];
#endif
    return;
  }

  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(TC_GATE_REGS));
  __half *sum0 = reinterpret_cast<__half *>(p.scratch) + (size_t)blockIdx.x * 2 * K::WT * T * UP; // [2][WT][T][UP]
  float *proj0 = p.ff2 + (size_t)blockIdx.x * 2 * K::WT * T * 16;                                 // [2][WT][T][16]
  float *q0 = p.qbuf + (size_t)blockIdx.x * 2 * K::WT * UP;                                       // [2][WT][UP]
  const float2 us = make_float2(p.b_unscale, p.b_unscale);
  int unit = 0;
  for (int64_t tile = tile_lo; tile < tile_hi; ++unit) {
    const int nt = (unit < lead || tile + 1 >= tile_hi) ? 1 : 2;
    const bool live1 = nt == 2;
    {
    // ===================== gate warps =====================
    const int quad = warp & 3, uq = warp >> 2;
    const int row = quad * 32 + lane;        // row of the tile = TMEM lane
    const int wl = row >> 1, dir = row & 1;  // window in tile, direction
    const float *tblp = s_P + uq * K::UPT;
    const uint32_t a_off = (uint32_t)((row >> 3) * K::SBO + (row & 7) * 16 + ((uq * K::UPT) >> 3) * 128);
    // this thread's constant part of the `sum` index: pass of its window, window within the pass, half
    const size_t sum_thr = ((size_t)(wl / p.wpp) * T * (UP / 8) * p.wpp + (size_t)(wl % p.wpp)) * 8 + (dir ? 4 : 0);
    const uint32_t oh_off = (uint32_t)((row >> 3) * K::SBO + (row & 7) * 16 + (UP / 8) * 128);   // the one-hot K chunk
    const uint32_t t_lane = tmem_base + ((uint32_t)(quad * 32) << 16);
    // The bases of a tile are one contiguous span of 63 * step + T codes: staged in shared memory once
    // per unit, so that the step loop has no global load (an L2 miss there stalls the whole tile).  Two
    // copies, already translated to input-table rows: forward (rows 0..3, 8 for 'N') and reversed +
    // complemented for the rc pass (rows 4..7, 9), so that both directions read position base + t.
    // Offset of this row's first base in its copy of tile slot 0's span; slot 1 is 2 * code_span further.
    // The reversed copy is laid out against the FULL span (63 * step + T) so that the offset does not
    // depend on the slot; what a short last tile does not cover is filled with 'N' rows (the windows
    // past the end compute on them; their results are never used).
    const int full_span = (K::WT - 1) * p.step + T;
    const int cbase = dir * p.code_span + (dir ? full_span - wl * p.step - T : wl * p.step);
    {
      const int nthr = TC_GATE_WARPS * 32;
      for (int s = 0; s < nt; ++s) {
        const TileRange tr = tile_range(p, tile + s, K::WT);
        const int64_t w_first = tr.w0;
        int64_t w_last = w_first + K::WT - 1;
        w_last = w_last < tr.hi ? w_last : tr.hi - 1;
        const int span = (int)((w_last - w_first) * p.step) + T;
        const uint8_t *src = p.codes + (w_first * (int64_t)p.step - p.codes_base);
        uint8_t *fwd_copy = s_codes + (size_t)(2 * s) * p.code_span, *rc_copy = fwd_copy + p.code_span;
        for (int i = tid; i < full_span; i += nthr) {
          const int c = i < span ? src[i] : 4;
          fwd_copy[i] = (uint8_t)(c < 4 ? c : 8);
          rc_copy[full_span - 1 - i] = (uint8_t)(c < 4 ? c + 4 : 9);
        }
      }
      gate_bar_sync();
    }
    float hprev[2][K::UPT];
#pragma unroll
    for (int s = 0; s < 2; ++s) {
#pragma unroll
      for (int j = 0; j < K::UPT; ++j) hprev[s][j] = 0.f;
      if (s == 1 && !live1) continue;
      // h[-1] = 0: zero this thread's slots of the A operand and let the issuer prime the accumulator
      unsigned char *a_tile = s_A + (size_t)s * 2 * K::A_BYTES + a_off;
#pragma unroll
      for (int c8 = 0; c8 < K::UPT / 8; ++c8)
#pragma unroll
        for (int pc = 0; pc < 2; ++pc)
          *reinterpret_cast<uint4 *>(a_tile + pc * K::A_BYTES + c8 * 128) = make_uint4(0u, 0u, 0u, 0u);
      if (uq == 0) {   // one_hot(x_0) in the hi piece's extra K chunk (its second half stays zero)
        unsigned char *oh = s_A + (size_t)s * 2 * K::A_BYTES + oh_off;
        *reinterpret_cast<uint4 *>(oh) = onehot_row(s_codes[cbase + s * 2 * p.code_span]);
        *reinterpret_cast<uint4 *>(oh + 128) = make_uint4(0u, 0u, 0u, 0u);
      }
      tc_fence_before();
      fence_async_smem();
      mbar_arrive(bar_ready + 8 * s);
      if (extra) {   // second priming round on the same all-zero operand
        mbar_wait(bar_done + 8 * s, 0u);
        mbar_arrive(bar_ready + 8 * s);
      }
    }
    TC_TRACE_DECL;
#pragma unroll 1
    for (int t = 0; t < T; ++t) {
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        if (s == 1 && !live1) continue;   // uniform over the CTA
        const int trow = s_codes[cbase + s * 2 * p.code_span + t];   // input-table row of this step's base
        TC_TRACE(4);
        mbar_wait(bar_done + 8 * s, (uint32_t)((t + extra) & 1));
        tc_fence_after();
        TC_TRACE(0);
        const float *prow = tblp + trow * K::PSTRIDE;
        const uint32_t t_tile = t_lane + (uint32_t)(s * K::TCOLS);
        unsigned char *a_tile = s_A + (size_t)s * 2 * K::A_BYTES + a_off;
        const size_t rt = (size_t)(s * K::WT + wl) * T + t;   // (window, t) row of the scratch arrays
        float pj[4];   // projection of h[t-1] (4 of the 16 extra columns per unit quarter)
        tmem_ld4(t_tile + (uint32_t)(K::NG + 4 * uq), pj);
        float2 hn2[K::UPT / 8][4];   // the new state of this thread's units
#pragma unroll
        for (int c8 = 0; c8 < K::UPT / 8; ++c8) {
          float az[8], ar[8], ah[8];
          {
            const uint32_t taddr = t_tile + (uint32_t)(uq * K::UPT + c8 * 8);
            tmem_ld8(taddr, az);
            tmem_ld8(taddr + UP, ar);
            tmem_ld8(taddr + 2 * UP, ah);
            tmem_ld_wait();
            if (c8 == 0) TC_TRACE(1);
          }
#pragma unroll
          for (int j4 = 0; j4 < 2; ++j4) {
            const float4 xh = *reinterpret_cast<const float4 *>(prow + 2 * UP + c8 * 8 + 4 * j4);
            gru_cell4(xh, az + 4 * j4, ar + 4 * j4, ah + 4 * j4, &hprev[s][c8 * 8 + 4 * j4], us, hn2[c8][2 * j4],
                      hn2[c8][2 * j4 + 1]);
          }
          // new state -> operand pieces in A (one 16-byte core-matrix row per piece)
          uint32_t hi[4], lo[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) split2h(hn2[c8][j], hi[j], lo[j]);
          *reinterpret_cast<uint4 *>(a_tile + c8 * 128) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
          *reinterpret_cast<uint4 *>(a_tile + K::A_BYTES + c8 * 128) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        }
        if (uq == 0 && t + 1 < T)   // the next step's base for the MMA's one-hot K columns
          *reinterpret_cast<uint4 *>(s_A + (size_t)s * 2 * K::A_BYTES + oh_off) =
              onehot_row(s_codes[cbase + s * 2 * p.code_span + t + 1]);
        TC_TRACE(2);
        // Hand the new A operand to the tensor core (the last step's MMA only feeds the projection).
        // The release fence waits for this thread's outstanding stores, so it comes BEFORE the scratch
        // stores of this step: only the A operand writes are in flight here.
        tc_fence_before();
        fence_async_smem();
        mbar_arrive(bar_ready + 8 * s);
        TC_TRACE(3);
        {
          // avg[t-1].K = h_fwd.(K/2) + h_rc.(K/2), stored by the fwd lane
          float4 o;
          o.x = pj[0] + __shfl_xor_sync(0xffffffffu, pj[0], 1);
          o.y = pj[1] + __shfl_xor_sync(0xffffffffu, pj[1], 1);
          o.z = pj[2] + __shfl_xor_sync(0xffffffffu, pj[2], 1);
          o.w = pj[3] + __shfl_xor_sync(0xffffffffu, pj[3], 1);
          o.x *= us.x; o.y *= us.x; o.z *= us.x; o.w *= us.x;
          if (dir == 0 && t > 0) *reinterpret_cast<float4 *>(proj0 + (rt - 1) * 16 + 4 * uq) = o;
        }
        TC_TRACE(5);
        if (p.attention) {
#pragma unroll
          for (int c8 = 0; c8 < K::UPT / 8; ++c8) {
            // h_fwd[t] + h_rc[t]: the partner row is the neighbouring lane; the fwd lane stores
            // units u0..u0+3, the rc lane u0+4..u0+7 (u0 = first unit of this block)
            float2 sm2[2];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
              const float2 send = dir ? hn2[c8][j] : hn2[c8][j + 2];
              const float2 mine = dir ? hn2[c8][j + 2] : hn2[c8][j];
              const float2 recv = make_float2(__shfl_xor_sync(0xffffffffu, send.x, 1),
                                              __shfl_xor_sync(0xffffffffu, send.y, 1));
              sm2[j] = __fadd2_rn(mine, recv);
            }
            const int u = uq * K::UPT + c8 * 8 + (dir ? 4 : 0);
            // [slot][pass][t][chunk][wpp windows][8 units]: the warp's 32 rows write 32 consecutive 4-unit groups
            __half *dst = sum0 + (size_t)s * K::WT * T * UP + sum_thr + ((size_t)t * (UP / 8) + (uq * (K::UPT / 8) + c8)) * p.wpp * 8;
            const __half2 h0 = __floats2half2_rn(sm2[0].x, sm2[0].y), h1 = __floats2half2_rn(sm2[1].x, sm2[1].y);
            *reinterpret_cast<uint2 *>(dst) =
                make_uint2(*reinterpret_cast<const uint32_t *>(&h0), *reinterpret_cast<const uint32_t *>(&h1));
            if (t == T - 1)   // the query avg[T-1] in full precision
              *reinterpret_cast<float4 *>(q0 + (size_t)(s * K::WT + wl) * UP + u) =
                  make_float4(0.5f * sm2[0].x, 0.5f * sm2[0].y, 0.5f * sm2[1].x, 0.5f * sm2[1].y);
          }
        }
        TC_TRACE(6);
      }
    }
    // projection of the last state h[T-1]
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      if (s == 1 && !live1) continue;
      mbar_wait(bar_done + 8 * s, (uint32_t)((T + extra) & 1));
      tc_fence_after();
      float pj[4];
      tmem_ld4(t_lane + (uint32_t)(s * K::TCOLS + K::NG + 4 * uq), pj);
      tmem_ld_wait();
      float4 o;
      o.x = pj[0] + __shfl_xor_sync(0xffffffffu, pj[0], 1);
      o.y = pj[1] + __shfl_xor_sync(0xffffffffu, pj[1], 1);
      o.z = pj[2] + __shfl_xor_sync(0xffffffffu, pj[2], 1);
      o.w = pj[3] + __shfl_xor_sync(0xffffffffu, pj[3], 1);
      o.x *= us.x; o.y *= us.x; o.z *= us.x; o.w *= us.x;
      if (dir == 0)
        *reinterpret_cast<float4 *>(proj0 + ((size_t)(s * K::WT + wl) * T + (T - 1)) * 16 + 4 * uq) = o;
    }
    tc_fence_before();
    }
    // ---- attention + FF + softmax + vote for the unit's tiles ------------------------------------
    __threadfence_block();
    gate_bar_sync();
#pragma unroll 1
    for (int s = 0; s < nt; ++s)
      attention_vote_sum_tile<UP, K::WT, TC_GATE_WARPS>(
          p, sum0 + (size_t)s * K::WT * T * UP, q0 + (size_t)s * K::WT * UP,
          proj0 + (size_t)s * K::WT * T * 16, tile_range(p, tile + s, K::WT), p.wpp, s_scale, s_score,
          p.smem_vote == 1 ? reinterpret_cast<float *>(s_A)            // A is idle: every MMA of the unit has completed
                           : (p.smem_vote == 2 ? reinterpret_cast<float *>(s_codes + 4 * (size_t)p.code_span) : nullptr));
    tile += nt;
  }

  // ---- teardown (the last "done" wait of every tile saw its MMAs complete) -----------------------
  tc_fence_before();
  gate_bar_sync();
#ifdef DGRP_TC_TRACE
  if (blockIdx.x == 0 && tid < 16 * 16) g_tc_trace[tid >> 4][(tid >> 3) & 1][tid & 7] += s_tc_trace[tid >> 4][(tid >> 3) & 1][tid & 7];
  if (blockIdx.x == 0 && tid < 16 * 8) g_tc_trace2[tid >> 3][tid & 7] += s_tc_trace2[tid >> 3][tid & 7];
#endif
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"(2 * K::TCOLS)
                 : "memory");
  }
}

template <int UP>
static size_t tc_smem_bytes(int T, int wpp, int code_span) {
  using K = TCfg<UP>;
  return (size_t)2 * K::B_BYTES + 2 * 2 * K::A_BYTES +
         sizeof(float) * ((size_t)10 * K::PSTRIDE + 2 * UP + (size_t)wpp * T) + 4 * (size_t)code_span + 128;
}

template <int UP>
static int launch_tc_t(dgrp_ctx *c, dgrp_model *m, FwdParams &p) {
  using K = TCfg<UP>;
  const int64_t n_windows = p.w_end - p.w_begin;
  if (n_windows <= 0 && p.w2_end <= p.w2_begin) return DGRP_OK;
  // windows per pass of the second phase: as many score rows as shared memory holds
  // staged base codes of a tile: 63 * step + T bytes; very large steps have no tcgen05 form
  const int64_t span = (int64_t)(K::WT - 1) * p.step + p.T;
  if (span > 16384) return DGRP_E_UNSUPPORTED;
  p.code_span = (int)((span + 15) & ~(int64_t)15);
  int wpp = K::WT;
  while (wpp > 8 && tc_smem_bytes<UP>(p.T, wpp, p.code_span) > 227 * 1024) wpp >>= 1;
  const size_t smem = tc_smem_bytes<UP>(p.T, wpp, p.code_span);
  if (smem > 227 * 1024) return DGRP_E_UNSUPPORTED;   // caller falls back to the fp32 kernel
  p.wpp = wpp;
  // the tile's span of rows, max-merged in the A operand's shared memory during the second phase
  // (1: in the A operand, idle in the second phase; 2: small models, whose A is smaller than the span -- a region of
  // its own behind the staged codes)
  const size_t vote_bytes = (size_t)span * p.C * sizeof(float);
  size_t smem_total = smem;
  p.smem_vote = 0;
  if (c->forward_smem_vote) {
    if (vote_bytes <= (size_t)2 * 2 * K::A_BYTES) p.smem_vote = 1;
    else if (smem + vote_bytes <= 227 * 1024) { p.smem_vote = 2; smem_total = smem + vote_bytes; }
  }
  if (p.query) return DGRP_OK;
  if (p.smem_vote) p.win_probs = nullptr;
  auto kern = gru_tc_attention_vote_kernel<UP>;
  DGRP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_total));
  const int64_t n_tiles = (n_windows > 0 ? (n_windows + K::WT - 1) / K::WT : 0) +
                          (p.w2_end > p.w2_begin ? (p.w2_end - p.w2_begin + K::WT - 1) / K::WT : 0);
  const int64_t n_pairs = (n_tiles + 1) / 2;
  const int grid = (int)(n_pairs < c->sm_count ? n_pairs : c->sm_count);
  const size_t rows = (size_t)grid * 2 * K::WT;   // window slots in flight
  DGRP_CHECK(c->avg.reserve(rows * p.T * UP * sizeof(__half) + rows * UP * sizeof(float)));
  DGRP_CHECK(c->io_c.reserve(rows * p.T * 16 * sizeof(float)));
  p.scratch = c->avg.as<float>();
  p.qbuf = reinterpret_cast<float *>(c->avg.as<unsigned char>() + rows * p.T * UP * sizeof(__half));
  p.ff2 = c->io_c.as<float>();
  // p.win_probs (window probabilities, max-merged by the caller's gather pass) or the atomic vote: forward.cu
  kern<<<grid, TC_THREADS, smem_total, c->stream>>>(p);
  c->launches++;
  DGRP_CUDA(cudaGetLastError());
  return DGRP_OK;
}

#ifdef DGRP_TC_TRACE
extern "C" int dgrp_debug_tc_trace(unsigned long long *out, int reset) {
  if (reset) {
    static unsigned long long zero[17][2][8];
    return (int)cudaMemcpyToSymbol(g_tc_trace, zero, sizeof(zero));
  }
  return (int)cudaMemcpyFromSymbol(out, g_tc_trace, sizeof(unsigned long long) * 17 * 2 * 8);
}
extern "C" int dgrp_debug_tc_trace2(unsigned long long *out, int reset) {
  if (reset) {
    static unsigned long long zero[16][8];
    return (int)cudaMemcpyToSymbol(g_tc_trace2, zero, sizeof(zero));
  }
  return (int)cudaMemcpyFromSymbol(out, g_tc_trace2, sizeof(unsigned long long) * 16 * 8);
}
#endif

// Returns DGRP_E_UNSUPPORTED when this model/shape has no tcgen05 form (the caller then uses the
// fp32 kernel): units > 64, or a window too long for the score buffer in shared memory.
int launch_forward_tc(dgrp_ctx *c, dgrp_model *m, FwdParams &p) {
  if (!m->d_Bsplit) return DGRP_E_UNSUPPORTED;
  p.Bsplit = m->d_Bsplit;
  p.b_unscale = ldexpf(1.0f, -(8 + m->b_shift));
  switch (m->UP) {
    case 32: return launch_tc_t<32>(c, m, p);
    case 64: return launch_tc_t<64>(c, m, p);
    default: return DGRP_E_UNSUPPORTED;
  }
}

}  // namespace dgrp
