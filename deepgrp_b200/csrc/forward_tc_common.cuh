// Pieces shared by the two tcgen05 forms of the forward (forward_tc.cu: two 128-row tiles in flight per SM,
// units <= 64; forward_tcw.cu: one tile per SM with N-split / CTA-pair MMAs, units <= 128 and LSTM): mbarrier,
// descriptor and TMEM wrappers, the operand split, the packed gate arithmetic and the second phase
// (attention scores, softmax over t, FF logits, class softmax, vote).
#pragma once
#include <cuda_fp16.h>

#include "forward_common.cuh"

namespace dgrp {

constexpr int TC_GATE_WARPS = 16;
constexpr int TC_THREADS = (TC_GATE_WARPS + 4) * 32;   // + one warpgroup: the issuer warp and three idle warps
constexpr int TC_GATE_REGS = 112, TC_AUX_REGS = 24;     // setmaxnreg split: the inc (16 warps x 16) must fit into what the dec releases (4 warps x 72);
                                                        // 120 (counting on the 4096 registers the launch leaves unallocated) HANGS at full grid -- measured, round 2
constexpr float kNegLog2e = -1.4426950408889634f;   // z, r columns are pre-scaled: ex2(arg) = e^{-x}
constexpr float kTwoLog2e = 2.8853900817779268f;    // h columns are pre-scaled:    ex2(arg) = e^{2x}

#ifdef DGRP_TC_TRACE
// Developer instrumentation (not compiled into the product): cycles of CTA 0's gate warps per segment
// of the step loop, [warp][tile slot][segment]: 0 wait for "done", 1 TMEM loads, 2 gates + A operand
// stores, 3 fences + arrive, 4 scratch stores + loop; [16][.][5..6] the issuer's wait / issue.
static __device__ unsigned long long g_tc_trace[17][2][8];
__shared__ unsigned int s_tc_trace[17][2][8];   // accumulated with fire-and-forget shared atomics
#define TC_TRACE_DECL unsigned int tr_t = (unsigned int)clock64()
#define TC_TRACE(seg)                                                         \
  do {                                                                        \
    const unsigned int now__ = (unsigned int)clock64();                       \
    if (lane == 0) atomicAdd(&s_tc_trace[warp][s][seg], now__ - tr_t);        \
    tr_t = now__;                                                             \
  } while (0)
#define TC_TRACE2(seg)                                                        \
  do {                                                                        \
    const unsigned int now__ = (unsigned int)clock64();                       \
    if (lane == 0) atomicAdd(&s_tc_trace2[warp][seg], now__ - tr_t);          \
    tr_t = now__;                                                             \
  } while (0)
__shared__ unsigned int s_tc_trace2[16][8];   // second phase: 0 scores, 1 barrier, 2 softmax over t, 3 vote, 4 barrier
static __device__ unsigned long long g_tc_trace2[16][8];
#else
#define TC_TRACE_DECL
#define TC_TRACE(seg)
#define TC_TRACE2(seg)
#endif

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        " selp.u32 %0, 1, 0, p;\n}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!done);
}
// the issuer's wait: back off between polls so that the spinning warp does not eat issue slots
__device__ __forceinline__ void mbar_wait_backoff(uint32_t bar, uint32_t parity) {
  uint32_t done;
  for (;;) {
    asm volatile(
        "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        " selp.u32 %0, 1, 0, p;\n}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) break;
    __nanosleep(64);
  }
}
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(lbo >> 4) << 16;
  d |= (uint64_t)(sbo >> 4) << 32;
  d |= 1ull << 46;  // descriptor version (sm_100)
  return d;         // layout_type = 0: no swizzle
}
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a, uint64_t b, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n"
      " tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}"
      ::"r"(d_tmem), "l"(a), "l"(b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
                 "=r"(r[7])
               : "r"(taddr)
               : "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, float (&v)[4]) {
  uint32_t r[4];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(taddr)
               : "memory");
#pragma unroll
  for (int i = 0; i < 4; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void fence_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// named barrier over the gate warps only (the issuer warp is in its own loop)
__device__ __forceinline__ void gate_bar_sync() {
  asm volatile("bar.sync 1, %0;" ::"n"(TC_GATE_WARPS * 32) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

// (a, b) * 2^8 = hi + lo in half-precision pieces (11 + 11 significant bits; the scale keeps the low piece a
// normal number for every |h| > 5e-4 and exact-to-2^-33 below); each output word packs a's piece (low half)
// and b's (high half).  The residual is formed with one packed FFMA2 (x - hi exactly, as the scalar
// subtraction would).
constexpr float kStateScale = 256.0f;
__device__ __forceinline__ void split2h(float2 ab, uint32_t &hi, uint32_t &lo) {
  const float2 x = __fmul2_rn(ab, make_float2(kStateScale, kStateScale));
  const __half2 h2 = __floats2half2_rn(x.x, x.y);
  hi = *reinterpret_cast<const uint32_t *>(&h2);
  const float2 hf = __half22float2(h2);
  const float2 r = __ffma2_rn(hf, make_float2(-1.0f, -1.0f), x);
  const __half2 l2 = __floats2half2_rn(r.x, r.y);
  lo = *reinterpret_cast<const uint32_t *>(&l2);
}

// The 16-byte core-matrix row that holds one_hot(x) * 2^8 (half precision, 0x5C00 = 256) for the
// input-table row `trow` (0..3 forward A,C,G,T; 4..7 the rc pass, already complemented; 8, 9 'N'):
// K position p = the base the table row stands for.
__device__ __forceinline__ uint4 onehot_row(int trow) {
  const int p = trow < 4 ? trow : (trow < 8 ? 7 - trow : 4);
  const uint32_t v = 0x5C00u << ((p & 1) * 16);
  const int j = p >> 1;
  return make_uint4(j == 0 ? v : 0u, j == 1 ? v : 0u, j == 2 ? v : 0u, 0u);
}

// GRU cell update for four units at once.  Packed fp32x2 arithmetic (FADD2 / FMUL2 / FFMA2 issue one
// instruction per pair, with the same IEEE rounding as the scalar forms); the accumulator and table
// values arrive pre-scaled (z, r by -log2 e; h by 2 log2 e):
//   z = 1/(1+2^sz) = 1/A, r = 1/(1+2^sr) = 1/B, hh = tanh = 1 - 2/D with D = 2^arg + 1, h' = hh + z (h - hh).
// The MUFU pipe (16 lanes/clk/SM) is what bounds this kernel, so reciprocals are shared: the four
// sigmoid denominators of two units cost ONE rcp (1/(A0 B0 A1 B1), then multiplied back), and so
// do the four tanh denominators of the quad: 3 ex2 + 0.75 rcp per unit instead of 3 + 2.  The clamps
// keep the products finite: sz, sr <= 28.85 is x >= -20 (sigmoid error < 2.1e-9), arg <= 30 is
// tanh = 1 - 2/(2^30 + 1), which rounds to 1.
__device__ __forceinline__ void sigmoid_pair(float2 sz, float2 sr, float2 &z, float2 &r) {
  const float2 one = make_float2(1.0f, 1.0f);
  const float2 ez = make_float2(ex2_approx(fminf(sz.x, 28.85f)), ex2_approx(fminf(sz.y, 28.85f)));
  const float2 er = make_float2(ex2_approx(fminf(sr.x, 28.85f)), ex2_approx(fminf(sr.y, 28.85f)));
  const float2 a = __fadd2_rn(ez, one), b = __fadd2_rn(er, one);
  const float2 ab = __fmul2_rn(a, b);
  const float inv = rcp_approx(ab.x * ab.y);
  const float2 iab = make_float2(inv * ab.y, inv * ab.x);   // 1/(a.x b.x), 1/(a.y b.y)
  z = __fmul2_rn(iab, b);
  r = __fmul2_rn(iab, a);
}
// The accumulators hold (state scale * weight scale) times the pre-activation and are multiplied by `us` on the
// way in.  The one-hot K columns of the MMA have already added the z / r input projection and the h gate's
// recurrent bias; only the h gate's input row `xh` stays outside r * (.) (reset_after=True).
__device__ __forceinline__ void gru_cell4(const float4 xh, const float *az, const float *ar, const float *ah, float *hp,
                                          float2 us, float2 &h01, float2 &h23) {
  const float2 one = make_float2(1.0f, 1.0f);
  float2 z0, r0, z1, r1;
  sigmoid_pair(__fmul2_rn(make_float2(az[0], az[1]), us), __fmul2_rn(make_float2(ar[0], ar[1]), us), z0, r0);
  sigmoid_pair(__fmul2_rn(make_float2(az[2], az[3]), us), __fmul2_rn(make_float2(ar[2], ar[3]), us), z1, r1);
  const float2 g0 = __fmul2_rn(make_float2(ah[0], ah[1]), us);
  const float2 g1 = __fmul2_rn(make_float2(ah[2], ah[3]), us);
  const float2 t0 = __ffma2_rn(r0, g0, make_float2(xh.x, xh.y));
  const float2 t1 = __ffma2_rn(r1, g1, make_float2(xh.z, xh.w));
  const float2 d0 = __fadd2_rn(make_float2(ex2_approx(fminf(t0.x, 30.0f)), ex2_approx(fminf(t0.y, 30.0f))), one);
  const float2 d1 = __fadd2_rn(make_float2(ex2_approx(fminf(t1.x, 30.0f)), ex2_approx(fminf(t1.y, 30.0f))), one);
  const float2 m = __fmul2_rn(d0, d1);              // {d0.x d1.x, d0.y d1.y}
  const float inv = rcp_approx(m.x * m.y);
  const float2 j = make_float2(inv * m.y, inv * m.x);
  const float2 i0 = __fmul2_rn(j, d1), i1 = __fmul2_rn(j, d0);   // 1/d0, 1/d1
  const float2 m2 = make_float2(-2.0f, -2.0f), neg1 = make_float2(-1.0f, -1.0f);
  const float2 hh0 = __ffma2_rn(m2, i0, one), hh1 = __ffma2_rn(m2, i1, one);
  h01 = __ffma2_rn(z0, __ffma2_rn(hh0, neg1, make_float2(hp[0], hp[1])), hh0);   // hh + z (h - hh)
  h23 = __ffma2_rn(z1, __ffma2_rn(hh1, neg1, make_float2(hp[2], hp[3])), hh1);
  hp[0] = h01.x; hp[1] = h01.y; hp[2] = h23.x; hp[3] = h23.y;
}

// Tiles of a launch: those of windows [w_begin, w_end), then those of [w2_begin, w2_end).
struct TileRange {
  int64_t w0;       // first window of the tile
  int64_t lo, hi;   // the window range it belongs to
};
__device__ __forceinline__ int64_t range_tiles(int64_t lo, int64_t hi, int WT) { return hi > lo ? (hi - lo + WT - 1) / WT : 0; }
__device__ __forceinline__ int64_t launch_tiles(const FwdParams &p, int WT) {
  return range_tiles(p.w_begin, p.w_end, WT) + range_tiles(p.w2_begin, p.w2_end, WT);
}
__device__ __forceinline__ TileRange tile_range(const FwdParams &p, int64_t tile, int WT) {
  const int64_t ta = range_tiles(p.w_begin, p.w_end, WT);
  TileRange r;
  if (tile < ta) { r.w0 = p.w_begin + tile * WT; r.lo = p.w_begin; r.hi = p.w_end; }
  else { r.w0 = p.w2_begin + (tile - ta) * WT; r.lo = p.w2_begin; r.hi = p.w2_end; }
  return r;
}

// Second phase for one tile, in passes of WPP windows (WPP * T floats of scores fit in shared memory).
//   sum   [T][UP/8 chunks][64 windows][8 units]  h_fwd[t] + h_rc[t]; the layout the gate warps can
//         write with full 128-byte lines (a warp's 32 rows are 16 windows x 2 directions x 4 units)
//   q     [64][UP]       avg[T-1]
//   proj  [64][T][16]    avg[t].K: ctx half in 0..4, avg half in 8..12
// (a) scores: score[t] = sum_u scale[u] tanh(q[u] + avg[t][u]) = S - 2 sum_u scale[u] / D[t][u] with
//     D = e^{2(q+avg)} + 1 and S = sum_u scale[u] the same for every t, so the softmax over t only needs
//     the second term.  A warp takes 8 adjacent windows x a slice of t; a lane takes one window and every
//     fourth chunk, so each load instruction reads whole 128-byte lines; four denominators share one rcp.
// (b) one warp per window, lanes over t: softmax over t, logits, class softmax and the max-vote.
// Ask the L2 to fetch `bytes` (multiple of 16) from HBM: one instruction, no registers, no L1 miss entries.
// The second phase reads scratch that left the L2 long ago; a single SM's demand loads sustain only
// ~17 B/clk against HBM latency, but ~4x that against L2 hits.
__device__ __forceinline__ void l2_prefetch(const void *ptr, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(ptr), "r"(bytes) : "memory");
}
// One 32-byte sector in one request (LDG.256): the softmax / vote passes read one sector of a `proj` row
// per lane, every lane a different line, and the LSU resolves one line per cycle -- the request count,
// not the bytes, bounds those passes.  `p` must be 32-byte aligned.
__device__ __forceinline__ void ldg256(const float *p, float (&v)[8]) {
  asm volatile("ld.global.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
               : "l"(p));
}
__device__ __forceinline__ float tanh_mufu(float x) {   // MUFU.TANH: relative error 2^-11
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float exp_fast(float x) {   // e^x through ex2.approx (2 ulp), e^{-inf} = 0
  return ex2_approx(x * 1.4426950408889634f);
}
template <int UP, int WT, int NWARPS>
__device__ __forceinline__ void attention_vote_sum_tile(const FwdParams &p, const __half *sum, const float *qbuf,
                                                        const float *proj, const TileRange tr, int wpp,
                                                        const float *s_scale, float *s_score, float *s_vote = nullptr) {
  const int64_t w_tile0 = tr.w0;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int T = p.T, C = p.C;
  // Shared-memory vote (s_vote: float[(WT - 1) * step + T][C], the idle A operand): the tile's windows overlap each
  // other, so their probabilities are max-merged on chip (shared-memory atomicMax on the int view, probabilities
  // are > 0) and every row of the tile's span leaves the SM once -- a plain store for the rows only this tile's
  // windows cover, a global atomicMax for the T - step rows at either end that the neighbouring tiles share and
  // for rows the displaced last batch (prediction.py:105) may land on.  The [windows][T][C] probabilities never
  // touch HBM (SURVEY.md section 7 step 6).
  const int vspan = (WT - 1) * p.step + T;
  if (s_vote) {
    for (int i = tid; i < vspan * C; i += NWARPS * 32) s_vote[i] = 0.f;   // ordered before the votes by the pass barrier
  }
  constexpr int NCH = UP / 8;          // 8-unit chunks per avg row
  constexpr int CPL = NCH / 4;         // chunks per lane: cj, cj + 4, ...
  constexpr int CH = CPL > 2 ? 2 : CPL;   // chunks per lane and sweep
  constexpr int UNR = 4;               // t's in flight per lane (scores)
  constexpr int PU = 11;               // rows in flight per lane (softmax / vote passes): all of T <= 352 at once
  TC_TRACE_DECL;
  for (int w0 = 0; w0 < WT; w0 += wpp) {
    if (w_tile0 + w0 >= tr.hi) break;
    if (p.attention) {
      const int ngrp = wpp >> 3, grp = warp % ngrp, sl = warp / ngrp, nsl = NWARPS / ngrp;
      const int wi = lane & 7, cj = lane >> 3;
      const int wl = w0 + grp * 8 + wi;
      const int t_begin = (int)((int64_t)T * sl / nsl), t_end = (int)((int64_t)T * (sl + 1) / nsl);
      // units > 64: two sweeps over t, each over half of the lane's chunks (the per-chunk constants of all
      // four chunks would not fit the register budget); the second sweep adds to the first one's scores
#pragma unroll 1
      for (int i0 = 0; i0 < CPL; i0 += CH) {
      float q2[CH][8], sc2[CH][8];   // q[u], scale[u]: score = sum_u scale[u] tanh.approx(q[u] + sum/2)
#pragma unroll
      for (int i = 0; i < CH; ++i) {
        const int u0 = (cj + 4 * (i0 + i)) * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          q2[i][j] = qbuf[(size_t)wl * UP + u0 + j];
          sc2[i][j] = s_scale[u0 + j];
        }
      }
      // the pass's windows are contiguous per (t, chunk): [pass][t][chunk][wpp windows][8 units]
      const __half *sum_pass = sum + (size_t)(w0 / wpp) * T * NCH * wpp * 8;
      const __half *base = sum_pass + ((size_t)(cj + 4 * i0) * wpp + (grp * 8 + wi)) * 8;
      // one warp per t-slice keeps the L2 PF_AHEAD rows ahead of the demand loads, PF_BLOCK rows at a time
      // (a t-row of the tile is NCH * WT * 8 contiguous elements)
      constexpr int PF_BLOCK = 4, PF_AHEAD = 12;
      const uint32_t ROW_BYTES = (uint32_t)(NCH * wpp * 8 * sizeof(__half));
      if (grp == 0 && lane == 0 && i0 == 0) {
        const int n0 = min(PF_AHEAD, t_end - t_begin);
        l2_prefetch(sum_pass + (size_t)t_begin * NCH * wpp * 8, (uint32_t)n0 * ROW_BYTES);
      }
      for (int t0 = t_begin; t0 < t_end; t0 += UNR) {
        if (grp == 0 && lane == 0 && i0 == 0 && (t0 - t_begin) % PF_BLOCK == 0) {
          const int ta = t0 + PF_AHEAD;
          if (ta < t_end) l2_prefetch(sum_pass + (size_t)ta * NCH * wpp * 8, (uint32_t)min(PF_BLOCK, t_end - ta) * ROW_BYTES);
        }
        uint4 v[UNR][CH];
#pragma unroll
        for (int k = 0; k < UNR; ++k) {
          const int t = min(t0 + k, t_end - 1);
#pragma unroll
          for (int i = 0; i < CH; ++i)
            v[k][i] = __ldcs(reinterpret_cast<const uint4 *>(base + ((size_t)t * NCH + 4 * i) * wpp * 8));
        }
#pragma unroll
        for (int k = 0; k < UNR; ++k) {
          float sacc = 0.f;
#pragma unroll
          for (int i = 0; i < CH; ++i) {
            float x[8];   // h_fwd[t] + h_rc[t] of 8 units
            const uint32_t wv[4] = {v[k][i].x, v[k][i].y, v[k][i].z, v[k][i].w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float2 f = __half22float2(*reinterpret_cast<const __half2 *>(&wv[j]));
              x[2 * j] = f.x; x[2 * j + 1] = f.y;
            }
            // The half-precision `sum` already limits a score to ~2^-11 per term; MUFU.TANH (tanh.approx.f32, relative
            // error 2^-11) is the matching arithmetic: 3.5 instead of ~8.5 instructions and 1 instead of 1.25 MUFU
            // operations per (t, unit) of the exact form -2 sum_u scale[u] / (e^{2(q + sum/2)} + 1).  Measured against
            // the exact form: max |dp| 3.5e-8 on random-init weights, 3.5e-5 on the x4 set (1.4e-5 from the
            // half-precision sum alone).
#pragma unroll
            for (int j = 0; j < 8; ++j) sacc = fmaf(sc2[i][j], tanh_mufu(fmaf(x[j], 0.5f, q2[i][j])), sacc);
          }
          sacc += __shfl_xor_sync(0xffffffffu, sacc, 8);
          sacc += __shfl_xor_sync(0xffffffffu, sacc, 16);
          if (cj == 0 && t0 + k < t_end) {
            float *dst = s_score + (size_t)(grp * 8 + wi) * T + t0 + k;
            *dst = (CH < CPL && i0 > 0) ? *dst + sacc : sacc;   // the same thread wrote the first sweep's value
          }
        }
      }
      }
    }
    if (lane == 0 && warp < wpp) l2_prefetch(proj + (size_t)(w0 + warp) * T * 16, (uint32_t)T * 64u);
    TC_TRACE2(0);
    asm volatile("bar.sync 1, %0;" ::"n"(NWARPS * 32) : "memory");
    TC_TRACE2(1);
    for (int wq = warp; wq < wpp; wq += NWARPS) {
      const int wl = w0 + wq;
      if (lane == 0 && wq + NWARPS < wpp)   // the next window of this warp
        l2_prefetch(proj + (size_t)(wl + NWARPS) * T * 16, (uint32_t)T * 64u);
      const int64_t w = w_tile0 + wl;
      if (w >= tr.hi) break;
      const float *pr = proj + (size_t)wl * T * 16;
      const float *sc = s_score + (size_t)wq * T;
      float ctxk[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
      if (p.attention) {
        // softmax over t and ctx.K1 = sum_t a_t (avg[t].K1); four rows per lane in flight
        float m_run = -INFINITY, l_run = 0.f, cacc[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
        for (int t0 = lane; t0 < T; t0 += 32 * PU) {
          float sv[PU], k1[PU][5];
#pragma unroll
          for (int k = 0; k < PU; ++k) {
            const int t = t0 + 32 * k;
            const bool ok = t < T;
            float row[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            if (ok) ldg256(pr + (size_t)t * 16, row);
#pragma unroll
            for (int c = 0; c < 5; ++c) k1[k][c] = row[c];
            sv[k] = ok ? sc[t] : -INFINITY;
          }
          float m_new = m_run;
#pragma unroll
          for (int k = 0; k < PU; ++k) m_new = fmaxf(m_new, sv[k]);
          if (m_new > -INFINITY) {
            const float corr = exp_fast(m_run - m_new);   // exp(-inf) = 0 on the first rows
            l_run *= corr;
#pragma unroll
            for (int c = 0; c < 5; ++c) cacc[c] *= corr;
#pragma unroll
            for (int k = 0; k < PU; ++k) {
              const float e = exp_fast(sv[k] - m_new);
              l_run += e;
#pragma unroll
              for (int c = 0; c < 5; ++c) cacc[c] = fmaf(e, k1[k][c], cacc[c]);
            }
            m_run = m_new;
          }
        }
        float m_all = m_run;
        for (int off = 16; off > 0; off >>= 1) m_all = fmaxf(m_all, __shfl_xor_sync(0xffffffffu, m_all, off));
        const float f = (m_run == -INFINITY) ? 0.f : exp_fast(m_run - m_all);
        float l = l_run * f;
#pragma unroll
        for (int c = 0; c < 5; ++c) cacc[c] *= f;
        for (int off = 16; off > 0; off >>= 1) {
          l += __shfl_xor_sync(0xffffffffu, l, off);
#pragma unroll
          for (int c = 0; c < 5; ++c) cacc[c] += __shfl_xor_sync(0xffffffffu, cacc[c], off);
        }
#pragma unroll
        for (int c = 0; c < 5; ++c) ctxk[c] = cacc[c] / l;
      }
      TC_TRACE2(2);
      // logits[t] = ctx.K1 + avg[t].K2 + b ; softmax over classes ; vote
      const int64_t place = (w < p.full_windows ? w * (int64_t)p.step
                                                : p.tail_base + (w - p.full_windows) * (int64_t)p.step) -
                            p.pred_row0;
      float cb[5];
#pragma unroll
      for (int c = 0; c < 5; ++c) cb[c] = c < C ? ctxk[c] + p.ffb[c] : 0.f;
      for (int t0 = lane; t0 < T; t0 += 32 * PU) {
        float k2[PU][5];
#pragma unroll
        for (int k = 0; k < PU; ++k) {
          const int t = t0 + 32 * k;
          const bool ok = t < T;
          float row[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
          if (ok) ldg256(pr + (size_t)t * 16 + 8, row);
#pragma unroll
          for (int c = 0; c < 5; ++c) k2[k][c] = row[c];
        }
#pragma unroll
        for (int k = 0; k < PU; ++k) {
          const int t = t0 + 32 * k;
          float lg[5], mx = -INFINITY;
#pragma unroll
          for (int c = 0; c < 5; ++c) {
            lg[c] = c < C ? k2[k][c] + cb[c] : -INFINITY;
            mx = fmaxf(mx, lg[c]);
          }
          float sum_e = 0.f;
#pragma unroll
          for (int c = 0; c < 5; ++c) { lg[c] = c < C ? exp_fast(lg[c] - mx) : 0.f; sum_e += lg[c]; }
          const float inv = 1.0f / sum_e;
          if (s_vote && w < p.full_windows) {
            if (t < T) {
              int *dst = reinterpret_cast<int *>(s_vote) + ((int)(w - w_tile0) * p.step + t) * C;
#pragma unroll
              for (int c = 0; c < 5; ++c)
                if (c < C) atomicMax(dst + c, __float_as_int(lg[c] * inv));
            }
          } else if (p.win_probs) {
            // plain stores of the window's probabilities; vote_gather_kernel max-merges them
            if (t < T) {
              float *dst = p.win_probs + ((size_t)(w - p.w_begin) * T + t) * C;
#pragma unroll
              for (int c = 0; c < 5; ++c)
                if (c < C) dst[c] = lg[c] * inv;
            }
          } else {
            const int64_t r = place + t;
            if (t < T && r >= 0 && r < p.pred_rows) {
              int *dst = reinterpret_cast<int *>(p.pred + (size_t)r * C);
#pragma unroll
              for (int c = 0; c < 5; ++c)
                if (c < C) atomicMax(dst + c, __float_as_int(lg[c] * inv));   // probs > 0
            }
          }
        }
      }
    }
    TC_TRACE2(3);
    asm volatile("bar.sync 1, %0;" ::"n"(NWARPS * 32) : "memory");   // s_score is rewritten by the next pass
    TC_TRACE2(4);
  }
  if (s_vote) {
    // the tile's merged rows -> pred.  Row r of the span is record row w_tile0 * step + r.
    const int64_t row0 = w_tile0 * (int64_t)p.step - p.pred_row0;
    const int64_t tail_lo = p.tail_base - p.pred_row0;                      // rows the displaced batch can touch
    const int64_t w_max = p.w2_end > p.w2_begin && p.w2_end > p.w_end ? p.w2_end : p.w_end;   // the launch's last window
    const int64_t tail_hi = tail_lo + (w_max > p.full_windows ? (w_max - p.full_windows - 1) * (int64_t)p.step + T : 0);
    const bool first = w_tile0 == tr.lo;
    const bool last = w_tile0 + WT >= (p.full_windows < tr.hi ? p.full_windows : tr.hi);
    const int own_lo = first ? 0 : T - p.step;                             // below: shared with the previous tile
    const int own_hi = last ? vspan : WT * p.step;                         // from here on: shared with the next tile
    for (int r = tid; r < vspan; r += NWARPS * 32) {
      const int64_t g = row0 + r;
      if (g < 0 || g >= p.pred_rows) continue;
      float v[5];
      bool any = false;
#pragma unroll
      for (int c = 0; c < 5; ++c) { v[c] = c < C ? s_vote[r * C + c] : 0.f; any |= v[c] != 0.f; }
      if (!any) continue;                                                   // no window of this tile covers the row
      float *dst = p.pred + (size_t)g * C;
      const bool shared_row = r < own_lo || r >= own_hi || (g >= tail_lo && g < tail_hi);
      if (shared_row) {
#pragma unroll
        for (int c = 0; c < 5; ++c)
          if (c < C) atomicMax(reinterpret_cast<int *>(dst) + c, __float_as_int(v[c]));
      } else {
#pragma unroll
        for (int c = 0; c < 5; ++c)
          if (c < C) dst[c] = v[c];
      }
    }
    asm volatile("bar.sync 1, %0;" ::"n"(NWARPS * 32) : "memory");   // the next tile zeroes s_vote
  }
}

}  // namespace dgrp
