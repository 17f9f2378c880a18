// Shared pieces of the two forward kernels (fp32 FFMA form in forward.cu, tcgen05 form in
// forward_tc.cu): launch parameters and the attention + FF + softmax + vote phase.
#pragma once
#include "dgrp_internal.cuh"

namespace dgrp {

constexpr int FWD_THREADS = 256;

struct FwdParams {
  const uint8_t *codes;   // code mode
  int64_t codes_base;     // record position of codes[0]
  const float *dense;     // dense mode: [n][T][5] windows (predict_on_batch semantics)
  float *probs_out;       // dense mode: [n][T][C]
  int64_t w_begin, w_end; // window index range
  int64_t w2_begin, w2_end;   // tcgen05 forms with the vote in shared memory: a second window range run by the same
                          // launch behind the first (tiles never mix the two) -- the windows of the displaced
                          // last batch (prediction.py:105) that land in a position range; empty: w2_end <= w2_begin
  int T, U, C, step, attention;
  int64_t full_windows, tail_base;
  const float *P, *Wk, *b0, *Rp, *b1, *scale, *ffk, *ffb;
  const uint16_t *Bsplit; // tcgen05 form: fp16 hi|lo pieces of [R | K/2]^T, UMMA layout
  int code_span;          // tcgen05 form: bytes per tile of the staged base codes (multiple of 16)
  int wpp;                // tcgen05 form: windows per pass of the second phase (8..64)
  float b_unscale;        // tcgen05 form: 1 / (state scale * weight scale), applied to the accumulator
  float *scratch, *ff2, *qbuf;
  float *pred;
  int64_t pred_row0, pred_rows;
  int smem_vote;          // tcgen05 form: max-merge a tile's windows in shared memory (the idle A operand) and write
                          // every row of the tile's span once; set by the launcher when the span fits
  int query;              // launcher: only decide (smem_vote, support) and return, do not launch
  float *win_probs;       // tcgen05 form: [w - w_begin][T][C] window probabilities instead of the vote
                          // (merged afterwards by vote_gather_kernel), or null: atomicMax into pred
};

// s_att[u][12] = {FF kernel ctx half [5], FF kernel avg half [5], attention scale, 0}
// 1 - 2/(e^{2x}+1): absolute error ~1e-7 (fp32 rounding of the quotient), exact limits +-1
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float tanh_fast(float x) {
  const float e = ex2_approx(x * 2.8853900817779268f);   // e^{2x}
  return fmaf(-2.0f, rcp_approx(e + 1.0f), 1.0f);
}

template <int UP, int NTHREADS = FWD_THREADS>
__device__ __forceinline__ void stage_attention_table(const FwdParams &p, float *s_att, int tid) {
  const int U = p.U, C = p.C;
  for (int i = tid; i < UP * 12; i += NTHREADS) {
    const int u = i / 12, j = i % 12;
    float v = 0.f;
    if (u < U) {
      if (p.attention) {
        if (j < 5) v = j < C ? p.ffk[(size_t)u * C + j] : 0.f;                  // ctx half (first)
        else if (j < 10) v = (j - 5) < C ? p.ffk[(size_t)(U + u) * C + (j - 5)] : 0.f;  // avg half
        else if (j == 10) v = p.scale[u];
      } else if (j >= 5 && j < 10) {
        v = (j - 5) < C ? p.ffk[(size_t)u * C + (j - 5)] : 0.f;
      }
    }
    s_att[i] = v;
  }
}

// Phase 2 for one tile of WT windows whose avg[t] rows are in `scratch` ([WT][T][UP]): additive
// attention (model.py:315), FF + softmax (model.py:325-329) and the max-vote (maxcalc.c:10-24),
// one warp per window.  Must be called by all FWD_THREADS threads after a __syncthreads().
// FAST: approximate-intrinsic tanh and a fully unrolled unit loop (all UP columns; the padded ones are
// zero in scratch and in s_att) so that the row's loads are in flight together.
template <int UP, bool DENSE, int WT, int NWARPS = FWD_THREADS / 32, bool FAST = false>
__device__ __forceinline__ void attention_vote_tile(const FwdParams &p, const float *scratch,
                                                    float *ff2, int64_t w_tile0, const float *s_att,
                                                    float *s_q, float *s_score) {
  const int tid = threadIdx.x;
  const int T = p.T, U = p.U, C = p.C;
  const int KU = FAST ? UP : ((U + 3) & ~3);
  {
    const int warp = tid >> 5, lane = tid & 31;
    if (warp >= NWARPS) return;
    float *qv = s_q + warp * UP;
    float *sc = s_score + (size_t)warp * T;
    for (int wl = warp; wl < WT; wl += NWARPS) {
      const int64_t w = w_tile0 + wl;
      if (w >= p.w_end) break;
      const float *av = scratch + (size_t)wl * T * UP;
      float *f2 = ff2 + (size_t)wl * T * 5;
      // query = (h_fwd[T-1] + h_rc[T-1]) / 2 = avg[T-1]   (model.py:311)
      for (int u = lane; u < UP; u += 32) qv[u] = av[(size_t)(T - 1) * UP + u];
      __syncwarp();
      float m_run = -INFINITY, l_run = 0.f, cacc[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
      for (int t = lane; t < T; t += 32) {
        const float *row = av + (size_t)t * UP;
        float s = 0.f, k1[5] = {0.f, 0.f, 0.f, 0.f, 0.f}, k2[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll(FAST ? UP / 4 : 1)
        for (int u = 0; u < KU; u += 4) {
          const float4 v4 = *reinterpret_cast<const float4 *>(row + u);
          const float vv[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float *a = s_att + (u + j) * 12;
            const float4 a0 = *reinterpret_cast<const float4 *>(a);
            const float4 a1 = *reinterpret_cast<const float4 *>(a + 4);
            const float4 a2 = *reinterpret_cast<const float4 *>(a + 8);
            const float v = vv[j];
            if (p.attention) {
              s = fmaf(a2.z, FAST ? tanh_fast(qv[u + j] + v) : tanhf(qv[u + j] + v), s);
              k1[0] = fmaf(v, a0.x, k1[0]); k1[1] = fmaf(v, a0.y, k1[1]);
              k1[2] = fmaf(v, a0.z, k1[2]); k1[3] = fmaf(v, a0.w, k1[3]);
              k1[4] = fmaf(v, a1.x, k1[4]);
            }
            k2[0] = fmaf(v, a1.y, k2[0]); k2[1] = fmaf(v, a1.z, k2[1]);
            k2[2] = fmaf(v, a1.w, k2[2]); k2[3] = fmaf(v, a2.x, k2[3]);
            k2[4] = fmaf(v, a2.y, k2[4]);
          }
        }
#pragma unroll
        for (int c = 0; c < 5; ++c) f2[(size_t)t * 5 + c] = k2[c];
        if (p.attention) {
          sc[t] = s;
          // online softmax over t of (score, avg[t].K1)
          const float m_new = fmaxf(m_run, s);
          const float corr = __expf(m_run - m_new);   // exp(-inf) = 0 on the first element
          const float e = expf(s - m_new);
          l_run = l_run * corr + e;
#pragma unroll
          for (int c = 0; c < 5; ++c) cacc[c] = cacc[c] * corr + e * k1[c];
          m_run = m_new;
        }
      }
      float ctxk[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
      if (p.attention) {
        float m_all = m_run;
        for (int off = 16; off > 0; off >>= 1) m_all = fmaxf(m_all, __shfl_xor_sync(0xffffffffu, m_all, off));
        const float f = (m_run == -INFINITY) ? 0.f : expf(m_run - m_all);
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
      __syncwarp();
      // logits[t] = ctx.K1 + avg[t].K2 + b ; softmax over classes ; vote
      int64_t place;
      if (DENSE) place = 0;
      else place = (w < p.full_windows ? w * (int64_t)p.step
                                       : p.tail_base + (w - p.full_windows) * (int64_t)p.step) -
                   p.pred_row0;
      for (int t = lane; t < T; t += 32) {
        float lg[5], mx = -INFINITY;
#pragma unroll
        for (int c = 0; c < 5; ++c) {
          lg[c] = c < C ? (ctxk[c] + f2[(size_t)t * 5 + c]) + p.ffb[c] : -INFINITY;
          mx = fmaxf(mx, lg[c]);
        }
        float sum = 0.f;
#pragma unroll
        for (int c = 0; c < 5; ++c) { lg[c] = c < C ? expf(lg[c] - mx) : 0.f; sum += lg[c]; }
        if (DENSE) {
          float *dst = p.probs_out + ((size_t)w * T + t) * C;
#pragma unroll
          for (int c = 0; c < 5; ++c) if (c < C) dst[c] = lg[c] / sum;
        } else {
          const int64_t r = place + t;
          if (r >= 0 && r < p.pred_rows) {
            int *dst = reinterpret_cast<int *>(p.pred + (size_t)r * C);
#pragma unroll
            for (int c = 0; c < 5; ++c)
              if (c < C) atomicMax(dst + c, __float_as_int(lg[c] / sum));   // probs > 0
          }
        }
      }
      __syncwarp();
    }
  }
}

}  // namespace dgrp
