// Training of GRU models (rnn="GRU", reset_after=True, units <= 64, n_classes <= MODEL_CMAX): forward with saved
// state, loss + head backward, BPTT, deterministic weight-gradient reduction and the optimiser update, all fp32 on CUDA
// cores.  The model is the one forward.cu computes (SURVEY.md section 3.2); the loss is Keras'
// categorical_crossentropy on the softmax probabilities, averaged over every position of the batch.
//
// Rows: a training step has 2n independent recurrences (window b, direction dir), row = 2b + dir.  A CTA runs
// TR_ROWS of them in lock step (256 threads = TR_ROWS rows x 64 units) with R in shared memory, so a 256-window
// batch is 128 CTAs -- the prediction kernels' 64-window tiles would give 4.
//
// Layout in HBM (rows = 2n, N = rows * T, U4 = 4U)
//   W      f32[P]            parameters, the Keras arrays concatenated (TrainLayout): kernel [5,3U],
//                            recurrent [U,3U], bias [2,3U], scale [U] (attention), FF kernel [F,C], FF bias [C]
//   Hs     f32[rows][T][U]   h after each step
//   GS     f32[rows][T][4][U]  z, r, hh, mh_h = (h.R)_h + b1_h of each step
//   D      f32[rows][T][U4]  dz, dr, da_h, da_h*r of each step (BPTT output, reduction input)
//   avg    f32[n][T][U]      (h_fwd[t] + h_rc[t]) / 2
//   dhin   f32[n][T][U]      dL/dh that the head adds at step t (the same for both directions)
//   hpart  f32[n][HP]        per-window head gradients: FF kernel, FF bias, scale
//   rpart  f32[chunks][KA][U4]  per-chunk partial products of the reduction
//   lpart  f32[n]            per-window sum of the position losses
//
// Determinism: every sum runs in a fixed order (thread-sequential loops, fixed-shape shuffle trees, per-chunk
// partials summed in chunk order); there are no float atomics, so a step is bit-reproducible on one GPU.
#include "dgrp_internal.cuh"

namespace dgrp {

constexpr int TR_ROWS = 4;          // recurrences per CTA (forward, BPTT)
constexpr int TR_THREADS = 256;     // TR_ROWS x TR_UMAX
constexpr int TR_UMAX = 64;
constexpr int TR_KAMAX = TR_UMAX + 6;   // reduction rows: h_prev[U], 1 (bias), one-hot x dropout scale [5]
constexpr int TR_TILE = 32;         // reduction items staged per pass
constexpr int TR_EVAL_CHUNK = 1024; // windows per forward pass of an evaluation
static_assert(TR_CMAX >= MODEL_CMAX, "the head kernel holds every class of a model in registers");

struct TrainArgs {
  int T, U, C, att, n;
  TrainLayout L;
  const float *w;
  const uint8_t *codes, *ymask;
  const int64_t *starts;
  const uint8_t *keep;   // [n][2][5] or null (evaluation: no dropout)
  float keep_scale;      // 1 / (1 - dropout)
  float inv_positions;   // 1 / (n * T)
  int backward;
  float *Hs, *GS, *D, *avg, *dhin, *probs, *hpart, *rpart, *lpart, *grad;
  int chunks;
};

__device__ __forceinline__ float tr_sigmoid(float x) { return 1.0f / (1.0f + expf(-x)); }

__device__ __forceinline__ int tr_code(const TrainArgs &a, int row, int t, float *scale) {
  const int b = row >> 1, dir = row & 1;
  const int64_t pos = a.starts[b] + (dir ? (a.T - 1 - t) : t);
  int code = a.codes[pos];
  if (dir && code < 4) code = 3 - code;   // the reverse complement's channel (model.py:233-237)
  if (scale) *scale = a.keep ? (a.keep[(b * 2 + dir) * 5 + code] ? a.keep_scale : 0.f) : 1.f;
  return code;
}

// ---- forward with saved state -------------------------------------------------------------------------------
__global__ void __launch_bounds__(TR_THREADS) train_forward_kernel(const TrainArgs a) {
  extern __shared__ __align__(16) float sm[];
  const int U = a.U, G3 = 3 * U, RS = G3 + 1, T = a.T;
  float *sR = sm;                      // [U][RS]
  float *sK = sR + U * RS;             // [5][3U]
  float *sb0 = sK + 5 * G3;            // [3U]
  float *sb1 = sb0 + G3;               // [3U]
  float *sh = sb1 + G3;                // [ROWS][U]   h of the previous step
  float *smh = sh + TR_ROWS * U;       // [ROWS][3U]  h.R + b1
  const int tid = threadIdx.x;
  for (int i = tid; i < U * G3; i += TR_THREADS) sR[(i / G3) * RS + i % G3] = a.w[a.L.oR + i];
  for (int i = tid; i < 5 * G3; i += TR_THREADS) sK[i] = a.w[a.L.oK + i];
  for (int i = tid; i < G3; i += TR_THREADS) { sb0[i] = a.w[a.L.oB + i]; sb1[i] = a.w[a.L.oB + G3 + i]; }
  for (int i = tid; i < TR_ROWS * U; i += TR_THREADS) sh[i] = 0.f;
  const int nrows = 2 * a.n;
  const int q = tid / TR_UMAX, u = tid % TR_UMAX;
  const int row = blockIdx.x * TR_ROWS + q;
  const bool act = u < U && row < nrows;
  __syncthreads();
  float h = 0.f;
  for (int t = 0; t < T; ++t) {
    if (tid < G3) {   // column tid of h.R for the CTA's rows, k ascending
      float acc[TR_ROWS];
#pragma unroll
      for (int r = 0; r < TR_ROWS; ++r) acc[r] = 0.f;
      for (int k = 0; k < U; ++k) {
        const float rw = sR[k * RS + tid];
#pragma unroll
        for (int r = 0; r < TR_ROWS; ++r) acc[r] = fmaf(sh[r * U + k], rw, acc[r]);
      }
#pragma unroll
      for (int r = 0; r < TR_ROWS; ++r) smh[r * G3 + tid] = acc[r] + sb1[tid];
    }
    __syncthreads();
    if (act) {
      float s;
      const int code = tr_code(a, row, t, &s);
      const float *kr = sK + code * G3;
      const float *mh = smh + q * G3;
      const float mxz = fmaf(s, kr[u], sb0[u]);
      const float mxr = fmaf(s, kr[U + u], sb0[U + u]);
      const float mxh = fmaf(s, kr[2 * U + u], sb0[2 * U + u]);
      const float z = tr_sigmoid(mxz + mh[u]);
      const float r = tr_sigmoid(mxr + mh[U + u]);
      const float hh = tanhf(mxh + r * mh[2 * U + u]);
      h = z * h + (1.0f - z) * hh;
      sh[q * U + u] = h;
      const size_t it = (size_t)row * T + t;
      a.Hs[it * U + u] = h;
      float *gs = a.GS + it * 4 * U;
      gs[u] = z; gs[U + u] = r; gs[2 * U + u] = hh; gs[3 * U + u] = mh[2 * U + u];
    }
    __syncthreads();
  }
}

// ---- head: attention, FF, softmax, loss and their backward; one CTA per window ------------------------------
__device__ __forceinline__ float tr_warp_sum(float v) {
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}
// fixed-shape block reduction (sum or max); every thread gets the result
template <bool MAX>
__device__ float tr_block_reduce(float v, float *sred) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int off = 16; off > 0; off >>= 1) {
    const float o = __shfl_xor_sync(0xffffffffu, v, off);
    v = MAX ? fmaxf(v, o) : v + o;
  }
  __syncthreads();
  if (lane == 0) sred[warp] = v;
  __syncthreads();
  v = sred[0];
  for (int w = 1; w < TR_THREADS / 32; ++w) v = MAX ? fmaxf(v, sred[w]) : v + sred[w];
  return v;
}

__global__ void __launch_bounds__(TR_THREADS) train_head_kernel(const TrainArgs a) {
  extern __shared__ __align__(16) float sm[];
  const int T = a.T, U = a.U, C = a.C, F = a.att ? 2 * U : U, b = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float *sFF = sm;                 // [F][C]
  float *sffb = sFF + F * C;       // [C]
  float *sscale = sffb + TR_CMAX;  // [U]
  float *sq = sscale + TR_UMAX;    // [U]   query
  float *sctx = sq + TR_UMAX;      // [U]
  float *sdctx = sctx + TR_UMAX;   // [U]
  float *sdq = sdctx + TR_UMAX;    // [U]
  float *sctxk = sdq + TR_UMAX;    // [C]   ctx . FF (ctx half)
  float *sdffb = sctxk + TR_CMAX;  // [C]
  float *sred = sdffb + TR_CMAX;   // [8]
  float *sa = sred + 8;            // [T]   attention weights
  float *sds = sa + T;             // [T]   scores, then dL/dscore
  float *sdl = sds + T;            // [T][C] dL/dlogits
  const float *W = a.w;
  for (int i = tid; i < F * C; i += TR_THREADS) sFF[i] = W[a.L.oF + i];
  for (int i = tid; i < C; i += TR_THREADS) sffb[i] = W[a.L.oFB + i];
  for (int i = tid; i < U; i += TR_THREADS) sscale[i] = a.att ? W[a.L.oS + i] : 0.f;
  const float *hf = a.Hs + (size_t)(2 * b) * T * U, *hr = a.Hs + (size_t)(2 * b + 1) * T * U;
  float *av = a.avg + (size_t)b * T * U;
  for (int i = tid; i < T * U; i += TR_THREADS) av[i] = (hf[i] + hr[i]) * 0.5f;   // not re-reversed (model.py:312)
  for (int i = tid; i < U; i += TR_THREADS) sq[i] = (hf[(size_t)(T - 1) * U + i] + hr[(size_t)(T - 1) * U + i]) * 0.5f;
  __syncthreads();   // av written by this CTA: visible to its threads after the barrier
  const float *FFa = sFF + (a.att ? U * C : 0);   // avg half of the FF kernel
  if (a.att) {
    // score[t] = sum_u scale_u tanh(q_u + avg[t,u]); softmax over t; ctx = sum_t a[t] avg[t]
    for (int t = warp; t < T; t += TR_THREADS / 32) {
      float s = 0.f;
      for (int uu = lane; uu < U; uu += 32) s = fmaf(sscale[uu], tanhf(sq[uu] + av[(size_t)t * U + uu]), s);
      s = tr_warp_sum(s);
      if (lane == 0) sds[t] = s;
    }
    __syncthreads();
    float m = -INFINITY;
    for (int t = tid; t < T; t += TR_THREADS) m = fmaxf(m, sds[t]);
    m = tr_block_reduce<true>(m, sred);
    float l = 0.f;
    for (int t = tid; t < T; t += TR_THREADS) { const float e = expf(sds[t] - m); sa[t] = e; l += e; }
    l = tr_block_reduce<false>(l, sred);
    for (int t = tid; t < T; t += TR_THREADS) sa[t] = sa[t] / l;
    __syncthreads();
    for (int uu = tid; uu < U; uu += TR_THREADS) {
      float c = 0.f;
      for (int t = 0; t < T; ++t) c = fmaf(sa[t], av[(size_t)t * U + uu], c);
      sctx[uu] = c;
    }
    __syncthreads();
    for (int c = tid; c < C; c += TR_THREADS) {
      float k = 0.f;
      for (int uu = 0; uu < U; ++uu) k = fmaf(sctx[uu], sFF[uu * C + c], k);
      sctxk[c] = k;
    }
  } else {
    for (int c = tid; c < C; c += TR_THREADS) sctxk[c] = 0.f;
  }
  __syncthreads();
  // logits, softmax, loss (p / sum p, clip to [1e-7, 1 - 1e-7], -sum y log p) and dL/dlogits of that form
  const float eps = 1e-7f;
  float lsum = 0.f;
  for (int t = tid; t < T; t += TR_THREADS) {
    float lg[TR_CMAX], mx = -INFINITY;
#pragma unroll
    for (int c = 0; c < TR_CMAX; ++c) if (c < C) lg[c] = sctxk[c];
    for (int uu = 0; uu < U; ++uu) {
      const float v = av[(size_t)t * U + uu];
#pragma unroll
      for (int c = 0; c < TR_CMAX; ++c) if (c < C) lg[c] = fmaf(v, FFa[uu * C + c], lg[c]);
    }
#pragma unroll
    for (int c = 0; c < TR_CMAX; ++c) if (c < C) { lg[c] += sffb[c]; mx = fmaxf(mx, lg[c]); }
    float sum = 0.f;
#pragma unroll
    for (int c = 0; c < TR_CMAX; ++c) if (c < C) { lg[c] = expf(lg[c] - mx); sum += lg[c]; }
    float p[TR_CMAX], S = 0.f;
#pragma unroll
    for (int c = 0; c < TR_CMAX; ++c) if (c < C) { p[c] = lg[c] / sum; S += p[c]; }
    if (a.probs) {
      float *dst = a.probs + ((size_t)b * T + t) * C;
#pragma unroll
      for (int c = 0; c < TR_CMAX; ++c) if (c < C) dst[c] = p[c];
    }
    const int y = a.ymask[a.starts[b] + t];
    float gn[TR_CMAX], gp_dot = 0.f;
#pragma unroll
    for (int c = 0; c < TR_CMAX; ++c) {
      gn[c] = 0.f;
      if (c < C && ((y >> c) & 1)) {
        const float pn = p[c] / S;
        const float pc = fminf(fmaxf(pn, eps), 1.0f - eps);
        lsum -= logf(pc);
        if (pn >= eps && pn <= 1.0f - eps) gn[c] = -a.inv_positions / pc;   // zero through clipped entries
      }
      if (c < C) gp_dot = fmaf(gn[c], p[c], gp_dot);
    }
    if (a.backward) {
      // through p / S: gp_k = gn_k / S - (gn . p) / S^2; through the softmax: p_k (gp_k - p . gp)
      float gp[TR_CMAX], pg = 0.f;
#pragma unroll
      for (int c = 0; c < TR_CMAX; ++c)
        if (c < C) { gp[c] = gn[c] / S - gp_dot / (S * S); pg = fmaf(p[c], gp[c], pg); }
#pragma unroll
      for (int c = 0; c < TR_CMAX; ++c) if (c < C) sdl[t * C + c] = p[c] * (gp[c] - pg);
    }
  }
  lsum = tr_block_reduce<false>(lsum, sred);
  if (tid == 0) a.lpart[b] = lsum;
  if (!a.backward) return;
  __syncthreads();
  float *hp = a.hpart + (size_t)b * a.L.HP;   // [F*C] FF kernel, [C] FF bias, [U] scale
  for (int c = tid; c < C; c += TR_THREADS) {
    float s = 0.f;
    for (int t = 0; t < T; ++t) s += sdl[t * C + c];
    sdffb[c] = s;
    hp[F * C + c] = s;
  }
  __syncthreads();
  const int fa = a.att ? U : 0;
  for (int i = tid; i < U * C; i += TR_THREADS) {
    const int uu = i / C, c = i % C;
    float s = 0.f;
    for (int t = 0; t < T; ++t) s = fmaf(av[(size_t)t * U + uu], sdl[t * C + c], s);
    hp[(fa + uu) * C + c] = s;
    if (a.att) hp[uu * C + c] = sctx[uu] * sdffb[c];
  }
  if (a.att) {
    for (int uu = tid; uu < U; uu += TR_THREADS) {   // dctx = sum_t dfeat[t, :U] = FF[:U] . sum_t dlogits[t]
      float s = 0.f;
      for (int c = 0; c < C; ++c) s = fmaf(sFF[uu * C + c], sdffb[c], s);
      sdctx[uu] = s;
    }
    __syncthreads();
    // da[t] = avg[t] . dctx;  dscore = a (da - sum a da)
    for (int t = warp; t < T; t += TR_THREADS / 32) {
      float s = 0.f;
      for (int uu = lane; uu < U; uu += 32) s = fmaf(av[(size_t)t * U + uu], sdctx[uu], s);
      s = tr_warp_sum(s);
      if (lane == 0) sds[t] = s;
    }
    __syncthreads();
    float dot = 0.f;
    for (int t = tid; t < T; t += TR_THREADS) dot = fmaf(sa[t], sds[t], dot);
    dot = tr_block_reduce<false>(dot, sred);
    for (int t = tid; t < T; t += TR_THREADS) sds[t] = sa[t] * (sds[t] - dot);
    __syncthreads();
    for (int uu = tid; uu < U; uu += TR_THREADS) {
      float ds = 0.f, dq = 0.f;
      for (int t = 0; t < T; ++t) {
        const float th = tanhf(sq[uu] + av[(size_t)t * U + uu]);
        ds = fmaf(sds[t], th, ds);
        dq = fmaf(sds[t] * sscale[uu], 1.0f - th * th, dq);
      }
      hp[F * C + C + uu] = ds;
      sdq[uu] = dq;
    }
    __syncthreads();
  }
  // dL/dh of both directions at step t: half of dL/davg[t] (+ half of dL/dq at T - 1)
  float *dh = a.dhin + (size_t)b * T * U;
  for (int i = tid; i < T * U; i += TR_THREADS) {
    const int t = i / U, uu = i % U;
    float g = 0.f;
    for (int c = 0; c < C; ++c) g = fmaf(sdl[t * C + c], FFa[uu * C + c], g);
    if (a.att) {
      const float th = tanhf(sq[uu] + av[i]);
      g += sa[t] * sdctx[uu] + sds[t] * sscale[uu] * (1.0f - th * th);
      if (t == T - 1) g += sdq[uu];
    }
    dh[i] = 0.5f * g;
  }
}

// ---- BPTT, reverse time, both directions --------------------------------------------------------------------
__global__ void __launch_bounds__(TR_THREADS) train_bptt_kernel(const TrainArgs a) {
  extern __shared__ __align__(16) float sm[];
  const int U = a.U, G3 = 3 * U, RS = G3 + 1, T = a.T, U4 = 4 * U;
  float *sR = sm;                 // [U][RS]
  float *sdm = sR + U * RS;       // [ROWS][3U]  dmh = [dz, dr, da_h * r]
  const int tid = threadIdx.x;
  for (int i = tid; i < U * G3; i += TR_THREADS) sR[(i / G3) * RS + i % G3] = a.w[a.L.oR + i];
  const int q = tid / TR_UMAX, u = tid % TR_UMAX;
  const int row = blockIdx.x * TR_ROWS + q;
  const bool act = u < U && row < 2 * a.n;
  const float *dhin = a.dhin + (size_t)(row >> 1) * T * U;
  __syncthreads();
  float dh_carry = 0.f;
  for (int t = T - 1; t >= 0; --t) {
    float dhz = 0.f;
    if (act) {
      const size_t it = (size_t)row * T + t;
      const float dh = dh_carry + dhin[(size_t)t * U + u];
      const float *gs = a.GS + it * 4 * U;
      const float z = gs[u], r = gs[U + u], hh = gs[2 * U + u], mhh = gs[3 * U + u];
      const float hp = t > 0 ? a.Hs[(it - 1) * U + u] : 0.f;
      const float dz = dh * (hp - hh) * z * (1.0f - z);
      const float dah = dh * (1.0f - z) * (1.0f - hh * hh);
      const float dr = dah * mhh * r * (1.0f - r);
      float *d = a.D + it * U4;
      d[u] = dz; d[U + u] = dr; d[2 * U + u] = dah; d[3 * U + u] = dah * r;
      sdm[q * G3 + u] = dz; sdm[q * G3 + U + u] = dr; sdm[q * G3 + 2 * U + u] = dah * r;
      dhz = dh * z;
    }
    __syncthreads();
    if (act) {   // dh_prev[k] = dh[k] z[k] + sum_j dmh[j] R[k, j]
      const float *dm = sdm + q * G3, *rk = sR + u * RS;
      float s = 0.f;
      for (int j = 0; j < G3; ++j) s = fmaf(dm[j], rk[j], s);
      dh_carry = dhz + s;
    }
    __syncthreads();
  }
}

// ---- weight gradients: out[KA][4U] = sum over items (row, t) of A[item]^T D[item], per chunk ----------------
// A[item] = [h_prev (U), 1, one_hot(code) * dropout scale (5)]; D[item] = [dz, dr, da_h, da_h * r]
__global__ void __launch_bounds__(TR_THREADS) train_reduce_kernel(const TrainArgs a) {
  __shared__ float sA[TR_TILE][TR_KAMAX];
  const int U = a.U, T = a.T, U4 = 4 * U, KA = U + 6;
  const int64_t N = (int64_t)2 * a.n * T;
  const int64_t per = (N + a.chunks - 1) / a.chunks;
  const int64_t lo = (int64_t)blockIdx.x * per, hi = lo + per < N ? lo + per : N;
  const int j = threadIdx.x;
  float acc[TR_KAMAX];
#pragma unroll
  for (int k = 0; k < TR_KAMAX; ++k) acc[k] = 0.f;
  for (int64_t base = lo; base < hi; base += TR_TILE) {
    const int nt = hi - base < TR_TILE ? (int)(hi - base) : TR_TILE;
    __syncthreads();
    for (int i = threadIdx.x; i < nt * KA; i += TR_THREADS) {
      const int m = i / KA, k = i % KA;
      const int64_t item = base + m;
      const int row = (int)(item / T), t = (int)(item % T);
      float v;
      if (k < U) v = t > 0 ? a.Hs[(item - 1) * U + k] : 0.f;
      else if (k == U) v = 1.f;
      else {
        float s;
        const int code = tr_code(a, row, t, &s);
        v = code == k - U - 1 ? s : 0.f;
      }
      sA[m][k] = v;
    }
    __syncthreads();
    if (j < U4) {
      for (int m = 0; m < nt; ++m) {
        const float d = a.D[(base + m) * U4 + j];
#pragma unroll
        for (int k = 0; k < TR_KAMAX; ++k)
          if (k < KA) acc[k] = fmaf(sA[m][k], d, acc[k]);
      }
    }
  }
  if (j < U4) {
    float *out = a.rpart + (size_t)blockIdx.x * KA * U4;
#pragma unroll
    for (int k = 0; k < TR_KAMAX; ++k)
      if (k < KA) out[(size_t)k * U4 + j] = acc[k];
  }
}

// every gradient in the parameter layout: chunk partials (GRU) and window partials (head) summed in order
__global__ void train_gather_grads_kernel(const TrainArgs a) {
  const TrainLayout &L = a.L;
  const int U = a.U, G3 = 3 * U, U4 = 4 * U, KA = U + 6;
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < L.n; p += gridDim.x * blockDim.x) {
    int k = -1, col = 0, hoff = -1;
    if (p < L.oR) { const int i = p - L.oK; k = U + 1 + i / G3; col = i % G3; }                 // kernel[c][j]
    else if (p < L.oB) {                                                                       // recurrent[k][j]
      const int i = p - L.oR, jj = i % G3;
      k = i / G3; col = jj < 2 * U ? jj : U4 - U + (jj - 2 * U);
    } else if (p < L.oB + 2 * G3) {                                                            // bias[0|1][j]
      const int i = p - L.oB, jj = i % G3;
      k = U; col = i < G3 ? jj : (jj < 2 * U ? jj : 3 * U + (jj - 2 * U));
    } else if (a.att && p < L.oS + U) hoff = L.F * a.C + a.C + (p - L.oS);                   // scale[u]
    else if (p < L.oFB) hoff = p - L.oF;                                                       // FF kernel
    else hoff = L.F * a.C + (p - L.oFB);                                                       // FF bias
    float s = 0.f;
    if (k >= 0)
      for (int ch = 0; ch < a.chunks; ++ch) s += a.rpart[((size_t)ch * KA + k) * U4 + col];
    else
      for (int b = 0; b < a.n; ++b) s += a.hpart[(size_t)b * L.HP + hoff];
    a.grad[p] = s;
  }
}

// one fused update of every parameter; state s1/s2: RMSprop ms / mom, Adam m / v
__global__ void train_update_kernel(float *w, const float *g, float *s1, float *s2, int n, int opt, float lr,
                                    float rho, float momentum, float eps, float b1, float b2) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float gi = g[i];
    if (opt == DGRP_OPT_RMSPROP) {
      const float ms = rho * s1[i] + (1.0f - rho) * gi * gi;
      s1[i] = ms;
      if (momentum > 0.f) {      // TF ApplyRMSProp
        const float mom = momentum * s2[i] + lr * gi / sqrtf(ms + eps);
        s2[i] = mom;
        w[i] -= mom;
      } else {
        w[i] -= lr * gi / (sqrtf(ms) + eps);
      }
    } else {                     // Adam; lr is lr_t = lr sqrt(1 - b2^t) / (1 - b1^t)
      const float m = b1 * s1[i] + (1.0f - b1) * gi;
      const float v = b2 * s2[i] + (1.0f - b2) * gi * gi;
      s1[i] = m; s2[i] = v;
      w[i] -= lr * m / (sqrtf(v) + eps);
    }
  }
}

// ---- launchers ------------------------------------------------------------------------------------------------
TrainLayout make_train_layout(int U, int C, bool att) {
  TrainLayout L;
  L.F = att ? 2 * U : U;
  L.oK = 0;
  L.oR = L.oK + 15 * U;
  L.oB = L.oR + 3 * U * U;
  L.oS = L.oB + 6 * U;
  L.oF = L.oS + (att ? U : 0);
  L.oFB = L.oF + L.F * C;
  L.n = L.oFB + C;
  L.HP = L.F * C + C + U;
  return L;
}

static size_t head_smem(int T, int U, int C, bool att) {
  const int F = att ? 2 * U : U;
  return ((size_t)F * C + 3 * TR_CMAX + 5 * TR_UMAX + 8 + 2 * (size_t)T + (size_t)T * C) * sizeof(float);
}

int train_check_shape(int T, int U, int C, bool att) {
  if (U > TR_UMAX) {
    set_error("training supports units <= %d, got %d", TR_UMAX, U);
    return DGRP_E_UNSUPPORTED;
  }
  DGRP_REQUIRE(U >= 1 && T >= 1, "vecsize and units must be positive");
  DGRP_REQUIRE(C >= MODEL_CMIN, "n_classes must be at least %d, got %d", MODEL_CMIN, C);
  if (C > MODEL_CMAX) {
    set_error("training supports n_classes <= %d, the most prediction can run, got %d", MODEL_CMAX, C);
    return DGRP_E_UNSUPPORTED;
  }
  if (head_smem(T, U, C, att) > 200 * 1024) {
    set_error("vecsize %d needs too much shared memory in the training head kernel", T);
    return DGRP_E_UNSUPPORTED;
  }
  return DGRP_OK;
}

// forward (+ head forward) of n windows; backward: also head backward, BPTT, reduction, gradients
static int train_pass(dgrp_ctx *c, dgrp_trainer *tr, int which, int64_t n, const int64_t *d_starts,
                      const uint8_t *d_keep, bool backward, float *d_probs) {
  const int T = tr->T, U = tr->U;
  const size_t rows = 2 * (size_t)n, items = rows * T;
  DGRP_CHECK(tr->Hs.reserve(items * U * sizeof(float)));
  DGRP_CHECK(tr->GS.reserve(items * 4 * U * sizeof(float)));
  DGRP_CHECK(tr->avg.reserve((size_t)n * T * U * sizeof(float)));
  DGRP_CHECK(tr->lpart.reserve((size_t)n * sizeof(float)));
  TrainArgs a = {};
  a.T = T; a.U = U; a.C = tr->C; a.att = tr->attention; a.n = (int)n;
  a.L = tr->L;
  a.w = tr->w.as<float>();
  a.codes = tr->codes[which].as<uint8_t>(); a.ymask = tr->ymask[which].as<uint8_t>();
  a.starts = d_starts; a.keep = d_keep;
  a.keep_scale = 1.0f / (1.0f - tr->dropout);
  a.inv_positions = (float)(1.0 / ((double)n * T));
  a.backward = backward ? 1 : 0;
  a.Hs = tr->Hs.as<float>(); a.GS = tr->GS.as<float>(); a.avg = tr->avg.as<float>();
  a.lpart = tr->lpart.as<float>(); a.probs = d_probs;
  a.chunks = 2 * c->sm_count;
  if (backward) {
    DGRP_CHECK(tr->D.reserve(items * 4 * U * sizeof(float)));
    DGRP_CHECK(tr->dhin.reserve((size_t)n * T * U * sizeof(float)));
    DGRP_CHECK(tr->hpart.reserve((size_t)n * tr->L.HP * sizeof(float)));
    DGRP_CHECK(tr->rpart.reserve((size_t)a.chunks * (U + 6) * 4 * U * sizeof(float)));
    a.D = tr->D.as<float>(); a.dhin = tr->dhin.as<float>(); a.hpart = tr->hpart.as<float>();
    a.rpart = tr->rpart.as<float>(); a.grad = tr->g.as<float>();
  }
  const int grid_rows = (int)((rows + TR_ROWS - 1) / TR_ROWS);
  const size_t fsm = ((size_t)U * (3 * U + 1) + 5 * 3 * U + 6 * U + TR_ROWS * U + TR_ROWS * 3 * U) * sizeof(float);
  DGRP_CUDA(cudaFuncSetAttribute(train_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsm));
  if (backward) cudaEventRecord(tr->ev[0], c->stream);
  train_forward_kernel<<<grid_rows, TR_THREADS, fsm, c->stream>>>(a);
  c->launches++;
  DGRP_CUDA(cudaGetLastError());
  if (backward) cudaEventRecord(tr->ev[1], c->stream);
  const size_t hsm = head_smem(T, U, tr->C, tr->attention);
  DGRP_CUDA(cudaFuncSetAttribute(train_head_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hsm));
  train_head_kernel<<<(int)n, TR_THREADS, hsm, c->stream>>>(a);
  c->launches++;
  DGRP_CUDA(cudaGetLastError());
  if (backward) cudaEventRecord(tr->ev[2], c->stream);
  if (!backward) return DGRP_OK;
  const size_t bsm = ((size_t)U * (3 * U + 1) + TR_ROWS * 3 * U) * sizeof(float);
  DGRP_CUDA(cudaFuncSetAttribute(train_bptt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bsm));
  train_bptt_kernel<<<grid_rows, TR_THREADS, bsm, c->stream>>>(a);
  c->launches++;
  DGRP_CUDA(cudaGetLastError());
  if (backward) cudaEventRecord(tr->ev[3], c->stream);
  train_reduce_kernel<<<a.chunks, TR_THREADS, 0, c->stream>>>(a);
  c->launches++;
  DGRP_CUDA(cudaGetLastError());
  train_gather_grads_kernel<<<(tr->L.n + 255) / 256, 256, 0, c->stream>>>(a);
  c->launches++;
  DGRP_CUDA(cudaGetLastError());
  if (backward) cudaEventRecord(tr->ev[4], c->stream);
  return DGRP_OK;
}

int train_run_step(dgrp_ctx *c, dgrp_trainer *tr, int64_t n, const int64_t *d_starts, const uint8_t *d_keep) {
  DGRP_CHECK(train_pass(c, tr, 0, n, d_starts, d_keep, true, nullptr));
  tr->steps++;
  float lr = tr->lr;
  const double b1 = 0.9, b2 = 0.999;
  if (tr->optimizer == DGRP_OPT_ADAM)
    lr = (float)(tr->lr * std::sqrt(1.0 - std::pow(b2, (double)tr->steps)) / (1.0 - std::pow(b1, (double)tr->steps)));
  const int n_par = tr->L.n;
  train_update_kernel<<<(n_par + 255) / 256, 256, 0, c->stream>>>(tr->w.as<float>(), tr->g.as<float>(),
                                                                   tr->s1.as<float>(), tr->s2.as<float>(), n_par,
                                                                   tr->optimizer, lr, tr->rho, tr->momentum,
                                                                   tr->epsilon, (float)b1, (float)b2);
  c->launches++;
  DGRP_CUDA(cudaGetLastError());
  cudaEventRecord(tr->ev[5], c->stream);
  tr->timed = true;
  return DGRP_OK;
}

int train_run_eval(dgrp_ctx *c, dgrp_trainer *tr, int which, int64_t n, const int64_t *d_starts, float *d_probs,
                   float *h_lpart) {
  for (int64_t w0 = 0; w0 < n; w0 += TR_EVAL_CHUNK) {
    const int64_t m = n - w0 < TR_EVAL_CHUNK ? n - w0 : TR_EVAL_CHUNK;
    DGRP_CHECK(train_pass(c, tr, which, m, d_starts + w0, nullptr, false,
                          d_probs ? d_probs + (size_t)w0 * tr->T * tr->C : nullptr));
    DGRP_CUDA(cudaMemcpyAsync(h_lpart + w0, tr->lpart.p, (size_t)m * sizeof(float), cudaMemcpyDeviceToHost,
                              c->stream));
  }
  return DGRP_OK;
}

}  // namespace dgrp
