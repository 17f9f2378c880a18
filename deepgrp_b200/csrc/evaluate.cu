// Evaluation helpers of deepgrp.prediction that the hyper-parameter search runs on every prediction
// (deepgrp/optimization.py:66-67): filter_segments (prediction.py:242-260) and confusion_matrix
// (prediction.py:200-218).  Both are one pass over the labels: HBM-bound integer kernels.
//
// K10, evaluation against an annotation (dgrp_evaluate_last): confusion counts of predicted rows against annotation
// runs, both as interval lists (eval_core.cuh); no per-base array is built.
#include "dgrp_internal.cuh"
#include "eval_core.cuh"

namespace dgrp {

// filter_segments: a run = maximal stretch of one identical positive label; runs shorter than
// min_len are zeroed.  One thread per position; the thread at a run start walks at most min_len
// elements (a run that reaches min_len is kept, so the walk stops there) and, for a short run,
// clears it in `out`.  `in` and `out` are different buffers (a cleared run must not change what the
// neighbouring run starts see).  Bytes: 1 read + 1 written per label, plus <= min_len re-reads per run.
__global__ void filter_segments_kernel(const uint8_t *__restrict__ in, uint8_t *__restrict__ out,
                                       int64_t n, int64_t min_len) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint8_t v = in[i];
  if (v == 0 || (i > 0 && in[i - 1] == v)) return;   // not a run start
  int64_t len = 1;
  while (len < min_len && i + len < n && in[i + len] == v) ++len;
  if (len >= min_len) return;
  for (int64_t k = 0; k < len; ++k) out[i + k] = 0;
}

// confusion_matrix: cnf[t][p] += 1 over all positions, labels < 16.  Per-block counters in shared
// memory (256 bins), one 64-bit global atomic per non-empty bin and block.
__global__ void confusion_kernel(const uint8_t *__restrict__ truth, const uint8_t *__restrict__ pred,
                                 int64_t n, unsigned long long *__restrict__ cnf, int *__restrict__ bad) {
  __shared__ unsigned int bins[256];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) bins[i] = 0u;
  __syncthreads();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const unsigned t = truth[i], p = pred[i];
    if (t >= 16u || p >= 16u) { *bad = 1; continue; }
    atomicAdd(&bins[t * 16u + p], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 256; i += blockDim.x)
    if (bins[i]) atomicAdd(&cnf[i], (unsigned long long)bins[i]);
}

int launch_filter_segments(dgrp_ctx *c, const uint8_t *d_in, uint8_t *d_out, int64_t n, int64_t min_len) {
  if (n <= 0) return DGRP_OK;
  DGRP_CUDA(cudaMemcpyAsync(d_out, d_in, (size_t)n, cudaMemcpyDeviceToDevice, c->stream));
  c->launches++;
  const int threads = 256;
  filter_segments_kernel<<<(unsigned)((n + threads - 1) / threads), threads, 0, c->stream>>>(d_in, d_out, n, min_len);
  c->launches++;
  DGRP_CUDA(cudaGetLastError());
  return DGRP_OK;
}

int launch_confusion(dgrp_ctx *c, const uint8_t *d_truth, const uint8_t *d_pred, int64_t n,
                     unsigned long long *d_cnf, int *d_bad) {
  DGRP_CUDA(cudaMemsetAsync(d_cnf, 0, 256 * sizeof(unsigned long long), c->stream));
  DGRP_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int), c->stream));
  if (n <= 0) return DGRP_OK;
  const int threads = 256;
  int64_t blocks = (n + threads * 16 - 1) / (threads * 16);
  const int64_t cap = (int64_t)c->sm_count * 8;   // a multiple of the SM count, grid-stride above it
  if (blocks > cap) blocks = cap;
  confusion_kernel<<<(unsigned)blocks, threads, 0, c->stream>>>(d_truth, d_pred, n, d_cnf, d_bad);
  c->launches++;
  DGRP_CUDA(cudaGetLastError());
  return DGRP_OK;
}

// One thread per WIN positions of one record's span, blocks never straddle records (block -> record by the table's
// block prefix).  Counts stay in registers (C^2 <= 25 bins of at most WIN each), are summed per warp with one
// reduction per bin, per block in shared memory, and reach counts[r][t][p] with one 64-bit atomic per non-zero bin
// and block: integer sums, so the result does not depend on the order.
template <int C>
__global__ void __launch_bounds__(eval::THREADS)
eval_confusion_kernel(const int64_t *__restrict__ tab, int64_t n_rec, int64_t o_span, int64_t o_row, int64_t o_run,
                      int64_t o_runs, const int64_t *__restrict__ tri, unsigned long long *__restrict__ counts) {
  __shared__ unsigned s_cnt[eval::THREADS / 32][C * C];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t r = eval::record_of_block(tab, n_rec, blockIdx.x);
  const int64_t sp = tab[o_span + 2 * r], len = tab[o_span + 2 * r + 1];
  const int64_t w0 = sp + (((int64_t)blockIdx.x - tab[r]) * eval::THREADS + threadIdx.x) * eval::WIN;
  unsigned cnt[C * C];
#pragma unroll
  for (int k = 0; k < C * C; ++k) cnt[k] = 0u;
  eval::window_counts<C>(tri, tab[o_row + r], tab[o_row + r + 1], tab + o_runs, tab + o_run + r * C, w0, sp + len,
                         cnt);
#pragma unroll
  for (int k = 0; k < C * C; ++k) {
    const unsigned v = __reduce_add_sync(0xffffffffu, cnt[k]);
    if (lane == 0) s_cnt[warp][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < C * C) {
    unsigned long long v = 0ull;
#pragma unroll
    for (int w = 0; w < eval::THREADS / 32; ++w) v += s_cnt[w][threadIdx.x];
    if (v) atomicAdd(&counts[r * C * C + threadIdx.x], v);
  }
}

template <int C>
static void launch_eval(dgrp_ctx *c, const eval::Table &t, const int64_t *d_tab, const int64_t *d_tri,
                        unsigned long long *d_counts) {
  eval_confusion_kernel<C><<<(unsigned)t.blocks, eval::THREADS, 0, c->stream>>>(d_tab, t.n_rec, t.o_span, t.o_row,
                                                                               t.o_run, t.o_runs, d_tri, d_counts);
}

int run_eval_confusion(dgrp_ctx *c, int C, const eval::Table &t, const int64_t *d_tab, const int64_t *d_tri,
                       int64_t *d_counts) {
  if (t.blocks == 0) return DGRP_OK;
  unsigned long long *cnt = reinterpret_cast<unsigned long long *>(d_counts);
  switch (C) {
    case 2: launch_eval<2>(c, t, d_tab, d_tri, cnt); break;
    case 3: launch_eval<3>(c, t, d_tab, d_tri, cnt); break;
    case 4: launch_eval<4>(c, t, d_tab, d_tri, cnt); break;
    case 5: launch_eval<5>(c, t, d_tab, d_tri, cnt); break;
    default: set_error("evaluation supports %d to %d classes, got %d", MODEL_CMIN, MODEL_CMAX, C); return DGRP_E_ARG;
  }
  c->launches++;
  DGRP_CUDA(cudaGetLastError());
  return DGRP_OK;
}

}  // namespace dgrp
