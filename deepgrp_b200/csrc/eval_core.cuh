// Evaluation against a repeat annotation (K10, evaluate.cu: eval_confusion_kernel) as __host__ __device__ code, so
// that tests/host/eval_host.cpp can run the exact kernel arithmetic on the CPU next to a numpy painter (the product
// only calls the window logic from the kernel and the table builder from dgrp_evaluate_last).
//
// Both sides are sorted, disjoint interval lists per record: the predicted rows (start, end, label) and, per class,
// the annotation runs (begin, end) after the host has sorted, merged and clipped them to the record's span.  No
// per-base array exists anywhere: a thread paints 128 positions into 128-bit masks and counts with popcounts.
#pragma once
#include <stdint.h>

#include <algorithm>
#include <utility>
#include <vector>

#if defined(__CUDACC__)
#define DGRP_EVAL_HD __host__ __device__ __forceinline__
#else
#define DGRP_EVAL_HD inline
#endif
#if defined(__CUDA_ARCH__)
#define DGRP_EVAL_UNROLL _Pragma("unroll")
#else
#define DGRP_EVAL_UNROLL
#endif

namespace dgrp {
namespace eval {

constexpr int WIN = 128;       // positions per thread
constexpr int THREADS = 256;   // threads per block; a block covers WIN * THREADS positions of one record
constexpr int64_t BLOCK_SPAN = (int64_t)WIN * THREADS;

struct M128 {
  uint64_t lo, hi;
};
DGRP_EVAL_HD M128 m_or(M128 a, M128 b) { return {a.lo | b.lo, a.hi | b.hi}; }
DGRP_EVAL_HD M128 m_and(M128 a, M128 b) { return {a.lo & b.lo, a.hi & b.hi}; }
DGRP_EVAL_HD M128 m_andnot(M128 a, M128 b) { return {a.lo & ~b.lo, a.hi & ~b.hi}; }
DGRP_EVAL_HD int m_popc(M128 a) {
#if defined(__CUDA_ARCH__)
  return __popcll(a.lo) + __popcll(a.hi);
#else
  return __builtin_popcountll(a.lo) + __builtin_popcountll(a.hi);
#endif
}
// bits [u, v) of one 64-bit word, 0 <= u, v <= 64
DGRP_EVAL_HD uint64_t bits64(int u, int v) {
  if (u >= v) return 0ull;
  return (v - u == 64 ? ~0ull : ((1ull << (v - u)) - 1ull)) << u;
}
// bits [u, v) of the window, 0 <= u, v <= WIN
DGRP_EVAL_HD M128 range_mask(int u, int v) {
  return {bits64(u < 64 ? u : 64, v < 64 ? v : 64), bits64((u > 64 ? u : 64) - 64, (v > 64 ? v : 64) - 64)};
}
// position p as an offset into the window [w0, w0 + WIN), clamped to [0, WIN]
DGRP_EVAL_HD int clamp_off(int64_t p, int64_t w0) {
  return p <= w0 ? 0 : (p >= w0 + WIN ? WIN : (int)(p - w0));
}
// first index in [a, b) of sorted, disjoint intervals (iv[stride i], iv[stride i + 1]) that ends after pos
DGRP_EVAL_HD int64_t first_ending_after(const int64_t *iv, int stride, int64_t a, int64_t b, int64_t pos) {
  while (a < b) {
    const int64_t m = (a + b) >> 1;
    if (iv[stride * m + 1] <= pos) a = m + 1; else b = m;
  }
  return a;
}
// union of the intervals [a, b) of iv (sorted, disjoint; (begin, end) pairs) inside the window [w0, w0 + WIN)
DGRP_EVAL_HD M128 paint_runs(const int64_t *iv, int64_t a, int64_t b, int64_t w0) {
  M128 m = {0ull, 0ull};
  for (int64_t x = first_ending_after(iv, 2, a, b, w0); x < b; ++x) {
    const int64_t s = iv[2 * x];
    if (s >= w0 + WIN) break;
    m = m_or(m, range_mask(clamp_off(s, w0), clamp_off(iv[2 * x + 1], w0)));
  }
  return m;
}

// Confusion counts of the window [w0, w0 + WIN) cut at span_end, added to cnt[t * C + p] (t = truth, p = prediction).
// rows [r0, r1) of tri: (start, end, label) with label in [1, C); run_off[c] .. run_off[c + 1]: the runs of class c
// (c = 1 .. C-1) in runs as (begin, end).  Truth is exclusive by priority -- the lowest class that covers a position
// -- and 0 where none does; the prediction is the label of the row that covers the position, 0 where none does.
template <int C>
DGRP_EVAL_HD void window_counts(const int64_t *tri, int64_t r0, int64_t r1, const int64_t *runs,
                                const int64_t *run_off, int64_t w0, int64_t span_end, unsigned (&cnt)[C * C]) {
  if (span_end <= w0) return;
  const M128 span = range_mask(0, clamp_off(span_end, w0));
  M128 P[C], T[C];
  DGRP_EVAL_UNROLL
  for (int c = 0; c < C; ++c) P[c] = {0ull, 0ull};
  for (int64_t x = first_ending_after(tri, 3, r0, r1, w0); x < r1; ++x) {
    const int64_t s = tri[3 * x], l = tri[3 * x + 2];
    if (s >= w0 + WIN) break;
    const M128 m = m_and(range_mask(clamp_off(s, w0), clamp_off(tri[3 * x + 1], w0)), span);
    DGRP_EVAL_UNROLL
    for (int c = 1; c < C; ++c)
      if (l == c) P[c] = m_or(P[c], m);
  }
  M128 any = {0ull, 0ull};
  DGRP_EVAL_UNROLL
  for (int c = 1; c < C; ++c) any = m_or(any, P[c]);
  P[0] = m_andnot(span, any);
  any = {0ull, 0ull};
  DGRP_EVAL_UNROLL
  for (int c = 1; c < C; ++c) {
    const M128 a = m_and(paint_runs(runs, run_off[c], run_off[c + 1], w0), span);
    T[c] = m_andnot(a, any);
    any = m_or(any, a);
  }
  T[0] = m_andnot(span, any);
  DGRP_EVAL_UNROLL
  for (int t = 0; t < C; ++t) {
    DGRP_EVAL_UNROLL
    for (int p = 0; p < C; ++p) cnt[t * C + p] += (unsigned)m_popc(m_and(T[t], P[p]));
  }
}

// the record whose blocks [blk[r], blk[r + 1]) hold block b (records without positions have no block)
DGRP_EVAL_HD int64_t record_of_block(const int64_t *blk, int64_t n_rec, int64_t b) {
  int64_t lo = 0, hi = n_rec;   // first record whose first block is after b
  while (lo < hi) {
    const int64_t m = (lo + hi) >> 1;
    if (blk[m] <= b) lo = m + 1; else hi = m;
  }
  return lo - 1;
}

// Host side.  The kernel's table, one int64 array: blk[n_rec + 1] (first block of every record, then the total), span[2 n_rec]
// (startpos, length), row_off[n_rec + 1], run_off[n_rec C + 1] (record r's runs of class c are
// [run_off[r C + c], run_off[r C + c + 1]); class 0 has none) and the runs as (begin, end) pairs.
struct Table {
  std::vector<int64_t> h;
  int64_t n_rec = 0, blocks = 0, o_span = 0, o_row = 0, o_run = 0, o_runs = 0;
};

// Sorts (begin, end) pairs by begin: LSD radix sort on begin - min(begin), 11 bits per pass, as many passes as the
// key range needs (three for a chromosome of up to 8.6 G positions).  std::sort took ~3 times as long on 150 000
// random annotations, the bulk of the entry point's time.
inline void sort_by_begin(std::vector<std::pair<int64_t, int64_t>> &v,
                          std::vector<std::pair<int64_t, int64_t>> &tmp) {
  if (v.size() < 2) return;
  int64_t lo = v[0].first, hi = v[0].first;
  bool sorted = true;
  for (size_t i = 1; i < v.size(); ++i) {
    lo = std::min(lo, v[i].first);
    hi = std::max(hi, v[i].first);
    sorted = sorted && v[i - 1].first <= v[i].first;
  }
  if (sorted) return;
  const uint64_t range = (uint64_t)(hi - lo);
  tmp.resize(v.size());
  for (int shift = 0; shift < 64 && (range >> shift) != 0; shift += 11) {
    size_t cnt[2049] = {};
    for (const auto &x : v) ++cnt[(((uint64_t)(x.first - lo)) >> shift & 2047u) + 1];
    for (int d = 0; d < 2048; ++d) cnt[d + 1] += cnt[d];
    for (const auto &x : v) tmp[cnt[((uint64_t)(x.first - lo)) >> shift & 2047u]++] = x;
    v.swap(tmp);
  }
}

// ann: (begin, end, class) triples of record r at [ann_off[r], ann_off[r + 1]), in any order, overlapping or not;
// classes in [1, C) and coordinates >= 0 (checked by the caller).  Each (record, class) list is sorted by begin,
// clipped to the record's span [startpos, startpos + length) and merged where intervals overlap or touch.
inline void build_table(int C, const int64_t *ann, const int64_t *ann_off, int64_t n_rec, const int64_t *startpos,
                        const int64_t *length, const int64_t *row_off, Table &t) {
  t.n_rec = n_rec;
  t.o_span = n_rec + 1;
  t.o_row = t.o_span + 2 * n_rec;
  t.o_run = t.o_row + n_rec + 1;
  t.o_runs = t.o_run + n_rec * C + 1;
  std::vector<int64_t> &h = t.h;
  h.assign((size_t)t.o_runs, 0);
  std::vector<std::pair<int64_t, int64_t>> iv[8], tmp;   // per class (C <= 5 < 8)
  int64_t blocks = 0;
  for (int64_t r = 0; r < n_rec; ++r) {
    const int64_t s0 = startpos[r], s1 = startpos[r] + length[r];
    h[r] = blocks;
    blocks += (length[r] + BLOCK_SPAN - 1) / BLOCK_SPAN;
    h[t.o_span + 2 * r] = startpos[r];
    h[t.o_span + 2 * r + 1] = length[r];
    h[t.o_row + r] = row_off[r];
    for (int c = 1; c < C; ++c) iv[c].clear();
    for (int64_t i = ann_off[r]; i < ann_off[r + 1]; ++i) {
      const int64_t b = std::max(ann[3 * i], s0), e = std::min(ann[3 * i + 1], s1);
      if (b < e) iv[ann[3 * i + 2]].emplace_back(b, e);
    }
    for (int c = 0; c < C; ++c) {
      h[t.o_run + r * C + c] = (int64_t)(h.size() - t.o_runs) / 2;
      if (c == 0) continue;
      sort_by_begin(iv[c], tmp);
      for (size_t k = 0; k < iv[c].size();) {
        const int64_t b = iv[c][k].first;
        int64_t e = iv[c][k].second;
        for (++k; k < iv[c].size() && iv[c][k].first <= e; ++k) e = std::max(e, iv[c][k].second);
        h.push_back(b);
        h.push_back(e);
      }
    }
  }
  h[n_rec] = blocks;
  h[t.o_row + n_rec] = row_off[n_rec];
  h[t.o_run + n_rec * C] = (int64_t)(h.size() - t.o_runs) / 2;
  t.blocks = blocks;
}

}  // namespace eval
}  // namespace dgrp
