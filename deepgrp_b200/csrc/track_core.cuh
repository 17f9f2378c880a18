// Probability tracks (K11, track.cu: dgrp_track_last) as __host__ __device__ code, so that tests/host/track_host.cpp
// can run the exact kernel arithmetic on the CPU next to a numpy restatement (the product only calls the bin, merge
// and line logic from the kernels and the table builder from dgrp_track_last).
//
// A record's span [sp, sp + len) is cut into bins [k n, (k + 1) n) aligned to 0 and clipped to the span.  A bin's
// value is the mean of the class column of the max-vote (prediction.py:89-111) over its positions, computed as
//   s = float64 sum of (double)pred[p][cls] in ascending p;  mean = s / count;  q = rint(mean * 1000.0)
// (IEEE float64, round half to even) and written as q / 1000 with three decimals.  The votes are probabilities, so
// 0 <= q <= 1000.  Consecutive bins of one record with the same q form one bedGraph line "chrom\tstart\tend\tvalue\n".
#pragma once
#include <math.h>
#include <stdint.h>

#include <vector>

#include "seg_core.cuh"

#if defined(__CUDACC__)
#define DGRP_TRACK_HD __host__ __device__ __forceinline__
#else
#define DGRP_TRACK_HD inline
#endif

namespace dgrp {
namespace track {

constexpr int THREADS = 256;
constexpr int64_t BIN_MAX = 1000000;
// bin word: q, with this bit set on the first bin of a record (a line never crosses records)
constexpr uint32_t RECORD_START = 1u << 31;

// bins of the span [sp, sp + len) with bin size n
DGRP_TRACK_HD int64_t bins_of(int64_t sp, int64_t len, int64_t n) {
  return len > 0 ? (sp + len - 1) / n - sp / n + 1 : 0;
}
// positions [b, e) of bin j (0-based within its record), clipped to the span
DGRP_TRACK_HD void bin_span(int64_t sp, int64_t len, int64_t n, int64_t j, int64_t &b, int64_t &e) {
  const int64_t k = sp / n + j;
  b = k * n > sp ? k * n : sp;
  e = (k + 1) * n < sp + len ? (k + 1) * n : sp + len;
}
// q of the rows [lo, hi) (hi > lo) of column cls of pred (row-major, C columns)
DGRP_TRACK_HD uint32_t bin_q(const float *pred, int C, int cls, int64_t lo, int64_t hi) {
  double s = 0.0;
  for (int64_t p = lo; p < hi; ++p) s += (double)pred[p * C + cls];
  const double mean = s / (double)(hi - lo);
  return (uint32_t)(int32_t)rint(mean * 1000.0);
}
// a line starts at bin g: the first bin of a record, or q differs from the bin before
DGRP_TRACK_HD bool line_starts(const uint32_t *words, int64_t g) {
  return (words[g] & RECORD_START) || ((words[g] ^ words[g - 1]) & ~RECORD_START);
}

// Record table of one dgrp_track_last, uploaded as int64: bin offsets (n_rec + 1), span starts, span lengths, first
// vote row of every record, prefix text offsets (n_rec + 1).  The prefix text ("chrom\t" per record) follows it.
struct Table {
  std::vector<int64_t> h;
  int64_t n_rec = 0, bins = 0, bin = 1;
  int64_t o_sp = 0, o_len = 0, o_row = 0, o_pfx = 0;
};
// tab[0, n_rec] = bin offsets: the last record r with tab[r] <= g holds bin g (records without bins are skipped)
DGRP_TRACK_HD int64_t record_of_bin(const int64_t *tab, int64_t n_rec, int64_t g) {
  int64_t lo = 0, hi = n_rec - 1;
  while (lo < hi) {
    const int64_t mid = (lo + hi + 1) >> 1;
    if (tab[mid] <= g) lo = mid;
    else hi = mid - 1;
  }
  return lo;
}
inline void build_table(int64_t n_rec, const int64_t *sp, const int64_t *len, const int64_t *row_off,
                        const int64_t *pfx_off, int64_t bin, Table &t) {
  t.n_rec = n_rec;
  t.bin = bin;
  t.o_sp = n_rec + 1;
  t.o_len = t.o_sp + n_rec;
  t.o_row = t.o_len + n_rec;
  t.o_pfx = t.o_row + n_rec;
  t.h.assign((size_t)(t.o_pfx + n_rec + 1), 0);
  int64_t b = 0;
  for (int64_t r = 0; r < n_rec; ++r) {
    t.h[r] = b;
    b += bins_of(sp[r], len[r], bin);
    t.h[t.o_sp + r] = sp[r];
    t.h[t.o_len + r] = len[r];
    t.h[t.o_row + r] = row_off[r];
  }
  t.h[n_rec] = b;
  for (int64_t r = 0; r <= n_rec; ++r) t.h[t.o_pfx + r] = pfx_off[r];
  t.bins = b;
}

// The bin word of bin g: q of the bin, RECORD_START on a record's first bin.  pred holds every record's vote rows.
DGRP_TRACK_HD uint32_t bin_word(const int64_t *tab, int64_t n_rec, int64_t o_sp, int64_t o_len, int64_t o_row,
                                int64_t bin, const float *pred, int C, int cls, int64_t g) {
  const int64_t r = record_of_bin(tab, n_rec, g);
  const int64_t sp = tab[o_sp + r], j = g - tab[r];
  int64_t b, e;
  bin_span(sp, tab[o_len + r], bin, j, b, e);
  const float *rows = pred + tab[o_row + r] * (int64_t)C;
  return bin_q(rows, C, cls, b - sp, e - sp) | (j == 0 ? RECORD_START : 0u);
}

struct Line {
  int64_t r, start, end;
  uint32_t q;
};
// line l: bins [line_bin[l], line_bin[l + 1]) (the last one up to the last bin); never more than one record
DGRP_TRACK_HD Line line_of(const int64_t *tab, int64_t n_rec, int64_t o_sp, int64_t o_len, int64_t bins, int64_t bin,
                           const uint32_t *words, const int64_t *line_bin, int64_t n_lines, int64_t l) {
  const int64_t g0 = line_bin[l], g1 = (l + 1 < n_lines ? line_bin[l + 1] : bins) - 1;
  Line out;
  out.r = record_of_bin(tab, n_rec, g0);
  const int64_t sp = tab[o_sp + out.r], len = tab[o_len + out.r];
  int64_t b, e;
  bin_span(sp, len, bin, g0 - tab[out.r], out.start, e);
  bin_span(sp, len, bin, g1 - tab[out.r], b, out.end);
  out.q = words[g0] & ~RECORD_START;
  return out;
}
// "chrom\t" + start + '\t' + end + '\t' + q / 1000 + '.' + three digits of q % 1000 + '\n'
DGRP_TRACK_HD unsigned line_len(int prefix_len, const Line &x) {
  return (unsigned)(prefix_len + seg::fmt_len(x.start) + seg::fmt_len(x.end) + seg::fmt_len(x.q / 1000u) + 7);
}
DGRP_TRACK_HD uint8_t *line_put(uint8_t *p, const uint8_t *prefix, int prefix_len, const Line &x) {
  for (int k = 0; k < prefix_len; ++k) p[k] = prefix[k];
  p += prefix_len;
  p = seg::fmt_put(p, x.start);  *p++ = '\t';
  p = seg::fmt_put(p, x.end);    *p++ = '\t';
  p = seg::fmt_put(p, x.q / 1000u);
  const unsigned f = x.q % 1000u;
  p[0] = '.';
  p[1] = (uint8_t)('0' + f / 100u);
  p[2] = (uint8_t)('0' + f / 10u % 10u);
  p[3] = (uint8_t)('0' + f % 10u);
  p[4] = '\n';
  return p + 5;
}

}  // namespace track
}  // namespace dgrp
