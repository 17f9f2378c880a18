// TEST INFRASTRUCTURE: runs deepgrp_b200/csrc/eval_core.cuh on the CPU -- the table dgrp_evaluate_last builds (sort,
// merge and clip of the annotation) and the window logic of eval_confusion_kernel, one "thread" at a time over the
// kernel's grid (blocks of 256 x 128 positions, block -> record by the table's prefix) -- so the evaluation kernel's
// arithmetic can be checked against a numpy painter without a GPU.
// Build: g++ -O2 -std=c++17 -shared -fPIC -o tests/host/libeval_host.so tests/host/eval_host.cpp
#include <stdint.h>
#include "../../deepgrp_b200/csrc/eval_core.cuh"

using namespace dgrp::eval;

template <int C>
static void grid(const Table &t, const int64_t *tri, int64_t *counts) {
  const int64_t *tab = t.h.data();
  for (int64_t b = 0; b < t.blocks; ++b) {
    const int64_t r = record_of_block(tab, t.n_rec, b);
    const int64_t sp = tab[t.o_span + 2 * r], len = tab[t.o_span + 2 * r + 1];
    for (int th = 0; th < THREADS; ++th) {
      unsigned cnt[C * C] = {};
      const int64_t w0 = sp + ((b - tab[r]) * THREADS + th) * WIN;
      window_counts<C>(tri, tab[t.o_row + r], tab[t.o_row + r + 1], tab + t.o_runs, tab + t.o_run + r * C, w0,
                       sp + len, cnt);
      for (int k = 0; k < C * C; ++k) counts[r * C * C + k] += cnt[k];
    }
  }
}

extern "C" {

// counts[n_rec][C][C] (zeroed here) of rows tri ((start, end, label), record r's at [row_off[r], row_off[r + 1]))
// against the annotation triples (begin, end, class) at [ann_off[r], ann_off[r + 1]), on the spans
// [startpos[r], startpos[r] + length[r]).  Returns the number of blocks of the grid, -1 for a C outside 2..5.
int64_t eval_host_counts(int C, const int64_t *tri, const int64_t *row_off, const int64_t *ann, const int64_t *ann_off,
                         const int64_t *startpos, const int64_t *length, int64_t n_rec, int64_t *counts) {
  Table t;
  build_table(C, ann, ann_off, n_rec, startpos, length, row_off, t);
  for (int64_t i = 0; i < n_rec * C * C; ++i) counts[i] = 0;
  switch (C) {
    case 2: grid<2>(t, tri, counts); break;
    case 3: grid<3>(t, tri, counts); break;
    case 4: grid<4>(t, tri, counts); break;
    case 5: grid<5>(t, tri, counts); break;
    default: return -1;
  }
  return t.blocks;
}

}  // extern "C"
