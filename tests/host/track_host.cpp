// TEST INFRASTRUCTURE: runs deepgrp_b200/csrc/track_core.cuh on the CPU -- the table dgrp_track_last builds and the
// per-thread logic of its kernels in their order (bin words, line starts in bin order, line lengths,
// exclusive scan, one line at its offset) -- so the track text can be checked against a numpy restatement without
// a GPU.
// Build: g++ -O2 -std=c++17 -shared -fPIC -o tests/host/libtrack_host.so tests/host/track_host.cpp
#include <stdint.h>
#include <vector>

#include "../../deepgrp_b200/csrc/track_core.cuh"

using namespace dgrp::track;

extern "C" {

// The bedGraph text of column cls of pred (f32[rows][C], record r's vote rows from row_off[r]) for the records with
// spans [startpos[r], startpos[r] + length[r]) and prefixes text[pfx_off[r], pfx_off[r + 1]).  Returns its length;
// writes it to out when it fits cap.  n_lines_out: the number of lines.
int64_t track_host_text(int C, int cls, int64_t bin, const float *pred, const int64_t *row_off,
                        const int64_t *startpos, const int64_t *length, const uint8_t *text, const int64_t *pfx_off,
                        int64_t n_rec, uint8_t *out, int64_t cap, int64_t *n_lines_out) {
  Table t;
  build_table(n_rec, startpos, length, row_off, pfx_off, bin, t);
  const int64_t *tab = t.h.data();
  std::vector<uint32_t> words((size_t)t.bins);
  for (int64_t g = 0; g < t.bins; ++g)
    words[g] = bin_word(tab, t.n_rec, t.o_sp, t.o_len, t.o_row, t.bin, pred, C, cls, g);
  std::vector<int64_t> line_bin;
  for (int64_t g = 0; g < t.bins; ++g)
    if (line_starts(words.data(), g)) line_bin.push_back(g);
  const int64_t n_lines = (int64_t)line_bin.size();
  *n_lines_out = n_lines;
  std::vector<int64_t> off((size_t)n_lines + 1, 0);
  for (int64_t l = 0; l < n_lines; ++l) {
    const Line x = line_of(tab, t.n_rec, t.o_sp, t.o_len, t.bins, t.bin, words.data(), line_bin.data(), n_lines, l);
    off[l + 1] = off[l] + line_len((int)(tab[t.o_pfx + x.r + 1] - tab[t.o_pfx + x.r]), x);
  }
  if (off[n_lines] > cap) return off[n_lines];
  for (int64_t l = 0; l < n_lines; ++l) {
    const Line x = line_of(tab, t.n_rec, t.o_sp, t.o_len, t.bins, t.bin, words.data(), line_bin.data(), n_lines, l);
    const int64_t p0 = tab[t.o_pfx + x.r];
    line_put(out + off[l], text + p0, (int)(tab[t.o_pfx + x.r + 1] - p0), x);
  }
  return off[n_lines];
}

}  // extern "C"
