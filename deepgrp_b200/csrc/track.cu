// K11: probability tracks (dgrp_track_last).  The max-vote rows of the last dgrp_predict_fasta[_tsv] (kept on the
// device with the "keep_votes" option) become the bedGraph text of one class, in the style of the TSV writer:
//   bins    one thread per bin: the float64 mean of its votes, rounded to thousandths (track_core.cuh)
//   lines   flags where the value changes or a record starts -> per-tile counts -> 64-bit exclusive scan -> ordered
//           scatter of the first bin of every line
//   text    line lengths -> 64-bit exclusive scan -> one thread per line writes at its offset
// Every step is integer work or a sequential sum inside one thread: no atomics, the text is deterministic.
#include "dgrp_internal.cuh"
#include "track_core.cuh"

namespace dgrp {

__global__ void tsv_scan_kernel(unsigned long long *a, int64_t m, unsigned long long *total);   // tsv.cu

struct TrackArgs {
  const int64_t *tab;
  int64_t n_rec, o_sp, o_len, bins, bin;
  const uint8_t *text;   // prefix text ("chrom\t" per record), offsets at tab[o_pfx ..]
  int64_t o_pfx;
};

__global__ void __launch_bounds__(track::THREADS)
track_bin_kernel(TrackArgs a, int64_t o_row, const float *__restrict__ pred, int C, int cls, uint32_t *words) {
  const int64_t g = (int64_t)blockIdx.x * track::THREADS + threadIdx.x;
  if (g >= a.bins) return;
  words[g] = track::bin_word(a.tab, a.n_rec, a.o_sp, a.o_len, o_row, a.bin, pred, C, cls, g);
}

// One tile of THREADS bins per block: the line-start flags of its bins as warp ballots, their count per warp in
// s_w; returns the flag of this thread's bin and the lanes of its warp below it that are flagged
__device__ __forceinline__ bool track_flags(const uint32_t *words, int64_t bins, unsigned *s_w, unsigned &below) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t g = (int64_t)blockIdx.x * track::THREADS + threadIdx.x;
  const bool f = g < bins && track::line_starts(words, g);
  const unsigned m = __ballot_sync(0xffffffffu, f);
  if (lane == 0) s_w[warp] = __popc(m);
  below = __popc(m & ((1u << lane) - 1u));
  __syncthreads();
  return f;
}

__global__ void __launch_bounds__(track::THREADS)
track_count_kernel(const uint32_t *__restrict__ words, int64_t bins, unsigned long long *tile_cnt) {
  __shared__ unsigned s_w[track::THREADS / 32];
  unsigned below;
  track_flags(words, bins, s_w, below);
  if (threadIdx.x == 0) {
    unsigned long long t = 0;
    for (int w = 0; w < track::THREADS / 32; ++w) t += s_w[w];
    tile_cnt[blockIdx.x] = t;
  }
}

// line_bin[line] = first bin of the line, at the tile's 64-bit offset + the lines before it in the tile
__global__ void __launch_bounds__(track::THREADS)
track_scatter_kernel(const uint32_t *__restrict__ words, int64_t bins, const unsigned long long *__restrict__ tile_off,
                     int64_t *__restrict__ line_bin) {
  __shared__ unsigned s_w[track::THREADS / 32];
  unsigned below;
  if (!track_flags(words, bins, s_w, below)) return;
  for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) below += s_w[w];
  line_bin[tile_off[blockIdx.x] + below] = (int64_t)blockIdx.x * track::THREADS + threadIdx.x;
}

__device__ __forceinline__ unsigned track_line(const TrackArgs &a, const uint32_t *words, const int64_t *line_bin,
                                               int64_t n_lines, int64_t l, track::Line &x) {
  x = track::line_of(a.tab, a.n_rec, a.o_sp, a.o_len, a.bins, a.bin, words, line_bin, n_lines, l);
  return track::line_len((int)(a.tab[a.o_pfx + x.r + 1] - a.tab[a.o_pfx + x.r]), x);
}

__global__ void __launch_bounds__(track::THREADS)
track_len_kernel(TrackArgs a, const uint32_t *__restrict__ words, const int64_t *__restrict__ line_bin,
                 int64_t n_lines, unsigned long long *tile_sum) {
  __shared__ unsigned long long s_sum;
  if (threadIdx.x == 0) s_sum = 0;
  __syncthreads();
  const int64_t l = (int64_t)blockIdx.x * track::THREADS + threadIdx.x;
  track::Line x;
  unsigned long long v = l < n_lines ? track_line(a, words, line_bin, n_lines, l, x) : 0;
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  if ((threadIdx.x & 31) == 0) atomicAdd(&s_sum, v);   // integer: the order does not matter
  __syncthreads();
  if (threadIdx.x == 0) tile_sum[blockIdx.x] = s_sum;
}

// one thread per line at tile_off[block] + the block's exclusive scan of the line lengths
__global__ void __launch_bounds__(track::THREADS)
track_write_kernel(TrackArgs a, const uint32_t *__restrict__ words, const int64_t *__restrict__ line_bin,
                   int64_t n_lines, const unsigned long long *__restrict__ tile_off, uint8_t *__restrict__ out) {
  __shared__ unsigned s_w[track::THREADS / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t l = (int64_t)blockIdx.x * track::THREADS + threadIdx.x;
  track::Line x;
  const unsigned len = l < n_lines ? track_line(a, words, line_bin, n_lines, l, x) : 0;
  unsigned incl = len;
  for (int off = 1; off < 32; off <<= 1) {
    const unsigned t = __shfl_up_sync(0xffffffffu, incl, off);
    if (lane >= off) incl += t;
  }
  if (lane == 31) s_w[warp] = incl;
  __syncthreads();
  if (l >= n_lines) return;
  unsigned before = incl - len;
  for (int w = 0; w < warp; ++w) before += s_w[w];
  const int64_t p0 = a.tab[a.o_pfx + x.r];
  track::line_put(out + tile_off[blockIdx.x] + before, a.text + p0, (int)(a.tab[a.o_pfx + x.r + 1] - p0), x);
}

int run_track(dgrp_ctx *c, const track::Table &t, const int64_t *d_tab, const uint8_t *d_text, const float *d_pred,
              int C, int cls, DevBuf &work, DevBuf &text, int64_t *n_bytes) {
  *n_bytes = 0;
  if (t.bins == 0) return DGRP_OK;
  const TrackArgs a{d_tab, t.n_rec, t.o_sp, t.o_len, t.bins, t.bin, d_text, t.o_pfx};
  // work: bin words (u32) | first bin of every line (i64); c->scan: tile counts, tile sums, totals
  const size_t words_bytes = ((size_t)t.bins * 4 + 15) / 16 * 16;
  DGRP_CHECK(work.reserve(words_bytes + (size_t)t.bins * 8));
  uint32_t *words = work.as<uint32_t>();
  int64_t *line_bin = reinterpret_cast<int64_t *>(work.as<uint8_t>() + words_bytes);
  // c->scan: 64-bit per-tile line counts of the bins, per-tile byte counts of the lines (lines <= bins), totals
  const int64_t bin_tiles = (t.bins + track::THREADS - 1) / track::THREADS;
  DGRP_CHECK(c->scan.reserve((size_t)bin_tiles * 16 + 64));
  unsigned long long *cnt = c->scan.as<unsigned long long>();
  unsigned long long *tile = cnt + bin_tiles;
  unsigned long long *total = tile + bin_tiles;   // [0] lines, [1] bytes
  DGRP_CHECK(c->pin_small.reserve(256));
  unsigned long long *h = c->pin_small.as<unsigned long long>();

  track_bin_kernel<<<(unsigned)bin_tiles, track::THREADS, 0, c->stream>>>(a, t.o_row, d_pred, C, cls, words);
  track_count_kernel<<<(unsigned)bin_tiles, track::THREADS, 0, c->stream>>>(words, t.bins, cnt);
  tsv_scan_kernel<<<1, 1024, 0, c->stream>>>(cnt, bin_tiles, total);
  track_scatter_kernel<<<(unsigned)bin_tiles, track::THREADS, 0, c->stream>>>(words, t.bins, cnt, line_bin);
  c->launches += 4;
  DGRP_CHECK(fetch_small(c, h, total, 8));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  const int64_t n_lines = (int64_t)h[0];
  const int64_t tiles = (n_lines + track::THREADS - 1) / track::THREADS;
  track_len_kernel<<<(unsigned)tiles, track::THREADS, 0, c->stream>>>(a, words, line_bin, n_lines, tile);
  tsv_scan_kernel<<<1, 1024, 0, c->stream>>>(tile, tiles, total + 1);
  c->launches += 2;
  DGRP_CHECK(fetch_small(c, h + 1, total + 1, 8));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  *n_bytes = (int64_t)h[1];
  DGRP_CHECK(text.reserve((size_t)*n_bytes + 16));
  track_write_kernel<<<(unsigned)tiles, track::THREADS, 0, c->stream>>>(a, words, line_bin, n_lines, tile,
                                                                       text.as<uint8_t>());
  c->launches++;
  DGRP_CUDA(cudaGetLastError());
  return DGRP_OK;
}

}  // namespace dgrp
