// Repeat-masked FASTA text (dgrp_mask_fasta, dgrp_mask_fasta_last): the input bytes with every sequence byte that
// a predicted row covers lower-cased (soft) or replaced by 'N' (hard), everything else copied unchanged.
//
// A position is a sequence byte as the decoder (csrc/fasta.cu) classifies it: a byte of a sequence line inside the
// line's strip() span.  Sequence bytes are ranked in file order over the whole buffer, so the bytes of records with
// an empty header and the text in front of the first '>' have ranks too; no row covers them, so they stay as
// they are.  Position p of kept record r is rank base[r] + p, base[r] being the header table's sequence count in
// front of the record (hdr_seq).
//
// Two launches after the decoder's classification (tile states and the scans of per-tile sequence counts):
//   mask_paint_kernel  rows -> one bit per sequence rank (n_seq / 8 bytes written);
//   fa_mask_kernel     one 4 KiB tile of the text per CTA: classify as fa_scatter_kernel does, rank every sequence
//                      byte, look its bit up, write the 16 output bytes of a thread with one 16-byte store.
// No floating point and no atomics: every output byte and bitmap word has exactly one writer.
#include "dgrp_internal.cuh"
#include "fasta_core.cuh"
#include "fasta_dev.cuh"

namespace dgrp {

using namespace fa;

constexpr int MASK_PAINT_THREADS = 256;
constexpr int MASK_RANKS = 128;   // sequence ranks per paint thread: one 16-byte store of the bitmap

// Bit q & 31 of word q >> 5 of `bits` is set when sequence rank q is masked.  Thread t paints ranks
// [128 t, 128 t + 128): it finds the first kept record that can overlap them and, in each record that does, the
// first row that ends past them (binary searches), then walks forward.  rec[2 r] = first rank of kept record r,
// rec[2 r + 1] = its first row in tri (rec[2 n_rec + 1] = rows in total); tri = (start, end, label) per row,
// record-relative, sorted and disjoint within a record.
__global__ void mask_paint_kernel(const int64_t *__restrict__ tri, const int64_t *__restrict__ rec, int64_t n_rec,
                                  int64_t n_seq, uint4 *__restrict__ bits) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t lo = t * MASK_RANKS, hi = lo + MASK_RANKS;
  if (lo >= n_seq) return;
  unsigned w[4] = {0u, 0u, 0u, 0u};
  int64_t a = 0, b = n_rec;                       // first record that starts after lo
  while (a < b) {
    const int64_t m = (a + b) >> 1;
    if (rec[2 * m] <= lo) a = m + 1; else b = m;
  }
  for (int64_t r = a > 0 ? a - 1 : 0; r < n_rec && rec[2 * r] < hi; ++r) {
    const int64_t base = rec[2 * r], r1 = rec[2 * r + 3];
    int64_t x = rec[2 * r + 1], y = r1;           // first row of the record that ends after lo
    while (x < y) {
      const int64_t m = (x + y) >> 1;
      if (base + tri[3 * m + 1] <= lo) x = m + 1; else y = m;
    }
    for (; x < r1; ++x) {
      const int64_t s = base + tri[3 * x], e = base + tri[3 * x + 1];
      if (s >= hi) break;
      const int bs = (int)((s > lo ? s : lo) - lo), be = (int)((e < hi ? e : hi) - lo);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int u = bs > 32 * j ? bs : 32 * j, v = be < 32 * j + 32 ? be : 32 * j + 32;
        if (u < v) w[j] |= (v - u == 32 ? 0xffffffffu : ((1u << (v - u)) - 1u)) << (u - 32 * j);
      }
    }
  }
  bits[t] = make_uint4(w[0], w[1], w[2], w[3]);
}

// One tile of the text per CTA.  A thread's sequence bytes have consecutive ranks, so its at most 16 mask bits
// come from one or two bitmap words.
__global__ void fa_mask_kernel(const uint8_t *__restrict__ raw, int64_t n, const uint8_t *__restrict__ tile_state,
                               const unsigned *__restrict__ seq_off, const unsigned *__restrict__ bits, int hard,
                               uint8_t *__restrict__ out) {
  __shared__ unsigned s_ws[FA_THREADS / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t base = (int64_t)blockIdx.x * FA_TILE + (int64_t)threadIdx.x * FA_ITEMS;
  Items it;
  load_items(raw, n, base, it);
  unsigned tot;
  const unsigned excl = block_scan_fn(items_fn(it), &tot);
  unsigned s = apply_fn(excl, tile_state[blockIdx.x]), ms = 0;
#pragma unroll
  for (int k = 0; k < FA_ITEMS; ++k) {
    if (k < it.cnt) {
      const bool term = it.term(k);
      ms |= (unsigned)classify(raw, n, base + k, it.b[k], term, s).seq << k;
      s = step_state(s, it.b[k], term);
    }
  }
  const unsigned cs = __popc(ms);
  unsigned incl = cs;
  for (int off = 1; off < 32; off <<= 1) {
    const unsigned v = __shfl_up_sync(0xffffffffu, incl, off);
    if (lane >= off) incl += v;
  }
  if (lane == 31) s_ws[warp] = incl;
  __syncthreads();
  unsigned ls = incl - cs;
  for (int w = 0; w < warp; ++w) ls += s_ws[w];
  unsigned m = 0;
  if (cs) {
    const int64_t r0 = (int64_t)seq_off[blockIdx.x] + ls;    // rank of the thread's first sequence byte
    const int64_t wi = r0 >> 5;
    const unsigned sh = (unsigned)(r0 & 31);
    unsigned long long v = bits[wi];
    if (sh + cs > 32) v |= (unsigned long long)bits[wi + 1] << 32;
    m = (unsigned)(v >> sh) & ((1u << cs) - 1u);
  }
  unsigned o[FA_ITEMS];
#pragma unroll
  for (int k = 0; k < FA_ITEMS; ++k) {
    unsigned c = it.b[k];
    if ((ms >> k) & 1u) {
      if (m & 1u) c = hard ? (unsigned)'N' : ((c >= 'A' && c <= 'Z') ? (c | 0x20u) : c);
      m >>= 1;
    }
    o[k] = c;
  }
  uint8_t *dst = out + base;
  if (it.cnt == FA_ITEMS && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
    unsigned w4[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) w4[j] = o[4 * j] | (o[4 * j + 1] << 8) | (o[4 * j + 2] << 16) | (o[4 * j + 3] << 24);
    *reinterpret_cast<uint4 *>(dst) = make_uint4(w4[0], w4[1], w4[2], w4[3]);
  } else {
#pragma unroll
    for (int k = 0; k < FA_ITEMS; ++k)
      if (k < it.cnt) dst[k] = (uint8_t)o[k];
  }
}

int run_mask(dgrp_ctx *c, const uint8_t *d_raw, int64_t n, const FastaScan &f, const int64_t *d_tri,
             const int64_t *d_rec, int64_t n_rec, int mode, uint8_t *d_out) {
  if (n <= 0) return DGRP_OK;
  const int64_t nthr = (f.n_seq + MASK_RANKS - 1) / MASK_RANKS;
  DGRP_CHECK(c->mask_bits.reserve((size_t)(nthr > 0 ? nthr : 1) * 16));
  if (nthr > 0) {
    mask_paint_kernel<<<(unsigned)((nthr + MASK_PAINT_THREADS - 1) / MASK_PAINT_THREADS), MASK_PAINT_THREADS, 0,
                        c->stream>>>(d_tri, d_rec, n_rec, f.n_seq, c->mask_bits.as<uint4>());
    c->launches++;
  }
  fa_mask_kernel<<<(unsigned)f.ntiles, FA_THREADS, 0, c->stream>>>(
      d_raw, n, f.tile_state, f.seq_off, c->mask_bits.as<unsigned>(), mode == DGRP_MASK_HARD, d_out);
  c->launches++;
  DGRP_CUDA(cudaGetLastError());
  return DGRP_OK;
}

}  // namespace dgrp
