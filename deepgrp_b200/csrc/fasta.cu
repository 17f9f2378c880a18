// K1 (file form): multi-FASTA text -> per-record sequence bytes, on the GPU.
// Replaces _read_multi_fasta, deepgrp/__main__.py:20-43, byte for byte:
//   * lines end at '\n' (Python's universal newlines: "\r\n" is one terminator, a lone '\r' too);
//   * every line is stripped of leading/trailing whitespace (str.strip(): 9-13, 28-32);
//   * a stripped line that is empty raises IndexError there -> DGRP_E_FASTA here;
//   * '>' as first character starts a record, the rest of the stripped line is its header;
//     a record with an empty header is dropped, so is sequence text before the first '>';
//   * other lines are sequence text (upper-casing is folded into the base-code table).
//
// The parse is a 3-state machine over bytes (line start / sequence line / header line).  Each byte
// is a function state -> state (3 x 2 bits); composing those functions is associative, so a
// block-level scan gives the state in front of every byte of a tile and a scan over tiles gives
// the state in front of every tile.  Sequence bytes are then compacted in order, and the number
// of sequence bytes in front of every header gives the record boundaries.
#include "dgrp_internal.cuh"
#include "fasta_core.cuh"
#include "fasta_dev.cuh"

namespace dgrp {

using namespace fa;

__global__ void fa_tile_fn_kernel(const uint8_t *__restrict__ raw, int64_t n, unsigned *tile_fn) {
  const int64_t base = (int64_t)blockIdx.x * FA_TILE + (int64_t)threadIdx.x * FA_ITEMS;
  Items it;
  load_items(raw, n, base, it);
  unsigned tot;
  block_scan_fn(items_fn(it), &tot);
  if (threadIdx.x == 0) tile_fn[blockIdx.x] = tot;
}

// One block: state in front of every tile (sequential over tiles in chunks of blockDim).
__global__ void fa_tile_state_kernel(const unsigned *__restrict__ tile_fn, int64_t ntiles,
                                     uint8_t *tile_state, unsigned *final_state) {
  __shared__ unsigned s_carry;
  if (threadIdx.x == 0) s_carry = ST_START;
  __syncthreads();
  for (int64_t base = 0; base < ntiles; base += FA_THREADS) {
    const int64_t t = base + threadIdx.x;
    const unsigned f = t < ntiles ? tile_fn[t] : FN_IDENT;
    unsigned tot;
    const unsigned excl = block_scan_fn(f, &tot);
    const unsigned carry = s_carry;
    if (t < ntiles) tile_state[t] = (uint8_t)apply_fn(excl, carry);
    __syncthreads();
    if (threadIdx.x == 0) s_carry = apply_fn(tot, carry);
    __syncthreads();
  }
  if (threadIdx.x == 0) *final_state = s_carry;
}

// pass 2: per tile counts of sequence bytes and headers, and the blank-line flag
__global__ void fa_count_kernel(const uint8_t *__restrict__ raw, int64_t n,
                                const uint8_t *__restrict__ tile_state, unsigned *seq_cnt,
                                unsigned *hdr_cnt, int *blank_flag) {
  __shared__ unsigned s_c[2];
  if (threadIdx.x == 0) { s_c[0] = 0; s_c[1] = 0; }
  const int64_t base = (int64_t)blockIdx.x * FA_TILE + (int64_t)threadIdx.x * FA_ITEMS;
  Items it;
  load_items(raw, n, base, it);
  unsigned tot;
  const unsigned excl = block_scan_fn(items_fn(it), &tot);
  unsigned s = apply_fn(excl, tile_state[blockIdx.x]);
  unsigned cs = 0, ch = 0;
  bool blank = false;
#pragma unroll
  for (int k = 0; k < FA_ITEMS; ++k) {
    if (k < it.cnt) {
      const bool term = it.term(k);
      const ByteClass c = classify(raw, n, base + k, it.b[k], term, s);
      cs += c.seq; ch += c.hdr; blank |= c.blank;
      s = step_state(s, it.b[k], term);
    }
  }
  for (int off = 16; off > 0; off >>= 1) {
    cs += __shfl_xor_sync(0xffffffffu, cs, off);
    ch += __shfl_xor_sync(0xffffffffu, ch, off);
  }
  if ((threadIdx.x & 31) == 0) { atomicAdd(&s_c[0], cs); atomicAdd(&s_c[1], ch); }
  if (blank) atomicOr(blank_flag, 1);
  __syncthreads();
  if (threadIdx.x == 0) { seq_cnt[blockIdx.x] = s_c[0]; hdr_cnt[blockIdx.x] = s_c[1]; }
}

// pass 3: ordered scatter.  seq_out[rank] = byte; hdr_pos[k] = offset of the k-th '>' in raw,
// hdr_seq[k] = number of sequence bytes in front of it.  The tile's sequence bytes are contiguous in
// seq_out: they are compacted in shared memory (shifted by the destination's offset inside its 16-byte
// vector) and leave as aligned 16-byte stores.
__global__ void fa_scatter_kernel(const uint8_t *__restrict__ raw, int64_t n,
                                  const uint8_t *__restrict__ tile_state,
                                  const unsigned *__restrict__ seq_off,
                                  const unsigned *__restrict__ hdr_off, int64_t seq_base,
                                  uint8_t *__restrict__ seq_out, int64_t *__restrict__ hdr_pos,
                                  int64_t *__restrict__ hdr_seq) {
  __shared__ unsigned s_ws[FA_THREADS / 32], s_wh[FA_THREADS / 32];
  __shared__ __align__(16) uint8_t s_buf[FA_TILE + 16];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t base = (int64_t)blockIdx.x * FA_TILE + (int64_t)threadIdx.x * FA_ITEMS;
  Items it;
  load_items(raw, n, base, it);
  unsigned tot;
  const unsigned excl = block_scan_fn(items_fn(it), &tot);
  const unsigned s0 = apply_fn(excl, tile_state[blockIdx.x]);
  // thread-local classes (bit k of ms / mh: byte k is a sequence byte / a record's '>') and counts
  unsigned s = s0, ms = 0, mh = 0;
#pragma unroll
  for (int k = 0; k < FA_ITEMS; ++k) {
    if (k < it.cnt) {
      const bool term = it.term(k);
      const ByteClass c = classify(raw, n, base + k, it.b[k], term, s);
      ms |= (unsigned)c.seq << k; mh |= (unsigned)c.hdr << k;
      s = step_state(s, it.b[k], term);
    }
  }
  const unsigned cs = __popc(ms), ch = __popc(mh);
  unsigned is_ = cs, ih = ch;
  for (int off = 1; off < 32; off <<= 1) {
    const unsigned a = __shfl_up_sync(0xffffffffu, is_, off), b = __shfl_up_sync(0xffffffffu, ih, off);
    if (lane >= off) { is_ += a; ih += b; }
  }
  if (lane == 31) { s_ws[warp] = is_; s_wh[warp] = ih; }
  __syncthreads();
  unsigned ls = is_ - cs, ph = hdr_off[blockIdx.x] + ih - ch, tile_total = 0;
  for (int w = 0; w < FA_THREADS / 32; ++w) {
    if (w < warp) { ls += s_ws[w]; ph += s_wh[w]; }
    tile_total += s_ws[w];
  }
  const int64_t tile_seq0 = seq_base + seq_off[blockIdx.x];          // rank of the tile's first sequence byte
  const unsigned shift = (unsigned)(reinterpret_cast<uintptr_t>(seq_out + tile_seq0) & 15);
#pragma unroll
  for (int k = 0; k < FA_ITEMS; ++k) {
    if ((ms >> k) & 1u) s_buf[shift + ls++] = (uint8_t)it.b[k];
    if ((mh >> k) & 1u) { hdr_pos[ph] = base + k; hdr_seq[ph] = tile_seq0 + ls; ++ph; }
  }
  __syncthreads();
  uint8_t *gbase = seq_out + tile_seq0 - shift;                      // 16-byte aligned
  const unsigned end = shift + tile_total;
  for (unsigned lo = threadIdx.x * 16; lo < end; lo += FA_THREADS * 16) {
    const unsigned hi = lo + 16;
    if (lo >= shift && hi <= end) {
      *reinterpret_cast<uint4 *>(gbase + lo) = *reinterpret_cast<const uint4 *>(s_buf + lo);
    } else {
      for (unsigned j = lo < shift ? shift : lo; j < (hi < end ? hi : end); ++j) gbase[j] = s_buf[j];
    }
  }
}

__global__ void cp_scan_kernel(unsigned int *a, int64_t m, unsigned long long *total);

// Classify `n` raw bytes on the device (the part of the decode that the mask kernels share, csrc/mask.cu):
// the state in front of every tile, and per tile the exclusive scans of the sequence-byte and header counts.
// Five launches and one synchronisation; a blank line is DGRP_E_FASTA.  The arrays live in c->scan.
int run_fasta_classify(dgrp_ctx *c, const uint8_t *d_raw, int64_t n, FastaScan *f) {
  DGRP_REQUIRE(n < (int64_t)4000000000LL, "FASTA buffers above 4e9 bytes must be split by record");
  const int64_t ntiles = (n + FA_TILE - 1) / FA_TILE;
  const size_t a = ((size_t)ntiles * 4 + 255) / 256 * 256;
  DGRP_CHECK(c->scan.reserve(a * 4 + 1024));
  unsigned char *pb = c->scan.as<unsigned char>();
  unsigned *tile_fn = reinterpret_cast<unsigned *>(pb);
  unsigned *seq_cnt = reinterpret_cast<unsigned *>(pb + a);
  unsigned *hdr_cnt = reinterpret_cast<unsigned *>(pb + 2 * a);
  uint8_t *tile_state = pb + 3 * a;
  unsigned long long *totals = reinterpret_cast<unsigned long long *>(pb + 4 * a);  // [0] seq [1] hdr
  unsigned *final_state = reinterpret_cast<unsigned *>(pb + 4 * a + 64);
  int *blank = reinterpret_cast<int *>(pb + 4 * a + 128);
  DGRP_CUDA(cudaMemsetAsync(pb + 4 * a, 0, 256, c->stream));
  fa_tile_fn_kernel<<<(unsigned)ntiles, FA_THREADS, 0, c->stream>>>(d_raw, n, tile_fn);
  fa_tile_state_kernel<<<1, FA_THREADS, 0, c->stream>>>(tile_fn, ntiles, tile_state, final_state);
  fa_count_kernel<<<(unsigned)ntiles, FA_THREADS, 0, c->stream>>>(d_raw, n, tile_state, seq_cnt, hdr_cnt, blank);
  cp_scan_kernel<<<1, 1024, 0, c->stream>>>(seq_cnt, ntiles, totals);
  cp_scan_kernel<<<1, 1024, 0, c->stream>>>(hdr_cnt, ntiles, totals + 1);
  c->launches += 5;
  DGRP_CHECK(c->pin_small.reserve(256));
  unsigned long long *h = c->pin_small.as<unsigned long long>() + 12;   // bytes 96..
  DGRP_CHECK(fetch_small(c, h, pb + 4 * a, 136));
  uint8_t *h_last = reinterpret_cast<uint8_t *>(c->pin_small.as<unsigned char>() + 240);
  DGRP_CHECK(fetch_small(c, h_last, d_raw + (n - 1), 1));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  const int64_t total_seq = (int64_t)h[0], total_hdr = (int64_t)h[1];
  const unsigned fin = *reinterpret_cast<unsigned *>(reinterpret_cast<unsigned char *>(h) + 64);
  const int blank_flag = *reinterpret_cast<int *>(reinterpret_cast<unsigned char *>(h) + 128);
  // a last line without terminator that holds only whitespace is also "blank"
  const bool last_is_term = (*h_last == '\n' || *h_last == '\r');
  if (blank_flag || (!last_is_term && fin == ST_START)) {
    set_error("string index out of range (blank line in FASTA input)");
    return DGRP_E_FASTA;
  }
  f->ntiles = ntiles;
  f->tile_state = tile_state;
  f->seq_off = seq_cnt;
  f->hdr_off = hdr_cnt;
  f->n_seq = total_seq;
  f->n_hdr = total_hdr;
  return DGRP_OK;
}

// Decode `n` raw bytes on the device.  Outputs (device): compacted sequence bytes in c->io_b,
// header table in c->rows (hdr_pos | hdr_seq).  Host: *n_seq, *n_hdr, and the header table copied
// into c->pin_b (hdr_pos[n_hdr], hdr_seq[n_hdr]).  *scan (if set) receives the classification, which stays
// valid until c->scan is reserved again.
int run_fasta_decode(dgrp_ctx *c, const uint8_t *d_raw, int64_t n, int64_t *n_seq, int64_t *n_hdr, FastaScan *scan) {
  *n_seq = 0; *n_hdr = 0;
  if (n <= 0) return DGRP_OK;
  FastaScan f;
  DGRP_CHECK(run_fasta_classify(c, d_raw, n, &f));
  const int64_t total_seq = f.n_seq, total_hdr = f.n_hdr;
  DGRP_CHECK(c->io_b.reserve((size_t)total_seq + 64));
  DGRP_CHECK(c->rows.reserve((size_t)(total_hdr + 1) * 16));
  int64_t *hdr_pos = c->rows.as<int64_t>();
  int64_t *hdr_seq = hdr_pos + (total_hdr + 1);
  if (total_seq > 0 || total_hdr > 0) {
    fa_scatter_kernel<<<(unsigned)f.ntiles, FA_THREADS, 0, c->stream>>>(
        d_raw, n, f.tile_state, f.seq_off, f.hdr_off, 0, c->io_b.as<uint8_t>(), hdr_pos, hdr_seq);
    c->launches++;
  }
  DGRP_CHECK(c->pin_b.reserve((size_t)(total_hdr + 1) * 16));
  if (total_hdr > 0) {
    if (total_hdr < 256) DGRP_CHECK(fetch_small(c, c->pin_b.p, hdr_pos, (size_t)(total_hdr + 1) * 16));
    else DGRP_CUDA(cudaMemcpyAsync(c->pin_b.p, hdr_pos, (size_t)(total_hdr + 1) * 16, cudaMemcpyDeviceToHost, c->stream));
    DGRP_CUDA(cudaStreamSynchronize(c->stream));
  }
  DGRP_CUDA(cudaGetLastError());
  *n_seq = total_seq;
  *n_hdr = total_hdr;
  if (scan) *scan = f;
  return DGRP_OK;
}

}  // namespace dgrp
