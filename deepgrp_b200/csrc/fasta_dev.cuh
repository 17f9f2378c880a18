// Block-level pieces of the GPU FASTA decode shared by its kernels (csrc/fasta.cu) and the mask kernel
// (csrc/mask.cu): the tile shape, the block scan of state functions and the per-thread byte load.
#pragma once
#include "fasta_core.cuh"

namespace dgrp {
namespace fa {

constexpr int FA_THREADS = 256;
constexpr int FA_TILE = FA_THREADS * FA_ITEMS;

// Exclusive block scan of per-thread functions; returns the function of everything before this
// thread in the tile, *total receives the whole tile's function.
__device__ __forceinline__ unsigned block_scan_fn(unsigned f, unsigned *total) {
  __shared__ unsigned s_w[FA_THREADS / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned incl = f;
  for (int off = 1; off < 32; off <<= 1) {
    const unsigned t = __shfl_up_sync(0xffffffffu, incl, off);
    if (lane >= off) incl = compose(t, incl);
  }
  if (lane == 31) s_w[warp] = incl;
  __syncthreads();
  unsigned before = FN_IDENT;
  for (int w = 0; w < warp; ++w) before = compose(before, s_w[w]);
  unsigned excl = __shfl_up_sync(0xffffffffu, incl, 1);
  if (lane == 0) excl = FN_IDENT;
  unsigned tot = FN_IDENT;
  for (int w = 0; w < FA_THREADS / 32; ++w) tot = compose(tot, s_w[w]);
  *total = tot;
  __syncthreads();
  return compose(before, excl);
}

// The FA_ITEMS bytes of one thread plus one look-ahead byte, in registers: one 16-byte load per thread
// (byte loads for the last, partial vector of the buffer or an unaligned source).  Bytes past the end
// read as 0, which is neither '\n' nor whitespace.  Every thread of the block must call load_items.
__device__ __forceinline__ void load_items(const uint8_t *__restrict__ raw, int64_t n, int64_t base, Items &it) {
  static_assert(FA_ITEMS == 16, "one uint4 per thread");
  const int64_t left = n - base;
  it.cnt = left <= 0 ? 0 : (left < FA_ITEMS ? (int)left : FA_ITEMS);
  if (it.cnt == FA_ITEMS && (reinterpret_cast<uintptr_t>(raw + base) & 15) == 0) {
    const uint4 v = __ldg(reinterpret_cast<const uint4 *>(raw + base));
    const unsigned w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < FA_ITEMS; ++k) it.b[k] = (w[k >> 2] >> (8 * (k & 3))) & 0xffu;
  } else {
#pragma unroll
    for (int k = 0; k < FA_ITEMS; ++k) it.b[k] = k < it.cnt ? (unsigned)raw[base + k] : 0u;
  }
  // look-ahead byte = first byte of the next thread; the last lane of a warp reads it from memory
  unsigned next = __shfl_down_sync(0xffffffffu, it.b[0], 1);
  if ((threadIdx.x & 31) == 31) next = left > FA_ITEMS ? (unsigned)raw[base + FA_ITEMS] : 0u;
  it.b[FA_ITEMS] = next;
}
}  // namespace fa
}  // namespace dgrp
