// C ABI of libdeepgrp_b200.so (include/deepgrp_b200.h): contexts, weight handles and the host-side
// sequencing of the kernels.  No CPU fallback: every entry point that computes needs a context, and a
// context needs an sm_100 GPU.
#include <math.h>
#include <stdarg.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <thread>

#include <cuda_fp16.h>
#include <cmath>

#include "dgrp_internal.cuh"

namespace dgrp {

static thread_local char g_err[1024] = "";

void set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof g_err, fmt, ap);
  va_end(ap);
}

int DevBuf::reserve(size_t bytes) {
  ++reserves;
  if (bytes <= cap && p) return DGRP_OK;
  if (bytes < 256) bytes = 256;
  if (p) { cudaFree(p); p = nullptr; cap = 0; }
  const size_t want = (bytes + (1u << 20) - 1) & ~((size_t)(1u << 20) - 1);
  DGRP_CUDA(cudaMalloc(&p, want));
  cap = want;
  return DGRP_OK;
}
void DevBuf::release() {
  if (p) cudaFree(p);
  p = nullptr; cap = 0;
}
int PinBuf::reserve(size_t bytes) {
  if (bytes <= cap && p) return DGRP_OK;
  if (bytes < 256) bytes = 256;
  if (p) { cudaFreeHost(p); p = nullptr; cap = 0; }
  DGRP_CUDA(cudaMallocHost(&p, bytes));
  cap = bytes;
  return DGRP_OK;
}
void PinBuf::release() {
  if (p) cudaFreeHost(p);
  p = nullptr; cap = 0;
}

__global__ void fetch_small_kernel(unsigned char *__restrict__ dst, const unsigned char *__restrict__ src, int n) {
  for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
}
int fetch_small(dgrp_ctx *c, void *pinned_dst, const void *d_src, size_t bytes) {
  if (bytes == 0) return DGRP_OK;
  void *mapped = nullptr;
  DGRP_CUDA(cudaHostGetDevicePointer(&mapped, pinned_dst, 0));
  fetch_small_kernel<<<1, 128, 0, c->stream>>>(static_cast<unsigned char *>(mapped),
                                               static_cast<const unsigned char *>(d_src), (int)bytes);
  c->launches++;
  DGRP_CUDA(cudaGetLastError());
  return DGRP_OK;
}

// sum of n scores (double): the direction the running sum of the MSS scan drifts in
__global__ void score_drift_kernel(const float *__restrict__ sc, int64_t n, double *out) {
  double acc = 0.0;
  const int64_t gs = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gs) acc += (double)sc[i];
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
  if ((threadIdx.x & 31) == 0) atomicAdd(out, acc);
}

// s0 = ln(0.99/0.01) and the two thresholds of pymss.pyx:46-53
static void mss_thresholds(int min_mss_len, int xdrop_len, double *min_sc, double *xdrop) {
  const double s0 = log(0.99 / (1.0 - 0.99));
  *xdrop = xdrop_len > 0 ? s0 * xdrop_len * 10.0 : -1.0;
  *min_sc = s0 * min_mss_len;
}

static void stamp(dgrp_ctx *c, int i) { cudaEventRecord(c->ev[i], c->stream); }

// codes (device, trimmed record of length L) -> predictions f32[L, C] in c->pred, or -- want_scores, when the vote
// and the score transform could be fused (c->fused_last) -- label u8[L] in c->labels and score f32[L] in
// c->scores32 with the predictions never materialised
static int core_predict(dgrp_ctx *c, dgrp_model *m, const uint8_t *d_codes, int64_t L, int step,
                        int batch_size, int compat, bool want_scores = false) {
  DGRP_REQUIRE(step > 0, "step_size must be positive");
  c->fused_last = 0;
  DGRP_CHECK(c->pred.reserve((size_t)(L > 0 ? L : 1) * m->C * sizeof(float)));
  const Placement pl = make_placement(L, m->T, step, batch_size, compat);
  c->timings.windows = pl.n_windows;
  c->timings.bases = L;
  if (want_scores && L > 0) {
    DGRP_CHECK(c->labels.reserve((size_t)L));
    DGRP_CHECK(c->scores32.reserve((size_t)L * 4));
    bool fused = false;
    DGRP_CHECK(run_forward_vote(c, m, d_codes, 0, 0, pl.n_windows, pl, c->pred.as<float>(), 0, L,
                                c->labels.as<uint8_t>(), c->scores32.as<float>(), &fused));
    c->fused_last = fused ? 1 : 0;
    return DGRP_OK;
  }
  if (L > 0) DGRP_CUDA(cudaMemsetAsync(c->pred.p, 0, (size_t)L * m->C * sizeof(float), c->stream));
  return run_forward_vote(c, m, d_codes, 0, 0, pl.n_windows, pl, c->pred.as<float>(), 0, L);
}

// core_labels on what core_predict left: fused label + score, or the predictions
static int core_labels(dgrp_ctx *c, const float *d_pred, const uint8_t *d_lab_in, const float *d_score_in, int64_t L,
                       int C, int use_mss, int min_mss_len, int xdrop_len);
static int core_labels_after_predict(dgrp_ctx *c, int64_t L, int C, int use_mss, int min_mss_len, int xdrop_len) {
  if (c->fused_last)
    return core_labels(c, nullptr, c->labels.as<uint8_t>(), c->scores32.as<float>(), L, C, use_mss, min_mss_len,
                       xdrop_len);
  return core_labels(c, c->pred.as<float>(), nullptr, nullptr, L, C, use_mss, min_mss_len, xdrop_len);
}

// predictions (device f32[L, C]) or ready (label, score) -> final labels in c->labels2
static int core_labels(dgrp_ctx *c, const float *d_pred, const uint8_t *d_lab_in,
                       const float *d_score_in, int64_t L, int C, int use_mss, int min_mss_len,
                       int xdrop_len) {
  DGRP_REQUIRE(L < 2147483647LL, "record longer than 2^31-1 bases (int indices in mss.h:16)");
  DGRP_CHECK(c->labels2.reserve((size_t)(L > 0 ? L : 1)));
  if (L <= 0) return DGRP_OK;
  if (use_mss) {
    const uint8_t *lab = d_lab_in;
    const float *sc = d_score_in;
    if (d_pred) {
      DGRP_CHECK(c->labels.reserve((size_t)L));
      DGRP_CHECK(c->scores32.reserve((size_t)L * 4));
      DGRP_CHECK(launch_score(c, d_pred, L, C, c->labels.as<uint8_t>(), c->scores32.as<float>(),
                              nullptr, nullptr));
      lab = c->labels.as<uint8_t>();
      sc = c->scores32.as<float>();
    }
    stamp(c, 3);
    double min_sc, xdrop;
    mss_thresholds(min_mss_len, xdrop_len, &min_sc, &xdrop);
    dgrp_seg_t *d_segs = nullptr;
    int n_seg = 0;
    DGRP_CHECK(run_mss_segments(c, nullptr, sc, (int)L, min_sc, xdrop, &d_segs, &n_seg));
    DGRP_CHECK(run_gap_fill(c, d_segs, n_seg, lab, nullptr, (int)L, C, c->labels2.as<uint8_t>()));
  } else {
    // softmax (prediction.py:62-65) then argmax (__main__.py:83)
    if (d_pred) {
      DGRP_CHECK(c->io_a.reserve((size_t)L * C * 4));
      DGRP_CHECK(launch_softmax_global(c, d_pred, L, C, c->io_a.as<float>()));
      DGRP_CHECK(launch_score(c, c->io_a.as<float>(), L, C, c->labels2.as<uint8_t>(), nullptr,
                              nullptr, nullptr));
    } else {
      DGRP_CUDA(cudaMemcpyAsync(c->labels2.p, d_lab_in, (size_t)L, cudaMemcpyDeviceToDevice, c->stream));
    }
    stamp(c, 3);
  }
  return DGRP_OK;
}

// final labels (c->labels2) -> rows on the host (label > 0 only, __main__.py:288-290)
static int core_rows(dgrp_ctx *c, int64_t L, int64_t startpos, int32_t record, bool to_host,
                     dgrp_row_t *rows, int64_t cap, int64_t *n_rows) {
  int64_t *d_tri = nullptr;
  int64_t cnt = 0;
  DGRP_CHECK(run_segments(c, c->labels2.as<uint8_t>(), nullptr, L, startpos, false, &d_tri, &cnt));
  *n_rows = cnt;
  if (!to_host || cnt == 0) return DGRP_OK;
  if (cnt > cap || !rows) {
    set_error("row buffer too small: %lld rows needed, capacity %lld", (long long)cnt, (long long)cap);
    return DGRP_E_CAPACITY;
  }
  DGRP_CHECK(c->pin_a.reserve((size_t)cnt * 24));
  DGRP_CUDA(cudaMemcpyAsync(c->pin_a.p, d_tri, (size_t)cnt * 24, cudaMemcpyDeviceToHost, c->stream));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  const int64_t *t = c->pin_a.as<int64_t>();
  for (int64_t i = 0; i < cnt; ++i) {
    rows[i].start = t[3 * i]; rows[i].end = t[3 * i + 1];
    rows[i].label = (int32_t)t[3 * i + 2]; rows[i].record = record;
  }
  return DGRP_OK;
}

static void finish_timings(dgrp_ctx *c, int64_t launches0) {
  cudaStreamSynchronize(c->stream);
  dgrp_timings_t &t = c->timings;
  cudaEventElapsedTime(&t.encode_ms, c->ev[0], c->ev[1]);
  cudaEventElapsedTime(&t.forward_ms, c->ev[1], c->ev[2]);
  cudaEventElapsedTime(&t.score_ms, c->ev[2], c->ev[3]);
  cudaEventElapsedTime(&t.mss_ms, c->ev[3], c->ev[4]);
  cudaEventElapsedTime(&t.segments_ms, c->ev[4], c->ev[5]);
  cudaEventElapsedTime(&t.total_ms, c->ev[0], c->ev[5]);
  t.attend_ms = 0.f;
  t.kernel_launches = c->launches - launches0;
}

// raw record bytes on the device -> (startpos, length) and codes in c->codes
static int core_encode(dgrp_ctx *c, const uint8_t *d_seq, int64_t n, int fold_case,
                       int64_t *startpos, int64_t *length) {
  DGRP_CHECK(c->small.reserve(256));
  DGRP_CHECK(c->pin_small.reserve(256));
  int64_t *d_fl = c->small.as<int64_t>() + 16;
  DGRP_CHECK(launch_trim(c, d_seq, n, fold_case, d_fl));
  int64_t *h = c->pin_small.as<int64_t>() + 8;
  DGRP_CHECK(fetch_small(c, h, d_fl, 16));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  *startpos = h[0];           // first non-'N' (n when there is none)
  *length = h[1] - h[0];      // (last non-'N' + 1) - startpos: -n for an all-'N' record
  if (*length > 0) {
    DGRP_CHECK(c->codes.reserve((size_t)*length + 16));
    DGRP_CHECK(launch_codes(c, d_seq, *startpos, *length, c->codes.as<uint8_t>()));
  }
  return DGRP_OK;
}

}  // namespace dgrp

using namespace dgrp;

extern "C" {

int dgrp_version(void) { return 100; }
const char *dgrp_last_error(void) { return g_err; }

int dgrp_device_count(int *count) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) {
    set_error("cudaGetDeviceCount: %s", cudaGetErrorString(e));
    *count = 0;
    return DGRP_E_NOGPU;
  }
  *count = n;
  return DGRP_OK;
}

int dgrp_ctx_create(int device, dgrp_ctx **out) {
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
    set_error("no CUDA device is visible; deepgrp_b200 has no CPU fallback");
    return DGRP_E_NOGPU;
  }
  DGRP_REQUIRE(device >= 0 && device < n, "device %d out of range (%d visible)", device, n);
  cudaDeviceProp prop;
  DGRP_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) {
    set_error("device %d (%s, sm_%d%d) is not a Blackwell sm_100 GPU", device, prop.name, prop.major,
              prop.minor);
    return DGRP_E_NOGPU;
  }
  DGRP_CUDA(cudaSetDevice(device));
  dgrp_ctx *c = new dgrp_ctx();
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) {
    set_error("cudaStreamCreate failed");
    delete c;
    return DGRP_E_CUDA;
  }
  for (auto &e : c->ev) cudaEventCreate(&e);
  for (int i = 0; i < 6; ++i) cudaEventRecord(c->ev[i], c->stream);
  *out = c;
  return DGRP_OK;
}

int dgrp_ctx_destroy(dgrp_ctx *c) {
  if (!c) return DGRP_OK;
  Use use(c->device);
  cudaStreamSynchronize(c->stream);
  DevBuf *bufs[] = {&c->raw, &c->codes, &c->onehot, &c->avg, &c->pred, &c->labels, &c->labels2,
                    &c->scores32, &c->scores64, &c->classes64, &c->io_a, &c->io_b, &c->io_c, &c->winprobs,
                    &c->small, &c->segs, &c->rows, &c->mss_a, &c->mss_b, &c->mss_c, &c->mss_d,
                    &c->mss_e, &c->scan, &c->gapfill};
  for (auto b : bufs) b->release();
  c->pin_small.release(); c->pin_a.release(); c->pin_b.release(); c->tsv_host.release();
  c->tsv_dev.release(); c->tsv_prefix.release();
  for (int i = 0; i < 2; ++i) { c->st_raw[i].release(); c->st_text[i].release(); c->st_stage[i].release(); }
  for (int i = 0; i < 4; ++i) c->st_slot[i].release();
  for (auto &e : c->ev) cudaEventDestroy(e);
  cudaStreamDestroy(c->stream);
  delete c;
  return DGRP_OK;
}

int dgrp_ctx_synchronize(dgrp_ctx *c) {
  Use use(c->device);
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  return DGRP_OK;
}
void *dgrp_ctx_stream(dgrp_ctx *c) { return (void *)c->stream; }
int dgrp_ctx_timings(dgrp_ctx *c, dgrp_timings_t *out) { *out = c->timings; return DGRP_OK; }
int64_t dgrp_ctx_launch_count(dgrp_ctx *c) { return c->launches; }

int dgrp_ctx_set_int(dgrp_ctx *c, const char *key, int64_t value) {
  if (!strcmp(key, "mss_chunk")) c->mss_chunk = (int)value;
  else if (!strcmp(key, "mss_max_rounds")) c->mss_max_rounds = (int)value;
  else if (!strcmp(key, "forward_tc")) c->forward_tc = (int)value;
  else if (!strcmp(key, "forward_sum16")) c->forward_sum16 = (int)value;
  else if (!strcmp(key, "forward_fp16x2")) c->forward_fp16x2 = (int)value;
  else if (!strcmp(key, "forward_gather")) c->forward_gather = (int)value;
  else if (!strcmp(key, "forward_fuse_score")) c->forward_fuse_score = (int)value;
  else if (!strcmp(key, "forward_smem_vote")) c->forward_smem_vote = (int)value;
  else if (!strcmp(key, "forward_wide")) c->forward_wide = (int)value;
  else if (!strcmp(key, "forward_overlap")) c->forward_overlap = (int)value;
  else if (!strcmp(key, "forward_ub")) c->forward_ub = (int)value;
  else if (!strcmp(key, "stream_slot_mb")) c->stream_slot_mb = (int)value;
  else if (!strcmp(key, "stream_early_rows")) c->stream_early_rows = (int)value;
  else if (!strcmp(key, "stream_early_slabs")) c->stream_early_slabs = (int)value;
  else if (!strcmp(key, "stream_early_unit")) c->stream_early_unit = (int)value;
  else if (!strcmp(key, "stream_early_ratio")) c->stream_early_ratio = (int)value;
  else if (!strcmp(key, "forward_slab_mb")) c->forward_slab_bytes = (int64_t)value << 20;
  else if (!strcmp(key, "shard_rank")) c->shard_rank = (int)value;
  else if (!strcmp(key, "shard_world")) c->shard_world = (int)value;
  else { set_error("unknown option %s", key); return DGRP_E_ARG; }
  return DGRP_OK;
}
int dgrp_ctx_get_int(dgrp_ctx *c, const char *key, int64_t *value) {
  if (!strcmp(key, "mss_chunk")) *value = c->mss_chunk;
  else if (!strcmp(key, "mss_max_rounds")) *value = c->mss_max_rounds;
  else if (!strcmp(key, "mss_rounds")) *value = c->mss_rounds;
  else if (!strcmp(key, "forward_tc")) *value = c->forward_tc;
  else if (!strcmp(key, "forward_sum16")) *value = c->forward_sum16;
  else if (!strcmp(key, "forward_fp16x2")) *value = c->forward_fp16x2;
  else if (!strcmp(key, "forward_gather")) *value = c->forward_gather;
  else if (!strcmp(key, "forward_fuse_score")) *value = c->forward_fuse_score;
  else if (!strcmp(key, "forward_smem_vote")) *value = c->forward_smem_vote;
  else if (!strcmp(key, "fused_last")) *value = c->fused_last;
  else if (!strcmp(key, "forward_wide")) *value = c->forward_wide;
  else if (!strcmp(key, "forward_overlap")) *value = c->forward_overlap;
  else if (!strcmp(key, "forward_ub")) *value = c->forward_ub;
  else if (!strcmp(key, "stream_slot_mb")) *value = c->stream_slot_mb;
  else if (!strcmp(key, "stream_early_rows")) *value = c->stream_early_rows;
  else if (!strcmp(key, "stream_early_slabs")) *value = c->stream_early_slabs;
  else if (!strcmp(key, "stream_early_unit")) *value = c->stream_early_unit;
  else if (!strcmp(key, "stream_early_ratio")) *value = c->stream_early_ratio;
  else if (!strcmp(key, "stream_early_parts")) *value = c->stream_early_parts;
  else if (!strcmp(key, "forward_slab_mb")) *value = c->forward_slab_bytes >> 20;
  else if (!strcmp(key, "forward_used_tc")) *value = c->forward_used_tc;
  else if (!strcmp(key, "sm_count")) *value = c->sm_count;
  else { set_error("unknown option %s", key); return DGRP_E_ARG; }
  return DGRP_OK;
}

/* ---------------------------------- deepgrp.sequence ---------------------------------- */

int dgrp_one_hot_stage(dgrp_ctx *c, const uint8_t *seq, int64_t n, int fold_case,
                       int64_t *startpos, int64_t *out_len) {
  Use use(c->device);
  DGRP_REQUIRE(n >= 0, "negative length");
  c->staged_len = -1;
  DGRP_CHECK(c->raw.reserve((size_t)n + 16));
  if (n > 0) DGRP_CUDA(cudaMemcpyAsync(c->raw.p, seq, (size_t)n, cudaMemcpyHostToDevice, c->stream));
  DGRP_CHECK(c->small.reserve(256));
  DGRP_CHECK(c->pin_small.reserve(256));
  int64_t *d_fl = c->small.as<int64_t>() + 16;
  DGRP_CHECK(launch_trim(c, c->raw.as<uint8_t>(), n, fold_case, d_fl));
  int64_t *h = c->pin_small.as<int64_t>() + 8;
  DGRP_CUDA(cudaMemcpyAsync(h, d_fl, 16, cudaMemcpyDeviceToHost, c->stream));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  *startpos = h[0];
  *out_len = h[1] - h[0];
  c->staged_n = n; c->staged_start = h[0]; c->staged_len = *out_len;
  if (*out_len < 0) {
    set_error("negative dimensions are not allowed (all-'N' sequence)");
    return DGRP_E_ALLN;
  }
  return DGRP_OK;
}

int dgrp_one_hot_fetch(dgrp_ctx *c, int8_t *fwd) {
  Use use(c->device);
  DGRP_REQUIRE(c->staged_len >= 0, "dgrp_one_hot_fetch without a successful dgrp_one_hot_stage");
  const int64_t len = c->staged_len;
  if (len == 0) return DGRP_OK;
  DGRP_CHECK(c->onehot.reserve((size_t)len * 5));
  DGRP_CHECK(launch_onehot(c, c->raw.as<uint8_t>(), c->staged_start, len, c->onehot.as<int8_t>()));
  DGRP_CUDA(cudaMemcpyAsync(fwd, c->onehot.p, (size_t)len * 5, cudaMemcpyDeviceToHost, c->stream));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  return DGRP_OK;
}

int dgrp_get_max_dev(dgrp_ctx *c, float *d_output, int64_t out_rows, const float *d_inputs,
                     int64_t batchsize, int64_t dim0, int64_t dim1, int64_t stride) {
  Use use(c->device);
  DGRP_REQUIRE(batchsize >= 0 && dim0 >= 0 && dim1 >= 0 && stride >= 0, "negative dimension");
  if (batchsize == 0 || dim0 == 0 || dim1 == 0) return DGRP_OK;
  DGRP_REQUIRE((batchsize - 1) * stride + dim0 <= out_rows,
               "get_max would write %lld rows but output has %lld",
               (long long)((batchsize - 1) * stride + dim0), (long long)out_rows);
  return launch_get_max(c, d_output, d_inputs, batchsize, dim0, dim1, stride);
}

int dgrp_get_max(dgrp_ctx *c, float *output, int64_t out_rows, const float *inputs,
                 int64_t batchsize, int64_t dim0, int64_t dim1, int64_t stride) {
  Use use(c->device);
  DGRP_REQUIRE(batchsize >= 0 && dim0 >= 0 && dim1 >= 0 && stride >= 0, "negative dimension");
  if (batchsize == 0 || dim0 == 0 || dim1 == 0) return DGRP_OK;
  const int64_t rows = (batchsize - 1) * stride + dim0;
  DGRP_REQUIRE(rows <= out_rows, "get_max would write %lld rows but output has %lld",
               (long long)rows, (long long)out_rows);
  const size_t ob = (size_t)rows * dim1 * 4, ib = (size_t)batchsize * dim0 * dim1 * 4;
  DGRP_CHECK(c->io_a.reserve(ob));
  DGRP_CHECK(c->io_b.reserve(ib));
  DGRP_CUDA(cudaMemcpyAsync(c->io_a.p, output, ob, cudaMemcpyHostToDevice, c->stream));
  DGRP_CUDA(cudaMemcpyAsync(c->io_b.p, inputs, ib, cudaMemcpyHostToDevice, c->stream));
  DGRP_CHECK(launch_get_max(c, c->io_a.as<float>(), c->io_b.as<float>(), batchsize, dim0, dim1, stride));
  DGRP_CUDA(cudaMemcpyAsync(output, c->io_a.p, ob, cudaMemcpyDeviceToHost, c->stream));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  return DGRP_OK;
}

int dgrp_get_segments(dgrp_ctx *c, const int64_t *classes, int64_t size, int64_t startpos,
                      int64_t out3[3]) {
  Use use(c->device);
  DGRP_REQUIRE(size > 0 && startpos >= 0 && startpos < size, "startpos %lld outside [0, %lld)",
               (long long)startpos, (long long)size);
  DGRP_CHECK(c->classes64.reserve((size_t)size * 8));
  DGRP_CHECK(c->small.reserve(256));
  DGRP_CUDA(cudaMemcpyAsync(c->classes64.p, classes, (size_t)size * 8, cudaMemcpyHostToDevice, c->stream));
  int64_t *d_out = c->small.as<int64_t>() + 24;
  DGRP_CHECK(launch_get_segments(c, c->classes64.as<int64_t>(), size, startpos, d_out));
  DGRP_CUDA(cudaMemcpyAsync(out3, d_out, 24, cudaMemcpyDeviceToHost, c->stream));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  return DGRP_OK;
}

int dgrp_yield_segments(dgrp_ctx *c, const int64_t *classes, int64_t size, int64_t start_offset,
                        int64_t *out, int64_t cap, int64_t *n_out) {
  Use use(c->device);
  *n_out = 0;
  if (size <= 0) return DGRP_OK;
  DGRP_CHECK(c->classes64.reserve((size_t)size * 8));
  DGRP_CUDA(cudaMemcpyAsync(c->classes64.p, classes, (size_t)size * 8, cudaMemcpyHostToDevice, c->stream));
  int64_t *d_tri = nullptr;
  int64_t cnt = 0;
  DGRP_CHECK(run_segments(c, nullptr, c->classes64.as<int64_t>(), size, start_offset, true, &d_tri, &cnt));
  *n_out = cnt;
  if (cnt == 0) return DGRP_OK;
  if (cnt > cap || !out) {
    set_error("segment buffer too small: %lld needed, capacity %lld", (long long)cnt, (long long)cap);
    return DGRP_E_CAPACITY;
  }
  DGRP_CUDA(cudaMemcpyAsync(out, d_tri, (size_t)cnt * 24, cudaMemcpyDeviceToHost, c->stream));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  return DGRP_OK;
}

/* ------------------------------------- deepgrp.mss ------------------------------------- */

int dgrp_mss_find_all(dgrp_ctx *c, int n, const double *S, double min_sc, double xdrop,
                      dgrp_seg_t *out, int64_t cap, int *n_seg) {
  Use use(c->device);
  *n_seg = 0;
  if (n <= 0) return DGRP_OK;
  DGRP_CHECK(c->scores64.reserve((size_t)n * 8));
  DGRP_CUDA(cudaMemcpyAsync(c->scores64.p, S, (size_t)n * 8, cudaMemcpyHostToDevice, c->stream));
  dgrp_seg_t *d_segs = nullptr;
  DGRP_CHECK(run_mss_segments(c, c->scores64.as<double>(), nullptr, n, min_sc, xdrop, &d_segs, n_seg));
  if (*n_seg == 0) return DGRP_OK;
  if (*n_seg > cap || !out) {
    set_error("segment buffer too small: %d needed, capacity %lld", *n_seg, (long long)cap);
    return DGRP_E_CAPACITY;
  }
  DGRP_CUDA(cudaMemcpyAsync(out, d_segs, (size_t)*n_seg * sizeof(dgrp_seg_t), cudaMemcpyDeviceToHost, c->stream));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  return DGRP_OK;
}

int dgrp_find_mss_labels(dgrp_ctx *c, const double *scores, const int64_t *label, int n,
                         int nof_labels, int min_mss_len, int xdrop_len, double *one_hot) {
  Use use(c->device);
  if (n <= 0) return DGRP_OK;
  double min_sc, xdrop;
  mss_thresholds(min_mss_len, xdrop_len, &min_sc, &xdrop);
  DGRP_CHECK(c->scores64.reserve((size_t)n * 8));
  DGRP_CHECK(c->classes64.reserve((size_t)n * 8));
  DGRP_CHECK(c->labels2.reserve((size_t)n));
  DGRP_CHECK(c->io_a.reserve((size_t)n * nof_labels * 8));
  DGRP_CUDA(cudaMemcpyAsync(c->scores64.p, scores, (size_t)n * 8, cudaMemcpyHostToDevice, c->stream));
  DGRP_CUDA(cudaMemcpyAsync(c->classes64.p, label, (size_t)n * 8, cudaMemcpyHostToDevice, c->stream));
  dgrp_seg_t *d_segs = nullptr;
  int n_seg = 0;
  DGRP_CHECK(run_mss_segments(c, c->scores64.as<double>(), nullptr, n, min_sc, xdrop, &d_segs, &n_seg));
  DGRP_CHECK(run_gap_fill(c, d_segs, n_seg, nullptr, c->classes64.as<int64_t>(), n, nof_labels,
                          c->labels2.as<uint8_t>()));
  DGRP_CHECK(launch_labels_to_onehot(c, c->labels2.as<uint8_t>(), n, nof_labels, c->io_a.as<double>()));
  DGRP_CUDA(cudaMemcpyAsync(one_hot, c->io_a.p, (size_t)n * nof_labels * 8, cudaMemcpyDeviceToHost, c->stream));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  return DGRP_OK;
}

int dgrp_filter_segments(dgrp_ctx *c, uint8_t *labels, int64_t n, int64_t min_len) {
  Use use(c->device);
  if (n <= 0) return DGRP_OK;
  DGRP_CHECK(c->labels.reserve((size_t)n));
  DGRP_CHECK(c->labels2.reserve((size_t)n));
  DGRP_CUDA(cudaMemcpyAsync(c->labels.p, labels, (size_t)n, cudaMemcpyHostToDevice, c->stream));
  DGRP_CHECK(launch_filter_segments(c, c->labels.as<uint8_t>(), c->labels2.as<uint8_t>(), n, min_len));
  DGRP_CUDA(cudaMemcpyAsync(labels, c->labels2.p, (size_t)n, cudaMemcpyDeviceToHost, c->stream));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  return DGRP_OK;
}

int dgrp_confusion_matrix(dgrp_ctx *c, const uint8_t *truelbl, const uint8_t *predictedlbl, int64_t n,
                          int64_t *cnf) {
  Use use(c->device);
  DGRP_REQUIRE(n >= 0, "n must be non-negative");
  DGRP_CHECK(c->labels.reserve((size_t)(n > 0 ? n : 1)));
  DGRP_CHECK(c->labels2.reserve((size_t)(n > 0 ? n : 1)));
  DGRP_CHECK(c->small.reserve(4096));
  DGRP_CHECK(c->pin_small.reserve(4096));
  if (n > 0) {
    DGRP_CUDA(cudaMemcpyAsync(c->labels.p, truelbl, (size_t)n, cudaMemcpyHostToDevice, c->stream));
    DGRP_CUDA(cudaMemcpyAsync(c->labels2.p, predictedlbl, (size_t)n, cudaMemcpyHostToDevice, c->stream));
  }
  unsigned long long *d_cnf = c->small.as<unsigned long long>() + 64;
  int *d_bad = reinterpret_cast<int *>(d_cnf + 256);
  DGRP_CHECK(launch_confusion(c, c->labels.as<uint8_t>(), c->labels2.as<uint8_t>(), n, d_cnf, d_bad));
  unsigned long long *h = c->pin_small.as<unsigned long long>() + 64;
  DGRP_CUDA(cudaMemcpyAsync(h, d_cnf, 257 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  DGRP_REQUIRE(*reinterpret_cast<int *>(h + 256) == 0, "confusion_matrix: labels must be < 16");
  for (int i = 0; i < 256; ++i) cnf[i] = (int64_t)h[i];
  return DGRP_OK;
}

/* ---------------------------------------- model ---------------------------------------- */

int dgrp_model_create(dgrp_ctx *c, int rnn, int vecsize, int units, int n_classes,
                      const float *kernel, const float *recurrent, const float *bias,
                      const float *att_scale, const float *ff_kernel, const float *ff_bias,
                      dgrp_model **out) {
  Use use(c->device);
  *out = nullptr;
  if (rnn != 0 && rnn != 1) {
    set_error("rnn must be 0 (GRU, reset_after=True) or 1 (LSTM)");
    return DGRP_E_UNSUPPORTED;
  }
  if (rnn == 1) att_scale = nullptr;   // attention is ignored for LSTM (deepgrp/model.py:308)
  DGRP_REQUIRE(vecsize > 0 && units > 0, "vecsize and units must be positive");
  DGRP_REQUIRE(n_classes >= MODEL_CMIN && n_classes <= MODEL_CMAX, "n_classes must be in [%d, %d], got %d",
               MODEL_CMIN, MODEL_CMAX, n_classes);
  if (units > 128) {
    set_error("units=%d not supported by the CUDA forward (max 128)", units);
    return DGRP_E_UNSUPPORTED;
  }
  int UP = 32;
  while (UP < units) UP <<= 1;
  const int U = units, G = rnn == 1 ? 4 : 3;   // LSTM: gates i, f, c, o and a single bias [4U]
  std::vector<float> P((size_t)5 * G * UP, 0.f), Wk((size_t)5 * G * UP, 0.f), b0((size_t)G * UP, 0.f),
      b1((size_t)G * UP, 0.f), Rp((size_t)UP * G * UP, 0.f);
  for (int cc = 0; cc < 5; ++cc)
    for (int g = 0; g < G; ++g)
      for (int u = 0; u < U; ++u) {
        const float w = kernel[(size_t)cc * G * U + g * U + u];
        Wk[((size_t)cc * G + g) * UP + u] = w;
        P[((size_t)cc * G + g) * UP + u] = w + bias[g * U + u];
      }
  for (int g = 0; g < G; ++g)
    for (int u = 0; u < U; ++u) {
      b0[(size_t)g * UP + u] = bias[g * U + u];
      b1[(size_t)g * UP + u] = rnn == 1 ? 0.f : bias[(size_t)G * U + g * U + u];
    }
  for (int k = 0; k < U; ++k)
    for (int g = 0; g < G; ++g)
      for (int u = 0; u < U; ++u)
        Rp[((size_t)k * G + g) * UP + u] = recurrent[(size_t)k * G * U + g * U + u];
  // bf16 hi|mid|lo pieces of recurrent^T in the tcgen05 operand layout (forward_tc.cu)
  std::vector<uint16_t> Bs, Bh;
  int b16_shift = 0;
  if (UP <= 64 && rnn == 0) {
    const int N = 3 * UP + 16, SBO = (UP / 8) * 128;   // 16 extra rows: FF kernel halves (forward_tc.cu)
    const bool att = att_scale != nullptr;
    Bs.assign((size_t)3 * N * UP, 0);
    auto f2bf = [](float f) -> uint16_t {
      uint32_t u;
      memcpy(&u, &f, 4);
      if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
      const uint32_t r = 0x7fffu + ((u >> 16) & 1u);
      return (uint16_t)((u + r) >> 16);
    };
    auto bf2f = [](uint16_t b) -> float {
      const uint32_t u = (uint32_t)b << 16;
      float f;
      memcpy(&f, &u, 4);
      return f;
    };
    // x(n, k): column n of [R | K/2] (pre-scaled gate columns, halved projection columns), row k
    auto entry = [&](int n, int k) -> float {
      if (n < 3 * UP) {
        // gate columns are pre-scaled so that the accumulator feeds ex2 directly (forward_tc.cu)
        const int g = n / UP, u = n % UP;
        return Rp[((size_t)k * G + g) * UP + u] * (g < 2 ? -1.4426950408889634f : 2.8853900817779268f);
      }
      if (k >= U) return 0.f;
      const int j = n - 3 * UP;          // 0..4: ctx half (attention only), 8..12: avg half
      // halved: the kernel adds the projections of the two directions, avg.K = h_fwd.K/2 + h_rc.K/2
      if (j < 5 && j < n_classes && att) return 0.5f * ff_kernel[(size_t)k * n_classes + j];
      if (j >= 8 && j - 8 < n_classes && j < 13)
        return 0.5f * ff_kernel[(size_t)((att ? U : 0) + k) * n_classes + (j - 8)];
      return 0.f;
    };
    float bmax = 0.f;
    for (int n = 0; n < N; ++n)
      for (int k = 0; k < UP; ++k) {
        const float x = entry(n, k);
        bmax = std::fmax(bmax, std::fabs(x));
        const uint16_t hi = f2bf(x);
        const float r1 = x - bf2f(hi);
        const uint16_t mid = f2bf(r1);
        const float r2 = r1 - bf2f(mid);
        const uint16_t lo = f2bf(r2);
        const size_t off = ((size_t)(n / 8) * SBO + (size_t)(k / 8) * 128 + (n % 8) * 16 + (k % 8) * 2) / 2;
        Bs[off] = hi;
        Bs[(size_t)N * UP + off] = mid;
        Bs[(size_t)2 * N * UP + off] = lo;
      }
    // fp16 hi|lo of the same matrix times 2^shift (largest entry just below 2^14, so that the low
    // pieces of all but negligible entries are normal half-precision numbers), with 16 more K rows:
    // rows UP + c (c = 0..4) hold the z / r entries of the input table for base c -- the kernel puts
    // one_hot(x_t) * 2^8 into the matching K columns of A, so the MMA adds the input projection of the
    // z and r gates (the h gate's stays outside r * (.), reset_after=True) and the h gate's recurrent bias.
    const int KP = UP + 16, SBO16 = (KP / 8) * 128;
    auto entry16 = [&](int n, int k) -> float {
      if (k < UP) return entry(n, k);
      const int cc = k - UP;
      if (cc >= 5 || n >= 3 * UP) return 0.f;
      if (n >= 2 * UP) return b1[n] * 2.8853900817779268f;   // h gate: its recurrent bias (inside r * (.))
      return (P[(size_t)cc * G * UP + n] + b1[n]) * -1.4426950408889634f;   // n = g * UP + u, g < 2
    };
    bmax = 0.f;
    for (int n = 0; n < N; ++n)
      for (int k = 0; k < KP; ++k) bmax = std::fmax(bmax, std::fabs(entry16(n, k)));
    if (bmax > 0.f && std::isfinite(bmax)) {
      int e = 0;
      std::frexp(bmax, &e);             // bmax = f * 2^e, f in [0.5, 1)
      b16_shift = 14 - e;
      if (b16_shift > 24) b16_shift = 24;
      if (b16_shift < -24) b16_shift = -24;
    }
    Bh.assign((size_t)2 * N * KP, 0);
    for (int n = 0; n < N; ++n)
      for (int k = 0; k < KP; ++k) {
        const float x = std::ldexp(entry16(n, k), b16_shift);
        const __half hi = __float2half_rn(x);
        const __half lo = __float2half_rn(x - __half2float(hi));
        const size_t off = ((size_t)(n / 8) * SBO16 + (size_t)(k / 8) * 128 + (n % 8) * 16 + (k % 8) * 2) / 2;
        memcpy(&Bh[off], &hi, 2);
        memcpy(&Bh[(size_t)N * KP + off], &lo, 2);
      }
  }
  std::vector<uint16_t> Bw[2][2];
  int bw_shift = 0;
  build_tcw_operands(rnn, U, UP, n_classes, att_scale != nullptr, Rp.data(), P.data(), b1.data(), ff_kernel, Bw,
                     &bw_shift);
  dgrp_model *m = new dgrp_model();
  m->device = c->device; m->rnn = rnn; m->T = vecsize; m->U = U; m->C = n_classes; m->UP = UP;
  m->attention = att_scale != nullptr;
  m->b16_shift = b16_shift;
  m->bw_shift = bw_shift;
  const int F = m->attention ? 2 * U : U;
  auto up = [&](float **dst, const float *src, size_t count) -> int {
    DGRP_CUDA(cudaMalloc((void **)dst, count * sizeof(float)));
    DGRP_CUDA(cudaMemcpyAsync(*dst, src, count * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    return DGRP_OK;
  };
  int rc = DGRP_OK;
  if ((rc = up(&m->d_P, P.data(), P.size())) || (rc = up(&m->d_Wk, Wk.data(), Wk.size())) ||
      (rc = up(&m->d_b0, b0.data(), b0.size())) || (rc = up(&m->d_b1, b1.data(), b1.size())) ||
      (rc = up(&m->d_Rp, Rp.data(), Rp.size())) ||
      (rc = up(&m->d_ffk, ff_kernel, (size_t)F * n_classes)) ||
      (rc = up(&m->d_ffb, ff_bias, (size_t)n_classes)) ||
      (m->attention && (rc = up(&m->d_scale, att_scale, (size_t)U))) ||
      (!Bs.empty() && (rc = up(reinterpret_cast<float **>(&m->d_Bsplit),
                               reinterpret_cast<const float *>(Bs.data()), Bs.size() / 2))) ||
      (!Bh.empty() && (rc = up(reinterpret_cast<float **>(&m->d_Bsplit16),
                               reinterpret_cast<const float *>(Bh.data()), Bh.size() / 2))) ||
      (!Bh.empty() && false)) {
    cudaStreamSynchronize(c->stream);
    dgrp_model_destroy(m);
    return rc;
  }
  for (int a = 0; a < 2 && rc == DGRP_OK; ++a)
    for (int b = 0; b < 2 && rc == DGRP_OK; ++b)
      if (!Bw[a][b].empty())
        rc = up(reinterpret_cast<float **>(&m->d_Bw[a][b]), reinterpret_cast<const float *>(Bw[a][b].data()),
                Bw[a][b].size() / 2);
  if (rc != DGRP_OK) {
    cudaStreamSynchronize(c->stream);
    dgrp_model_destroy(m);
    return rc;
  }
  DGRP_CUDA(cudaStreamSynchronize(c->stream));   // host vectors go out of scope
  *out = m;
  return DGRP_OK;
}

int dgrp_model_destroy(dgrp_model *m) {
  if (!m) return DGRP_OK;
  Use use(m->device);
  float *ptrs[] = {m->d_kernel, m->d_bias, m->d_recurrent, m->d_P, m->d_Wk, m->d_b0, m->d_Rp,
                   m->d_b1, m->d_scale, m->d_ffk, m->d_ffb};
  for (float *p : ptrs)
    if (p) cudaFree(p);
  if (m->d_Bsplit) cudaFree(m->d_Bsplit);
  if (m->d_Bsplit16) cudaFree(m->d_Bsplit16);
  for (auto &a : m->d_Bw)
    for (uint16_t *q : a)
      if (q) cudaFree(q);
  delete m;
  return DGRP_OK;
}

int dgrp_forward_windows(dgrp_ctx *c, dgrp_model *m, const float *batch, int64_t nbatch,
                         float *probs) {
  Use use(c->device);
  if (nbatch <= 0) return DGRP_OK;
  const size_t ib = (size_t)nbatch * m->T * 5 * 4, ob = (size_t)nbatch * m->T * m->C * 4;
  DGRP_CHECK(c->io_a.reserve(ib));
  DGRP_CHECK(c->io_b.reserve(ob));
  DGRP_CUDA(cudaMemcpyAsync(c->io_a.p, batch, ib, cudaMemcpyHostToDevice, c->stream));
  DGRP_CHECK(run_forward_dense(c, m, c->io_a.as<float>(), nbatch, c->io_b.as<float>()));
  DGRP_CUDA(cudaMemcpyAsync(probs, c->io_b.p, ob, cudaMemcpyDeviceToHost, c->stream));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  return DGRP_OK;
}

/* ---------------------------------- deepgrp.prediction --------------------------------- */

int dgrp_predict_onehot(dgrp_ctx *c, dgrp_model *m, const int8_t *fwd, int64_t length, int step,
                        int batch_size, int compat, float *predictions) {
  Use use(c->device);
  DGRP_REQUIRE(length >= 0, "negative length");
  if (length == 0) return DGRP_OK;
  DGRP_CHECK(c->onehot.reserve((size_t)length * 5));
  DGRP_CHECK(c->codes.reserve((size_t)length + 16));
  DGRP_CUDA(cudaMemcpyAsync(c->onehot.p, fwd, (size_t)length * 5, cudaMemcpyHostToDevice, c->stream));
  DGRP_CHECK(launch_onehot_to_codes(c, c->onehot.as<int8_t>(), length, c->codes.as<uint8_t>()));
  DGRP_CHECK(c->pin_small.reserve(256));
  int *h_flag = c->pin_small.as<int>() + 40;
  DGRP_CUDA(cudaMemcpyAsync(h_flag, c->small.p, 4, cudaMemcpyDeviceToHost, c->stream));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  DGRP_REQUIRE(*h_flag == 0, "input matrix is not one-hot int8[5, L] (use forward_windows for dense input)");
  DGRP_CHECK(core_predict(c, m, c->codes.as<uint8_t>(), length, step, batch_size, compat));
  DGRP_CUDA(cudaMemcpyAsync(predictions, c->pred.p, (size_t)length * m->C * 4, cudaMemcpyDeviceToHost, c->stream));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  return DGRP_OK;
}

int dgrp_mss_scores(dgrp_ctx *c, const float *probs, int64_t n, int n_classes, double *scores,
                    int64_t *classes) {
  Use use(c->device);
  if (n <= 0) return DGRP_OK;
  DGRP_CHECK(c->io_a.reserve((size_t)n * n_classes * 4));
  DGRP_CHECK(c->scores64.reserve((size_t)n * 8));
  DGRP_CHECK(c->classes64.reserve((size_t)n * 8));
  DGRP_CUDA(cudaMemcpyAsync(c->io_a.p, probs, (size_t)n * n_classes * 4, cudaMemcpyHostToDevice, c->stream));
  DGRP_CHECK(launch_score(c, c->io_a.as<float>(), n, n_classes, nullptr, nullptr,
                          c->scores64.as<double>(), c->classes64.as<int64_t>()));
  if (scores) DGRP_CUDA(cudaMemcpyAsync(scores, c->scores64.p, (size_t)n * 8, cudaMemcpyDeviceToHost, c->stream));
  if (classes) DGRP_CUDA(cudaMemcpyAsync(classes, c->classes64.p, (size_t)n * 8, cudaMemcpyDeviceToHost, c->stream));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  return DGRP_OK;
}

int dgrp_apply_mss(dgrp_ctx *c, const float *probs, int n, int n_classes, int min_mss_len,
                   int xdrop_len, double *one_hot) {
  Use use(c->device);
  if (n <= 0) return DGRP_OK;
  DGRP_CHECK(c->io_a.reserve((size_t)n * n_classes * 4));
  DGRP_CUDA(cudaMemcpyAsync(c->io_a.p, probs, (size_t)n * n_classes * 4, cudaMemcpyHostToDevice, c->stream));
  DGRP_CHECK(core_labels(c, c->io_a.as<float>(), nullptr, nullptr, n, n_classes, 1, min_mss_len, xdrop_len));
  DGRP_CHECK(c->io_b.reserve((size_t)n * n_classes * 8));
  DGRP_CHECK(launch_labels_to_onehot(c, c->labels2.as<uint8_t>(), n, n_classes, c->io_b.as<double>()));
  DGRP_CUDA(cudaMemcpyAsync(one_hot, c->io_b.p, (size_t)n * n_classes * 8, cudaMemcpyDeviceToHost, c->stream));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  return DGRP_OK;
}

int dgrp_softmax(dgrp_ctx *c, const float *array, int64_t n, int n_classes, float *out) {
  Use use(c->device);
  if (n <= 0) return DGRP_OK;
  const size_t b = (size_t)n * n_classes * 4;
  DGRP_CHECK(c->io_a.reserve(b));
  DGRP_CHECK(c->io_b.reserve(b));
  DGRP_CUDA(cudaMemcpyAsync(c->io_a.p, array, b, cudaMemcpyHostToDevice, c->stream));
  DGRP_CHECK(launch_softmax_global(c, c->io_a.as<float>(), n, n_classes, c->io_b.as<float>()));
  DGRP_CUDA(cudaMemcpyAsync(out, c->io_b.p, b, cudaMemcpyDeviceToHost, c->stream));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  return DGRP_OK;
}

/* ----------------------------------- deepgrp.__main__ ---------------------------------- */

int dgrp_predict_sequence(dgrp_ctx *c, dgrp_model *m, const uint8_t *seq, int64_t n,
                          int fold_case, int step, int batch_size, int use_mss, int min_mss_len,
                          int xdrop_len, int compat, int64_t *startpos, int64_t *length,
                          uint8_t *labels, dgrp_row_t *rows, int64_t cap, int64_t *n_rows) {
  Use use(c->device);
  DGRP_REQUIRE(n >= 0, "negative length");
  const int64_t launches0 = c->launches;
  *n_rows = 0;
  stamp(c, 0);
  DGRP_CHECK(c->raw.reserve((size_t)n + 16));
  if (n > 0) DGRP_CUDA(cudaMemcpyAsync(c->raw.p, seq, (size_t)n, cudaMemcpyHostToDevice, c->stream));
  DGRP_CHECK(core_encode(c, c->raw.as<uint8_t>(), n, fold_case, startpos, length));
  if (*length < 0) {
    set_error("negative dimensions are not allowed (all-'N' sequence)");
    return DGRP_E_ALLN;
  }
  stamp(c, 1);
  const int64_t L = *length;
  DGRP_CHECK(core_predict(c, m, c->codes.as<uint8_t>(), L, step, batch_size, compat, use_mss != 0));
  stamp(c, 2);
  DGRP_CHECK(core_labels_after_predict(c, L, m->C, use_mss, min_mss_len, xdrop_len));
  stamp(c, 4);
  if (labels && L > 0)
    DGRP_CUDA(cudaMemcpyAsync(labels, c->labels2.p, (size_t)L, cudaMemcpyDeviceToHost, c->stream));
  int rc = DGRP_OK;
  if (L > 0) rc = core_rows(c, L, *startpos, 0, true, rows, cap, n_rows);
  stamp(c, 5);
  finish_timings(c, launches0);
  return rc;
}

// filename == nullptr: rows are copied to the host (c->fa_rows); else the TSV text is produced on
// the device and lands in c->tsv_host.
static int predict_fasta_impl(dgrp_ctx *c, dgrp_model *m, const uint8_t *fasta, int64_t nbytes,
                              const char *filename, int step, int batch_size, int use_mss,
                              int min_mss_len, int xdrop_len, int compat, int64_t *n_rows,
                              int64_t *n_records) {
  Use use(c->device);
  c->tsv_len = 0;
  int64_t total_rows = 0;
  const size_t fn_len = filename ? strlen(filename) : 0;
  const int64_t launches0 = c->launches;
  *n_rows = 0; *n_records = 0;
  c->fa_rows.clear(); c->fa_hdr_off.clear(); c->fa_hdr_len.clear();
  c->fa_startpos.clear(); c->fa_length.clear();
  c->fa_tsv_off.clear(); c->fa_tsv_len.clear(); c->fa_owner.clear();
  DGRP_REQUIRE(nbytes >= 0, "negative length");
  stamp(c, 0);
  DGRP_CHECK(c->raw.reserve((size_t)nbytes + 16));
  if (nbytes > 0) DGRP_CUDA(cudaMemcpyAsync(c->raw.p, fasta, (size_t)nbytes, cudaMemcpyHostToDevice, c->stream));
  int64_t n_seq = 0, n_hdr = 0;
  DGRP_CHECK(run_fasta_decode(c, c->raw.as<uint8_t>(), nbytes, &n_seq, &n_hdr));
  std::vector<int64_t> hpos(n_hdr), hseq(n_hdr + 1);
  if (n_hdr > 0) {
    const int64_t *t = c->pin_b.as<int64_t>();
    for (int64_t k = 0; k < n_hdr; ++k) { hpos[k] = t[k]; hseq[k] = t[(n_hdr + 1) + k]; }
  }
  hseq[n_hdr] = n_seq;
  auto ws = [](uint8_t b) { return (b >= 9 && b <= 13) || (b >= 28 && b <= 32); };
  // Contig sharding (SURVEY.md section 8e): every rank decodes the file and derives the same
  // largest-first assignment of the kept records to ranks; it then processes only its own.
  std::vector<int64_t> owner_of(n_hdr, -1);
  {
    std::vector<int64_t> kept;
    for (int64_t k = 0; k < n_hdr; ++k) {
      int64_t b = hpos[k] + 1, e = b;
      while (e < nbytes && fasta[e] != '\n' && !(fasta[e] == '\r' && !(e + 1 < nbytes && fasta[e + 1] == '\n'))) ++e;
      while (e > b && ws(fasta[e - 1])) --e;
      if (e > b) kept.push_back(k);
    }
    std::vector<int64_t> order(kept);
    std::stable_sort(order.begin(), order.end(), [&](int64_t a, int64_t b2) {
      return (hseq[a + 1] - hseq[a]) > (hseq[b2 + 1] - hseq[b2]);
    });
    const int world = c->shard_world > 0 ? c->shard_world : 1;
    std::vector<int64_t> load(world, 0);
    for (int64_t k : order) {
      int best = 0;
      for (int r = 1; r < world; ++r)
        if (load[r] < load[best]) best = r;
      owner_of[k] = best;
      load[best] += hseq[k + 1] - hseq[k];
    }
  }
  float enc_ms = 0.f, fwd_ms = 0.f, score_ms = 0.f, mss_ms = 0.f, seg_ms = 0.f;
  int64_t windows = 0, bases = 0;
  cudaEvent_t e_begin = c->ev[6], e_end = c->ev[7];
  cudaEventRecord(e_begin, c->stream);
  int rc = DGRP_OK;
  for (int64_t k = 0; k < n_hdr && rc == DGRP_OK; ++k) {
    // header = stripped line without its '>' (__main__.py:38)
    int64_t b = hpos[k] + 1, e = b;
    while (e < nbytes && fasta[e] != '\n' && !(fasta[e] == '\r' && !(e + 1 < nbytes && fasta[e + 1] == '\n'))) ++e;
    while (e > b && ws(fasta[e - 1])) --e;
    if (e == b) continue;                         // empty header: record dropped (__main__.py:36)
    const int32_t rec = (int32_t)c->fa_hdr_off.size();
    if (owner_of[k] != c->shard_rank) {   // another rank's record: table entry only
      c->fa_hdr_off.push_back(b); c->fa_hdr_len.push_back(e - b);
      c->fa_startpos.push_back(-1); c->fa_length.push_back(hseq[k + 1] - hseq[k]);
      c->fa_tsv_off.push_back(c->tsv_len); c->fa_tsv_len.push_back(0); c->fa_owner.push_back(owner_of[k]);
      continue;
    }
    const uint8_t *d_seq = c->io_b.as<uint8_t>() + hseq[k];
    const int64_t n = hseq[k + 1] - hseq[k];
    int64_t startpos = 0, length = 0;
    stamp(c, 0);
    rc = core_encode(c, d_seq, n, 1, &startpos, &length);
    if (rc != DGRP_OK) break;
    if (length < 0) {
      set_error("negative dimensions are not allowed (all-'N' record %d)", rec);
      rc = DGRP_E_ALLN;
      break;
    }
    c->fa_hdr_off.push_back(b); c->fa_hdr_len.push_back(e - b);
    c->fa_startpos.push_back(startpos); c->fa_length.push_back(length);
    c->fa_tsv_off.push_back(c->tsv_len); c->fa_tsv_len.push_back(0); c->fa_owner.push_back(owner_of[k]);
    stamp(c, 1);
    if ((rc = core_predict(c, m, c->codes.as<uint8_t>(), length, step, batch_size, compat, use_mss != 0))) break;
    windows += c->timings.windows; bases += length;
    stamp(c, 2);
    if ((rc = core_labels_after_predict(c, length, m->C, use_mss, min_mss_len, xdrop_len))) break;
    stamp(c, 4);
    if (length > 0) {
      int64_t *d_tri = nullptr;
      int64_t cnt = 0;
      if ((rc = run_segments(c, c->labels2.as<uint8_t>(), nullptr, length, startpos, false, &d_tri, &cnt))) break;
      total_rows += cnt;
      if (cnt > 0 && filename) {
        // prefix = "<filename>\t<header>\t"
        std::string prefix(filename, fn_len);
        prefix.push_back('\t');
        prefix.append(reinterpret_cast<const char *>(fasta + b), (size_t)(e - b));
        prefix.push_back('\t');
        int64_t need = 0;
        if ((rc = c->tsv_prefix.reserve(prefix.size() + 16))) break;
        if (cudaMemcpyAsync(c->tsv_prefix.p, prefix.data(), prefix.size(), cudaMemcpyHostToDevice, c->stream) != cudaSuccess) {
          set_error("uploading the TSV prefix failed"); rc = DGRP_E_CUDA; break;
        }
        if ((rc = run_tsv_measure(c, d_tri, cnt, (int)prefix.size(), &need))) break;   // syncs
        if ((rc = c->tsv_dev.reserve((size_t)need + 16))) break;
        if ((size_t)(c->tsv_len + need) > c->tsv_host.cap) {
          // grow the pinned text buffer, keeping what earlier records wrote
          PinBuf bigger;
          size_t want = std::max<size_t>((size_t)(c->tsv_len + need), c->tsv_host.cap * 2);
          if ((rc = bigger.reserve(want + 4096))) break;
          if (c->tsv_len > 0) memcpy(bigger.p, c->tsv_host.p, (size_t)c->tsv_len);
          c->tsv_host.release();
          c->tsv_host = bigger;
        }
        if ((rc = run_tsv_write(c, d_tri, cnt, c->tsv_prefix.as<uint8_t>(), (int)prefix.size(),
                                c->tsv_dev.as<uint8_t>()))) break;
        if (cudaMemcpyAsync(c->tsv_host.as<uint8_t>() + c->tsv_len, c->tsv_dev.p, (size_t)need,
                            cudaMemcpyDeviceToHost, c->stream) != cudaSuccess) {
          set_error("copying the TSV text failed"); rc = DGRP_E_CUDA; break;
        }
        c->tsv_len += need;
        c->fa_tsv_len.back() = need;
      } else if (cnt > 0) {
        if ((rc = c->pin_a.reserve((size_t)cnt * 24))) break;
        if (cudaMemcpyAsync(c->pin_a.p, d_tri, (size_t)cnt * 24, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
            cudaStreamSynchronize(c->stream) != cudaSuccess) {
          set_error("copying rows failed");
          rc = DGRP_E_CUDA;
          break;
        }
        const int64_t *t = c->pin_a.as<int64_t>();
        const size_t base = c->fa_rows.size();
        c->fa_rows.resize(base + (size_t)cnt);
        for (int64_t i = 0; i < cnt; ++i) {
          dgrp_row_t &r = c->fa_rows[base + i];
          r.start = t[3 * i]; r.end = t[3 * i + 1]; r.label = (int32_t)t[3 * i + 2]; r.record = rec;
        }
      }
    }
    stamp(c, 5);
    cudaStreamSynchronize(c->stream);
    float ms;
    cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]); enc_ms += ms;
    cudaEventElapsedTime(&ms, c->ev[1], c->ev[2]); fwd_ms += ms;
    cudaEventElapsedTime(&ms, c->ev[2], c->ev[3]); score_ms += ms;
    cudaEventElapsedTime(&ms, c->ev[3], c->ev[4]); mss_ms += ms;
    cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]); seg_ms += ms;
  }
  cudaEventRecord(e_end, c->stream);
  cudaStreamSynchronize(c->stream);
  dgrp_timings_t &t = c->timings;
  t.encode_ms = enc_ms; t.forward_ms = fwd_ms; t.score_ms = score_ms; t.mss_ms = mss_ms;
  t.segments_ms = seg_ms; t.attend_ms = 0.f; t.windows = windows; t.bases = bases;
  cudaEventElapsedTime(&t.total_ms, e_begin, e_end);
  t.kernel_launches = c->launches - launches0;
  *n_rows = total_rows;
  *n_records = (int64_t)c->fa_hdr_off.size();
  return rc;
}

int dgrp_predict_fasta(dgrp_ctx *c, dgrp_model *m, const uint8_t *fasta, int64_t nbytes, int step,
                       int batch_size, int use_mss, int min_mss_len, int xdrop_len, int compat,
                       int64_t *n_rows, int64_t *n_records) {
  return predict_fasta_impl(c, m, fasta, nbytes, nullptr, step, batch_size, use_mss, min_mss_len,
                            xdrop_len, compat, n_rows, n_records);
}

int dgrp_predict_fasta_tsv(dgrp_ctx *c, dgrp_model *m, const uint8_t *fasta, int64_t nbytes,
                           const char *filename, int step, int batch_size, int use_mss,
                           int min_mss_len, int xdrop_len, int compat, const uint8_t **tsv,
                           int64_t *tsv_len, int64_t *n_rows, int64_t *n_records) {
  *tsv = nullptr; *tsv_len = 0;
  DGRP_REQUIRE(filename != nullptr, "filename is required");
  const int rc = predict_fasta_impl(c, m, fasta, nbytes, filename, step, batch_size, use_mss,
                                    min_mss_len, xdrop_len, compat, n_rows, n_records);
  if (rc == DGRP_OK) { *tsv = c->tsv_host.as<uint8_t>(); *tsv_len = c->tsv_len; }
  return rc;
}

int dgrp_fasta_rows(dgrp_ctx *c, dgrp_row_t *rows, int64_t cap) {
  DGRP_REQUIRE((int64_t)c->fa_rows.size() <= cap, "row buffer too small: %lld needed",
               (long long)c->fa_rows.size());
  if (!c->fa_rows.empty()) memcpy(rows, c->fa_rows.data(), c->fa_rows.size() * sizeof(dgrp_row_t));
  return DGRP_OK;
}

int dgrp_fasta_records(dgrp_ctx *c, int64_t *hdr_off, int64_t *hdr_len, int64_t *startpos,
                       int64_t *length, int64_t cap) {
  const size_t n = c->fa_hdr_off.size();
  DGRP_REQUIRE((int64_t)n <= cap, "record buffer too small: %lld needed", (long long)n);
  if (n == 0) return DGRP_OK;
  if (hdr_off) memcpy(hdr_off, c->fa_hdr_off.data(), n * 8);
  if (hdr_len) memcpy(hdr_len, c->fa_hdr_len.data(), n * 8);
  if (startpos) memcpy(startpos, c->fa_startpos.data(), n * 8);
  if (length) memcpy(length, c->fa_length.data(), n * 8);
  return DGRP_OK;
}

int dgrp_fasta_record_tsv(dgrp_ctx *c, int64_t *owner, int64_t *tsv_off, int64_t *tsv_len, int64_t cap) {
  const size_t n = c->fa_owner.size();
  DGRP_REQUIRE((int64_t)n <= cap, "record buffer too small: %lld needed", (long long)n);
  if (n == 0) return DGRP_OK;
  if (owner) memcpy(owner, c->fa_owner.data(), n * 8);
  if (tsv_off) memcpy(tsv_off, c->fa_tsv_off.data(), n * 8);
  if (tsv_len) memcpy(tsv_len, c->fa_tsv_len.data(), n * 8);
  return DGRP_OK;
}

int dgrp_predict_codes_dev(dgrp_ctx *c, dgrp_model *m, const uint8_t *d_codes, int64_t length,
                           int step, int batch_size, int use_mss, int min_mss_len, int xdrop_len,
                           int compat, int64_t *n_rows) {
  Use use(c->device);
  const int64_t launches0 = c->launches;
  *n_rows = 0;
  c->codes_dev_length = -1;
  stamp(c, 0);
  stamp(c, 1);
  DGRP_CHECK(core_predict(c, m, d_codes, length, step, batch_size, compat, use_mss != 0));
  stamp(c, 2);
  DGRP_CHECK(core_labels_after_predict(c, length, m->C, use_mss, min_mss_len, xdrop_len));
  stamp(c, 4);
  int rc = DGRP_OK;
  if (length > 0) rc = core_rows(c, length, 0, 0, false, nullptr, 0, n_rows);
  stamp(c, 5);
  finish_timings(c, launches0);
  if (rc == DGRP_OK) {
    c->codes_dev_length = length;
    c->codes_dev_rows = *n_rows;
    c->codes_dev_reserves[0] = c->labels2.reserves;
    c->codes_dev_reserves[1] = c->segs.reserves;
  }
  return rc;
}

int dgrp_predict_codes_dev_results(dgrp_ctx *c, uint8_t *labels, int64_t length, int64_t *rows, int64_t n_rows) {
  Use use(c->device);
  DGRP_REQUIRE(c->codes_dev_length >= 0 && c->codes_dev_reserves[0] == c->labels2.reserves &&
                   c->codes_dev_reserves[1] == c->segs.reserves,
               "no dgrp_predict_codes_dev result to fetch: none ran, or another call has used its buffers since");
  DGRP_REQUIRE(length == c->codes_dev_length && n_rows == c->codes_dev_rows,
               "the last dgrp_predict_codes_dev has length %lld and %lld rows", (long long)c->codes_dev_length,
               (long long)c->codes_dev_rows);
  if (labels && length > 0)
    DGRP_CUDA(cudaMemcpyAsync(labels, c->labels2.p, (size_t)length, cudaMemcpyDeviceToHost, c->stream));
  if (rows && n_rows > 0)
    DGRP_CUDA(cudaMemcpyAsync(rows, c->segs.p, (size_t)n_rows * 24, cudaMemcpyDeviceToHost, c->stream));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  return DGRP_OK;
}

/* -------------------------------------- training --------------------------------------- */

// the Keras arrays <-> the trainer's flat parameter vector (TrainLayout)
static void train_pack(const dgrp_trainer *tr, std::vector<float> &flat, const float *kernel, const float *recurrent,
                       const float *bias, const float *att_scale, const float *ff_kernel, const float *ff_bias) {
  const TrainLayout &L = tr->L;
  const int U = tr->U, C = tr->C;
  flat.assign(L.n, 0.f);
  std::copy(kernel, kernel + 15 * U, flat.begin() + L.oK);
  std::copy(recurrent, recurrent + 3 * U * U, flat.begin() + L.oR);
  std::copy(bias, bias + 6 * U, flat.begin() + L.oB);
  if (tr->attention) std::copy(att_scale, att_scale + U, flat.begin() + L.oS);
  std::copy(ff_kernel, ff_kernel + L.F * C, flat.begin() + L.oF);
  std::copy(ff_bias, ff_bias + C, flat.begin() + L.oFB);
}

static int train_unpack(dgrp_trainer *tr, const DevBuf &src, float *kernel, float *recurrent, float *bias,
                        float *att_scale, float *ff_kernel, float *ff_bias) {
  dgrp_ctx *c = tr->ctx;
  const TrainLayout &L = tr->L;
  const int U = tr->U, C = tr->C;
  std::vector<float> flat(L.n);
  DGRP_CUDA(cudaMemcpyAsync(flat.data(), src.p, (size_t)L.n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  auto put = [&](float *dst, int off, int count) { if (dst) std::copy(flat.begin() + off, flat.begin() + off + count, dst); };
  put(kernel, L.oK, 15 * U);
  put(recurrent, L.oR, 3 * U * U);
  put(bias, L.oB, 6 * U);
  if (tr->attention) put(att_scale, L.oS, U);
  put(ff_kernel, L.oF, L.F * C);
  put(ff_bias, L.oFB, C);
  return DGRP_OK;
}

int dgrp_train_create(dgrp_ctx *c, int rnn, int vecsize, int units, int n_classes, int attention,
                      const float *kernel, const float *recurrent, const float *bias, const float *att_scale,
                      const float *ff_kernel, const float *ff_bias, int optimizer, float learning_rate, float rho,
                      float momentum, float epsilon, float dropout, dgrp_trainer **out) {
  Use use(c->device);
  *out = nullptr;
  if (rnn != 0) {
    set_error("training supports rnn=\"GRU\" only (LSTM is not implemented)");
    return DGRP_E_UNSUPPORTED;
  }
  DGRP_CHECK(train_check_shape(vecsize, units, n_classes, attention != 0));
  DGRP_REQUIRE(optimizer == DGRP_OPT_RMSPROP || optimizer == DGRP_OPT_ADAM,
               "optimizer must be DGRP_OPT_RMSPROP or DGRP_OPT_ADAM, got %d", optimizer);
  DGRP_REQUIRE(dropout >= 0.f && dropout < 1.f, "dropout must be in [0, 1), got %g", (double)dropout);
  DGRP_REQUIRE(learning_rate >= 0.f && epsilon >= 0.f && rho >= 0.f && momentum >= 0.f,
               "learning_rate, rho, momentum and epsilon must not be negative");
  DGRP_REQUIRE(kernel && recurrent && bias && ff_kernel && ff_bias && (!attention || att_scale),
               "a weight array is NULL");
  dgrp_trainer *tr = new dgrp_trainer();
  tr->ctx = c;
  tr->T = vecsize; tr->U = units; tr->C = n_classes; tr->attention = attention != 0;
  tr->optimizer = optimizer; tr->lr = learning_rate; tr->rho = rho; tr->momentum = momentum;
  tr->epsilon = epsilon; tr->dropout = dropout;
  tr->L = make_train_layout(units, n_classes, tr->attention);
  std::vector<float> flat;
  train_pack(tr, flat, kernel, recurrent, bias, att_scale, ff_kernel, ff_bias);
  const size_t bytes = (size_t)tr->L.n * sizeof(float);
  int rc = DGRP_OK;
  for (auto &e : tr->ev)
    if (rc == DGRP_OK && cudaEventCreate(&e) != cudaSuccess) { set_error("cudaEventCreate failed"); rc = DGRP_E_CUDA; }
  if (rc == DGRP_OK) rc = tr->w.reserve(bytes);
  if (rc == DGRP_OK) rc = tr->g.reserve(bytes);
  if (rc == DGRP_OK) rc = tr->s1.reserve(bytes);
  if (rc == DGRP_OK) rc = tr->s2.reserve(bytes);
  if (rc == DGRP_OK && cudaMemcpyAsync(tr->w.p, flat.data(), bytes, cudaMemcpyHostToDevice, c->stream) != cudaSuccess) {
    set_error("uploading the weights failed");
    rc = DGRP_E_CUDA;
  }
  if (rc == DGRP_OK && (cudaMemsetAsync(tr->g.p, 0, bytes, c->stream) != cudaSuccess ||
                        cudaMemsetAsync(tr->s1.p, 0, bytes, c->stream) != cudaSuccess ||
                        cudaMemsetAsync(tr->s2.p, 0, bytes, c->stream) != cudaSuccess)) {
    set_error("clearing the optimiser state failed");
    rc = DGRP_E_CUDA;
  }
  if (rc == DGRP_OK && cudaStreamSynchronize(c->stream) != cudaSuccess) {
    set_error("creating the trainer failed");
    rc = DGRP_E_CUDA;
  }
  if (rc != DGRP_OK) {
    dgrp_train_destroy(tr);
    return rc;
  }
  *out = tr;
  return DGRP_OK;
}

int dgrp_train_set_data(dgrp_trainer *tr, int which, const uint8_t *codes, const uint8_t *ymask, int64_t length) {
  dgrp_ctx *c = tr->ctx;
  Use use(c->device);
  DGRP_REQUIRE(which == 0 || which == 1, "which must be 0 (training) or 1 (validation), got %d", which);
  DGRP_REQUIRE(length >= tr->T, "record length %lld is shorter than vecsize %d", (long long)length, tr->T);
  DGRP_REQUIRE(codes && ymask, "codes and ymask must not be NULL");
  for (int64_t i = 0; i < length; ++i) {
    DGRP_REQUIRE(codes[i] <= 4, "code %d at position %lld is not a base code 0..4", codes[i], (long long)i);
    DGRP_REQUIRE((ymask[i] >> tr->C) == 0, "label mask 0x%x at position %lld names a class >= %d", ymask[i],
                 (long long)i, tr->C);
  }
  tr->length[which] = -1;
  DGRP_CHECK(tr->codes[which].reserve((size_t)length));
  DGRP_CHECK(tr->ymask[which].reserve((size_t)length));
  DGRP_CUDA(cudaMemcpyAsync(tr->codes[which].p, codes, (size_t)length, cudaMemcpyHostToDevice, c->stream));
  DGRP_CUDA(cudaMemcpyAsync(tr->ymask[which].p, ymask, (size_t)length, cudaMemcpyHostToDevice, c->stream));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  tr->length[which] = length;
  return DGRP_OK;
}

static int train_upload_starts(dgrp_trainer *tr, int which, const int64_t *starts, int64_t n) {
  dgrp_ctx *c = tr->ctx;
  DGRP_REQUIRE(which == 0 || which == 1, "which must be 0 (training) or 1 (validation), got %d", which);
  DGRP_REQUIRE(tr->length[which] >= 0, "no %s data set: call dgrp_train_set_data first",
               which ? "validation" : "training");
  DGRP_REQUIRE(n >= 1, "n must be at least 1, got %lld", (long long)n);
  DGRP_REQUIRE(starts, "starts must not be NULL");
  const int64_t last = tr->length[which] - tr->T;
  for (int64_t b = 0; b < n; ++b)
    DGRP_REQUIRE(starts[b] >= 0 && starts[b] <= last, "window start %lld (window %lld) is outside [0, %lld]",
                 (long long)starts[b], (long long)b, (long long)last);
  DGRP_CHECK(tr->starts.reserve((size_t)n * sizeof(int64_t)));
  DGRP_CUDA(cudaMemcpyAsync(tr->starts.p, starts, (size_t)n * sizeof(int64_t), cudaMemcpyHostToDevice, c->stream));
  return DGRP_OK;
}

static float train_mean_loss(const std::vector<float> &lpart, int64_t n, int T) {
  double s = 0.0;
  for (int64_t b = 0; b < n; ++b) s += lpart[b];
  return (float)(s / ((double)n * T));
}

int dgrp_train_step(dgrp_trainer *tr, const int64_t *starts, const uint8_t *keep, int64_t n, float *loss) {
  dgrp_ctx *c = tr->ctx;
  Use use(c->device);
  DGRP_CHECK(train_upload_starts(tr, 0, starts, n));
  DGRP_REQUIRE(keep, "keep must not be NULL");
  DGRP_CHECK(tr->keep.reserve((size_t)n * 10));
  DGRP_CUDA(cudaMemcpyAsync(tr->keep.p, keep, (size_t)n * 10, cudaMemcpyHostToDevice, c->stream));
  DGRP_CHECK(train_run_step(c, tr, n, tr->starts.as<int64_t>(), tr->keep.as<uint8_t>()));
  tr->h_lpart.resize((size_t)n);
  DGRP_CUDA(cudaMemcpyAsync(tr->h_lpart.data(), tr->lpart.p, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost,
                            c->stream));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  if (loss) *loss = train_mean_loss(tr->h_lpart, n, tr->T);
  return DGRP_OK;
}

int dgrp_train_eval(dgrp_trainer *tr, int which, const int64_t *starts, int64_t n, float *loss, float *probs) {
  dgrp_ctx *c = tr->ctx;
  Use use(c->device);
  DGRP_CHECK(train_upload_starts(tr, which, starts, n));
  float *d_probs = nullptr;
  if (probs) {
    DGRP_CHECK(tr->probs.reserve((size_t)n * tr->T * tr->C * sizeof(float)));
    d_probs = tr->probs.as<float>();
  }
  tr->h_lpart.resize((size_t)n);
  DGRP_CHECK(train_run_eval(c, tr, which, n, tr->starts.as<int64_t>(), d_probs, tr->h_lpart.data()));
  if (probs)
    DGRP_CUDA(cudaMemcpyAsync(probs, d_probs, (size_t)n * tr->T * tr->C * sizeof(float), cudaMemcpyDeviceToHost,
                              c->stream));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  if (loss) *loss = train_mean_loss(tr->h_lpart, n, tr->T);
  return DGRP_OK;
}

int dgrp_train_get_weights(dgrp_trainer *tr, float *kernel, float *recurrent, float *bias, float *att_scale,
                           float *ff_kernel, float *ff_bias) {
  Use use(tr->ctx->device);
  return train_unpack(tr, tr->w, kernel, recurrent, bias, att_scale, ff_kernel, ff_bias);
}

int dgrp_train_get_grads(dgrp_trainer *tr, float *kernel, float *recurrent, float *bias, float *att_scale,
                         float *ff_kernel, float *ff_bias) {
  Use use(tr->ctx->device);
  return train_unpack(tr, tr->g, kernel, recurrent, bias, att_scale, ff_kernel, ff_bias);
}

int dgrp_train_timings(dgrp_trainer *tr, float *out5) {
  Use use(tr->ctx->device);
  DGRP_REQUIRE(tr->timed, "no training step has run");
  DGRP_CUDA(cudaEventSynchronize(tr->ev[5]));
  for (int i = 0; i < 5; ++i) DGRP_CUDA(cudaEventElapsedTime(&out5[i], tr->ev[i], tr->ev[i + 1]));
  return DGRP_OK;
}

int dgrp_train_destroy(dgrp_trainer *tr) {
  if (!tr) return DGRP_OK;
  Use use(tr->ctx->device);
  cudaStreamSynchronize(tr->ctx->stream);
  DevBuf *bufs[] = {&tr->w, &tr->g, &tr->s1, &tr->s2, &tr->codes[0], &tr->codes[1], &tr->ymask[0], &tr->ymask[1],
                    &tr->starts, &tr->keep, &tr->Hs, &tr->GS, &tr->D, &tr->avg, &tr->dhin, &tr->hpart,
                    &tr->rpart, &tr->lpart, &tr->probs};
  for (auto b : bufs) b->release();
  for (auto &e : tr->ev)
    if (e) cudaEventDestroy(e);
  delete tr;
  return DGRP_OK;
}

}  // extern "C"

// positions [pos0, pos1) of a record from device codes: label + score into device buffers
static int core_predict_range(dgrp_ctx *c, dgrp_model *m, const uint8_t *d_codes, int64_t codes_base,
                              int64_t codes_len, int64_t length, int64_t pos0, int64_t pos1, int step,
                              int batch_size, int compat, uint8_t *d_labels, float *d_scores) {
  DGRP_REQUIRE(0 <= pos0 && pos0 <= pos1 && pos1 <= length, "bad range [%lld, %lld) of %lld",
               (long long)pos0, (long long)pos1, (long long)length);
  DGRP_REQUIRE(step > 0, "step_size must be positive");
  const int64_t rows = pos1 - pos0;
  if (rows == 0) return DGRP_OK;
  const Placement pl = make_placement(length, m->T, step, batch_size, compat);
  const int T = m->T;
  // windows whose PLACED rows [place, place+T) intersect [pos0, pos1)
  auto range_for = [&](int64_t w_lo, int64_t w_hi, int64_t base, int64_t *b, int64_t *e) {
    // window w (w_lo <= w < w_hi) is placed at base + (w - w_lo) * step
    int64_t first = 0, last = w_hi - w_lo;  // local indices
    if (pos0 - T + 1 - base > 0) first = (pos0 - T + 1 - base + step - 1) / step;
    if (pos1 - base <= 0) last = 0;
    else last = std::min<int64_t>(last, (pos1 - 1 - base) / step + 1);
    if (first > last) first = last;
    *b = w_lo + first; *e = w_lo + last;
  };
  int64_t a0, a1, t0, t1;
  range_for(0, pl.full_windows, 0, &a0, &a1);
  range_for(pl.full_windows, pl.n_windows, pl.tail_base, &t0, &t1);
  // codes needed: true window positions [w*step, w*step + T)
  int64_t need_lo = length, need_hi = 0;
  if (a1 > a0) { need_lo = std::min(need_lo, a0 * step); need_hi = std::max(need_hi, (a1 - 1) * step + T); }
  if (t1 > t0) { need_lo = std::min(need_lo, t0 * step); need_hi = std::max(need_hi, (t1 - 1) * step + T); }
  if (need_hi > need_lo)
    DGRP_REQUIRE(codes_base <= need_lo && need_hi <= codes_base + codes_len,
                 "codes [%lld, %lld) do not cover the needed bases [%lld, %lld)", (long long)codes_base,
                 (long long)(codes_base + codes_len), (long long)need_lo, (long long)need_hi);
  c->timings.windows = (a1 - a0) + (t1 - t0);
  c->timings.bases = rows;
  DGRP_CHECK(c->pred.reserve((size_t)rows * m->C * 4));
  DGRP_CUDA(cudaMemsetAsync(c->pred.p, 0, (size_t)rows * m->C * 4, c->stream));
  DGRP_CHECK(run_forward_vote(c, m, d_codes, codes_base, a0, a1, pl, c->pred.as<float>(), pos0, rows, nullptr, nullptr,
                              nullptr, t0, t1));
  return launch_score(c, c->pred.as<float>(), rows, m->C, d_labels, d_scores, nullptr, nullptr);
}

extern "C" {

int dgrp_predict_range(dgrp_ctx *c, dgrp_model *m, const uint8_t *codes, int64_t codes_base,
                       int64_t codes_len, int64_t length, int64_t pos0, int64_t pos1, int step,
                       int batch_size, int compat, uint8_t *labels, float *scores) {
  Use use(c->device);
  DGRP_REQUIRE(0 <= pos0 && pos0 <= pos1 && pos1 <= length, "bad range [%lld, %lld) of %lld",
               (long long)pos0, (long long)pos1, (long long)length);
  const int64_t rows = pos1 - pos0;
  if (rows == 0) return DGRP_OK;
  DGRP_CHECK(c->codes.reserve((size_t)codes_len + 16));
  DGRP_CUDA(cudaMemcpyAsync(c->codes.p, codes, (size_t)codes_len, cudaMemcpyHostToDevice, c->stream));
  DGRP_CHECK(c->labels.reserve((size_t)rows));
  DGRP_CHECK(c->scores32.reserve((size_t)rows * 4));
  DGRP_CHECK(core_predict_range(c, m, c->codes.as<uint8_t>(), codes_base, codes_len, length, pos0, pos1, step,
                                batch_size, compat, c->labels.as<uint8_t>(), c->scores32.as<float>()));
  if (labels) DGRP_CUDA(cudaMemcpyAsync(labels, c->labels.p, (size_t)rows, cudaMemcpyDeviceToHost, c->stream));
  if (scores) DGRP_CUDA(cudaMemcpyAsync(scores, c->scores32.p, (size_t)rows * 4, cudaMemcpyDeviceToHost, c->stream));
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  return DGRP_OK;
}

int dgrp_predict_range_dev(dgrp_ctx *c, dgrp_model *m, const uint8_t *d_codes, int64_t codes_base,
                           int64_t codes_len, int64_t length, int64_t pos0, int64_t pos1, int step,
                           int batch_size, int compat, uint8_t *d_labels, float *d_scores) {
  Use use(c->device);
  const int64_t launches0 = c->launches;
  stamp(c, 0);
  stamp(c, 1);
  const int rc = core_predict_range(c, m, d_codes, codes_base, codes_len, length, pos0, pos1, step, batch_size,
                                    compat, d_labels, d_scores);
  stamp(c, 2); stamp(c, 3); stamp(c, 4); stamp(c, 5);
  finish_timings(c, launches0);
  return rc;
}

int dgrp_finish_record(dgrp_ctx *c, const uint8_t *labels, const float *scores, int64_t length,
                       int n_classes, int use_mss, int min_mss_len, int xdrop_len, int64_t startpos,
                       uint8_t *labels_out, dgrp_row_t *rows, int64_t cap, int64_t *n_rows) {
  Use use(c->device);
  *n_rows = 0;
  if (length <= 0) return DGRP_OK;
  DGRP_CHECK(c->labels.reserve((size_t)length));
  DGRP_CHECK(c->scores32.reserve((size_t)length * 4));
  DGRP_CUDA(cudaMemcpyAsync(c->labels.p, labels, (size_t)length, cudaMemcpyHostToDevice, c->stream));
  if (use_mss)
    DGRP_CUDA(cudaMemcpyAsync(c->scores32.p, scores, (size_t)length * 4, cudaMemcpyHostToDevice, c->stream));
  DGRP_CHECK(core_labels(c, nullptr, c->labels.as<uint8_t>(), c->scores32.as<float>(), length,
                         n_classes, use_mss, min_mss_len, xdrop_len));
  if (labels_out)
    DGRP_CUDA(cudaMemcpyAsync(labels_out, c->labels2.p, (size_t)length, cudaMemcpyDeviceToHost, c->stream));
  const int rc = core_rows(c, length, startpos, 0, true, rows, cap, n_rows);
  DGRP_CUDA(cudaStreamSynchronize(c->stream));
  return rc;
}

int dgrp_finish_record_dev(dgrp_ctx *c, const uint8_t *d_labels, const float *d_scores, int64_t length,
                           int n_classes, int use_mss, int min_mss_len, int xdrop_len, int64_t *n_rows) {
  Use use(c->device);
  const int64_t launches0 = c->launches;
  *n_rows = 0;
  stamp(c, 0); stamp(c, 1); stamp(c, 2);
  DGRP_CHECK(core_labels(c, nullptr, d_labels, d_scores, length, n_classes, use_mss, min_mss_len, xdrop_len));
  stamp(c, 4);
  int rc = DGRP_OK;
  if (length > 0) rc = core_rows(c, length, 0, 0, false, nullptr, 0, n_rows);
  stamp(c, 5);
  finish_timings(c, launches0);
  return rc;
}

}  // extern "C"

/* ------------------------- streaming whole-file driver (pipelined) ------------------------- */
// deepgrp/__main__.py:275-295 reads a file record by record and writes a record's rows as soon as the record is
// done.  dgrp_fasta_stream does the same as a three-stage pipeline with bounded memory:
//   compute thread  cuts the text into slices at header lines (host memchr index), uploads ONLY this rank's
//                   slices (pinned staging ring, one cudaMemcpyAsync per chunk, a stream of its own), decodes a
//                   slice on the GPU and runs encode -> forward -> MSS -> segments -> TSV text per record; the
//                   text of a record lands in one of two device buffers;
//   copier thread   moves a finished record's text to the host in pieces through a ring of pinned slots on a
//                   third stream, while the compute thread is already on the next record;
//   caller          dgrp_fasta_stream_next() hands out one piece at a time (valid until the next call).
namespace {

constexpr int kSlots = 4;
constexpr int64_t kSlotBytesDefault = (int64_t)64 << 20;    // one piece of TSV text ("stream_slot_mb")
constexpr int64_t kStageBytes = (int64_t)32 << 20;   // one chunk of the upload
constexpr int64_t kMinSlice = (int64_t)8 << 20;      // adjacent records are merged into slices of at least this size

struct StreamPiece {
  int slot;
  int64_t bytes, slice, ordinal, rows;
  int last;   // last piece of its record
};
struct StreamRecord {
  int buf;    // device text buffer
  int64_t bytes, slice, ordinal, rows;
  int final_part;   // 0: rows of a record that is still being computed ("early rows"), more text follows
};

}  // namespace

struct dgrp_fasta_stream {
  dgrp_ctx *c = nullptr;
  dgrp_model *m = nullptr;
  const uint8_t *fasta = nullptr;
  int64_t nbytes = 0;
  std::string filename;
  int step = 0, batch_size = 0, use_mss = 0, min_mss_len = 0, xdrop_len = 0, compat = 0;
  std::vector<int64_t> cuts;     // slice k = [cuts[k], cuts[k + 1])
  std::vector<int64_t> mine;     // this rank's slices, in file order
  DevBuf *raw = nullptr, *text = nullptr;     // [2] each; the buffers live in the context and are reused by the next stream
  PinBuf *stage = nullptr, *slot = nullptr;   // [2], [kSlots]
  cudaStream_t s_in = nullptr, s_out = nullptr;
  cudaEvent_t ev_in[2] = {}, ev_stage[2] = {}, ev_text[2] = {}, ev_slot[kSlots] = {};
  bool src_pinned = false;
  int64_t slot_bytes = kSlotBytesDefault;
  std::thread compute, copier, uploader;
  int up_done = 0, dec_done = 0;    // slices (of `mine`) whose upload has been enqueued / that have been decoded
  int up_rc = DGRP_OK;
  std::string up_err;
  std::mutex mu;
  std::condition_variable cv;
  std::deque<StreamRecord> ready;   // compute -> copier
  std::deque<StreamPiece> pieces;   // copier -> caller
  int text_busy[2] = {0, 0};        // device text buffer handed to the copier
  int slot_state[kSlots] = {};      // 0 free, 1 being filled / queued, 2 held by the caller
  int held = -1;
  bool compute_done = false, copier_done = false, cancel = false, cancel_upload = false;
  int rc = DGRP_OK;
  std::string err;
  // totals
  int64_t rows = 0, records = 0, bases = 0, windows = 0, launches = 0, h2d_bytes = 0, d2h_bytes = 0;
  double forward_ms = 0.0, gpu_ms = 0.0;
  // where the threads waited, ms: [0] compute for the upload, [1] compute for a free text buffer, [2] copier for a
  // finished record, [3] copier for a free slot, [4] copier in event waits (the copies), [5] uploader for a free raw
  // buffer, [6] uploader in memcpy + enqueue, [7] compute thread total
  double waits[12] = {};   // [8] slice decode, [9] records (host wall), [10] TSV measure + write enqueue, [11] encode
};

namespace {

struct WaitClock {   // adds the scope's wall time to a counter
  double &acc;
  std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
  explicit WaitClock(double &a) : acc(a) {}
  ~WaitClock() { acc += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); }
};

// Header lines start a slice: a '>' that is the first byte of a line.  (A '>' after leading whitespace is a
// header too, __main__.py:34-35; it simply stays inside the preceding slice, which the GPU parser handles.)
// slices [cuts[k], cuts[k+1]) of the text and their owners; pure host code (also exported as dgrp_fasta_index)
void index_slices(const uint8_t *f, int64_t n, int world, std::vector<int64_t> &cuts, std::vector<int> &owner) {
  // candidate header positions: '>' right after a line terminator; found by memchr, in parallel for large inputs
  // (a 3 GB genome is 0.15 s of single-threaded scanning per rank otherwise)
  const int nt = n > ((int64_t)64 << 20) ? 8 : (n > ((int64_t)8 << 20) ? 4 : 1);
  std::vector<std::vector<int64_t>> found(nt);
  auto scan = [&](int t) {
    int64_t p = std::max<int64_t>(1, n * t / nt);
    const int64_t end = n * (t + 1) / nt;
    while (p < end) {
      const void *q = memchr(f + p, '>', (size_t)(end - p));
      if (!q) break;
      p = (const uint8_t *)q - f;
      if (f[p - 1] == '\n' || f[p - 1] == '\r') found[t].push_back(p);
      ++p;
    }
  };
  if (nt == 1) scan(0);
  else {
    std::vector<std::thread> th;
    for (int t = 0; t < nt; ++t) th.emplace_back(scan, t);
    for (auto &x : th) x.join();
  }
  cuts.clear();
  cuts.push_back(0);
  for (int t = 0; t < nt; ++t)
    for (int64_t p : found[t])
      if (p - cuts.back() >= kMinSlice) cuts.push_back(p);
  cuts.push_back(n);
  // largest-first assignment of slices to ranks (every rank derives the same table)
  const int64_t ns = (int64_t)cuts.size() - 1;
  if (world < 1) world = 1;
  std::vector<int64_t> order(ns);
  for (int64_t k = 0; k < ns; ++k) order[k] = k;
  std::stable_sort(order.begin(), order.end(), [&](int64_t a, int64_t b) {
    return (cuts[a + 1] - cuts[a]) > (cuts[b + 1] - cuts[b]);
  });
  std::vector<int64_t> load(world, 0);
  owner.assign(ns, 0);
  for (int64_t k : order) {
    int best = 0;
    for (int r = 1; r < world; ++r)
      if (load[r] < load[best]) best = r;
    owner[k] = best;
    load[best] += cuts[k + 1] - cuts[k];
  }
}

void stream_index(dgrp_fasta_stream *s) {
  std::vector<int> owner;
  index_slices(s->fasta, s->nbytes, s->c->shard_world, s->cuts, owner);
  s->mine.clear();
  for (int64_t k = 0; k + 1 < (int64_t)s->cuts.size(); ++k)
    if (owner[k] == s->c->shard_rank && s->cuts[k + 1] > s->cuts[k]) s->mine.push_back(k);
}

#define STREAM_CUDA(call)                                                                     \
  do {                                                                                        \
    cudaError_t e__ = (call);                                                                 \
    if (e__ != cudaSuccess) {                                                                 \
      dgrp::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
      return DGRP_E_CUDA;                                                                     \
    }                                                                                         \
  } while (0)

// enqueue the upload of slice `k` into raw[b] on s_in and record ev_in[b]
int stream_upload(dgrp_fasta_stream *s, int64_t k, int b, int *stage_turn) {
  const int64_t off = s->cuts[k], n = s->cuts[k + 1] - off;
  DGRP_CHECK(s->raw[b].reserve((size_t)n + 16));
  if (s->src_pinned) {
    STREAM_CUDA(cudaMemcpyAsync(s->raw[b].p, s->fasta + off, (size_t)n, cudaMemcpyHostToDevice, s->s_in));
  } else {
    for (int64_t o = 0; o < n; o += kStageBytes) {
      const int t = (*stage_turn)++ & 1;
      const int64_t len = std::min<int64_t>(kStageBytes, n - o);
      STREAM_CUDA(cudaEventSynchronize(s->ev_stage[t]));   // the chunk that used this staging buffer has left
      memcpy(s->stage[t].p, s->fasta + off + o, (size_t)len);
      STREAM_CUDA(cudaMemcpyAsync(s->raw[b].as<uint8_t>() + o, s->stage[t].p, (size_t)len, cudaMemcpyHostToDevice, s->s_in));
      STREAM_CUDA(cudaEventRecord(s->ev_stage[t], s->s_in));
    }
  }
  s->h2d_bytes += n;
  STREAM_CUDA(cudaEventRecord(s->ev_in[b], s->s_in));
  return DGRP_OK;
}

// Slab ends (positions) of a long record for the early-rows route; fewer than two = not worth it.  A slab is a
// whole number of forward "units" (unit_w windows = one round of two tiles on every SM) minus the halo windows a
// position range recomputes, so that the persistent kernel's CTAs get equal tile counts.  The slabs shrink
// geometrically (ratio_pct per cent each) because only the LAST slab's text cannot overlap any compute; the default
// (6 slabs, 80 %: 27 / 22 / 17 / 14 / 11 / 9 % of the record) also keeps the FIRST slab small, so that the copies
// start early where several ranks share one host's memory and a rank's text takes as long as its forward
// (DESIGN.md section 6); on one GPU it measures the same as 4 slabs at 55 % (profiles/r02s2_summary.md).
void plan_slabs(int64_t length, int T, int step, int64_t unit_w, int n_slabs, int ratio_pct,
                std::vector<int64_t> &ends) {
  ends.clear();
  if (step <= 0 || unit_w <= 0) return;
  const double K = (double)(length / step) / (double)unit_w;   // units in the record
  int n = n_slabs;
  if ((double)n > K / 2.0) n = (int)(K / 2.0);
  if (n < 2) return;
  const double ratio = (ratio_pct > 0 && ratio_pct <= 100 ? ratio_pct : 80) / 100.0;
  double wsum = 0.0, w = 1.0;
  for (int i = 0; i < n; ++i) { wsum += w; w *= ratio; }
  const int64_t halo = (T + step - 1) / step + 8;
  auto rows_of = [&](int64_t k) {
    int64_t rows = (k * unit_w - halo) * step;
    if (rows <= 0) rows = k * unit_w * step;
    if (rows > 64) rows &= ~(int64_t)63;
    return rows;
  };
  int64_t pos = 0;
  w = 1.0;
  for (int i = 0; i + 1 < n; ++i, w *= ratio) {
    int64_t k = (int64_t)(w / wsum * K + 0.5);
    if (k < 1) k = 1;
    const int64_t rows = rows_of(k);
    if (pos + rows + unit_w * step >= length) break;
    pos += rows;
    ends.push_back(pos);
  }
  ends.push_back(length);
}

// one slice (already on the device in raw[b]): decode, then every record of it
int stream_slice(dgrp_fasta_stream *s, int64_t k, int b, int *text_turn, bool last_slice) {
  dgrp_ctx *c = s->c;
  dgrp_model *m = s->m;
  const uint8_t *fasta = s->fasta + s->cuts[k];          // host view of the slice (headers)
  const int64_t nbytes = s->cuts[k + 1] - s->cuts[k];
  STREAM_CUDA(cudaStreamWaitEvent(c->stream, s->ev_in[b], 0));
  int64_t n_seq = 0, n_hdr = 0;
  int drc;
  {
    WaitClock wc(s->waits[8]);
    drc = run_fasta_decode(c, s->raw[b].as<uint8_t>(), nbytes, &n_seq, &n_hdr);
  }
  {
    std::lock_guard<std::mutex> lk(s->mu);   // the raw bytes have been consumed (the decode synchronises)
    s->dec_done += 1;
  }
  s->cv.notify_all();
  DGRP_CHECK(drc);
  std::vector<int64_t> hpos(n_hdr), hseq(n_hdr + 1);
  if (n_hdr > 0) {
    const int64_t *t = c->pin_b.as<int64_t>();
    for (int64_t i = 0; i < n_hdr; ++i) { hpos[i] = t[i]; hseq[i] = t[(n_hdr + 1) + i]; }
  }
  hseq[n_hdr] = n_seq;
  auto ws = [](uint8_t x) { return (x >= 9 && x <= 13) || (x >= 28 && x <= 32); };
  int64_t ordinal = 0;
  for (int64_t i = 0; i < n_hdr; ++i) {
    {
      std::lock_guard<std::mutex> lk(s->mu);
      if (s->cancel) return DGRP_OK;
    }
    int64_t hb = hpos[i] + 1, he = hb;
    while (he < nbytes && fasta[he] != '\n' && !(fasta[he] == '\r' && !(he + 1 < nbytes && fasta[he + 1] == '\n'))) ++he;
    while (he > hb && ws(fasta[he - 1])) --he;
    if (he == hb) continue;                         // empty header: record dropped (__main__.py:36)
    const uint8_t *d_seq = c->io_b.as<uint8_t>() + hseq[i];
    const int64_t n = hseq[i + 1] - hseq[i];
    int64_t startpos = 0, length = 0;
    WaitClock wrec(s->waits[9]);
    stamp(c, 0);
    {
      WaitClock wc(s->waits[11]);
      DGRP_CHECK(core_encode(c, d_seq, n, 1, &startpos, &length));
    }
    if (length < 0) {
      set_error("negative dimensions are not allowed (all-'N' record in slice %lld)", (long long)k);
      return DGRP_E_ALLN;
    }
    s->bases += length;
    std::string prefix(s->filename);
    prefix.push_back('\t');
    prefix.append(reinterpret_cast<const char *>(fasta + hb), (size_t)(he - hb));
    prefix.push_back('\t');
    bool prefix_up = false;
    bool cancelled = false;
    // rows (device triples) -> TSV text in one of the two device text buffers -> the copier.  final_part = 0: rows of
    // a record whose later positions are still being computed; its text travels like a record's, without the
    // end-of-record mark.  Synchronises the stream.
    auto emit = [&](const int64_t *d_tri, int64_t cnt, int final_part) -> int {
      int64_t need = 0;
      int tb = -1;
      if (cnt > 0) {
        WaitClock wc(s->waits[10]);
        if (!prefix_up) {
          DGRP_CHECK(c->tsv_prefix.reserve(prefix.size() + 16));
          STREAM_CUDA(cudaMemcpyAsync(c->tsv_prefix.p, prefix.data(), prefix.size(), cudaMemcpyHostToDevice, c->stream));
          prefix_up = true;
        }
        DGRP_CHECK(run_tsv_measure(c, d_tri, cnt, (int)prefix.size(), &need));   // syncs
        tb = (*text_turn)++ & 1;
        {
          WaitClock wc1(s->waits[1]);
          std::unique_lock<std::mutex> lk(s->mu);   // the copier still drains the text before last
          s->cv.wait(lk, [&] { return s->text_busy[tb] == 0 || s->cancel; });
          if (s->cancel) { cancelled = true; return DGRP_OK; }
        }
        DGRP_CHECK(s->text[tb].reserve((size_t)need + 16));
        DGRP_CHECK(run_tsv_write(c, d_tri, cnt, c->tsv_prefix.as<uint8_t>(), (int)prefix.size(),
                                 s->text[tb].as<uint8_t>()));
        STREAM_CUDA(cudaEventRecord(s->ev_text[tb], c->stream));
      }
      if (final_part) stamp(c, 5);
      STREAM_CUDA(cudaStreamSynchronize(c->stream));
      s->rows += cnt;
      if (cnt > 0 || final_part) {
        std::lock_guard<std::mutex> lk(s->mu);
        if (tb >= 0) s->text_busy[tb] = 1;
        s->ready.push_back(StreamRecord{tb, need, k, ordinal, cnt, final_part});   // records without rows travel as empty pieces
      }
      s->cv.notify_all();
      return DGRP_OK;
    };
    // Long records with MSS: positions in slabs, see stream_record_slabs
    std::vector<int64_t> slab_end;
    // (by default only for the rank's LAST record: the text of every other record crosses PCIe under the next
    // record's forward anyway, and the slabs cost a few per cent of kernel efficiency; 2 = every long record)
    if (s->use_mss && length > 0 &&
        (c->stream_early_rows >= 2 || (c->stream_early_rows == 1 && last_slice && i + 1 == n_hdr)))
      plan_slabs(length, m->T, s->step, c->stream_early_unit > 0 ? c->stream_early_unit : (int64_t)c->sm_count * 128,
                 c->stream_early_slabs > 0 ? c->stream_early_slabs : 6, c->stream_early_ratio, slab_end);
    c->stream_early_parts = 0;
    float ms = 0.f;
    if (slab_end.size() >= 2) {
      // "Early rows".  MSS needs the whole record before the LAST candidate is final, but not before the first:
      // whenever a run of positive scores finds no candidate with a smaller running sum the reference flushes its
      // stack (mss.c:78-81) and nothing before that run can change any more.  The record is computed in position
      // slabs (halo recompute, as for chunk sharding); after each slab MSS runs over [restart, slab end) from the
      // carried running sum, the part before the last flush is gap-filled, cut into rows and formatted, and its
      // text crosses PCIe while the next slab's forward runs.  Scores that drift upwards never flush: the first
      // slab that makes little progress ends the probing and the record finishes as a whole.  Identical rows
      // either way (tests/test_gpu_stream.py; the resumed scan is pinned on the CPU in tests/test_host.py).
      DGRP_CHECK(c->labels.reserve((size_t)length));
      DGRP_CHECK(c->scores32.reserve((size_t)length * 4));
      DGRP_CHECK(c->labels2.reserve((size_t)length));
      DGRP_REQUIRE(length < 2147483647LL, "record longer than 2^31-1 bases (int indices in mss.h:16)");
      uint8_t *lab = c->labels.as<uint8_t>(), *lab2 = c->labels2.as<uint8_t>();
      float *sc = c->scores32.as<float>();
      double min_sc, xdrop;
      mss_thresholds(s->min_mss_len, s->xdrop_len, &min_sc, &xdrop);
      int64_t p0 = 0, r = 0, e = 0;   // slab start; MSS resumes at r (running sum L0); rows are out up to e
      double L0 = 0.0;
      bool probing = true;
      for (size_t q = 0; q < slab_end.size() && !cancelled; ++q) {
        const int64_t p1 = slab_end[q];
        const bool last = q + 1 == slab_end.size();
        stamp(c, 1);
        DGRP_CHECK(core_predict_range(c, m, c->codes.as<uint8_t>(), 0, length, length, p0, p1, s->step, s->batch_size,
                                      s->compat, lab + p0, sc + p0));
        stamp(c, 2);
        s->windows += c->timings.windows;
        p0 = p1;
        dgrp_seg_t *d_segs = nullptr;
        int n_seg = 0;
        int64_t *d_tri = nullptr;
        int64_t cnt = 0;
        if (last) {
          DGRP_CHECK(run_mss_segments(c, nullptr, sc + r, (int)(length - r), min_sc, xdrop, &d_segs, &n_seg, L0, nullptr));
          DGRP_CHECK(run_gap_fill(c, d_segs, n_seg, lab + r, nullptr, (int)(length - r), m->C, lab2 + r));
          stamp(c, 4);
          DGRP_CHECK(run_segments(c, lab2 + e, nullptr, length - e, startpos + e, false, &d_tri, &cnt));
          DGRP_CHECK(emit(d_tri, cnt, 1));
        } else if (probing) {
          if (q == 0) {
            // Which way do the scores drift?  Upwards (confident class-0 calls score positive: the x4 weight set,
            // config 5b) the running sum keeps rising, no run ever finds the stack without a smaller L and
            // nothing is final before the record ends: the MSS pass over the slab would be wasted (it is the
            // expensive rounding regime, too), so the rest of the record runs as one call.
            DGRP_CHECK(c->small.reserve(256));
            DGRP_CHECK(c->pin_small.reserve(256));
            double *d_sum = reinterpret_cast<double *>(c->small.as<unsigned char>() + 192);
            STREAM_CUDA(cudaMemsetAsync(d_sum, 0, 8, c->stream));
            score_drift_kernel<<<c->sm_count * 8, 256, 0, c->stream>>>(sc, p1, d_sum);
            c->launches++;
            double *h_sum = reinterpret_cast<double *>(c->pin_small.as<unsigned char>() + 96);
            DGRP_CHECK(fetch_small(c, h_sum, d_sum, 8));
            STREAM_CUDA(cudaStreamSynchronize(c->stream));
            if (*h_sum > 0.0) probing = false;
          }
        }
        if (!last && probing) {
          MssResume rs;
          DGRP_CHECK(run_mss_segments(c, nullptr, sc + r, (int)(p1 - r), min_sc, xdrop, &d_segs, &n_seg, L0, &rs));
          if (rs.restart > 0) {
            DGRP_CHECK(run_gap_fill(c, d_segs, n_seg, lab + r, nullptr, rs.restart, m->C, lab2 + r));
            if (rs.restart < (p1 - r) / 2) probing = false;
            r += rs.restart;
            L0 = rs.L0;
            int64_t tail = 0;
            DGRP_CHECK(run_segments(c, lab2 + e, nullptr, r - e, startpos + e, false, &d_tri, &cnt, &tail));
            e += tail;
            DGRP_CHECK(emit(d_tri, cnt, 0));
            if (cnt > 0) c->stream_early_parts += 1;
          } else {
            probing = false;
          }
        }
        STREAM_CUDA(cudaEventSynchronize(c->ev[2]));
        cudaEventElapsedTime(&ms, c->ev[1], c->ev[2]); s->forward_ms += ms;
        // nothing (more) to gain from slabs: the rest of the record in one call
        if (!probing && q + 2 < slab_end.size()) slab_end.erase(slab_end.begin() + (q + 1), slab_end.end() - 1);
      }
      if (cancelled) return DGRP_OK;
    } else {
      stamp(c, 1);
      DGRP_CHECK(core_predict(c, m, c->codes.as<uint8_t>(), length, s->step, s->batch_size, s->compat, s->use_mss != 0));
      s->windows += c->timings.windows;
      stamp(c, 2);
      DGRP_CHECK(core_labels_after_predict(c, length, m->C, s->use_mss, s->min_mss_len, s->xdrop_len));
      stamp(c, 4);
      int64_t cnt = 0;
      int64_t *d_tri = nullptr;
      if (length > 0) DGRP_CHECK(run_segments(c, c->labels2.as<uint8_t>(), nullptr, length, startpos, false, &d_tri, &cnt));
      DGRP_CHECK(emit(d_tri, cnt, 1));
      if (cancelled) return DGRP_OK;
      cudaEventElapsedTime(&ms, c->ev[1], c->ev[2]); s->forward_ms += ms;
    }
    cudaEventElapsedTime(&ms, c->ev[0], c->ev[5]); s->gpu_ms += ms;
    s->records += 1;
    ++ordinal;
  }
  return DGRP_OK;
}

// The upload runs ahead of the compute thread by one slice: the staging memcpy (page faults of a mapped file
// included) overlaps the GPU work on the slice before.
void stream_uploader_main(dgrp_fasta_stream *s) {
  cudaSetDevice(s->c->device);
  int stage_turn = 0, rc = DGRP_OK;
  for (size_t i = 0; i < s->mine.size() && rc == DGRP_OK; ++i) {
    {
      WaitClock wc(s->waits[5]);
      std::unique_lock<std::mutex> lk(s->mu);   // raw[i & 1] is free once slice i - 2 has been decoded
      s->cv.wait(lk, [&] { return (int)i < s->dec_done + 2 || s->cancel || s->cancel_upload; });
      if (s->cancel || s->cancel_upload) break;
    }
    {
      WaitClock wc(s->waits[6]);
      rc = stream_upload(s, s->mine[i], (int)(i & 1), &stage_turn);
    }
    {
      std::lock_guard<std::mutex> lk(s->mu);
      if (rc != DGRP_OK) { s->up_rc = rc; s->up_err = dgrp_last_error(); }
      s->up_done = (int)i + 1;
    }
    s->cv.notify_all();
  }
}

void stream_compute_main(dgrp_fasta_stream *s) {
  cudaSetDevice(s->c->device);
  const int64_t launches0 = s->c->launches;
  int rc = DGRP_OK, text_turn = 0;
  WaitClock total(s->waits[7]);
  for (size_t i = 0; i < s->mine.size() && rc == DGRP_OK; ++i) {
    {
      WaitClock wc(s->waits[0]);
      std::unique_lock<std::mutex> lk(s->mu);
      s->cv.wait(lk, [&] { return s->up_done > (int)i || s->cancel; });
      if (s->cancel) break;
      if (s->up_rc != DGRP_OK) { rc = s->up_rc; set_error("%s", s->up_err.c_str()); break; }
    }
    rc = stream_slice(s, s->mine[i], (int)(i & 1), &text_turn, i + 1 == s->mine.size());
    std::lock_guard<std::mutex> lk(s->mu);
    if (s->cancel) break;
  }
  s->launches = s->c->launches - launches0;
  {
    std::lock_guard<std::mutex> lk(s->mu);
    if (rc != DGRP_OK) { s->rc = rc; s->err = dgrp_last_error(); s->cancel_upload = true; }
    s->compute_done = true;
  }
  s->cv.notify_all();
}

void stream_copier_main(dgrp_fasta_stream *s) {
  cudaSetDevice(s->c->device);
  std::deque<StreamPiece> inflight;
  auto publish_oldest = [&]() {
    StreamPiece p = inflight.front();
    inflight.pop_front();
    if (p.slot >= 0) { WaitClock wc(s->waits[4]); cudaEventSynchronize(s->ev_slot[p.slot]); }
    {
      std::lock_guard<std::mutex> lk(s->mu);
      s->pieces.push_back(p);
    }
    s->cv.notify_all();
  };
  for (;;) {
    StreamRecord r;
    {
      WaitClock wc(s->waits[2]);
      std::unique_lock<std::mutex> lk(s->mu);
      s->cv.wait(lk, [&] { return !s->ready.empty() || s->compute_done || s->cancel; });
      if (s->cancel) break;
      if (s->ready.empty()) break;   // compute finished and everything is copied
      r = s->ready.front();
      s->ready.pop_front();
    }
    if (r.buf < 0 || r.bytes == 0) {   // a record without rows
      inflight.push_back(StreamPiece{-1, 0, r.slice, r.ordinal, r.rows, r.final_part});
      while (!inflight.empty()) publish_oldest();
      continue;
    }
    cudaStreamWaitEvent(s->s_out, s->ev_text[r.buf], 0);
    bool stop = false;
    for (int64_t off = 0; off < r.bytes && !stop; off += s->slot_bytes) {
      const int64_t len = std::min<int64_t>(s->slot_bytes, r.bytes - off);
      int slot = -1;
      for (;;) {
        {
          std::lock_guard<std::mutex> lk(s->mu);
          if (s->cancel) { stop = true; break; }
          for (int q = 0; q < kSlots; ++q)
            if (s->slot_state[q] == 0) { slot = q; s->slot_state[q] = 1; break; }
        }
        if (slot >= 0) break;
        if (!inflight.empty()) { publish_oldest(); continue; }   // the caller needs something to release
        WaitClock wc(s->waits[3]);
        std::unique_lock<std::mutex> lk(s->mu);
        s->cv.wait(lk, [&] {
          if (s->cancel) return true;
          for (int q = 0; q < kSlots; ++q) if (s->slot_state[q] == 0) return true;
          return false;
        });
      }
      if (stop) break;
      cudaMemcpyAsync(s->slot[slot].p, s->text[r.buf].as<uint8_t>() + off, (size_t)len, cudaMemcpyDeviceToHost, s->s_out);
      cudaEventRecord(s->ev_slot[slot], s->s_out);
      s->d2h_bytes += len;
      inflight.push_back(StreamPiece{slot, len, r.slice, r.ordinal, off + len >= r.bytes ? r.rows : 0,
                                     (off + len >= r.bytes && r.final_part) ? 1 : 0});
      if ((int)inflight.size() >= kSlots - 1) publish_oldest();
    }
    while (!inflight.empty()) publish_oldest();   // the record's last copy has completed: its device buffer is free
    {
      std::lock_guard<std::mutex> lk(s->mu);
      s->text_busy[r.buf] = 0;
    }
    s->cv.notify_all();
    if (stop) break;
  }
  {
    std::lock_guard<std::mutex> lk(s->mu);
    s->copier_done = true;
  }
  s->cv.notify_all();
}

}  // namespace

extern "C" {

int dgrp_fasta_index(const uint8_t *fasta, int64_t nbytes, int world, int64_t *cuts, int32_t *owner, int64_t cap,
                     int64_t *n_slices) {
  std::vector<int64_t> cv;
  std::vector<int> ov;
  if (nbytes < 0 || !n_slices) { set_error("bad arguments"); return DGRP_E_ARG; }
  index_slices(fasta, nbytes, world, cv, ov);
  *n_slices = (int64_t)ov.size();
  if ((int64_t)ov.size() > cap) { set_error("slice table too small: %lld needed", (long long)ov.size()); return DGRP_E_CAPACITY; }
  for (size_t k = 0; k < ov.size(); ++k) { if (cuts) cuts[k] = cv[k]; if (owner) owner[k] = ov[k]; }
  if (cuts) cuts[ov.size()] = cv[ov.size()];
  return DGRP_OK;
}

int dgrp_fasta_stream_plan(int64_t length, int vecsize, int step, int64_t unit_windows, int n_slabs, int ratio_pct,
                           int64_t *ends, int cap, int *n_out) {
  if (!n_out || length < 0 || vecsize <= 0 || step <= 0) { set_error("bad arguments"); return DGRP_E_ARG; }
  std::vector<int64_t> e;
  plan_slabs(length, vecsize, step, unit_windows > 0 ? unit_windows : (int64_t)148 * 128, n_slabs > 0 ? n_slabs : 6,
             ratio_pct, e);
  if (e.size() < 2) e.clear();
  *n_out = (int)e.size();
  if ((int)e.size() > cap) { set_error("slab table too small: %d needed", (int)e.size()); return DGRP_E_CAPACITY; }
  for (size_t i = 0; i < e.size(); ++i) ends[i] = e[i];
  return DGRP_OK;
}

int dgrp_fasta_stream_open(dgrp_ctx *c, dgrp_model *m, const uint8_t *fasta, int64_t nbytes, const char *filename,
                           int step, int batch_size, int use_mss, int min_mss_len, int xdrop_len, int compat,
                           dgrp_fasta_stream **out) {
  Use use(c->device);
  *out = nullptr;
  DGRP_REQUIRE(nbytes >= 0 && filename != nullptr, "bad arguments");
  DGRP_REQUIRE(step > 0, "step_size must be positive");
  dgrp_fasta_stream *s = new dgrp_fasta_stream();
  s->c = c; s->m = m; s->fasta = fasta; s->nbytes = nbytes; s->filename = filename;
  s->step = step; s->batch_size = batch_size; s->use_mss = use_mss; s->min_mss_len = min_mss_len;
  s->xdrop_len = xdrop_len; s->compat = compat;
  s->raw = c->st_raw; s->text = c->st_text; s->stage = c->st_stage; s->slot = c->st_slot;
  if (c->stream_slot_mb > 0) s->slot_bytes = (int64_t)c->stream_slot_mb << 20;
  stream_index(s);
  cudaPointerAttributes attr;
  if (nbytes > 0 && cudaPointerGetAttributes(&attr, fasta) == cudaSuccess) s->src_pinned = attr.type == cudaMemoryTypeHost;
  cudaGetLastError();
  int rc = DGRP_OK;
  auto ck = [&](cudaError_t e) { if (e != cudaSuccess && rc == DGRP_OK) { set_error("stream setup: %s", cudaGetErrorString(e)); rc = DGRP_E_CUDA; } };
  ck(cudaStreamCreateWithFlags(&s->s_in, cudaStreamNonBlocking));
  ck(cudaStreamCreateWithFlags(&s->s_out, cudaStreamNonBlocking));
  for (int i = 0; i < 2; ++i) {
    ck(cudaEventCreateWithFlags(&s->ev_in[i], cudaEventDisableTiming));
    ck(cudaEventCreateWithFlags(&s->ev_stage[i], cudaEventDisableTiming));
    ck(cudaEventCreateWithFlags(&s->ev_text[i], cudaEventDisableTiming));
    if (!s->src_pinned && rc == DGRP_OK) rc = s->stage[i].reserve((size_t)kStageBytes);
  }
  for (int i = 0; i < kSlots; ++i) {
    ck(cudaEventCreateWithFlags(&s->ev_slot[i], cudaEventDisableTiming | cudaEventBlockingSync));
    if (rc == DGRP_OK) rc = s->slot[i].reserve((size_t)s->slot_bytes);
  }
  if (rc != DGRP_OK) { dgrp_fasta_stream_close(s); return rc; }
  s->uploader = std::thread(stream_uploader_main, s);
  s->compute = std::thread(stream_compute_main, s);
  s->copier = std::thread(stream_copier_main, s);
  *out = s;
  return DGRP_OK;
}

int dgrp_fasta_stream_next(dgrp_fasta_stream *s, const uint8_t **tsv, int64_t *tsv_len, int64_t *slice,
                           int64_t *ordinal, int64_t *n_rows, int *last_of_record, int *done) {
  *tsv = nullptr; *tsv_len = 0; *done = 0;
  if (slice) *slice = -1;
  if (ordinal) *ordinal = -1;
  if (n_rows) *n_rows = 0;
  if (last_of_record) *last_of_record = 0;
  std::unique_lock<std::mutex> lk(s->mu);
  if (s->held >= 0) { s->slot_state[s->held] = 0; s->held = -1; s->cv.notify_all(); }
  s->cv.wait(lk, [&] { return !s->pieces.empty() || s->copier_done; });
  if (s->pieces.empty()) {
    // everything that was produced has been handed out; an error of the compute thread surfaces now, after the
    // rows of the records before it (the reference has written those when it raises)
    *done = 1;
    if (s->rc != DGRP_OK) { set_error("%s", s->err.c_str()); return s->rc; }
    return DGRP_OK;
  }
  const StreamPiece p = s->pieces.front();
  s->pieces.pop_front();
  if (p.slot >= 0) { s->slot_state[p.slot] = 2; s->held = p.slot; *tsv = s->slot[p.slot].as<uint8_t>(); }
  *tsv_len = p.bytes;
  if (slice) *slice = p.slice;
  if (ordinal) *ordinal = p.ordinal;
  if (n_rows) *n_rows = p.rows;
  if (last_of_record) *last_of_record = p.last;
  return DGRP_OK;
}

int dgrp_fasta_stream_stats(dgrp_fasta_stream *s, int64_t *rows, int64_t *records, int64_t *bases, int64_t *windows,
                            int64_t *launches, int64_t *h2d_bytes, int64_t *d2h_bytes, double *forward_ms,
                            double *gpu_ms) {
  std::lock_guard<std::mutex> lk(s->mu);
  if (rows) *rows = s->rows;
  if (records) *records = s->records;
  if (bases) *bases = s->bases;
  if (windows) *windows = s->windows;
  if (launches) *launches = s->launches;
  if (h2d_bytes) *h2d_bytes = s->h2d_bytes;
  if (d2h_bytes) *d2h_bytes = s->d2h_bytes;
  if (forward_ms) *forward_ms = s->forward_ms;
  if (gpu_ms) *gpu_ms = s->gpu_ms;
  return DGRP_OK;
}

int dgrp_fasta_stream_waits(dgrp_fasta_stream *s, double *out12) {
  std::lock_guard<std::mutex> lk(s->mu);
  for (int i = 0; i < 12; ++i) out12[i] = s->waits[i];
  return DGRP_OK;
}

int dgrp_fasta_stream_close(dgrp_fasta_stream *s) {
  if (!s) return DGRP_OK;
  Use use(s->c->device);
  {
    std::lock_guard<std::mutex> lk(s->mu);
    s->cancel = true;
    if (s->held >= 0) { s->slot_state[s->held] = 0; s->held = -1; }
  }
  s->cv.notify_all();
  if (s->uploader.joinable()) s->uploader.join();
  if (s->compute.joinable()) s->compute.join();
  {
    std::lock_guard<std::mutex> lk(s->mu);
    s->compute_done = true;
  }
  s->cv.notify_all();
  if (s->copier.joinable()) s->copier.join();
  cudaStreamSynchronize(s->c->stream);
  if (s->s_in) { cudaStreamSynchronize(s->s_in); cudaStreamDestroy(s->s_in); }
  if (s->s_out) { cudaStreamSynchronize(s->s_out); cudaStreamDestroy(s->s_out); }
  for (int i = 0; i < 2; ++i) {
    if (s->ev_in[i]) cudaEventDestroy(s->ev_in[i]);
    if (s->ev_stage[i]) cudaEventDestroy(s->ev_stage[i]);
    if (s->ev_text[i]) cudaEventDestroy(s->ev_text[i]);
  }
  for (int i = 0; i < kSlots; ++i)
    if (s->ev_slot[i]) cudaEventDestroy(s->ev_slot[i]);
  delete s;
  return DGRP_OK;
}

}  // extern "C"
