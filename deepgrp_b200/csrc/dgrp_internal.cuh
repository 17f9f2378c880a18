// Internal declarations shared by the translation units of libdeepgrp_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <utility>
#include <vector>

#include "../../include/deepgrp_b200.h"

namespace dgrp {

// class counts a model may have: the prediction kernels' output layout holds at most 5 classes, and the trainer
// accepts only models that prediction can run
constexpr int MODEL_CMIN = 2, MODEL_CMAX = 5;

void set_error(const char *fmt, ...);

#define DGRP_CUDA(call)                                                                      \
  do {                                                                                       \
    cudaError_t e__ = (call);                                                                \
    if (e__ != cudaSuccess) {                                                                \
      dgrp::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
      return DGRP_E_CUDA;                                                                    \
    }                                                                                        \
  } while (0)

#define DGRP_CHECK(call)          \
  do {                            \
    int rc__ = (call);            \
    if (rc__ != DGRP_OK) return rc__; \
  } while (0)

#define DGRP_REQUIRE(cond, ...)      \
  do {                               \
    if (!(cond)) {                   \
      dgrp::set_error(__VA_ARGS__);  \
      return DGRP_E_ARG;             \
    }                                \
  } while (0)

// Grow-only device buffer.
struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  // reserve() calls so far.  Every call that writes a buffer reserves it first, so an unchanged count means
  // unchanged contents (dgrp_predict_codes_dev_results relies on it).
  uint64_t reserves = 0;
  int reserve(size_t bytes);
  void release();
  template <typename T>
  T *as() const { return reinterpret_cast<T *>(p); }
};

// Grow-only pinned host buffer.
struct PinBuf {
  void *p = nullptr;
  size_t cap = 0;
  int reserve(size_t bytes);
  void release();
  template <typename T>
  T *as() const { return reinterpret_cast<T *>(p); }
};

}  // namespace dgrp

struct dgrp_model {
  int device = 0;
  int rnn = 0;
  int T = 0, U = 0, C = 0, UP = 0;  // UP: units padded to a multiple of 16
  bool attention = false;
  // device arrays
  float *d_kernel = nullptr;     // [5, 3U]     raw Keras kernel
  float *d_bias = nullptr;       // [2, 3U]
  float *d_recurrent = nullptr;  // [U, 3U]     raw Keras recurrent kernel
  float *d_P = nullptr;          // [5, 3, UP]  kernel[c, g*U+u] + bias[0, g*U+u], zero padded
  float *d_Wk = nullptr;         // [5, 3, UP]  kernel alone (dense float input), zero padded
  float *d_b0 = nullptr;         // [3, UP]     bias[0, g*U+u], zero padded
  float *d_Rp = nullptr;         // [UP, 3, UP] recurrent[k, g*U+u], zero padded
  float *d_b1 = nullptr;         // [3, UP]     bias[1, g*U+u], zero padded
  // two-tile tcgen05 form (forward_tc.cu): [2][(3UP + 16) x (UP + 16)] fp16 hi|lo of ([R | K/2]^T * 2^b_shift)
  // (+ 16 one-hot K rows), UMMA K-major core matrices; null where the shape has no such form
  uint16_t *d_Bsplit = nullptr;
  int b_shift = 0;
  // wide tcgen05 form (forward_tcw.cu): fp16 hi|lo pieces of the blocked [R | K/2]^T (+ 16 one-hot K rows), for one
  // CTA per tile and for a CTA pair ([rank][piece][rows of the rank]); null where the shape has no such form
  uint16_t *d_Bw[2] = {};   // [0 one CTA | 1 CTA pair]
  int bw_shift = 0;
  float *d_scale = nullptr;      // [U] or null
  float *d_ffk = nullptr;        // [F, C]
  float *d_ffb = nullptr;        // [C]
};

struct dgrp_ctx {
  int device = 0;
  int sm_count = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[8] = {};
  int64_t launches = 0;
  dgrp_timings_t timings = {};
  // workspaces (grow-only)
  dgrp::DevBuf raw, codes, onehot, avg, pred, labels, labels2, scores32, scores64, classes64,
      io_a, io_b, io_c, small, segs, rows, mss_a, mss_b, mss_c, mss_d, mss_e, scan, winprobs, gapfill;
  dgrp::PinBuf pin_small, pin_a, pin_b;
  // tuning knobs / diagnostics (dgrp_ctx_set_int / dgrp_ctx_get_int)
  int mss_chunk = 0;       // elements per MSS scan chunk (0 = automatic)
  int mss_max_rounds = 0;  // Jacobi rounds before the sequential completion (0 = default)
  int mss_rounds = 0;      // rounds used by the last MSS call (negative: completed sequentially)
  int forward_tc = 1;      // 1: tcgen05 recurrence where available, 0: fp32 FFMA kernel
  int forward_gather = 1;  // tcgen05 forward: write window probabilities and max-merge them in a gather pass
                           // (1) instead of 5 atomicMax per window-step (0); falls back to 0 above 40 GB
  int forward_wide = 0;    // 0: the wide tcgen05 kernel (forward_tcw.cu) only where the two-tile kernel has no form
                           // (units > 64, LSTM); 1 / 2: force its single-CTA / CTA-pair variant where it exists
  int stream_slot_mb = 0;  // dgrp_fasta_stream: size of one host piece of TSV text, MiB (0 = 64)
  int stream_early_rows = 1;   // dgrp_fasta_stream: a long record is computed in position slabs and the rows that are
                               // final after a slab (everything before the last MSS flush) leave while the next slab runs:
                               // 1 = the rank's last record (whose text nothing else would hide), 2 = every long record, 0 = off
  int stream_early_slabs = 0;  // number of slabs of a long record (0 = default: 6)
  int stream_early_unit = 0;   // windows per unit of a slab (0 = one wave of the forward kernel: 128 x SM count)
  int stream_early_ratio = 0;  // size of a slab relative to the one before it, per cent (0 = default: 80)
  int stream_early_parts = 0;  // diagnostic: parts of the last record's text that left before its last slab
  int64_t forward_slab_bytes = (int64_t)8 << 30;   // bound of the window-probability buffer: the windows of a
                           // record run in slabs of at most this many bytes of [windows][T][C] probabilities
  int forward_smem_vote = 1;    // tcgen05 forward: max-merge a tile's windows in shared memory (no window probabilities in HBM)
  int forward_fuse_score = 1;   // whole-record calls: fuse vote + score transform when the windows fit one slab
  int fused_last = 0;      // the last core_predict produced label + score directly (no predictions in HBM)
  int forward_used_tc = 0; // what the last forward launch used: 0 fp32 kernel, 1 two-tile tcgen05, 2 wide, 3 wide CTA pair
  // results of the last dgrp_predict_fasta (fetched with dgrp_fasta_rows / dgrp_fasta_records)
  std::vector<dgrp_row_t> fa_rows;
  std::vector<int64_t> fa_hdr_off, fa_hdr_len, fa_startpos, fa_length, fa_tsv_off, fa_tsv_len, fa_owner;
  // the last dgrp_predict_codes_dev: record length, row count, and the reserve counts of labels2 and segs when it
  // returned (its labels in labels2 and rows in segs are fetched with dgrp_predict_codes_dev_results while neither
  // buffer has been reserved since)
  int64_t codes_dev_length = -1, codes_dev_rows = 0;
  uint64_t codes_dev_reserves[2] = {};
  // the last dgrp_predict_fasta[_tsv] for dgrp_mask_fasta_last and dgrp_evaluate_last: every kept record's first
  // sequence rank and first row (one more row entry: the total), its rows on the device as (start, end, label)
  // triples, its byte count (-1: it failed, was sharded, or none ran) and the reserve count of c->raw (its text)
  // when it returned
  std::vector<int64_t> fa_seq_base, fa_row_off;
  dgrp::DevBuf fa_tri;
  int64_t mask_nbytes = -1;
  uint64_t mask_raw_reserves = 0;
  int fa_classes = 0;                  // the model classes of that call (dgrp_evaluate_last)
  dgrp::DevBuf eval_tab, eval_counts;  // dgrp_evaluate_last: record / run table, per-record counts
  int64_t eval_kernel_ns = 0;          // device time of the last evaluation kernel (CUDA events)
  // dgrp_track_last: with keep_votes set, dgrp_predict_fasta[_tsv] also keeps every kept record's max-vote rows
  // (f32[length][C], record r's from row fa_pred_off[r]) and its chromosome (first word of the header, fa_chrom at
  // fa_chrom_off[r]); fa_votes: the last call did so and succeeded.  fa_pred holds the votes of the largest call
  // (grow-only while keep_votes is set) and is freed by the next call without keep_votes.  track_* hold the table, the
  // bin words, the line starts, the text on the device and in pinned host memory (the view dgrp_track_last returns)
  int keep_votes = 0;
  bool fa_votes = false;
  dgrp::DevBuf fa_pred;
  std::vector<int64_t> fa_pred_off, fa_chrom_off;
  std::string fa_chrom;
  dgrp::DevBuf track_tab, track_work, track_text;
  dgrp::PinBuf track_host;
  int64_t votes_append_ns = 0;         // device time of the vote appends of the last dgrp_predict_fasta[_tsv]
  int64_t track_kernel_ns = 0;         // device time of the kernels of the last dgrp_track_last (CUDA events)
  cudaEvent_t tev[2] = {};
  dgrp::DevBuf mask_rec, mask_bits, mask_out;   // dgrp_mask_fasta*: record table, rank bitmap, masked text
  int shard_rank = 0, shard_world = 1;   // contig sharding of dgrp_predict_fasta* (dgrp_ctx_set_int)
  dgrp::PinBuf tsv_host;     // finished TSV text of the last dgrp_predict_fasta_tsv
  int64_t tsv_len = 0;
  dgrp::DevBuf tsv_dev, tsv_prefix;
  // buffers of dgrp_fasta_stream (kept across streams): uploaded slices, finished record text, upload staging,
  // host pieces
  dgrp::DevBuf st_raw[2], st_text[2];
  dgrp::PinBuf st_stage[2], st_slot[4];
  // staged one-hot state (dgrp_one_hot_stage -> dgrp_one_hot_fetch)
  int64_t staged_n = 0, staged_start = 0, staged_len = -1;
};

namespace dgrp {
// offsets into a trainer's flat parameter vector: the Keras arrays of a GRU model concatenated
struct TrainLayout {
  int F;                        // FF kernel rows (2U with attention, else U)
  int oK, oR, oB, oS, oF, oFB;  // kernel [5,3U], recurrent [U,3U], bias [2,3U], scale [U], FF kernel [F,C], FF bias [C]
  int n;                        // parameter count
  int HP;                       // per-window head gradient floats: F*C + C + U
};
}  // namespace dgrp

struct dgrp_trainer {
  dgrp_ctx *ctx = nullptr;
  int T = 0, U = 0, C = 0;
  bool attention = false;
  int optimizer = 0;
  float lr = 0.f, rho = 0.f, momentum = 0.f, epsilon = 0.f, dropout = 0.f;
  int64_t steps = 0;
  int64_t length[2] = {-1, -1};   // record length of the training / validation data (-1: not set)
  dgrp::TrainLayout L = {};
  // parameters, gradients of the last step, optimiser state (RMSprop ms / mom, Adam m / v)
  dgrp::DevBuf w, g, s1, s2;
  dgrp::DevBuf codes[2], ymask[2], starts, keep;
  dgrp::DevBuf Hs, GS, D, avg, dhin, hpart, rpart, lpart, probs;
  std::vector<float> h_lpart;
  cudaEvent_t ev[6] = {};   // forward | head | BPTT | reduction | update of the last step
  bool timed = false;
};

namespace dgrp {

struct Use {  // RAII: make the context's device current
  int prev = -1;
  explicit Use(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~Use() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

// A few bytes (counts, flags, sizes) from the device into PINNED host memory, written by a one-block kernel
// through the mapped address instead of a D2H memcpy: a copy would queue on the copy engine behind the multi-MB
// pieces of TSV text that dgrp_fasta_stream moves on its own stream (measured: ~8 ms per FASTA slice decode
// instead of 0.3).  Visible to the host after the stream has been synchronised.
int fetch_small(dgrp_ctx *c, void *pinned_dst, const void *d_src, size_t bytes);

// ---- kernel launchers (device pointers, enqueue on ctx->stream) ------------------------------
// encode.cu
int launch_trim(dgrp_ctx *c, const uint8_t *d_seq, int64_t n, int fold_case, int64_t *d_first_last);
int launch_onehot(dgrp_ctx *c, const uint8_t *d_seq, int64_t start, int64_t len, int8_t *d_fwd);
int launch_codes(dgrp_ctx *c, const uint8_t *d_seq, int64_t start, int64_t len, uint8_t *d_codes);
int launch_onehot_to_codes(dgrp_ctx *c, const int8_t *d_fwd, int64_t len, uint8_t *d_codes);
// vote.cu
int launch_vote_gather(dgrp_ctx *c, const float *d_win, int64_t w_begin, int64_t w_end, int T, int C,
                       int64_t full_windows, int64_t tail_base, int step, float *d_pred, int64_t pred_row0,
                       int64_t pred_rows, uint8_t *d_label = nullptr, float *d_score = nullptr);
int launch_get_max(dgrp_ctx *c, float *d_out, const float *d_in, int64_t batch, int64_t dim0,
                   int64_t dim1, int64_t stride);
int launch_score(dgrp_ctx *c, const float *d_pred, int64_t n, int C, uint8_t *d_label,
                 float *d_score32, double *d_score64, int64_t *d_class64);
int launch_softmax_global(dgrp_ctx *c, const float *d_in, int64_t n, int C, float *d_out);
// forward.cu
struct Placement {  // where window w is max-merged (prediction.py:105 compatibility)
  int64_t n_windows;    // W
  int64_t full_windows; // windows in complete batches (= W when compat is FIXED)
  int64_t tail_base;    // row offset of the first window of the short last batch
  int step;
};
Placement make_placement(int64_t length, int T, int step, int batch_size, int compat);
// Run GRU + attention + FF + softmax for windows [w_begin, w_end) of the code array and
// max-merge into d_pred (rows relative to pred_row0; rows outside [0, pred_rows) are dropped).
// [w2_begin, w2_end): a second window range voted into the same rows (not with d_label / d_score).
// With d_label / d_score (whole record, pred_row0 = 0): when the windows fit one slab of the tcgen05 path the vote
// and the score transform are fused (*fused = true: label + score written, d_pred untouched and NOT zero-filled by
// the caller beforehand); otherwise *fused = false and d_pred (zero-initialised by the caller) holds the votes.
int run_forward_vote(dgrp_ctx *c, dgrp_model *m, const uint8_t *d_codes, int64_t codes_base,
                     int64_t w_begin, int64_t w_end, const Placement &pl, float *d_pred,
                     int64_t pred_row0, int64_t pred_rows, uint8_t *d_label = nullptr, float *d_score = nullptr,
                     bool *fused = nullptr, int64_t w2_begin = 0, int64_t w2_end = 0);
// dense float windows [B, T, 5] -> probs [B, T, C] (predict_on_batch semantics)
int run_forward_dense(dgrp_ctx *c, dgrp_model *m, const float *d_batch, int64_t nbatch,
                      float *d_probs);
// forward_tcw.cu: host-side packing of the wide tcgen05 kernel's weight operand (empty where the shape has no form)
void build_tcw_operands(int rnn, int U, int UP, int C, bool att, const float *Rp, const float *P, const float *b1,
                        const float *ffk, std::vector<uint16_t> (&out)[2], int *shift);
// mss.cu
// L0: the running sum the scan starts from (0 at the start of a record).  resume != nullptr: the scores are a
// PREFIX of a record ("open end"): only the segments that are final whatever follows are returned -- those the
// last FLUSH run (mss.c:78-81) or an earlier event flushed -- and *resume receives where and with which running
// sum the record can be resumed (restart = -1: nowhere yet; the caller then passes the same prefix start again).
struct MssResume {
  int restart;   // index of the first element of the last FLUSH run
  double L0;     // running sum before it
};
int run_mss_segments(dgrp_ctx *c, const double *d_s64, const float *d_s32, int n, double min_sc,
                     double xdrop, dgrp_seg_t **d_segs_out, int *n_seg, double L0 = 0.0,
                     MssResume *resume = nullptr);
int run_gap_fill(dgrp_ctx *c, const dgrp_seg_t *d_segs, int n_seg, const uint8_t *d_label_in,
                 const int64_t *d_label64_in, int n, int nof_labels, uint8_t *d_label_out);
int launch_labels_to_onehot(dgrp_ctx *c, const uint8_t *d_label, int64_t n, int C, double *d_out);
// fasta.cu
struct FastaScan {              // classification of a FASTA buffer (device arrays in c->scan)
  int64_t ntiles;
  uint8_t *tile_state;          // [ntiles] line state in front of every tile
  unsigned *seq_off, *hdr_off;  // [ntiles] sequence bytes / headers in front of every tile
  int64_t n_seq, n_hdr;         // totals
};
int run_fasta_classify(dgrp_ctx *c, const uint8_t *d_raw, int64_t n, FastaScan *f);
int run_fasta_decode(dgrp_ctx *c, const uint8_t *d_raw, int64_t n, int64_t *n_seq, int64_t *n_hdr,
                     FastaScan *scan = nullptr);
// mask.cu
// Masked copy of the FASTA buffer d_raw[n] (classified in f) into d_out[n]: a sequence byte of rank q is masked
// when a row of kept record r covers q - rec[2 r] (rec[2 r]: rank of the record's first sequence byte,
// rec[2 r + 1]: index of its first row in d_tri; rec[2 n_rec + 1] = number of rows).  d_tri: (start, end, label)
// triples, sorted and disjoint within a record, records in rank order.
int run_mask(dgrp_ctx *c, const uint8_t *d_raw, int64_t n, const FastaScan &f, const int64_t *d_tri,
             const int64_t *d_rec, int64_t n_rec, int mode, uint8_t *d_out);
// tsv.cu
int run_tsv_measure(dgrp_ctx *c, const int64_t *d_tri, int64_t n, int prefix_len, int64_t *need);
int run_tsv_write(dgrp_ctx *c, const int64_t *d_tri, int64_t n, const uint8_t *d_prefix,
                  int prefix_len, uint8_t *d_out);
// evaluate.cu
int launch_filter_segments(dgrp_ctx *c, const uint8_t *d_in, uint8_t *d_out, int64_t n, int64_t min_len);
int launch_confusion(dgrp_ctx *c, const uint8_t *d_truth, const uint8_t *d_pred, int64_t n,
                     unsigned long long *d_cnf, int *d_bad);
namespace eval { struct Table; }
// K10: adds the confusion counts of every record of the table t (uploaded to d_tab) against the rows d_tri of
// dgrp_predict_fasta to d_counts[r][t][p] (int64, zeroed by the caller); one launch
int run_eval_confusion(dgrp_ctx *c, int C, const eval::Table &t, const int64_t *d_tab, const int64_t *d_tri,
                       int64_t *d_counts);
// track.cu
namespace track { struct Table; }
// K11: the bedGraph text of class cls for every record of the table t (uploaded to d_tab, prefix text at d_text)
// from the vote rows d_pred into text (device, reserved here); *n_bytes = its length.  Bin words and line starts go
// to work; synchronises twice (line count, byte count)
int run_track(dgrp_ctx *c, const track::Table &t, const int64_t *d_tab, const uint8_t *d_text, const float *d_pred,
              int C, int cls, DevBuf &work, DevBuf &text, int64_t *n_bytes);
// segments.cu
// open_tail != nullptr: the labels are a prefix of a record whose continuation is not known yet.  The
// reference's special case of the record's last element does not apply, and a run that reaches the end of
// the prefix is NOT emitted: *open_tail receives its first index (n when the prefix ends on a zero).
int run_segments(dgrp_ctx *c, const uint8_t *d_label, const int64_t *d_label64, int64_t n,
                 int64_t offset, bool keep_zero, int64_t **d_triples, int64_t *n_out,
                 int64_t *open_tail = nullptr);
int launch_get_segments(dgrp_ctx *c, const int64_t *d_classes, int64_t size, int64_t startpos,
                        int64_t *d_out3);
// train.cu
constexpr int TR_CMAX = 8;   // classes the head kernel's per-thread arrays hold (>= MODEL_CMAX)
TrainLayout make_train_layout(int U, int C, bool att);
int train_check_shape(int T, int U, int C, bool att);
// one training step on n windows of the training record (starts, keep on the device); leaves the gradients in
// tr->g, the per-window losses in tr->lpart, and updates tr->w
int train_run_step(dgrp_ctx *c, dgrp_trainer *tr, int64_t n, const int64_t *d_starts, const uint8_t *d_keep);
// forward only, no dropout: per-window losses into h_lpart[n] (host), probabilities [n][T][C] into d_probs if set
int train_run_eval(dgrp_ctx *c, dgrp_trainer *tr, int which, int64_t n, const int64_t *d_starts, float *d_probs,
                   float *h_lpart);

}  // namespace dgrp
