/* deepgrp_b200.h -- C ABI of libdeepgrp_b200.so, the B200-native replacement for DeepGRP's
 * prediction hot path.
 *
 * Everything here is `extern "C"`, plain pointers and sizes.  Each entry point names the
 * reference interface it replaces (paths relative to the reference repo fhausmann/deepgrp).
 * INTEGRATION.md shows the ctypes / Cython stubs a reference maintainer would add.
 *
 * Conventions
 *  - every function returns 0 on success or a negative DGRP_E_* code; dgrp_last_error() gives
 *    the message of the last failure on the calling thread;
 *  - "host" entry points take HOST pointers and do their own H2D/D2H copies on the context's
 *    stream (they are what the Python shims of deepgrp.sequence / deepgrp.mss call);
 *  - "_dev" entry points take DEVICE pointers resident on the context's GPU and only enqueue
 *    kernels on the context's stream (no implicit synchronisation);
 *  - there is NO CPU fallback: without a usable sm_100 GPU dgrp_ctx_create fails.
 */
#ifndef DEEPGRP_B200_H_
#define DEEPGRP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DGRP_OK 0
#define DGRP_E_CUDA (-1)        /* a CUDA runtime call failed */
#define DGRP_E_ARG (-2)         /* invalid argument */
#define DGRP_E_NOGPU (-3)       /* no CUDA device / wrong architecture */
#define DGRP_E_ALLN (-4)        /* all-'N' sequence: the reference raises ValueError (sequence.pyx:32) */
#define DGRP_E_CAPACITY (-5)    /* caller-provided output too small; required size is reported */
#define DGRP_E_UNSUPPORTED (-6) /* model variant not implemented by the CUDA path */
#define DGRP_E_FASTA (-7)       /* malformed FASTA (blank line: the reference raises IndexError) */

/* Window-placement compatibility (SURVEY.md section 0 fact 3):
 * DGRP_COMPAT_REFERENCE reproduces deepgrp/prediction.py:105, where the final short batch is
 * max-merged at offset i*len(batch)*step; DGRP_COMPAT_FIXED places every window at w*step. */
#define DGRP_COMPAT_REFERENCE 0
#define DGRP_COMPAT_FIXED 1

typedef struct dgrp_ctx dgrp_ctx;     /* one GPU: device id, stream, workspace */
typedef struct dgrp_model dgrp_model; /* device-resident weights of one model */

/* Same layout as msseg_t, deepgrp/_mss/mss.h:11-14 */
typedef struct {
  int st, en;
  double sc;
} dgrp_seg_t;

/* One output row of `deepgrp predict` before formatting (deepgrp/__main__.py:288-292):
 * 0-based half-open [start, end) in ORIGINAL (untrimmed) record coordinates, label in 1..C-1. */
typedef struct {
  int64_t start, end;
  int32_t label;
  int32_t record; /* index of the FASTA record (dgrp_predict_fasta only; else 0) */
} dgrp_row_t;

/* Per-stage device times of the last dgrp_predict_* call, milliseconds (CUDA events). */
typedef struct {
  float encode_ms, forward_ms, attend_ms, score_ms, mss_ms, segments_ms, total_ms;
  int64_t windows, bases;
  int64_t kernel_launches;
} dgrp_timings_t;

/* ---- library / context ---------------------------------------------------------------- */
int dgrp_version(void);
const char *dgrp_last_error(void);
int dgrp_device_count(int *count);
int dgrp_ctx_create(int device, dgrp_ctx **out);
int dgrp_ctx_destroy(dgrp_ctx *ctx);
int dgrp_ctx_synchronize(dgrp_ctx *ctx);
/* CUDA stream of the context as a void* (cudaStream_t), for callers that enqueue their own work */
void *dgrp_ctx_stream(dgrp_ctx *ctx);
int dgrp_ctx_timings(dgrp_ctx *ctx, dgrp_timings_t *out);
/* number of kernels this library has launched on the context since creation */
int64_t dgrp_ctx_launch_count(dgrp_ctx *ctx);
/* tuning knobs and diagnostics: "mss_chunk" (elements per MSS scan chunk, 0 = automatic),
 * "mss_max_rounds" (parallel rounds before the sequential completion), "forward_tc" (1 = tcgen05
 * recurrence where available, 0 = fp32 kernel), "shard_rank" / "shard_world" (contig sharding of
 * dgrp_predict_fasta*: records are assigned largest-first to the least loaded rank; a rank
 * computes only its own records), and read-only "mss_rounds" (rounds the last MSS call used;
 * negative = completed sequentially), "forward_used_tc" (what the last forward used: 0 fp32 kernel, 1 two-tile tcgen05, 2 wide tcgen05 with one CTA per
 * tile, 3 wide tcgen05 CTA pair), "fused_last", "sm_count".  Round 2: "forward_wide" (0 auto, 1 / 2 force the wide
 * kernel's one-CTA / CTA-pair variant where it exists), "forward_slab_mb" (bound of the
 * window-probability buffer), "forward_fuse_score" (fuse vote + score transform for whole-record calls),
 * "stream_slot_mb" (host piece size of dgrp_fasta_stream), "stream_early_rows" / "stream_early_slabs" /
 * "stream_early_ratio" / "stream_early_unit" (position slabs of a long record in dgrp_fasta_stream; get-only
 * "stream_early_parts": parts of the last record's text that left before its last slab); get-only "eval_kernel_ns"
 * (device time of the last dgrp_evaluate_last kernel, nanoseconds); "keep_votes" (0 / 1, default 0: whether
 * dgrp_predict_fasta[_tsv] keeps every record's max-vote rows on the device for dgrp_track_last -- 4 C bytes per base
 * of the call, held until the next dgrp_predict_fasta[_tsv] without it or the context's destruction); get-only
 * "votes_append_ns" (device time of those copies in the last call) and "track_kernel_ns" (device time of the last
 * dgrp_track_last from its first kernel to its last, nanoseconds). */
int dgrp_ctx_set_int(dgrp_ctx *ctx, const char *key, int64_t value);
int dgrp_ctx_get_int(dgrp_ctx *ctx, const char *key, int64_t *value);

/* ---- deepgrp.sequence (deepgrp/sequence.pyx + deepgrp/maxcalc.c) --------------------- */

/* one_hot_encode_dna_sequence, sequence.pyx:55-58 / :21-36.  Two steps so the caller can size
 * the int8[5, L] array: _stage uploads the bytes and finds the edge-'N' trim on the GPU;
 * _fetch writes the one-hot matrix (C order [5, out_len]) into `fwd`.
 * fold_case != 0 treats 'n' like 'N' for trimming (the CLI upper-cases first, __main__.py:41).
 * Returns DGRP_E_ALLN when the trimmed length is negative (all-'N' input). */
int dgrp_one_hot_stage(dgrp_ctx *ctx, const uint8_t *seq, int64_t n, int fold_case,
                       int64_t *startpos, int64_t *out_len);
int dgrp_one_hot_fetch(dgrp_ctx *ctx, int8_t *fwd);

/* _get_max, maxcalc.c:10-24 / get_max, sequence.pyx:67-76: window b (dim0 x dim1 floats) is
 * max-merged into `output` at row b*stride.  `out_rows` is the number of rows of `output`
 * (the reference does not know it and never checks; rows beyond it are an error here). */
int dgrp_get_max(dgrp_ctx *ctx, float *output, int64_t out_rows, const float *inputs,
                 int64_t batchsize, int64_t dim0, int64_t dim1, int64_t stride);
int dgrp_get_max_dev(dgrp_ctx *ctx, float *d_output, int64_t out_rows, const float *d_inputs,
                     int64_t batchsize, int64_t dim0, int64_t dim1, int64_t stride);

/* get_segments, sequence.pyx:40-53 (including its size-1 loop bounds). out3 = start,end,label */
int dgrp_get_segments(dgrp_ctx *ctx, const int64_t *classes, int64_t size, int64_t startpos,
                      int64_t out3[3]);
/* yield_segments, sequence.pyx:79-85, materialised: all (start+off, end+off, label) triples in
 * order, label 0 included.  `out` holds cap triples; *n_out is the true count (DGRP_E_CAPACITY
 * if cap is too small; call again with a larger buffer). */
int dgrp_yield_segments(dgrp_ctx *ctx, const int64_t *classes, int64_t size, int64_t start_offset,
                        int64_t *out, int64_t cap, int64_t *n_out);

/* ---- deepgrp.mss (deepgrp/_mss/pymss.pyx + deepgrp/_mss/mss.c) ---------------------- */

/* mss_find_all, mss.c:50-101 (min_sc is truncated to int as at the reference call site,
 * mss.c:35).  Writes at most cap segments sorted by start; *n_seg is the true count. */
int dgrp_mss_find_all(dgrp_ctx *ctx, int n, const double *S, double min_sc, double xdrop,
                      dgrp_seg_t *out, int64_t cap, int *n_seg);
/* find_mss_labels, pymss.pyx:16-27: one_hot is double[n, nof_labels], written completely. */
int dgrp_find_mss_labels(dgrp_ctx *ctx, const double *scores, const int64_t *label, int n,
                         int nof_labels, int min_mss_len, int xdrop_len, double *one_hot);

/* ---- model (deepgrp/model.py:293-336; weights as stored by Keras) ---------------------- */

/* rnn: 0 = GRU (reset_after, gate order z,r,h): kernel[5,3U], recurrent[U,3U], bias[2,3U];
 *      1 = LSTM (gate order i,f,c,o): kernel[5,4U], recurrent[U,4U], bias[4U]; att_scale is ignored
 *          (the reference builds no attention for LSTM, deepgrp/model.py:308) and ff_kernel is [U,C].
 * att_scale[U] or NULL (no attention), ff_kernel[F,C] (F = 2U with attention else U), ff_bias[C].
 * tcgen05 recurrence: GRU with units <= 64 on the two-tile kernel, 65..128 on a CTA pair (cta_group::2), LSTM with
 * units <= 64 on the one-tile kernel; LSTM with 65..128 units runs the fp32 kernel; units > 128 are refused. */
int dgrp_model_create(dgrp_ctx *ctx, int rnn, int vecsize, int units, int n_classes,
                      const float *kernel, const float *recurrent, const float *bias,
                      const float *att_scale, const float *ff_kernel, const float *ff_bias,
                      dgrp_model **out);
int dgrp_model_destroy(dgrp_model *model);

/* keras.Model.predict_on_batch as used in deepgrp/prediction.py:106:
 * batch float32[B, T, 5] (host) -> probs float32[B, T, C] (host). */
int dgrp_forward_windows(dgrp_ctx *ctx, dgrp_model *model, const float *batch, int64_t nbatch,
                         float *probs);

/* ---- deepgrp.prediction ---------------------------------------------------------------- */

/* fetch_validation_batch + predict (prediction.py:14-37, 89-111) on a one-hot int8[5, L] matrix:
 * windows start at range(0, L-T, step); every window's softmax output is max-merged into the
 * zero-initialised predictions float32[L, C].  batch_size only matters for
 * DGRP_COMPAT_REFERENCE placement. */
int dgrp_predict_onehot(dgrp_ctx *ctx, dgrp_model *model, const int8_t *fwd, int64_t length,
                        int step, int batch_size, int compat, float *predictions);

/* apply_mss (prediction.py:40-59): probs float32[n, C] -> one-hot float64[n, C]. */
int dgrp_apply_mss(dgrp_ctx *ctx, const float *probs, int n, int n_classes, int min_mss_len,
                   int xdrop_len, double *one_hot);
/* The score transform alone (prediction.py:51-57): float64 scores + int64 classes. */
int dgrp_mss_scores(dgrp_ctx *ctx, const float *probs, int64_t n, int n_classes, double *scores,
                    int64_t *classes);
/* softmax (prediction.py:62-65): exp(x - global max) / row sum, float32[n, C]. */
int dgrp_softmax(dgrp_ctx *ctx, const float *array, int64_t n, int n_classes, float *out);

/* filter_segments (prediction.py:242-260): runs of one identical positive label shorter than
 * min_len are set to 0; labels uint8[n] (host), filtered in place. */
int dgrp_filter_segments(dgrp_ctx *ctx, uint8_t *labels, int64_t n, int64_t min_len);
/* confusion_matrix (prediction.py:200-218) for labels < 16: cnf[16*t + p] = number of positions with
 * true label t and predicted label p (int64[256], host).  DGRP_E_ARG for a label >= 16. */
int dgrp_confusion_matrix(dgrp_ctx *ctx, const uint8_t *truelbl, const uint8_t *predictedlbl, int64_t n,
                          int64_t *cnf);

/* ---- deepgrp.__main__ ------------------------------------------------------------------ */

/* _predict (__main__.py:46-83) for one record given as raw sequence bytes (no header, no
 * newlines): encode (fold_case as the CLI), forward, vote, then MSS (use_mss) or plain argmax.
 * labels (uint8[n]) receives labels for the trimmed record, *length its length. labels may be
 * NULL.  Rows (yield_segments + label>0 filter, __main__.py:288-290) are written to `rows`
 * (cap entries; DGRP_E_CAPACITY with *n_rows = required if too small). */
int dgrp_predict_sequence(dgrp_ctx *ctx, dgrp_model *model, const uint8_t *seq, int64_t n,
                          int fold_case, int step, int batch_size, int use_mss, int min_mss_len,
                          int xdrop_len, int compat, int64_t *startpos, int64_t *length,
                          uint8_t *labels, dgrp_row_t *rows, int64_t cap, int64_t *n_rows);

/* The same on a window range of one record, for multi-GPU sharding (SURVEY.md section 8e):
 * computes label (uint8) and float32 score for positions [pos0, pos1) of the TRIMMED record of
 * length `length` whose codes (0..4, 5 = non-ACGTN) are given for the whole record or at least
 * for [pos0 - T, pos1 + T) via `codes_base` (position of codes[0]). Outputs are host arrays. */
int dgrp_predict_range(dgrp_ctx *ctx, dgrp_model *model, const uint8_t *codes, int64_t codes_base,
                       int64_t codes_len, int64_t length, int64_t pos0, int64_t pos1, int step,
                       int batch_size, int compat, uint8_t *labels, float *scores);
/* MSS gap fill + segment rows from gathered (label, score) of a whole record.  use_mss = 0 is refused
 * (DGRP_E_UNSUPPORTED), here and in _finish_record_dev: without MSS the reference's labels are the argmax
 * after a softmax over the record's global maximum, which can round two close probabilities into a tie
 * that the ranges' raw-vote labels do not reproduce.  Predict such a record whole. */
int dgrp_finish_record(dgrp_ctx *ctx, const uint8_t *labels, const float *scores, int64_t length,
                       int n_classes, int use_mss, int min_mss_len, int xdrop_len,
                       int64_t startpos, uint8_t *labels_out, dgrp_row_t *rows, int64_t cap,
                       int64_t *n_rows);
/* Device-pointer forms of the two calls above, for chunk sharding inside one box: the codes, the
 * per-range (label, score) outputs and the gathered inputs of the owner stay in HBM and travel
 * between GPUs with one NCCL gather (bench.py --shard chunk).  _finish_record_dev leaves labels and
 * segment triples on the device and returns the row count (like dgrp_predict_codes_dev). */
int dgrp_predict_range_dev(dgrp_ctx *ctx, dgrp_model *model, const uint8_t *d_codes, int64_t codes_base,
                           int64_t codes_len, int64_t length, int64_t pos0, int64_t pos1, int step,
                           int batch_size, int compat, uint8_t *d_labels, float *d_scores);
int dgrp_finish_record_dev(dgrp_ctx *ctx, const uint8_t *d_labels, const float *d_scores, int64_t length,
                           int n_classes, int use_mss, int min_mss_len, int xdrop_len, int64_t *n_rows);

/* Whole-file driver (__main__.py:275-292 for one FASTA): raw FASTA text in, rows out.  The text is
 * decoded on the GPU (_read_multi_fasta, __main__.py:20-43: line stripping, '>' records, records
 * with an empty header dropped, case folding) and every record runs encode -> forward -> vote ->
 * MSS -> segments without leaving the device.  Results stay in the context until the next call:
 * *n_rows rows in record order and *n_records records; fetch them with the two calls below.
 * A blank line gives DGRP_E_FASTA (IndexError in the reference), an all-'N' record DGRP_E_ALLN. */
int dgrp_predict_fasta(dgrp_ctx *ctx, dgrp_model *model, const uint8_t *fasta, int64_t nbytes,
                       int step, int batch_size, int use_mss, int min_mss_len, int xdrop_len,
                       int compat, int64_t *n_rows, int64_t *n_records);
/* The same, but the rows are formatted on the GPU exactly as __main__.py:288-292 writes them
 * ("{filename}\t{header}\t{start}\t{end}\t{label}\n", label > 0 only): *tsv points at *tsv_len
 * bytes of finished text in pinned host memory owned by the context (valid until the next call).
 * The record table is available through dgrp_fasta_records; rows are NOT copied to the host. */
int dgrp_predict_fasta_tsv(dgrp_ctx *ctx, dgrp_model *model, const uint8_t *fasta, int64_t nbytes,
                           const char *filename, int step, int batch_size, int use_mss,
                           int min_mss_len, int xdrop_len, int compat, const uint8_t **tsv,
                           int64_t *tsv_len, int64_t *n_rows, int64_t *n_records);
/* Repeat-masked FASTA text: out[nbytes] (host) is the input with every position that a row covers lower-cased
 * (DGRP_MASK_SOFT: ASCII 'A'-'Z' only, other bytes unchanged) or replaced by 'N' (DGRP_MASK_HARD); every other
 * byte (headers, terminators, strip() whitespace, text in front of the first '>', records with an empty header,
 * unmasked positions) is copied unchanged.  A position is a byte of a sequence line inside the line's strip()
 * span, as _read_multi_fasta counts them (__main__.py:20-43); position p of record r is masked when a row of r has
 * start <= p < end (untrimmed coordinates).  rows[i].record indexes the kept records in file order, as in
 * dgrp_fasta_records.  The text is decoded on the GPU by the call.  DGRP_E_ARG for a bad mode, a record index out
 * of range, start < 0 or end > the record's untrimmed length or start >= end, label <= 0, or rows that are not
 * sorted by (record, start) or overlap within a record; DGRP_E_FASTA for a blank line. */
#define DGRP_MASK_SOFT 0
#define DGRP_MASK_HARD 1
int dgrp_mask_fasta(dgrp_ctx *ctx, const uint8_t *fasta, int64_t nbytes, const dgrp_row_t *rows, int64_t n_rows,
                    int mode, uint8_t *out);
/* The same with the record table and rows that the last dgrp_predict_fasta[_tsv] on this context left on the
 * device (no row goes to the host); `fasta` and `nbytes` must be that call's text.  DGRP_E_ARG when that call
 * failed or was sharded (shard_world > 1), when nbytes differs from its, or when another call has overwritten
 * its text on the device since. */
int dgrp_mask_fasta_last(dgrp_ctx *ctx, const uint8_t *fasta, int64_t nbytes, int mode, uint8_t *out);
/* Evaluation against a repeat annotation (the per-base multi-class confusion matrix that deepgrp/optimization.py:58-69
 * scores models with): counts[r][t][p] (int64[n_records][C][C], host) = positions of kept record r's span
 * [startpos, startpos + length) (dgrp_fasta_records) whose true class is t and whose predicted class is p, for the rows
 * the last dgrp_predict_fasta[_tsv] left on the device.  The predicted class of a position is the label of the row
 * that covers it, 0 where none does.  ann holds (begin, end, class) triples, 0-based half-open in untrimmed record
 * coordinates, record r's at [ann_off[r], ann_off[r + 1]) in any order, overlapping or not; they are clipped to the
 * span, and begin >= end contributes nothing.  The true class of a position is the lowest class among the triples that
 * cover it, 0 where none does (preprocess_y(...).argmax(axis=0), deepgrp/preprocessing.py:9-46).  No per-base array is
 * built: the rows and the sorted, merged runs of every (record, class) are compared as interval lists.  DGRP_E_ARG
 * when there is no such prediction (as in dgrp_mask_fasta_last), when n_records or n_classes differ from that call's
 * kept records and model classes, for a class outside [1, n_classes), a negative coordinate, a decreasing ann_off, or
 * a NULL pointer.  The device time of the kernel is read with dgrp_ctx_get_int(ctx, "eval_kernel_ns", ...). */
int dgrp_evaluate_last(dgrp_ctx *ctx, int n_classes, const int64_t *ann, const int64_t *ann_off, int64_t n_records,
                       int64_t *counts);
/* Probability track (bedGraph) of class cls for every kept record of the last dgrp_predict_fasta[_tsv], which must
 * have run with the option "keep_votes" set.  The value of a position is its max-vote pred[p][cls] before MSS or
 * softmax (the predictions of deepgrp/prediction.py:89-111).  Bins [k bin, (k + 1) bin) in untrimmed record
 * coordinates, clipped to the record's span [startpos, startpos + length); a bin's value is the float64 mean of its
 * positions' votes summed in ascending order, rounded half-to-even to thousandths (rint(mean * 1000.0)) and written
 * as "%d.%03d".  Consecutive bins of one record with the same value form one line "chrom\tstart\tend\tvalue\n";
 * chrom is the first word of the header; no track line, records in file order.  *text is pinned host memory owned by
 * the context, valid until the next call of this function or the context's destruction.  DGRP_E_ARG when there is no
 * such prediction (as in dgrp_mask_fasta_last), when it did not keep its votes, for cls outside [1, C), a bin outside
 * [1, 1000000] or a NULL pointer. */
int dgrp_track_last(dgrp_ctx *ctx, int cls, int bin, const uint8_t **text, int64_t *len);
/* rows[i].record indexes the record table */
int dgrp_fasta_rows(dgrp_ctx *ctx, dgrp_row_t *rows, int64_t cap);
/* per record: header text = fasta[hdr_off, hdr_off + hdr_len); startpos = leading 'N' count;
 * length = trimmed length.  Any of the four arrays may be NULL. */
int dgrp_fasta_records(dgrp_ctx *ctx, int64_t *hdr_off, int64_t *hdr_len, int64_t *startpos,
                       int64_t *length, int64_t cap);
/* per record: owning rank, and where its rows are in the TSV text of dgrp_predict_fasta_tsv
 * (tsv_len 0 for records owned by another rank; their startpos is -1 and length untrimmed). */
int dgrp_fasta_record_tsv(dgrp_ctx *ctx, int64_t *owner, int64_t *tsv_off, int64_t *tsv_len,
                          int64_t cap);

/* Streaming, pipelined form of the whole-file driver.  deepgrp/__main__.py:275-295 writes the rows of a record as
 * soon as the record is done; this does the same with bounded memory and with the copies off the critical path:
 * the text is cut into slices at header lines on the host ('>' at a line start), a rank uploads ONLY its own slices
 * ("shard_rank" / "shard_world": largest slice first to the least loaded rank) through a pinned staging ring, and a
 * record's finished TSV text travels to the host in pieces of <= 64 MiB on a second stream while the next record is
 * being computed.  `fasta` must stay valid until _close.  _next returns the next piece of text in file order of this
 * rank's records (*tsv valid until the following call): (*slice, *ordinal) identify the record (slice number in the
 * file, record number within the slice), *last_of_record marks its final piece; *n_rows is the number of rows that
 * are complete with this piece (the counts of a record's pieces add up to its rows); a record without rows yields
 * one empty piece.  A long record (>= ~4 waves of the forward kernel) with MSS is computed in position slabs and the
 * rows that are already final -- everything before the last run at which mss.c:78-81 flushes its candidate stack --
 * leave as pieces while the later slabs are still being computed ("stream_early_rows": 1, the default, for the last
 * record of the rank's share -- the only one whose text no later record's compute would hide --, 2 for every long
 * record, 0 never; the text is the same bytes in the same order either way).  *done = 1 when everything has been handed out -- an error met on the way (blank line,
 * all-'N' record, CUDA) is returned by that last call, after the text of the records before it, as the reference
 * has written those rows when it raises.  One stream per context at a time; the context must not be used for
 * other calls while a stream is open. */
typedef struct dgrp_fasta_stream dgrp_fasta_stream;
/* The stream's host index alone (no GPU needed): the text is cut at header lines into slices of >= 8 MiB,
 * cuts[0 .. n_slices] (cap + 1 entries) are their byte offsets and owner[k] the rank slice k goes to among `world`
 * ranks (largest slice first to the least loaded rank).  DGRP_E_CAPACITY with *n_slices = required if cap is too small. */
int dgrp_fasta_index(const uint8_t *fasta, int64_t nbytes, int world, int64_t *cuts, int32_t *owner, int64_t cap,
                     int64_t *n_slices);
/* The position slabs the stream would cut a record of `length` bases into (host arithmetic only, no GPU needed):
 * ends[0 .. *n_slabs) are the slab ends, the last one = length; *n_slabs = 0 when the record is too short for the
 * early-rows route.  unit_windows = windows of one forward wave (0: 128 x 148), n_slabs / ratio_pct = 0: the defaults
 * (6 slabs, each 80 % of the one before).  DGRP_E_CAPACITY when cap is too small. */
int dgrp_fasta_stream_plan(int64_t length, int vecsize, int step, int64_t unit_windows, int n_slabs, int ratio_pct,
                           int64_t *ends, int cap, int *n_out);
int dgrp_fasta_stream_open(dgrp_ctx *ctx, dgrp_model *model, const uint8_t *fasta, int64_t nbytes,
                           const char *filename, int step, int batch_size, int use_mss, int min_mss_len,
                           int xdrop_len, int compat, dgrp_fasta_stream **out);
int dgrp_fasta_stream_next(dgrp_fasta_stream *stream, const uint8_t **tsv, int64_t *tsv_len, int64_t *slice,
                           int64_t *ordinal, int64_t *n_rows, int *last_of_record, int *done);
/* totals so far (any pointer may be NULL): rows, records, trimmed bases, windows, kernel launches, bytes uploaded /
 * copied back, forward-kernel and whole-GPU milliseconds (CUDA events, summed over records) */
int dgrp_fasta_stream_stats(dgrp_fasta_stream *stream, int64_t *rows, int64_t *records, int64_t *bases,
                            int64_t *windows, int64_t *launches, int64_t *h2d_bytes, int64_t *d2h_bytes,
                            double *forward_ms, double *gpu_ms);
/* diagnostics: milliseconds the pipeline's threads spent waiting -- [0] compute for the upload, [1] compute for a
 * free device text buffer, [2] copier for a finished record, [3] copier for a free host slot, [4] copier for its
 * copies, [5] uploader for a free device buffer, [6] uploader copying, [7] the compute thread in total, [8] slice
 * decodes, [9] records (host wall clock), [10] TSV measure + write, [11] trim + encode */
int dgrp_fasta_stream_waits(dgrp_fasta_stream *stream, double *out12);
int dgrp_fasta_stream_close(dgrp_fasta_stream *stream);

/* Device-resident step used by bench.py's `value` leg: codes already in HBM (d_codes, length L),
 * runs forward + vote + score + MSS + segment extraction entirely on the device and leaves the
 * row count in *n_rows (rows stay on the device).  No host copies except the 8-byte count. */
int dgrp_predict_codes_dev(dgrp_ctx *ctx, dgrp_model *model, const uint8_t *d_codes,
                           int64_t length, int step, int batch_size, int use_mss,
                           int min_mss_len, int xdrop_len, int compat, int64_t *n_rows);
/* Copies what the last dgrp_predict_codes_dev left on the device to the host: the final label of each of its
 * `length` positions (labels, may be NULL) and its n_rows rows as (start, end, label) int64 triples (rows, may be
 * NULL).  `length` and `n_rows` must be those of that call, and no call that overwrites them (one computing labels
 * or rows) may have run on the context since, even one that failed (DGRP_E_ARG otherwise). */
int dgrp_predict_codes_dev_results(dgrp_ctx *ctx, uint8_t *labels, int64_t length, int64_t *rows, int64_t n_rows);

/* ---- training (deepgrp/training.py, deepgrp/model.py:202-215) ----------------------------------------------- */

/* A trainer holds one GRU model's weights, its optimiser state and its training / validation records on the
 * context's GPU.  Supported: rnn = 0 (GRU, reset_after=True) with 1 <= units <= 64, n_classes 2..5 (the classes
 * dgrp_model_create accepts), with or without attention; LSTM, units > 64 and n_classes > 5 give
 * DGRP_E_UNSUPPORTED.  Every step is fp32 on CUDA cores and bit-reproducible on one GPU (no float atomics).  Weights and gradients use the Keras layouts of dgrp_model_create: kernel[5,3U],
 * recurrent[U,3U], bias[2,3U], att_scale[U] (NULL without attention), ff_kernel[F,C], ff_bias[C].
 * optimizer: DGRP_OPT_RMSPROP (momentum > 0: TF ApplyRMSProp, ms = rho ms + (1-rho) g^2, mom = momentum mom +
 * lr g / sqrt(ms + eps), w -= mom; momentum = 0: w -= lr g / (sqrt(ms) + eps)) or DGRP_OPT_ADAM (Keras: beta1 0.9,
 * beta2 0.999, w -= lr sqrt(1-beta2^t) / (1-beta1^t) m / (sqrt(v) + eps)).  dropout in [0, 1) is the GRU's input
 * dropout (recurrent dropout 0). */
#define DGRP_OPT_RMSPROP 0
#define DGRP_OPT_ADAM 1
typedef struct dgrp_trainer dgrp_trainer;
int dgrp_train_create(dgrp_ctx *ctx, int rnn, int vecsize, int units, int n_classes, int attention,
                      const float *kernel, const float *recurrent, const float *bias, const float *att_scale,
                      const float *ff_kernel, const float *ff_bias, int optimizer, float learning_rate, float rho,
                      float momentum, float epsilon, float dropout, dgrp_trainer **out);
/* Uploads one record: which = 0 training, 1 validation; codes[L] base codes 0..4 (A, C, G, T, N: the row of the
 * one-hot matrix), ymask[L] bit c set where class c is annotated (several bits where annotations overlap).
 * DGRP_E_ARG when L < vecsize or a code / bit is out of range. */
int dgrp_train_set_data(dgrp_trainer *tr, int which, const uint8_t *codes, const uint8_t *ymask, int64_t length);
/* One step on n windows of the training record: window b covers [starts[b], starts[b] + vecsize); keep[b][dir][c]
 * (0/1) is the input dropout mask of direction dir (0 forward, 1 reverse complement) for the channel c the GRU
 * sees.  *loss receives the batch's mean loss before the update. */
int dgrp_train_step(dgrp_trainer *tr, const int64_t *starts, const uint8_t *keep, int64_t n, float *loss);
/* Forward only (no dropout, no update) on n windows of record `which`: *loss = mean loss, probs [n][T][C] or NULL. */
int dgrp_train_eval(dgrp_trainer *tr, int which, const int64_t *starts, int64_t n, float *loss, float *probs);
/* Current weights / gradients of the last step (before its update), host arrays in the Keras layouts above. */
int dgrp_train_get_weights(dgrp_trainer *tr, float *kernel, float *recurrent, float *bias, float *att_scale,
                           float *ff_kernel, float *ff_bias);
int dgrp_train_get_grads(dgrp_trainer *tr, float *kernel, float *recurrent, float *bias, float *att_scale,
                         float *ff_kernel, float *ff_bias);
/* Device milliseconds of the last step's phases: forward, head, BPTT, weight-gradient reduction, update. */
int dgrp_train_timings(dgrp_trainer *tr, float *out5);
int dgrp_train_destroy(dgrp_trainer *tr);

#ifdef __cplusplus
}
#endif
#endif /* DEEPGRP_B200_H_ */
