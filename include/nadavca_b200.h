/*
 * nadavca_b200.h -- C ABI of libnadavca_b200.so: the B200 (sm_100a) replacement for nadavca's native DP core.
 *
 * The reference exposes its hot path through ONE foreign-function boundary, the pybind11 module `nadavca.dtw`
 * (/root/reference/nadavca/dtw/dtwmodule.cpp:10-29), called from nadavca/estimator.py:77,99,172.  Every entry
 * point below names the reference interface it replaces.  The boundary is batched: one call handles a whole
 * batch of reads (CSR layout: a value array plus an int64 offsets array of n_reads+1 entries per field), because
 * one read exposes far too little parallelism for a GPU.  A batch of one read is exactly the reference call.
 *
 * Conventions
 *   - plain C, no torch / CUDA types in signatures; `stream` is a cudaStream_t passed as void* (NULL = default
 *     stream); device pointers are named d_*; everything else is host memory owned by the caller.
 *   - every int-returning function returns 0 on success, a negative NVB_E* code on failure; nvb_last_error()
 *     gives the message (thread-local).  There is NO CPU fallback: without a usable CUDA device every compute
 *     entry point fails with NVB_ECUDA.
 *   - the library keeps nothing of the caller's buffers after a call returns.
 */
#ifndef NADAVCA_B200_H
#define NADAVCA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NVB_OK 0
#define NVB_EINVAL (-1)   /* bad argument */
#define NVB_ECUDA (-2)    /* CUDA runtime error / no device */
#define NVB_ENOMEM (-3)   /* workspace does not fit the device */
#define NVB_ESTATE (-4)   /* call order (e.g. download before run) */

/* per-read status written by the refine / estimate calls */
#define NVB_READ_OK 0
#define NVB_READ_NO_PATH 1  /* reference: RefineAlignment returns an empty vector (dtw.cpp:211-213) */
#define NVB_READ_BAD_BAND 2 /* anchors give an empty band row (the reference would throw std::length_error) */

typedef struct nvb_model nvb_model;
typedef struct nvb_batch nvb_batch;

int nvb_abi_version(void);
const char *nvb_last_error(void);
/* number of usable CUDA devices (0 when there is no driver/GPU); never fails */
int nvb_device_count(void);
/* Device buffers of destroyed batches / models are kept in a per-device cache for re-use (cudaFree costs far more
 * than a batch's kernels); this hands the cached blocks back to the driver. */
int nvb_trim_memory(int device);
/* Schedule of the forward / backward row sweeps (a tuning knob without a reference counterpart; results are
 * identical): AUTO picks per wave by batch size, ROTATE = one rotating wavefront per (read, direction), STRIPES =
 * pipelined 31-row stripes.  Returns the previous setting. */
#define NVB_SWEEP_AUTO 0
#define NVB_SWEEP_ROTATE 1
#define NVB_SWEEP_STRIPES 2
int nvb_set_sweep_schedule(int schedule);

/* ---- k-mer model: replaces class KmerModel (dtwmodule.cpp:12-18, kmer_model.cpp:6-42) -------------------- */
/* mean/sigma have alphabet_size^k entries; tables (mean, log(1/sqrt(2 pi s^2)), 1/(2 s^2)) are built on the host
 * with the same libm expressions as kmer_model.cpp:10-13 and uploaded to `device`. */
nvb_model *nvb_model_create(int k, int central_position, int alphabet_size, const double *mean,
                            const double *sigma, int64_t n_kmers, int device);
void nvb_model_destroy(nvb_model *model);
int nvb_model_k(const nvb_model *model);                 /* KmerModel::GetK */
int nvb_model_central_position(const nvb_model *model);  /* KmerModel::GetCentralPosition */
int nvb_model_alphabet_size(const nvb_model *model);
/* bytes of device memory held by the model's DP workspaces, summed over every stream it has run on (each workspace
 * grows to the largest wave seen on its stream and is kept until the model is destroyed, see nvb_batch_refine) */
int64_t nvb_model_workspace_bytes(const nvb_model *model);
/* KmerModel::GetExpectedSignal (kmer_model.cpp:32-42), batched; runs as a CUDA kernel.
 * reference/context arrays as in nvb_reads; out has reference_off[n_reads] doubles (host). */
int nvb_model_expected_signal(nvb_model *model, int32_t n_reads, const int32_t *reference,
                              const int64_t *reference_off, const int32_t *context_before,
                              const int64_t *context_before_off, const int32_t *context_after,
                              const int64_t *context_after_off, double *out);

/* ---- a batch of reads: the arguments shared by refine_alignment / estimate_log_likelihoods ------------- */
/* (dtwmodule.cpp:19-28: signal, reference, context_before, context_after, approximate_alignment, bandwidth,
 *  min_event_length).  All pointers are HOST memory. */
typedef struct nvb_reads {
  int32_t n_reads;
  const double *signal;           /* concatenated signal slices */
  const int64_t *signal_off;      /* [n_reads+1] */
  const int32_t *reference;       /* concatenated numeric bases (0..alphabet-1) */
  const int64_t *reference_off;   /* [n_reads+1] */
  const int32_t *context_before;  /* may be NULL when context_before_off is all zero */
  const int64_t *context_before_off;
  const int32_t *context_after;
  const int64_t *context_after_off;
  const int32_t *anchors;         /* approximate_alignment: pairs (signal index, reference index) */
  const int64_t *anchor_off;      /* [n_reads+1], counted in pairs */
  int32_t bandwidth;
  int32_t min_event_length;
} nvb_reads;

/* One-shot calls with HOST buffers (upload -> kernels -> download).  These are the drop-in for the two pybind
 * functions; host<->device copies happen inside. */

/* refine_alignment (dtwmodule.cpp:24-28 -> RefineAlignment dtw.cpp:133-228).
 * events: int32[reference_off[n_reads]][2] = (event start, event end) sample offsets into each read's slice;
 * status: int32[n_reads] (NVB_READ_*); rows of reads without a path are filled with -1. */
int nvb_refine_alignment_batch(nvb_model *model, const nvb_reads *reads, int model_transitions, int32_t *events,
                               int32_t *status);
/* estimate_log_likelihoods (dtwmodule.cpp:19-23 -> EstimateLogLikelihoods dtw.cpp:37-131).
 * out: double[reference_off[n_reads]][alphabet_size] raw log-likelihoods; status: int32[n_reads]. */
int nvb_estimate_log_likelihoods_batch(nvb_model *model, const nvb_reads *reads, int model_wobbling, double *out,
                                       int32_t *status);

/* ---- resident batches: inputs uploaded once, results kept in HBM ----------------------------------------- */
/* Upload a batch and compute its band geometry (ComputeBandStarts/Ends dtw.cpp:7-35) on the device. */
nvb_batch *nvb_batch_create(nvb_model *model, const nvb_reads *reads);
void nvb_batch_destroy(nvb_batch *batch);
/* limit for the DP matrices kept in HBM at one time (bytes; 0 = 70% of the free device memory).  Batches that
 * need more are processed in several waves of reads. */
int nvb_batch_set_workspace_limit(nvb_batch *batch, int64_t bytes);
/* run the kernels on `stream`; asynchronous with respect to the host except for wave planning.  The DP matrices live
 * in workspaces owned by the MODEL, one per stream (each grows to the largest wave seen on its stream and is freed with
 * the model): runs on one stream are ordered by the stream, runs on different streams use different workspaces, so
 * batches of one model may be in flight on several streams at once.  The result getters (nvb_batch_get_*, event
 * means, alignment table) read back on the stream of the batch's latest run and wait for that stream only. */
int nvb_batch_refine(nvb_batch *batch, int model_transitions, void *stream);
int nvb_batch_estimate(nvb_batch *batch, int model_wobbling, void *stream);
/* results of the last run (blocking copies) */
int nvb_batch_get_events(nvb_batch *batch, int32_t *events, int32_t *status);
int nvb_batch_get_log_likelihoods(nvb_batch *batch, double *out, int32_t *status);
/* band geometry, for tests and cell counting: starts/ends int32[reference_off[n]+n_reads] (n_r+1 rows per read) */
int nvb_batch_get_bands(nvb_batch *batch, int32_t *starts, int32_t *ends);
/* DP cell counts of the batch by the formulas of SURVEY.md 8(d): [0] refine with transitions, [1] refine without,
 * [2] estimate forward+backward, [3] estimate SNP loop */
int nvb_batch_cell_counts(nvb_batch *batch, int model_wobbling, int64_t counts[4]);
/* debugging aid: the stored DP rows of read `read` after nvb_batch_estimate (plane 0 = prefix, 1 = suffix) as
 * log-probabilities, packed band rows 0..n (cells = sum of band widths); the read must be in the last wave */
int nvb_batch_debug_rows(nvb_batch *batch, int read, int plane, double *out_log, int64_t n_cells);
/* number of kernels launched by this batch object so far (bench.py reports it as gpu_launches) */
int64_t nvb_batch_launch_count(const nvb_batch *batch);
/* per-stage device timing with CUDA events recorded on the run's stream (measurement only; no reference
 * counterpart).  Stages: 0 forward/backward rows, 1 path + traceback, 2 no-SNP total, 3 SNP loop. */
#define NVB_N_STAGES 4
int nvb_batch_enable_timing(nvb_batch *batch, int on);
/* synchronises the device; ms / launches are accumulated since the last call (then reset) */
int nvb_batch_get_timing(nvb_batch *batch, double ms[NVB_N_STAGES], int64_t launches[NVB_N_STAGES]);
/* sustained FP64 FMA issue rate of `device` in FMA/s (a register-resident DFMA loop on every SM, best of 3);
 * the denominator of the ALU roofline reported by bench.py */
int nvb_measure_fp64_fma_rate(int device, double *fma_per_second);

/* ---- estimator post-processing on the device (nadavca/estimator.py) ------------------------------------------ */
/* (n,3) alignment table of get_refined_alignment (estimator.py:187-195):
 * out int64[sum n][3] = (reference position, event_start + start_in_signal, event_end + start_in_signal);
 * reference position = ref_start + i (forward) or ref_end - i - 1 (reverse strand). Host buffers. */
int nvb_batch_get_alignment_table(nvb_batch *batch, const int64_t *start_in_signal, const int64_t *ref_start,
                                  const int64_t *ref_end, const int32_t *reverse, int64_t *out);
/* Mean of the signal samples of every refined event, out double[sum n] (host): the numpy.mean calls of
 * Read.tweak_signal_normalization (read.py:86) and of the align_signal renormalisation (align_signal.py:66-70),
 * reproduced bit for bit (numpy's pairwise summation order) from the resident signal and events.  NaN for reads
 * without a path and for empty events. */
int nvb_batch_event_means(nvb_batch *batch, double *out);
/* Evaluation half of Read.tweak_signal_normalization (read.py:94, scipy.interpolate.splev, FITPACK splev/fpbspl with
 * extrapolation): every sample x of a read's resident signal is replaced by spline_r(x).  The splines come from the
 * host fit (scipy.interpolate.splrep, read.py:93) as FITPACK's knots t and coefficients c, both of length
 * spline_off[r+1] - spline_off[r] per read (0 = leave the read's signal as it is); degree = 3 for the reference. */
int nvb_batch_apply_splines(nvb_batch *batch, const double *knots, const double *coefs, const int64_t *spline_off,
                            int degree, void *stream);
/* the resident signal values (after nvb_batch_apply_splines), double[signal_off[n_reads]] */
int nvb_batch_get_signal(nvb_batch *batch, double *out);
/* _normalize_log_likelihoods + reverse-strand complement/flip (estimator.py:45-47,111-119) applied to the
 * resident raw log-likelihoods; d_chunks: double[sum n][4] device buffer (alphabet must be 4).  Asynchronous: the
 * per-read `reverse` (and `dest` of nvb_batch_scatter_add_rows) arrays are kept on the device and re-uploaded only
 * when they change. */
int nvb_batch_chunk_values(nvb_batch *batch, const int32_t *reverse, double normalization_event_length,
                           double *d_chunks, void *stream);
/* ---- batched anchor construction: replaces the per-read CIGAR walk and signal-alignment glue of
 * ApproximateAligner (alignment.py:109-140 parse the CIGAR and keep matching bases; alignment.py:142-186 convert them
 * to signal anchors and ranges).  Mapping the reads (BWA) stays on the host; its hits come in as CSR arrays. ---------- */
typedef struct nvb_hits {
  int32_t n_reads;
  const int32_t *cigar_len;       /* CIGAR operations of all reads: lengths ... */
  const int8_t *cigar_op;         /* ... and codes 0 = M, 1 = I, 2 = D, 3 = S */
  const int64_t *cigar_off;       /* [n_reads + 1] */
  const int64_t *mapped_position; /* 0-based position of the hit in the contig (SAM pos - 1) */
  const int32_t *reverse;         /* 1 = the read maps to the reverse strand */
  const int8_t *read_sequence;    /* basecalled bases 0..3 of all reads (Read.sequence) ... */
  const int32_t *base_to_sample;  /* ... and the sample index of each base, -1 = not placed
                                   * (Read.sequence_to_signal_mapping) */
  const int64_t *read_off;        /* [n_reads + 1] */
  const int32_t *n_signal;        /* len(Read.normalized_signal) per read */
  const int8_t *d_genome;         /* DEVICE pointer: contig bases 0..3 (anything else: 4) */
  int64_t genome_length;
  int32_t bandwidth;
} nvb_hits;
/* anchors: host int32[2 * read_off[n_reads]]; the anchors of read b are the first meta[7b] (sample index - extended
 * signal start, reference index - first anchored reference index) pairs from anchors + 2 * read_off[b].
 * meta: host int64[7 * n_reads] = per read [n_anchors, reference_start, reference_end, signal_start, signal_end,
 * read_sequence_start, read_sequence_end] in the conventions of ApproximateSignalAlignment (alignment.py:10-17,
 * 153-186); n_anchors = 0 and -1s for a read without usable anchors. */
int nvb_signal_anchors_batch(int device, const nvb_hits *hits, int32_t *anchors, int64_t *meta, void *stream);

/* ---- pooled median / MAD normalisation on the device: replaces Read.normalize_reads (read.py:67-81) ------------
 * One pass of an exact most-significant-digit radix select over the order-preserving 64-bit keys of d_values (or of
 * |d_values - shift| when absolute_deviation != 0): ADDS to d_hist[256] the histogram of the 8 key bits below the
 * `fixed_bits` (0, 8, .. 56) leading bits, over the values whose leading bits equal `prefix`.  Eight passes find an
 * order statistic; a job sharded over GPUs all-reduces d_hist between the kernel and the bin choice.  Enqueues only. */
int nvb_radix_histogram_d(int device, const double *d_values, int64_t n, int absolute_deviation, double shift,
                          uint64_t prefix, int fixed_bits, uint64_t *d_hist, void *stream);
/* Every read normalised on its own (align_signal.py:54 calls Read.normalize_reads with one read at a time): values / out
 * are HOST arrays, CSR over reads by off[n_reads + 1]; out = clip((values - median) / MAD, lo, hi) with the exact
 * per-read median and MAD (one CTA per read, radix select in shared memory); shift_scale (optional, host,
 * 2 * n_reads) receives them. */
int nvb_normalize_each(int device, const double *values, const int64_t *off, int32_t n_reads, double lo, double hi,
                       double *out, double *shift_scale, void *stream);
/* d_out = clip((d_values - shift) / scale, lo, hi)  (read.py:80-81).  Enqueues only. */
int nvb_normalize_clip_d(int device, const double *d_values, int64_t n, double shift, double scale, double lo, double hi,
                         double *d_out, void *stream);

/* Consensus accumulator as ROWS of 5 doubles [sum A, sum C, sum G, sum T, coverage] (estimator.py:226-231): sums and
 * coverage travel in one buffer, so the exchange between GPUs is one collective (reduce-scatter by genome slice, or
 * all-reduce).  d_rows is a zero-initialised device buffer of (total rows, 5) doubles: d_rows[dest[r] + i][j] +=
 * chunk_r[i][j] and d_rows[dest[r] + i][4] += 1 for every read r with dest[r] >= 0 and status OK.  dest is a HOST
 * array of n_reads row offsets. */
int nvb_batch_scatter_add_rows(nvb_batch *batch, const double *d_chunks, const int64_t *dest, double *d_rows,
                               void *stream);
/* _compute_posterior (estimator.py:123-156) for the global rows [row_lo, row_hi) of the concatenated groups, from
 * consensus rows that start at global row base_row (a rank's slice plus its k-1 halo rows); d_ref and d_group_off
 * are indexed by global rows, d_ref int8 (0..3, anything else = no base matches), d_group_off int64[n_groups+1].
 * d_out_rows: (row_hi - row_lo, 5) doubles = [P(A), P(C), P(G), P(T), coverage].  Only enqueues the kernel on
 * `stream`. */
int nvb_posterior_rows_d(int device, const double *d_rows, int64_t base_row, int64_t row_lo, int64_t row_hi,
                         const int8_t *d_ref, const int64_t *d_group_off, int32_t n_groups, int k, double snp_prior,
                         double *d_out_rows, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* NADAVCA_B200_H */
