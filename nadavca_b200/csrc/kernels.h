// kernels.h -- host-side launchers of the sm_100a kernels (one per stage of the hot path).
#pragma once
#include "common.cuh"

// band.cu
void nvbk_band(const BatchDev &B, int64_t *d_summary, cudaStream_t st);
// d_out[total][4] = {mean, ac * scale, mc * scale, 0} of the k-mer at every reference position (BatchDev::row_emis)
void nvbk_row_emission(const ModelDev &M, const BatchDev &B, int64_t total, double scale, double *d_out, cudaStream_t st);
double nvbk_emission_scale();  // NVB_EXP_SCALE of dp3.cuh
void nvbk_expected_signal(const ModelDev &M, const BatchDev &B, int64_t total, double *d_out, cudaStream_t st);

// rows4.cu: forward + backward banded rows for reads [b0,b1): one CTA per (read, direction), stripes pipelined over
// its warps; rows are stored as a mantissa plane (double) and an exponent plane (int32).  wave_maxw = widest band
// row of the wave.  Returns -1 for an unsupported min_event_length, -2 when the hand-off rows do not fit shared memory.
// g_handoff: global scratch for the hand-off rows of band rows too wide for shared memory (size from
// nvbk_sweep2_global_handoff_doubles, 0 = not needed).
int64_t nvbk_sweep2_global_handoff_doubles(int mode, int n_reads, int wave_maxw);
int nvbk_sweep2(const ModelDev &M, const BatchDev &B, int mode, int b0, int b1, int wave_maxw,
                const int64_t *d_mat_base, double *pF, int32_t *pX, double *sF, int32_t *sX, double *g_handoff,
                cudaStream_t st);
// rows5.cu: the same rows with one continuously rotating wavefront per (read, direction); for reads whose bands allow
// it (band.cu flags the others).  Returns -1 for an unsupported min_event_length.
int nvbk_sweep_rotate(const ModelDev &M, const BatchDev &B, int mode, int b0, int b1, const int64_t *d_mat_base,
                      double *pF, int32_t *pX, double *sF, int32_t *sX, cudaStream_t st);
// no-SNP total (dtw.cpp:83-85) written into the reference-base column of out_ll
void nvbk_no_snp2(const ModelDev &M, const BatchDev &B, int b0, int b1, const int64_t *d_mat_base, const double *pF,
                  const int32_t *pX, const double *sF, const int32_t *sX, double *d_out_ll, cudaStream_t st);

// snp3.cu: the SNP re-run loop (dtw.cpp:93-129)
int nvbk_snp2(const ModelDev &M, const BatchDev &B, int wobbling, int b0, int b1, int64_t g0, int64_t g1,
              const int64_t *d_mat_base, const double *pF, const int32_t *pX, const double *sF, const int32_t *sX,
              double *d_out_ll, cudaStream_t st);

// path2.cu: posterior scores (in place over the prefix mantissa plane), max-product path with one record bit per
// cell, traceback (dtw.cpp:199-227).  nvbk_path2 returns -1 when the shared-memory reservation fails.
int nvbk_path2_columns_per_lane(int maxw);
void nvbk_score(int64_t total_cells, double *pF, const int32_t *pX, const double *sF, const int32_t *sX,
                cudaStream_t st);
int nvbk_path2(const BatchDev &B, int mode, int b0, int b1, int pk, const int64_t *d_mat_base, const double *score,
               uint32_t *d_records, const int64_t *d_rec_base, double *d_dp, const int64_t *d_dp_base, int wave_maxw,
               int32_t *d_events, int32_t *d_status, cudaStream_t st);

// finalize.cu
void nvbk_alignment_table(const BatchDev &B, const int32_t *d_events, const int32_t *d_status,
                          const int64_t *d_sig_start, const int64_t *d_ref_start, const int64_t *d_ref_end,
                          const int32_t *d_reverse, int64_t total, int64_t *d_out, cudaStream_t st);
void nvbk_event_means(const BatchDev &B, const int32_t *d_events, const int32_t *d_status, int64_t total, double *d_out,
                      cudaStream_t st);
void nvbk_apply_splines(const BatchDev &B, double *d_signal, const double *d_knots, const double *d_coefs,
                        const int64_t *d_spl_off, int degree, int64_t total, cudaStream_t st);
void nvbk_chunk_values(const BatchDev &B, const double *d_ll, const int32_t *d_reverse, double nel, int64_t total,
                       double *d_chunks, cudaStream_t st);
void nvbk_scatter_add_rows(const BatchDev &B, const double *d_chunks, const int64_t *d_dest, const int32_t *d_status,
                           int64_t total, double *d_rows, cudaStream_t st);
void nvbk_posterior_rows(const double *d_rows, int64_t base, int64_t row_lo, int64_t row_hi, const int8_t *d_ref,
                         const int64_t *d_group_off, int n_groups, int k, double snp_prior, double *d_out,
                         cudaStream_t st);
void nvbk_fill_status(const BatchDev &B, int32_t *d_status, double *d_ll, int alphabet, cudaStream_t st);

// select.cu: pooled median / MAD normalisation (read.py:67-81)
void nvbk_radix_hist(const double *d_values, int64_t n, int mode, double shift, unsigned long long prefix, int fixed,
                     unsigned long long *d_hist, cudaStream_t st);
void nvbk_normalize_each(const double *d_values, const int64_t *d_off, int n_reads, double lo, double hi, double *d_out,
                         double *d_shift_scale, cudaStream_t st);
void nvbk_normalize_clip(const double *d_values, int64_t n, double shift, double scale, double lo, double hi,
                         double *d_out, cudaStream_t st);

// anchors.cu: CIGAR -> matching-base anchors -> signal anchors and ranges (alignment.py:109-186), one warp per read
void nvbk_anchors(const AnchorBatch &A, int32_t *d_anchors, int64_t *d_meta, cudaStream_t st);

// microbench.cu
float nvbk_fp64_fma_probe(int iters, int blocks, cudaStream_t st, double *d_sink);
