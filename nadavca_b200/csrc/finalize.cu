// finalize.cu -- elementwise post-processing of the estimator glue, kept on the device so that a batch makes one
// round trip: alignment table (estimator.py:187-195), normalised / strand-flipped chunks (estimator.py:45-47,
// 111-119), consensus scatter-add (estimator.py:226-231) and the Bayesian posterior stencil (estimator.py:123-156).
#include "common.cuh"
#include "kernels.h"

namespace {

__device__ __forceinline__ int find_read(const BatchDev &B, int64_t g) {
  int lo = 0, hi = B.n_reads;  // last read with ref_off <= g (empty reads are skipped by construction)
  while (hi - lo > 1) {
    int mid = (lo + hi) >> 1;
    if (B.ref_off[mid] <= g) lo = mid; else hi = mid;
  }
  return lo;
}

__global__ void alignment_table_kernel(BatchDev B, const int32_t *events, const int32_t *status,
                                       const int64_t *sig_start, const int64_t *ref_start, const int64_t *ref_end,
                                       const int32_t *reverse, int64_t total, int64_t *out) {
  int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (g >= total) return;
  const int b = find_read(B, g);
  const int64_t i = g - B.ref_off[b];
  if (status[b] != 0) { out[3 * g] = -1; out[3 * g + 1] = -1; out[3 * g + 2] = -1; return; }
  out[3 * g] = reverse[b] ? ref_end[b] - i - 1 : ref_start[b] + i;
  out[3 * g + 1] = events[2 * g] + sig_start[b];
  out[3 * g + 2] = events[2 * g + 1] + sig_start[b];
}

// numpy's float64 add.reduce over a contiguous 1-D array (pairwise_sum in numpy/_core/src/umath/loops_utils.h.src):
// fewer than 8 terms are added in order, up to 128 terms go through 8 interleaved accumulators combined as
// ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)) plus an in-order tail, longer blocks are split at n/2 rounded down to a multiple
// of 8.  Reproduced operation for operation (the file is compiled without FMA contraction) so that event means equal
// numpy.mean bit for bit -- they feed the spline tweak (read.py:86-88) and the linear renormalisation
// (align_signal.py:66-72), whose results the alignment must match exactly.
__device__ double numpy_pairwise_sum(const double *a, int n) {
  if (n < 8) {
    double res = 0.0;
    for (int i = 0; i < n; i++) res += a[i];
    return res;
  }
  if (n <= 128) {
    double r[8];
#pragma unroll
    for (int j = 0; j < 8; j++) r[j] = a[j];
    int i;
    for (i = 8; i < n - (n % 8); i += 8) {
#pragma unroll
      for (int j = 0; j < 8; j++) r[j] += a[i + j];
    }
    double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; i++) res += a[i];
    return res;
  }
  int n2 = n / 2;
  n2 -= n2 % 8;
  return numpy_pairwise_sum(a, n2) + numpy_pairwise_sum(a + n2, n - n2);
}

// Mean of the signal samples of every refined event (read.py:86, align_signal.py:66-70): one thread per base.
__global__ void event_means_kernel(BatchDev B, const int32_t *events, const int32_t *status, int64_t total,
                                   double *out) {
  int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (g >= total) return;
  const int b = find_read(B, g);
  const double nan = __longlong_as_double(0x7ff8000000000000LL);
  if (status[b] != 0) { out[g] = nan; return; }
  const int s = events[2 * g], e = events[2 * g + 1];
  const int n = e - s;
  if (n <= 0) { out[g] = nan; return; }  // numpy.mean of an empty slice
  out[g] = numpy_pairwise_sum(B.signal + B.sig_off[b] + s, n) / (double)n;
}

// FITPACK splev (ext = 0) / fpbspl, degree k <= 5, for one abscissa: the evaluation half of
// Read.tweak_signal_normalization (read.py:94, scipy.interpolate.splev).  Same operations in the same order as the
// Fortran (no FMA contraction in this file), so the result equals scipy's up to the compiler's rounding of a/b.
__device__ double fitpack_splev(const double *t, const double *c, int n, int k, double x) {
  const int k1 = k + 1, nk1 = n - k1;
  // l (1-based) = last knot <= x, clamped to [k1, nk1]
  int lo = 0, hi = n;  // count of knots <= x
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (t[mid] <= x) lo = mid + 1; else hi = mid;
  }
  const int l = min(max(lo, k1), nk1);
  double h[6], hh[5];
  h[0] = 1.0;
  for (int j = 1; j <= k; j++) {
    for (int i = 0; i < j; i++) hh[i] = h[i];
    h[0] = 0.0;
    for (int i = 1; i <= j; i++) {
      const int li = l + i, lj = li - j;  // 1-based knot indices
      const double tli = t[li - 1], tlj = t[lj - 1];
      if (tli == tlj) {
        h[i] = 0.0;
      } else {
        const double f = hh[i - 1] / (tli - tlj);
        h[i - 1] = h[i - 1] + f * (tli - x);
        h[i] = f * (x - tlj);
      }
    }
  }
  double sp = 0.0;
  for (int j = 1; j <= k1; j++) sp = sp + c[l - k1 + j - 1] * h[j - 1];
  return sp;
}

// signal[g] <- spline_b(signal[g]) for every sample of every read that has a spline (n_knots > 0), in place.
__global__ void apply_splines_kernel(BatchDev B, double *signal, const double *knots, const double *coefs,
                                     const int64_t *spl_off, int degree, int64_t total) {
  int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (g >= total) return;
  int lo = 0, hi = B.n_reads;  // last read with sig_off <= g
  while (hi - lo > 1) {
    int mid = (lo + hi) >> 1;
    if (B.sig_off[mid] <= g) lo = mid; else hi = mid;
  }
  const int64_t o = spl_off[lo];
  const int n = (int)(spl_off[lo + 1] - o);
  if (n < 2 * (degree + 1)) return;
  signal[g] = fitpack_splev(knots + o, coefs + o, n, degree, signal[g]);
}

// (LL - LL[0][ref[0]]) / normalization_event_length; reverse strand: complement the columns, flip the rows.
__global__ void chunk_values_kernel(BatchDev B, const double *ll, const int32_t *reverse, double nel, int64_t total,
                                    double *chunks) {
  int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (g >= total) return;
  const int b = find_read(B, g);
  const int64_t r0 = B.ref_off[b];
  const int64_t n = B.ref_off[b + 1] - r0;
  const int64_t i = g - r0;
  const double shift = ll[r0 * 4 + B.ref[r0]];
  if (reverse[b]) {
    const double *src = ll + (r0 + (n - 1 - i)) * 4;
#pragma unroll
    for (int j = 0; j < 4; j++) chunks[g * 4 + j] = (src[3 - j] - shift) / nel;
  } else {
    const double *src = ll + g * 4;
#pragma unroll
    for (int j = 0; j < 4; j++) chunks[g * 4 + j] = (src[j] - shift) / nel;
  }
}

// Consensus accumulator as ROWS of 5 doubles [A, C, G, T, coverage]: the sums of estimator.py:226-231 and the coverage
// count of estimator.py:229-230 in one buffer, so that the exchange between GPUs is ONE collective (coverage counts
// are small integers, exact in a double).
__global__ void scatter_add_rows_kernel(BatchDev B, const double *chunks, const int64_t *dest, const int32_t *status,
                                        int64_t total, double *rows) {
  int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (g >= total) return;
  const int b = find_read(B, g);
  if (dest[b] < 0 || status[b] != 0) return;
  const int64_t p = dest[b] + (g - B.ref_off[b]);
#pragma unroll
  for (int j = 0; j < 4; j++) atomicAdd(rows + p * 5 + j, chunks[g * 4 + j]);
  atomicAdd(rows + p * 5 + 4, 1.0);
}

// _compute_posterior (estimator.py:131-156) at global row g: window [max(0,i-k+1), min(i+k,L)) inside the position's
// group, same accumulation order as the reference.  `rows` holds consensus rows of 5 doubles starting at global row
// `base` (the whole buffer, or a slice with its k-1 halo rows).
__device__ __forceinline__ void posterior_at(const double *rows, int64_t base, const int8_t *ref,
                                             const int64_t *group_off, int n_groups, int64_t g, int k, double snp_prior,
                                             double pr_out[4]) {
  int lo = 0, hi = n_groups;
  while (hi - lo > 1) {
    int mid = (lo + hi) >> 1;
    if (group_off[mid] <= g) lo = mid; else hi = mid;
  }
  const int64_t gs = group_off[lo], ge = group_off[lo + 1];
  const int64_t i = g - gs, L = ge - gs;
  const int64_t cs = max((int64_t)0, i - k + 1), ce = min(i + k, L);
  const double *row0 = rows + (gs - base) * 5;  // row of the group's first position
  double mx = nvb_neg_inf();
  for (int64_t i2 = cs; i2 < ce; i2++)
    for (int j = 0; j < 4; j++) mx = fmax(mx, row0[i2 * 5 + j]);
  // _corrected_priors (estimator.py:123-129)
  const double c = 3.0;
  const double p1 = 1 - snp_prior, p2 = snp_prior / c;
  const double snp_h = 1 / (p1 / p2 + (1 - (double)(ce - cs - 1)) * c);
  const double nonsnp_h = 1 - snp_h * c;
  double pr[4];
  const int rb = ref[g];
  for (int j = 0; j < 4; j++) {
    const double prior = (j != rb) ? snp_h : nonsnp_h;
    double v = exp(row0[i * 5 + j] - mx) * prior;
    if (j == rb) {
      for (int64_t i2 = cs; i2 < ce; i2++) {
        if (i2 == i) continue;
        const int rb2 = ref[gs + i2];
        for (int j2 = 0; j2 < 4; j2++) {
          if (j2 == rb2) continue;
          v += exp(row0[i2 * 5 + j2] - mx) * snp_h;
        }
      }
    }
    pr[j] = v;
  }
  double sum = 0.0;  // Python's builtin sum() starts from int 0
  for (int j = 0; j < 4; j++) sum += pr[j];
  for (int j = 0; j < 4; j++) pr_out[j] = pr[j] / sum;
}

// Posterior of the global rows [row_lo, row_hi) from consensus rows of 5 doubles that start at global row `base`
// (base <= row_lo - (k-1) unless row_lo opens a group): out rows of 5 = [P(A), P(C), P(G), P(T), coverage].
__global__ void posterior_rows_kernel(const double *rows, int64_t base, int64_t row_lo, int64_t row_hi,
                                      const int8_t *ref, const int64_t *group_off, int n_groups, int k, double snp_prior,
                                      double *out) {
  int64_t g = row_lo + blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (g >= row_hi) return;
  double pr[4];
  posterior_at(rows, base, ref, group_off, n_groups, g, k, snp_prior, pr);
  double *o = out + (g - row_lo) * 5;
  for (int j = 0; j < 4; j++) o[j] = pr[j];
  o[4] = rows[(g - base) * 5 + 4];
}

__global__ void fill_status_kernel(BatchDev B, int32_t *status, double *ll, int alphabet) {
  const int b = blockIdx.x;
  const int f = B.flags[b];
  if (threadIdx.x == 0) status[b] = f;
  if (f && ll) {
    const int64_t r0 = B.ref_off[b] * alphabet, r1 = B.ref_off[b + 1] * alphabet;
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    for (int64_t x = r0 + threadIdx.x; x < r1; x += blockDim.x) ll[x] = nan;
  }
}

inline unsigned blocks_for(int64_t total) { return (unsigned)((total + 255) / 256); }

}  // namespace

void nvbk_alignment_table(const BatchDev &B, const int32_t *d_events, const int32_t *d_status,
                          const int64_t *d_sig_start, const int64_t *d_ref_start, const int64_t *d_ref_end,
                          const int32_t *d_reverse, int64_t total, int64_t *d_out, cudaStream_t st) {
  if (total > 0)
    alignment_table_kernel<<<blocks_for(total), 256, 0, st>>>(B, d_events, d_status, d_sig_start, d_ref_start,
                                                              d_ref_end, d_reverse, total, d_out);
}

void nvbk_event_means(const BatchDev &B, const int32_t *d_events, const int32_t *d_status, int64_t total, double *d_out,
                      cudaStream_t st) {
  if (total > 0) event_means_kernel<<<blocks_for(total), 256, 0, st>>>(B, d_events, d_status, total, d_out);
}

void nvbk_apply_splines(const BatchDev &B, double *d_signal, const double *d_knots, const double *d_coefs,
                        const int64_t *d_spl_off, int degree, int64_t total, cudaStream_t st) {
  if (total > 0)
    apply_splines_kernel<<<blocks_for(total), 256, 0, st>>>(B, d_signal, d_knots, d_coefs, d_spl_off, degree, total);
}

void nvbk_chunk_values(const BatchDev &B, const double *d_ll, const int32_t *d_reverse, double nel, int64_t total,
                       double *d_chunks, cudaStream_t st) {
  if (total > 0) chunk_values_kernel<<<blocks_for(total), 256, 0, st>>>(B, d_ll, d_reverse, nel, total, d_chunks);
}

void nvbk_scatter_add_rows(const BatchDev &B, const double *d_chunks, const int64_t *d_dest, const int32_t *d_status,
                           int64_t total, double *d_rows, cudaStream_t st) {
  if (total > 0) scatter_add_rows_kernel<<<blocks_for(total), 256, 0, st>>>(B, d_chunks, d_dest, d_status, total, d_rows);
}

void nvbk_posterior_rows(const double *d_rows, int64_t base, int64_t row_lo, int64_t row_hi, const int8_t *d_ref,
                         const int64_t *d_group_off, int n_groups, int k, double snp_prior, double *d_out,
                         cudaStream_t st) {
  if (row_hi > row_lo)
    posterior_rows_kernel<<<blocks_for(row_hi - row_lo), 256, 0, st>>>(d_rows, base, row_lo, row_hi, d_ref, d_group_off,
                                                                     n_groups, k, snp_prior, d_out);
}

void nvbk_fill_status(const BatchDev &B, int32_t *d_status, double *d_ll, int alphabet, cudaStream_t st) {
  if (B.n_reads > 0) fill_status_kernel<<<B.n_reads, 128, 0, st>>>(B, d_status, d_ll, alphabet);
}
