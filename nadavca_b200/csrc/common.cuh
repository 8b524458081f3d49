// common.cuh -- device-side data layout and helpers shared by all kernels of libnadavca_b200.so (sm_100a).
//
// Data layout in HBM (all per batch, CSR over reads; see DESIGN.md "Data layout"):
//   signal   double[sum N]          sig_off[b]   .. sig_off[b+1]
//   ref      int32 [sum n]          ref_off[b]   .. ref_off[b+1]       numeric bases
//   bs, be   int32 [sum (n+1)]      index ref_off[b] + b + j           inclusive band of band-row j = 0..n
//   cell_off int64 [sum (n+2)]      index ref_off[b] + 2b + j          exclusive scan of band widths (j = n+1: total)
//   prefix/suffix matrices: packed band rows, row j of read b at mat_base[b] + cell_off[j] + (c - bs[j])
//   (with transitions the 2n rows interleave band rows i and i+1, see trans_row_off()).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define NVB_WARP 32
#define NVB_FULL 0xffffffffu

enum { NVB_MODE_PLAIN = 0, NVB_MODE_TRANS = 1, NVB_MODE_WOBBLE = 2 };

struct ModelDev {
  int k, central, alphabet;
  int64_t n_kmers;
  const double *mean, *ac, *mc;  // per k-mer tables (kmer_model.cpp:6-14)
  // Padding to 56 bytes: kernels take BatchDev right after ModelDev, and ptxas pairs the constant-bank loads of its
  // fields by their 16-byte alignment.  At 48 bytes the wobbling rotating sweep measured 1 % slower (B200, 1000 W).
  int64_t pad;
};

struct BatchDev {
  int n_reads;
  const double *signal;
  const int64_t *sig_off;
  const int32_t *ref;
  const int64_t *ref_off;
  const int32_t *ctxb;
  const int64_t *ctxb_off;
  const int32_t *ctxa;
  const int64_t *ctxa_off;
  const int32_t *anchors;
  const int64_t *anc_off;
  int bandwidth, mel;
  int32_t *bs, *be;
  int64_t *cell_off;
  int32_t *flags;      // per read NVB_READ_* (bad band)
  int32_t *max_width;  // per read
  const double *row_emis;  // per reference position [mu, ac * S, mc * S, same-mean flags]: Gaussian emission of the unmodified k-mer
                           // there, ac and mc scaled for exp_ext_scaled (dp3.cuh); filled once per batch (band.cu)
};

// Inputs of the batched anchor construction (anchors.cu), CSR over reads.
struct AnchorBatch {
  int n_reads;
  const int32_t *cigar_len;   // operations of every read's CIGAR ...
  const int8_t *cigar_op;     // ... 0 = M, 1 = I, 2 = D, 3 = S
  const int64_t *cigar_off;
  const int64_t *mapped_pos;  // 0-based position of the hit in the contig
  const int32_t *reverse;
  const int8_t *read_seq;     // basecalled bases 0..3 ...
  const int32_t *mapping;     // ... and the sample index of each base (-1: not placed), Read.sequence_to_signal_mapping
  const int64_t *read_off;
  const int32_t *n_signal;    // len(read.normalized_signal)
  const int8_t *genome;       // contig bases 0..3 (4 = other)
  int64_t genome_len;
  int bandwidth;
};

struct ReadView {
  int n, N, nb, na;
  const double *sig;
  const int32_t *ref, *cb, *ca;
  const int32_t *bs, *be;
  const int64_t *coff;
  const double *emis;  // BatchDev::row_emis of this read
};

__device__ __forceinline__ double nvb_neg_inf() { return __longlong_as_double(0xfff0000000000000LL); }

__device__ __forceinline__ ReadView read_view(const BatchDev &B, int b) {
  ReadView v;
  int64_t r0 = B.ref_off[b];
  v.n = (int)(B.ref_off[b + 1] - r0);
  v.N = (int)(B.sig_off[b + 1] - B.sig_off[b]);
  v.nb = (int)(B.ctxb_off[b + 1] - B.ctxb_off[b]);
  v.na = (int)(B.ctxa_off[b + 1] - B.ctxa_off[b]);
  v.sig = B.signal + B.sig_off[b];
  v.ref = B.ref + r0;
  v.cb = B.ctxb + B.ctxb_off[b];
  v.ca = B.ctxa + B.ctxa_off[b];
  v.bs = B.bs + r0 + b;
  v.be = B.be + r0 + b;
  v.coff = B.cell_off + r0 + 2 * (int64_t)b;
  v.emis = B.row_emis + 4 * r0;
  return v;
}

// ExtendedSequence / ModifiedSequence (sequence.cpp:6-38): context ++ reference ++ context, base 0 outside,
// one optional overridden position.
__device__ __forceinline__ int base_at(const ReadView &v, int idx, int mod_pos, int mod_val) {
  if (idx == mod_pos) return mod_val;
  int j = idx + v.nb;
  if (j < 0 || j >= v.nb + v.n + v.na) return 0;
  if (j < v.nb) return v.cb[j];
  if (j < v.nb + v.n) return v.ref[j - v.nb];
  return v.ca[j - v.nb - v.n];
}

// KmerModel::GetKmerId (kmer_model.cpp:22-30)
__device__ __forceinline__ int kmer_id(const ModelDev &M, const ReadView &v, int i, int mod_pos, int mod_val) {
  int id = 0;
  for (int p = i - M.central; p < i - M.central + M.k; p++) id = id * M.alphabet + base_at(v, p, mod_pos, mod_val);
  return id;
}

// Row offset of row rho (0..2n-1) in the transition layout: rows 2i / 2i+1 live on band rows i / i+1.
__device__ __forceinline__ int64_t trans_row_off(const ReadView &v, int rho) {
  int i = rho >> 1;
  if (rho & 1) return 2 * v.coff[i + 1] - v.coff[1];
  return v.coff[i] + v.coff[i + 1] - v.coff[1];
}
