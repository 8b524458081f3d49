// snp3.cu -- the per-position SNP refinement DP (reference dtw.cpp:93-129), scaled linear domain (dp3.cuh).
//
// Task = (read, position i, alternative base).  Lanes of a task: LOADER (streams the stored prefix row `first` from
// HBM and evaluates the emission of base first-1), one PAIR lane per influenced base j = first..last (wobble row on
// band j + model row on band j+1 under the modified sequence, dtw.cpp:103-115), JOIN (the trailing wobble row on
// band `last` -- dtw.cpp:116-123 -- and Node::TotalLikelihood against the stored suffix row last+1).  That is k+2
// lanes; 32/(k+2) tasks share a warp (4 for the 6-mer model).  Every lane evaluates exactly one exp per step and all
// roles run the same instruction stream (dp3.cuh).
#include "dp3.cuh"
#include "kernels.h"

namespace {

// Renormalisation period of the SNP kernel: 16 steps instead of the 8 of the sweeps (dp3.cuh NVB_RENORM_MASK).  A task
// is a chain of k+2 lanes, so stale-mantissa slack compounds over at most k+2 hops: with <= 2 bits per step and hop
// (emission mantissa < 2, one addition) 16 steps stay below 2^(2*16*(k+2)): 2^256 for the 6-mer model, 2^416 at k = 11,
// inside the double range (2^1022) up to k = 29, beyond any k-mer table that fits a device; the sweeps, whose chains
// are 32 lanes long, keep 8.  Measured: 71.1 -> 69.8 ms at 1000 reads (the renormalisation was 6.5 % of the kernel's
// instructions), parity suite and fuzz unchanged (profiles/r02ad).
#ifndef NVB_SNP_RENORM_MASK
#define NVB_SNP_RENORM_MASK 15
#endif

template <int MEL, int MODE>
__global__ void __launch_bounds__(128) snp3_kernel(ModelDev M, BatchDev B, int b0, int b1, int64_t g0, int64_t n_tasks,
                                                   int LT, int TPW, const int64_t *mat_base, const double *pF,
                                                   const int32_t *pX, const double *sF, const int32_t *sX,
                                                   double *out_ll) {
  constexpr bool wobbling = (MODE == NVB_MODE_WOBBLE);
  const unsigned exp_tab = exp_table_init();
  const int wic = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t warp_id = blockIdx.x * (int64_t)(blockDim.x >> 5) + wic;
  const int A = M.alphabet;
  const double C_E2 = 0.1353352832366127;  // exp(-2): the "/ 2" of kmer_model.cpp:60 is "- 2.0" in log space

  const int slot = lane / LT, ri = lane - slot * LT;
  const int64_t task = warp_id * TPW + slot;
  const bool have = slot < TPW && task < n_tasks;

  LaneCfg L;
  lane_cfg_clear(L);
  const double *rowF = nullptr;   // LOADER: prefix row; JOIN: suffix row
  const int32_t *rowX = nullptr;
  const double *sig = B.signal;
  int N = 1, C0 = 0, T = 0;
  double *out = nullptr;

  if (have) {
    const int64_t g = g0 + task / (A - 1);
    const int alt = (int)(task % (A - 1));
    int lo = b0, hi = b1;  // last read with ref_off <= g
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (B.ref_off[mid] <= g) lo = mid; else hi = mid;
    }
    const int b = lo;
    if (!B.flags[b]) {
      ReadView v = read_view(B, b);
      const int n = v.n;
      const int i = (int)(g - B.ref_off[b]);
      const int refbase = v.ref[i];
      const int base = alt + (alt >= refbase ? 1 : 0);
      const int back = M.k - M.central - 1, fwd = M.central;  // dtw.cpp:88-89
      const int first = max(0, i - back), last = min(n - 1, i + fwd);
      const int npairs = last - first + 1;
      N = v.N; sig = v.sig;
      C0 = v.bs[first];
      const int64_t mb = mat_base[b];
      int kmer_at = -1;
      bool hasA = false;
      if (ri == 0) {
        L.role = NVB_ROLE_LOADER;
        L.ms = v.bs[first]; L.me = v.be[first];
        rowF = pF + mb + v.coff[first]; rowX = pX + mb + v.coff[first];
        kmer_at = first > 0 ? first - 1 : first;
      } else if (ri <= npairs) {
        const int j = first + ri - 1;
        L.role = NVB_ROLE_PAIR;
        hasA = wobbling && j > 0;
        if (hasA) { L.ws = v.bs[j]; L.we = v.be[j]; }
        L.ms = v.bs[j + 1]; L.me = v.be[j + 1];
        kmer_at = j;
      } else if (ri == npairs + 1) {
        L.role = NVB_ROLE_JOIN;
        hasA = wobbling && last + 1 < n;
        if (hasA) { L.ws = v.bs[last]; L.we = v.be[last]; }  // band row `last`, not last+1 (dtw.cpp:120-121)
        L.ms = v.bs[last + 1]; L.me = v.be[last + 1];  // band of the closing suffix row
        rowF = sF + mb + v.coff[last + 1]; rowX = sX + mb + v.coff[last + 1];
        kmer_at = last + 1 < n ? last + 1 : last;
        out = out_ll + (B.ref_off[b] + i) * A + base;
        const int endcol = hasA ? L.we : L.me;         // range of the row that is joined
        T = endcol - C0 + ri + 1 + MEL;                // + MEL: the joined cells pass through the B-row delay line
      }
      if (hasA) { L.cm = C_E2; L.abias = 0; }
      if (kmer_at >= 0) {
        const int id = kmer_id(M, v, kmer_at, i, base);  // ModifiedSequence (sequence.cpp:30-38)
        lane_set_emission(L, M.mean[id], M.ac[id], M.mc[id]);
      }
    }
  }
  T = __reduce_max_sync(NVB_FULL, T);  // (a REDUX result is warp-uniform for the compiler as well: uniform loop bounds)

  LaneState<MEL> S;
  lane_reset(S);
  LaneOut res;
  res.f = 0.0; res.E = NVB_EZERO; res.p = 1.0; res.k = 0;
  const bool is_loader = L.role == NVB_ROLE_LOADER, is_join = L.role == NVB_ROLE_JOIN;
  const bool reads_row = is_loader || is_join;
  const bool passes = L.role == NVB_ROLE_PAIR;  // lanes whose B-row cell feeds the next lane
  // Blocks of NVB_SNP_RENORM_MASK + 1 steps with the renormalisation between them: a test inside the step loop made
  // every loop-carried value take a register move per step (the two paths had to meet in the same registers).
  for (int t0 = 0; t0 < T; t0 += NVB_SNP_RENORM_MASK + 1) {
    const int t1 = min(t0 + NVB_SNP_RENORM_MASK + 1, T);
#pragma unroll 1
    for (int t = t0; t < t1; t++) {
      const int c = C0 + (t - ri);
      const double x = __ldg(sig + min(max(c - 1, 0), N - 1));
      LaneOut in = shfl_up_out<MODE>(res);
      double rF = 0.0;
      int rX = NVB_EZERO;
      if (reads_row && c >= L.ms && c <= L.me) {
        rF = __ldg(rowF + (c - L.ms));
        rX = __ldg(rowX + (c - L.ms));
      }
      XD aout;
      // JOIN lanes multiply their A-row cell by the closing suffix cell, every other lane by (1.0, 0)
      lane_step<MEL, MODE, true, false>(L, S, exp_tab, c, x, in, is_join ? rF : 1.0, is_join ? rX : 0, res, aout);
      if (is_loader) {  // the loader's output is the stored prefix row (zero outside its band)
        res.f = rF; res.E = rX;
      } else if (!passes) {
        res.f = 0.0; res.E = NVB_EZERO;
      }
    }
    lane_renorm(S);
  }
  if (is_join) {
    xd_renorm(S.mod);  // canonical mantissa
    *out = log_ext(S.mod.f, S.mod.e);
  }
}

template <int MEL>
void launch_snp3(const ModelDev &M, const BatchDev &B, int wobbling, int b0, int b1, int64_t g0, int64_t n_tasks, int LT,
                 int TPW, const int64_t *mb, const double *pF, const int32_t *pX, const double *sF, const int32_t *sX,
                 double *out, cudaStream_t st) {
  const int warps = 4;
  const int64_t n_warps = (n_tasks + TPW - 1) / TPW;
  const unsigned grid = (unsigned)((n_warps + warps - 1) / warps);
  if (wobbling)
    snp3_kernel<MEL, NVB_MODE_WOBBLE><<<grid, warps * NVB_WARP, 0, st>>>(M, B, b0, b1, g0, n_tasks, LT, TPW, mb, pF, pX,
                                                                         sF, sX, out);
  else
    snp3_kernel<MEL, NVB_MODE_PLAIN><<<grid, warps * NVB_WARP, 0, st>>>(M, B, b0, b1, g0, n_tasks, LT, TPW, mb, pF, pX,
                                                                        sF, sX, out);
}

}  // namespace

int nvbk_snp2(const ModelDev &M, const BatchDev &B, int wobbling, int b0, int b1, int64_t g0, int64_t g1,
              const int64_t *d_mat_base, const double *pF, const int32_t *pX, const double *sF, const int32_t *sX,
              double *d_out_ll, cudaStream_t st) {
  const int LT = M.k + 2;  // LOADER + k pairs + JOIN
  if (LT > NVB_WARP) return -1;
  const int TPW = NVB_WARP / LT;
  const int64_t n_tasks = (g1 - g0) * (M.alphabet - 1);
  if (n_tasks <= 0) return 0;
#define NVB_SNP3(MEL) \
  launch_snp3<MEL>(M, B, wobbling, b0, b1, g0, n_tasks, LT, TPW, d_mat_base, pF, pX, sF, sX, d_out_ll, st)
  switch (B.mel) {
    case 0: NVB_SNP3(0); break;
    case 1: NVB_SNP3(1); break;
    case 2: NVB_SNP3(2); break;
    case 3: NVB_SNP3(3); break;
    case 4: NVB_SNP3(4); break;
    case 5: NVB_SNP3(5); break;
    case 6: NVB_SNP3(6); break;
    default: return -1;
  }
#undef NVB_SNP3
  return 0;
}
