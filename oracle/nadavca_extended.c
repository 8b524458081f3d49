/*
 * nadavca_extended.c -- extended-precision restatement of EstimateLogLikelihoods.   *** TEST INFRASTRUCTURE ***
 *
 * The pinned oracle (nadavca_oracle.c) repeats the reference's double log-space arithmetic operation for operation, so
 * its own rounding error grows with |log-likelihood| (every a + log(1 + exp(b - a)) rounds at the magnitude of a).
 * This file computes the same mathematics -- reference nadavca/dtw/dtw.cpp:37-131 on the model's own double tables
 * (kmer_model.cpp:10-13) -- with an error that does not grow with the magnitude of the values, so that the GPU
 * kernels can be held to an absolute bar on log-likelihood RATIOS.
 *
 * Representation: a value is m * 2^e with a long double (x86 80-bit, 64-bit significand) mantissa m in [0.5, 1) and
 * an int64 exponent e; every product and sum is renormalised, so each operation costs about 2^-64 relative error
 * whatever the value's magnitude, and nothing over- or underflows.  Emissions are the reference's formulas
 * evaluated in long double on the double tables: Gaussian exp(ac - d^2 mc) (kmer_model.cpp:44-52), wobble mixture
 * (e1 + e2) * exp(-2) (kmer_model.cpp:54-62, "/ 2" is "- 2.0" in log space).
 *
 * Only tests/ load this file (through oracle/oracle.py); the product never does.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef struct { long double m; int64_t e; } xv; /* m * 2^e; m in [0.5, 1), or m == 0 for an exact zero */

static const xv XV0 = {0.0L, 0}, XV1 = {0.5L, 1};
static const long double LN2L = 0.693147180559945309417232121458176568L;
/* Cody-Waite split of ln 2: k * LN2_HI is exact for |k| < 2^31, LN2_LO carries the next 64 bits */
static const long double LN2_HI = 0x1.62e42feep-1L, LN2_LO = 0xd1cf79abc9e3b398p-96L;

static inline xv xv_norm(long double m, int64_t e) {
  xv r;
  if (m == 0) return XV0;
  int ex;
  r.m = frexpl(m, &ex);
  r.e = e + ex;
  return r;
}

static inline xv xv_mul(xv a, xv b) {
  if (a.m == 0 || b.m == 0) return XV0;
  return xv_norm(a.m * b.m, a.e + b.e);
}

static inline xv xv_add(xv a, xv b) {
  if (b.m == 0) return a;
  if (a.m == 0) return b;
  if (a.e < b.e) { xv t = a; a = b; b = t; }
  int64_t d = b.e - a.e;
  if (d < -96) return a; /* below half an ulp of a's mantissa */
  return xv_norm(a.m + ldexpl(b.m, (int)d), a.e);
}

/* exp(l) for any finite l: l = k ln2 + r, 0 <= r < ln2 */
static inline xv xv_exp(long double l) {
  long double k = floorl(l / LN2L);
  long double r = (l - k * LN2_HI) - k * LN2_LO;
  return xv_norm(expl(r), (int64_t)k);
}

static inline long double xv_logl(xv a) { return logl(a.m) + (long double)a.e * LN2L; }
static inline double xv_log(xv a) { return a.m == 0 ? -INFINITY : (double)xv_logl(a); }

/* ---- k-mer model: kmer_model.cpp:6-30, the double tables as the reference builds them ------------------------------ */

typedef struct {
  int k, central, alphabet;
  int64_t size;
  double *mean, *ac, *mc;
} nvx_model;

nvx_model *nvx_model_create(int k, int central, int alphabet, const double *mean, const double *sigma, int64_t size) {
  nvx_model *m = (nvx_model *)calloc(1, sizeof(nvx_model));
  m->k = k; m->central = central; m->alphabet = alphabet; m->size = size;
  m->mean = (double *)malloc(sizeof(double) * size);
  m->ac = (double *)malloc(sizeof(double) * size);
  m->mc = (double *)malloc(sizeof(double) * size);
  for (int64_t i = 0; i < size; i++) {
    double s = sigma[i];
    m->mean[i] = mean[i];
    m->ac[i] = log(1 / sqrt(2 * M_PI * s * s)); /* kmer_model.cpp:11 */
    m->mc[i] = 1 / (2 * s * s);                 /* kmer_model.cpp:12 */
  }
  return m;
}

void nvx_model_destroy(nvx_model *m) {
  if (!m) return;
  free(m->mean); free(m->ac); free(m->mc); free(m);
}

/* extended sequence (sequence.cpp:6-38): context_before ++ reference ++ context_after, base 0 outside, optional
 * single-base override (ModifiedSequence) */
typedef struct {
  const int *ref, *before, *after;
  int n, nb, na, mod_pos, mod_val;
} nvx_seq;

static inline int seq_at(const nvx_seq *s, int idx) {
  if (idx == s->mod_pos) return s->mod_val;
  int j = idx + s->nb;
  if (j < 0 || j >= s->nb + s->n + s->na) return 0;
  if (j < s->nb) return s->before[j];
  if (j < s->nb + s->n) return s->ref[j - s->nb];
  return s->after[j - s->nb - s->n];
}

static inline int kmer_id(const nvx_model *m, const nvx_seq *s, int i) { /* kmer_model.cpp:22-30 */
  int id = 0;
  for (int p = i - m->central; p < i - m->central + m->k; p++) id = id * m->alphabet + seq_at(s, p);
  return id;
}

/* One row's emission: Gaussian of k-mer a, or (mix) the wobble mixture of k-mers a and b. */
typedef struct { int mix, a, b; } nvx_emis;

static inline xv gauss(const nvx_model *m, int id, double x) { /* kmer_model.cpp:44-52 in long double */
  long double d = (long double)x - (long double)m->mean[id];
  return xv_exp((long double)m->ac[id] - d * d * (long double)m->mc[id]);
}

static xv emis(const nvx_model *m, const nvx_emis *em, double x) {
  if (!em->mix) return gauss(m, em->a, x);
  static xv e2 = {0.0L, 0};
  if (e2.m == 0) e2 = xv_exp(-2.0L); /* kmer_model.cpp:60 */
  return xv_mul(xv_add(gauss(m, em->a, x), gauss(m, em->b, x)), e2);
}

/* ---- bands: dtw.cpp:7-35 ------------------------------------------------------------------------------------------- */

static void band_bounds(const int *anchors, int n_anchors, int n_signal, int n_ref, int bandwidth, int *starts,
                        int *ends) {
  for (int i = 0; i <= n_ref; i++) { starts[i] = 0; ends[i] = n_signal; }
  for (int a = 0; a < n_anchors; a++) {
    int sig = anchors[2 * a], ref = anchors[2 * a + 1];
    int lo = sig - bandwidth, hi = sig + bandwidth;
    starts[ref] = lo > 0 ? lo : 0;
    ends[ref] = hi < n_signal ? hi : n_signal;
  }
  for (int i = 1; i <= n_ref; i++)
    if (starts[i - 1] > starts[i]) starts[i] = starts[i - 1];
  for (int i = n_ref - 1; i >= 0; i--)
    if (ends[i + 1] < ends[i]) ends[i] = ends[i + 1];
}

/* ---- one banded row: node.cpp:5-37, node_next_row.h:6-61 --------------------------------------------------------- */

typedef struct { int s, e; xv *v; } xrow; /* inclusive [s, e]; v[i - s] */

static inline xv row_at(const xrow *r, int i) { return (i < r->s || i > r->e) ? XV0 : r->v[i - r->s]; }

typedef struct {
  const nvx_model *model;
  const double *signal;
  int n_signal;
  xv *em; /* emission of the row being computed at every signal sample (scratch of n_signal entries) */
} nvx_ctx;

/* emissions of samples [lo, hi] (clipped to the signal) */
static void fill_emis(nvx_ctx *c, const nvx_emis *em, int lo, int hi) {
  if (lo < 0) lo = 0;
  if (hi > c->n_signal - 1) hi = c->n_signal - 1;
  for (int t = lo; t <= hi; t++) c->em[t] = emis(c->model, em, c->signal[t]);
}

static void next_row(nvx_ctx *c, xrow *res, int s, int e, const xrow *pred, const nvx_emis *em, int m, int reverse,
                     xv *storage) {
  res->s = s; res->e = e; res->v = storage;
  for (int i = 0; i <= e - s; i++) storage[i] = XV0;
  if (e < s) return;
  const xv *E = c->em;
  if (!reverse) {
    fill_emis(c, em, (pred->s < s ? pred->s : s) - m - 1, e);
    if (s >= m) { /* node_next_row.h:37-48: the first cell sums every predecessor at least m samples back */
      xv p = XV1;
      for (int i = s; i >= pred->s; i--) {
        if (i < s) p = xv_mul(p, E[i]);
        if (s - i >= m) res->v[0] = xv_add(res->v[0], xv_mul(p, row_at(pred, i)));
      }
    }
    for (int i = (s + 1 > m ? s + 1 : m); i <= e; i++) { /* node_next_row.h:49-58: an m-sample event or a stay */
      xv p = XV1;
      for (int j = i - 1; j >= i - m; j--) p = xv_mul(p, E[j]);
      res->v[i - s] = xv_add(xv_mul(p, row_at(pred, i - m)), xv_mul(E[i - 1], row_at(res, i - 1)));
    }
  } else {
    fill_emis(c, em, s, (pred->e > e ? pred->e : e) + m);
    if (e + m <= c->n_signal) { /* node_next_row.h:13-24: the last cell sums every successor at least m samples on */
      xv p = XV1;
      for (int i = e; i <= pred->e; i++) {
        if (i > e) p = xv_mul(p, E[i - 1]);
        if (i - e >= m) res->v[e - s] = xv_add(res->v[e - s], xv_mul(p, row_at(pred, i)));
      }
    }
    int top = e - 1 < c->n_signal - m ? e - 1 : c->n_signal - m;
    for (int i = top; i >= s; i--) { /* node_next_row.h:25-35 */
      xv p = XV1;
      for (int j = i; j < i + m; j++) p = xv_mul(p, E[j]);
      res->v[i - s] = xv_add(xv_mul(p, row_at(pred, i + m)), xv_mul(E[i], row_at(res, i + 1)));
    }
  }
}

static xv total_likelihood(const xrow *prefix, const xrow *suffix) { /* node.cpp:31-37 */
  xv r = XV0;
  for (int i = prefix->s; i <= prefix->e; i++) r = xv_add(r, xv_mul(prefix->v[i - prefix->s], row_at(suffix, i)));
  return r;
}

static void row_fill(xrow *r, int s, int e, xv fill, xv *storage) {
  r->s = s; r->e = e; r->v = storage;
  for (int i = 0; i <= e - s; i++) storage[i] = fill;
}

/* ---- EstimateLogLikelihoods: dtw.cpp:37-131 -------------------------------------------------------------------------
 * out_ll     n x alphabet log-likelihoods (rounded once to double);
 * out_ratio  n x alphabet log(L[i][b] / L[i][ref_i]), rounded once (NULL to skip);
 * dbg_prefix / dbg_suffix  the stored rows 0..n packed back to back, as log values (NULL to skip);
 * row_dev    n+1 values sum_c P[j][c] S[j][c] / (the same for row n) - 1 (NULL to skip; plain mode only, where that
 *            sum is the same total for every row). */
void nvx_estimate_log_likelihoods(const nvx_model *model, const double *signal, int n_signal, const int *ref, int n_ref,
                                  const int *before, int nb, const int *after, int na, const int *anchors,
                                  int n_anchors, int bandwidth, int m_len, int wobbling, double *out_ll,
                                  double *out_ratio, double *dbg_prefix, double *dbg_suffix, double *row_dev) {
  if (n_ref <= 0) return;
  nvx_seq seq = {ref, before, after, n_ref, nb, na, INT32_MIN, 0};
  const int n = n_ref, A = model->alphabet;
  int *bs = (int *)malloc(sizeof(int) * (n + 1)), *be = (int *)malloc(sizeof(int) * (n + 1));
  band_bounds(anchors, n_anchors, n_signal, n, bandwidth, bs, be);
  int64_t *off = (int64_t *)malloc(sizeof(int64_t) * (n + 2));
  int wmax = 1;
  off[0] = 0;
  for (int r = 0; r <= n; r++) {
    int w = be[r] - bs[r] + 1;
    if (w > wmax) wmax = w;
    off[r + 1] = off[r] + (w > 0 ? w : 0);
  }
  xv *P = (xv *)malloc(sizeof(xv) * (off[n + 1] + 1)), *S = (xv *)malloc(sizeof(xv) * (off[n + 1] + 1));
  xrow *Pr = (xrow *)calloc(n + 1, sizeof(xrow)), *Sr = (xrow *)calloc(n + 1, sizeof(xrow));
  xv *ta = (xv *)malloc(sizeof(xv) * wmax), *tb = (xv *)malloc(sizeof(xv) * wmax);
  nvx_ctx c = {model, signal, n_signal, (xv *)malloc(sizeof(xv) * (n_signal > 0 ? n_signal : 1))};

  row_fill(&Pr[0], bs[0], be[0], XV1, P); /* dtw.cpp:50 */
  for (int i = 0; i < n; i++) {          /* dtw.cpp:51-64 */
    xrow pred = Pr[i], wob;
    if (i > 0 && wobbling) {
      nvx_emis mix = {1, kmer_id(model, &seq, i - 1), kmer_id(model, &seq, i)};
      next_row(&c, &wob, bs[i], be[i], &pred, &mix, 0, 0, ta);
      pred = wob;
    }
    nvx_emis g = {0, kmer_id(model, &seq, i), 0};
    next_row(&c, &Pr[i + 1], bs[i + 1], be[i + 1], &pred, &g, m_len, 0, P + off[i + 1]);
  }
  row_fill(&Sr[n], bs[n], be[n], XV1, S + off[n]); /* dtw.cpp:66-67 */
  for (int i = n; i > 0; i--) {                     /* dtw.cpp:68-81 */
    xrow pred = Sr[i], wob;
    if (i < n && wobbling) {
      nvx_emis mix = {1, kmer_id(model, &seq, i), kmer_id(model, &seq, i - 1)};
      next_row(&c, &wob, bs[i], be[i], &pred, &mix, 0, 1, ta);
      pred = wob;
    }
    nvx_emis g = {0, kmer_id(model, &seq, i - 1), 0};
    next_row(&c, &Sr[i - 1], bs[i - 1], be[i - 1], &pred, &g, m_len, 1, S + off[i - 1]);
  }
  if (dbg_prefix) for (int64_t x = 0; x < off[n + 1]; x++) dbg_prefix[x] = xv_log(P[x]);
  if (dbg_suffix) for (int64_t x = 0; x < off[n + 1]; x++) dbg_suffix[x] = xv_log(S[x]);

  xv no_snp = total_likelihood(&Pr[n], &Sr[n]); /* dtw.cpp:83-85 */
  if (row_dev) {
    for (int j = 0; j <= n; j++) {
      xv t = total_likelihood(&Pr[j], &Sr[j]);
      row_dev[j] = (t.m == 0 || no_snp.m == 0) ? NAN : (double)(ldexpl(t.m / no_snp.m, (int)(t.e - no_snp.e)) - 1.0L);
    }
  }
  const int back = model->k - model->central - 1, fwd = model->central; /* dtw.cpp:88-89 */
  for (int i = 0; i < n; i++) { /* dtw.cpp:93-129 */
    const int first = i - back > 0 ? i - back : 0;
    const int last = i + fwd < n - 1 ? i + fwd : n - 1;
    const int rb = seq_at(&seq, i);
    for (int base = 0; base < A; base++) {
      xv L = no_snp;
      if (base != rb) {
        nvx_seq mod = seq;
        mod.mod_pos = i; mod.mod_val = base;
        xrow cur = Pr[first], nxt;
        xv *buf = ta, *other = tb;
        for (int j = first; j <= last; j++) {
          if (j > 0 && wobbling) {
            nvx_emis mix = {1, kmer_id(model, &mod, j - 1), kmer_id(model, &mod, j)};
            next_row(&c, &nxt, bs[j], be[j], &cur, &mix, 0, 0, buf);
            cur = nxt; { xv *t = buf; buf = other; other = t; }
          }
          nvx_emis g = {0, kmer_id(model, &mod, j), 0};
          next_row(&c, &nxt, bs[j + 1], be[j + 1], &cur, &g, m_len, 0, buf);
          cur = nxt; { xv *t = buf; buf = other; other = t; }
        }
        if (last + 1 < n && wobbling) { /* dtw.cpp:116-123: band row `last`, not last+1 */
          nvx_emis mix = {1, kmer_id(model, &mod, last), kmer_id(model, &mod, last + 1)};
          next_row(&c, &nxt, bs[last], be[last], &cur, &mix, 0, 0, buf);
          cur = nxt;
        }
        L = total_likelihood(&cur, &Sr[last + 1]);
      }
      out_ll[i * A + base] = xv_log(L);
      if (out_ratio) {
        if (L.m == 0 || no_snp.m == 0)
          out_ratio[i * A + base] = (L.m == 0) ? -INFINITY : NAN;
        else
          out_ratio[i * A + base] = (double)(logl(L.m / no_snp.m) + (long double)(L.e - no_snp.e) * LN2L);
      }
    }
  }
  free(c.em); free(ta); free(tb); free(Pr); free(Sr); free(P); free(S); free(off); free(bs); free(be);
}
