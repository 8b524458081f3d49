"""The GPU's SNP log-likelihood ratios, stored rows, chunks, consensus sums and posteriors against extended precision.

The pinned oracle works in double log space; its error grows with |LL| (1e3..1e4 per read), so raw log-likelihoods
can only be held to rtol 1e-9, which lets a kernel lose about 1e-5 of a read's probability mass unnoticed
(tests/test_extended_reference.py::test_old_bar_is_blind).  Here the truth is oracle/nadavca_extended.c (mantissa +
int64 exponent, about 2^-64 per operation whatever the magnitude), and the bars are absolute, from an error model:

  a. every ratio LL[i][b] - LL[i][ref_i] and the no-SNP total: |GPU - truth| <= 64 eps (N + n) + 2 E, eps = 2^-52:
     a few roundings per DP step along a path of N + n steps, plus E = `exponent_term`, the rounding of the Gaussian
     exponent ac - d^2 mc in double summed along a path.  The reference evaluates that exponent in double too
     (kmer_model.cpp:44-52); E is below 64 eps (N + n) on ordinary reads and 74-97 times it on the outlier bursts of
     the dynamic-range cases.  Finite exactly where the truth is;
  b. stored rows (locator): the zero pattern equals the truth's; cells holding >= 2^-200 of the read's posterior mass
     within 64 eps (row + column depth) in log;
  c. chunk_values_kernel: bit-exact against numpy on the GPU's own raw LLs;
  d. scatter_add_rows_kernel: |GPU - fsum| <= (m - 1) eps sum|x| for m summands (any summation order), coverage exact;
  e. posterior_rows_kernel, directly and through ProbabilityEstimator._compute_posterior: rtol 1e-13 against 50-digit
     mpmath on the GPU's own input rows; 0/0 rows of the reference's double arithmetic are NaN; a halo slice is
     bit-identical to the unsliced call;
  f. ProbabilityEstimator.estimate_probabilities, consensus and independent, against extended ratios -> long double
     chunks -> fsum -> 50-digit posterior: rtol 1e-8 on probabilities >= 1e-12, 1e-15 below; coverage exact.

Every GPU test prints the worst error / bar ratio per case; part a also prints the error and E against the base term
64 eps (N + n) alone.
"""
import math
import os

import numpy as np
import pytest

from test_extended_reference import full_size_inputs

EPS = 2.0 ** -52
LL_BAR = 64  # the bar is LL_BAR * eps * (N + n)


# ---- cases -----------------------------------------------------------------------------------------------------------

class XCase:
    """A batch of reads under one model for part a/b: reads are (signal, reference, ctx_before, ctx_after, anchors)."""

    def __init__(self, name, model_key, bw, mel, reads, schedules=(None,), limit=0, rows=False):
        self.name, self.model_key, self.bw, self.mel, self.reads = name, model_key, bw, mel, reads
        self.schedules, self.limit, self.rows = tuple(schedules), limit, rows


def _model_arrays(key):
    if key == 'default':
        from conftest import ROOT
        from nadavca_b200.kmer_model import KmerModel
        km = KmerModel.load_from_hdf5(os.path.join(ROOT, 'nadavca_b200', 'default', 'kmer_model.hdf5'))
        return km.get_k(), km.get_central_position(), km.mean, km.sigma
    from test_gpu_kernel_edges import model_arrays
    k, cp, seed, lo, hi = key
    mean, sigma = model_arrays(k, seed, lo, hi)
    return k, cp, mean, sigma


def full_size_cases():
    """8 seeded full-size reads of the shipped 6-mer model, both strands, bandwidth 150 and 30."""
    out = []
    for bw in (150, 30):
        reads = []
        for i in range(4):
            c = full_size_inputs(10 + i, bw, strand='+-'[i % 2])
            reads.append(c[2:7])
        out.append(XCase('full-size bw %d' % bw, 'default', bw, 2, reads, rows=True))
    return out


def narrow_cases():
    """Reads whose band is so narrow against the anchor jitter that band-edge columns carry real posterior mass
    (test_narrow_cases_have_edge_mass checks >= 1e-3 of some row's mass on the truth)."""
    reads = [full_size_inputs(40 + i, 8, strand='+-'[i % 2], n_bases=300, jitter=10)[2:7] for i in range(4)]
    return [XCase('narrow bw 8', 'default', 8, 2, reads, schedules=(None, 'r', 's'), rows=True)]


def edge_cases(sm_count):
    """The dispatch-threshold table of test_gpu_kernel_edges.py (estimate ops)."""
    from test_gpu_kernel_edges import all_cases
    return [XCase(c.name, c.model.key, c.bw, c.mel, c.reads, c.schedules, c.limit) for c in all_cases(sm_count)]


# ---- truth in a pool -------------------------------------------------------------------------------------------------

_WORKER = {}


def _truth_job(task):
    from oracle import oracle as orc
    key, read, bw, mel, wob, rows = task
    if key not in _WORKER:
        k, cp, mean, sigma = _model_arrays(key)
        if len(_WORKER) >= 3:
            _WORKER.clear()
        _WORKER[key] = orc.ExtendedModel(k, cp, 4, mean, sigma)
    sig, ref, cb, ca, anc = read
    return orc.estimate_log_likelihoods_extended(sig, ref, cb, ca, anc, bw, mel, _WORKER[key], wob, rows=rows)


@pytest.fixture(scope='module')
def pool():
    import multiprocessing as mp
    p = mp.get_context('spawn').Pool(min(os.cpu_count() or 1, 48))
    yield p
    p.terminate()


def _edge_mass(truth):
    """Per row of a plain-mode truth: share of the row's posterior mass in its two band-edge columns."""
    bs, be = truth['bs'], truth['be']
    w = (be - bs + 1).astype(np.int64)
    off = np.concatenate([[0], np.cumsum(w)])
    total = truth['ll'][0].max()  # every entry of row 0 that is not a SNP is the no-SNP total; the max is >= it
    tot = np.log(np.sum(np.exp(truth['prefix'][off[-2]:off[-1]] + truth['suffix'][off[-2]:off[-1]] - total))) + total
    out = []
    for j in range(len(w)):
        p = truth['prefix'][off[j]:off[j + 1]] + truth['suffix'][off[j]:off[j + 1]] - tot
        out.append(float(np.exp(p[0]) + (np.exp(p[-1]) if len(p) > 1 else 0.0)))
    return np.array(out)


def test_narrow_cases_have_edge_mass():
    """The narrow-band reads keep their teeth: in each of them some band row has >= 1e-3 of its posterior mass in its
    edge columns (computed from the extended truth, plain mode)."""
    from oracle import oracle as orc
    k, cp, mean, sigma = _model_arrays('default')
    xm = orc.ExtendedModel(k, cp, 4, mean, sigma)
    c = narrow_cases()[0]
    for r in c.reads:
        t = orc.estimate_log_likelihoods_extended(*r, c.bw, c.mel, xm, False, rows=True)
        assert _edge_mass(t).max() >= 1e-3, _edge_mass(t).max()


# ---- a / b: log-likelihood ratios and stored rows --------------------------------------------------------------------

def exponent_term(k, cp, mean, sigma, read, bw):
    """eps * sum over samples t of max |l| over the band rows that can emit t, where l = ac - d^2 mc is the Gaussian
    exponent (kmer_model.cpp:44-52).  The kernels round l in double (dp3.cuh lane_step: fma(-(d*d), mc, ac) on
    constants scaled by 256/ln 2), as the reference does, so each emission carries a relative error of about eps |l|;
    this sums that over a path (absolute, in log units)."""
    from oracle import oracle as orc
    from test_gpu_kernel_edges import kmer_levels

    class M:
        pass
    m = M()
    m.k, m.cp, m.mean, m.sigma = k, cp, mean, sigma
    sig, ref, _, _, anc = read
    mu, sd = kmer_levels(m, ref)
    ac = np.log(1 / np.sqrt(2 * np.pi * sd * sd))
    mc = 1 / (2 * sd * sd)
    bs, be = orc.band_bounds(anc, len(sig), len(ref), bw)
    a = np.zeros(len(sig))
    for j in range(len(ref)):  # row j emits the samples of its cells and of the cells of row j + 1
        lo, hi = max(int(min(bs[j], bs[j + 1])) - 8, 0), min(int(be[j + 1]), len(sig))
        x = sig[lo:hi]
        a[lo:hi] = np.maximum(a[lo:hi], np.abs(ac[j] - (x - mu[j]) ** 2 * mc[j]))
    return EPS * float(a.sum())


def ll_bar(N, n, term):
    """The error model of part a: a few roundings per DP step along a path of N + n steps, plus twice the exponent
    rounding `exponent_term` (d*d, the scaled mc and the fma each round once in dp3.cuh)."""
    return LL_BAR * EPS * (N + n) + 2 * term


def _check_read(res, truth, N, n, ref, term):
    """-> (worst err/bar over ratios, worst over no-SNP total, worst err / (64 eps (N + n)), message or None)."""
    bar = ll_bar(N, n, term)
    fin = np.isfinite(truth['ll'])
    if not np.array_equal(np.isfinite(res), fin):
        bad = np.argwhere(np.isfinite(res) != fin)[0]
        return np.inf, np.inf, np.inf, 'finite pattern differs first at (%d, %d)' % tuple(bad)
    tot_err = abs(res[0, ref[0]] - truth['ll'][0, ref[0]]) / bar if fin[0, ref[0]] else 0.0
    rows = np.arange(n)
    gr = res - res[rows, ref][:, None]
    m = fin & fin[rows, ref][:, None]
    err = np.abs(gr[m] - truth['ratio'][m]) / bar if m.any() else np.zeros(1)
    worst = float(err.max())
    base = max(worst, tot_err) * bar / (LL_BAR * EPS * (N + n))
    msg = None
    if worst > 1 or tot_err > 1:
        idx = np.argwhere(m)[int(np.argmax(err))]
        msg = 'ratio err/bar %.3g at (%d, %d), total err/bar %.3g (bar %.2e)' % (worst, idx[0], idx[1], tot_err, bar)
    return worst, float(tot_err), base, msg


def _check_rows(batch, ri, truth, N, n):
    """Stored rows of read ri against the truth: the zero pattern of every cell, and the log value of every cell that
    holds >= 2^-200 of the read's mass within 64 eps (row + column depth).  -> (worst err/bar, message or None)."""
    bs, be = truth['bs'], truth['be']
    w = (be - bs + 1).astype(np.int64)
    rows_of = np.repeat(np.arange(n + 1), w)
    cols_of = np.concatenate([np.arange(s, e + 1) for s, e in zip(bs, be)])
    tot = truth['ll'][0].max()
    tot = np.log(np.sum(np.exp(truth['prefix'][-w[-1]:] + truth['suffix'][-w[-1]:] - tot))) + tot
    mass = truth['prefix'] + truth['suffix'] - tot
    worst = 0.0
    for plane, name in ((0, 'prefix'), (1, 'suffix')):
        got = batch.debug_rows(ri, plane)
        want = truth[name]
        z = np.isneginf(want)
        if not np.array_equal(np.isneginf(got), z):
            c = int(np.argmax(np.isneginf(got) != z))
            return np.inf, 'zero pattern differs first at row %d column %d plane %s' % (rows_of[c], cols_of[c], name)
        depth = (rows_of + cols_of) if plane == 0 else ((n - rows_of) + (N - cols_of))
        sel = (mass >= -200 * math.log(2)) & ~z
        err = np.abs(got[sel] - want[sel]) / (LL_BAR * EPS * np.maximum(depth[sel], 1))
        if err.size:
            worst = max(worst, float(err.max()))
            if err.max() > 1:
                c = np.flatnonzero(sel)[int(np.argmax(err > 1))]
                return worst, 'cell differs first at row %d column %d plane %s: %.17g vs %.17g' % (
                    rows_of[c], cols_of[c], name, got[c], want[c])
    return worst, None


@pytest.mark.gpu
def test_log_likelihood_ratios_match_extended(lib_built, pool):
    """Part a (and b for the full-size and narrow reads): every case, both modes, every sweep schedule of the case."""
    import time
    import torch
    from nadavca_b200 import dtw
    t0 = time.time()
    sm_count = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    cases = full_size_cases() + narrow_cases() + edge_cases(sm_count)
    jobs = []
    for ci, c in enumerate(cases):
        for ri, r in enumerate(c.reads):
            for wob in (True, False):
                jobs.append((len(r[0]) * len(r[1]), (ci, ri, wob), (c.model_key, r, c.bw, c.mel, wob, c.rows)))
    jobs.sort(key=lambda j: -j[0])
    pending = {key: pool.apply_async(_truth_job, (task,)) for _, key, task in jobs}
    failures = []
    overall = {'ratio': 0.0, 'total': 0.0, 'rows': 0.0, 'base': 0.0}
    for ci, c in enumerate(cases):
        k, cp, mean, sigma = _model_arrays(c.model_key)
        gm = dtw.KmerModel(k, cp, 4, mean, sigma)
        lists = [[r[i] for r in c.reads] for i in range(5)]
        worst = {'ratio': 0.0, 'total': 0.0, 'rows': 0.0, 'base': 0.0}
        terms = [exponent_term(k, cp, mean, sigma, r, c.bw) for r in c.reads]
        term_share = max(t / (LL_BAR * EPS * (len(r[0]) + len(r[1]))) for t, r in zip(terms, c.reads))
        try:
            for sched in c.schedules:
                dtw.set_sweep_schedule(sched)
                with dtw.Batch(gm, *lists, c.bw, c.mel, workspace_limit=c.limit) as batch:
                    for wob in (True, False):
                        batch.estimate(wob)
                        ll, status = batch.log_likelihoods()
                        for ri, r in enumerate(c.reads):
                            truth = pending[(ci, ri, wob)].get(timeout=3000)
                            N, n = len(r[0]), len(r[1])
                            where = '%s [%s] %s read %d' % (c.name, sched or 'auto', 'wobble' if wob else 'plain', ri)
                            if status[ri] != 0:
                                failures.append('%s: status %d' % (where, status[ri]))
                                continue
                            wr, wt, wb, msg = _check_read(ll[ri], truth, N, n, r[1], terms[ri])
                            worst['ratio'] = max(worst['ratio'], wr)
                            worst['total'] = max(worst['total'], wt)
                            worst['base'] = max(worst['base'], wb)
                            if msg:
                                failures.append('%s: %s' % (where, msg))
                            if c.rows:
                                wrow, msg = _check_rows(batch, ri, truth, N, n)
                                worst['rows'] = max(worst['rows'], wrow)
                                if msg:
                                    failures.append('%s: rows: %s' % (where, msg))
        finally:
            dtw.set_sweep_schedule(None)
        for key in overall:
            overall[key] = max(overall[key], worst[key])
        print('%-28s worst err/bar: ratio %.2e  no-SNP total %.2e%s | err / 64 eps (N + n) %.2e, exponent term / '
              '64 eps (N + n) %.2f' % (c.name, worst['ratio'], worst['total'],
                                       '  stored rows %.2e' % worst['rows'] if c.rows else '', worst['base'],
                                       term_share))
    print('extended LL: %d cases, worst err/bar ratio %.2e total %.2e rows %.2e (err / 64 eps (N + n) %.2e), %.0f s'
          % (len(cases), overall['ratio'], overall['total'], overall['rows'], overall['base'], time.time() - t0))
    assert not failures, '\n'.join(failures[:40])


# ---- c / d: chunk values and consensus sums --------------------------------------------------------------------------

def _glue_batch():
    """64 short reads of a 3-mer model, one of a single base, two with an empty band row (NVB_READ_BAD_BAND)."""
    from test_gpu_kernel_edges import Model, make_read
    rng = np.random.default_rng(31)
    m = Model(3, 1, 500)
    reads = [make_read(rng, m, int(rng.integers(20, 40)), 10, 2, spacing=5) for _ in range(61)]
    reads.insert(5, make_read(rng, m, 1, 10, 2, spacing=5))
    for pos in (17, 40):
        sig, ref, cb, ca, _ = make_read(rng, m, 20, 10, 2, spacing=5)
        reads.insert(pos, (sig, ref, cb, ca, np.array([[60, 3], [5, 5]])))  # rows 3..4 end before they start
    return m, reads


@pytest.mark.gpu
def test_chunk_values_and_scatter_add_rows(lib_built):
    """Part c: chunk_values_kernel bit-exact against numpy on the GPU's own raw LLs -- both strands, a read of one
    base, failed reads inside the batch, normalization_event_length 10 and 7.3.
    Part d: scatter_add_rows_kernel over up to 64 overlapping reads (some with dest -1, the failed ones skipped):
    |GPU - fsum| <= (m - 1) eps sum|x| per entry, coverage exact."""
    import torch
    from nadavca_b200 import dtw
    m, reads = _glue_batch()
    rng = np.random.default_rng(32)
    gm = dtw.KmerModel(m.k, m.cp, 4, m.mean, m.sigma)
    lists = [[r[i] for r in reads] for i in range(5)]
    worst_d = 0.0
    with dtw.Batch(gm, *lists, 10, 2) as batch:
        batch.estimate(True)
        ll, status = batch.log_likelihoods()
        assert status[17] == status[40] == 2 and (np.delete(status, [17, 40]) == 0).all(), status
        total = batch.pack.total_reference
        for nel in (10.0, 7.3):
            reverse = rng.integers(0, 2, size=len(reads)).astype(np.int32)
            d_chunks = torch.empty((total, 4), dtype=torch.float64, device='cuda')
            batch.chunk_values(reverse, nel, d_chunks.data_ptr())
            got = d_chunks.cpu().numpy()
            off = batch.pack.reference_off
            for i, r in enumerate(reads):
                x = ll[i]
                want = (x - x[0, int(r[1][0])]) / nel
                if reverse[i]:
                    want = want[::-1, ::-1]
                assert np.array_equal(got[off[i]:off[i + 1]], want, equal_nan=True), 'chunk of read %d (nel %g)' % (
                    i, nel)
            # consensus rows: every read starts within 12 rows of the origin, so up to 64 overlap
            dest = rng.integers(0, 12, size=len(reads)).astype(np.int64)
            dest[rng.choice(len(reads), 6, replace=False)] = -1
            rows_n = int(max(dest[i] + len(r[1]) for i, r in enumerate(reads)))
            d_rows = torch.zeros((rows_n, 5), dtype=torch.float64, device='cuda')
            batch.scatter_add_rows(d_chunks.data_ptr(), dest, d_rows.data_ptr())
            rows = d_rows.cpu().numpy()
            contrib = [[[] for _ in range(4)] for _ in range(rows_n)]
            cov = np.zeros(rows_n)
            for i, r in enumerate(reads):
                if dest[i] < 0 or status[i] != 0:
                    continue
                for p in range(len(r[1])):
                    cov[dest[i] + p] += 1
                    for j in range(4):
                        contrib[dest[i] + p][j].append(got[off[i] + p, j])
            assert np.array_equal(rows[:, 4], cov), 'coverage'
            assert cov.max() >= 40
            for p in range(rows_n):
                for j in range(4):
                    xs = contrib[p][j]
                    if not xs:
                        assert rows[p, j] == 0.0
                        continue
                    want = math.fsum(xs)
                    bound = (len(xs) - 1) * EPS * math.fsum(abs(v) for v in xs)
                    err = abs(rows[p, j] - want)
                    assert err <= bound, 'row %d column %d: %.17g vs fsum %.17g (bound %.3g)' % (p, j, rows[p, j],
                                                                                                 want, bound)
                    if bound > 0:
                        worst_d = max(worst_d, err / bound)
    print('chunk_values bit-exact; scatter_add_rows worst err/bar %.2e (coverage up to %d)' % (worst_d, cov.max()))


# ---- e: posterior ----------------------------------------------------------------------------------------------------

def _posterior_inputs(k, seed):
    """Groups of lengths 1, k-1, k, 2k-1, 2k and 60; entries like summed chunk values (reference entries 0, the others
    a few nats either way), reference code 4 at some positions, and windows whose maximum is a neighbour's reference
    entry 800 nats above every summed term (0/0 rows of the reference's double arithmetic)."""
    rng = np.random.default_rng(seed)
    lens = [x for x in (1, k - 1, k, 2 * k - 1, 2 * k, 60) if x > 0]
    total = sum(lens)
    group_off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    ref = rng.integers(0, 4, size=total).astype(np.int8)
    ref[rng.choice(total, max(2, total // 15), replace=False)] = 4
    ll = rng.normal(0, 6, size=(total, 4))
    ll[np.arange(total), np.minimum(ref, 3)] = np.where(ref < 4, 0.0, ll[np.arange(total), np.minimum(ref, 3)])
    big = group_off[-2] + 30  # inside the long group: a towering reference entry
    ref[big] = 1
    ll[big] = [-3.0, 800.0, -2.0, -4.0]
    cov = rng.integers(1, 9, size=total).astype(np.float64)
    return ll, ref, group_off, cov


def _mp_posterior(ll, ref, group_off, k, prior):
    import mpmath
    mpmath.mp.dps = 50
    out = np.zeros(ll.shape)
    E = [[mpmath.exp(mpmath.mpf(float(x))) for x in row] for row in ll]  # every term is exp of one entry
    for g in range(len(group_off) - 1):
        gs, ge = int(group_off[g]), int(group_off[g + 1])
        L = ge - gs
        for i in range(L):
            cs, ce = max(0, i - k + 1), min(i + k, L)
            c = mpmath.mpf(3)
            p1, p2 = 1 - mpmath.mpf(prior), mpmath.mpf(prior) / c
            snp = 1 / (p1 / p2 + (1 - (ce - cs - 1)) * c)
            nonsnp = 1 - snp * c
            rb = int(ref[gs + i])
            terms = []
            for j in range(4):
                v = E[gs + i][j] * (nonsnp if j == rb else snp)
                if j == rb:
                    for i2 in range(cs, ce):
                        if i2 == i:
                            continue
                        for j2 in range(4):
                            if j2 != int(ref[gs + i2]):
                                v += E[gs + i2][j2] * snp
                terms.append(v)
            s = mpmath.fsum(terms)
            out[gs + i] = [float(t / s) for t in terms]
    return out


def _nan_rows(ll, ref, group_off, k, prior):
    """Rows where the reference's double arithmetic divides 0 by 0 (oracle.OracleEstimator.compute_posterior)."""
    import warnings
    from oracle import oracle as orc

    class K:
        def get_k(self):
            return k
    est = orc.OracleEstimator(K(), None, {'snp_prior_probability': prior})
    letters = np.array(list('ACGTN'))
    out = []
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        for g in range(len(group_off) - 1):
            gs, ge = int(group_off[g]), int(group_off[g + 1])
            out.append(np.isnan(est.compute_posterior(ll[gs:ge], letters[ref[gs:ge]])).any(axis=1))
    return np.concatenate(out)


@pytest.mark.gpu
def test_posterior_rows_match_mpmath(lib_built):
    """Part e: posterior_rows_kernel, called directly and through ProbabilityEstimator._compute_posterior once per
    group, at k 1, 2, 6, 11 and snp_prior 0.001, 0.3 against 50-digit mpmath, rtol 1e-13 (atol 1e-290 for
    probabilities the double exp leaves subnormal); the 0/0 rows NaN.  Halo slices [row_lo, row_hi) -- every group
    boundary and seeded random ones -- from a buffer that starts at row_lo - (k-1) (the group start when row_lo opens
    one) and is NaN outside the rows the window can reach: bit-identical to the unsliced call, coverage column
    included."""
    import torch
    from nadavca_b200 import dtw
    from nadavca_b200.estimator import ProbabilityEstimator
    dev = torch.cuda.current_device()
    worst = 0.0
    nan_rows_seen = 0
    for k in (1, 2, 6, 11):
        for prior in (0.001, 0.3):
            ll, ref, goff, cov = _posterior_inputs(k, 100 * k + int(prior * 1000))
            total = len(ref)
            truth = _mp_posterior(ll, ref, goff, k, prior)
            nan_rows = _nan_rows(ll, ref, goff, k, prior)
            nan_rows_seen += int(nan_rows.sum())
            # _compute_posterior reads only k and the device of its model: constant tables, no model on the device
            km = dtw.KmerModel(k, 0, 4, np.zeros(4 ** k), np.ones(4 ** k), device=dev)
            est = ProbabilityEstimator(km, None, dict(E2E_CONFIG, snp_prior_probability=prior))
            p4 = np.concatenate([est._compute_posterior(ll[gs:ge], ref[gs:ge]) for gs, ge in zip(goff[:-1], goff[1:])])
            d_ref = torch.as_tensor(ref, device='cuda')
            d_goff = torch.as_tensor(goff, device='cuda')
            rows = torch.as_tensor(np.concatenate([ll, cov[:, None]], axis=1), device='cuda')
            full = torch.empty((total, 5), dtype=torch.float64, device='cuda')
            dtw.posterior_rows(dev, rows.data_ptr(), 0, 0, total, d_ref.data_ptr(), d_goff.data_ptr(), len(goff) - 1,
                               k, prior, full.data_ptr())
            torch.cuda.synchronize()
            p5 = full.cpu().numpy()
            assert np.array_equal(p5[:, 4], cov)
            for got, name in ((p4, '_compute_posterior'), (p5[:, :4], 'posterior_rows')):
                assert np.array_equal(np.isnan(got).any(axis=1), nan_rows), '%s k %d prior %g: NaN rows' % (name, k,
                                                                                                             prior)
                ok = ~nan_rows
                err = np.abs(got[ok] - truth[ok])
                tol = 1e-13 * np.abs(truth[ok]) + 1e-290
                assert (err <= tol).all(), '%s k %d prior %g: row %d' % (name, k, prior,
                                                                         np.flatnonzero(ok)[np.argwhere(err > tol)[0][0]])
                worst = max(worst, float((err / tol).max()))
            # halo slices
            rng = np.random.default_rng(k)
            cuts = sorted(set(goff.tolist()))
            slices = [(a, b) for a, b in zip(cuts[:-1], cuts[1:])]
            slices += [(int(g), min(total, int(g) + 3)) for g in goff[1:-1]]
            slices += [(max(0, int(g) - 2), min(total, int(g) + 2)) for g in goff[1:-1]]
            for _ in range(30):
                a = int(rng.integers(0, total))
                slices.append((a, int(rng.integers(a + 1, total + 1))))
            full_np = p5
            for lo, hi in slices:
                base = lo if lo in goff else max(0, lo - (k - 1))
                top = min(total, hi + k - 1)
                local = np.full((top - base, 5), np.nan)
                keep_lo = max(base, lo - (k - 1))
                local[keep_lo - base:] = np.concatenate([ll, cov[:, None]], axis=1)[keep_lo:top]
                d_local = torch.as_tensor(local, device='cuda')
                o = torch.empty((hi - lo, 5), dtype=torch.float64, device='cuda')
                dtw.posterior_rows(dev, d_local.data_ptr(), base, lo, hi, d_ref.data_ptr(), d_goff.data_ptr(),
                                   len(goff) - 1, k, prior, o.data_ptr())
                got = o.cpu().numpy()
                assert np.array_equal(got.view(np.int64), full_np[lo:hi].view(np.int64)), \
                    'k %d prior %g: slice [%d, %d) base %d differs from the unsliced call' % (k, prior, lo, hi, base)
    assert nan_rows_seen > 0
    print('posterior: worst err/tol %.2e over k 1/2/6/11, priors 0.001/0.3; %d 0/0 rows NaN; halo slices bit-exact' % (
        worst, nan_rows_seen))


# ---- f: end to end ---------------------------------------------------------------------------------------------------

E2E_CONFIG = dict(bandwidth=30, snp_prior_probability=0.001, min_event_length=2, model_wobbling=True,
                  model_transitions=True, tweak_signal_normalization=False, normalization_event_length=10)


def _e2e_reads():
    """16 full-size reads of the shipped 6-mer model on an 8 kb synthetic genome, alternating strands, so they overlap
    about four deep; normalised on the host (the tweak is off, so these are the signals the DP sees)."""
    import copy
    from conftest import ROOT
    from nadavca_b200 import synthetic
    from nadavca_b200.kmer_model import KmerModel
    from nadavca_b200.read import Read
    km = KmerModel.load_from_hdf5(os.path.join(ROOT, 'nadavca_b200', 'default', 'kmer_model.hdf5'))
    genome = synthetic.make_genome(8000, seed=21)
    reads = [synthetic.make_read(genome, km, 200 + i, bandwidth=E2E_CONFIG['bandwidth'], strand='+-'[i % 2])
             for i in range(16)]
    Read.normalize_reads(reads)
    return km, genome, reads, [copy.deepcopy(r) for r in reads]


def _e2e_inputs(km, genome, read):
    """DP inputs of one read as estimator.py:59-110 builds them (oracle glue), plus its reference range and strand."""
    from nadavca_b200 import synthetic
    from oracle import oracle as orc
    bw = E2E_CONFIG['bandwidth']
    apx = synthetic.SyntheticAligner(genome).get_signal_alignment(read, bw)
    s_ref, e_ref = apx.reference_range
    part = genome[s_ref:e_ref]
    if apx.reverse_complement:
        part = orc.reverse_complement(part)
    k, cp = km.get_k(), km.get_central_position()
    start, end = apx.read_sequence_range
    s0, e0 = apx.signal_range
    dp = (np.asarray(read.normalized_signal[s0:e0], dtype=np.float64), orc.to_numerical(part),
          orc.to_numerical(read.sequence[start - cp:start]), orc.to_numerical(read.sequence[end:end + k - cp - 1]),
          np.asarray(apx.alignment))
    return dp, (s_ref, e_ref), bool(apx.reverse_complement)


def _truth_chunk(ratio, reverse):
    """estimator.py:45-47,111-119 on the extended ratios: L[i][b] / L[0][ref_0] is the ratio of row i (every row's
    reference entry is the same no-SNP total), divided by normalization_event_length in long double."""
    v = np.asarray(ratio, dtype=np.longdouble) / np.longdouble(E2E_CONFIG['normalization_event_length'])
    return v[::-1, ::-1] if reverse else v


@pytest.mark.gpu
def test_end_to_end_probabilities_match_extended(lib_built, pool):
    """Part f: ProbabilityEstimator.estimate_probabilities, consensus and independent, against the truth pipeline --
    extended log-likelihood ratios, long double chunks, math.fsum over the reads of a position, 50-digit posterior.
    Probabilities >= 1e-12 within rtol 1e-8, smaller ones within 1e-15; coverage exact."""
    import time
    from nadavca_b200.estimator import ProbabilityEstimator, _ref_codes, group_intervals
    t0 = time.time()
    km, genome, reads, host_reads = _e2e_reads()
    inputs = [_e2e_inputs(km, genome, r) for r in host_reads]
    k, cp = km.get_k(), km.get_central_position()
    pending = [pool.apply_async(_truth_job, (('default', dp, E2E_CONFIG['bandwidth'], E2E_CONFIG['min_event_length'],
                                              E2E_CONFIG['model_wobbling'], False),)) for dp, _, _ in inputs]
    est = ProbabilityEstimator(km, synthetic_aligner(genome), E2E_CONFIG)
    got = {False: est.estimate_probabilities(genome, reads), True: est.estimate_probabilities(genome, reads,
                                                                                              independent=True)}
    chunks = [_truth_chunk(p.get(timeout=3000)['ratio'], rev) for p, (_, _, rev) in zip(pending, inputs)]
    intervals = [iv for _, iv, _ in inputs]
    prior = E2E_CONFIG['snp_prior_probability']
    worst, small = 0.0, 0.0
    for independent in (False, True):
        groups = [(s, e, [i]) for i, (s, e) in enumerate(intervals)] if independent else group_intervals(intervals)
        out = got[independent]
        assert len(out) == len(groups)
        if not independent:
            out = sorted(out, key=lambda c: (c.start, c.end))
        for (start, end, members), chunk in zip(groups, out):
            assert (chunk.start, chunk.end) == (start, end)
            L = end - start
            cols = [[[] for _ in range(4)] for _ in range(L)]
            cov = np.zeros(L, dtype=int)
            for i in members:
                s, e = intervals[i]
                cov[s - start:e - start] += 1
                for p in range(e - s):
                    for j in range(4):
                        cols[s - start + p][j].append(float(chunks[i][p, j]))
            assert np.array_equal(np.asarray(chunk.coverage), cov), 'coverage of group [%d, %d)' % (start, end)
            ll = np.array([[math.fsum(c) for c in row] for row in cols])
            truth = _mp_posterior(ll, _ref_codes(genome[start:end]), np.array([0, L]), k, prior)
            g = np.asarray(chunk.values)
            big = truth >= 1e-12
            rel = np.abs(g[big] - truth[big]) / truth[big]
            absd = np.abs(g[~big] - truth[~big])
            mode = 'independent' if independent else 'consensus'
            assert rel.max() <= 1e-8, '%s group [%d, %d): rtol %.3g' % (mode, start, end, rel.max())
            assert absd.size == 0 or absd.max() <= 1e-15, '%s group [%d, %d): atol %.3g' % (mode, start, end,
                                                                                            absd.max())
            worst = max(worst, float(rel.max()) / 1e-8)
            if absd.size:
                small = max(small, float(absd.max()) / 1e-15)
    print('end to end: 16 reads, consensus and independent, worst err/bar %.2e (p >= 1e-12), %.2e (smaller p), '
          'coverage exact, %.0f s' % (worst, small, time.time() - t0))


def synthetic_aligner(genome):
    from nadavca_b200 import synthetic
    return synthetic.SyntheticAligner(genome)
