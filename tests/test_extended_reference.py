"""The extended-precision reference of EstimateLogLikelihoods (oracle/nadavca_extended.c), validated on the CPU.

The pinned oracle's own rounding error grows with |LL|, so it cannot hold the GPU to an absolute bar on log-likelihood
ratios.  This reference can, and it is checked here: against a 50-digit mpmath restatement of the recurrence on tiny
cases, against the pinned port (same mathematics) on the golden and on random cases, and for the identity
sum_c P[j][c] S[j][c] = total that every row of the plain mode satisfies.  test_old_bar_is_blind shows why a tighter,
absolute bar is needed.
"""
import math
import time

import mpmath
import numpy as np

from conftest import make_case

EPS = 2.0 ** -52


def _ext(case, wob, rows=False):
    from oracle import oracle as orc
    mean, sigma, sig, ref, cb, ca, anc, k, cp, bw, mel = case
    xm = orc.ExtendedModel(k, cp, 4, mean, sigma)
    return orc.estimate_log_likelihoods_extended(sig, ref, cb, ca, anc, bw, mel, xm, wob, rows=rows)


# ---- an independent restatement in mpmath (probabilities, not logs) -------------------------------------------------

def _mp_estimate(mean, sigma, sig, ref, cb, ca, anc, k, cp, bw, mel, wob):
    """dtw.cpp:37-131 with every value an mpmath number at 50 digits; returns the n x 4 log-likelihoods."""
    from oracle import oracle as orc
    mpmath.mp.dps = 50
    n, N = len(ref), len(sig)
    bs, be = orc.band_bounds(anc, N, n, bw)
    zero, one = mpmath.mpf(0), mpmath.mpf(1)

    def tables(i):  # kmer_model.cpp:11-12 in double, as the reference builds them
        s = float(sigma[i])
        return math.log(1 / math.sqrt(2 * math.pi * s * s)), 1 / (2 * s * s)

    def seq_at(seq, idx):
        j = idx + len(cb)
        if j < 0 or j >= len(cb) + n + len(ca):
            return 0
        return int(np.concatenate([cb, seq, ca])[j])

    def kid(seq, i):
        v = 0
        for p in range(i - cp, i - cp + k):
            v = v * 4 + seq_at(seq, p)
        return v

    def gauss(kmer, x):
        ac, mc = tables(kmer)
        d = mpmath.mpf(float(x)) - mpmath.mpf(float(mean[kmer]))
        return mpmath.exp(mpmath.mpf(ac) - d * d * mpmath.mpf(mc))

    def emis(e, x):
        if e[0] == 'g':
            return gauss(e[1], x)
        return (gauss(e[1], x) + gauss(e[2], x)) * mpmath.exp(-2)

    def at(row, i):
        s, e, v = row
        return v[i - s] if s <= i <= e else zero

    def nxt(s, e, pred, em, m, reverse):  # node_next_row.h:6-61
        v = [zero] * max(e - s + 1, 0)
        if e < s:
            return (s, e, v)
        ps, pe, _ = pred
        E = lambda t: emis(em, sig[t])
        if not reverse:
            if s >= m:
                p = one
                for i in range(s, ps - 1, -1):
                    if i < s:
                        p *= E(i)
                    if s - i >= m:
                        v[0] += p * at(pred, i)
            for i in range(max(s + 1, m), e + 1):
                p = one
                for j in range(i - 1, i - m - 1, -1):
                    p *= E(j)
                v[i - s] = p * at(pred, i - m) + E(i - 1) * at((s, e, v), i - 1)
        else:
            if e + m <= N:
                p = one
                for i in range(e, pe + 1):
                    if i > e:
                        p *= E(i - 1)
                    if i - e >= m:
                        v[e - s] += p * at(pred, i)
            for i in range(min(e - 1, N - m), s - 1, -1):
                p = one
                for j in range(i, i + m):
                    p *= E(j)
                v[i - s] = p * at(pred, i + m) + E(i) * at((s, e, v), i + 1)
        return (s, e, v)

    def total(pre, suf):
        return mpmath.fsum(x * at(suf, i) for i, x in zip(range(pre[0], pre[1] + 1), pre[2]))

    P = [(bs[0], be[0], [one] * (be[0] - bs[0] + 1))]
    for i in range(n):
        pred = P[i]
        if i > 0 and wob:
            pred = nxt(bs[i], be[i], pred, ('m', kid(ref, i - 1), kid(ref, i)), 0, False)
        P.append(nxt(bs[i + 1], be[i + 1], pred, ('g', kid(ref, i)), mel, False))
    S = [None] * (n + 1)
    S[n] = (bs[n], be[n], [one] * (be[n] - bs[n] + 1))
    for i in range(n, 0, -1):
        pred = S[i]
        if i < n and wob:
            pred = nxt(bs[i], be[i], pred, ('m', kid(ref, i), kid(ref, i - 1)), 0, True)
        S[i - 1] = nxt(bs[i - 1], be[i - 1], pred, ('g', kid(ref, i - 1)), mel, True)
    no_snp = total(P[n], S[n])
    back, fwd = k - cp - 1, cp
    out = np.zeros((n, 4), dtype=object)
    for i in range(n):
        first, last = max(i - back, 0), min(i + fwd, n - 1)
        for b in range(4):
            if b == ref[i]:
                out[i, b] = no_snp
                continue
            mod = np.array(ref).copy()
            mod[i] = b
            cur = P[first]
            for j in range(first, last + 1):
                if j > 0 and wob:
                    cur = nxt(bs[j], be[j], cur, ('m', kid(mod, j - 1), kid(mod, j)), 0, False)
                cur = nxt(bs[j + 1], be[j + 1], cur, ('g', kid(mod, j)), mel, False)
            if last + 1 < n and wob:
                cur = nxt(bs[last], be[last], cur, ('m', kid(mod, last), kid(mod, last + 1)), 0, False)
            out[i, b] = total(cur, S[last + 1])
    return out


def _tiny_cases():
    rng = np.random.default_rng(77)
    cases = []
    for k in (1, 2, 3):
        for mel in (0, 1, 2):
            made = 0
            while made < 2:
                cp = int(rng.integers(0, k))
                n = int(rng.integers(1, 5))
                c = make_case(rng, k, cp, n, 2, mel, spacing=2)
                if len(c[2]) > 12:
                    continue
                cases.append(c + (k, cp, 2, mel))
                made += 1
    return cases


def test_extended_matches_mpmath_on_tiny_cases():
    """n <= 4, N <= 12, k 1..3, mel 0..2, both modes: the extended reference equals a 50-digit evaluation of the same
    recurrence to 1e-15 in every log-likelihood and every ratio, beyond the final rounding to double."""
    checked = 0
    for case in _tiny_cases():
        for wob in (False, True):
            truth = _mp_estimate(*case, wob)
            got = _ext(case, wob)
            ref = case[3]
            for i in range(truth.shape[0]):
                for b in range(4):
                    t = truth[i, b]
                    if t == 0:
                        assert got['ll'][i, b] == -np.inf
                        continue
                    lt = float(mpmath.log(t))
                    assert abs(got['ll'][i, b] - lt) <= 1e-15 + np.spacing(abs(lt)) / 2, (case[-4:], wob, i, b)
                    if truth[i, ref[i]] != 0:
                        rt = float(mpmath.log(t / truth[i, ref[i]]))
                        assert abs(got['ratio'][i, b] - rt) <= 1e-15 + np.spacing(abs(rt)) / 2, (case[-4:], wob, i, b)
                    checked += 1
    assert checked > 250


def _random_cases(count, seed):
    rng = np.random.default_rng(seed)
    out = []
    for t in range(count):
        k = int(rng.integers(1, 7))
        cp = int(rng.integers(0, k))
        mel = int(rng.integers(0, 4))
        bw = int(rng.integers(3, 25))
        c = make_case(rng, k, cp, int(rng.integers(1, 60)), bw, mel, sparse=bool(t % 3 == 0),
                      homopolymer=bool(t % 5 == 0))
        out.append(c + (k, cp, bw, mel))
    return out


def _golden_cases(golden):
    out = []
    for tag in [str(x) for x in golden['names']]:
        c = golden.case(tag)
        k, cp, bw, mel = (int(x) for x in c['params'])
        out.append((c['mean'], c['sigma'], c['signal'], c['reference'], c['context_before'], c['context_after'],
                    c['anchors'], k, cp, bw, mel))
    return out


def test_extended_is_the_ports_mathematics(golden_dp):
    """On the golden dp_cases and on random cases the extended reference and the pinned port agree in every entry to
    eps (N + n) max(|LL|, 1): the port's own error model, one rounding of a + log(1 + exp(b - a)) at magnitude |LL| per
    DP step along N + n steps.  A cell of 1e-6 of the mass dropped from either recurrence moves LL by 1e-6, far above
    that bar.  The finite pattern is the same, and in plain mode every row j gives the same total
    sum_c P[j][c] S[j][c] to 1e-16 relative."""
    from oracle import oracle as orc
    worst, worst_row, cnt = 0.0, 0.0, 0
    for case in _golden_cases(golden_dp) + _random_cases(40, 5):
        mean, sigma, sig, ref, cb, ca, anc, k, cp, bw, mel = case
        om = orc.OracleModel(k, cp, 4, mean, sigma, 'port')
        for wob in (False, True):
            port = np.array(orc.estimate_log_likelihoods(sig, ref, cb, ca, anc, bw, mel, om, wob))
            got = _ext(case, wob, rows=not wob)
            fin = np.isfinite(port)
            assert np.array_equal(np.isfinite(got['ll']), fin)
            if fin.any():
                bar = EPS * (len(sig) + len(ref)) * np.maximum(np.abs(got['ll'][fin]), 1.0)
                err = np.abs(got['ll'][fin] - port[fin]) / bar
                assert err.max() <= 1, 'k %d bw %d mel %d: err/bar %.3g' % (k, bw, mel, err.max())
                worst = max(worst, float(err.max()))
            if not wob:
                dev = got['row_dev']
                assert np.isnan(dev).all() or np.abs(dev).max() <= 1e-16, dev
                if not np.isnan(dev).any():
                    worst_row = max(worst_row, float(np.abs(dev).max()))
            cnt += 1
    print('extended vs port: %d runs, worst err/bar %.3f (bar eps (N + n) |LL|); max row-total deviation %.1e' % (cnt, worst,
                                                                                                        worst_row))


def full_size_inputs(read_index, bandwidth, strand='+', genome_seed=5, genome_length=30000, n_bases=None, jitter=20):
    """DP inputs of one full-size synthetic read (~2 kb, ~20k samples) on the shipped 6-mer model, as the estimator
    builds them without the normalisation tweak (estimator.py:59-110)."""
    import os
    from conftest import ROOT
    from nadavca_b200 import synthetic
    from nadavca_b200.kmer_model import KmerModel
    from nadavca_b200.read import Read
    from oracle import oracle as orc
    km = KmerModel.load_from_hdf5(os.path.join(ROOT, 'nadavca_b200', 'default', 'kmer_model.hdf5'))
    genome = synthetic.make_genome(genome_length, seed=genome_seed)
    read = synthetic.make_read(genome, km, read_index, n_bases=n_bases, bandwidth=bandwidth, jitter=jitter,
                                strand=strand)
    Read.normalize_reads([read])
    apx = synthetic.SyntheticAligner(genome).get_signal_alignment(read, bandwidth)
    s0, e0 = apx.signal_range
    k, cp = km.get_k(), km.get_central_position()
    start, end = apx.read_sequence_range
    cb = orc.to_numerical(read.sequence[start - cp:start])
    ca = orc.to_numerical(read.sequence[end:end + k - cp - 1])
    return (km.mean, km.sigma, np.asarray(read.normalized_signal[s0:e0], dtype=np.float64),
            orc.to_numerical(apx.reference_part), cb, ca, np.asarray(apx.alignment), k, cp, bandwidth, 2)


def test_old_bar_is_blind():
    """A full-size read (bandwidth 150): drop from the truth's no-SNP total one cell of the closing row -- the cell
    whose share of the total is nearest 1e-6, the weight a band-edge column carries in a narrow band (the last column
    itself carries e^-600 here).  rtol = 1e-9 on the raw log-likelihood accepts the damaged total; an absolute bar of
    64 eps (N + n), which this reference can support, rejects it.  Also reports the reference's CPU time per read."""
    case = full_size_inputs(0, 150)
    N, n = len(case[2]), len(case[3])
    times = []
    for wob in (False, True):
        t0 = time.process_time()
        got = _ext(case, wob, rows=True)
        times.append(time.process_time() - t0)
    total = float(got['ll'][0, case[3][0]])
    w = got['be'] - got['bs'] + 1
    closing = got['prefix'][-w[-1]:] + got['suffix'][-w[-1]:] - total  # log share of each closing-row cell
    cell = int(np.argmin(np.abs(closing - math.log(1e-6))))
    share = math.exp(closing[cell])
    assert 1e-7 < share < 1e-5
    damaged = total + math.log1p(-share)
    assert abs(damaged - total) <= 1e-9 * abs(total), 'the old bar would catch this'
    bar = 64 * EPS * (N + n)
    assert abs(damaged - total) > bar
    print('full-size read N %d n %d: dropped share %.2e moves LL by %.2e; old bar %.2e accepts, new bar %.2e rejects '
          '(x%.0f); extended reference CPU time %.1f s plain, %.1f s wobble' % (
              N, n, share, abs(damaged - total), 1e-9 * abs(total), bar, abs(damaged - total) / bar, *times))
