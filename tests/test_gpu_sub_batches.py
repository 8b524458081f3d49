"""ProbabilityEstimator on workloads of several sub-batches: split against whole, against the oracle pipeline, and the
DP workspaces the model keeps across calls.

``_run_estimate`` cuts the reads into sub-batches of ``sub_batch_reads`` on up to four streams (reused as j % 4); per
sub-batch it refines, takes the event means on the device, fits the tweak splines on the host, evaluates them on the
device and estimates; reads that refine finds no path for are dropped and the sub-batch is rebuilt from the survivors
(or dropped whole).  ``posterior_stage`` then adds the chunks of every sub-batch into one set of consensus rows.

The small case: 42 reads of 400-800 bases of the shipped 6-mer model on a 4 kb genome, both strands, drawn from a copy
of the genome with 1 % substitutions so that the SNP posteriors are not all trivial.  One read does not align; eleven
fail refine because a stretch of their signal was cut to one sample per base (with min_event_length 2 the band holds no
path).  ``test_case_plan`` checks, without a GPU, what each split claims: more than four sub-batches (streams reused),
uneven sizes, a sub-batch whose first and last reads fail, one in which every read fails, and a consensus group whose
reads come from at least three sub-batches, reverse-strand reads included.

Bars (tests/test_gpu_estimator.py): chunks rtol 1e-7 (atol 1e-9), posteriors rtol 1e-6 (atol 1e-12), coverage and
group ranges exact.  Split against whole in independent mode: bit-identical.  In consensus mode the sums differ by the
order of the fp64 atomics; each run is within (m - 1) eps sum|x| of the exact sum (DESIGN.md 3(d)), so two runs differ
by at most D = 2 (m - 1) eps sum|x|, and a posterior, a ratio of sums of exp of such sums over its window, by at most
p (2 D_window + 2e-13) (2e-13: the posterior kernel's own rounding in each run, DESIGN.md 3(e)).
"""
import copy
import os
import time

import numpy as np
import pytest

EPS = 2.0 ** -52
CHUNK_RTOL, CHUNK_ATOL = 1e-7, 1e-9
PROB_RTOL, PROB_ATOL = 1e-6, 1e-12

CONFIG = dict(bandwidth=30, snp_prior_probability=0.001, min_event_length=2, model_wobbling=True,
              model_transitions=True, tweak_signal_normalization=True, normalization_event_length=10)
SPLITS = (3, 4, 7)
N_READS = 42
UNALIGNED = 9                                         # input index of the read the aligner cannot place
FAILED = (20, 21, 22, 23, 24, 25, 26, 34, 37, 38, 40)  # indices among the ALIGNED reads whose refine has no path
WHOLE = 1 << 20


def sub_bounds(n, per):
    """The bounds formula of ProbabilityEstimator._run_estimate (estimator.py)."""
    per = max(1, int(per))
    n_sub = -(-n // per)
    return [n * j // n_sub for j in range(n_sub + 1)]


def _model():
    from conftest import ROOT
    from nadavca_b200.kmer_model import KmerModel
    return KmerModel.load_from_hdf5(os.path.join(ROOT, 'nadavca_b200', 'default', 'kmer_model.hdf5'))


def _squeeze(read, first, count):
    """Keep only the first sample of each of the molecule bases [first, first + count): the approximate alignment still
    places the read, but the band cannot hold min_event_length 2 samples per base there."""
    from nadavca_b200.read import Read
    t = read.truth
    keep = np.ones(len(read.raw_signal), dtype=bool)
    for b in range(first, first + count):
        keep[t['event_starts'][b] + 1:t['event_starts'][b] + t['event_lengths'][b]] = False
    kept = np.flatnonzero(keep)
    mapping = {b: int(np.searchsorted(kept, s)) for b, s in read.sequence_to_signal_mapping.items()}
    out = Read.from_arrays(read.raw_signal[keep], read.sequence, mapping, name=read.fastq.split('\n')[0][1:])
    out.truth = t
    return out


def small_case(km):
    """(genome, reads, planted SNP positions): the reads normalised together, as estimate_snps does."""
    from nadavca_b200 import synthetic
    from nadavca_b200.read import Read
    genome = synthetic.make_genome(4000, seed=61)
    rng = np.random.default_rng(62)
    sample = genome.copy()
    snps = np.sort(rng.choice(len(genome), 40, replace=False))
    for p in snps:
        sample[p] = 'ACGT'[('ACGT'.index(genome[p]) + int(rng.integers(1, 4))) % 4]
    reads = []
    for i in range(N_READS):
        r = synthetic.make_read(sample, km, i, n_bases=int(rng.integers(400, 800)), bandwidth=CONFIG['bandwidth'],
                                strand='+-'[i % 2], seed_base=500)
        item = i - (i > UNALIGNED)
        if i == UNALIGNED:
            r.truth = None
        elif item in FAILED:
            r = _squeeze(r, 150, 120)
        reads.append(r)
    Read.normalize_reads(reads)
    return genome, reads, snps


def _aligned(reads, genome):
    from nadavca_b200 import synthetic
    aligner = synthetic.SyntheticAligner(genome)
    return [(i, apx) for i, apx in ((i, aligner.get_signal_alignment(r, CONFIG['bandwidth']))
                                    for i, r in enumerate(reads)) if apx is not None]


def test_case_plan():
    """No GPU: every claim the small case makes for each split, and the refine failures against the oracle."""
    from nadavca_b200.estimator import group_intervals
    from nadavca_b200.genome import Genome
    from oracle import oracle as orc
    km = _model()
    genome, reads, _ = small_case(km)
    aligned = _aligned(reads, genome)
    assert [i for i, _ in aligned] == [i for i in range(N_READS) if i != UNALIGNED]
    n = len(aligned)
    # refine (tweak: model_transitions False) has no path exactly for the planned reads, on the oracle
    om = orc.OracleModel(km.get_k(), km.get_central_position(), 4, km.mean, km.sigma, 'port')
    k, cp = km.get_k(), km.get_central_position()
    no_path = []
    for item, (i, apx) in enumerate(aligned):
        r = reads[i]
        s0, s1 = apx.signal_range
        a, b = apx.read_sequence_range
        ev = orc.refine_alignment(r.normalized_signal[s0:s1], Genome.to_numerical(apx.reference_part),
                                  Genome.to_numerical(r.sequence[a - cp:a]),
                                  Genome.to_numerical(r.sequence[b:b + k - cp - 1]), apx.alignment,
                                  CONFIG['bandwidth'], CONFIG['min_event_length'], om, False)
        if not ev:
            no_path.append(item)
    assert tuple(no_path) == FAILED
    survivors = [item for item in range(n) if item not in FAILED]
    intervals = [tuple(aligned[item][1].reference_range) for item in survivors]
    reverse = [aligned[item][1].reverse_complement for item in survivors]
    assert any(reverse) and not all(reverse)
    for per in SPLITS + (WHOLE,):
        bounds = sub_bounds(n, per)
        sizes = np.diff(bounds)
        if per == WHOLE:
            assert len(sizes) == 1
            continue
        fails = [[item in FAILED for item in range(lo, hi)] for lo, hi in zip(bounds[:-1], bounds[1:])]
        assert len(sizes) > 4, per                                                 # streams are reused (j % 4)
        assert len(set(sizes.tolist())) > 1, per                                   # uneven sub-batches
        assert any(f[0] and f[-1] and not all(f) for f in fails), per              # first and last reads dropped
        assert any(all(f) for f in fails), per                                     # the batch = None branch
        sub_of = np.searchsorted(bounds, survivors, side='right') - 1
        spans = [(len({sub_of[m] for m in members}), any(reverse[m] for m in members))
                 for _, _, members in group_intervals(intervals)]
        assert any(s >= 3 and rev for s, rev in spans), per                       # one group, several sub-batches


# ---- the oracle pipeline in worker processes -------------------------------------------------------------------------

_ORACLE = {}


def _oracle_job(task):
    """estimator.py:59-121 and 131-156 for one read on the oracle (port back end), tweak included: ('ok', (start,
    end, chunk values, independent posterior)), ('unaligned', None) or ('failed', message) -- the reference crashes in
    its tweak on a read without a refined path, and so does the oracle."""
    from nadavca_b200 import synthetic
    from oracle import oracle as orc
    spec, cfg, genome, read = task
    if spec[0] not in _ORACLE:
        _ORACLE.clear()
        _ORACLE[spec[0]] = orc.OracleModel(*spec[1:], 'port')
    est = orc.OracleEstimator(_ORACLE[spec[0]], synthetic.SyntheticAligner(genome), cfg)
    try:
        chunk = est.estimate_log_likelihoods(genome, read)
    except Exception as e:  # noqa: BLE001 -- the tweak's splrep / broadcasting error on an empty path
        return 'failed', repr(e)
    if chunk is None:
        return 'unaligned', None
    posterior = est.compute_posterior(chunk.values, genome[chunk.start:chunk.end])
    return 'ok', (chunk.start, chunk.end, chunk.values, posterior)


def _spec(km, key):
    return (key, km.get_k(), km.get_central_position(), 4, km.mean, km.sigma)


def oracle_consensus(km, cfg, genome, reads, results):
    """The oracle's estimate_probabilities (sorted chunk sums, posterior per group) over the reads it could process,
    from the per-read chunks the workers computed."""
    from oracle import oracle as orc
    om = orc.OracleModel(km.get_k(), km.get_central_position(), 4, km.mean, km.sigma, 'port')
    est = orc.OracleEstimator(om, None, cfg)
    chunks = {id(r): orc.OracleChunk(*res[1][:3]) for r, res in zip(reads, results) if res[0] == 'ok'}
    est.estimate_log_likelihoods = lambda reference, read: chunks[id(read)]
    return est.estimate_probabilities(genome, [r for r in reads if id(r) in chunks])


@pytest.fixture(scope='module')
def pool():
    import multiprocessing as mp
    p = mp.get_context('spawn').Pool(min(os.cpu_count() or 1, 48))
    yield p
    p.terminate()


class Worst:
    """Largest err / bar seen per comparison."""

    def __init__(self):
        self.v = {}

    def add(self, name, got, want, rtol, atol):
        got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
        assert got.shape == want.shape, name
        r = float((np.abs(got - want) / (atol + rtol * np.abs(want))).max()) if got.size else 0.0
        self.v[name] = max(self.v.get(name, 0.0), r)
        return r <= 1

    def __str__(self):
        return ', '.join('%s %.2e' % kv for kv in sorted(self.v.items()))


# ---- the small case on the GPU: every split under both forced schedules ----------------------------------------------

@pytest.fixture(scope='module')
def small_runs(default_model, pool):
    """Oracle results (started first, so they run while the GPU works) and the GPU results of every split:
    runs[(schedule, per)] = dict(chunks, independent, consensus, sub_batches)."""
    from nadavca_b200 import dtw, synthetic
    from nadavca_b200.estimator import ProbabilityEstimator
    t0 = time.time()
    km = default_model
    genome, reads, snps = small_case(km)
    pending = [pool.apply_async(_oracle_job, ((_spec(km, 'default'), CONFIG, genome, copy.deepcopy(r)),))
               for r in reads]
    aligner = synthetic.SyntheticAligner(genome)
    runs = {}
    try:
        for sched in ('r', 's'):
            dtw.set_sweep_schedule(sched)
            for per in SPLITS + (WHOLE,):
                est = ProbabilityEstimator(km, aligner, dict(CONFIG, sub_batch_reads=per))
                out = {'chunks': est.estimate_log_likelihood_chunks(genome, reads),
                       'independent': est.estimate_probabilities(genome, reads, independent=True)}
                out['consensus'] = est.estimate_probabilities(genome, reads)
                out['sub_batches'] = est.last_stats['sub_batches']
                runs[(sched, per)] = out
    finally:
        dtw.set_sweep_schedule(None)
    oracle = [p.get(timeout=3000) for p in pending]
    return dict(km=km, genome=genome, reads=reads, snps=snps, runs=runs, oracle=oracle, seconds=time.time() - t0)


def _consensus_bar(whole_chunks, groups, k):
    """Per row of the concatenated groups: the relative bar 2 D_window + 2e-13 of a split-vs-whole posterior, where
    D = 2 (m - 1) eps sum|x| per (position, base), maximised over the posterior's window (rows i-k+1 .. i+k-1 of its
    group, every base)."""
    bars = []
    for g in groups:
        L = g.end - g.start
        absum = np.zeros((L, 4))
        for c in whole_chunks:
            if c.start >= g.start and c.end <= g.end:
                absum[c.start - g.start:c.end - g.start] += np.abs(c.values)
        m = np.asarray(g.coverage, dtype=np.float64)
        d = (2 * np.maximum(m - 1, 0) * EPS)[:, None] * absum
        dmax = d.max(axis=1)
        win = np.array([dmax[max(0, i - k + 1):min(L, i + k)].max() for i in range(L)])
        bars.append(2 * win + 2e-13)
    return bars


@pytest.mark.gpu
def test_split_matches_whole(small_runs):
    """sub_batch_reads 3, 4, 7 against one batch, tweak and wobble on, under each forced sweep schedule: independent
    chunks, probabilities and coverage bit-identical; consensus coverage and ranges exact, posteriors within the bar of
    the atomics' order; failed and unaligned reads None, results in input order."""
    s = small_runs
    n_aligned = N_READS - 1
    missing = {UNALIGNED} | {f + (f >= UNALIGNED) for f in FAILED}
    k = s['km'].get_k()
    failures, identical, worst_cons = [], {}, 0.0
    for sched in ('r', 's'):
        whole = s['runs'][(sched, WHOLE)]
        assert whole['sub_batches'] == 1
        bars = _consensus_bar(whole['chunks'], whole['consensus'], k)
        for per in SPLITS:
            run = s['runs'][(sched, per)]
            where = '[%s] sub_batch_reads %d' % (sched, per)
            assert run['sub_batches'] == sum(
                1 for lo, hi in zip(sub_bounds(n_aligned, per)[:-1], sub_bounds(n_aligned, per)[1:])
                if any(item not in FAILED for item in range(lo, hi))), where
            ind = run['independent']
            assert len(ind) == N_READS and {i for i, c in enumerate(ind) if c is None} == missing, where
            same = len(run['chunks']) == len(whole['chunks']) == N_READS - len(missing)
            for a, b in zip(run['chunks'], whole['chunks']):
                same &= (a.start, a.end) == (b.start, b.end) and np.array_equal(a.values, b.values)
            for a, b in zip(ind, whole['independent']):
                if a is None or b is None:
                    same &= a is None and b is None
                    continue
                same &= (a.start, a.end) == (b.start, b.end) and np.array_equal(a.values, b.values) and \
                    np.array_equal(a.coverage, b.coverage)
            identical[(sched, per)] = bool(same)
            if not same:
                failures.append('%s: independent results are not bit-identical to the whole batch' % where)
            cons, wcons = run['consensus'], whole['consensus']
            assert [(c.start, c.end) for c in cons] == [(c.start, c.end) for c in wcons], where
            for c, w, bar in zip(cons, wcons, bars):
                assert np.array_equal(c.coverage, w.coverage), where
                err = np.abs(c.values - w.values)
                lim = bar[:, None] * np.abs(w.values) + 1e-300
                worst_cons = max(worst_cons, float((err / lim).max()))
                if (err > lim).any():
                    failures.append('%s: consensus group [%d, %d) beyond the atomics bar (%.3g)' % (
                        where, c.start, c.end, float((err / lim).max())))
    print('split vs whole (42 reads, %s): independent bit-identical %s; consensus worst err/bar %.2e' % (
        '/'.join(map(str, SPLITS)), ', '.join('%s/%d %s' % (a, b, 'yes' if v else 'NO')
                                             for (a, b), v in sorted(identical.items())), worst_cons))
    assert not failures, '\n'.join(failures)


@pytest.mark.gpu
def test_split_matches_oracle_pipeline(small_runs):
    """Every split and schedule against the oracle's own pipeline (host numpy.mean, splrep, splev, sorted chunk
    sums, posterior) at the pinned bars; the oracle fails on exactly the planned reads."""
    s = small_runs
    km, genome, reads, oracle = s['km'], s['genome'], s['reads'], s['oracle']
    status = [o[0] for o in oracle]
    missing_failed = {f + (f >= UNALIGNED) for f in FAILED}
    assert {i for i, st in enumerate(status) if st == 'unaligned'} == {UNALIGNED}
    assert {i for i, st in enumerate(status) if st == 'failed'} == missing_failed
    ok = [i for i, st in enumerate(status) if st == 'ok']
    consensus = oracle_consensus(km, CONFIG, genome, reads, oracle)
    # the planted substitutions are called: some reference bases lose the posterior
    called = sum(int((c.values[np.arange(c.end - c.start), ['ACGT'.index(b) for b in genome[c.start:c.end]]]
                      < 0.5).sum()) for c in consensus)
    assert called >= 5, called
    worst = Worst()
    failures = []
    for (sched, per), run in sorted(s['runs'].items()):
        where = '[%s] sub_batch_reads %d' % (sched, per if per != WHOLE else -1)
        assert len(run['chunks']) == len(ok), where
        for c, i in zip(run['chunks'], ok):
            start, end, values, _ = oracle[i][1]
            assert (c.start, c.end) == (start, end), where
            if not worst.add('chunks', c.values, values, CHUNK_RTOL, CHUNK_ATOL):
                failures.append('%s: chunk of read %d' % (where, i))
        for i, c in enumerate(run['independent']):
            if i not in ok:
                assert c is None, (where, i)
                continue
            start, end, _, post = oracle[i][1]
            assert (c.start, c.end) == (start, end) and np.array_equal(c.coverage, np.ones(end - start)), where
            if not worst.add('independent', c.values, post, PROB_RTOL, PROB_ATOL):
                failures.append('%s: independent posterior of read %d' % (where, i))
        assert [(c.start, c.end) for c in run['consensus']] == [(c.start, c.end) for c in consensus], where
        for c, w in zip(run['consensus'], consensus):
            assert np.array_equal(c.coverage, w.coverage), where
            if not worst.add('consensus', c.values, w.values, PROB_RTOL, PROB_ATOL):
                failures.append('%s: consensus group [%d, %d)' % (where, c.start, c.end))
    print('small case vs oracle (%d reads ok, %d failed refine, 1 unaligned; %d groups, %d reference bases called '
          'against): worst err/bar %s; %.0f s' % (len(ok), len(missing_failed), len(consensus), called, worst,
                                                 s['seconds']))
    assert not failures, '\n'.join(failures[:20])


# ---- the benchmark's shape -------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_benchmark_shape_two_sub_batches(default_model, pool):
    """300 full-size reads (~2000 bases, bandwidth 150) under the default config: sub_batch_reads 256 gives two
    sub-batches of 150 on their own streams.  Schedule auto.  Independent mode, against the oracle on 32 reads of the
    SECOND sub-batch and against the whole batch (which sits above the 295/296-read schedule threshold while each
    sub-batch is below it) at the pinned bars."""
    from nadavca_b200 import defaults, dtw, synthetic
    from nadavca_b200.estimator import ProbabilityEstimator
    from nadavca_b200.read import Read
    t0 = time.time()
    km = default_model
    cfg = defaults.load_config()
    assert 'sub_batch_reads' not in cfg and cfg['bandwidth'] == 150 and cfg['tweak_signal_normalization']
    genome = synthetic.make_genome(300_000, seed=71)
    reads = [synthetic.make_read(genome, km, 3000 + i) for i in range(300)]
    Read.normalize_reads(reads)
    bounds = sub_bounds(len(reads), 256)
    assert bounds == [0, 150, 300]
    picked = list(range(bounds[1], bounds[2], 4))[:32]
    assert len(picked) == 32
    pending = {i: pool.apply_async(_oracle_job, ((_spec(km, 'default'), cfg, genome, copy.deepcopy(reads[i])),))
               for i in picked}
    aligner = synthetic.SyntheticAligner(genome)
    got = {}
    dtw.set_sweep_schedule(None)
    for name, c in (('split', cfg), ('whole', dict(cfg, sub_batch_reads=len(reads)))):
        est = ProbabilityEstimator(km, aligner, c)
        chunks = est.estimate_log_likelihood_chunks(genome, reads)
        ind = est.estimate_probabilities(genome, reads, independent=True)
        got[name] = (chunks, ind, est.last_stats['sub_batches'])
    assert got['split'][2] == 2 and got['whole'][2] == 1
    worst = Worst()
    failures = []
    split, whole = got['split'], got['whole']
    assert len(split[0]) == len(whole[0]) == len(reads) and all(c is not None for c in split[1] + whole[1])
    identical = True
    for i in range(len(reads)):
        a, b = split[0][i], whole[0][i]
        assert (a.start, a.end) == (b.start, b.end)
        identical &= np.array_equal(a.values, b.values) and np.array_equal(split[1][i].values, whole[1][i].values)
        if not worst.add('split/whole chunks', a.values, b.values, CHUNK_RTOL, CHUNK_ATOL):
            failures.append('chunk of read %d: split vs whole' % i)
        if not worst.add('split/whole posteriors', split[1][i].values, whole[1][i].values, PROB_RTOL, PROB_ATOL):
            failures.append('posterior of read %d: split vs whole' % i)
        assert np.array_equal(split[1][i].coverage, whole[1][i].coverage)
    for i in picked:
        st, res = pending[i].get(timeout=3000)
        assert st == 'ok', (i, st, res)
        start, end, values, post = res
        assert (split[0][i].start, split[0][i].end) == (split[1][i].start, split[1][i].end) == (start, end)
        if not worst.add('oracle chunks', split[0][i].values, values, CHUNK_RTOL, CHUNK_ATOL):
            failures.append('chunk of read %d: split vs oracle' % i)
        if not worst.add('oracle posteriors', split[1][i].values, post, PROB_RTOL, PROB_ATOL):
            failures.append('posterior of read %d: split vs oracle' % i)
    print('benchmark shape (300 reads, 2 sub-batches, auto): split vs whole bit-identical %s; worst err/bar %s; '
          '%.0f s' % ('yes' if identical else 'no', worst, time.time() - t0))
    assert not failures, '\n'.join(failures[:20])


# ---- DP workspaces across calls --------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_workspace_does_not_grow_across_calls(lib_built):
    """Ten estimate_probabilities calls on one estimator with eleven sub-batches each, then three estimate_snps calls
    (a new estimator each) with the same model: the model's DP workspace bytes (its own counter, not the device's
    free memory) stay those of the first call, within one sub-batch's workspace."""
    import nadavca_b200
    from nadavca_b200 import _cabi, synthetic
    from nadavca_b200.estimator import ProbabilityEstimator
    km = _model()  # a model of its own: its workspaces start empty
    genome, reads, _ = small_case(km)
    cfg = dict(CONFIG, sub_batch_reads=4)
    assert len(sub_bounds(N_READS - 1, 4)) - 1 == 11
    aligner = synthetic.SyntheticAligner(genome)
    est = ProbabilityEstimator(km, aligner, cfg)
    lib = _cabi.load()
    sizes = []
    for _ in range(10):
        est.estimate_probabilities(genome, reads, independent=True)
        sizes.append(int(lib.nvb_model_workspace_bytes(km.handle)))
    for _ in range(3):
        nadavca_b200.estimate_snps(None, copy.deepcopy(reads), reference=genome, config=cfg, kmer_model=km,
                                   independent=True, aligner=aligner)
        sizes.append(int(lib.nvb_model_workspace_bytes(km.handle)))
    one = sizes[0] // 4  # four streams' workspaces after the first call: one sub-batch's is about a quarter
    print('workspace bytes: after call 1 %d, after call 10 %d, after 3 estimate_snps calls %d' % (
        sizes[0], sizes[9], sizes[-1]))
    assert sizes[0] > 0
    assert max(sizes) - sizes[0] <= one, sizes
