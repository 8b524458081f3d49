"""GPU parity, API level: the drop-in Python surface (ProbabilityEstimator / estimate_snps / align_signal) on the
B200 kernels against (a) the golden outputs of the reference's own estimator.py and (b) the oracle, plus
size-independent properties at the full BASELINE read size.

Tolerances (north_star: alignments bit-exact, log-likelihoods / probabilities <= 1e-5 relative):
  alignment tables, coverage, group ranges : exact
  normalised log-likelihood chunks          : rtol 1e-7 (atol 1e-9: entries that are exactly 0 in the reference)
  SNP posterior probabilities               : rtol 1e-6, atol 1e-12
"""
import numpy as np
import pytest

from conftest import GOLDEN_CONFIG, golden_reads

pytestmark = pytest.mark.gpu

CHUNK_RTOL, CHUNK_ATOL = 1e-7, 1e-9
PROB_RTOL, PROB_ATOL = 1e-6, 1e-12


def _setup(golden_estimator, default_model, tweak):
    from nadavca_b200 import synthetic
    from nadavca_b200.estimator import ProbabilityEstimator
    from nadavca_b200.read import Read
    genome = golden_estimator['genome']
    reads = golden_reads(golden_estimator)
    Read.normalize_reads(reads)
    aligner = synthetic.SyntheticAligner(genome)
    cfg = dict(GOLDEN_CONFIG, tweak_signal_normalization=bool(tweak))
    return genome, reads, aligner, ProbabilityEstimator(default_model, aligner, cfg), cfg


@pytest.mark.parametrize('tweak', [1, 0])
def test_estimator_matches_reference_golden(golden_estimator, default_model, tweak):
    g = golden_estimator
    genome, reads, aligner, est, cfg = _setup(g, default_model, tweak)
    pre = 'tweak%d/' % tweak
    # path A: refined alignment tables, bit-exact
    tables = est.get_refined_alignments(reads)
    for i, res in enumerate(tables):
        assert res is not None
        assert np.array_equal(res[1], g[pre + 'read%d/alignment_table' % i]), i
        assert res[1].dtype.kind == 'i' and res[1].shape[1] == 3
    one = est.get_refined_alignment(reads[2])
    assert np.array_equal(one[1], g[pre + 'read2/alignment_table'])
    # path B: per-read normalised chunks
    chunks = est.estimate_log_likelihood_chunks(genome, reads)
    assert len(chunks) == len(reads)
    for i, c in enumerate(chunks):
        assert [c.start, c.end] == g[pre + 'read%d/chunk_range' % i].tolist()
        np.testing.assert_allclose(c.values, g[pre + 'read%d/chunk_values' % i], rtol=CHUNK_RTOL, atol=CHUNK_ATOL)
    # independent posteriors (estimate_snps.py:63-68) and the consensus groups (estimator.py:205-236)
    ind = est.estimate_probabilities(genome, reads, independent=True)
    for i, c in enumerate(ind):
        np.testing.assert_allclose(c.values, g[pre + 'read%d/independent_probabilities' % i], rtol=PROB_RTOL,
                                   atol=PROB_ATOL)
        assert np.array_equal(c.coverage, np.ones(c.end - c.start, dtype=int))
    groups = est.estimate_probabilities(genome, reads, independent=False)
    assert len(groups) == int(g[pre + 'n_groups'])
    for gi, c in enumerate(groups):
        assert [c.start, c.end] == g[pre + 'group%d/range' % gi].tolist()
        assert np.array_equal(c.coverage, g[pre + 'group%d/coverage' % gi])
        np.testing.assert_allclose(c.values, g[pre + 'group%d/probabilities' % gi], rtol=PROB_RTOL, atol=PROB_ATOL)
        np.testing.assert_allclose(c.values.sum(axis=1), 1.0, rtol=1e-12)


def test_estimate_snps_api(golden_estimator, default_model):
    """Public entry point with Read instances, a dict config and an injected aligner."""
    import nadavca_b200
    from nadavca_b200 import synthetic
    g = golden_estimator
    genome = g['genome']
    aligner = synthetic.SyntheticAligner(genome)
    for independent in (True, False):
        reads = golden_reads(g)
        out = nadavca_b200.estimate_snps(None, reads, reference=genome, config=GOLDEN_CONFIG,
                                         kmer_model=default_model, independent=independent, aligner=aligner)
        if independent:
            assert len(out) == len(reads)
            for i, c in enumerate(out):
                np.testing.assert_allclose(c.values, g['tweak1/read%d/independent_probabilities' % i],
                                           rtol=PROB_RTOL, atol=PROB_ATOL)
        else:
            assert [(c.start, c.end) for c in out] == [tuple(g['tweak1/group%d/range' % i]) for i in range(4)]
            assert out == sorted(out)
    assert nadavca_b200.estimate_snps(None, [], reference=genome, config='/nonexistent.yaml',
                                      kmer_model=default_model, aligner=aligner) is None


def test_align_signal_api_matches_oracle_loop(golden_estimator, default_model):
    """align_signal's renormalisation rounds (align_signal.py:52-81) against the same loop driven by the oracle."""
    import nadavca_b200
    from nadavca_b200 import synthetic
    from nadavca_b200.read import Read
    from oracle import oracle as orc
    from scipy.stats import linregress
    g = golden_estimator
    genome = g['genome']
    aligner = synthetic.SyntheticAligner(genome)
    km = default_model
    got = list(nadavca_b200.align_signal(None, golden_reads(g), config=GOLDEN_CONFIG, kmer_model=km,
                                         aligner=aligner, reference=genome))
    om = orc.OracleModel(km.get_k(), km.get_central_position(), 4, km.mean, km.sigma, 'port')
    est = orc.OracleEstimator(om, aligner, GOLDEN_CONFIG)
    reads = golden_reads(g)
    assert len(got) == len(reads)
    for (read_out, res), read in zip(got, reads):
        Read.normalize_reads([read])
        apx, al = est.get_refined_alignment(read)
        for r in range(3):
            if r % 2 == 0:
                expected = np.array(om.get_expected_signal(orc.to_numerical(apx.reference_part), [], []))
                cut = read.normalized_signal[al[0][1]:al[-1][2]]
                means = [np.mean(cut[s - al[0][1]:e - al[0][1]]) for _, s, e in al]
                slope, intercept, _, _, _ = linregress(expected, means)
                read.normalized_signal = (read.normalized_signal - intercept) / slope
            else:
                apx, al = est.get_refined_alignment(read)
        assert res is not None
        assert np.array_equal(res[1], al)
        np.testing.assert_allclose(read_out.normalized_signal, read.normalized_signal, rtol=1e-12)


def test_unaligned_reads_are_none(golden_estimator, default_model):
    from nadavca_b200.read import Read
    g = golden_estimator
    genome, reads, aligner, est, cfg = _setup(g, default_model, 1)
    stranger = Read.from_arrays(np.arange(50.0), 'ACGT' * 3, {i: 4 * i for i in range(12)})
    Read.normalize_reads([stranger])
    res = est.get_refined_alignments([reads[0], stranger, reads[1]])
    assert res[1] is None and res[0] is not None and res[2] is not None
    chunks = est.estimate_probabilities(genome, [stranger], independent=True)
    assert chunks == [None]
    chunks = est.estimate_probabilities(genome, [reads[0], stranger, reads[1]], independent=True)
    assert chunks[1] is None and chunks[0] is not None and chunks[2] is not None
    assert est.estimate_probabilities(genome, [stranger], independent=False) == []


def test_full_size_reads_properties_and_oracle(default_model):
    """BASELINE read size (~2000 bases, ~20k samples, bandwidth 150): two reads against the oracle, the rest
    through size-independent properties."""
    from nadavca_b200 import dtw, synthetic
    from nadavca_b200.genome import Genome
    from nadavca_b200.read import Read
    from oracle import oracle as orc
    km = default_model
    genome = synthetic.make_genome(100_000, seed=4)
    reads = [synthetic.make_read(genome, km, 900 + i, n_bases=1900 + 40 * i) for i in range(6)]
    Read.normalize_reads(reads)
    aligner = synthetic.SyntheticAligner(genome)
    args = []
    for r in reads:
        apx = aligner.get_signal_alignment(r, 150)
        s0, s1 = apx.signal_range
        a, b = apx.read_sequence_range
        args.append((r.normalized_signal[s0:s1], Genome.to_numerical(apx.reference_part),
                     Genome.to_numerical(r.sequence[a - 2:a]), Genome.to_numerical(r.sequence[b:b + 3]),
                     apx.alignment))
    om = orc.OracleModel(6, 2, 4, km.mean, km.sigma, 'port')
    with dtw.Batch(km, *[list(x) for x in zip(*args)], 150, 2) as batch:
        for flag in (False, True):
            batch.refine(flag)
            events, status = batch.events()
            assert np.all(status == 0)
            for ev in events:
                assert np.all(ev[:, 1] - ev[:, 0] >= 2) and np.all(ev[1:, 0] >= ev[:-1, 1])
                if not flag:
                    assert np.array_equal(ev[1:, 0], ev[:-1, 1])
            for i in (0, 5):
                assert events[i].tolist() == orc.refine_alignment(*args[i], 150, 2, om, flag)
        batch.estimate(True)
        lls, _ = batch.log_likelihoods()
        for ll, a in zip(lls, args):
            ref_col = ll[np.arange(len(ll)), a[1]]
            assert np.all(ref_col == ref_col[0]) and np.all(np.isfinite(ll))
            # the true base is the most likely one at (nearly) every position of an error-free synthetic read
            assert np.mean(np.argmax(ll, axis=1) == a[1]) > 0.97
        want = np.array(orc.estimate_log_likelihoods(*args[0], 150, 2, om, True))
        np.testing.assert_allclose(lls[0], want, rtol=1e-9)
        np.testing.assert_allclose((lls[0] - lls[0][0, args[0][1][0]]) / 10, (want - want[0, args[0][1][0]]) / 10,
                                   rtol=CHUNK_RTOL, atol=CHUNK_ATOL)


def test_wide_band_and_long_read(default_model):
    """Band-width sweep corner (BASELINE configs[4]): bandwidth 400 (801-column rows: several warps per sweep
    direction, three chunks per row in the path search) against the oracle, and a 6000-base read with the default
    band through size-independent properties (BASELINE configs[3] in miniature)."""
    from nadavca_b200 import dtw, synthetic
    from nadavca_b200.genome import Genome
    from nadavca_b200.read import Read
    from oracle import oracle as orc
    km = default_model
    genome = synthetic.make_genome(50_000, seed=9)
    om = orc.OracleModel(6, 2, 4, km.mean, km.sigma, 'port')

    def prepare(read, bw):
        apx = synthetic.SyntheticAligner(genome).get_signal_alignment(read, bw)
        s0, s1 = apx.signal_range
        a, b = apx.read_sequence_range
        return (read.normalized_signal[s0:s1], Genome.to_numerical(apx.reference_part),
                Genome.to_numerical(read.sequence[a - 2:a]), Genome.to_numerical(read.sequence[b:b + 3]), apx.alignment)

    wide = [synthetic.make_read(genome, km, 300 + i, n_bases=500 + 60 * i, bandwidth=400) for i in range(2)]
    Read.normalize_reads(wide)
    args = [prepare(r, 400) for r in wide]
    with dtw.Batch(km, *[list(x) for x in zip(*args)], 400, 2) as batch:
        assert max(int((be - bs + 1).max()) for bs, be in batch.bands()) > 704  # > 2 chunks of 352 columns
        for flag in (True, False):
            batch.refine(flag)
            events, status = batch.events()
            for ev, a in zip(events, args):
                assert ev.tolist() == orc.refine_alignment(*a, 400, 2, om, flag)
        batch.estimate(True)
        lls, _ = batch.log_likelihoods()
        want = np.array(orc.estimate_log_likelihoods(*args[0], 400, 2, om, True))
        np.testing.assert_allclose(lls[0], want, rtol=1e-9)

    long_read = [synthetic.make_read(genome, km, 400, n_bases=6000)]
    Read.normalize_reads(long_read)
    a = prepare(long_read[0], 150)
    with dtw.Batch(km, *[[x] for x in a], 150, 2) as batch:
        batch.refine(True)
        events, status = batch.events()
        ev = events[0]
        assert status[0] == 0 and len(ev) == len(a[1])
        assert np.all(ev[:, 1] - ev[:, 0] >= 2) and np.all(ev[1:, 0] >= ev[:-1, 1])
        batch.estimate(True)
        ll = batch.log_likelihoods()[0][0]
        assert np.all(np.isfinite(ll)) and np.mean(np.argmax(ll, axis=1) == a[1]) > 0.97


def test_event_means_equal_numpy_mean_bit_for_bit(golden_estimator, default_model):
    """nvb_batch_event_means reproduces numpy.mean (pairwise summation order) exactly, including events longer than
    8 and 128 samples and reads without a path."""
    from nadavca_b200 import dtw
    rng = np.random.default_rng(77)
    k, cp, mel, bw = 2, 1, 2, 40
    mean = rng.normal(0, 1.2, size=16)
    sigma = rng.uniform(0.2, 0.5, size=16)
    gm = dtw.KmerModel(k, cp, 4, mean, sigma)
    cases = [make_case_local(rng, k, cp, n, bw, mel, spacing) for n, spacing in ((30, 6), (8, 150), (20, 40), (12, 12))]
    sig = rng.normal(0, 1, 12)
    cases.append((sig, rng.integers(0, 4, 10), [], [], np.array([[0, 0], [11, 9]])))  # no path
    lists = [[c[i] for c in cases] for i in range(5)]
    with dtw.Batch(gm, *lists, bw, mel) as batch:
        for flag in (False, True):
            batch.refine(flag)
            events, status = batch.events()
            means = batch.event_means()
            longest = 0
            for ev, m, c in zip(events, means, cases):
                if ev is None:
                    assert np.all(np.isnan(m))
                    continue
                want = np.array([np.mean(c[0][s:e]) for s, e in ev])
                assert np.array_equal(m, want)
                longest = max(longest, int((ev[:, 1] - ev[:, 0]).max()))
            assert longest > 128  # the recursive split of numpy's pairwise sum was exercised


def make_case_local(rng, k, cp, n, bw, mel, spacing):
    from conftest import make_case
    return make_case(rng, k, cp, n, bw, mel, spacing=spacing)[2:]


def test_device_spline_evaluation_matches_scipy(golden_estimator, default_model):
    """nvb_batch_apply_splines == scipy.interpolate.splev (FITPACK) on the splines the tweak fits, including
    extrapolation beyond the knots and reads left untouched."""
    from scipy import interpolate
    from nadavca_b200 import dtw, synthetic
    from nadavca_b200.genome import Genome
    from nadavca_b200.read import Read
    g = golden_estimator
    genome = g['genome']
    reads = golden_reads(g)
    Read.normalize_reads(reads)
    aligner = synthetic.SyntheticAligner(genome)
    km = default_model
    args, splines = [], []
    for i, r in enumerate(reads):
        apx = aligner.get_signal_alignment(r, 30)
        s0, s1 = apx.signal_range
        a, b = apx.read_sequence_range
        ref = Genome.to_numerical(apx.reference_part)
        cb, ca = Genome.to_numerical(r.sequence[a - 2:a]), Genome.to_numerical(r.sequence[b:b + 3])
        args.append((r.normalized_signal[s0:s1], ref, cb, ca, apx.alignment))
        table = g['tweak1/read%d/alignment_table' % i]
        expected = km.get_expected_signal(ref, cb, ca)
        splines.append(None if i == 3 else r.fit_tweak_spline(table[:, 1:], expected))
    with dtw.Batch(km, *[list(x) for x in zip(*args)], 30, 2) as batch:
        batch.apply_splines(splines)
        got = batch.signals()
    for sig, spl, a in zip(got, splines, args):
        want = a[0] if spl is None else interpolate.splev(a[0], spl)
        if spl is not None:  # some samples lie outside the knot range: the extrapolation branch is exercised
            assert a[0].min() < spl[0][0] or a[0].max() > spl[0][-1]
        np.testing.assert_allclose(sig, want, rtol=1e-13, atol=1e-13)


def test_full_size_batch_alignments_bit_exact(default_model):
    """32 reads of the BASELINE size (~2000 bases, ~20k samples, bandwidth 150, both strands) through both alignment
    modes: every event boundary equals the oracle's; split into waves by a small workspace limit on the way."""
    from nadavca_b200 import dtw, synthetic
    from nadavca_b200.genome import Genome
    from nadavca_b200.read import Read
    from oracle import oracle as orc
    km = default_model
    genome = synthetic.make_genome(200_000, seed=12)
    reads = [synthetic.make_read(genome, km, 5000 + i) for i in range(32)]
    Read.normalize_reads(reads)
    aligner = synthetic.SyntheticAligner(genome)
    args = []
    for r in reads:
        apx = aligner.get_signal_alignment(r, 150)
        s0, s1 = apx.signal_range
        a, b = apx.read_sequence_range
        args.append((r.normalized_signal[s0:s1], Genome.to_numerical(apx.reference_part),
                     Genome.to_numerical(r.sequence[a - 2:a]), Genome.to_numerical(r.sequence[b:b + 3]),
                     apx.alignment))
    om = orc.OracleModel(6, 2, 4, km.mean, km.sigma, 'port')
    total = 0
    with dtw.Batch(km, *[list(x) for x in zip(*args)], 150, 2, workspace_limit=400_000_000) as batch:
        for flag in (False, True):
            batch.refine(flag)
            events, status = batch.events()
            assert np.all(status == 0)
            for ev, a in zip(events, args):
                assert ev.tolist() == orc.refine_alignment(*a, 150, 2, om, flag)
                total += len(ev)
    assert total > 2 * 32 * 1500


def test_detect_meth_api(golden_estimator, default_model, tmp_path):
    """detect_meth end to end on the GPU path: CSV layout of the reference, scores consistent with the returned
    alignments and the renormalised signals."""
    import csv
    import nadavca_b200
    from nadavca_b200 import synthetic
    from nadavca_b200.detect_meth import calculate_meth_scores, maxs3
    g = golden_estimator
    genome = g['genome']
    aligner = synthetic.SyntheticAligner(genome)
    reads = golden_reads(g)
    out = tmp_path / 'meth.csv'
    rows = nadavca_b200.detect_meth(None, reads, 'CG', str(out), config=GOLDEN_CONFIG, kmer_model=default_model,
                                    aligner=aligner, reference=genome, names=['r%d' % i for i in range(len(reads))])
    with open(out) as fh:
        lines = list(csv.reader(fh))
    assert lines[0] == ['Filename', 'Position', 'Sequence context', 'Position scores', 'Aggregated score']
    assert len(lines) == len(rows) + 1 and len(rows) >= 10
    # recompute from an independent align_signal run over fresh copies of the reads
    again = list(nadavca_b200.align_signal(None, golden_reads(g), config=GOLDEN_CONFIG, kmer_model=default_model,
                                           aligner=aligner, reference=genome))
    want = []
    for i, (read, (apx, alignment)) in enumerate(again):
        cut = read.normalized_signal[alignment[0][1]:alignment[-1][2]]
        for pos, context, scores in calculate_meth_scores(cut, alignment, apx, 'CG', default_model):
            assert len(context) == 11 and context[5:7] == 'CG' and len(scores) == 11
            want.append(('r%d' % i, pos, context, ','.join(map(str, scores)), maxs3(scores)))
    assert rows == want


def test_bench_line_contract():
    """bench.py on a tiny workload prints one JSON line with every key of the measurement contract."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--reads', '24', '--bases', '400', '--steps',
                          '2', '--warmup', '3', '--cpu-sample', '2'], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith('{')][-1])
    for key in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
                'vs_baseline', 'dtype', 'data', 'config', 'e2e', 'gpu_launches', 'clocks', 'roofline', 'cpu_baseline'):
        assert key in line, key
    assert line['n_gpus'] == 1 and line['steps'] == 2 and line['dtype'] == 'f64' and line['data'] == 'synthetic'
    assert line['value'] > 0 and line['e2e']['value'] > 0 and line['e2e']['h2d_bytes_per_step'] > 0
    assert line['gpu_launches'] >= 2 * 8  # sweeps, score, path, no-SNP, SNP, chunk, scatter, posterior per step
    assert set(line['roofline']) >= {'bound', 'achieved', 'peak', 'unit', 'frac', 'traffic'}
    assert line['roofline']['bound'] == 'hbm' and 0 < line['roofline']['frac'] < 1
    assert line['cpu_baseline']['kind'] in ('reference', 'port') and line['cpu_baseline']['cores'] >= 1
    assert 'workload' in line['config']
    assert line['consensus']['ranks_identical'] and line['consensus']['value'] > 0
    assert line['api']['estimate_snps']['value'] > 0 and line['api']['align_signal']['aligned'] == 24
    assert line['alu']['kernel'] == 'snp3_kernel' and line['alu']['dp_cells_per_sec'] > 0
    # the benchmarked reads themselves are checked against the reference inside the CPU leg
    par = line['parity']
    assert par['reads'] == 2 and par['event_mismatches'] == 0 and par['ll_mismatches'] == 0
    assert par['events_compared'] > 0 and par['max_ll_rel'] < 1e-9


def test_bench_dump_outputs_are_reproducible(tmp_path):
    """bench.py --dump-outputs: float arrays of what the last timed step computed, consistent with each other, under
    64 MB, and bit-identical between two runs with the same arguments (seeded inputs, deterministic kernels)."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    names = ['chunks', 'coverage', 'events', 'log_likelihoods', 'probabilities']
    runs = []
    for tag in ('a', 'b'):
        out = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--reads', '24', '--bases', '400',
                              '--steps', '2', '--warmup', '1', '--no-api', '--no-consensus', '--no-cpu-baseline',
                              '--dump-outputs', str(tmp_path / tag)], capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-3000:]
        assert sorted(os.listdir(tmp_path / tag)) == [n + '.npy' for n in names]
        assert sum(os.path.getsize(tmp_path / tag / (n + '.npy')) for n in names) <= 64 << 20
        runs.append({n: np.load(tmp_path / tag / (n + '.npy')) for n in names})
    d = runs[0]
    for arr in d.values():
        assert arr.dtype in (np.float32, np.float64)
    assert d['chunks'][:, 0].tolist() == list(range(24))  # a small batch is written whole
    rows = int((d['chunks'][:, 2] - d['chunks'][:, 1]).sum())
    assert d['probabilities'].shape == d['log_likelihoods'].shape == (rows, 4) and d['events'].shape == (rows, 2)
    np.testing.assert_allclose(d['probabilities'].sum(axis=1), 1.0, rtol=1e-12)
    assert np.all(d['coverage'] == 1) and np.all(d['events'][:, 1] - d['events'][:, 0] >= 2)
    for n in names:
        assert np.array_equal(runs[0][n], runs[1][n]), n


def test_estimator_on_a_non_default_torch_stream(golden_estimator, default_model):
    """The estimator enqueues every kernel on torch's CURRENT stream (PyTorch's side streams are not ordered against
    the legacy default stream): results under ``with torch.cuda.stream(s)`` equal the golden ones."""
    import torch
    g = golden_estimator
    genome, reads, aligner, est, cfg = _setup(g, default_model, 1)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        # keep the default stream busy so that an unordered read of the results would see stale data
        junk = torch.empty(64 << 20, device='cuda')
        for _ in range(4):
            junk.normal_()
        groups = est.estimate_probabilities(genome, reads, independent=False)
        tables = est.get_refined_alignments(reads)
    side.synchronize()
    assert len(groups) == int(g['tweak1/n_groups'])
    for gi, c in enumerate(groups):
        np.testing.assert_allclose(c.values, g['tweak1/group%d/probabilities' % gi], rtol=PROB_RTOL, atol=PROB_ATOL)
        assert np.array_equal(c.coverage, g['tweak1/group%d/coverage' % gi])
    for i, res in enumerate(tables):
        assert np.array_equal(res[1], g['tweak1/read%d/alignment_table' % i])


def test_meth_scores_on_gpu_alignments_match_reference_golden(golden_estimator, default_model):
    """detect_meth's scoring (detect_meth.py:26-60) fed by the GPU path -- refined alignments and expected levels
    from the device -- equals the golden scores the REFERENCE's detect_meth computed on its own alignments of the same
    reads, bit for bit."""
    from nadavca_b200.detect_meth import calculate_meth_scores, maxs3
    g = golden_estimator
    genome, reads, aligner, est, cfg = _setup(g, default_model, 1)
    results = est.get_refined_alignments(reads)
    total = 0
    for i, (read, res) in enumerate(zip(reads, results)):
        apx, table = res
        cut = read.normalized_signal[table[0][1]:table[-1][2]]
        feats = calculate_meth_scores(cut, table, apx, 'CG', default_model)
        assert [f[0] for f in feats] == g['meth/read%d/positions' % i].tolist()
        assert [f[1] for f in feats] == g['meth/read%d/contexts' % i].tolist()
        assert np.array_equal(np.array([f[2] for f in feats]).reshape(-1, 11), g['meth/read%d/scores' % i])
        assert [maxs3(f[2]) for f in feats] == g['meth/read%d/aggregated' % i].tolist()
        total += len(feats)
    assert total >= 10


@pytest.mark.parametrize('n_reads', [1, 4, 7])
def test_device_normalisation_equals_numpy_bit_for_bit(lib_built, n_reads):
    """Read.normalize_reads(device=...) == the host path (numpy.median twice + clip, read.py:67-81): exact radix
    select on the GPU, odd and even pooled counts, repeated values around the medians, integer raw signals."""
    from nadavca_b200.read import Read
    rng = np.random.default_rng(200 + n_reads)
    raws = []
    for i in range(n_reads):
        n = int(rng.integers(50, 4000)) + (i == 0)
        raw = np.round(rng.normal(90, 15, size=n) * 4) / 4.0          # many ties
        raw[rng.integers(0, n, size=5)] = rng.choice([-300.0, 800.0], size=5)  # outliers beyond the clip
        raws.append(raw.astype(np.int16) if i % 3 == 2 else raw)
    host = [Read.from_arrays(r, 'ACGT', {0: 0}) for r in raws]
    gpu = [Read.from_arrays(r, 'ACGT', {0: 0}) for r in raws]
    Read.normalize_reads(host)
    Read.normalize_reads(gpu, device=0)
    for a, b in zip(host, gpu):
        assert b.normalized_signal.dtype == np.float64
        assert np.array_equal(a.normalized_signal, b.normalized_signal)
    assert max(abs(b.normalized_signal).max() for b in gpu) == 5.0


def test_per_read_normalisation_equals_numpy_bit_for_bit(lib_built):
    """Read.normalize_each == Read.normalize_reads([read]) read by read (align_signal.py:54): one CTA per read, exact
    per-read median / MAD; odd and even lengths, heavy ties, a constant-but-one read, a one-sample-over-two read."""
    from nadavca_b200.read import Read
    rng = np.random.default_rng(77)
    raws = []
    for i in range(40):
        n = int(rng.integers(3, 6000))
        raw = np.round(rng.normal(90, 15, size=n) * 2) / 2.0
        if n > 20:
            raw[rng.integers(0, n, size=4)] = rng.choice([-300.0, 800.0], size=4)
        raws.append(raw.astype(np.int16) if i % 4 == 3 else raw)
    raws.append(np.array([1.0, 2.0, 4.0, 8.0]))
    raws.append(np.array([5.0, 5.0, 5.0, 9.0, 1.0]))
    host = [Read.from_arrays(r, 'ACGT', {0: 0}) for r in raws]
    gpu = [Read.from_arrays(r, 'ACGT', {0: 0}) for r in raws]
    with np.errstate(divide='ignore', invalid='ignore'):
        for read in host:
            Read.normalize_reads([read])
    Read.normalize_each(gpu, 0)
    for a, b in zip(host, gpu):
        assert b.normalized_signal.dtype == np.float64
        assert np.array_equal(a.normalized_signal, b.normalized_signal, equal_nan=True)  # MAD 0: 0/0 stays NaN in both


def test_batched_anchor_construction_matches_host_glue(lib_built):
    """csrc/anchors.cu (CIGAR walk -> matching-base anchors -> signal anchors and ranges) against the host functions
    that restate alignment.py:109-186, field by field: both strands, insertions / deletions / soft clips, mismatches,
    bases the basecaller did not place, a hit without any usable anchor and an unmapped read."""
    from nadavca_b200 import alignment
    from nadavca_b200.genome import Genome
    from nadavca_b200.read import Read
    rng = np.random.default_rng(301)
    alpha = np.array(list('ACGT'))
    G = 5000
    genome = alpha[rng.integers(0, 4, size=G)]
    reads, hits, want = [], [], []
    for i in range(40):
        is_rc = bool(i % 2)
        start = int(rng.integers(0, G - 700))
        ops, oriented, ref_pos = [], [], start
        if rng.random() < 0.5:
            n = int(rng.integers(1, 20)); ops.append((n, 'S')); oriented.extend(alpha[rng.integers(0, 4, size=n)])
        for _ in range(int(rng.integers(3, 40))):
            n = int(rng.integers(1, 45))
            seg = genome[ref_pos:ref_pos + n].copy()
            flip = rng.random(n) < 0.08
            seg[flip] = alpha[rng.integers(0, 4, size=int(flip.sum()))]
            ops.append((n, 'M')); oriented.extend(seg); ref_pos += n
            kind = rng.random()
            if kind < 0.3:
                n = int(rng.integers(1, 6)); ops.append((n, 'I')); oriented.extend(alpha[rng.integers(0, 4, size=n)])
            elif kind < 0.6:
                n = int(rng.integers(1, 6)); ops.append((n, 'D')); ref_pos += n
        if rng.random() < 0.5:
            n = int(rng.integers(1, 20)); ops.append((n, 'S')); oriented.extend(alpha[rng.integers(0, 4, size=n)])
        oriented = np.array(oriented)
        sequence = Genome.reverse_complement(oriented) if is_rc else oriented
        L = len(sequence)
        samples = np.cumsum(rng.integers(2, 15, size=L)) + 100
        placed = rng.random(L) < (0.0 if i == 7 else 0.9)   # read 7: no base was placed in the signal
        read = Read.from_arrays(rng.normal(90, 15, size=int(samples[-1]) + 150), sequence,
                                {int(b): int(samples[b]) for b in range(L) if placed[b]})
        Read.normalize_reads([read])
        cigar = ''.join('%d%s' % op for op in ops)
        reads.append(read)
        hits.append(None if i == 11 else (cigar, start, is_rc))
        if i == 11:
            want.append(None)
            continue
        mapping = alignment.base_mapping_from_cigar(cigar, start, sequence, genome, is_rc)
        want.append(alignment.signal_alignment_from_base_mapping(read, mapping, is_rc, 'contig', genome, 37))
    got = alignment.batch_signal_alignments(reads, hits, genome, 37, contig_name='contig')
    assert want[7] is None and want[11] is None and sum(w is not None for w in want) >= 36
    for g, w in zip(got, want):
        if w is None:
            assert g is None
            continue
        assert np.array_equal(g.alignment, w.alignment)
        assert g.signal_range == tuple(w.signal_range) and g.reference_range == tuple(w.reference_range)
        assert g.read_sequence_range == tuple(w.read_sequence_range)
        assert g.reverse_complement == w.reverse_complement and g.contig_name == w.contig_name
        assert np.array_equal(g.reference_part, w.reference_part)
