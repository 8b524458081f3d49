"""CPU suite, part 2: host-side logic of the drop-in (no GPU, no oracle compute): model file reader, packing,
overlap groups, sharding, alignment contract, config handling, cell/byte accounting used by bench.py."""
import io
import os

import numpy as np
import pytest

from conftest import GOLDEN_CONFIG, ROOT, golden_reads


def test_hdf5_mini_reads_shipped_model(default_model_host):
    """kmer_model.hdf5 without h5py: 4096 6-mers, central_pos 2, constant sd (SURVEY.md 8c)."""
    km = default_model_host
    assert (km.get_k(), km.get_central_position(), km.get_alphabet_size()) == (6, 2, 4)
    assert km.mean.shape == (4096,) and km.sigma.shape == (4096,)
    assert np.all(km.sigma == 0.3328800486427912)
    assert abs(km.mean.min() + 3.178) < 1e-3 and abs(km.mean.max() - 2.831) < 1e-3
    from nadavca_b200.kmer_model import kmer_to_id
    assert kmer_to_id('AAAAAA') == 0 and kmer_to_id('TTTTTT') == 4095 and kmer_to_id('ACGTAC') == 0b000110110001


def test_genome_helpers():
    from nadavca_b200.genome import Genome
    assert Genome.to_numerical('ACGTTG').tolist() == [0, 1, 2, 3, 3, 2]
    assert ''.join(Genome.reverse_complement('AACGT')) == 'ACGTT'
    assert ''.join(Genome.reverse_complement(np.array(list('TTGA')))) == 'TCAA'
    with pytest.raises(KeyError):
        Genome.to_numerical('ACGN')
    fq = Genome.create_from_fastq_string('@r1\nACGT\n+\nIIII\n')
    assert ''.join(fq[0].bases) == 'ACGT'


def test_fasta_loader(tmp_path):
    from nadavca_b200.genome import Genome
    p = tmp_path / 'x.fa'
    p.write_text('>chr1 test\nACGT\nTTAA\n>chr2\nGG\n')
    gs = Genome.load_from_fasta(str(p))
    assert [g.description for g in gs] == ['>chr1 test', '>chr2']
    assert ''.join(gs[0].bases) == 'ACGTTTAA' and ''.join(gs[1].bases) == 'GG'


def test_group_intervals_touching_chunks_split():
    """estimator.py:216 uses '>=': a chunk starting exactly at the running end opens a new group (SURVEY Q9)."""
    from nadavca_b200.estimator import group_intervals
    iv = [(100, 200), (0, 50), (40, 90), (90, 100), (150, 260), (300, 310)]
    groups = group_intervals(iv)
    assert [(g[0], g[1]) for g in groups] == [(0, 90), (90, 100), (100, 260), (300, 310)]
    assert [sorted(g[2]) for g in groups] == [[1, 2], [3], [0, 4], [5]]
    assert group_intervals([]) == []
    # a contained interval does not shorten the group
    assert [(g[0], g[1]) for g in group_intervals([(0, 100), (10, 20), (99, 120)])] == [(0, 120)]


def test_plan_groups_host_consensus_and_independent():
    from nadavca_b200.estimator import plan_groups_host
    iv = [(10, 30), (20, 50), (50, 60)]
    groups, off, dest = plan_groups_host(iv, independent=False)
    assert [(g[0], g[1]) for g in groups] == [(10, 50), (50, 60)]
    assert off.tolist() == [0, 40, 50] and dest.tolist() == [0, 10, 40]
    groups, off, dest = plan_groups_host(iv, independent=True)
    assert off.tolist() == [0, 20, 50, 60] and dest.tolist() == [0, 20, 50]
    assert plan_groups_host([], independent=False) is None


def test_shard_reads_balances_work():
    from nadavca_b200.estimator import shard_reads
    rng = np.random.default_rng(0)
    work = rng.integers(1000, 3000, size=203).astype(float)
    for world in (1, 2, 4, 8):
        shards = shard_reads(work, world)
        assert sorted(i for s in shards for i in s) == list(range(203))
        loads = [work[s].sum() for s in shards]
        assert max(loads) - min(loads) <= work.max()
        assert all(s == sorted(s) for s in shards)


def test_reads_pack_layout_and_validation():
    from nadavca_b200._cabi import ReadsPack
    pack = ReadsPack([[0.5, 1.5, 2.5], [], [1.0]], [[0, 1], [], [3]], [[], [2], []], [[1], [], []],
                     [[[0, 0], [2, 1]], np.zeros((0, 2)), [[0, 0]]], 7, 2)
    assert pack.n_reads == 3
    assert pack.signal_off.tolist() == [0, 3, 3, 4] and pack.signal.dtype == np.float64
    assert pack.reference_off.tolist() == [0, 2, 2, 3] and pack.reference.dtype == np.int32
    assert pack.context_before_off.tolist() == [0, 0, 1, 1] and pack.context_after_off.tolist() == [0, 1, 1, 1]
    assert pack.anchor_off.tolist() == [0, 2, 2, 3] and pack.anchors.tolist() == [0, 0, 2, 1, 0, 0]
    assert (pack.struct.n_reads, pack.struct.bandwidth, pack.struct.min_event_length) == (3, 7, 2)
    assert pack.total_reference == 3 and pack.total_signal == 4
    with pytest.raises(ValueError):
        ReadsPack([[1.0]], [[0]], [[]], [[]], [[1, 2, 3]], 1, 1)      # anchors must be pairs
    with pytest.raises(ValueError):
        ReadsPack([[1.0]], [[0], [1]], [[]], [[]], [[[0, 0]]], 1, 1)  # ragged argument lists
    again = ReadsPack.from_packed(pack.signal, pack.signal_off, pack.reference, pack.reference_off,
                                  pack.context_before, pack.context_before_off, pack.context_after,
                                  pack.context_after_off, pack.anchors, pack.anchor_off, 7, 2)
    assert again.signal is pack.signal and again.n_reads == 3
    with pytest.raises(ValueError):
        ReadsPack.from_packed(pack.signal.astype(np.float32), pack.signal_off, pack.reference, pack.reference_off,
                              pack.context_before, pack.context_before_off, pack.context_after,
                              pack.context_after_off, pack.anchors, pack.anchor_off, 7, 2)


def test_chunk_contract():
    from nadavca_b200.estimator import Chunk
    a, b, c = Chunk(5, 9, np.zeros((4, 4))), Chunk(5, 7, np.zeros((2, 4))), Chunk(1, 20, np.zeros((19, 4)))
    assert sorted([a, b, c]) == [c, b, a]
    assert a.coverage.tolist() == [1, 1, 1, 1]
    out = io.StringIO()
    Chunk.print_head(out)
    Chunk(1, 3, np.array([[.25] * 4, [1, 0, 0, 0]]), np.array([2, 3])).print(out, 'ACGT')
    lines = out.getvalue().splitlines()
    assert lines[0] == 'index\tbase\tcoverage\tA\tC\tG\tT'
    assert lines[1] == '1\tC\t2\t' + '\t'.join(['0.2500000000000000'] * 4)
    assert lines[2].startswith('2\tG\t3\t1.0000000000000000\t0.0')


def test_config_loading(tmp_path):
    from nadavca_b200 import defaults
    cfg = defaults.load_config()
    assert cfg == dict(bandwidth=150, snp_prior_probability=0.001, min_event_length=2, model_wobbling=True,
                       model_transitions=True, tweak_signal_normalization=True, normalization_event_length=10)
    assert defaults.load_config(dict(cfg, bandwidth=30))['bandwidth'] == 30
    with pytest.raises(KeyError):
        defaults.load_config({'bandwidth': 3})
    with pytest.raises(FileNotFoundError):
        defaults.load_config(str(tmp_path / 'missing.yaml'))


def test_synthetic_aligner_contract(golden_estimator):
    """Layout of ApproximateSignalAlignment (alignment.py:142-186) on both strands."""
    from nadavca_b200 import synthetic
    from nadavca_b200.genome import Genome
    from nadavca_b200.read import Read
    genome = golden_estimator['genome']
    reads = golden_reads(golden_estimator)
    Read.normalize_reads(reads)
    aligner = synthetic.SyntheticAligner(genome)
    for r in reads:
        apx = aligner.get_signal_alignment(r, 30)
        n = apx.reference_range[1] - apx.reference_range[0]
        assert apx.alignment[0][1] == 0 and apx.alignment[-1][1] == n - 1
        assert np.all(np.diff(apx.alignment[:, 1]) > 0) and np.all(np.diff(apx.alignment[:, 0]) >= 0)
        s0, s1 = apx.signal_range
        assert 0 <= s0 < s1 <= len(r.normalized_signal)
        assert apx.alignment[0][0] == min(30, apx.alignment[0][0] + s0)  # first anchor sits `bandwidth` in
        part = genome[apx.reference_range[0]:apx.reference_range[1]]
        if apx.reverse_complement:
            part = Genome.reverse_complement(part)
        assert np.array_equal(apx.reference_part, part) and len(part) == n
        a, b = apx.read_sequence_range
        assert b - a >= n  # anchored bases of the read span the reference part (substitutions never add bases)
    assert aligner.get_signal_alignment(Read(), 30) is None


def test_cigar_base_mapping():
    from nadavca_b200.alignment import base_mapping_from_cigar, parse_cigar
    assert parse_cigar('3S10M2D4M1I') == [(3, 'S'), (10, 'M'), (2, 'D'), (4, 'M'), (1, 'I')]
    ref = np.array(list('AACCGGTTAC'))
    read = np.array(list('TACCGTTT'))  # 1S 4M 1D 2M 1S against ref[1:]
    m = base_mapping_from_cigar('1S4M1D2M1S', 1, read, ref, False)
    assert m.tolist() == [[1, 1], [2, 2], [3, 3], [4, 4], [5, 6], [6, 7]]
    with pytest.raises(ValueError):
        base_mapping_from_cigar('3X', 0, read, ref, False)


def test_read_normalisation_and_tweak_match_reference(golden_estimator):
    """Read.normalize_reads == the reference's (stored normalised signals); the tweak is the same scipy call."""
    from nadavca_b200.read import Read
    reads = golden_reads(golden_estimator)
    Read.normalize_reads(reads)
    for i, r in enumerate(reads):
        assert np.array_equal(r.normalized_signal, golden_estimator['read%d/normalized_signal' % i])
        assert r.normalized_signal.min() >= -5 and r.normalized_signal.max() <= 5
    with pytest.raises(NotImplementedError):
        Read.load_from_fast5('x.fast5', 'Analyses/Basecall_1D_000')


def test_band_stats_matches_oracle_counts(golden_dp):
    """bench.py's cell accounting == the oracle's count_cells on the same bands."""
    import bench
    from oracle import oracle as orc
    for tag in ['model6_0', 'model6_1', 'rnd09']:
        c = golden_dp.case(tag)
        k, cp, bw, mel = (int(x) for x in c['params'])
        n, N = len(c['reference']), len(c['signal'])
        bs, be = orc.band_bounds(c['anchors'], N, n, bw)
        cells, nbytes = bench.band_stats([(bs, be)], k, cp, True)
        want = orc.count_cells(c['anchors'], N, n, bw, k, cp)
        assert cells['refine_plain'] == want['refine_plain']
        assert cells['estimate_fb'] == want['estimate_fb']
        assert cells['estimate_snp'] == want['estimate_snp']
        assert all(v > 0 for v in nbytes.values())


def test_product_never_imports_oracle():
    """The oracle is test infrastructure: nothing under nadavca_b200/ may import or execute it."""
    pkg = os.path.join(ROOT, 'nadavca_b200')
    for dirpath, _, files in os.walk(pkg):
        for name in files:
            if name.endswith(('.py', '.cu', '.cuh', '.h')):
                text = open(os.path.join(dirpath, name), errors='replace').read()
                assert 'import oracle' not in text and 'from oracle' not in text and 'oracle/' not in text, name


def test_tweak_with_precomputed_event_means(golden_estimator):
    """Read.tweak_signal_normalization gives the same spline whether the event means come from its own numpy.mean
    loop (reference behaviour, read.py:83-94) or are passed in (the device-computed ones are bit-identical)."""
    from nadavca_b200.read import Read
    reads = golden_reads(golden_estimator)
    Read.normalize_reads(reads)
    r = reads[0]
    table = golden_estimator['tweak1/read0/alignment_table']
    events = table[:, 1:]
    rng = np.random.default_rng(3)
    expected = [float(np.mean(r.normalized_signal[s:e])) + rng.normal(0, 0.2) for s, e in events]
    r.tweak_signal_normalization(events, expected)
    a = r.tweaked_normalized_signal.copy()
    means = [float(np.mean(r.normalized_signal[s:e])) for s, e in events]
    r.tweak_signal_normalization(events, expected, means)
    assert np.array_equal(a, r.tweaked_normalized_signal)


def test_meth_scores_match_reference_golden(golden_estimator, default_model_host):
    """calculate_meth_scores / maxs3 == nadavca/detect_meth.py:26-60 on the reference's own refined alignments
    (golden, pattern "CG"); the expected levels come from the oracle model so the test needs no GPU."""
    from nadavca_b200 import synthetic
    from nadavca_b200.detect_meth import calculate_meth_scores, maxs3
    from nadavca_b200.read import Read
    from oracle import oracle as orc
    g = golden_estimator
    km = default_model_host
    om = orc.OracleModel(km.get_k(), km.get_central_position(), 4, km.mean, km.sigma, 'port')
    reads = golden_reads(g)
    Read.normalize_reads(reads)
    aligner = synthetic.SyntheticAligner(g['genome'])
    total = 0
    for i, r in enumerate(reads):
        table = g['tweak1/read%d/alignment_table' % i]
        apx = aligner.get_signal_alignment(r, 30)
        cut = r.normalized_signal[table[0][1]:table[-1][2]]
        feats = calculate_meth_scores(cut, table, apx, 'CG', om)
        assert [f[0] for f in feats] == g['meth/read%d/positions' % i].tolist()
        assert [f[1] for f in feats] == g['meth/read%d/contexts' % i].tolist()
        got = np.array([f[2] for f in feats]).reshape(-1, 11)
        assert np.array_equal(got, g['meth/read%d/scores' % i])
        assert [maxs3(f[2]) for f in feats] == g['meth/read%d/aggregated' % i].tolist()
        total += len(feats)
    assert total >= 10


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the reference's own CPU path on the host cores) prints one JSON line with the
    contract's keys; a tiny sample keeps the CPU suite fast."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--cpu-sample', '2',
                          '--bases', '150', '--steps', '1', '--warmup', '1'], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith('{')][-1])
    assert line['impl'] == 'reference' and line['metric'] == 'signal_samples_aligned_per_sec'
    assert line['unit'] == 'samples/s' and line['higher_is_better'] is True and line['value'] > 0
    assert line['cpu_baseline']['kind'] in ('reference', 'port') and line['cpu_baseline']['cores'] >= 1
    assert line['e2e'] == {'value': line['value'], 'unit': 'samples/s', 'h2d_bytes_per_step': 0,
                           'd2h_bytes_per_step': 0}
    assert 'workload' in line['config'] and line['vs_baseline'] is None


def test_bench_dump_selection():
    """--dump-outputs writes every read when the batch fits its budget, otherwise the same seeded sample on every
    call, within the budget."""
    import bench
    rng = np.random.default_rng(5)
    small = rng.integers(300, 500, size=24)
    assert bench.dump_selection(small).tolist() == list(range(24))
    big = rng.integers(1800, 2200, size=1000)
    keep = bench.dump_selection(big)
    assert np.array_equal(keep, bench.dump_selection(big.copy()))
    assert np.all(np.diff(keep) > 0) and 100 < len(keep) < 1000
    cost = big[keep] * bench.DUMP_BYTES_PER_ROW + bench.DUMP_BYTES_PER_READ
    assert cost.sum() <= bench.DUMP_BYTES < 64 << 20
    assert len(bench.dump_selection([bench.DUMP_BYTES])) == 0  # one read larger than the budget: nothing fits


def test_bench_rejects_bad_arguments():
    import subprocess
    import sys
    for extra in (['--steps', '0'], ['--impl', 'reference', '--dump-outputs', 'unused']):
        out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + extra, capture_output=True, text=True,
                             timeout=120)
        assert out.returncode == 2 and 'error' in out.stderr, extra


def test_output_writers_keep_the_reference_layout(tmp_path):
    """.npz of `nadavca align` (align_signal.py:83-132) and the SNP table of `nadavca snp` (estimator.py:21-31)."""
    from nadavca_b200 import output
    from nadavca_b200.alignment import ApproximateSignalAlignment
    from nadavca_b200.estimator import Chunk
    from nadavca_b200.read import Read
    read = Read.from_arrays(np.arange(100, 160), 'ACGTAC', {i: 10 * i for i in range(6)})
    apx = ApproximateSignalAlignment(np.zeros((0, 2), dtype=int), (0, 60), (7, 11), (1, 5), True,
                                     np.array(list('GATT')), 'chr1')
    table = np.array([[10, 5, 12], [9, 12, 20], [8, 20, 31], [7, 31, 40]])
    path = output.write_alignment_npz(str(tmp_path / 'r0'), read, apx, table)
    z = np.load(path)
    assert z['arr_0'].tolist() == list(range(105, 131))          # raw signal from the first to the last event START
    labels = z['arr_1']
    assert len(labels) == 26 and labels[0] == 'G' and labels[7] == 'A' and labels[15] == 'T'
    assert (labels != 'N').sum() == 3                            # the last base gets no label (alignment[:-1])
    assert z['arr_2'].tolist() == ['7', '-', 'chr1', 'ACGTAC']
    bad = table.copy()
    bad[2, 1] = 12
    with pytest.raises(output.AlignException):
        output.sample_labels(apx, bad)
    assert output.write_alignment_npz(str(tmp_path / 'e'), read, apx, np.array([[1, 5, 5], [2, 5, 9]])) is None
    chunk = Chunk(2, 4, np.array([[0.25, 0.25, 0.25, 0.25], [1.0, 0.0, 0.0, 0.0]]), np.array([3, 1]))
    output.write_snp_tables([chunk], 'ACGTACGT', str(tmp_path / 'snps.txt'))
    lines = open(tmp_path / 'snps.txt').read().splitlines()
    assert lines[0] == 'index\tbase\tcoverage\tA\tC\tG\tT'
    assert lines[1] == '2\tG\t3\t' + '\t'.join(['0.2500000000000000'] * 4)
    assert lines[2].startswith('3\tT\t1\t1.0000000000000000\t0.0000000000000000')
    output.write_snp_tables([chunk, None], 'ACGTACGT', str(tmp_path / 'ind'), independent=True, names=['a.fast5', 'b'])
    assert sorted(os.listdir(tmp_path / 'ind')) == ['a.txt']


def test_linear_fit_equals_scipy_linregress():
    """align_signal's fast slope / intercept == scipy.stats.linregress bit for bit (align_signal.py:73)."""
    from scipy.stats import linregress
    from nadavca_b200.align_signal import linear_fit
    rng = np.random.default_rng(17)
    for n in (2, 3, 17, 500, 2000, 2311):
        x = rng.normal(0, 1.3, size=n)
        y = 0.93 * x + 0.07 + rng.normal(0, 0.2, size=n)
        want = linregress(x, y)
        slope, intercept = linear_fit(x, list(y))
        assert slope == want.slope and intercept == want.intercept, n
    with_nan = np.array([0.1, np.nan, 0.5])
    s, i = linear_fit(np.array([0.0, 1.0, 2.0]), with_nan)
    assert np.isnan(s) and np.isnan(i)


def test_fit_splines_pool_equals_inline(golden_estimator):
    """The worker-process pool of the spline fits returns exactly what the inline scipy call returns."""
    from nadavca_b200.read import fit_spline, fit_splines_async
    rng = np.random.default_rng(23)
    jobs = []
    for i in range(40):
        n = int(rng.integers(30, 200))
        expected = rng.normal(0, 1.2, size=n)
        means = expected + rng.normal(0, 0.15, size=n)
        means[::17] += 3.0  # dropped by the |expected - mean| <= 1 filter
        jobs.append((means, expected))
    inline = [fit_spline(*j) for j in jobs]
    pooled = fit_splines_async(jobs, workers=3).get()
    few = fit_splines_async(jobs[:5], workers=3).get()
    for a, b in zip(inline, pooled):
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and a[2] == b[2]
    for a, b in zip(inline, few):
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_device_exp_restated_in_numpy():
    """The emission exp of csrc/dp3.cuh (exp_ext_scaled: scaled argument, 256-entry table, degree-4 polynomial),
    restated with the table and the constants READ FROM THE SOURCE, against 60-digit arithmetic: every table entry is
    the correctly rounded 2^(j/256) and p * 2^k is within 3e-16 of exp over the whole range of emission exponents."""
    import re
    import mpmath
    mpmath.mp.prec = 200
    src = open(os.path.join(ROOT, 'nadavca_b200', 'csrc', 'dp3.cuh')).read()
    body = src[src.index('g_exp_tab[256] = {') + len('g_exp_tab[256] = {'):]
    tab = np.array([float(x) for x in body[:body.index('};')].replace('\n', ' ').split(',')])
    assert len(tab) == 256
    for j in range(256):
        assert tab[j] == float(mpmath.power(2, mpmath.mpf(j) / 256))
    step, c4, c3 = [float(x) for x in re.search(r'c_exp_k\[3\] = \{([^}]*)\}', src).group(1).split(',')]
    scale = float(re.search(r'#define NVB_EXP_SCALE ([0-9.]+)', src).group(1))
    assert scale == float(256 / mpmath.log(2)) and step == float(mpmath.log(2) / 256)
    assert np.float64(c4).view(np.uint64) & np.uint64(0xffffffff) == 0 and abs(c4 * 24 - 1) < 2e-6

    def fma(a, b, c):
        return float(mpmath.mpf(a) * mpmath.mpf(b) + mpmath.mpf(c))

    rng = np.random.default_rng(0)
    logs = np.concatenate([rng.uniform(-60, 3, 1500), rng.uniform(-3300, -60, 400), -np.abs(rng.normal(0, 1e-3, 100)),
                           [0.0, -1e-300, 2.5]])
    magic = 6755399441055744.0
    worst = 0.0
    for ls in logs * scale:
        t = ls + magic
        n = int(t - magic)
        r = (ls - (t - magic)) * step
        q = fma(r, c4, c3)
        q = fma(q, r, 0.5)
        q = fma(q, r, 1.0)
        q = q * r
        p = fma(tab[n & 255], q, tab[n & 255])
        assert 0.99 < p < 2.0
        true = mpmath.exp(mpmath.mpf(ls) * mpmath.log(2) / 256)
        worst = max(worst, abs(float((mpmath.mpf(p) * mpmath.power(2, n >> 8) - true) / true)))
    assert worst < 3e-16, worst
