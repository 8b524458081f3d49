"""Reads whose DP cells sit more than 2^31 elements into the planes of a wave.

The library plans a batch into waves of consecutive reads that share the model's DP workspace (api.cu plan_waves): read
b's prefix and suffix matrices start at cell mat_base[b] of the planes, and the kernels add per-read row offsets
(cell_off) and column terms to it.  A default wave is sized to 70 % of free HBM, so at the benchmark's shape (~2 kb
reads, bandwidth 150, ~0.6 M cells per read and plane) production waves hold more than 2^31 cells, while every other
check in this repository stays far below that: one missing 64-bit promotion in an offset would corrupt the tail of
a large wave unnoticed.

This file runs one batch of N_READS such reads under an explicit workspace limit (the bytes of one refine wave holding
them all) that puts every op's waves past 2^31 cells:
  - refine without transitions, estimate plain and wobble: one wave of every read;
  - refine with transitions (twice the cells): two waves of half the reads each, both past 2^31.
Each such wave has a straddling read (mat_base < 2^31 < mat_base + cells: its own rows cross the boundary) and at
least MIN_TAIL tail reads (mat_base >= 2^31).  `op_plan` restates the planner with citations, and
test_large_offset_plan checks all of this on the host, without a GPU.

On the GPU, under the automatic sweep schedule (the rotating wavefront of rows5.cu at these band widths) and the forced
stripes (rows4.cu):
  1. the straddling and tail reads give bit-identical results in the large batch and in a batch of only those reads,
     where their offsets are near 0: bands, events and event means of both refine modes, alignment tables,
     log-likelihoods, chunk values and both stored planes of both estimate modes;
  2. every read gives bit-identical events and log-likelihoods when the same batch runs as about 8 waves;
  3. the straddling and tail reads match the oracle port (events bit-exact, structural ties counted; raw
     log-likelihoods rtol 1e-9), and two of them, one per strand, match the extended-precision reference
     (test_gpu_extended_precision.py part a) in both estimate modes;
  4. the private model's workspace is exactly the planned peak, and the device's free memory comes back when the
     batches and the model are gone and the library's block cache is trimmed.

Out of scope: record words and reference positions stay below 2^31 at this size (about 1e9 words and 7e6 positions);
a single read of more than 2^31 cells (over 50 GB of planes and hours of oracle time); multi-rank consensus.
"""
import functools
import hashlib
import os
import time

import numpy as np
import pytest

from conftest import ROOT
from test_gpu_extended_precision import _check_read, _truth_job, exponent_term
from test_gpu_kernel_edges import B200_SMS, Geom, path_columns_per_lane, rotates

MODEL_PATH = os.path.join(ROOT, 'nadavca_b200', 'default', 'kmer_model.hdf5')
N_READS = 3640
GENOME_LENGTH, GENOME_SEED, READ_SEED = 1_000_000, 31, 310_000
BW, MEL = 150, 2
NORMALIZATION_EVENT_LENGTH = 10.0
BOUNDARY = 2 ** 31  # the first cell index a signed 32-bit offset cannot hold
MIN_TAIL = 16
SMALL_WAVES = 8  # the second run: the same batch in about this many waves
MAX_PEAK = 60e9  # the GPU is shared: the case stays below this many bytes of workspace
MEMORY_MARGIN = 4 << 30
RELEASE_SLACK = 1 << 30
LL_RTOL = 1e-9
SCHEDULES = (None, 's')

# (label, kind, flag, mode), in the order they run: the first op's waves are the largest in cells, path scratch and
# record words (test_large_offset_plan checks it), so the model's workspace is allocated once and never regrows
OPS = (('refine-plain', 'refine', False, 'plain'), ('refine-trans', 'refine', True, 'trans'),
       ('estimate-plain', 'estimate', False, 'plain'), ('estimate-wobble', 'estimate', True, 'wobble'))


# ---- the case and the wave plan, on the host -------------------------------------------------------------------------

class LargeCase:
    """N_READS reads: `reads` (signal, reference, ctx_before, ctx_after, anchors) as the estimator passes them to the
    DP, `meta` (start_in_signal, ref_start, ref_end, reverse) as it passes them to the alignment table, and the band
    geometry of each (test_gpu_kernel_edges.Geom, from orc.band_bounds)."""

    def __init__(self, reads, meta):
        self.reads, self.meta = reads, meta
        self.geoms = [Geom(r, BW) for r in reads]
        self.pk = path_columns_per_lane(max(g.maxw for g in self.geoms if not g.bad))  # api.cu batch_init


@functools.lru_cache(maxsize=1)
def large_case():
    """Seeded reads of the benchmark's shape (synthetic.make_read defaults: ~2000 bases, ~10 samples per base, random
    strand) on a 1 Mb genome, normalised together, bandwidth 150, min_event_length 2."""
    from nadavca_b200 import synthetic
    from nadavca_b200.kmer_model import KmerModel
    from nadavca_b200.read import Read
    from oracle import oracle as orc
    km = KmerModel.load_from_hdf5(MODEL_PATH)  # host tables only: this model never gets a device handle
    k, cp = km.get_k(), km.get_central_position()
    genome = synthetic.make_genome(GENOME_LENGTH, seed=GENOME_SEED)
    raw = [synthetic.make_read(genome, km, i, seed_base=READ_SEED) for i in range(N_READS)]
    Read.normalize_reads(raw)
    aligner = synthetic.SyntheticAligner(genome)
    reads, meta = [], []
    for r in raw:
        apx = aligner.get_signal_alignment(r, BW)
        s0, s1 = apx.signal_range
        a, b = apx.read_sequence_range
        reads.append((np.asarray(r.normalized_signal[s0:s1], dtype=np.float64), orc.to_numerical(apx.reference_part),
                      orc.to_numerical(r.sequence[a - cp:a]), orc.to_numerical(r.sequence[b:b + k - cp - 1]),
                      np.asarray(apx.alignment)))
        meta.append((s0, apx.reference_range[0], apx.reference_range[1], int(bool(apx.reverse_complement))))
    return LargeCase(reads, meta)


def op_plan(geoms, mode, need_dp, limit, pk):
    """api.cu plan_waves with an explicit workspace limit: a wave takes consecutive reads while its bytes -- 24 per
    matrix cell (api.cu matrix_cells: two double mantissa and two int32 exponent planes), and for refine 8 per double
    of path scratch (two rows of the read's widest band row) and 4 per record word (api.cu record_words) -- stay
    within `limit`.  -> (waves as dicts b0, b1, cells, dp, rec; mat_base per read, the first cell of its matrices in
    its wave's planes)."""
    n = len(geoms)
    mat_base = np.zeros(n, dtype=np.int64)
    waves, i = [], 0
    while i < n:
        cells = dp = rec = 0
        j = i
        while j < n:
            g = geoms[j]
            c = g.matrix_cells(mode)
            d = 2 * g.maxw if need_dp else 0
            rw = g.record_words(mode, pk) if need_dp else 0
            if 24 * (cells + c) + 8 * (dp + d) + 4 * (rec + rw) > limit:
                assert j > i, 'read %d alone exceeds the workspace limit' % j
                break
            mat_base[j] = cells
            cells, dp, rec = cells + c, dp + d, rec + rw
            j += 1
        waves.append(dict(b0=i, b1=j, cells=cells, dp=dp, rec=rec))
        i = j
    return waves, mat_base


def crossings(geoms, mode, waves, mat_base):
    """Per wave past 2^31 cells: its straddling read (mat_base < 2^31 < mat_base + cells) and its tail reads
    (mat_base >= 2^31)."""
    out = []
    for wi, w in enumerate(waves):
        if w['cells'] <= BOUNDARY:
            continue
        idx = range(w['b0'], w['b1'])
        straddle = [j for j in idx if mat_base[j] < BOUNDARY < mat_base[j] + geoms[j].matrix_cells(mode)]
        tail = [j for j in idx if mat_base[j] >= BOUNDARY]
        out.append(dict(wave=wi, straddle=straddle, tail=tail))
    return out


def launches(kind, n_waves):
    """Kernel launches counted by the batch for one op: api.cu nvb_batch_refine counts 3 per wave (sweep, score, path),
    nvb_batch_estimate 1 (fill_status) + 3 per wave (sweep, no-SNP total, SNP)."""
    return 3 * n_waves if kind == 'refine' else 1 + 3 * n_waves


def full_plan(case):
    """The two limits, the wave plans of every op under each, the reads to check and the peak workspace bytes."""
    geoms, pk = case.geoms, case.pk
    whole = op_plan(geoms, 'plain', True, 1 << 62, pk)[0][0]
    limit = 24 * whole['cells'] + 8 * whole['dp'] + 4 * whole['rec']  # refine without transitions, every read at once
    # every wave but the last of the second run holds more than limit / SMALL_WAVES bytes: at most SMALL_WAVES waves
    small = -(-limit // SMALL_WAVES) + max(g.wave_bytes('trans', True, pk) for g in geoms)
    plans, small_plans = {}, {}
    for label, kind, _, mode in OPS:
        waves, mat_base = op_plan(geoms, mode, kind == 'refine', limit, pk)
        plans[label] = dict(waves=waves, mat_base=mat_base, crossings=crossings(geoms, mode, waves, mat_base))
        small_plans[label] = op_plan(geoms, mode, kind == 'refine', small, pk)[0]
    checked = sorted({j for p in plans.values() for c in p['crossings'] for j in c['straddle'] + c['tail']})
    top = {key: max(w[key] for p in plans.values() for w in p['waves']) for key in ('cells', 'dp', 'rec')}
    peak = 24 * top['cells'] + 8 * top['dp'] + 4 * top['rec']
    return dict(limit=limit, small=small, plans=plans, small_plans=small_plans, checked=checked, top=top, peak=peak)


def describe_plan(case, plan):
    lines = ['%d reads, limit %d bytes (%.2f GB), second run %d bytes; peak workspace %d bytes (%.2f GB: %d cells, '
             '%d path-scratch doubles, %d record words)' % (
                 N_READS, plan['limit'], plan['limit'] / 1e9, plan['small'], plan['peak'], plan['peak'] / 1e9,
                 plan['top']['cells'], plan['top']['dp'], plan['top']['rec'])]
    for label, _, _, mode in OPS:
        p = plan['plans'][label]
        parts = []
        for c in p['crossings']:
            s = c['straddle'][0]
            parts.append('wave %d: %.4f x 2^31 cells, straddling read %d at cells [%d, %d), %d tail reads %d..%d' % (
                c['wave'], p['waves'][c['wave']]['cells'] / BOUNDARY, s, p['mat_base'][s],
                p['mat_base'][s] + case.geoms[s].matrix_cells(mode), len(c['tail']), c['tail'][0], c['tail'][-1]))
        lines.append('  %-15s %d wave(s) (second run %d); %s' % (label, len(p['waves']), len(plan['small_plans'][label]),
                                                               '; '.join(parts)))
    lines.append('  %d reads checked against the batch of only them and against the oracle' % len(plan['checked']))
    return '\n'.join(lines)


def test_large_offset_plan():
    """On the host: in every op some wave exceeds 2^31 cells and holds a straddling read and at least MIN_TAIL tail
    reads; refine without transitions and both estimates run as one wave, refine with transitions as two; the first op
    sizes every workspace buffer; the peak stays below MAX_PEAK; the second run has about SMALL_WAVES waves; the
    automatic schedule runs the rotating sweep on every wave."""
    case = large_case()
    plan = full_plan(case)
    print(describe_plan(case, plan))
    assert not any(g.bad for g in case.geoms)
    for label, kind, _, mode in OPS:
        p = plan['plans'][label]
        assert len(p['waves']) == (2 if mode == 'trans' else 1), label
        assert p['crossings'], '%s: no wave exceeds 2^31 cells' % label
        for c in p['crossings']:
            assert len(c['straddle']) == 1, '%s wave %d: no straddling read' % (label, c['wave'])
            assert len(c['tail']) >= MIN_TAIL, '%s wave %d: %d tail reads' % (label, c['wave'], len(c['tail']))
        first = plan['plans'][OPS[0][0]]['waves']
        for key in ('cells', 'dp', 'rec'):
            assert max(w[key] for w in p['waves']) <= max(w[key] for w in first), '%s regrows %s' % (label, key)
        for w in p['waves']:
            maxw = max(g.maxw for g in case.geoms[w['b0']:w['b1']])
            no_rot = any(g.no_rotation for g in case.geoms[w['b0']:w['b1']])
            assert rotates(mode, maxw, w['b1'] - w['b0'], no_rot, None, B200_SMS), label
            assert not rotates(mode, maxw, w['b1'] - w['b0'], no_rot, 's', B200_SMS), label
        n_small = len(plan['small_plans'][label])
        assert SMALL_WAVES - 1 <= n_small // (2 if mode == 'trans' else 1) <= SMALL_WAVES, (label, n_small)
    assert BOUNDARY * 24 < plan['peak'] <= MAX_PEAK
    assert len({case.meta[j][3] for j in plan['checked']}) == 2, 'the checked reads cover both strands'


# ---- the GPU runs ------------------------------------------------------------------------------------------------------

def _digest(a):
    return hashlib.blake2b(np.ascontiguousarray(a).tobytes(), digest_size=16).hexdigest()


def _stored_rows(batch, read, cells):
    """Both stored planes of one read after estimate (nvb_batch_debug_rows) as digests; the cell count comes from the
    host geometry (Batch.debug_rows would copy the bands of the whole batch for every call)."""
    import ctypes
    from nadavca_b200 import _cabi
    out = []
    for plane in (0, 1):
        rows = np.zeros(cells, dtype=np.float64)
        _cabi.check(batch.lib.nvb_batch_debug_rows(batch.handle, int(read), plane, _cabi.ptr(rows, ctypes.c_double),
                                                   int(cells)), 'nvb_batch_debug_rows')
        out.append(_digest(rows))
    return tuple(out)


def _run(km, case, idx, limit, keep):
    """One batch of the reads `idx` (in that order) under the current sweep schedule, every op of OPS.  -> dict:
    'launches' per op; 'all' per op the events or log-likelihoods of every read, with the status; 'kept' for the batch
    positions `keep`, in that order: bands, and per op (events, event means, alignment table) or (log-likelihoods,
    chunk values, stored rows)."""
    import torch
    from nadavca_b200 import dtw
    reads = [case.reads[j] for j in idx]
    meta = np.array([case.meta[j] for j in idx], dtype=np.int64)
    out = {'launches': {}, 'all': {}, 'kept': {}}
    with dtw.Batch(km, *[[r[f] for r in reads] for f in range(5)], BW, MEL, workspace_limit=limit) as batch:
        bands = batch.bands()
        out['kept']['bands'] = [(bands[p][0].copy(), bands[p][1].copy()) for p in keep]
        off = batch.pack.reference_off
        for label, kind, flag, mode in OPS:
            before = batch.launch_count
            if kind == 'refine':
                batch.refine(flag)
                out['launches'][label] = batch.launch_count - before
                events, status = batch.events()
                out['all'][label] = (events, status)
                means = batch.event_means()
                tables = batch.alignment_tables(meta[:, 0], meta[:, 1], meta[:, 2], meta[:, 3].astype(np.int32))
                kept = [(events[p], means[p], tables[p]) for p in keep]
            else:
                batch.estimate(flag)
                out['launches'][label] = batch.launch_count - before
                ll, status = batch.log_likelihoods()
                out['all'][label] = (ll, status)
                chunks = torch.empty((batch.pack.total_reference, 4), dtype=torch.float64, device='cuda')
                batch.chunk_values(meta[:, 3].astype(np.int32), NORMALIZATION_EVENT_LENGTH, chunks.data_ptr())
                chunks = chunks.cpu().numpy()
                kept = [(ll[p], chunks[off[p]:off[p + 1]].copy(), _stored_rows(batch, p, case.geoms[idx[p]].cells))
                        for p in keep]
            out['kept'][label] = kept
    return out


def _same(a, b):
    """Bit-identical (NaN and signed zeros included), None only against None."""
    if a is None or b is None:
        return a is None and b is None
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


def _diff_all(one, other):
    """Reads whose events / log-likelihoods differ between two runs of the whole batch, per op."""
    out = {}
    for label, _, _, _ in OPS:
        (x, sx), (y, sy) = one['all'][label], other['all'][label]
        out[label] = [j for j in range(N_READS) if sx[j] != sy[j] or not _same(x[j], y[j])]
    return out


@pytest.fixture(scope='module')
def pool():
    import multiprocessing as mp
    p = mp.get_context('spawn').Pool(min(os.cpu_count() or 1, 48))
    yield p
    p.terminate()


@pytest.fixture(scope='module')
def large_runs(lib_built, pool):
    """Every GPU run of this file, on a private model, then the release: the batches closed, the model destroyed, the
    library's block cache trimmed.  The oracle and the extended reference start first in the pool and run meanwhile."""
    import torch
    from nadavca_b200 import _cabi, dtw
    from nadavca_b200.kmer_model import KmerModel
    from oracle import parity
    t0 = time.time()
    case = large_case()
    plan = full_plan(case)
    # an empty block cache: the workspace gets blocks of exactly its size, and the free memory is measured without them
    dtw.trim_memory()
    torch.cuda.synchronize()
    free_before = torch.cuda.mem_get_info()[0]
    if free_before < plan['peak'] + MEMORY_MARGIN:
        pytest.skip('%d bytes of device memory free, the case needs %d bytes of DP workspace + %d' % (
            free_before, plan['peak'], MEMORY_MARGIN))
    checked = plan['checked']
    km = KmerModel.load_from_hdf5(MODEL_PATH)
    spec = (km.get_k(), km.get_central_position(), km.mean, km.sigma, 'port')
    oracle = {(j, label): pool.apply_async(parity.job, ((kind, spec, case.reads[j] + (BW, MEL, flag)),))
              for j in checked for label, kind, flag, _ in OPS}
    straddler = plan['plans']['refine-plain']['crossings'][0]['straddle'][0]
    other = next(j for j in checked if case.meta[j][3] != case.meta[straddler][3])
    extended = {(j, wob): pool.apply_async(_truth_job, (('default', case.reads[j], BW, MEL, wob, False),))
                for j in (straddler, other) for wob in (False, True)}
    runs = {}
    try:
        for sched in SCHEDULES:
            dtw.set_sweep_schedule(sched)
            one = _run(km, case, list(range(N_READS)), plan['limit'], checked)
            small = _run(km, case, list(range(N_READS)), plan['small'], [])
            alone = _run(km, case, checked, 0, list(range(len(checked))))
            runs[sched] = dict(launches=one['launches'], kept=one['kept'], small_launches=small['launches'],
                               small_diff=_diff_all(one, small), alone=alone['kept'])
            del one, small, alone
        workspace = int(_cabi.load().nvb_model_workspace_bytes(km.handle))
    finally:
        dtw.set_sweep_schedule(None)
        km.__del__()  # destroys the device model and its workspace now, whatever still refers to the object
        dtw.trim_memory()
        torch.cuda.empty_cache()
        torch.cuda.synchronize()
    free_after = torch.cuda.mem_get_info()[0]
    print('GPU runs and release: %.0f s' % (time.time() - t0))
    return dict(case=case, plan=plan, runs=runs, oracle=oracle, extended=extended, extended_reads=(straddler, other),
                workspace=workspace, free=(free_before, free_after), t0=t0)


@pytest.mark.gpu
def test_tail_reads_equal_reads_alone(large_runs):
    """The straddling and tail reads, at their offsets past 2^31 in the large batch and near 0 in a batch of only
    them: bands, events, event means and alignment tables of both refine modes, log-likelihoods, chunk values and both
    stored planes of both estimate modes bit-identical, under both schedules; each op ran the planned waves."""
    s = large_runs
    plan, case, checked = s['plan'], s['case'], s['plan']['checked']
    print(describe_plan(case, plan))
    failures = []
    for sched, run in s['runs'].items():
        name = sched or 'auto'
        for label, kind, _, _ in OPS:
            want = launches(kind, len(plan['plans'][label]['waves']))
            if run['launches'][label] != want:
                failures.append('[%s] %s: %d launches, the plan gives %d' % (name, label, run['launches'][label], want))
            want = launches(kind, len(plan['small_plans'][label]))
            if run['small_launches'][label] != want:
                failures.append('[%s] %s, second run: %d launches, the plan gives %d' % (
                    name, label, run['small_launches'][label], want))
        big, alone = run['kept'], run['alone']
        for p, j in enumerate(checked):
            if not all(_same(a, b) for a, b in zip(big['bands'][p], alone['bands'][p])):
                failures.append('[%s] read %d: bands differ' % (name, j))
            for label, kind, _, _ in OPS:
                parts = ('events', 'event means', 'alignment table') if kind == 'refine' else \
                    ('log-likelihoods', 'chunk values', 'stored rows')
                for part, a, b in zip(parts, big[label][p], alone[label][p]):
                    if not _same(a, b):
                        failures.append('[%s] %s read %d: %s differ from the read alone' % (name, label, j, part))
    print('%d straddling and tail reads bit-identical to the reads alone under schedules %s: %s' % (
        len(checked), '/'.join(x or 'auto' for x in s['runs']), 'yes' if not failures else 'NO'))
    assert not failures, '\n'.join(failures[:40])


@pytest.mark.gpu
def test_waves_match_one_wave(large_runs):
    """The same batch as about SMALL_WAVES waves (every wave re-plans mat_base from 0): events of both refine modes and
    log-likelihoods of both estimate modes of every read bit-identical to the run in one wave (two for transitions)."""
    s = large_runs
    failures = []
    for sched, run in s['runs'].items():
        for label, _, _, _ in OPS:
            bad = run['small_diff'][label]
            if bad:
                failures.append('[%s] %s: %d reads differ between %d waves and %d, first %s' % (
                    sched or 'auto', label, len(bad), len(s['plan']['small_plans'][label]),
                    len(s['plan']['plans'][label]['waves']), bad[:8]))
    print('%d reads, %s: bit-identical in %s waves and in %s: %s' % (
        N_READS, ', '.join(label for label, _, _, _ in OPS),
        '/'.join(str(len(s['plan']['small_plans'][label])) for label, _, _, _ in OPS),
        '/'.join(str(len(s['plan']['plans'][label]['waves'])) for label, _, _, _ in OPS), 'yes' if not failures else 'NO'))
    assert not failures, '\n'.join(failures)


@pytest.mark.gpu
def test_tail_reads_match_references(large_runs):
    """The straddling and tail reads of the large batch under both schedules against the oracle port: events
    bit-exact, structural ties counted (none on this 6-mer workload); raw log-likelihoods within rtol 1e-9, finite
    exactly where the oracle's are.  Two of them, one per strand, against the extended-precision reference in both
    estimate modes: every ratio LL[i][b] - LL[i][ref_i] and the no-SNP total within ll_bar (64 eps (N + n) + 2 E)."""
    from nadavca_b200.kmer_model import KmerModel
    from oracle import oracle as orc
    from oracle import parity
    s = large_runs
    case, checked = s['case'], s['plan']['checked']
    km = KmerModel.load_from_hdf5(MODEL_PATH)  # host tables only
    om = orc.OracleModel(km.get_k(), km.get_central_position(), 4, km.mean, km.sigma, 'port')
    tally = {'exact': 0, 'tie': 0}
    worst_ll, failures = 0.0, []
    for p, j in enumerate(checked):
        r = case.reads[j]
        for label, kind, flag, _ in OPS:
            want = s['oracle'][(j, label)].get(timeout=3000)
            for sched, run in s['runs'].items():
                got = run['kept'][label][p][0]
                where = '[%s] %s read %d' % (sched or 'auto', label, j)
                try:
                    if kind == 'refine':
                        tally[parity.compare_events(got, *r, BW, MEL, om, flag, want=want)] += 1
                    else:
                        worst_ll = max(worst_ll, parity.ll_max_rel(got, want))
                        np.testing.assert_allclose(got, want, rtol=LL_RTOL)
                except AssertionError as e:
                    failures.append('%s: %s' % (where, str(e).strip().splitlines()[-1]))
    k, cp = km.get_k(), km.get_central_position()
    worst = {'ratio': 0.0, 'total': 0.0, 'base': 0.0}
    for j in s['extended_reads']:
        p = checked.index(j)
        r = case.reads[j]
        N, n = len(r[0]), len(r[1])
        term = exponent_term(k, cp, km.mean, km.sigma, r, BW)
        for label, wob in (('estimate-plain', False), ('estimate-wobble', True)):
            truth = s['extended'][(j, wob)].get(timeout=3000)
            for sched, run in s['runs'].items():
                wr, wt, wb, msg = _check_read(run['kept'][label][p][0], truth, N, n, r[1], term)
                worst = {'ratio': max(worst['ratio'], wr), 'total': max(worst['total'], wt),
                         'base': max(worst['base'], wb)}
                if msg:
                    failures.append('[%s] %s read %d: extended: %s' % (sched or 'auto', label, j, msg))
    print('%d straddling and tail reads vs the oracle port: %d alignments exact, %d structural ties, max rel LL error '
          '%.2e; reads %s vs the extended reference: worst err/bar ratio %.2e, no-SNP total %.2e (err / 64 eps (N + n) '
          '%.2e)' % (len(checked), tally['exact'], tally['tie'], worst_ll, list(s['extended_reads']), worst['ratio'],
                     worst['total'], worst['base']))
    assert not failures, '\n'.join(failures[:40])
    assert tally['tie'] == 0, 'structural ties on the 6-mer workload'


@pytest.mark.gpu
def test_workspace_released(large_runs):
    """The private model's DP workspace was exactly the planned peak (each of its six buffers rounded up to the block
    cache's 512 bytes), and with the batches closed, the model destroyed and the library's block cache trimmed the
    device's free memory is back within RELEASE_SLACK of its value before the runs."""
    s = large_runs
    before, after = s['free']
    print('workspace %d bytes, planned %d; free device memory %d bytes before, %d after (%+.3f GB); file %.0f s so far'
          % (s['workspace'], s['plan']['peak'], before, after, (after - before) / 1e9, time.time() - s['t0']))
    assert 0 <= s['workspace'] - s['plan']['peak'] < 6 * 512
    assert after >= before - RELEASE_SLACK, 'free memory %d bytes after, %d before' % (after, before)
