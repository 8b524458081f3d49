"""Kernel dispatch thresholds against the oracle.

The CUDA kernels change schedule, slot use, shared-memory layout or lane layout at hard thresholds of a band width or a
count.  This file builds ragged batches that sit exactly on both sides of each of them and holds every case to the
bars of test_gpu_parity.py: bands equal to the oracle's, events bit-exact (structural ties counted, expected 0 because
no reference here has two neighbouring positions with identical emissions), log-likelihoods within rtol = atol = 1e-9 and finite exactly where the
oracle's are.

Cases are built on the host by searching with orc.band_bounds until the geometry is exact, and every case states
which side of which threshold it is on.  `plan` below restates the dispatch decisions of the library with a citation
for each; test_thresholds_pinned_to_sources reads the constants back out of the .cu files, and
test_case_geometry_is_exact checks every case against `plan` without a GPU, so a retuned threshold or a bad case fails
before any GPU time is spent.
"""
import os
import re

import numpy as np
import pytest

from conftest import ROOT
from test_gpu_parity import LL_ATOL, LL_RTOL

CSRC = os.path.join(ROOT, 'nadavca_b200', 'csrc')
B200_SMS = 148

# ---- the dispatch decisions, restated ------------------------------------------------------------------------------
ROT_MAX = 640          # api.cu run_sweep: band rows wider than the rotating sweep's signal window go to the stripes
ROT_ONE_SLOT = 352     # api.cu run_sweep: steps a lane has per row pair; wider rows keep every second slot busy
ROT_WARPS_PER_SM = 16  # api.cu run_sweep: resident sweep warps per SM (auto rule 4 * items >= sm_count * 16)
ROT_SPAN = 63          # band.cu band_kernel: row j is checked against row j + 63 ...
ROT_OVERLAP = 48       # ... and must end at most 48 columns beyond its start (else NVB_READ_NO_ROTATION)
PATH_PK3_MAX = 384     # path2.cu nvbk_path2_columns_per_lane: 3 columns per lane up to 384 columns,
PATH_PK6_MAX = 1536    # 6 up to 1536, 11 beyond
PATH_MAX_WARPS = 8     # path2.cu launch_path: warps per read
PATH_GB = 64           # path2.cu: rows per geometry block
PATH_D = {3: 4, 6: 3, 11: 2}  # path2.cu nvbk_path2: score-ring depth of each layout
SMEM_BUDGET = 200 * 1024      # path2.cu launch_path and rows4.cu plan_sweep
PAIRS = 31             # rows4.cu: pair lanes per stripe
STRIPE_MAX_WARPS = 7   # rows4.cu plan_sweep
STRIPE_TS = 8          # rows4.cu NVB_STRIPE_TS
STRIPE_ROWMETA = 16    # rows4.cu RowMeta: long long + 2 int
RING_STATE = 40        # dp3.cuh RingState: one pointer + 7 ints, 8-byte aligned
STRIPE_TILE = 32 * (STRIPE_TS + 1) * (8 + 4) + 32 * STRIPE_ROWMETA  # rows4.cu kTileBytes
STRIPE_RING = (4 * 256 + 4 * 8 + RING_STATE + 15) // 16 * 16      # rows4.cu kRingStride (ring_bytes(4))
SNP_WARPS_PER_CTA = 4  # snp3.cu launch_snp3

MODES = ('plain', 'trans', 'wobble')
# (label, kind, flag, mode): refine(False) / refine(True) / estimate(True) / estimate(False)
OPS = (('refine-plain', 'refine', False, 'plain'), ('refine-trans', 'refine', True, 'trans'),
       ('estimate-wobble', 'estimate', True, 'wobble'), ('estimate-plain', 'estimate', False, 'plain'))


def path_columns_per_lane(maxw):
    """path2.cu nvbk_path2_columns_per_lane (from the batch's widest row, api.cu batch_init)."""
    return 3 if maxw <= PATH_PK3_MAX else (6 if maxw <= PATH_PK6_MAX else 11)


def path_plan(pk, wave_maxw):
    """path2.cu launch_path: warps per read, rounds of chunks, prefix-max rows in global memory, full staging area."""
    chunk = pk * 32
    nch = -(-wave_maxw // chunk)
    warps = max(1, min(PATH_MAX_WARPS, nch))
    head = (16 + 2 * (PATH_GB + PATH_D[pk] + 1) + PATH_D[pk] * warps * 32 * pk) * 8
    want_stage = 32 * nch * 32 * 4
    rows_bytes = 2 * wave_maxw * 8
    global_rows = head + rows_bytes > SMEM_BUDGET
    if global_rows:
        rows_bytes = 0
    body = max(rows_bytes, want_stage)
    if head + body > SMEM_BUDGET:
        body = rows_bytes
    return dict(pk=pk, path_warps=warps, path_rounds=-(-nch // warps), global_rows=global_rows,
                stage_full=body >= want_stage)


def stripe_plan(mode, wave_maxw):
    """rows4.cu plan_sweep: warps per (read, direction) and global hand-off rows."""
    width = (wave_maxw + 1) & ~1
    nw = max(1, min(STRIPE_MAX_WARPS, (wave_maxw + 12 * PAIRS + 11 * PAIRS - 1) // (11 * PAIRS)))
    tpw = 2 if mode == 'trans' else 1

    def tiles(w):
        return 64 + 16 + w * (tpw * STRIPE_TILE + STRIPE_RING)

    def total(w):
        return tiles(w) + (w + 1) * width * 12
    handoff = total(1) > SMEM_BUDGET
    if not handoff:
        while nw > 1 and total(nw) > SMEM_BUDGET:
            nw -= 1
    return dict(stripe_warps=nw, global_handoff=handoff)


def rotates(mode, wave_maxw, n_wave, no_rotation, schedule, sm_count):
    """api.cu run_sweep: rotating wavefront (rows5.cu) or stripes (rows4.cu) for one wave."""
    items = 2 * n_wave
    if schedule is None:
        rot = wave_maxw <= ROT_MAX and (wave_maxw <= ROT_ONE_SLOT or mode == 'plain' or
                                       4 * items >= sm_count * ROT_WARPS_PER_SM)
    else:
        rot = wave_maxw <= ROT_MAX and schedule == 'r'
    return rot and not no_rotation


class Geom:
    """Band geometry of one read from orc.band_bounds, plus the band kernel's summary (band.cu)."""

    def __init__(self, read, bw):
        from oracle import oracle as orc
        sig, ref, _, _, anc = read
        self.n, self.N = len(ref), len(sig)
        self.bs, self.be = orc.band_bounds(anc, self.N, self.n, bw)
        w = self.be.astype(np.int64) - self.bs + 1
        self.bad = bool((w <= 0).any()) or self.n <= 0 or self.N <= 0
        w = np.maximum(w, 0)
        self.rows = self.n + 1
        self.cells = int(w.sum())
        self.w0, self.wn = int(w[0]), int(w[-1])
        self.maxw = int(w.max())
        r = self.rows - ROT_SPAN
        self.overlap = int((self.be[:r].astype(np.int64) - self.bs[ROT_SPAN:]).max()) if r > 0 else None
        self.no_rotation = self.overlap is not None and self.overlap > ROT_OVERLAP

    def matrix_cells(self, mode):  # api.cu matrix_cells
        if self.bad:
            return 0
        return 2 * self.cells - self.w0 - self.wn if mode == 'trans' else self.cells

    def record_words(self, mode, pk):  # api.cu record_words
        if self.bad:
            return 0
        rows = 2 * self.n if mode == 'trans' else self.n + 1
        return rows * -(-self.maxw // (32 * pk)) * 32

    def wave_bytes(self, mode, need_dp, pk):  # api.cu plan_waves
        dp = 2 * self.maxw if need_dp and not self.bad else 0
        rec = self.record_words(mode, pk) if need_dp else 0
        return self.matrix_cells(mode) * 2 * 12 + dp * 8 + rec * 4


def plan_waves(geoms, mode, need_dp, limit, pk):
    """api.cu plan_waves with an explicit workspace limit (0: the whole batch in one wave)."""
    if limit <= 0:
        return [(0, len(geoms))]
    waves, i = [], 0
    while i < len(geoms):
        total, j = 0, i
        while j < len(geoms):
            b = geoms[j].wave_bytes(mode, need_dp, pk)
            if total + b > limit and j > i:
                break
            assert total + b <= limit, 'read %d alone exceeds the workspace limit' % j
            total += b
            j += 1
        waves.append((i, j))
        i = j
    return waves


def plan(geoms, mode, need_dp, schedule, limit, sm_count):
    """Per wave: what the library launches for `mode` (refine: need_dp) under `schedule` (None, 'r', 's')."""
    good = [g.maxw for g in geoms if not g.bad]
    pk = path_columns_per_lane(max(good) if good else 0)
    out = []
    for b0, b1 in plan_waves(geoms, mode, need_dp, limit, pk):
        ws = [g for g in geoms[b0:b1] if not g.bad]
        maxw = max([g.maxw for g in ws] or [0])
        d = dict(reads=(b0, b1), maxw=maxw,
                 rotate=rotates(mode, maxw, b1 - b0, any(g.no_rotation for g in geoms[b0:b1]), schedule, sm_count))
        d.update(stripe_plan(mode, maxw))
        if need_dp:
            d.update(path_plan(pk, maxw))
        out.append(d)
    return out


def describe(waves, need_dp):
    parts = []
    for w in waves:
        s = 'rot' if w['rotate'] else 'str%d%s' % (w['stripe_warps'], '+gh' if w['global_handoff'] else '')
        if need_dp:
            s += '/pk%d.w%d.r%d%s%s' % (w['pk'], w['path_warps'], w['path_rounds'], '+gm' if w['global_rows'] else '',
                                         '' if w['stage_full'] else '+part')
        parts.append(s)
    return ','.join(parts)


# ---- case construction ---------------------------------------------------------------------------------------------

def model_arrays(k, seed, sigma_lo=0.2, sigma_hi=0.6):
    """A random k-mer model; all 4^k means are distinct, so no two positions tie structurally."""
    rng = np.random.default_rng(seed)
    return rng.normal(0, 1.2, size=4 ** k), rng.uniform(sigma_lo, sigma_hi, size=4 ** k)


class Model:
    def __init__(self, k, cp, seed, sigma_lo=0.2, sigma_hi=0.6):
        self.k, self.cp, self.seed = k, cp, seed
        self.key = (k, cp, seed, sigma_lo, sigma_hi)
        self.mean, self.sigma = model_arrays(k, seed, sigma_lo, sigma_hi)


def kmer_levels(model, ref):
    n, k = len(ref), model.k
    padded = np.zeros(n + k, dtype=int)
    padded[model.cp:model.cp + n] = ref
    ids = np.zeros(n, dtype=int)
    for j in range(k):
        ids = ids * 4 + padded[j:j + n]
    return model.mean[ids], model.sigma[ids]


def tie_free_reference(rng, model, n, cb, ca):
    """A random reference in which no position has a neighbour with an identical emission (oracle/parity.py
    tie_rows: a run of k+1 equal bases, or any repeated base under a 1-mer model).  There the posterior cells of the
    boundary tie mathematically and the oracle's own argmax is rounding noise, so a path may differ from the oracle's
    as a counted structural tie; without such positions every path must be bit-exact."""
    from oracle import parity
    ref = rng.integers(0, 4, size=n)
    for _ in range(100):
        mask = parity.tie_rows(ref, cb, ca, model.k, model.cp, model.mean, model.sigma)
        if not mask.any():
            return ref
        ref[mask] = rng.integers(0, 4, size=int(mask.sum()))
    raise AssertionError('no tie-free reference found')


def make_read(rng, model, n, bw, mel, spacing=6, lengths=None, width=None, drop=(), bursts=()):
    """One read slice under `model`: bw samples of noise, the events (levels and noise of the model), a tail of noise;
    one anchor per base at its event start except the bases in `drop`.  With `width`, the tail is searched (through
    orc.band_bounds) until the widest band row has exactly `width` columns.  `bursts`: (position, length) pairs of
    the signal overwritten with outliers clipped at +-5."""
    cb = rng.integers(0, 4, size=rng.integers(0, model.cp + 1))
    ca = rng.integers(0, 4, size=rng.integers(0, model.k - model.cp))
    ref = tie_free_reference(rng, model, n, cb, ca)
    if lengths is None:
        lengths = np.maximum(max(mel, 1), rng.poisson(spacing, size=n))
    lengths = np.asarray(lengths)
    mu, sd = kmer_levels(model, ref)
    starts = np.concatenate([[0], np.cumsum(lengths)[:-1]]) + bw
    body = np.repeat(mu, lengths) + rng.normal(0, 1, lengths.sum()) * np.repeat(sd, lengths)
    keep = np.array([j for j in range(n) if j not in drop], dtype=int)
    anchors = np.stack([starts[keep], keep], axis=1)
    tail = bw
    if width is not None:
        for _ in range(30):
            g = Geom((np.zeros(bw + lengths.sum() + tail), ref, [], [], anchors), bw)
            if g.maxw == width:
                break
            tail += width - g.maxw
            assert tail >= 0, 'no tail gives %d columns (bw %d)' % (width, bw)
        else:
            raise AssertionError('tail search for width %d did not converge' % width)
    sig = np.concatenate([rng.normal(0, 1, bw), body, rng.normal(0, 1, tail)])
    for pos, ln in bursts:
        sig[pos:pos + ln] = rng.normal(0, 8, ln)
    sig = np.clip(sig, -5, 5)
    return sig, ref, cb, ca, anchors


def read_with_overlap(rng, model, n, bw, mel, target, p_long):
    """A read whose band overlap (band.cu: max be[j] - bs[j+63]) is exactly `target`: events of `mel` samples, one
    sample longer with probability `p_long`, redrawn until orc.band_bounds gives it."""
    for _ in range(2000):
        lengths = mel + (rng.random(n) < p_long)
        anchors = np.stack([np.concatenate([[0], np.cumsum(lengths)[:-1]]) + bw, np.arange(n)], axis=1)
        g = Geom((np.zeros(2 * bw + lengths.sum()), np.zeros(n, dtype=int), [], [], anchors), bw)
        if g.overlap == target:
            return make_read(rng, model, n, bw, mel, lengths=lengths)
    raise AssertionError('no read with overlap %d found' % target)


class Case:
    """A ragged batch plus its model.  `claims`: (mode, schedule, wave, key, value) that `plan` must give."""

    def __init__(self, name, model, bw, mel, reads, schedules=(None,), claims=(), limit=0):
        self.name, self.model, self.bw, self.mel, self.reads = name, model, bw, mel, reads
        self.schedules, self.claims, self.limit = tuple(schedules), list(claims), limit
        self.geoms = [Geom(r, bw) for r in reads]

    def plan(self, mode, need_dp, schedule, sm_count):
        return plan(self.geoms, mode, need_dp, schedule, self.limit, sm_count)

    def check_claims(self, sm_count):
        for mode, sched, wave, key, value in self.claims:
            for need_dp in ((True, False) if mode == 'plain' else ((True,) if mode == 'trans' else (False,))):
                if key.startswith('path') or key in ('pk', 'global_rows', 'stage_full'):
                    if not need_dp:
                        continue
                waves = self.plan(mode, need_dp, sched, sm_count)
                got = waves[wave][key] if wave is not None else [w[key] for w in waves]
                assert got == value, '%s: %s/%s wave %s: %s is %r, the case claims %r' % (
                    self.name, mode, sched, wave, key, got, value)

    def summary(self, sm_count):
        g = self.geoms
        ov = [x.overlap for x in g if x.overlap is not None]
        head = '%s: %d reads, n %d..%d, maxw %d, overlap %s' % (
            self.name, len(g), min(x.n for x in g), max(x.n for x in g), max(x.maxw for x in g),
            max(ov) if ov else '-')
        paths = []
        for sched in self.schedules:
            d = ' '.join('%s=%s' % (lab[:3] + lab[lab.index('-') + 1:][:1], describe(self.plan(mode, kind == 'refine', sched, sm_count),
                                                                                   kind == 'refine'))
                         for lab, kind, flag, mode in OPS)
            paths.append('[%s] %s' % (sched or 'auto', d))
        return head + ' | ' + ' | '.join(paths)


def _width_cases(rng):
    """Group A: rotate against stripes at 352/353 and 640/641 columns (api.cu run_sweep)."""
    m = Model(4, 2, 101)
    cases = []
    for width in (352, 353, 640, 641):
        bw = (width - 1) // 2
        spacing = 13 if width > 600 else 9
        reads = [make_read(rng, m, n, bw, 2, spacing=spacing, width=w)
                 for n, w in ((70, width), (45, 2 * bw + 1), (90, width))]
        over = width > ROT_ONE_SLOT
        claims = [('plain', None, 0, 'rotate', width <= ROT_MAX), ('plain', 's', 0, 'rotate', False)]
        for mode in ('trans', 'wobble'):
            claims += [(mode, None, 0, 'rotate', not over), (mode, 'r', 0, 'rotate', width <= ROT_MAX),
                       (mode, 's', 0, 'rotate', False)]
        cases.append(Case('A width %d' % width, m, bw, 2, reads, (None, 'r', 's'), claims))
    return cases


def _legality_cases(rng):
    """Group A: the rotation legality limit of band.cu (be[j] - bs[j+63] <= 48)."""
    m = Model(3, 1, 102)
    bw, mel = 87, 2
    cases = []
    for target in (ROT_OVERLAP, ROT_OVERLAP + 1):
        reads = [read_with_overlap(rng, m, 90, bw, mel, target, 0.03)]
        legal = target <= ROT_OVERLAP
        cases.append(Case('A overlap %d' % target, m, bw, mel, reads, (None, 'r'),
                          [(md, s, 0, 'rotate', legal) for md in MODES for s in (None, 'r')]))
    # 63, 64 and 65 band rows at an overlap far beyond the limit: only the reads of 64 and more rows are checked
    for rows in (63, 64, 65):
        read = make_read(rng, m, rows - 1, 120, mel, lengths=np.full(rows - 1, 2))
        c = Case('A %d rows dense' % rows, m, 120, mel, [read], (None, 'r'),
                 [(md, s, 0, 'rotate', rows <= ROT_SPAN) for md in MODES for s in (None, 'r')])
        assert rows <= ROT_SPAN or c.geoms[0].overlap > 2 * ROT_OVERLAP
        cases.append(c)
    # one wave: one non-rotatable read among rotatable ones
    good = [make_read(rng, m, n, bw, mel, spacing=7) for n in (80, 120, 66)]
    bad = read_with_overlap(rng, m, 100, bw, mel, ROT_OVERLAP + 1, 0.03)
    c = Case('A one bad read', m, bw, mel, good[:2] + [bad] + good[2:], (None, 'r'),
             [(md, s, 0, 'rotate', False) for md in MODES for s in (None, 'r')])
    assert [g.no_rotation for g in c.geoms] == [False, False, True, False]
    cases.append(c)
    # several waves (workspace limit): the first, holding the non-rotatable read, runs the stripes, the last rotates
    reads = [bad] + good + [make_read(rng, m, 70, bw, mel, spacing=7)]
    probe = Case('', m, bw, mel, reads)
    limit = find_limit(probe, lambda waves: not waves[0]['rotate'] and waves[-1]['rotate'])
    cases.append(Case('A two waves', m, bw, mel, reads, (None, 'r'),
                      [(md, s, w, 'rotate', w == -1) for md in MODES for s in (None, 'r') for w in (0, -1)],
                      limit=limit))
    return cases


def find_limit(case, want, sm_count=B200_SMS):
    """Smallest workspace limit for which every mode's wave plan satisfies `want` (searched over the byte sums the
    planner compares)."""
    pk = path_columns_per_lane(max(g.maxw for g in case.geoms if not g.bad))
    cands = set()
    for mode in MODES:
        for dp in (True, False):
            b = [g.wave_bytes(mode, dp, pk) for g in case.geoms]
            for i in range(len(b)):
                cands.update(np.cumsum(b[i:]).tolist())
    floor = max(g.wave_bytes(md, dp, pk) for g in case.geoms for md in MODES for dp in (True, False))
    for lim in sorted(c for c in cands if c >= floor):
        case.limit = lim
        if all(want(case.plan(mode, kind == 'refine', None, sm_count)) for _, kind, _, mode in OPS):
            return lim
    raise AssertionError('no workspace limit gives the wanted waves')


def _big_batch_cases(rng, sm_count):
    """Group A: the auto rule for big batches, 4 * items >= sm_count * 16 with items = 2 reads (api.cu run_sweep)."""
    m = Model(3, 1, 103)
    bw, mel = 200, 2
    need = -(-sm_count * ROT_WARPS_PER_SM // 8)
    reads = [make_read(rng, m, int(rng.integers(14, 22)), bw, mel, spacing=12, width=int(rng.integers(401, 641)))
             for _ in range(need)]
    cases = []
    for cnt in (need - 1, need):
        claims = [(md, None, 0, 'rotate', md == 'plain' or cnt >= need) for md in MODES]
        cases.append(Case('A %d reads auto' % cnt, m, bw, mel, reads[:cnt], (None,), claims))
    return cases


def _wavefront_cases(rng):
    """Group A: reads of 1, 2, 31..33, 64, 65 band rows-ish around a 31-pair stripe and a 32-lane generation."""
    m = Model(3, 1, 104)
    bw, mel = 12, 2
    reads = [make_read(rng, m, n, bw, mel, spacing=5) for n in (1, 2, 30, 31, 32, 33, 63, 64, 65)]
    return [Case('A wavefront edges', m, bw, mel, reads, ('r', 's'),
                 [('wobble', 'r', 0, 'rotate', True), ('wobble', 's', 0, 'rotate', False)])]


def path_thresholds():
    """Column counts at which the path search changes layout, computed from path_plan (path2.cu launch_path)."""
    out = {}
    prev = path_plan(11, PATH_PK6_MAX + 1)
    for w in range(PATH_PK6_MAX + 2, 40_000):
        p = path_plan(11, w)
        if p['global_rows'] and not prev['global_rows']:
            out['global_rows'] = w
        if not p['stage_full'] and prev['stage_full'] and p['global_rows']:
            out['stage_partial'] = w
            break
        prev = p
    return out


def _path_cases(rng):
    """Group B: the path search layouts of path2.cu (warps, columns per lane, rounds, global prefix rows, staging)."""
    m = Model(3, 1, 105)
    th = path_thresholds()
    widths = [96, 97, 192, 193, 288, 289, 384, 385, 1536, 1537, 2816, 2817, th['global_rows'] - 1, th['global_rows'],
              th['stage_partial'] - 1, th['stage_partial']]
    cases = []
    for w in widths:
        bw = 40 if w > 100 else 20
        reads = [make_read(rng, m, 25, bw, 2, spacing=6, width=w), make_read(rng, m, 40, bw, 2, spacing=6)]
        pk = path_columns_per_lane(w)
        p = path_plan(pk, w)
        claims = [('trans', None, 0, key, p[key]) for key in ('pk', 'path_warps', 'path_rounds', 'global_rows',
                                                                 'stage_full')]
        c = Case('B path %d' % w, m, bw, 2, reads, (None,), claims)
        cases.append(c)
    # the widest read (11 columns per lane) in a wave of its own, narrow reads in another
    wide = make_read(rng, m, 30, 40, 2, spacing=6, width=3000)
    narrow = [make_read(rng, m, int(rng.integers(40, 80)), 40, 2, spacing=6) for _ in range(8)]
    probe = Case('', m, 40, 2, [wide] + narrow)
    limit = find_limit(probe, lambda waves: len(waves) >= 2 and all(w['maxw'] < 200 for w in waves[1:]))
    cases.append(Case('B wide read own wave', m, 40, 2, [wide] + narrow, (None,),
                      [('trans', None, 0, 'pk', 11), ('trans', None, 1, 'path_warps', 1)], limit=limit))
    return cases


def stripe_thresholds(mode):
    """Widths at which plan_sweep (rows4.cu) cuts the warps per read or moves the hand-off rows to global memory."""
    out, prev = [], stripe_plan(mode, 1)
    for w in range(2, 12_000):
        p = stripe_plan(mode, w)
        if p['stripe_warps'] < prev['stripe_warps'] or p['global_handoff'] != prev['global_handoff']:
            out.append(w)
        prev = p
    return out


def _stripe_cases(rng):
    """Group C: both sides of every width at which shared memory cuts the striped sweep's warps, and of the global
    hand-off switch; every band row of the read that wide, enough pairs for every warp to take a stripe."""
    m = Model(3, 1, 106)
    cases = []
    for mode in ('plain', 'trans'):
        for edge in stripe_thresholds(mode):
            for w in (edge - 1, edge):
                bw = (w - 1) // 2
                nw = stripe_plan(mode, w)['stripe_warps']
                n = PAIRS * nw + 3
                read = make_read(rng, m, n, bw, 2, spacing=4, width=w)
                p = stripe_plan(mode, w)
                cases.append(Case('C %s %d' % (mode, w), m, bw, 2, [read], ('s',),
                                  [(mode, 's', 0, 'stripe_warps', p['stripe_warps']),
                                   (mode, 's', 0, 'global_handoff', p['global_handoff'])]))
    return cases


def snp_geometry(k, total_ref):
    """snp3.cu nvbk_snp2 / launch_snp3: tasks, lanes per task, tasks per warp, whether the last warp / CTA is
    partial."""
    lt = k + 2
    tpw = 32 // lt
    tasks = 3 * total_ref
    warps = -(-tasks // tpw)
    return dict(lt=lt, tpw=tpw, partial_warp=tasks % tpw != 0, partial_cta=warps % SNP_WARPS_PER_CTA != 0)


def _snp_cases(rng):
    """Group D: the SNP kernel at odd and extreme k and central positions, reads shorter than / as long as k, and a
    task count that leaves the last warp and CTA partial."""
    cases = []
    for k in (1, 2, 5, 7, 9, 11):
        for cp in sorted({0, k - 1, k // 2}):
            m = Model(k, cp, 200 + 10 * k + cp)
            bw, mel = 10, 2
            reads = [make_read(rng, m, n, bw, mel, spacing=5) for n in sorted({1, max(1, k - 1), k, k + 1, 30})]
            base = sum(len(r[1]) for r in reads)
            # a last read whose length leaves the last warp (when tasks per warp allow it) and CTA partial
            tpw = 32 // (k + 2)
            for extra in range(5, 200):
                g = snp_geometry(k, base + extra)
                if g['partial_cta'] and (g['partial_warp'] or 3 % tpw == 0):
                    break
            reads.append(make_read(rng, m, extra, bw, mel, spacing=5))
            g = snp_geometry(k, base + extra)
            assert g['partial_cta'] and (g['partial_warp'] or 3 % tpw == 0)
            cases.append(Case('D k%d cp%d' % (k, cp), m, bw, mel, reads, (None,)))
    m = Model(3, 1, 300)
    for mel in range(7):
        reads = [make_read(rng, m, n, 14, mel, spacing=mel + 4) for n in (1, 3, 40, 75)]
        cases.append(Case('D mel %d' % mel, m, 14, mel, reads, (None, 'r', 's'),
                          [('wobble', 'r', 0, 'rotate', True), ('trans', 's', 0, 'rotate', False)]))
    return cases


def _range_cases(rng):
    """Group E: dynamic range -- sigmas of 0.03..0.05, outlier bursts of 50..300 samples clipped at +-5, one event of
    over 500 samples -- for the renormalisation periods of the sweeps (dp3.cuh) and the SNP kernel (snp3.cu)."""
    cases = []
    for k, cp in ((6, 2), (11, 5)):
        m = Model(k, cp, 400 + k, 0.03, 0.05)
        bw, mel = 25, 2
        reads = []
        for i in range(3):
            n = 70
            lengths = np.maximum(mel, rng.poisson(8, size=n))
            lengths[30] = 520 + 20 * i
            starts = np.concatenate([[0], np.cumsum(lengths)[:-1]]) + bw
            # a short burst early in the read and a long one inside the long event
            bursts = [(int(starts[8]) + 2, int(rng.integers(50, 120))), (int(starts[30]) + 100, int(rng.integers(200, 301)))]
            reads.append(make_read(rng, m, n, bw, mel, lengths=lengths, drop=(31,), bursts=bursts))
        c = Case('E range k%d' % k, m, bw, mel, reads, (None, 'r', 's'),
                 [(md, 'r', 0, 'rotate', True) for md in MODES])
        assert ROT_ONE_SLOT < max(g.maxw for g in c.geoms) <= ROT_MAX
        cases.append(c)
    return cases


def all_cases(sm_count):
    rng = np.random.default_rng(2026)
    return (_width_cases(rng) + _legality_cases(rng) + _big_batch_cases(rng, sm_count) + _wavefront_cases(rng) +
            _path_cases(rng) + _stripe_cases(rng) + _snp_cases(rng) + _range_cases(rng))


# ---- CPU half ------------------------------------------------------------------------------------------------------

def _src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def test_thresholds_pinned_to_sources():
    """Every threshold `plan` restates, read back out of the kernels' sources: a retuned threshold fails here instead
    of leaving the boundary cases on one side of it."""
    api, band, path, rows4, rows5, dp3, snp = (_src(x) for x in ('api.cu', 'band.cu', 'path2.cu', 'rows4.cu',
                                                                  'rows5.cu', 'dp3.cuh', 'snp3.cu'))
    m = re.search(r'bool rotate = w\.maxw <= (\d+) && \(w\.maxw <= (\d+) \|\| mode == NVB_MODE_PLAIN \|\| '
                  r'4 \* items >= resident\);', api)
    assert m and (int(m.group(1)), int(m.group(2))) == (ROT_MAX, ROT_ONE_SLOT)
    assert re.search(r'rotate = w\.maxw <= %d && g_opt\.sweep == NVB_SWEEP_ROTATE;' % ROT_MAX, api)
    assert re.search(r'const int items = 2 \* \(w\.b1 - w\.b0\);', api)
    assert int(re.search(r'const int resident = b->model->sm_count \* (\d+);', api).group(1)) == ROT_WARPS_PER_SM
    assert re.search(r'rotate = !b->no_rotation\[i\];', api)
    m = re.search(r'if \(j \+ (\d+) < rows\) overlap = max\(overlap, be\[j\] - bs\[j \+ (\d+)\]\);', band)
    assert m and int(m.group(1)) == int(m.group(2)) == ROT_SPAN
    assert int(re.search(r'no_rotation = s_overlap > (\d+);', band).group(1)) == ROT_OVERLAP
    m = re.search(r'return maxw <= (\d+) \? 3 : \(maxw <= (\d+) \? 6 : 11\);', path)
    assert m and (int(m.group(1)), int(m.group(2))) == (PATH_PK3_MAX, PATH_PK6_MAX)
    assert re.search(r'warps = warps < 1 \? 1 : \(warps > %d \? %d : warps\);' % (PATH_MAX_WARPS, PATH_MAX_WARPS), path)
    assert int(re.search(r'constexpr int GB = (\d+);', path).group(1)) == PATH_GB
    for pk, d in PATH_D.items():
        assert re.search(r'launch_path<%d, %d>\(' % (pk, d), path)
    assert 'const size_t head = (16 + 2 * (GB + D + 1) + (size_t)D * warps * NVB_WARP * PK) * sizeof(double);' in path
    assert 'const size_t want_stage = (size_t)32 * nch * NVB_WARP * sizeof(uint32_t);' in path
    m = re.search(r'if \(head \+ rows_bytes > (\d+) \* 1024\) \{ smem_width = 0; rows_bytes = 0; \}\n.*\n'
                  r'\s+if \(head \+ body > (\d+) \* 1024\) body = rows_bytes;', path)
    assert m and int(m.group(1)) * 1024 == int(m.group(2)) * 1024 == SMEM_BUDGET
    assert re.search(r'constexpr int PAIRS = NVB_WARP - 1;', rows4) and PAIRS == 31
    assert int(re.search(r'#define NVB_STRIPE_TS (\d+)', rows4).group(1)) == STRIPE_TS
    assert 'int NW = (wave_maxw + 12 * PAIRS + 11 * PAIRS - 1) / (11 * PAIRS);' in rows4
    assert 'NW = NW < 1 ? 1 : (NW > %d ? %d : NW);' % (STRIPE_MAX_WARPS, STRIPE_MAX_WARPS) in rows4
    assert 'return (size_t)64 + 16 + (size_t)nw * (tiles_per_warp * kTileBytes + kRingStride);' in rows4
    assert 'return tile_bytes(nw) + (size_t)(nw + 1) * p.width * (sizeof(double) + sizeof(int32_t));' in rows4
    assert int(re.search(r'const size_t limit = (\d+) \* 1024;', rows4).group(1)) * 1024 == SMEM_BUDGET
    assert 'struct RowMeta {\n  long long off;  // offset of the row\'s first cell in the matrix planes\n  int s, e;' \
        in rows4
    body = dp3[dp3.index('struct RingState {'):]
    body = body[:body.index('};')]
    assert len(re.findall(r'^\s+const double \*\w+;', body, re.M)) == 1
    assert sum(len(re.findall(r'\w+', d)) for d in re.findall(r'^\s+(?:int|unsigned) ([^;]+);', body, re.M)) == 7
    assert 'constexpr int ring_bytes(int NS) { return NS * 256 + NS * 8 + (int)sizeof(RingState); }' in dp3
    assert 'const int LT = M.k + 2;' in snp and 'const int TPW = NVB_WARP / LT;' in snp
    assert int(re.search(r'const int warps = (\d+);', snp).group(1)) == SNP_WARPS_PER_CTA
    assert '8 is the largest value the slot-reuse guarantee of band.cu (be[j] - bs[j+63] <= 48) allows.' in rows5


def test_case_geometry_is_exact():
    """Every case of the GPU table, built on the host: geometry exact, each case on the side it claims."""
    cases = all_cases(B200_SMS)
    names = [c.name for c in cases]
    assert len(set(names)) == len(names)
    from oracle import parity
    for c in cases:
        c.check_claims(B200_SMS)
        for r in c.reads:  # no structural ties: every path must be bit-exact
            assert not parity.tie_rows(r[1], r[2], r[3], c.model.k, c.model.cp, c.model.mean, c.model.sigma).any()
    by = {c.name: c for c in cases}
    for w in (352, 353, 640, 641):
        assert max(g.maxw for g in by['A width %d' % w].geoms) == w
    assert [by['A overlap %d' % t].geoms[0].overlap for t in (48, 49)] == [48, 49]
    assert [by['A %d rows dense' % r].geoms[0].rows for r in (63, 64, 65)] == [63, 64, 65]
    assert [by['A %d rows dense' % r].geoms[0].no_rotation for r in (63, 64, 65)] == [False, True, True]
    assert sorted(g.rows for g in by['A wavefront edges'].geoms) == [2, 3, 31, 32, 33, 34, 64, 65, 66]
    th = path_thresholds()
    for w in (96, 97, 192, 193, 288, 289, 384, 385, 1536, 1537, 2816, 2817, th['global_rows'] - 1, th['global_rows'],
              th['stage_partial'] - 1, th['stage_partial']):
        assert max(g.maxw for g in by['B path %d' % w].geoms) == w
    assert [path_plan(3, w)['path_warps'] for w in (96, 97, 192, 193, 288, 289, 384)] == [1, 2, 2, 3, 3, 4, 4]
    assert path_plan(11, 2816)['path_rounds'] == 1 and path_plan(11, 2817)['path_rounds'] == 2
    for mode in ('plain', 'trans'):
        edges = stripe_thresholds(mode)
        for w in edges[:-1]:  # one warp fewer at each shared-memory cut, down to one warp
            assert stripe_plan(mode, w)['stripe_warps'] == stripe_plan(mode, w - 1)['stripe_warps'] - 1
        assert stripe_plan(mode, edges[-2])['stripe_warps'] == 1
        assert stripe_plan(mode, edges[-1])['global_handoff'] and not stripe_plan(mode, edges[-1] - 1)['global_handoff']
        for w in edges:
            for side in (w - 1, w):
                assert max(g.maxw for g in by['C %s %d' % (mode, side)].geoms) == side
    ks = {(c.model.k, c.model.cp) for c in cases if c.name.startswith('D k')}
    assert {k for k, _ in ks} == {1, 2, 5, 7, 9, 11} and all((k, k - 1) in ks and (k, 0) in ks for k, _ in ks)
    assert {c.mel for c in cases if c.name.startswith('D mel')} == set(range(7))
    for c in cases:
        if c.name.startswith('D k'):
            k = c.model.k
            ns = [g.n for g in c.geoms]
            assert 1 in ns and k in ns and any(n < k for n in ns) == (k > 1)
        if c.name.startswith('E'):
            assert c.model.sigma.min() >= 0.03 and c.model.sigma.max() <= 0.05
            assert all(np.abs(r[0]).max() <= 5 and (np.abs(r[0]) == 5).sum() >= 20 for r in c.reads)


# ---- GPU half ------------------------------------------------------------------------------------------------------

_WORKER_MODELS = {}


def _oracle_job(task):
    """One oracle call in a pool worker; the model is rebuilt from its seed (a 4^11-entry model is not shipped
    through a pipe for every read)."""
    from oracle import oracle as orc
    key, kind, args = task
    if key not in _WORKER_MODELS:
        k, cp, seed, lo, hi = key
        mean, sigma = model_arrays(k, seed, lo, hi)
        _WORKER_MODELS.clear()
        _WORKER_MODELS[key] = orc.OracleModel(k, cp, 4, mean, sigma, 'port')
    model = _WORKER_MODELS[key]
    sig, ref, cb, ca, anc, bw, mel, flag = args
    if kind == 'refine':
        return orc.refine_alignment(sig, ref, cb, ca, anc, bw, mel, model, flag)
    return np.array(orc.estimate_log_likelihoods(sig, ref, cb, ca, anc, bw, mel, model, flag))


@pytest.fixture(scope='module')
def pool():
    import multiprocessing as mp
    p = mp.get_context('spawn').Pool(min(os.cpu_count() or 1, 48))
    yield p
    p.terminate()


def _run_case(case, sm_count):
    """Every op under every schedule of the case -> {(schedule, label): per-read results}; bands checked."""
    from nadavca_b200 import dtw
    from oracle import oracle as orc
    m = case.model
    gm = dtw.KmerModel(m.k, m.cp, 4, m.mean, m.sigma)
    lists = [[r[i] for r in case.reads] for i in range(5)]
    out = {}
    try:
        for sched in case.schedules:
            dtw.set_sweep_schedule(sched)
            with dtw.Batch(gm, *lists, case.bw, case.mel, workspace_limit=case.limit) as batch:
                if sched == case.schedules[0]:
                    for (bs, be), r, g in zip(batch.bands(), case.reads, case.geoms):
                        obs, obe = orc.band_bounds(r[4], len(r[0]), len(r[1]), case.bw)
                        assert np.array_equal(bs, obs) and np.array_equal(be, obe), 'bands differ'
                for label, kind, flag, _ in OPS:
                    if kind == 'refine':
                        batch.refine(flag)
                        ev, st = batch.events()
                        out[(sched, label)] = ([None if e is None else e.copy() for e in ev], st.copy())
                    else:
                        batch.estimate(flag)
                        ll, st = batch.log_likelihoods()
                        out[(sched, label)] = ([x.copy() for x in ll], st.copy())
    finally:
        dtw.set_sweep_schedule(None)
    return out


@pytest.mark.gpu
def test_kernel_edges_match_oracle(lib_built, pool):
    """The whole case table on the GPU against the oracle; one line per case (geometry, predicted launch per op and
    schedule, exact / tie counts, largest relative log-likelihood error), every failure listed at the end."""
    import time
    import torch
    from oracle import oracle as orc
    from oracle import parity
    t_start = time.time()
    sm_count = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    cases = all_cases(sm_count)
    for c in cases:
        c.check_claims(sm_count)
    # the oracle first, fanned out over the pool, largest jobs first; the GPU runs meanwhile
    jobs = []
    for ci, c in enumerate(cases):
        for ri, (r, g) in enumerate(zip(c.reads, c.geoms)):
            for label, kind, flag, _ in OPS:
                cost = g.cells * (8 * c.model.k if kind == 'estimate' else 1)
                jobs.append((cost, (ci, ri, label), (c.model.key, kind, tuple(r) + (c.bw, c.mel, flag))))
    jobs.sort(key=lambda j: -j[0])
    pending = {key: pool.apply_async(_oracle_job, (task,)) for _, key, task in jobs}
    failures, lines = [], []
    tally = {'exact': 0, 'tie': 0}
    for ci, c in enumerate(cases):
        line = c.summary(sm_count)
        try:
            got = _run_case(c, sm_count)
            om = orc.OracleModel(c.model.k, c.model.cp, 4, c.model.mean, c.model.sigma, 'port')
            counts, worst = {'exact': 0, 'tie': 0}, 0.0
            for label, kind, flag, _ in OPS:
                wants = [pending[(ci, ri, label)].get(timeout=3000) for ri in range(len(c.reads))]
                for sched in c.schedules:
                    res, status = got[(sched, label)]
                    for ri, (r, want) in enumerate(zip(c.reads, wants)):
                        where = '%s [%s] read %d' % (label, sched or 'auto', ri)
                        if kind == 'refine':
                            assert (res[ri] is None) == (status[ri] == 1), where + ': status'
                            try:
                                counts[parity.compare_events(res[ri], *r, c.bw, c.mel, om, flag, want=want)] += 1
                            except AssertionError as e:
                                raise AssertionError('%s: %s' % (where, e))
                        else:
                            want = np.asarray(want)
                            finite = np.isfinite(want)
                            assert np.array_equal(np.isfinite(res[ri]), finite), where + ': finite pattern'
                            try:
                                np.testing.assert_allclose(res[ri][finite], want[finite], rtol=LL_RTOL, atol=LL_ATOL)
                            except AssertionError as e:
                                raise AssertionError('%s: %s' % (where, str(e).strip().splitlines()[-3:]))
                            worst = max(worst, parity.ll_max_rel(res[ri], want))
            for key in tally:
                tally[key] += counts[key]
            line += ' | exact %d tie %d max-rel-LL %.1e' % (counts['exact'], counts['tie'], worst)
            if counts['tie']:
                failures.append('%s: %d structural ties with a model without identical emissions' % (c.name,
                                                                                                    counts['tie']))
        except AssertionError as e:
            failures.append('%s: %s' % (c.name, e))
            line += ' | FAILED'
        print(line)
        lines.append(line)
    print('kernel edges: %d cases, %d alignments exact, %d ties, %.0f s' % (len(cases), tally['exact'], tally['tie'],
                                                                           time.time() - t_start))
    assert not failures, '\n'.join(failures)
