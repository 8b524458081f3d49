#!/usr/bin/env python
"""bench.py -- throughput of the nadavca hot path on B200 (DESIGN.md "Measurement").

Workload (BASELINE.json configs[1]): estimate_snps(independent=True) over synthetic reads (~2 kb bases, ~20 k
samples each, default config: bandwidth 150, min_event_length 2, wobbling, tweak) simulated from the shipped 6-mer
model.  One "step" = one pass of the device hot path over the whole batch of reads:

    refine_alignment(model_transitions=False) on the normalised signals       (estimator.py:77-87)
    estimate_log_likelihoods(model_wobbling=True) on the tweaked signals      (estimator.py:99-109)
    normalise / strand flip -> per-read posterior                               (estimator.py:111-156)

The host-side spline tweak between the two DP calls (scipy, estimator.py:89-97) is prepared once, untimed, for both
arms: it is the same scipy call in the reference and here and is not part of the path being accelerated.

  value  = signal samples aligned per second with every input already resident in HBM (CUDA events, max over ranks)
  e2e    = the same metric through the C-ABI calls with (pinned) HOST buffers: H2D of all inputs, kernels, D2H of
           events and probabilities inside the timed region
  --impl reference : the reference's own CPU implementation of the same two DP calls (oracle/_ref = the unmodified
           nadavca C++ compiled by oracle/Makefile; the C port when it is missing) on all host cores, one read per
           worker, on a bounded sample of the same workload.
  --dump-outputs DIR : after the timed steps, what the last step computed as DIR/<name>.npy (see `dump_outputs`),
           so that two builds can be compared output for output on identical seeded inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DEFAULT_CONFIG = dict(bandwidth=150, snp_prior_probability=0.001, min_event_length=2, model_wobbling=True,
                      model_transitions=True, tweak_signal_normalization=True, normalization_event_length=10)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', type=int, default=1, choices=[0, 1, 2, 3, 4],
                    help='BASELINE.json configs index: 1 = the headline workload (default; its line also carries the '
                         'consensus step of configs[2]), 2 = the same line, 0 / 3 / 4 = bench_configs.py')
    ap.add_argument('--reads', type=int, default=None, help='reads per GPU (weak scaling); default per config')
    ap.add_argument('--bases', type=int, default=None, help='bases per read; default per config')
    ap.add_argument('--sweep-bandwidths', default='50,100,150,250,400,650,1000', help='--config 4')
    ap.add_argument('--sweep-batches', default='1,8,64,512,4096', help='--config 4: reads per GPU')
    ap.add_argument('--genome', type=int, default=4_600_000, help='synthetic genome length (E. coli-sized: configs[2])')
    ap.add_argument('--no-api', action='store_true', help='skip the public-API timing block')
    ap.add_argument('--no-consensus', action='store_true', help='skip the consensus-mode (configs[2]) step')
    ap.add_argument('--bandwidth', type=int, default=None, help='default 150 (400 for --config 3)')
    ap.add_argument('--cpu-sample', type=int, default=0, help='reads in the CPU sample (0 = one per host core)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-overlap', action='store_true', help='accepted for older scripts; no effect')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step computed as DIR/<name>.npy (at most 64 MB: a fixed, seeded '
                         'sample of the reads when the batch is larger)')
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if a.dump_outputs and (a.impl != 'ours' or a.config not in (1, 2)):
        ap.error('--dump-outputs applies to the estimate_snps step of --config 1 / 2')
    per_config = {0: (100, 2000, 150), 1: (1000, 2000, 150), 2: (1000, 2000, 150), 3: (62, 100_000, 400),
                  4: (None, 2000, 150)}[a.config]
    a.reads = a.reads if a.reads is not None else per_config[0]
    a.bases = a.bases if a.bases is not None else per_config[1]
    a.bandwidth = a.bandwidth if a.bandwidth is not None else per_config[2]
    return a


# ---- workload ----------------------------------------------------------------------------------------------------

def load_model():
    from nadavca_b200.kmer_model import KmerModel
    return KmerModel.load_from_hdf5(os.path.join(ROOT, 'nadavca_b200', 'default', 'kmer_model.hdf5'))


def make_workload(km, n_reads, first_index, bases, genome_len, bandwidth):
    """Seeded synthetic reads + everything the estimator prepares on the host before the first DP call."""
    from nadavca_b200 import synthetic
    from nadavca_b200.genome import Genome
    from nadavca_b200.read import Read
    genome = synthetic.make_genome(genome_len, seed=0)
    reads = []
    for i in range(n_reads):
        rng = np.random.default_rng(500_000 + first_index + i)
        nb = int(round(rng.normal(bases, bases / 10.0)))
        reads.append(synthetic.make_read(genome, km, first_index + i, n_bases=nb, bandwidth=bandwidth))
    Read.normalize_reads(reads)
    aligner = synthetic.SyntheticAligner(genome)
    k, cp = km.get_k(), km.get_central_position()
    items = []
    for r in reads:
        apx = aligner.get_signal_alignment(r, bandwidth)
        s0, s1 = apx.signal_range
        a, b = apx.read_sequence_range
        ref_part = genome[apx.reference_range[0]:apx.reference_range[1]]
        if apx.reverse_complement:
            ref_part = Genome.reverse_complement(ref_part)
        items.append(dict(read=r, apx=apx, signal=r.normalized_signal[s0:s1], reference=Genome.to_numerical(ref_part),
                          cb=Genome.to_numerical(r.sequence[a - cp:a]),
                          ca=Genome.to_numerical(r.sequence[b:b + k - cp - 1])))
    return genome, items


def tweak_on_host(items, events_per_read, expected_per_read):
    """Read.tweak_signal_normalization per read (scipy spline) -> tweaked signal slices."""
    out = []
    for it, ev, exp_sig in zip(items, events_per_read, expected_per_read):
        s0, s1 = it['apx'].signal_range
        it['read'].tweak_signal_normalization(np.asarray(ev, dtype=int) + s0, exp_sig)
        out.append(np.ascontiguousarray(it['read'].tweaked_normalized_signal[s0:s1]))
    return out


def band_stats(bands, k, cp, wobbling=True):
    """DP cell counts (SURVEY.md 8d) and algorithmic HBM bytes per stage from the band widths (DESIGN.md)."""
    cells = dict(refine_plain=0, estimate_fb=0, estimate_snp=0)
    bytes_ = dict(rows_refine=0, path=0, rows_estimate=0, snp=0)
    back, fwd = k - cp - 1, cp
    for bs, be in bands:
        w = (be - bs + 1).astype(np.int64)
        n = len(w) - 1
        tot = int(w.sum())
        cells['refine_plain'] += int(w[1:].sum() + w[:-1].sum())
        cells['estimate_fb'] += int(w[1:].sum() + w[:-1].sum() + (2 * w[1:n].sum() if wobbling else 0))
        csum = np.concatenate([[0], np.cumsum(w)])
        i = np.arange(n)
        first = np.maximum(0, i - back)
        last = np.minimum(n - 1, i + fwd)
        model_rows = csum[last + 2] - csum[first + 1]                    # sum_{j=first..last} W[j+1]
        wob_rows = csum[last + 1] - csum[np.maximum(first, 1)] if wobbling else 0  # sum_{j=max(first,1)..last} W[j]
        trail = np.where(last + 1 < n, w[last], 0) if wobbling else 0
        cells['estimate_snp'] += int(3 * (model_rows + wob_rows + trail).sum())
        # algorithmic traffic (DESIGN.md section 6): a stored cell is 12 B (f64 mantissa + i32 exponent);
        # sweeps write prefix and suffix once ...
        bytes_['rows_refine'] += 2 * tot * 12
        bytes_['rows_estimate'] += 2 * tot * 12
        # ... the score kernel reads both (24 B) and writes the score (8 B), the path kernel reads the score (8 B) and
        # writes one record bit per cell
        bytes_['path'] += tot * (24 + 8 + 8) + tot // 8
        # ... every SNP task streams its start prefix row and its closing suffix row and writes one double
        bytes_['snp'] += int(3 * ((w[first] + w[last + 1]) * 12 + 8).sum())
    return cells, bytes_


def band_cells_transitions(band):
    """NextRow cells of refine_alignment(transitions) for one read's (starts, ends) band (SURVEY.md 8d)."""
    bs, be = band
    w = (be - bs + 1).astype(np.int64)
    return int(2 * (2 * w.sum() - w[0] - w[-1]) - w[0] - w[-1])


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    QUERY = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.proc = None
        self.first = 0

    def mark(self):
        """Start of the timed region: earlier samples are not summarised."""
        self.first = len(self.lines)

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.QUERY,
                                          '--format=csv,noheader,nounits', '-lms', '200'], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in self.lines[self.first:]:
            parts = [p.strip() for p in line.split(',')]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(max(mx)), 'reasons': sorted(reasons),
                'samples': len(sm)}


# ---- CPU reference arm ----------------------------------------------------------------------------------------

_WORKER = {}


def _cpu_worker_init(k, cp, mean, sigma, backend):
    from oracle import oracle as orc
    _WORKER['model'] = orc.OracleModel(k, cp, 4, mean, sigma, backend)
    _WORKER['orc'] = orc


def _cpu_worker(task):
    """The two DP calls of estimator.py:77-109 for one read on one core; the results go back to the parent, which
    checks the GPU's results for the same reads against them (the `parity` block of the bench line)."""
    orc, model = _WORKER['orc'], _WORKER['model']
    signal, tweaked, ref, cb, ca, anchors, bw, mel = task
    ev = orc.refine_alignment(signal, ref, cb, ca, anchors, bw, mel, model, False)
    ll = orc.estimate_log_likelihoods(tweaked, ref, cb, ca, anchors, bw, mel, model, True)
    return np.asarray(ev, dtype=np.int32).reshape(-1, 2), np.asarray(ll, dtype=np.float64)


class CpuArm:
    def __init__(self, km, cores, method='fork'):
        import multiprocessing as mp
        from oracle import oracle as orc
        self.kind = 'reference' if orc.ref_module() is not None else 'port'
        self.backend = 'ref' if self.kind == 'reference' else 'port'
        self.cores = cores
        self.pool = mp.get_context(method).Pool(cores, initializer=_cpu_worker_init,
                                                initargs=(km.get_k(), km.get_central_position(), km.mean, km.sigma,
                                                          self.backend))

    def run(self, tasks):
        t0 = time.perf_counter()
        self.results = self.pool.map(_cpu_worker, tasks, chunksize=1)
        return time.perf_counter() - t0

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_tasks(km, items, tweaked, bandwidth, mel):
    return [(it['signal'], tw, it['reference'], it['cb'], it['ca'], it['apx'].alignment, bandwidth, mel)
            for it, tw in zip(items, tweaked)]


def cpu_tweak(km, items, bandwidth, mel):
    """Tweaked signals computed with the oracle only (for the reference arm, which must not need a GPU)."""
    from oracle import oracle as orc
    backend = 'ref' if orc.ref_module() is not None else 'port'
    model = orc.OracleModel(km.get_k(), km.get_central_position(), 4, km.mean, km.sigma, backend)
    evs, exps = [], []
    for it in items:
        evs.append(orc.refine_alignment(it['signal'], it['reference'], it['cb'], it['ca'], it['apx'].alignment,
                                        bandwidth, mel, model, False))
        exps.append(model.get_expected_signal(it['reference'], it['cb'], it['ca']))
    return tweak_on_host(items, evs, exps)


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    km = load_model()
    cores = os.cpu_count() or 1
    n_sample = args.cpu_sample or cores
    cfg = DEFAULT_CONFIG
    _, items = make_workload(km, n_sample, 0, args.bases, args.genome, args.bandwidth)
    tweaked = cpu_tweak(km, items, args.bandwidth, cfg['min_event_length'])
    tasks = cpu_tasks(km, items, tweaked, args.bandwidth, cfg['min_event_length'])
    from oracle import oracle as orc
    counts = dict(refine_plain=0, estimate_fb=0, estimate_snp=0)
    for it in items:
        c = orc.count_cells(it['apx'].alignment, len(it['signal']), len(it['reference']), args.bandwidth,
                            km.get_k(), km.get_central_position())
        for key in counts:
            counts[key] += c[key]
    samples = sum(len(it['signal']) for it in items)
    cells = sum(counts.values())
    arm = CpuArm(km, min(cores, n_sample))
    for _ in range(args.warmup):
        arm.run(tasks)
    t = 0.0
    for _ in range(args.steps):
        t += arm.run(tasks)
    arm.close()
    value = samples * args.steps / t
    sample_desc = '%d reads of the workload (one per worker), refine_alignment(no transitions) + ' \
                  'estimate_log_likelihoods(wobbling) per read' % n_sample
    line = {
        'impl': 'reference', 'metric': 'signal_samples_aligned_per_sec', 'value': value, 'unit': 'samples/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * t / args.steps,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'dp_cells_per_sec': cells * args.steps / t,
        'config': workload_config(args, n_sample),
        'cpu_baseline': {'value': value, 'unit': 'samples/s', 'cores': arm.cores, 'kind': arm.kind,
                         'sample': sample_desc},
        'e2e': {'value': value, 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line))


def workload_config(args, reads_per_gpu):
    return {'workload': 'configs[1]: estimate_snps independent=True, synthetic reads (~%d bases, ~%dk samples), '
                        'default config (bandwidth %d, min_event_length 2, wobbling, tweak), kmer_model.hdf5 6-mer'
                        % (args.bases, args.bases // 100, args.bandwidth),
            'reads_per_gpu': reads_per_gpu, 'bandwidth': args.bandwidth, 'genome_bases': args.genome,
            'step': 'refine_alignment(plain) + estimate_log_likelihoods(wobbling) + chunk normalise + posterior',
            'l2': 'inputs larger than L2 (DP matrices of several GB per step)'}


# ---- --dump-outputs ------------------------------------------------------------------------------------------------

DUMP_BYTES = 60 << 20        # stays under the 64 MB --dump-outputs promises, .npy headers included
DUMP_BYTES_PER_ROW = 84      # probabilities 4 x f64 + coverage f32 + log-likelihoods 4 x f64 + events 2 x f64
DUMP_BYTES_PER_READ = 24     # chunks 3 x f64
DUMP_SEED = 20_261_020


def dump_selection(rows_per_read, budget=DUMP_BYTES):
    """Indices (ascending) of the reads --dump-outputs writes: all of them when they fit into `budget`, otherwise the
    longest prefix of one fixed seeded permutation that does, so that runs with the same arguments pick the same
    reads."""
    rows = np.asarray(rows_per_read, dtype=np.int64)
    cost = rows * DUMP_BYTES_PER_ROW + DUMP_BYTES_PER_READ
    if cost.sum() <= budget:
        return np.arange(len(rows))
    order = np.random.default_rng(DUMP_SEED).permutation(len(rows))
    n = int(np.searchsorted(np.cumsum(cost[order]), budget, side='right'))
    return np.sort(order[:n])


def dump_outputs(out_dir, result, events, log_likelihoods):
    """What one step of estimate_snps(independent=True) computed, for the reads of `dump_selection` in read order:

      probabilities.npy    float64 (rows, 4)  posterior of A, C, G, T per reference position: the `values` of the
                                              Chunk objects the call returns, the reads' chunks concatenated
      coverage.npy         float32 (rows,)    the chunks' `coverage`
      chunks.npy           float64 (n, 3)     read index, reference start, reference end of each chunk
      log_likelihoods.npy  float64 (rows, 4)  raw log-likelihoods of estimate_log_likelihoods(wobbling), read
                                              orientation
      events.npy           float64 (rows, 2)  event boundaries of refine_alignment(no transitions), relative to the
                                              start of the read's signal range

    `result` is what ``posterior_stage`` returned; `events` / `log_likelihoods` the per-read arrays of the batches.
    With several GPUs only rank 0 writes, its own reads."""
    groups, group_off, probs, cov = result
    probs, cov = probs.cpu().numpy(), cov.cpu().numpy()
    keep = dump_selection(np.diff(group_off))

    def rows_of(per_read, width):
        return np.concatenate([np.zeros((0, width))] + [per_read[i] for i in keep]).astype(np.float64)

    rows = np.concatenate([np.zeros(0, np.int64)] + [np.arange(group_off[i], group_off[i + 1]) for i in keep])
    out = {'probabilities': probs[rows].astype(np.float64),
           'coverage': cov[rows].astype(np.float32),
           'chunks': np.array([(i, groups[i][0], groups[i][1]) for i in keep], dtype=np.float64).reshape(-1, 3),
           'log_likelihoods': rows_of(log_likelihoods, 4),
           'events': rows_of(events, 2)}
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in out.items():
        np.save(os.path.join(out_dir, name + '.npy'), arr)


# ---- GPU arm ------------------------------------------------------------------------------------------------------

def first_read_index(rank, reads_per_gpu):
    """Weak scaling: rank r simulates (and owns) reads [r*R, (r+1)*R) of the seeded workload; no read is shared."""
    return rank * reads_per_gpu


def reduce_over_ranks(value, op, device):
    """max / sum of a host scalar over all ranks (identity for a single process)."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return value
    t = torch.tensor([value], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX if op == 'max' else dist.ReduceOp.SUM)
    return float(t.item())


def run_ours(args):
    import torch
    import torch.distributed as dist
    from nadavca_b200 import _cabi, dtw
    from nadavca_b200.estimator import ProbabilityEstimator

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device (the product path has no CPU fallback)')
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    dev = torch.device('cuda', local_rank)
    stream = torch.cuda.current_stream()
    cfg = dict(DEFAULT_CONFIG, bandwidth=args.bandwidth)
    mel = cfg['min_event_length']

    km = load_model()
    km._device = local_rank
    genome, items = make_workload(km, args.reads, first_read_index(rank, args.reads), args.bases, args.genome, args.bandwidth)
    est = ProbabilityEstimator(km, None, cfg)

    lists = ([it['signal'] for it in items], [it['reference'] for it in items], [it['cb'] for it in items],
             [it['ca'] for it in items], [it['apx'].alignment for it in items])
    reverse = [int(it['apx'].reverse_complement) for it in items]
    intervals = [tuple(it['apx'].reference_range) for it in items]

    # untimed preparation: first refine, host spline tweak, second resident batch with the tweaked signals
    batch_n = dtw.Batch(km, *lists, args.bandwidth, mel)
    batch_n.refine(False, stream)
    events, status = batch_n.events()
    assert all(ev is not None for ev in events), 'synthetic read without a path'
    expected = km.get_expected_signal_batch(lists[1], lists[2], lists[3])
    tweaked = tweak_on_host(items, events, expected)
    batch_t = dtw.Batch(km, tweaked, *lists[1:], args.bandwidth, mel)
    plan = est.plan_groups(intervals, genome, independent=True)
    cells, abytes = band_stats(batch_n.bands(), km.get_k(), km.get_central_position(), True)
    samples = int(batch_n.pack.total_signal)
    total_cells = sum(cells.values())

    def step():
        batch_n.refine(False, stream)
        batch_t.estimate(True, stream)
        return est.posterior_stage(batch_t, reverse, intervals, genome, independent=True, plan=plan)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # The sampler is started BEFORE the warm-up: the first nvidia-smi on a fresh box takes a second or two to attach
    # to the driver and slows kernel launches while it does (measured: +20 ms per step on the first run of a box);
    # only the samples taken during the timed region are summarised.
    with ClockSampler(local_rank) as clocks:
        for _ in range(args.warmup):
            step()
        barrier()
        l0 = batch_n.launch_count + batch_t.launch_count
        batch_n.enable_timing(True)
        batch_t.enable_timing(True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        clocks.mark()
        e0.record(stream)
        for _ in range(args.steps):
            out = step()
        e1.record(stream)
        barrier()
    ms = e0.elapsed_time(e1)
    launches = (batch_n.launch_count + batch_t.launch_count - l0) + args.steps  # + posterior kernel per step
    tn, tt = batch_n.timing(), batch_t.timing()
    batch_n.enable_timing(False)
    batch_t.enable_timing(False)
    if args.dump_outputs and rank == 0:
        # before the consensus step below, which runs the same batches again
        dump_outputs(args.dump_outputs, out, batch_n.events()[0], batch_t.log_likelihoods()[0])
    # what the timed steps left resident for the reads of the CPU sample (checked against the reference below)
    n_check = cpu_sample_size(args, len(items)) if (world == 1 and not args.no_cpu_baseline) else 0
    gpu_events = batch_n.events()[0][:n_check] if n_check else []
    gpu_ll = batch_t.log_likelihoods()[0][:n_check] if n_check else []

    # ---- consensus mode (configs[2]: estimate_snps independent=False, reads sharded over the ranks) ------------------
    # Same resident reads, same DP work per step, but the per-position sums go over the reads of ALL ranks
    # (estimator.py:226-231): timed region = refine -> estimate -> chunk normalise -> scatter-add into the consensus
    # rows -> the exchange (reduce-scatter by genome slice + halo + all-gather over NCCL) -> posterior on the owned
    # slice.  The overlap groups over all ranks' intervals are planned once (host, untimed), like `plan` above.
    consensus = None
    if not args.no_consensus:
        pg = dist.group.WORLD if world > 1 else None
        plan_c = est.plan_groups(intervals, genome, independent=False, process_group=pg)
        ev_log = []

        def consensus_step(collective='auto', log=None):
            batch_n.refine(False, stream)
            batch_t.estimate(True, stream)
            return est.posterior_stage(batch_t, reverse, intervals, genome, independent=False, process_group=pg,
                                       plan=plan_c, collective=collective, events=log)

        for _ in range(2):
            res_c = consensus_step()
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record(stream)
        for _ in range(args.steps):
            log = {}
            res_c = consensus_step(log=log)
            ev_log.append(log)
        c1.record(stream)
        barrier()
        c_ms = c0.elapsed_time(c1) / args.steps
        x_ms = [sum(a.elapsed_time(b) for a, b in log.get('exchange', [])) for log in ev_log]
        probs_c, cov_c = res_c[2], res_c[3]
        # every rank must hold the same consensus; the two exchange variants must agree
        check = torch.stack([probs_c.sum(), probs_c.square().sum(), cov_c.sum().double()])
        hi_, lo_ = check.clone(), check.clone()
        modes_diff = 0.0
        if world > 1:
            dist.all_reduce(hi_, op=dist.ReduceOp.MAX)
            dist.all_reduce(lo_, op=dist.ReduceOp.MIN)
            other = consensus_step(collective='allreduce')
            modes_diff = float((other[2] - probs_c).abs().max().item())
            barrier()
        consensus = {
            'ms_per_step': reduce_over_ranks(c_ms, 'max', dev),
            'exchange_ms_per_step': reduce_over_ranks(float(np.mean(x_ms)) if x_ms else 0.0, 'max', dev),
            'collective': ev_log[-1].get('mode', 'none (one rank)') if ev_log else None,
            'bus_bytes_per_step': ev_log[-1].get('bus_bytes', 0.0) if ev_log else 0.0,
            'positions': int(probs_c.shape[0]), 'groups': len(res_c[0]),
            'mean_coverage': float(cov_c.double().mean().item()),
            'ranks_identical': bool(torch.equal(hi_, lo_)),
            'reduce_scatter_vs_allreduce_max_abs_diff': modes_diff,
            'rows_sum_to_one_max_err': float((probs_c.sum(dim=1) - 1).abs().max().item()),
        }

    # ---- end to end through the C ABI with pinned host buffers -----------------------------------------------
    def pinned(arr):
        t = torch.from_numpy(np.ascontiguousarray(arr)).pin_memory()
        return t, t.numpy()

    pk = batch_n.pack
    keep = []
    host = {}
    for name in ('signal', 'signal_off', 'reference', 'reference_off', 'context_before', 'context_before_off',
                 'context_after', 'context_after_off', 'anchors', 'anchor_off'):
        t, a = pinned(getattr(pk, name))
        keep.append(t)
        host[name] = a
    # the tweak splines were fitted on the host during the (untimed) preparation; the product path evaluates them on
    # the device (estimator._run_estimate), so the end-to-end step uploads knots and coefficients, not signals
    splines = [it['read'].tweak_spline for it in items]
    spline_bytes = sum(2 * 8 * len(sp[0]) for sp in splines) + 8 * (len(splines) + 1)
    pack = _cabi.ReadsPack.from_packed(bandwidth=args.bandwidth, min_event_length=mel, **host)
    h2d = sum(a.nbytes for a in host.values()) + spline_bytes
    ev_host = torch.empty((pk.total_reference, 2), dtype=torch.int32).pin_memory()
    st_host = torch.empty(pk.n_reads, dtype=torch.int32).pin_memory()
    prob_host = torch.empty((pk.total_reference, 4), dtype=torch.float64).pin_memory()
    d2h = ev_host.numel() * 4 + st_host.numel() * 4 + prob_host.numel() * 8 + pk.total_reference * 8
    import ctypes
    lib = _cabi.load()

    def e2e_step():
        b = dtw.Batch.from_pack(km, pack)                       # H2D of every input + band kernel
        b.refine(False, stream)
        _cabi.check(lib.nvb_batch_get_events(b.handle, ctypes.cast(ev_host.data_ptr(), _cabi.c_i32p),
                                             ctypes.cast(st_host.data_ptr(), _cabi.c_i32p)), 'get_events')  # D2H
        b.event_means()                                          # D2H of the per-event means (input of the fit)
        b.apply_splines(splines, stream)                         # H2D of the splines, evaluation on the device
        b.estimate(True, stream)
        res = est.posterior_stage(b, reverse, intervals, genome, independent=True, plan=plan)
        prob_host.copy_(res[2], non_blocking=True)               # D2H of the step's result
        torch.cuda.synchronize()
        b.close()

    # free the resident batches first: the e2e batch allocates its own workspace
    batch_n.close()
    batch_t.close()
    e2e_steps = args.steps
    for _ in range(2):  # warm-up: the first pass also fills the library's device block cache
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0

    # ---- the public API (what a user of the reference calls), host glue included -------------------------------------
    # estimate_snps: pooled normalisation (device), aligner glue, packing, refine, spline fits (worker pool), SNP DP,
    # posterior, Chunk objects.  align_signal: per-read normalisation, two alignment rounds with transitions, linear
    # renormalisation.  Reported next to `e2e` (the C-ABI path both arms are compared on); raw samples per second.
    api = None
    if not args.no_api:
        import nadavca_b200
        from nadavca_b200 import synthetic
        reads_api = [it['read'] for it in items]
        aligner = synthetic.SyntheticAligner(genome)
        raw_samples = float(sum(len(r.raw_signal) for r in reads_api))

        def timed_call(fn):
            fn()  # warm-up: worker pool, workspaces
            best, out = None, None
            for _ in range(2):  # best of two: a single wall-clock call is at the mercy of the host's other processes
                barrier()
                t0 = time.perf_counter()
                out = fn()
                barrier()
                dt = time.perf_counter() - t0
                best = dt if best is None else min(best, dt)
            return best, out

        snp_s, chunks = timed_call(lambda: nadavca_b200.estimate_snps(None, reads_api, reference=genome, config=cfg,
                                                                      kmer_model=km, independent=True, aligner=aligner))
        align_s, aligned = timed_call(lambda: list(nadavca_b200.align_signal(None, reads_api, config=cfg, kmer_model=km,
                                                                             aligner=aligner, reference=genome)))
        api = {'estimate_snps_s': reduce_over_ranks(snp_s, 'max', dev),
               'align_signal_s': reduce_over_ranks(align_s, 'max', dev),
               'raw_samples': reduce_over_ranks(raw_samples, 'sum', dev),
               'chunks': len([c for c in chunks if c is not None]),
               'aligned': sum(1 for _, res in aligned if res is not None)}

    # ---- reductions over ranks -----------------------------------------------------------------------------------
    ms_max = reduce_over_ranks(ms, 'max', dev)
    e2e_max = reduce_over_ranks(e2e_s, 'max', dev)
    samples_all = reduce_over_ranks(float(samples), 'sum', dev)
    cells_all = reduce_over_ranks(float(total_cells), 'sum', dev)
    launches_all = reduce_over_ranks(float(launches), 'sum', dev)

    if rank == 0:
        value = samples_all * args.steps / (ms_max * 1e-3)
        peaks = {}
        try:
            with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as fh:
                peaks = json.load(fh)
        except OSError:
            pass
        hbm_peak = peaks.get('hbm_gbs', 6650.0)
        peak_src = 'measured' if 'hbm_gbs' in peaks else 'fallback'
        snp_ms, snp_n = tt['snp']
        snp_launch_ms = snp_ms / max(snp_n, 1)
        snp_bytes_per_launch = abytes['snp'] * args.steps / max(snp_n, 1)
        achieved = snp_bytes_per_launch / (snp_launch_ms * 1e-3) / 1e9 if snp_launch_ms > 0 else 0.0
        fma_rate = dtw.measure_fp64_fma_rate(local_rank)
        snp_cells_per_s = cells['estimate_snp'] * args.steps / (snp_ms * 1e-3) if snp_ms > 0 else 0.0
        line = {
            'metric': 'signal_samples_aligned_per_sec', 'value': value, 'unit': 'samples/s', 'n_gpus': world,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_max / args.steps,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'dp_cells_per_sec': cells_all * args.steps / (ms_max * 1e-3),
            'config': workload_config(args, args.reads),
            'e2e': {'value': samples_all * e2e_steps / e2e_max, 'unit': 'samples/s', 'h2d_bytes_per_step': h2d,
                    'd2h_bytes_per_step': d2h, 'steps': e2e_steps},
            'gpu_launches': int(launches_all),
            'clocks': clocks.summary(),
            'roofline': {'bound': 'hbm', 'kernel': 'snp3_kernel', 'achieved': achieved, 'peak': hbm_peak,
                         'unit': 'GB/s', 'frac': achieved / hbm_peak, 'traffic': ncu_traffic(args.reads), 'peak_source': peak_src,
                         'launch_ms': snp_launch_ms, 'algorithmic_bytes_per_launch': snp_bytes_per_launch,
                         'note': 'the SNP kernel is instruction-issue / FP64-pipe bound, not HBM bound: see alu'},
            'alu': alu_block(snp_cells_per_s, snp_launch_ms, fma_rate, clocks.summary().get('sm_mhz'), args.reads),
            'stage_ms_per_step': {'rows_refine': tn['rows'][0] / args.steps, 'path': tn['path'][0] / args.steps,
                                  'rows_estimate': tt['rows'][0] / args.steps, 'no_snp': tt['no_snp'][0] / args.steps,
                                  'snp': tt['snp'][0] / args.steps},
            'cells_per_step_per_gpu': cells,
            'api': None if api is None else {
                'estimate_snps': {'call': 'nadavca_b200.estimate_snps(reads, independent=True)',
                                  'seconds': api['estimate_snps_s'], 'unit': 'raw samples/s',
                                  'value': api['raw_samples'] / api['estimate_snps_s'], 'chunks': api['chunks']},
                'align_signal': {'call': 'nadavca_b200.align_signal(reads)  (two alignment rounds, transitions)',
                                 'seconds': api['align_signal_s'], 'unit': 'raw samples/s',
                                 'value': api['raw_samples'] / api['align_signal_s'], 'aligned': api['aligned']},
                'reads_per_gpu': args.reads},
            'consensus': None if consensus is None else dict(
                consensus, value=samples_all / (consensus['ms_per_step'] * 1e-3), unit='samples/s',
                bus_GBs=(consensus['bus_bytes_per_step'] / (consensus['exchange_ms_per_step'] * 1e-3) / 1e9
                         if consensus['exchange_ms_per_step'] > 0 else None),
                nvlink_peak_GBs_per_direction=900.0,
                workload='configs[2] shape: estimate_snps independent=False, %d reads per GPU over a %.1f Mb '
                         'synthetic genome; timed region includes the NCCL exchange' % (args.reads, args.genome / 1e6)),
        }
        if world == 1 and not args.no_cpu_baseline:
            line['cpu_baseline'], line['parity'] = cpu_baseline(km, items, tweaked, args, mel, gpu_events, gpu_ll)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def alu_block(snp_cells_per_s, snp_launch_ms, fma_rate, sm_mhz, reads_per_gpu):
    """The bound that matters for the dominant kernel: instruction issue and the FP64 pipe, not HBM.  A B200 SM issues
    4 warp instructions per clock (one per scheduler).  `issue_frac` = warp instructions of one launch (counted by ncu
    in the committed capture of the same workload, profiles/snp_traffic.json: the kernel executes the same
    instructions for the same reads) / the launch time measured LIVE in this run / the issue peak at the SM clock
    sampled live.  `fp64_pipe_frac`: the capture's FP64-pipe utilisation rescaled by the same time ratio."""
    out = {'kernel': 'snp3_kernel', 'dp_cells_per_sec': snp_cells_per_s, 'fp64_fma_per_sec_measured': fma_rate,
           'issue_frac': None, 'fp64_pipe_frac': None,
           'source': 'profiles/snp_traffic.json (ncu --set full of the same kernel and workload) + live launch time'}
    try:
        with open(os.path.join(ROOT, 'profiles', 'snp_traffic.json')) as fh:
            cap = json.load(fh)
        if cap.get('reads_per_gpu') != reads_per_gpu or snp_launch_ms <= 0:
            return out
        issue_peak = 148 * 4 * (sm_mhz or 1965.0) * 1e6  # warp instructions per second
        out['warp_instructions_per_launch'] = cap['warp_instructions_per_launch']
        out['issue_frac'] = cap['warp_instructions_per_launch'] / (snp_launch_ms * 1e-3) / issue_peak
        out['fp64_pipe_frac'] = cap['fp64_pipe_pct'] / 100.0 * cap['launch_ms'] / snp_launch_ms
        out['captured'] = {'issue_active_pct': cap['issue_active_pct'], 'fp64_pipe_pct': cap['fp64_pipe_pct'],
                           'alu_pipe_pct': cap.get('alu_pipe_pct'), 'launch_ms': cap['launch_ms']}
    except (OSError, ValueError, KeyError, AttributeError, TypeError):
        pass
    return out


def ncu_traffic(reads_per_gpu):
    """dram__bytes_read.sum + dram__bytes_write.sum of one snp3_kernel launch from the committed ncu --set full capture
    (profiles/snp_traffic.json, written by tools/ncu_traffic.py); null when the capture is for another batch size."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'snp_traffic.json')) as fh:
            t = json.load(fh)
        return t['dram_bytes_per_launch'] if t.get('reads_per_gpu') == reads_per_gpu else None
    except (OSError, ValueError, KeyError, AttributeError, TypeError):
        return None


def cpu_sample_size(args, n_items):
    """Reads of the CPU leg: at least 64 (a multiple of the host cores, so that every core is busy to the end)."""
    cores = os.cpu_count() or 1
    want = args.cpu_sample or max(64, cores)
    if not args.cpu_sample and want % cores:
        want += cores - want % cores
    return min(n_items, want)


def cpu_baseline(km, items, tweaked, args, mel, gpu_events, gpu_ll):
    """The reference's CPU implementation on the first reads of the benchmarked workload, timed on the host cores,
    and -- with its results -- the check of what the GPU computed for the same reads during the timed steps."""
    from oracle import oracle as orc
    from oracle import parity
    cores = os.cpu_count() or 1
    n_sample = cpu_sample_size(args, len(items))
    tasks = cpu_tasks(km, items[:n_sample], tweaked[:n_sample], args.bandwidth, mel)
    arm = CpuArm(km, min(cores, n_sample), method='spawn')  # CUDA is initialised in this process: do not fork
    t = arm.run(tasks)
    results = arm.results
    arm.close()
    samples = sum(len(it['signal']) for it in items[:n_sample])
    base = {'value': samples / t, 'unit': 'samples/s', 'cores': arm.cores, 'kind': arm.kind,
            'sample': 'first %d reads of the workload, one per worker process, %.1f s wall' % (n_sample, t)}
    om = orc.OracleModel(km.get_k(), km.get_central_position(), 4, km.mean, km.sigma, 'port')
    par = {'reads': n_sample, 'against': arm.kind, 'event_mismatches': 0, 'tie_accepts': 0, 'max_ll_rel': 0.0,
           'll_mismatches': 0, 'events_compared': 0, 'll_rtol': 1e-9}
    for i, (task, (ev, ll)) in enumerate(zip(tasks, results)):
        signal, _, ref, cb, ca, anchors, bw, _ = task
        par['events_compared'] += len(ev)
        try:
            kind = parity.compare_events(gpu_events[i], signal, ref, cb, ca, anchors, bw, mel, om, False, want=ev)
            par['tie_accepts'] += kind == 'tie'
        except AssertionError:
            par['event_mismatches'] += 1
        try:
            rel = parity.ll_max_rel(gpu_ll[i], ll)
            par['max_ll_rel'] = max(par['max_ll_rel'], rel)
            par['ll_mismatches'] += rel > par['ll_rtol']
        except AssertionError:
            par['ll_mismatches'] += 1
    return base, par


def relaunch_under_torchrun(args):
    """`python bench.py --gpus N` (N > 1) without a launcher: start one rank per GPU on this node ourselves."""
    import socket
    with socket.socket() as sock:
        sock.bind(('127.0.0.1', 0))
        port = sock.getsockname()[1]
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(args.gpus),
           '--master-addr', '127.0.0.1', '--master-port', str(port), os.path.abspath(__file__)] + sys.argv[1:]
    raise SystemExit(subprocess.call(cmd))


if __name__ == '__main__':
    a = parse_args()
    if a.gpus > 1 and 'WORLD_SIZE' not in os.environ:
        relaunch_under_torchrun(a)
    if a.impl == 'reference':
        run_reference(a)
    elif a.config in (0, 3, 4):
        import bench_configs
        bench_configs.run(sys.modules[__name__], a)
    else:
        run_ours(a)
