"""Batched estimator glue on top of the B200 kernels (reference nadavca/estimator.py).

Same classes and method names as the reference (``Chunk``, ``ProbabilityEstimator`` with
``get_refined_alignment``, ``_estimate_log_likelihoods``, ``estimate_probabilities``, ``_compute_posterior``), but
every method that touches the DP gathers ALL reads first and makes one trip to the GPU per stage:

    host: approximate alignment, slicing, contexts            (estimator.py:60-74, 159-170)
    GPU : refine_alignment(model_transitions=False) batch     (estimator.py:77-87)
    host: Read.tweak_signal_normalization (scipy spline)      (estimator.py:89-97)
    GPU : estimate_log_likelihoods batch -> normalise / strand flip -> [consensus scatter-add -> all-reduce]
          -> Bayesian posterior                                (estimator.py:99-121, 199-236)

torch is used only for device buffers, the current stream and (consensus mode, several ranks) the NCCL all-reduce.
"""
import numpy

from . import dtw
from .alphabet import alphabet
from .genome import Genome, _as_bytes

_REF_LUT = numpy.full(256, 4, dtype=numpy.int8)
for _i, _b in enumerate(alphabet):
    _REF_LUT[ord(_b)] = _i


def _ref_codes(reference_slice):
    """Reference characters -> int8 codes 0..3, 4 for anything else (never equal to a base, like the reference's
    string comparison in estimator.py:141,150)."""
    arr = numpy.asarray(reference_slice) if not isinstance(reference_slice, str) else reference_slice
    if not isinstance(arr, str) and arr.dtype.kind in 'iu':
        return arr.astype(numpy.int8)
    if len(arr) == 0:
        return numpy.zeros(0, dtype=numpy.int8)
    return _REF_LUT[_as_bytes(arr)]  # (arrays of 1-char strings are read as UCS4 code points: no per-element cast)


class Chunk:
    """estimator.py:7-31."""

    def __init__(self, start, end, values, coverage=None):
        self.start = start
        self.end = end
        self.values = values
        self.coverage = coverage
        if coverage is None:
            self.coverage = numpy.ones(end - start, dtype=int)

    def __lt__(self, other):
        if self.start == other.start:
            return self.end < other.end
        return self.start < other.start

    @staticmethod
    def print_head(file):
        file.write('index\tbase\tcoverage\t{}\n'.format('\t'.join(alphabet)))

    def print(self, file, reference):
        for i in range(self.start, self.end):
            values_string = '\t'.join(map('{:18.16f}'.format, self.values[i - self.start]))
            file.write('{}\t{}\t{}\t{}\n'.format(i, reference[i], self.coverage[i - self.start], values_string))


class _Prepared:
    """Per-read host preparation shared by both paths."""
    __slots__ = ('read', 'apx', 'reference_part', 'signal_range', 'context_before', 'context_after')


def group_intervals(intervals):
    """Overlap groups of (start, end) intervals sorted by (start, end) -- estimator.py:205-220; a chunk starting
    exactly at the running end opens a new group ('>=').  Returns [(group_start, group_end, [member indices])]."""
    order = sorted(range(len(intervals)), key=lambda i: (intervals[i][0], intervals[i][1]))
    groups = []
    members, cur_start, cur_end = [], None, None
    for pos, idx in enumerate(order):
        start, end = intervals[idx]
        if cur_start is None:
            cur_start, cur_end = start, end
        members.append(idx)
        cur_end = max(cur_end, end)
        if pos + 1 >= len(order) or intervals[order[pos + 1]][0] >= cur_end:
            groups.append((cur_start, cur_end, members))
            members, cur_start, cur_end = [], None, None
    return groups


class ProbabilityEstimator:
    def __init__(self, kmer_model, aligner, config):
        self.kmer_model = kmer_model
        self.aligner = aligner
        self.bandwidth = config['bandwidth']
        self.snp_prior = config['snp_prior_probability']
        self.min_event_length = config['min_event_length']
        self.model_wobbling = config['model_wobbling']
        self.model_transitions = config['model_transitions']
        self.normalization_event_length = config['normalization_event_length']
        self.tweak_signal_normalization = config['tweak_signal_normalization']
        self.workspace_limit = config.get('workspace_limit_bytes', 0) if hasattr(config, 'get') else 0
        self.sub_batch_reads = config.get('sub_batch_reads', 256) if hasattr(config, 'get') else 256
        self.last_stats = {}

    # ---- small host helpers with the reference's names ------------------------------------------------------
    def _normalize_log_likelihoods(self, likelihoods, reference):
        shift = likelihoods[0][reference[0]]
        return (likelihoods - shift) / self.normalization_event_length

    def _get_read_context(self, read, read_sequence_range):
        start, end = read_sequence_range
        k = self.kmer_model.get_k()
        central_position = self.kmer_model.get_central_position()
        lo = start - central_position
        # Python slicing semantics of the reference (estimator.py:53): a negative lower bound wraps around
        context_before = read.sequence[lo:start]
        context_after = read.sequence[end:end + k - central_position - 1]
        return Genome.to_numerical(context_before), Genome.to_numerical(context_after)

    def _corrected_priors(self, context_positions):
        c = len(alphabet) - 1
        p_1 = 1 - self.snp_prior
        p_2 = self.snp_prior / c
        snp_hypothesis_prior = 1 / (p_1 / p_2 + (1 - context_positions) * c)
        nonsnp_hypothesis_prior = 1 - snp_hypothesis_prior * c
        return snp_hypothesis_prior, nonsnp_hypothesis_prior

    def _prepare(self, read, reference=None):
        apx = self.aligner.get_signal_alignment(read, self.bandwidth)
        if apx is None:
            return None
        item = _Prepared()
        item.read = read
        item.apx = apx
        if reference is None:  # get_refined_alignment uses the aligner's reference part (estimator.py:164)
            part = apx.reference_part
        else:                  # _estimate_log_likelihoods slices the given reference (estimator.py:64-68)
            start, end = apx.reference_range
            part = reference[start:end]
            if apx.reverse_complement:
                part = Genome.reverse_complement(part)
        item.reference_part = Genome.to_numerical(part)
        item.signal_range = apx.signal_range
        item.context_before, item.context_after = self._get_read_context(read, apx.read_sequence_range)
        return item

    def _batch(self, items, signals):
        return dtw.Batch(self.kmer_model, signals, [it.reference_part for it in items],
                         [it.context_before for it in items], [it.context_after for it in items],
                         [it.apx.alignment for it in items], self.bandwidth, self.min_event_length,
                         workspace_limit=self.workspace_limit)

    # ---- path A: refined alignments ---------------------------------------------------------------------------
    def get_refined_alignments(self, reads, with_event_means=False, prepared=None):
        """Batched get_refined_alignment: list (one per read) of (ApproximateSignalAlignment, int (n,3) array) or
        None for reads that are unaligned or have no valid path.  With `with_event_means` every result carries a third
        item, the mean signal level of each event (``numpy.mean(normalized_signal[start:end])`` bit for bit, computed
        on the device) -- what the renormalisation rounds of align_signal need (align_signal.py:66-70).

        `prepared`: the value of ``self.last_prepared`` after an earlier call with the same reads -- the approximate
        alignments (which depend on the base sequence only, not on the signal normalisation) are then reused instead
        of asking the aligner again."""
        if prepared is None:
            prepared = [self._prepare(read) for read in reads]
        self.last_prepared = prepared
        items = [it for it in prepared if it is not None]
        results = [None] * len(reads)
        if not items:
            return results
        signals = [it.read.normalized_signal[it.signal_range[0]:it.signal_range[1]] for it in items]
        with self._batch(items, signals) as batch:
            # every kernel of the batch runs on the caller's current torch stream; the getters below read back on it
            batch.refine(self.model_transitions, _current_stream(self.kmer_model))
            tables = batch.alignment_tables([it.signal_range[0] for it in items],
                                            [it.apx.reference_range[0] for it in items],
                                            [it.apx.reference_range[1] for it in items],
                                            [int(it.apx.reverse_complement) for it in items])
            means = batch.event_means() if with_event_means else None
            self.last_stats = {'launches': batch.launch_count}
        pos = 0
        for i, it in enumerate(prepared):
            if it is None:
                continue
            table = tables[pos]
            if table is not None:
                results[i] = (it.apx, table.astype(int)) + ((means[pos].copy(),) if with_event_means else ())
            pos += 1
        return results

    def get_refined_alignment(self, read):
        """estimator.py:158-196 (a batch of one)."""
        return self.get_refined_alignments([read])[0]

    # ---- path B: log-likelihood chunks ---------------------------------------------------------------------------
    def _run_estimate(self, reference, reads):
        """Shared front half of path B.  Returns (items, subs): the prepared reads that aligned and have a path, and
        a list of (batch, count) sub-batches covering them in order, raw log-likelihoods resident on the device -- or
        ([], []).  Reads whose approximate alignment or refinement fails are dropped (the reference returns None /
        crashes in splrep for them).

        The reads are cut into sub-batches of ``sub_batch_reads`` (config key, default 256), each on its own CUDA
        stream (per-stream DP workspaces, csrc/api.cu), so that the host work between the two DP calls -- D2H of the
        event means, the FITPACK spline fits (worker processes), H2D of the splines -- of one sub-batch overlaps the
        kernels of the others.

        The model keeps one DP workspace per stream until it is destroyed, so the sub-batch streams are created once
        per device and process (``_sub_batch_streams``) and reused by every call and every estimator: a process that
        calls this over and over holds at most four sub-batch workspaces per model, not one per stream torch hands
        out.  Work on a caller's own current stream (a single sub-batch runs there) is the caller's business: every
        distinct stream a caller runs on keeps its own workspace."""
        from .read import fit_splines_async
        items = [it for it in (self._prepare(read, reference) for read in reads) if it is not None]
        if not items:
            return [], []
        main = _current_stream(self.kmer_model)
        per = max(1, int(self.sub_batch_reads))
        n_sub = -(-len(items) // per)
        bounds = [len(items) * j // n_sub for j in range(n_sub + 1)]
        streams = _sub_batch_streams(_device(self.kmer_model), min(n_sub, 4)) if n_sub > 1 else [main]
        subs = []
        for j in range(n_sub):
            sub_items = items[bounds[j]:bounds[j + 1]]
            st = streams[j % len(streams)]
            st.wait_stream(main)
            batch = self._batch(sub_items, [it.read.normalized_signal[it.signal_range[0]:it.signal_range[1]]
                                            for it in sub_items])
            if self.tweak_signal_normalization:
                batch.refine(False, st)
            subs.append([batch, sub_items, st])
        if self.tweak_signal_normalization:
            fits = []
            for sub in subs:
                batch, sub_items, st = sub
                events, _ = batch.events()
                event_means = batch.event_means()  # per-event signal means, computed next to the resident events
                keep = [i for i, ev in enumerate(events) if ev is not None]
                if len(keep) != len(sub_items):
                    batch.close()
                    sub_items = [sub_items[i] for i in keep]
                    event_means = [event_means[i] for i in keep]
                    if sub_items:
                        batch = self._batch(sub_items, [it.read.normalized_signal[it.signal_range[0]:it.signal_range[1]]
                                                        for it in sub_items])
                    else:
                        batch = None
                    sub[0], sub[1] = batch, sub_items
                expected = self.kmer_model.get_expected_signal_batch([it.reference_part for it in sub_items],
                                                                     [it.context_before for it in sub_items],
                                                                     [it.context_after for it in sub_items]) \
                    if sub_items else []
                # host: the smoothing-spline FIT per read (scipy splrep, read.py:93), in worker processes
                fits.append(fit_splines_async(zip(event_means, expected)))
            for (batch, sub_items, st), fit in zip(subs, fits):
                if batch is None:
                    continue
                splines = fit.get()
                for it, spline in zip(sub_items, splines):
                    it.read.tweak_spline = spline
                    it.read.tweaked_normalized_signal = None
                # device: the spline EVALUATION over the resident signal slices (read.py:94), which therefore never
                # travel back to the host
                batch.apply_splines(splines, st)
                batch.estimate(self.model_wobbling, st)
        else:
            for batch, sub_items, st in subs:
                batch.estimate(self.model_wobbling, st)
        for _, _, st in subs:
            main.wait_stream(st)
        subs = [(batch, sub_items) for batch, sub_items, _ in subs if batch is not None]
        return [it for _, sub_items in subs for it in sub_items], [(batch, len(sub_items)) for batch, sub_items in subs]

    def _estimate_log_likelihoods(self, reference, read):
        """estimator.py:59-121 for one read: Chunk of normalised, strand-corrected log-likelihoods or None."""
        chunks = self.estimate_log_likelihood_chunks(reference, [read])
        return chunks[0] if chunks else None

    def estimate_log_likelihood_chunks(self, reference, reads):
        import torch
        items, subs = self._run_estimate(reference, reads)
        if not subs:
            return []
        stream = _current_stream(self.kmer_model)
        out = []
        try:
            lo = 0
            for batch, count in subs:
                sub_items = items[lo:lo + count]
                lo += count
                d_chunks = torch.empty((batch.pack.total_reference, 4), dtype=torch.float64,
                                       device=_device(self.kmer_model))
                batch.chunk_values([int(it.apx.reverse_complement) for it in sub_items],
                                   self.normalization_event_length, d_chunks.data_ptr(), stream)
                values = d_chunks.cpu().numpy()
                off = batch.pack.reference_off
                out.extend(Chunk(it.apx.reference_range[0], it.apx.reference_range[1], values[off[i]:off[i + 1]].copy())
                           for i, it in enumerate(sub_items))
        finally:
            for batch, _ in subs:
                batch.close()
        return out

    def _compute_posterior(self, log_likelihoods, reference):
        """estimator.py:131-156 for one group, on the device: the log-likelihoods go through the consensus-row
        posterior kernel as a group of rows of 5 doubles (coverage column 0)."""
        import torch
        dev = _device(self.kmer_model)
        ll = torch.as_tensor(numpy.asarray(log_likelihoods, dtype=numpy.float64), device=dev)
        L = ll.shape[0]
        rows = torch.zeros((L, 5), dtype=torch.float64, device=dev)
        rows[:, :4] = ll
        ref = torch.as_tensor(_ref_codes(reference), device=dev)
        group_off = torch.tensor([0, L], dtype=torch.int64, device=dev)
        out = torch.empty_like(rows)
        dtw.posterior_rows(dev.index, rows.data_ptr(), 0, 0, L, ref.data_ptr(), group_off.data_ptr(), 1,
                           self.kmer_model.get_k(), self.snp_prior, out.data_ptr(), torch.cuda.current_stream())
        return out[:, :4].cpu().numpy()

    def estimate_probabilities(self, reference, reads, independent=False, process_group=None):
        """estimator.py:199-236.  `independent=True` treats every read as its own group (what estimate_snps does
        with one call per read, estimate_snps.py:63-68) and returns one entry per input read in input order: its
        Chunk, or None when the read did not align / has no path.
        Otherwise chunks are summed per overlap group; with an initialised torch.distributed `process_group` the
        reads given to each rank are that rank's shard and the per-position sums are all-reduced over NCCL."""
        items, subs = self._run_estimate(reference, reads)
        try:
            stage = self.posterior_stage(subs, [int(it.apx.reverse_complement) for it in items],
                                         [tuple(it.apx.reference_range) for it in items], reference, independent,
                                         process_group)
            if stage is None:
                return [None] * len(reads) if independent else []
            groups, group_off, out, cov = stage
            # D2H through a cached pinned buffer; the Chunks below take their own copies of their rows
            from .read import _staging
            import torch
            count = out.numel()
            pinned = _staging('probabilities', count)
            pinned[:count].copy_(out.reshape(-1), non_blocking=True)
            coverage = cov.cpu().numpy().astype(int)  # (synchronises the stream: the pinned copy has landed too)
            torch.cuda.current_stream(out.device).synchronize()
            probabilities = pinned.numpy()[:count].reshape(tuple(out.shape))
            self.last_stats = {'launches': sum(batch.launch_count for batch, _ in subs) + 1,
                               'groups': len(groups), 'positions': int(group_off[-1]), 'sub_batches': len(subs)}
        finally:
            for batch, _ in subs:
                batch.close()
        chunks = [Chunk(g[0], g[1], probabilities[group_off[i]:group_off[i + 1]].copy(),
                        coverage[group_off[i]:group_off[i + 1]].copy()) for i, g in enumerate(groups)]
        if not independent:
            return chunks
        # one entry per input read, in input order; None for reads that did not align or have no path (the reference
        # indexes chunks[0] per read, estimate_snps.py:65-67, and crashes on those)
        position = {id(it.read): i for i, it in enumerate(items)}
        return [chunks[position[id(read)]] if id(read) in position else None for read in reads]

    def posterior_stage(self, batch, reverse, intervals, reference, independent=False, process_group=None,
                        plan=None, collective='auto', events=None):
        """Device half of estimate_probabilities after the raw log-likelihoods exist in `batch` (one ``dtw.Batch``,
        None, or the list of (batch, read count) sub-batches of ``_run_estimate``; `reverse` / `intervals` cover the
        reads of all sub-batches in order): normalise / flip,
        scatter-add into the concatenated groups, the exchange between ranks (consensus mode only, see
        ``consensus_exchange``), posterior stencil.  Returns (groups, group_off, probabilities tensor (total,4),
        coverage tensor (total,)) or None.  `plan` (from ``plan_groups``) can be reused between calls with the same
        intervals; `events`, a dict, receives CUDA event pairs around the exchange (``events['exchange']``) and its
        payload in bytes."""
        import torch
        dev = _device(self.kmer_model)
        stream = torch.cuda.current_stream()
        dist = _dist(process_group)
        if plan is None:
            plan = self.plan_groups(intervals, reference, independent, process_group)
        if plan is None:
            return None
        groups, group_off, dest, d_ref = plan[:4]
        d_group_off = plan[4] if len(plan) > 4 else torch.as_tensor(group_off, device=dev)
        total = int(group_off[-1])
        k = self.kmer_model.get_k()
        world = dist.get_world_size(process_group) if (dist is not None and not independent) else 1
        slice_rows, total_pad = slice_geometry(total, world)
        # consensus rows [sum A, sum C, sum G, sum T, coverage] (estimator.py:226-231): one buffer, one collective
        rows = torch.zeros((total_pad, 5), dtype=torch.float64, device=dev)
        subs = batch if isinstance(batch, (list, tuple)) else ([(batch, len(reverse))] if batch is not None else [])
        lo = 0
        for sub, count in subs:
            d_chunks = torch.empty((sub.pack.total_reference, 4), dtype=torch.float64, device=dev)
            sub.chunk_values(reverse[lo:lo + count], self.normalization_event_length, d_chunks.data_ptr(), stream)
            sub.scatter_add_rows(d_chunks.data_ptr(), dest[lo:lo + count], rows.data_ptr(), stream)
            lo += count

        def posterior_rows(local, base_row, row_lo, row_hi, out_rows):
            dtw.posterior_rows(dev.index, local.data_ptr(), base_row, row_lo, row_hi, d_ref.data_ptr(),
                               d_group_off.data_ptr(), len(groups), k, self.snp_prior, out_rows.data_ptr(), stream)

        out = consensus_exchange(rows, total, k - 1, process_group if world > 1 else None, posterior_rows, collective,
                                 events)
        return groups, group_off, out[:total, :4].contiguous(), out[:total, 4].to(torch.int32)

    def _reference_codes(self, reference):
        """int8 codes of the whole reference, converted once per reference object (character arrays convert at
        ~10 ns per base, but one call per read cost 0.2 ms each: 0.2 s per 1000 reads in ``plan_groups``)."""
        cached = getattr(self, '_codes_cache', None)
        if cached is None or cached[0] is not reference or cached[1] != len(reference):
            cached = (reference, len(reference), _ref_codes(reference))
            self._codes_cache = cached
        return cached[2]

    def plan_groups(self, intervals, reference, independent=False, process_group=None):
        """Host planning of the overlap groups (estimator.py:205-220): (groups, group_off, dest rows of the local
        chunks, device int8 reference codes) or None when no read aligned anywhere."""
        import torch
        dev = _device(self.kmer_model)
        host = plan_groups_host(intervals, independent, process_group)
        if host is None:
            return None
        groups, group_off, dest = host
        codes = self._reference_codes(reference)  # the whole reference once, not one conversion per group
        ref_codes = numpy.concatenate([codes[g[0]:g[1]] for g in groups])
        d_ref = torch.as_tensor(ref_codes, device=dev)
        d_group_off = torch.as_tensor(group_off, device=dev)
        return groups, group_off, dest, d_ref, d_group_off


def slice_geometry(total, world):
    """Rows per rank and padded row count when the concatenated groups are cut into `world` equal genome slices."""
    rows = -(-max(total, 1) // world)
    return rows, rows * world


def consensus_exchange(rows, total, halo, process_group, posterior_rows, collective='auto', events=None):
    """The one exchange step of consensus mode (estimator.py:226-231: per-position sums over the reads of ALL ranks)
    followed by the posterior stencil.  `rows` is this rank's (total_pad, 5) accumulator [A, C, G, T, coverage].

      'reduce_scatter' (default for several ranks): ONE reduce-scatter leaves every rank with the reduced rows of its
          own genome slice; a tiny all-gather brings in the k-1 = `halo` reduced rows either side of it (the posterior
          window, estimator.py:135-136); each rank computes the posterior of its slice only; ONE all-gather
          distributes probabilities and coverage.  Traffic per rank: (N-1)/N of the buffer each way.
      'allreduce': one all-reduce of the whole buffer, posterior replicated on every rank.
      no process group: posterior over the local rows.

    `posterior_rows(local, base_row, row_lo, row_hi, out_rows)` computes rows [row_lo, row_hi) from `local`, whose
    first row is global row `base_row`, into `out_rows` (rows of 5 = probabilities + coverage).  Works on CUDA tensors
    (NCCL) and on CPU tensors (gloo, the CPU tests).  Returns (>= total, 5) rows."""
    import torch
    if process_group is None:
        out = torch.empty_like(rows)
        posterior_rows(rows, 0, 0, total, out)
        return out
    import torch.distributed as dist
    world, rank = dist.get_world_size(process_group), dist.get_rank(process_group)
    slice_rows, total_pad = slice_geometry(total, world)
    assert rows.shape[0] == total_pad and rows.shape[1] == 5
    mode = collective
    if mode == 'auto':
        mode = 'reduce_scatter' if (world > 1 and slice_rows >= halo) else 'allreduce'
    timing = events is not None and rows.is_cuda
    if timing:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    if mode == 'allreduce':
        dist.all_reduce(rows, group=process_group)
        if timing:
            e1.record()
            events['exchange'] = [(e0, e1)]
            events['bus_bytes'] = rows.numel() * 8 * 2 * (world - 1) / world
        out = torch.empty_like(rows)
        posterior_rows(rows, 0, 0, total, out)
        if events is not None:
            events['mode'] = mode
        return out
    local = torch.zeros((slice_rows + 2 * halo, 5), dtype=rows.dtype, device=rows.device)
    dist.reduce_scatter_tensor(local[halo:halo + slice_rows].view(-1), rows.view(-1), group=process_group)
    if halo > 0:
        edges = torch.cat([local[halo:2 * halo], local[slice_rows:slice_rows + halo]])  # own first / last halo rows
        all_edges = torch.empty((world, 2 * halo, 5), dtype=rows.dtype, device=rows.device)
        dist.all_gather_into_tensor(all_edges.view(-1), edges.reshape(-1), group=process_group)
        if rank > 0:
            local[:halo] = all_edges[rank - 1, halo:]
        if rank < world - 1:
            local[halo + slice_rows:] = all_edges[rank + 1, :halo]
    if timing:
        e1.record()
    lo = rank * slice_rows
    hi = max(lo, min(lo + slice_rows, total))
    out_slice = torch.zeros((slice_rows, 5), dtype=rows.dtype, device=rows.device)
    posterior_rows(local, lo - halo, lo, hi, out_slice)
    if timing:
        e2 = torch.cuda.Event(enable_timing=True)
        e3 = torch.cuda.Event(enable_timing=True)
        e2.record()
    out = torch.empty((total_pad, 5), dtype=rows.dtype, device=rows.device)
    dist.all_gather_into_tensor(out.view(-1), out_slice.view(-1), group=process_group)
    if timing:
        e3.record()
        events['exchange'] = [(e0, e1), (e2, e3)]
        events['bus_bytes'] = 2 * rows.numel() * 8 * (world - 1) / world
    if events is not None:
        events['mode'] = mode
    return out


def plan_groups_host(intervals, independent=False, process_group=None):
    """Pure host half of ``plan_groups`` (no device access, so it runs under the gloo backend in the CPU tests):
    the overlap groups over the reads of ALL ranks, the concatenated row offset of every group and, for each LOCAL
    read, the row of the concatenated accumulator its chunk is added at.  In consensus mode over several ranks the
    (start, end) intervals are exchanged with one all_gather_object; `independent` needs no exchange."""
    dist = _dist(process_group)
    if dist is not None and not independent:
        gathered = [None] * dist.get_world_size(process_group)
        dist.all_gather_object(gathered, [tuple(map(int, iv)) for iv in intervals], group=process_group)
        all_intervals = [tuple(iv) for part in gathered for iv in part]
    else:
        all_intervals = [tuple(iv) for iv in intervals]
    if not all_intervals:
        return None
    if independent:
        groups = [(s, e, [i]) for i, (s, e) in enumerate(intervals)]
    else:
        groups = group_intervals(all_intervals)
    group_off = numpy.zeros(len(groups) + 1, dtype=numpy.int64)
    group_off[1:] = numpy.cumsum([g[1] - g[0] for g in groups])
    starts = numpy.array([g[0] for g in groups], dtype=numpy.int64)
    if independent:
        dest = group_off[:-1].copy()
    elif len(intervals):
        local_starts = numpy.array([iv[0] for iv in intervals], dtype=numpy.int64)
        gi = numpy.searchsorted(starts, local_starts, side='right') - 1
        dest = group_off[gi] + (local_starts - starts[gi])
    else:
        dest = numpy.zeros(0, dtype=numpy.int64)
    return groups, group_off, dest


def shard_reads(work, world_size):
    """Deal reads to ranks by longest-processing-time-first on a per-read work estimate (DP cells ~ bases x band
    width): returns a list of `world_size` index lists, each in ascending read order.  Reads are independent units
    (estimator.py:201-204), so this is the whole multi-GPU partitioning; ties and equal work fall back to a
    round-robin deal."""
    work = numpy.asarray(work, dtype=numpy.float64)
    order = numpy.argsort(-work, kind='stable')
    load = numpy.zeros(world_size)
    shards = [[] for _ in range(world_size)]
    for idx in order:
        r = int(numpy.argmin(load))
        shards[r].append(int(idx))
        load[r] += work[idx]
    return [sorted(s) for s in shards]


def _current_stream(kmer_model):
    """torch's current stream on the model's device (the kernels of a call are enqueued on it, so the estimator may
    be used under ``with torch.cuda.stream(s)``)."""
    import torch
    return torch.cuda.current_stream(_device(kmer_model))


_SUB_BATCH_STREAMS = {}


def _sub_batch_streams(dev, count):
    """The first `count` sub-batch streams of device `dev`, created on first use and kept for the process
    (``torch.cuda.Stream()`` hands out a different pooled stream on every call, and each new stream would cost the
    model a new DP workspace)."""
    import torch
    cache = _SUB_BATCH_STREAMS.setdefault(dev.index, [])
    while len(cache) < count:
        cache.append(torch.cuda.Stream(device=dev))
    return cache[:count]


def _device(kmer_model):
    import torch
    if not torch.cuda.is_available():
        raise dtw.NadavcaCudaError('no CUDA device available: nadavca_b200 has no CPU fallback')
    dev = torch.device('cuda', kmer_model.device)
    torch.cuda.set_device(dev)
    return dev


def _dist(process_group):
    """torch.distributed when the caller passed a process group, else None: collectives are never implied by an
    initialised default group (a rank may well run a single-GPU estimate next to a distributed job)."""
    if process_group is None:
        return None
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist
    return None
