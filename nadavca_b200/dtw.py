"""Drop-in for the reference's native module ``nadavca.dtw`` (nadavca/dtw/dtwmodule.cpp:10-29) on top of the
B200 kernels: ``KmerModel``, ``refine_alignment`` and ``estimate_log_likelihoods`` keep the reference's keyword
signatures (a batch of one read); ``Batch`` is the batched, device-resident form the estimator uses.
"""
import ctypes

import numpy as np

from . import _cabi
from ._cabi import NadavcaCudaError, ReadsPack  # noqa: F401  (re-exported)


class KmerModel:
    """KmerModel(k, central_position, alphabet_size, mean, sigma) -- dtwmodule.cpp:12-18.

    The per-k-mer tables live on the GPU (created lazily on first use so that a model can be described on a host
    without CUDA, e.g. by ``KmerModel.load_from_hdf5``)."""

    def __init__(self, k, central_position, alphabet_size, mean, sigma, device=None):
        self._k = int(k)
        self._central_position = int(central_position)
        self._alphabet_size = int(alphabet_size)
        self.mean = np.ascontiguousarray(mean, dtype=np.float64)
        self.sigma = np.ascontiguousarray(sigma, dtype=np.float64)
        if self.mean.shape != self.sigma.shape or self.mean.size != self._alphabet_size ** self._k:
            raise ValueError('mean and sigma need alphabet_size**k entries')
        self._device = device
        self._handle = None

    def get_k(self):
        return self._k

    def get_central_position(self):
        return self._central_position

    def get_alphabet_size(self):
        return self._alphabet_size

    @property
    def device(self):
        if self._device is None:
            self._device = _current_device()
        return self._device

    @property
    def handle(self):
        if self._handle is None:
            lib = _cabi.require_device()
            h = lib.nvb_model_create(self._k, self._central_position, self._alphabet_size,
                                     _cabi.ptr(self.mean, ctypes.c_double), _cabi.ptr(self.sigma, ctypes.c_double),
                                     self.mean.size, self.device)
            if not h:
                raise NadavcaCudaError('nvb_model_create failed: ' + _cabi.last_error())
            self._handle = ctypes.c_void_p(h)
        return self._handle

    def __del__(self):
        if getattr(self, '_handle', None) is not None:
            try:
                _cabi.load().nvb_model_destroy(self._handle)
            except Exception:
                pass
            self._handle = None

    def get_expected_signal(self, reference, context_before, context_after):
        """KmerModel::GetExpectedSignal (kmer_model.cpp:32-42): list of the k-mer means along `reference`."""
        return self.get_expected_signal_batch([reference], [context_before], [context_after])[0].tolist()

    def get_expected_signal_batch(self, references, contexts_before, contexts_after):
        n = len(references)
        pack = ReadsPack([[]] * n, references, contexts_before, contexts_after, [[]] * n, 0, 0)
        out = np.zeros(pack.total_reference, dtype=np.float64)
        lib = _cabi.load()
        _cabi.check(lib.nvb_model_expected_signal(
            self.handle, n, pack.struct.reference, pack.struct.reference_off, pack.struct.context_before,
            pack.struct.context_before_off, pack.struct.context_after, pack.struct.context_after_off,
            _cabi.ptr(out, ctypes.c_double)), 'nvb_model_expected_signal')
        return [out[pack.reference_off[i]:pack.reference_off[i + 1]] for i in range(n)]


def _current_device():
    """Device ordinal for this process: LOCAL_RANK under torchrun, else torch's current device when torch is
    already in use, else 0."""
    import os
    import sys
    if 'LOCAL_RANK' in os.environ:
        return int(os.environ['LOCAL_RANK'])
    torch = sys.modules.get('torch')
    if torch is not None and torch.cuda.is_available():
        return torch.cuda.current_device()
    return 0


class Batch:
    """A batch of reads resident in HBM (nvb_batch_* of the C ABI)."""

    def __init__(self, kmer_model, signals, references, contexts_before, contexts_after, alignments, bandwidth,
                 min_event_length, workspace_limit=0, pack=None):
        self.model = kmer_model
        self.pack = pack if pack is not None else ReadsPack(signals, references, contexts_before, contexts_after,
                                                            alignments, bandwidth, min_event_length)
        self.lib = _cabi.require_device()
        h = self.lib.nvb_batch_create(kmer_model.handle, ctypes.byref(self.pack.struct))
        if not h:
            raise NadavcaCudaError('nvb_batch_create failed: ' + _cabi.last_error())
        self.handle = ctypes.c_void_p(h)
        if workspace_limit:
            _cabi.check(self.lib.nvb_batch_set_workspace_limit(self.handle, int(workspace_limit)),
                        'nvb_batch_set_workspace_limit')

    @classmethod
    def from_pack(cls, kmer_model, pack, workspace_limit=0):
        """Batch over an existing ReadsPack (e.g. ReadsPack.from_packed over pinned host arrays)."""
        return cls(kmer_model, None, None, None, None, None, pack.bandwidth, pack.min_event_length,
                   workspace_limit=workspace_limit, pack=pack)

    def close(self):
        if getattr(self, 'handle', None) is not None:
            self.lib.nvb_batch_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- inputs -----------------------------------------------------------------------------------------------
    @property
    def n_reads(self):
        return self.pack.n_reads

    def apply_splines(self, splines, stream=None):
        """Replace every read's resident signal x by spline(x); `splines` holds one FITPACK (t, c, k) tuple per read
        as returned by scipy.interpolate.splrep, or None to leave that read untouched."""
        degree = next((int(s[2]) for s in splines if s is not None), 3)
        off = np.zeros(self.n_reads + 1, dtype=np.int64)
        knots, coefs = [], []
        for i, s in enumerate(splines):
            n = 0
            if s is not None:
                if int(s[2]) != degree:
                    raise ValueError('all splines of a batch must have the same degree')
                n = len(s[0])
                knots.append(np.asarray(s[0], dtype=np.float64))
                coefs.append(np.asarray(s[1], dtype=np.float64)[:n])
            off[i + 1] = off[i] + n
        t = np.ascontiguousarray(np.concatenate(knots) if knots else np.zeros(0))
        c = np.ascontiguousarray(np.concatenate(coefs) if coefs else np.zeros(0))
        _cabi.check(self.lib.nvb_batch_apply_splines(self.handle, _cabi.ptr(t, ctypes.c_double),
                                                     _cabi.ptr(c, ctypes.c_double), _cabi.ptr(off, ctypes.c_int64),
                                                     degree, _stream(stream)), 'nvb_batch_apply_splines')

    def signals(self):
        """The resident signal values per read (after apply_splines)."""
        out = np.zeros(self.pack.total_signal, dtype=np.float64)
        _cabi.check(self.lib.nvb_batch_get_signal(self.handle, _cabi.ptr(out, ctypes.c_double)), 'nvb_batch_get_signal')
        off = self.pack.signal_off
        return [out[off[i]:off[i + 1]] for i in range(self.n_reads)]

    # -- kernels ----------------------------------------------------------------------------------------------
    def refine(self, model_transitions, stream=None):
        _cabi.check(self.lib.nvb_batch_refine(self.handle, int(bool(model_transitions)), _stream(stream)),
                    'nvb_batch_refine')

    def estimate(self, model_wobbling, stream=None):
        _cabi.check(self.lib.nvb_batch_estimate(self.handle, int(bool(model_wobbling)), _stream(stream)),
                    'nvb_batch_estimate')

    # -- results ----------------------------------------------------------------------------------------------
    def events(self):
        """-> (list of int32 (n,2) arrays or None for reads without a path, status array)."""
        ev = np.zeros((self.pack.total_reference, 2), dtype=np.int32)
        status = np.zeros(self.n_reads, dtype=np.int32)
        _cabi.check(self.lib.nvb_batch_get_events(self.handle, _cabi.ptr(ev, ctypes.c_int32),
                                                  _cabi.ptr(status, ctypes.c_int32)), 'nvb_batch_get_events')
        off = self.pack.reference_off
        return [ev[off[i]:off[i + 1]] if status[i] == 0 else None for i in range(self.n_reads)], status

    def log_likelihoods(self):
        a = self.model.get_alphabet_size()
        out = np.zeros((self.pack.total_reference, a), dtype=np.float64)
        status = np.zeros(self.n_reads, dtype=np.int32)
        _cabi.check(self.lib.nvb_batch_get_log_likelihoods(self.handle, _cabi.ptr(out, ctypes.c_double),
                                                           _cabi.ptr(status, ctypes.c_int32)),
                    'nvb_batch_get_log_likelihoods')
        off = self.pack.reference_off
        return [out[off[i]:off[i + 1]] for i in range(self.n_reads)], status

    def bands(self):
        cnt = self.pack.total_reference + self.n_reads
        starts = np.zeros(cnt, dtype=np.int32)
        ends = np.zeros(cnt, dtype=np.int32)
        _cabi.check(self.lib.nvb_batch_get_bands(self.handle, _cabi.ptr(starts, ctypes.c_int32),
                                                 _cabi.ptr(ends, ctypes.c_int32)), 'nvb_batch_get_bands')
        off = self.pack.reference_off
        return [(starts[off[i] + i:off[i + 1] + i + 1], ends[off[i] + i:off[i + 1] + i + 1])
                for i in range(self.n_reads)]

    def cell_counts(self, model_wobbling=True):
        """DP cell counts (SURVEY.md 8d): dict refine_transitions / refine_plain / estimate_fb / estimate_snp."""
        c = np.zeros(4, dtype=np.int64)
        _cabi.check(self.lib.nvb_batch_cell_counts(self.handle, int(bool(model_wobbling)),
                                                   _cabi.ptr(c, ctypes.c_int64)), 'nvb_batch_cell_counts')
        return {'refine_transitions': int(c[0]), 'refine_plain': int(c[1]), 'estimate_fb': int(c[2]),
                'estimate_snp': int(c[3])}

    def alignment_tables(self, start_in_signal, ref_start, ref_end, reverse):
        """(n,3) int64 tables of get_refined_alignment (estimator.py:187-195), None for reads without a path."""
        out = np.zeros((self.pack.total_reference, 3), dtype=np.int64)
        s = _cabi.as_array(start_in_signal, np.int64)
        a = _cabi.as_array(ref_start, np.int64)
        b = _cabi.as_array(ref_end, np.int64)
        r = _cabi.as_array(reverse, np.int32)
        _cabi.check(self.lib.nvb_batch_get_alignment_table(
            self.handle, _cabi.ptr(s, ctypes.c_int64), _cabi.ptr(a, ctypes.c_int64), _cabi.ptr(b, ctypes.c_int64),
            _cabi.ptr(r, ctypes.c_int32), _cabi.ptr(out, ctypes.c_int64)), 'nvb_batch_get_alignment_table')
        off = self.pack.reference_off
        return [out[off[i]:off[i + 1]] if (off[i + 1] > off[i] and out[off[i], 1] >= 0) else None
                for i in range(self.n_reads)]

    def event_means(self):
        """Per read: mean signal level of every refined event (bit-identical to numpy.mean over the event's samples);
        NaN rows for reads without a path."""
        out = np.zeros(self.pack.total_reference, dtype=np.float64)
        _cabi.check(self.lib.nvb_batch_event_means(self.handle, _cabi.ptr(out, ctypes.c_double)),
                    'nvb_batch_event_means')
        off = self.pack.reference_off
        return [out[off[i]:off[i + 1]] for i in range(self.n_reads)]

    def chunk_values(self, reverse, normalization_event_length, d_chunks, stream=None):
        """Normalised, strand-corrected chunk values into the device buffer `d_chunks` (a data pointer)."""
        r = _cabi.as_array(reverse, np.int32)
        _cabi.check(self.lib.nvb_batch_chunk_values(self.handle, _cabi.ptr(r, ctypes.c_int32),
                                                    float(normalization_event_length), ctypes.c_void_p(d_chunks),
                                                    _stream(stream)), 'nvb_batch_chunk_values')

    def scatter_add_rows(self, d_chunks, dest, d_rows, stream=None):
        """Add the chunks into consensus rows of 5 doubles [A, C, G, T, coverage] (one buffer, one collective)."""
        d = _cabi.as_array(dest, np.int64)
        _cabi.check(self.lib.nvb_batch_scatter_add_rows(self.handle, ctypes.c_void_p(d_chunks),
                                                        _cabi.ptr(d, ctypes.c_int64), ctypes.c_void_p(d_rows),
                                                        _stream(stream)), 'nvb_batch_scatter_add_rows')

    def debug_rows(self, read, plane, transitions=False):
        """Stored DP rows of one read after estimate() as log-probabilities (plane 0 prefix, 1 suffix)."""
        bs, be = self.bands()[read]
        w = be - bs + 1
        cells = int(2 * w.sum() - w[0] - w[-1]) if transitions else int(w.sum())
        out = np.zeros(cells, dtype=np.float64)
        _cabi.check(self.lib.nvb_batch_debug_rows(self.handle, int(read), int(plane),
                                                  _cabi.ptr(out, ctypes.c_double), cells), 'nvb_batch_debug_rows')
        return out

    @property
    def launch_count(self):
        return int(self.lib.nvb_batch_launch_count(self.handle))

    STAGES = ('rows', 'path', 'no_snp', 'snp')

    def enable_timing(self, on=True):
        _cabi.check(self.lib.nvb_batch_enable_timing(self.handle, int(on)), 'nvb_batch_enable_timing')

    def timing(self):
        """Per-stage device milliseconds / launches accumulated since the last call (CUDA events)."""
        ms = np.zeros(4, dtype=np.float64)
        cnt = np.zeros(4, dtype=np.int64)
        _cabi.check(self.lib.nvb_batch_get_timing(self.handle, _cabi.ptr(ms, ctypes.c_double),
                                                  _cabi.ptr(cnt, ctypes.c_int64)), 'nvb_batch_get_timing')
        return {name: (float(ms[i]), int(cnt[i])) for i, name in enumerate(self.STAGES)}


SWEEP_SCHEDULES = {None: 0, 'auto': 0, 'r': 1, 'rotate': 1, 's': 2, 'stripes': 2}


def set_sweep_schedule(schedule):
    """Force the schedule of the row sweeps ('r' rotating wavefront, 's' pipelined stripes, None automatic); returns
    the previous setting as an int.  Results do not depend on it."""
    return int(_cabi.load().nvb_set_sweep_schedule(SWEEP_SCHEDULES[schedule]))


def trim_memory(device=None):
    """Hand the library's cached device blocks back to the driver (nvb_trim_memory) and free the pinned staging
    buffers of the device normalisation."""
    from .read import trim_staging
    lib = _cabi.require_device()
    _cabi.check(lib.nvb_trim_memory(_current_device() if device is None else int(device)), 'nvb_trim_memory')
    trim_staging()


def measure_fp64_fma_rate(device=0):
    """FP64 FMA/s of the device (nvb_measure_fp64_fma_rate)."""
    lib = _cabi.require_device()
    out = ctypes.c_double(0)
    _cabi.check(lib.nvb_measure_fp64_fma_rate(int(device), ctypes.byref(out)), 'nvb_measure_fp64_fma_rate')
    return out.value


def _stream(stream):
    if stream is None:
        return ctypes.c_void_p(0)
    return ctypes.c_void_p(int(getattr(stream, 'cuda_stream', stream)))


def posterior_rows(device, d_rows, base_row, row_lo, row_hi, d_ref, d_group_off, n_groups, k, snp_prior, d_out_rows,
                   stream=None):
    """_compute_posterior for the global rows [row_lo, row_hi) from consensus rows of 5 doubles starting at global row
    `base_row`; writes rows of 5 = [P(A), P(C), P(G), P(T), coverage].  Enqueues only."""
    lib = _cabi.require_device()
    _cabi.check(lib.nvb_posterior_rows_d(int(device), ctypes.c_void_p(d_rows), int(base_row), int(row_lo), int(row_hi),
                                         ctypes.c_void_p(d_ref), ctypes.c_void_p(d_group_off), int(n_groups), int(k),
                                         float(snp_prior), ctypes.c_void_p(d_out_rows), _stream(stream)),
                'nvb_posterior_rows_d')


# ---- the two functions of the reference module, one read per call ------------------------------------------

def refine_alignment(signal, reference, context_before, context_after, approximate_alignment, bandwidth,
                     min_event_length, kmer_model, model_transitions):
    """dtwmodule.cpp:24-28: -> list of [event_start, event_end] per reference base, [] when there is no path."""
    with Batch(kmer_model, [signal], [reference], [context_before], [context_after], [approximate_alignment],
               bandwidth, min_event_length) as batch:
        batch.refine(model_transitions)
        events, _ = batch.events()
    return [] if events[0] is None else events[0].tolist()


def estimate_log_likelihoods(signal, reference, context_before, context_after, approximate_alignment, bandwidth,
                             min_event_length, kmer_model, model_wobbling):
    """dtwmodule.cpp:19-23: -> n x alphabet_size list of raw log-likelihoods."""
    with Batch(kmer_model, [signal], [reference], [context_before], [context_after], [approximate_alignment],
               bandwidth, min_event_length) as batch:
        batch.estimate(model_wobbling)
        ll, _ = batch.log_likelihoods()
    return ll[0].tolist()
