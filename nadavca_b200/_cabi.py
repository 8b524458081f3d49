"""ctypes binding of libnadavca_b200.so (the C ABI declared in include/nadavca_b200.h).

The library is built in-tree by ``nadavca_b200.build``.  Nothing here computes on the CPU: when the shared library
or a CUDA device is missing, the compute entry points raise ``NadavcaCudaError``.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libnadavca_b200.so')

NVB_READ_OK, NVB_READ_NO_PATH, NVB_READ_BAD_BAND = 0, 1, 2


class NadavcaCudaError(RuntimeError):
    pass


c_i32p = ctypes.POINTER(ctypes.c_int32)
c_i64p = ctypes.POINTER(ctypes.c_int64)
c_f64p = ctypes.POINTER(ctypes.c_double)
c_i8p = ctypes.POINTER(ctypes.c_int8)


class NvbReads(ctypes.Structure):
    _fields_ = [
        ('n_reads', ctypes.c_int32),
        ('signal', c_f64p), ('signal_off', c_i64p),
        ('reference', c_i32p), ('reference_off', c_i64p),
        ('context_before', c_i32p), ('context_before_off', c_i64p),
        ('context_after', c_i32p), ('context_after_off', c_i64p),
        ('anchors', c_i32p), ('anchor_off', c_i64p),
        ('bandwidth', ctypes.c_int32), ('min_event_length', ctypes.c_int32),
    ]


class NvbHits(ctypes.Structure):
    _fields_ = [
        ('n_reads', ctypes.c_int32),
        ('cigar_len', c_i32p), ('cigar_op', c_i8p), ('cigar_off', c_i64p),
        ('mapped_position', c_i64p), ('reverse', c_i32p),
        ('read_sequence', c_i8p), ('base_to_sample', c_i32p), ('read_off', c_i64p),
        ('n_signal', c_i32p),
        ('d_genome', ctypes.c_void_p), ('genome_length', ctypes.c_int64), ('bandwidth', ctypes.c_int32),
    ]


# name -> (restype, argtypes); every symbol declared in include/nadavca_b200.h
SIGNATURES = {
    'nvb_abi_version': (ctypes.c_int, []),
    'nvb_last_error': (ctypes.c_char_p, []),
    'nvb_device_count': (ctypes.c_int, []),
    'nvb_trim_memory': (ctypes.c_int, [ctypes.c_int]),
    'nvb_set_sweep_schedule': (ctypes.c_int, [ctypes.c_int]),
    'nvb_model_create': (ctypes.c_void_p, [ctypes.c_int, ctypes.c_int, ctypes.c_int, c_f64p, c_f64p, ctypes.c_int64,
                                           ctypes.c_int]),
    'nvb_model_destroy': (None, [ctypes.c_void_p]),
    'nvb_model_k': (ctypes.c_int, [ctypes.c_void_p]),
    'nvb_model_central_position': (ctypes.c_int, [ctypes.c_void_p]),
    'nvb_model_alphabet_size': (ctypes.c_int, [ctypes.c_void_p]),
    'nvb_model_workspace_bytes': (ctypes.c_int64, [ctypes.c_void_p]),
    'nvb_model_expected_signal': (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32, c_i32p, c_i64p, c_i32p, c_i64p,
                                                 c_i32p, c_i64p, c_f64p]),
    'nvb_refine_alignment_batch': (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(NvbReads), ctypes.c_int, c_i32p,
                                                  c_i32p]),
    'nvb_estimate_log_likelihoods_batch': (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(NvbReads), ctypes.c_int,
                                                          c_f64p, c_i32p]),
    'nvb_batch_create': (ctypes.c_void_p, [ctypes.c_void_p, ctypes.POINTER(NvbReads)]),
    'nvb_batch_destroy': (None, [ctypes.c_void_p]),
    'nvb_batch_set_workspace_limit': (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64]),
    'nvb_batch_refine': (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]),
    'nvb_batch_estimate': (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]),
    'nvb_batch_get_events': (ctypes.c_int, [ctypes.c_void_p, c_i32p, c_i32p]),
    'nvb_batch_get_log_likelihoods': (ctypes.c_int, [ctypes.c_void_p, c_f64p, c_i32p]),
    'nvb_batch_get_bands': (ctypes.c_int, [ctypes.c_void_p, c_i32p, c_i32p]),
    'nvb_batch_cell_counts': (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, c_i64p]),
    'nvb_batch_launch_count': (ctypes.c_int64, [ctypes.c_void_p]),
    'nvb_batch_debug_rows': (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, c_f64p, ctypes.c_int64]),
    'nvb_batch_enable_timing': (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    'nvb_batch_get_timing': (ctypes.c_int, [ctypes.c_void_p, c_f64p, c_i64p]),
    'nvb_measure_fp64_fma_rate': (ctypes.c_int, [ctypes.c_int, c_f64p]),
    'nvb_batch_get_alignment_table': (ctypes.c_int, [ctypes.c_void_p, c_i64p, c_i64p, c_i64p, c_i32p, c_i64p]),
    'nvb_batch_event_means': (ctypes.c_int, [ctypes.c_void_p, c_f64p]),
    'nvb_batch_apply_splines': (ctypes.c_int, [ctypes.c_void_p, c_f64p, c_f64p, c_i64p, ctypes.c_int, ctypes.c_void_p]),
    'nvb_batch_get_signal': (ctypes.c_int, [ctypes.c_void_p, c_f64p]),
    'nvb_batch_chunk_values': (ctypes.c_int, [ctypes.c_void_p, c_i32p, ctypes.c_double, ctypes.c_void_p,
                                              ctypes.c_void_p]),
    'nvb_signal_anchors_batch': (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(NvbHits), c_i32p, c_i64p,
                                                ctypes.c_void_p]),
    'nvb_radix_histogram_d': (ctypes.c_int, [ctypes.c_int, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int,
                                             ctypes.c_double, ctypes.c_uint64, ctypes.c_int, ctypes.c_void_p,
                                             ctypes.c_void_p]),
    'nvb_normalize_each': (ctypes.c_int, [ctypes.c_int, c_f64p, c_i64p, ctypes.c_int32, ctypes.c_double,
                                          ctypes.c_double, c_f64p, c_f64p, ctypes.c_void_p]),
    'nvb_normalize_clip_d': (ctypes.c_int, [ctypes.c_int, ctypes.c_void_p, ctypes.c_int64, ctypes.c_double,
                                            ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_void_p,
                                            ctypes.c_void_p]),
    'nvb_batch_scatter_add_rows': (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, c_i64p, ctypes.c_void_p,
                                                  ctypes.c_void_p]),
    'nvb_posterior_rows_d': (ctypes.c_int, [ctypes.c_int, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64,
                                            ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32,
                                            ctypes.c_int, ctypes.c_double, ctypes.c_void_p, ctypes.c_void_p]),
}

_lib = None


def load():
    """Load the shared library (no CUDA call is made)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NadavcaCudaError(
                '{} not found: build it with `python -m nadavca_b200.build` (there is no CPU fallback)'.format(LIB_PATH))
        lib = ctypes.CDLL(LIB_PATH)
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = lib
    return _lib


def last_error():
    return load().nvb_last_error().decode('utf-8', 'replace')


def check(rc, what):
    if rc != 0:
        raise NadavcaCudaError('{} failed ({}): {}'.format(what, rc, last_error()))


def require_device():
    lib = load()
    if lib.nvb_device_count() <= 0:
        raise NadavcaCudaError('no CUDA device available: nadavca_b200 has no CPU fallback')
    return lib


def ptr(arr, ctype):
    return arr.ctypes.data_as(ctypes.POINTER(ctype))


def as_array(values, dtype):
    return np.ascontiguousarray(values, dtype=dtype)


class ReadsPack:
    """Host-side CSR packing of a list of per-read arguments; keeps the numpy arrays alive for the C struct."""

    def __init__(self, signals, references, contexts_before, contexts_after, alignments, bandwidth,
                 min_event_length):
        n = len(signals)
        if not (len(references) == len(contexts_before) == len(contexts_after) == len(alignments) == n):
            raise ValueError('per-read argument lists differ in length')

        def pack(items, dtype, width=1):
            arrs = [np.asarray(x, dtype=dtype).reshape(-1) for x in items]
            off = np.zeros(n + 1, dtype=np.int64)
            if n:
                off[1:] = np.cumsum([a.size // width for a in arrs])
            flat = np.concatenate(arrs) if n and off[-1] > 0 else np.zeros(0, dtype=dtype)
            return np.ascontiguousarray(flat, dtype=dtype), off

        self.n_reads = n
        self.signal, self.signal_off = pack(signals, np.float64)
        self.reference, self.reference_off = pack(references, np.int32)
        self.context_before, self.context_before_off = pack(contexts_before, np.int32)
        self.context_after, self.context_after_off = pack(contexts_after, np.int32)
        for a in alignments:
            a = np.asarray(a)
            if a.size and (a.ndim != 2 or a.shape[1] != 2):
                raise ValueError('approximate_alignment must be a sequence of (signal index, reference index) pairs')
        self.anchors, self.anchor_off = pack(alignments, np.int32, width=2)
        self.bandwidth = int(bandwidth)
        self.min_event_length = int(min_event_length)
        self._make_struct()

    @classmethod
    def from_packed(cls, signal, signal_off, reference, reference_off, context_before, context_before_off,
                    context_after, context_after_off, anchors, anchor_off, bandwidth, min_event_length):
        """Wrap already packed CSR arrays WITHOUT copying (they may live in pinned host memory); dtypes must be
        float64 / int32 / int64 as in the C struct."""
        self = cls.__new__(cls)
        self.n_reads = len(signal_off) - 1
        for name, arr, dtype in (('signal', signal, np.float64), ('signal_off', signal_off, np.int64),
                                 ('reference', reference, np.int32), ('reference_off', reference_off, np.int64),
                                 ('context_before', context_before, np.int32),
                                 ('context_before_off', context_before_off, np.int64),
                                 ('context_after', context_after, np.int32),
                                 ('context_after_off', context_after_off, np.int64),
                                 ('anchors', anchors, np.int32), ('anchor_off', anchor_off, np.int64)):
            if arr.dtype != dtype or not arr.flags['C_CONTIGUOUS']:
                raise ValueError('{} must be a contiguous {} array'.format(name, np.dtype(dtype).name))
            setattr(self, name, arr)
        self.bandwidth = int(bandwidth)
        self.min_event_length = int(min_event_length)
        self._make_struct()
        return self

    def _make_struct(self):
        n = self.n_reads
        self.struct = NvbReads(
            n, ptr(self.signal, ctypes.c_double), ptr(self.signal_off, ctypes.c_int64),
            ptr(self.reference, ctypes.c_int32), ptr(self.reference_off, ctypes.c_int64),
            ptr(self.context_before, ctypes.c_int32), ptr(self.context_before_off, ctypes.c_int64),
            ptr(self.context_after, ctypes.c_int32), ptr(self.context_after_off, ctypes.c_int64),
            ptr(self.anchors, ctypes.c_int32), ptr(self.anchor_off, ctypes.c_int64),
            self.bandwidth, self.min_event_length)

    @property
    def total_reference(self):
        return int(self.reference_off[-1])

    @property
    def total_signal(self):
        return int(self.signal_off[-1])
