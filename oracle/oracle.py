"""CPU oracle for the nadavca hot path.   *** TEST INFRASTRUCTURE -- never imported by nadavca_b200 ***

Two back ends behind one interface:
  * ``port``  -- oracle/libnadavca_oracle.so, the plain-C restatement in oracle/nadavca_oracle.c (``extended``,
                 oracle/libnadavca_extended.so, restates its EstimateLogLikelihoods in extended precision, see
                 ``estimate_log_likelihoods_extended``);
  * ``ref``   -- oracle/_ref/dtw*.so, the UNMODIFIED reference C++ compiled by oracle/Makefile (present whenever
                 `make -C oracle ref` ran in a container that has /root/reference; the built file travels to the
                 GPU box).
plus a pure-Python restatement of the estimator glue (reference nadavca/estimator.py:45-57,111-156,187-236), written
to keep the reference's accumulation order.

Parity status: PINNED -- oracle/check_against_ref.py requires the port to be bit-identical to ``ref`` and the glue
restatement to be bit-identical to the reference's own estimator.py (imported from /root/reference under shims);
tests/golden/*.npz holds vectors produced from ``ref`` by oracle/make_golden.py.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this module.
"""
import ctypes
import glob
import importlib.util
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PORT_LIB = os.path.join(HERE, 'libnadavca_oracle.so')

ALPHABET = ['A', 'C', 'G', 'T']
NUM_COMPLEMENT = {0: 3, 1: 2, 2: 1, 3: 0}

_i32p = ctypes.POINTER(ctypes.c_int32)
_f64p = ctypes.POINTER(ctypes.c_double)
_i64p = ctypes.POINTER(ctypes.c_int64)


def build(which='all'):
    subprocess.run(['make', '-s', '-C', HERE, which], check=True)


def _load_port():
    if not os.path.exists(PORT_LIB) or os.path.getmtime(PORT_LIB) < os.path.getmtime(
            os.path.join(HERE, 'nadavca_oracle.c')):
        build('port')
    lib = ctypes.CDLL(PORT_LIB)
    lib.nvo_model_create.restype = ctypes.c_void_p
    lib.nvo_model_create.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, _f64p, _f64p, ctypes.c_int64]
    lib.nvo_model_destroy.argtypes = [ctypes.c_void_p]
    lib.nvo_expected_signal.argtypes = [ctypes.c_void_p, _i32p, ctypes.c_int, _i32p, ctypes.c_int, _i32p,
                                        ctypes.c_int, _f64p]
    lib.nvo_band_bounds.argtypes = [_i32p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, _i32p, _i32p]
    lib.nvo_refine_cells.restype = ctypes.c_int64
    lib.nvo_refine_cells.argtypes = [_i32p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    lib.nvo_refine_alignment.restype = ctypes.c_int
    lib.nvo_refine_alignment.argtypes = [ctypes.c_void_p, _f64p, ctypes.c_int, _i32p, ctypes.c_int, _i32p,
                                         ctypes.c_int, _i32p, ctypes.c_int, _i32p, ctypes.c_int, ctypes.c_int,
                                         ctypes.c_int, ctypes.c_int, _i32p, _f64p, _f64p, _i32p, _i32p]
    lib.nvo_estimate_log_likelihoods.argtypes = [ctypes.c_void_p, _f64p, ctypes.c_int, _i32p, ctypes.c_int, _i32p,
                                                 ctypes.c_int, _i32p, ctypes.c_int, _i32p, ctypes.c_int,
                                                 ctypes.c_int, ctypes.c_int, ctypes.c_int, _f64p, _f64p, _f64p]
    lib.nvo_count_cells.argtypes = [_i32p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                    ctypes.c_int, _i64p, _i64p, _i64p, _i64p]
    return lib


_port = None


def port_lib():
    global _port
    if _port is None:
        _port = _load_port()
    return _port


_ref = False


def ref_module():
    """The compiled reference module (oracle/_ref/dtw*.so) or None."""
    global _ref
    if _ref is False:
        found = glob.glob(os.path.join(HERE, '_ref', 'dtw*.so'))
        if not found and os.path.isdir('/root/reference/nadavca/dtw'):
            try:
                build('ref')
            except Exception:
                pass
            found = glob.glob(os.path.join(HERE, '_ref', 'dtw*.so'))
        if found:
            spec = importlib.util.spec_from_file_location('dtw', found[0])
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
            _ref = mod
        else:
            _ref = None
    return _ref


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32).reshape(-1)


def _p(a, t):
    return a.ctypes.data_as(ctypes.POINTER(t))


class OracleModel:
    """KmerModel for either back end (reference dtwmodule.cpp:12-18)."""

    def __init__(self, k, central_position, alphabet_size, mean, sigma, backend='port'):
        self.k, self.central_position, self.alphabet_size = int(k), int(central_position), int(alphabet_size)
        self.mean = np.ascontiguousarray(mean, dtype=np.float64)
        self.sigma = np.ascontiguousarray(sigma, dtype=np.float64)
        self.backend = backend
        if backend == 'ref':
            mod = ref_module()
            if mod is None:
                raise RuntimeError('oracle/_ref is not built')
            self.handle = mod.KmerModel(self.k, self.central_position, self.alphabet_size, self.mean.tolist(),
                                        self.sigma.tolist())
        else:
            lib = port_lib()
            self.handle = ctypes.c_void_p(lib.nvo_model_create(self.k, self.central_position, self.alphabet_size,
                                                               _p(self.mean, ctypes.c_double),
                                                               _p(self.sigma, ctypes.c_double), self.mean.size))

    def __del__(self):
        if getattr(self, 'backend', None) == 'port' and getattr(self, 'handle', None):
            try:
                port_lib().nvo_model_destroy(self.handle)
            except Exception:
                pass
            self.handle = None

    def get_k(self):
        return self.k

    def get_central_position(self):
        return self.central_position

    def get_expected_signal(self, reference, context_before, context_after):
        if self.backend == 'ref':
            return self.handle.get_expected_signal(list(map(int, reference)), list(map(int, context_before)),
                                                   list(map(int, context_after)))
        ref, cb, ca = _i32(reference), _i32(context_before), _i32(context_after)
        out = np.zeros(ref.size, dtype=np.float64)
        port_lib().nvo_expected_signal(self.handle, _p(ref, ctypes.c_int32), ref.size, _p(cb, ctypes.c_int32),
                                       cb.size, _p(ca, ctypes.c_int32), ca.size, _p(out, ctypes.c_double))
        return out.tolist()


def band_bounds(approximate_alignment, n_signal, n_ref, bandwidth):
    """ComputeBandStarts / ComputeBandEnds (dtw.cpp:7-35) -> (starts, ends) int32[n_ref+1]."""
    anc = _i32(approximate_alignment)
    bs = np.zeros(n_ref + 1, dtype=np.int32)
    be = np.zeros(n_ref + 1, dtype=np.int32)
    port_lib().nvo_band_bounds(_p(anc, ctypes.c_int32), anc.size // 2, n_signal, n_ref, bandwidth,
                               _p(bs, ctypes.c_int32), _p(be, ctypes.c_int32))
    return bs, be


def count_cells(approximate_alignment, n_signal, n_ref, bandwidth, k, central):
    anc = _i32(approximate_alignment)
    vals = [ctypes.c_int64(0) for _ in range(4)]
    port_lib().nvo_count_cells(_p(anc, ctypes.c_int32), anc.size // 2, n_signal, n_ref, bandwidth, k, central,
                               *[ctypes.byref(v) for v in vals])
    return {'refine_transitions': vals[0].value, 'refine_plain': vals[1].value, 'estimate_fb': vals[2].value,
            'estimate_snp': vals[3].value}


def refine_alignment(signal, reference, context_before, context_after, approximate_alignment, bandwidth,
                     min_event_length, kmer_model, model_transitions, debug=False):
    """RefineAlignment (dtw.cpp:133-228) -> list of [start, end] per base, [] for no path.  With debug=True (port
    only) also returns dict(prefix, suffix, bs, be) of the packed DP rows."""
    if kmer_model.backend == 'ref':
        return ref_module().refine_alignment(
            signal=np.asarray(signal, dtype=float).tolist(), reference=list(map(int, reference)),
            context_before=list(map(int, context_before)), context_after=list(map(int, context_after)),
            approximate_alignment=np.asarray(approximate_alignment, dtype=int).reshape(-1, 2).tolist(),
            bandwidth=int(bandwidth), min_event_length=int(min_event_length), kmer_model=kmer_model.handle,
            model_transitions=bool(model_transitions))
    lib = port_lib()
    sig = np.ascontiguousarray(signal, dtype=np.float64)
    ref, cb, ca, anc = _i32(reference), _i32(context_before), _i32(context_after), _i32(approximate_alignment)
    events = np.zeros((max(ref.size, 1), 2), dtype=np.int32)
    dbg = None
    args = [None, None, None, None]
    if debug:
        cells = lib.nvo_refine_cells(_p(anc, ctypes.c_int32), anc.size // 2, sig.size, ref.size, bandwidth,
                                     int(bool(model_transitions)))
        rows = 2 * ref.size if model_transitions else ref.size + 1
        dbg = {'prefix': np.zeros(cells), 'suffix': np.zeros(cells), 'bs': np.zeros(rows, dtype=np.int32),
               'be': np.zeros(rows, dtype=np.int32)}
        args = [_p(dbg['prefix'], ctypes.c_double), _p(dbg['suffix'], ctypes.c_double),
                _p(dbg['bs'], ctypes.c_int32), _p(dbg['be'], ctypes.c_int32)]
    ok = lib.nvo_refine_alignment(kmer_model.handle, _p(sig, ctypes.c_double), sig.size, _p(ref, ctypes.c_int32),
                                  ref.size, _p(cb, ctypes.c_int32), cb.size, _p(ca, ctypes.c_int32), ca.size,
                                  _p(anc, ctypes.c_int32), anc.size // 2, int(bandwidth), int(min_event_length),
                                  int(bool(model_transitions)), _p(events, ctypes.c_int32), *args)
    result = events[:ref.size].tolist() if ok else []
    return (result, dbg) if debug else result


def estimate_log_likelihoods(signal, reference, context_before, context_after, approximate_alignment, bandwidth,
                             min_event_length, kmer_model, model_wobbling, debug=False):
    """EstimateLogLikelihoods (dtw.cpp:37-131) -> n x alphabet list of lists.  debug=True (port only) also returns
    dict(prefix, suffix) with the packed stored rows 0..n."""
    if kmer_model.backend == 'ref':
        return ref_module().estimate_log_likelihoods(
            signal=np.asarray(signal, dtype=float).tolist(), reference=list(map(int, reference)),
            context_before=list(map(int, context_before)), context_after=list(map(int, context_after)),
            approximate_alignment=np.asarray(approximate_alignment, dtype=int).reshape(-1, 2).tolist(),
            bandwidth=int(bandwidth), min_event_length=int(min_event_length), kmer_model=kmer_model.handle,
            model_wobbling=bool(model_wobbling))
    sig = np.ascontiguousarray(signal, dtype=np.float64)
    ref, cb, ca, anc = _i32(reference), _i32(context_before), _i32(context_after), _i32(approximate_alignment)
    out = np.zeros((ref.size, kmer_model.alphabet_size), dtype=np.float64)
    dbg, args = None, [None, None]
    if debug:
        bs, be = band_bounds(approximate_alignment, sig.size, ref.size, bandwidth)
        cells = int((be - bs + 1).sum())
        dbg = {'prefix': np.zeros(cells), 'suffix': np.zeros(cells), 'bs': bs, 'be': be}
        args = [_p(dbg['prefix'], ctypes.c_double), _p(dbg['suffix'], ctypes.c_double)]
    port_lib().nvo_estimate_log_likelihoods(
        kmer_model.handle, _p(sig, ctypes.c_double), sig.size, _p(ref, ctypes.c_int32), ref.size,
        _p(cb, ctypes.c_int32), cb.size, _p(ca, ctypes.c_int32), ca.size, _p(anc, ctypes.c_int32), anc.size // 2,
        int(bandwidth), int(min_event_length), int(bool(model_wobbling)), _p(out, ctypes.c_double), *args)
    return (out.tolist(), dbg) if debug else out.tolist()


# ---- extended-precision EstimateLogLikelihoods (oracle/nadavca_extended.c) -----------------------------------------

EXT_LIB = os.path.join(HERE, 'libnadavca_extended.so')
_ext = None


def extended_lib():
    global _ext
    if _ext is None:
        if not os.path.exists(EXT_LIB) or os.path.getmtime(EXT_LIB) < os.path.getmtime(
                os.path.join(HERE, 'nadavca_extended.c')):
            build('extended')
        lib = ctypes.CDLL(EXT_LIB)
        lib.nvx_model_create.restype = ctypes.c_void_p
        lib.nvx_model_create.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, _f64p, _f64p, ctypes.c_int64]
        lib.nvx_model_destroy.argtypes = [ctypes.c_void_p]
        lib.nvx_estimate_log_likelihoods.argtypes = [ctypes.c_void_p, _f64p, ctypes.c_int, _i32p, ctypes.c_int, _i32p,
                                                     ctypes.c_int, _i32p, ctypes.c_int, _i32p, ctypes.c_int,
                                                     ctypes.c_int, ctypes.c_int, ctypes.c_int, _f64p, _f64p, _f64p,
                                                     _f64p, _f64p]
        _ext = lib
    return _ext


class ExtendedModel:
    """The model tables of nadavca_extended.c (the reference's double ac / mc, kmer_model.cpp:10-13)."""

    def __init__(self, k, central_position, alphabet_size, mean, sigma):
        self.k, self.central_position, self.alphabet_size = int(k), int(central_position), int(alphabet_size)
        self.mean = np.ascontiguousarray(mean, dtype=np.float64)
        self.sigma = np.ascontiguousarray(sigma, dtype=np.float64)
        self.handle = ctypes.c_void_p(extended_lib().nvx_model_create(
            self.k, self.central_position, self.alphabet_size, _p(self.mean, ctypes.c_double),
            _p(self.sigma, ctypes.c_double), self.mean.size))

    def __del__(self):
        if getattr(self, 'handle', None):
            try:
                extended_lib().nvx_model_destroy(self.handle)
            except Exception:
                pass
            self.handle = None


def estimate_log_likelihoods_extended(signal, reference, context_before, context_after, approximate_alignment,
                                      bandwidth, min_event_length, model, model_wobbling, rows=False):
    """EstimateLogLikelihoods (dtw.cpp:37-131) in extended precision -> dict with
      ll     (n, alphabet) log-likelihoods, each rounded once to double;
      ratio  (n, alphabet) log(L[i][b] / L[i][ref_i]), rounded once (0 on the reference base);
    and with rows=True also bs, be (band bounds), prefix, suffix (stored rows 0..n packed, as log values) and row_dev
    (n+1: sum_c P[j][c] S[j][c] relative to row n's, minus 1; the same total for every row in plain mode)."""
    sig = np.ascontiguousarray(signal, dtype=np.float64)
    ref, cb, ca, anc = _i32(reference), _i32(context_before), _i32(context_after), _i32(approximate_alignment)
    a = model.alphabet_size
    out = {'ll': np.zeros((ref.size, a)), 'ratio': np.zeros((ref.size, a))}
    extra = [None, None, None]
    if rows:
        bs, be = band_bounds(approximate_alignment, sig.size, ref.size, bandwidth)
        cells = int(np.maximum(be.astype(np.int64) - bs + 1, 0).sum())
        out.update(bs=bs, be=be, prefix=np.zeros(cells), suffix=np.zeros(cells), row_dev=np.zeros(ref.size + 1))
        extra = [_p(out['prefix'], ctypes.c_double), _p(out['suffix'], ctypes.c_double),
                 _p(out['row_dev'], ctypes.c_double)]
    extended_lib().nvx_estimate_log_likelihoods(
        model.handle, _p(sig, ctypes.c_double), sig.size, _p(ref, ctypes.c_int32), ref.size, _p(cb, ctypes.c_int32),
        cb.size, _p(ca, ctypes.c_int32), ca.size, _p(anc, ctypes.c_int32), anc.size // 2, int(bandwidth),
        int(min_event_length), int(bool(model_wobbling)), _p(out['ll'], ctypes.c_double),
        _p(out['ratio'], ctypes.c_double), *extra)
    return out


# ---- estimator glue, restated (reference nadavca/estimator.py) -----------------------------------------------

def to_numerical(sequence):
    inv = {c: i for i, c in enumerate(ALPHABET)}
    return np.array([inv[b] for b in sequence], dtype=int)


def reverse_complement(sequence):
    comp = {'A': 'T', 'C': 'G', 'G': 'C', 'T': 'A'}
    res = [comp[x] for x in sequence]
    res.reverse()
    return np.array(res)


class OracleChunk:
    def __init__(self, start, end, values, coverage=None):
        self.start, self.end, self.values = start, end, values
        self.coverage = np.ones(end - start, dtype=int) if coverage is None else coverage

    def __lt__(self, other):
        if self.start == other.start:
            return self.end < other.end
        return self.start < other.start


class OracleEstimator:
    """Restatement of ProbabilityEstimator (estimator.py:33-236) driving either oracle back end."""

    def __init__(self, kmer_model, aligner, config):
        self.kmer_model = kmer_model
        self.aligner = aligner
        self.cfg = config

    def _context(self, read, read_sequence_range):  # estimator.py:49-57
        start, end = read_sequence_range
        k, cp = self.kmer_model.get_k(), self.kmer_model.get_central_position()
        return to_numerical(read.sequence[start - cp:start]), to_numerical(read.sequence[end:end + k - cp - 1])

    def get_refined_alignment(self, read):  # estimator.py:158-196
        c = self.cfg
        apx = self.aligner.get_signal_alignment(read, c['bandwidth'])
        if apx is None:
            return None
        s_ref, e_ref = apx.reference_range
        ref_part = to_numerical(apx.reference_part)
        s_sig, e_sig = apx.signal_range
        signal = read.normalized_signal[s_sig:e_sig]
        cb, ca = self._context(read, apx.read_sequence_range)
        refined = refine_alignment(signal, ref_part, cb, ca, apx.alignment, c['bandwidth'], c['min_event_length'],
                                   self.kmer_model, c['model_transitions'])
        if len(refined) == 0:
            return None
        result = np.zeros((len(refined), 3), dtype=int)
        for pos, (ev_s, ev_e) in enumerate(refined):
            result[pos][1] = ev_s + s_sig
            result[pos][2] = ev_e + s_sig
            result[pos][0] = e_ref - pos - 1 if apx.reverse_complement else s_ref + pos
        return apx, result

    def estimate_log_likelihoods(self, reference, read, return_raw=False):  # estimator.py:59-121
        c = self.cfg
        apx = self.aligner.get_signal_alignment(read, c['bandwidth'])
        if apx is None:
            return None
        s_ref, e_ref = apx.reference_range
        ref_part = reference[s_ref:e_ref]
        if apx.reverse_complement:
            ref_part = reverse_complement(ref_part)
        ref_part = to_numerical(ref_part)
        s_sig, e_sig = apx.signal_range
        signal = read.normalized_signal[s_sig:e_sig]
        cb, ca = self._context(read, apx.read_sequence_range)
        if c['tweak_signal_normalization']:
            refined = refine_alignment(signal, ref_part, cb, ca, apx.alignment, c['bandwidth'],
                                       c['min_event_length'], self.kmer_model, False)
            refined = np.array(refined) + s_sig
            expected = self.kmer_model.get_expected_signal(ref_part, cb, ca)
            read.tweak_signal_normalization(refined, expected)
            signal = read.tweaked_normalized_signal[s_sig:e_sig]
        ll = np.array(estimate_log_likelihoods(signal, ref_part, cb, ca, apx.alignment, c['bandwidth'],
                                               c['min_event_length'], self.kmer_model, c['model_wobbling']))
        raw = ll
        ll = (ll - ll[0][ref_part[0]]) / c['normalization_event_length']  # estimator.py:45-47
        if apx.reverse_complement:  # estimator.py:114-119
            comp = np.zeros(ll.shape, dtype=float)
            for i, line in enumerate(ll):
                for j in range(4):
                    comp[i][j] = line[NUM_COMPLEMENT[j]]
            ll = np.flipud(comp)
        chunk = OracleChunk(s_ref, e_ref, ll)
        return (chunk, raw) if return_raw else chunk

    def corrected_priors(self, context_positions):  # estimator.py:123-129
        c = 3
        p_1 = 1 - self.cfg['snp_prior_probability']
        p_2 = self.cfg['snp_prior_probability'] / c
        snp = 1 / (p_1 / p_2 + (1 - context_positions) * c)
        return snp, 1 - snp * c

    def compute_posterior(self, log_likelihoods, reference):  # estimator.py:131-156
        prob = np.zeros(log_likelihoods.shape, dtype=float)
        k = self.kmer_model.get_k()
        for i in range(len(prob)):
            cs, ce = max(0, i - k + 1), min(i + k, len(prob))
            mx = np.max(log_likelihoods[cs:ce])
            snp, nonsnp = self.corrected_priors(ce - cs - 1)
            for j, base in enumerate(ALPHABET):
                prior = snp if base != reference[i] else nonsnp
                prob[i][j] = np.exp(log_likelihoods[i][j] - mx) * prior
                if base == reference[i]:
                    for i2 in range(cs, ce):
                        if i2 == i:
                            continue
                        for j2, base2 in enumerate(ALPHABET):
                            if base2 == reference[i2]:
                                continue
                            prob[i][j] += np.exp(log_likelihoods[i2][j2] - mx) * snp
            prob[i] /= sum(prob[i])
        return prob

    def estimate_probabilities(self, reference, reads):  # estimator.py:199-236
        chunks = []
        for read in reads:
            chunk = self.estimate_log_likelihoods(reference, read)
            if chunk is not None:
                chunks.append(chunk)
        chunks.sort()
        groups, cur, cs, ce = [], [], None, None
        for i, chunk in enumerate(chunks):
            if cs is None:
                cs, ce = chunk.start, chunk.end
            cur.append(chunk)
            ce = max(ce, chunk.end)
            if i + 1 >= len(chunks) or chunks[i + 1].start >= ce:
                groups.append(((cs, ce), cur))
                cur, cs, ce = [], None, None
        result = []
        for (start, end), members in groups:
            coverage = np.zeros(end - start, dtype=int)
            ll = np.zeros((end - start, 4), dtype=float)
            for chunk in members:
                coverage[chunk.start - start:chunk.end - start] += 1
                ll[chunk.start - start:chunk.end - start] += chunk.values
            result.append(OracleChunk(start, end, self.compute_posterior(ll, reference[start:end]), coverage))
        return result
