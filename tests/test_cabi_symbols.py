"""CPU suite, part 3: the C-ABI shared library builds for sm_100a, loads without a GPU, exports every symbol that
include/nadavca_b200.h declares, and fails LOUDLY (no CPU fallback) when no CUDA device is present."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT

HEADER = os.path.join(ROOT, 'include', 'nadavca_b200.h')


def declared_functions():
    text = open(HEADER).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    text = re.sub(r'typedef struct nvb_reads \{.*?\} nvb_reads;', '', text, flags=re.S)
    text = re.sub(r'typedef struct nvb_hits \{.*?\} nvb_hits;', '', text, flags=re.S)
    names = re.findall(r'\b(nvb_[a-z0-9_]+)\s*\(', text)
    return sorted(set(names))


def test_header_declares_the_boundary():
    names = declared_functions()
    for must in ('nvb_model_create', 'nvb_model_expected_signal', 'nvb_refine_alignment_batch',
                 'nvb_estimate_log_likelihoods_batch', 'nvb_batch_create', 'nvb_batch_refine', 'nvb_batch_estimate',
                 'nvb_posterior_rows_d', 'nvb_batch_scatter_add_rows', 'nvb_last_error'):
        assert must in names
    # every entry point cites the reference interface it replaces
    text = open(HEADER).read()
    for cite in ('dtwmodule.cpp:10-29', 'dtwmodule.cpp:19-23', 'dtwmodule.cpp:24-28', 'kmer_model.cpp:32-42',
                 'dtw.cpp:7-35', 'estimator.py:187-195', 'estimator.py:123-156', 'estimator.py:226-231'):
        assert cite in text, cite


def test_header_compiles_as_plain_c(tmp_path):
    """No torch / CUDA / C++ types in the signatures: the header must compile as C99 on its own."""
    src = tmp_path / 'use.c'
    src.write_text('#include "nadavca_b200.h"\nint main(void) { nvb_reads r; (void)r; return NVB_OK; }\n')
    subprocess.run(['gcc', '-std=c99', '-Wall', '-Werror', '-I', os.path.join(ROOT, 'include'), '-c', str(src),
                    '-o', str(tmp_path / 'use.o')], check=True)


def test_library_exports_every_declared_symbol(lib_built):
    from nadavca_b200 import _cabi
    lib = ctypes.CDLL(lib_built)
    names = declared_functions()
    assert len(names) >= 30
    for name in names:
        assert hasattr(lib, name), 'libnadavca_b200.so does not export ' + name
    # the ctypes table binds exactly the declared functions
    assert sorted(_cabi.SIGNATURES) == names
    bound = _cabi.load()
    assert bound.nvb_abi_version() == 1
    assert isinstance(bound.nvb_device_count(), int)


def test_library_is_sm100a_only(lib_built):
    out = subprocess.run(['cuobjdump', '--list-elf', lib_built], capture_output=True, text=True).stdout
    archs = set(re.findall(r'sm_\d+a?', out))
    assert archs == {'sm_100a'}, archs


def test_compute_fails_loudly_without_gpu(lib_built):
    """No CPU fallback: without a CUDA device every compute entry point raises."""
    from nadavca_b200 import _cabi, dtw
    if _cabi.load().nvb_device_count() > 0:
        pytest.skip('a CUDA device is present')
    km = dtw.KmerModel(1, 0, 4, [0, 1, 2, 3], [.5] * 4)
    assert km.get_k() == 1 and km.get_central_position() == 0  # describing a model needs no device
    with pytest.raises(dtw.NadavcaCudaError):
        km.get_expected_signal([0, 1], [], [])
    with pytest.raises(dtw.NadavcaCudaError):
        dtw.refine_alignment(signal=[0.1, 0.2, 0.3], reference=[0], context_before=[], context_after=[],
                             approximate_alignment=[[0, 0]], bandwidth=2, min_event_length=1, kmer_model=km,
                             model_transitions=True)
    with pytest.raises(dtw.NadavcaCudaError):
        dtw.estimate_log_likelihoods(signal=[0.1, 0.2, 0.3], reference=[0], context_before=[], context_after=[],
                                     approximate_alignment=[[0, 0]], bandwidth=2, min_event_length=1, kmer_model=km,
                                     model_wobbling=True)
    with pytest.raises(dtw.NadavcaCudaError):
        dtw.measure_fp64_fma_rate(0)
    # direct C call: NULL handle + error string
    lib = _cabi.load()
    mean = np.zeros(4)
    h = lib.nvb_model_create(1, 0, 4, _cabi.ptr(mean, ctypes.c_double), _cabi.ptr(mean + 1, ctypes.c_double), 4, 0)
    assert not h
    assert 'no CPU fallback' in _cabi.last_error()


def test_model_argument_validation(lib_built):
    from nadavca_b200 import _cabi, dtw
    with pytest.raises(ValueError):
        dtw.KmerModel(2, 0, 4, [0, 1, 2, 3], [.5] * 4)  # needs 16 entries
    lib = _cabi.load()
    mean = np.zeros(4)
    assert not lib.nvb_model_create(1, 3, 4, _cabi.ptr(mean, ctypes.c_double), _cabi.ptr(mean, ctypes.c_double), 4, 0)
    assert 'bad arguments' in _cabi.last_error()
    assert not lib.nvb_model_create(2, 0, 4, _cabi.ptr(mean, ctypes.c_double), _cabi.ptr(mean, ctypes.c_double), 4, 0)
    assert 'expected 16' in _cabi.last_error()
    assert lib.nvb_batch_refine(None, 1, None) == -1
    assert lib.nvb_batch_get_events(None, None, None) == -1
