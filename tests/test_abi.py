"""CPU: the C-ABI library loads and exports every symbol include/re2nn_b200.h declares."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, 'include', 're2nn_b200.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(re2nn_[a-z0-9_]+)\s*\(', src)))


def test_header_symbols_exported():
    from re2nn_seq_b200 import _lib
    names = _declared()
    assert len(names) >= 15
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), 'missing export: ' + n
    assert sorted(_lib.SYMBOLS.keys()) == names          # the ctypes binding covers the whole header


def test_version_and_error_channel():
    from re2nn_seq_b200 import _lib
    assert _lib.fn["re2nn_abi_version"]() == 4
    # argument validation happens before any CUDA call, so this is safe without a GPU
    rc = _lib.fn['re2nn_decompose_recurrence'](None, None)
    assert rc != 0
    assert b'null args' in _lib.fn['re2nn_last_error']()
    assert _lib.fn['re2nn_debug_set_viterbi_seqs'](4) != 0
    assert b'expected 0, 1 or 2' in _lib.fn['re2nn_last_error']()
    # a precision outside the enum is refused before anything is launched or sized from it (dummy pointers, ample ws)
    bad, p, ws = 7, ctypes.c_void_p(0x1000), 1 << 40
    a = _lib.RecurrenceArgs()
    a.B, a.Lpad, a.L, a.S, a.R, a.precision = 4, 8, 8, 32, 16, bad
    for f in ('x', 'lengths', 'vtab', 'S1', 'S2', 'W', 'o', 'h0', 'hT', 'alpha', 'beta', 'ws'):
        setattr(a, f, p)
    a.ws_bytes = ws
    calls = {
        're2nn_label_scores': lambda f: f(p, p, p, 4, 8, 32, p, 5, None, None, 0, bad, p, p, ws, None),
        're2nn_label_scores_ab': lambda f: f(p, 4, 8, 32, p, 5, None, None, bad, p, p, ws, None),
        're2nn_gemm_nt': lambda f: f(bad, p, p, 16, 16, 16, p, p, ws, None),
        're2nn_decompose_weight_prep': lambda f: f(ctypes.byref(a), p, None),
        're2nn_decompose_recurrence': lambda f: f(ctypes.byref(a), None),
    }
    for name, call in calls.items():
        assert call(_lib.fn[name]) != 0, name
        assert b'unknown precision' in _lib.fn['re2nn_last_error'](), (name, _lib.fn['re2nn_last_error']())


def test_no_oracle_in_product():
    """The product package must not import or reference the oracle (no CPU fallback)."""
    pkg = os.path.join(ROOT, 're2nn_seq_b200')
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                txt = open(os.path.join(root, f)).read()
                assert 'import oracle' not in txt and 'from oracle' not in txt and 're2nn_oracle' not in txt, f


def test_torch_library_registration():
    """TORCH_LIBRARY(re2nn, ...): the hot-path ops are registered PyTorch custom ops with CUDA kernels only
    (csrc/torch_ops.cpp); calling one with CPU tensors fails loudly instead of falling back."""
    import pytest
    import torch
    from re2nn_seq_b200 import _lib
    assert int(_lib.tops.abi_version()) == 4
    for name in ('ifst_decompose_forward', 'ifst_onehot_forward', 'label_scores', 'argmax_decode', 'crf_viterbi', 'crf_nll',
                 'crf_nll_backward'):
        assert hasattr(_lib.tops, name), name
        schema = str(getattr(_lib.tops, name).default._schema)
        assert schema.startswith('re2nn::' + name + '('), schema
    f = torch.zeros(2, 3, 5)
    with pytest.raises((RuntimeError, NotImplementedError)):       # no CPU implementation is registered
        _lib.tops.crf_viterbi(f, torch.zeros(5, 5), torch.tensor([3, 2]), None, 0, -1, 0.0, 0, False, True, None)
