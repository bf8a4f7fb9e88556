"""GPU: the path queries of the decompose recurrence against what a call launches.  bench.py reports
re2nn_decompose_recurrence_launches as gpu_launches and picks its roofline class and its fused leg from
re2nn_decompose_recurrence_resident / _fuses; here each query is checked against the kernels torch.profiler sees."""
import ctypes as C
import re

import pytest
import torch
from torch.autograd import DeviceType
from torch.profiler import ProfilerActivity, profile

pytestmark = pytest.mark.gpu

B, L, V = 200, 6, 50
# precision, S, R, farnn, save_for_backward, full_pad, ab_out, wprep
CASES = [
    ('fp32', 96, 48, 0, False, False, False, False),
    ('fp32', 96, 48, 2, False, False, False, False),
    ('fp16x3', 96, 48, 0, False, False, False, False),
    ('fp16x3', 96, 48, 2, False, False, False, True),
    ('tf32x3', 96, 48, 0, False, False, True, False),
    ('tf32x3', 96, 48, 2, False, False, False, False),
    ('bf16', 96, 48, 0, False, False, False, True),
    ('bf16', 96, 48, 2, False, False, False, False),
    ('fp16x3', 1024, 64, 0, False, False, False, False),
    ('fp16x3', 1024, 64, 0, False, False, True, False),
    ('bf16', 1024, 64, 0, False, False, True, True),
    ('tf32x3', 1024, 64, 1, False, False, False, True),
    ('fp16x3', 1024, 64, 0, False, True, True, False),
    ('fp16x3', 96, 48, 0, False, True, False, False),
    ('fp32', 96, 48, 1, True, False, False, False),
    ('tf32x3', 96, 48, 0, True, False, False, False),
    ('fp16x3', 96, 48, 2, True, False, False, True),
]
# EpiH<PREC, NL, FARNN, TRAIN, FUSE = true>, demangled or mangled
FUSED_EPI = re.compile(r'EpiH<[-\d, ]+, (?:false|true), true>|EpiHI(?:Lin?\d+E){3}Lb[01]ELb1E')


def _case_id(c):
    prec, S, R, farnn, save, full_pad, ab, wprep = c
    return '%s-S%d-farnn%d%s%s%s%s' % (prec, S, farnn, '-train' if save else '', '-full_pad' if full_pad else '',
                                      '-ab' if ab else '', '-wprep' if wprep else '')


@pytest.mark.parametrize('case', CASES, ids=_case_id)
def test_recurrence_path_queries_match_launches(case):
    from re2nn_seq_b200 import _lib, ops
    prec, S, R, farnn, save, full_pad, ab, wprep = case
    if prec != 'fp32' and not ops.has_tcgen05():
        pytest.skip('no tcgen05 device')
    g = torch.Generator(device='cuda').manual_seed(7)
    f32 = lambda *shape, scale=0.1: (torch.rand(shape, device='cuda', generator=g) - 0.5) * scale
    keep = []                                            # every buffer the argument block points at

    def ptr(t):
        keep.append(t)
        return C.c_void_p(t.data_ptr())

    lengths = torch.randint(1, L + 1, (B,), device='cuda', generator=g)
    lengths[0] = L
    x = torch.randint(0, V, (B, L), device='cuda', generator=g)
    S1, S2, W, Wss1, Wss2 = f32(S, R), f32(S, R), f32(S, S), f32(S, S), f32(S, S)
    a = ops._rec_args(S, R, farnn, prec, B, L, update_nonlinear='tanh', full_pad=full_pad, save_for_backward=save,
                      sigmoid_exponent=1.0)
    a.x, a.lengths, a.vtab = ptr(x), ptr(lengths), ptr(f32(V, R, scale=2.0))
    a.gtab = ptr(f32(V, S * farnn)) if farnn else None
    a.S1, a.S2, a.W, a.o, a.h0, a.hT = ptr(S1), ptr(S2), ptr(W), ptr(f32(S, scale=2.0)), ptr(f32(S)), ptr(f32(S))
    a.Wss1 = ptr(Wss1) if farnn >= 1 else None
    a.Wss2 = ptr(Wss2) if farnn == 2 else None
    a.alpha, a.beta = ptr(torch.empty(B, L, S, device='cuda')), ptr(torch.empty(B, L, S, device='cuda'))
    if save:
        a.hbar_save, a.hst_save = ptr(torch.zeros(2, L + 1, B, S, device='cuda')), ptr(torch.zeros(2, L + 1, B, S, device='cuda'))
        a.u_save, a.a_save = ptr(torch.zeros(2, L, B, R, device='cuda')), ptr(torch.zeros(2, L, B, S, device='cuda'))
        a.zsave = ptr(torch.zeros(2, L, B, S, device='cuda')) if farnn >= 1 else None
        a.rsave = ptr(torch.zeros(2, L, B, S, device='cuda')) if farnn == 2 else None
    if ab:
        nbytes = _lib.fn['re2nn_label_scores_ab_bytes'](B, L, S, _lib.PREC[prec])
        a.ab_out = ptr(torch.empty(nbytes, dtype=torch.uint8, device='cuda'))
    if wprep:
        a.wprep = ptr(ops.weight_prep(S1, S2, W, Wss1 if farnn >= 1 else None, Wss2 if farnn == 2 else None, farnn, prec))
    need = _lib.fn['re2nn_decompose_recurrence_workspace'](C.byref(a))
    a.ws, a.ws_bytes = ptr(torch.empty(need, dtype=torch.uint8, device='cuda')), need

    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    run = lambda: _lib.check(_lib.fn['re2nn_decompose_recurrence'](C.byref(a), stream), 'decompose_recurrence')
    run()                                                # module loads and smem attributes outside the profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run()
        torch.cuda.synchronize()
    kernels = [e.name for e in prof.events()
               if e.device_type == DeviceType.CUDA and not e.name.startswith(('Memcpy', 'Memset'))]

    launches = _lib.fn['re2nn_decompose_recurrence_launches'](C.byref(a))
    resident = _lib.fn['re2nn_decompose_recurrence_resident'](C.byref(a))
    fuses = _lib.fn['re2nn_decompose_recurrence_fuses'](C.byref(a))
    assert len(kernels) == launches, kernels
    assert any('tc_resident_kernel' in k for k in kernels) == bool(resident), kernels
    assert any(FUSED_EPI.search(k) for k in kernels) == bool(fuses and ab), kernels
