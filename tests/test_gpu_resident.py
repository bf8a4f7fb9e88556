"""GPU: the resident recurrence kernel (one launch for all steps, a CTA pair per 128-row tile) against the
one-launch-per-step path and the float64 oracle: more tiles than SM pairs (a pair walks several tiles), ragged
lengths (tiles stop at their own last step), batches that are not a multiple of 128, pad semantics (full_pad),
pre-computed rank factors (FARNN_S_SF), every tensor-core precision."""
import numpy as np
import pytest
import torch

from helpers import oracle_params, rel_err
from oracle import re2nn_oracle as orc

pytestmark = pytest.mark.gpu


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _need_tc():
    from re2nn_seq_b200 import ops
    if not ops.has_tcgen05():
        pytest.skip('no tcgen05 device')


def _set_resident(on):
    from re2nn_seq_b200 import _lib
    _lib.check(_lib.fn['re2nn_debug_set_resident'](1 if on else 0), 'resident')


def _launches(m, xt, lt):
    from re2nn_seq_b200 import ops
    l0 = ops.launches()
    with torch.no_grad():
        s = m.forward_scores(xt, lt)
    return s, ops.launches() - l0


class _Z(dict):
    files = property(lambda self: list(self.keys()))


def _truth(m, args, x, lens):
    z = _Z({'p.' + k: v.detach().cpu().numpy() for k, v in m.state_dict().items()})
    sc, _, _ = orc.decompose_scores(oracle_params(z, np.float64), x, lens, args)
    return sc


@pytest.mark.parametrize('prec,tol', [('fp16x3', 1e-5), ('tf32x3', 1e-5), ('bf16', 3e-2)])
@pytest.mark.parametrize('B,S,R,L,nl', [(5000, 96, 48, 9, 'tanh'), (333, 300, 200, 12, 'tanh'), (130, 64, 40, 7, 'relu')])
def test_resident_matches_per_step_and_oracle(B, S, R, L, nl, prec, tol):
    from test_gpu_parity import _random_decompose
    _need_tc()
    m, args, x, lens, lab = _random_decompose(11, 500, S, R, 20, 50, B, L, farnn=0, use_crf=0, update_nonlinear=nl,
                                              beta=0.1)
    m.precision = prec
    m.use_cuda_graph = False
    xt, lt = _t(x), _t(lens)
    try:
        _set_resident(True)
        s_res, n_res = _launches(m, xt, lt)
        _set_resident(False)
        s_step, n_step = _launches(m, xt, lt)
    finally:
        _set_resident(True)
    Lmax = int(lens.max())
    assert n_res < n_step and (n_step - n_res) % 2 == 1   # one resident launch replaces two step GEMMs per step
    mask = orc.length_mask(lens, Lmax)
    a, b = s_res.cpu().numpy()[mask], s_step.cpu().numpy()[mask]
    if prec != 'bf16':
        assert np.array_equal(a, b)                  # same summation order as the per-step path: same bits
    truth = _truth(m, args, x, lens)[mask]
    assert rel_err(a, truth) < tol
    assert rel_err(b, truth) < tol


def test_resident_full_pad_positions():
    """KD / PR read the scores at pad positions: with full_pad every tile runs all L steps (reference semantics)."""
    from test_gpu_parity import _random_decompose
    _need_tc()
    m, args, x, lens, lab = _random_decompose(3, 400, 80, 48, 12, 50, 300, 10, farnn=0, use_crf=0, update_nonlinear='tanh',
                                              beta=0.1)
    m.use_cuda_graph = False
    m.full_pad = True
    xt, lt = _t(x), _t(lens)
    out = {}
    try:
        for prec in ('fp32', 'fp16x3'):
            m.precision = prec
            with torch.no_grad():
                out[prec] = m.forward_scores(xt, lt).cpu().numpy()
    finally:
        m.full_pad = False
    assert rel_err(out['fp16x3'], out['fp32']) < 1e-5            # every position, pads included


def test_resident_precomputed_factors():
    """FARNN_S_SF (v_t supplied as B x L x R floats) through the resident kernel."""
    import re2nn_seq_b200 as r
    from re2nn_seq_b200 import synth
    _need_tc()
    S, R, C, B, L = 120, 72, 15, 700, 8
    args = synth.make_args(farnn=0, use_crf=0, update_nonlinear='tanh', beta=0.1)
    f = synth.make_decompose_factors(2, 300, S, R, C, 50, dtype=np.float32)
    keep = ('S1', 'S2', 'C_output_mat', 'wildcard_mat', 'wildcard_output_vector', 'final_vector', 'start_vector')
    m = r.FARNN_S_SF(args=args, o_idx=0, is_cuda=True, priority_mat=None, **{k: f[k] for k in keep}).cuda()
    m.use_cuda_graph = False
    rs = np.random.RandomState(5)
    v = (rs.randn(B, L, R) * 0.3).astype(np.float32)
    lens = rs.randint(3, L + 1, size=B).astype(np.int64)
    lens[0] = L
    vt, lt = _t(v), _t(lens)
    out = {}
    for prec in ('fp32', 'fp16x3'):
        m.precision = prec
        with torch.no_grad():
            out[prec] = m.forward_scores(vt, lt).cpu().numpy()
    mask = orc.length_mask(lens, L)
    assert rel_err(out['fp16x3'][mask], out['fp32'][mask]) < 1e-5


@pytest.mark.parametrize('prec', ['fp16x3', 'tf32x3', 'bf16'])
@pytest.mark.parametrize('farnn', [1, 2])
@pytest.mark.parametrize('B,S,R,L', [(5000, 96, 48, 7), (300, 300, 200, 12)])
def test_resident_gated_matches_per_step_and_oracle(B, S, R, L, farnn, prec):
    """farnn = 1 / 2: the gate GEMM runs as one (z) or two (z, r) extra phases of the resident kernel."""
    from test_gpu_parity import _random_decompose
    _need_tc()
    m, args, x, lens, lab = _random_decompose(13, 500, S, R, 20, 50, B, L, farnn=farnn, use_crf=0, update_nonlinear='tanh',
                                              beta=0.1)
    m.precision = prec
    m.use_cuda_graph = False
    xt, lt = _t(x), _t(lens)
    try:
        _set_resident(True)
        s_res, n_res = _launches(m, xt, lt)
        _set_resident(False)
        s_step, n_step = _launches(m, xt, lt)
    finally:
        _set_resident(True)
    assert n_res < n_step
    mask = orc.length_mask(lens, int(lens.max()))
    a, b = s_res.cpu().numpy()[mask], s_step.cpu().numpy()[mask]
    if prec != 'bf16':
        assert np.array_equal(a, b)
    truth = _truth(m, args, x, lens)[mask]
    tol = 3e-2 if prec == 'bf16' else 1e-5
    assert rel_err(a, truth) < tol
    assert rel_err(b, truth) < tol


@pytest.mark.parametrize('farnn,crf', [(0, 1), (2, 0)])
def test_chunked_multi_stream_inference_matches_single_stream(farnn, crf):
    """The graphed inference body forks one stream per chunk of the length-sorted batch (scoring + decode of the
    short chunks overlap the recurrence of the longest): same predictions as the single-stream and eager paths."""
    from test_gpu_parity import _random_decompose
    _need_tc()
    m, args, x, lens, lab = _random_decompose(17, 400, 96, 48, 14, 50, 1500, 11, farnn=farnn, use_crf=crf,
                                              update_nonlinear='tanh', beta=0.1)
    m.precision = 'fp16x3'
    xt, lt, yt = _t(x), _t(lens), _t(lab)
    out = {}
    with torch.no_grad():
        for chunks in (1, 4, 3):
            m.infer_chunks = chunks
            for _ in range(2):                       # capture, then replay
                _, pred, true = m.forward_local(xt, yt, lt, train=False)
            out[chunks] = (pred.clone(), true.clone())
        m.use_cuda_graph = False
        _, pred_e, true_e = m.forward_local(xt, yt, lt, train=False)
    for chunks in (1, 4, 3):
        assert torch.equal(out[chunks][0], pred_e), chunks
        assert torch.equal(out[chunks][1], true_e), chunks
    assert pred_e.shape[0] == int(lens.sum())


def test_chunked_multi_stream_inference_precomputed_factors():
    """FARNN_S_SF (dense B x L x R input) through the chunked, graphed inference body."""
    import re2nn_seq_b200 as r
    from re2nn_seq_b200 import synth
    _need_tc()
    S, R, C, B, L = 96, 48, 11, 1300, 9
    args = synth.make_args(farnn=0, use_crf=1, update_nonlinear='tanh', beta=0.1)
    f = synth.make_decompose_factors(6, 300, S, R, C, 50, dtype=np.float32)
    keep = ('S1', 'S2', 'C_output_mat', 'wildcard_mat', 'wildcard_output_vector', 'final_vector', 'start_vector')
    torch.manual_seed(2)
    m = r.FARNN_S_SF(args=args, o_idx=0, is_cuda=True, priority_mat=None, **{k: f[k] for k in keep}).cuda()
    with torch.no_grad():
        m.crf.transitions.copy_(torch.from_numpy(synth.crf_transitions(6, m.C)))
    m.precision = 'fp16x3'
    rs = np.random.RandomState(7)
    v = _t((rs.randn(B, L, R) * 0.3).astype(np.float32))
    lens = rs.randint(2, L + 1, size=B).astype(np.int64)
    lens[0] = L
    lt, yt = _t(lens), _t(rs.randint(0, C, size=(B, L)).astype(np.int64))
    out = {}
    with torch.no_grad():
        for chunks in (1, 4):
            m.infer_chunks = chunks
            for _ in range(2):
                _, pred, true = m(v, yt, lt, train=False)
            out[chunks] = pred.clone()
        m.use_cuda_graph = False
        _, pred_e, _ = m(v, yt, lt, train=False)
    assert torch.equal(out[1], pred_e) and torch.equal(out[4], pred_e)


def test_graph_policy_over_an_evaluation_sweep():
    """val.py-style sweep: batch shapes change from batch to batch and the parameters change between sweeps.  A key is
    captured only on its second sighting, captures are bounded and evicted (stale parameter versions first), in-place
    `.data` writes are picked up after invalidate_caches(), and every result equals the eager path."""
    import re2nn_seq_b200 as r
    from re2nn_seq_b200 import synth
    args = synth.make_args(farnn=0, use_crf=1, update_nonlinear='tanh', beta=0.1)
    f = synth.make_decompose_factors(3, 300, 96, 64, 9, 16, dtype=np.float32)
    torch.manual_seed(3)
    m = r.FARNN_S_D_W_I_S(args=args, o_idx=0, **f)
    with torch.no_grad():
        m.crf.transitions.copy_(torch.from_numpy(synth.crf_transitions(3, m.C)))
    m = m.cuda().eval()
    rs = np.random.RandomState(0)
    shapes = [(256, 9), (256, 12), (130, 9), (256, 9), (256, 12), (256, 9), (384, 7), (256, 12)] + \
             [(256, int(l)) for l in rs.randint(5, 20, size=14)]

    def sweep():
        out = []
        for i, (B, Lmax) in enumerate(shapes):
            x, lens, lab = synth.make_batch(100 + i, B, Lmax, 300, 9)
            xt, lt, yt = _t(x), _t(lens), _t(lab)
            with torch.no_grad():
                _, pred, _ = m.forward_local(xt, yt, lt, train=False)
                m.use_cuda_graph = False
                _, want, _ = m.forward_local(xt, yt, lt, train=False)
                m.use_cuda_graph = True
            assert torch.equal(pred, want), 'batch %d (B=%d, L<=%d)' % (i, B, Lmax)
            out.append(pred.clone())
        return out

    first = sweep()
    assert 1 <= len(m._graphs) <= m._GRAPH_MAX_ENTRIES          # repeated keys were captured, the rest ran eagerly
    n_captured = len(m._graphs)
    again = sweep()                                              # same parameters: captures are reused / extended, bounded
    assert len(m._graphs) <= m._GRAPH_MAX_ENTRIES and len(m._graphs) >= n_captured
    for a, b in zip(first, again):
        assert torch.equal(a, b)
    with torch.no_grad():                                        # an in-place write that does NOT bump _version ...
        m.S1.data.mul_(1.5)
    m.invalidate_caches()                                        # ... needs the documented call
    assert len(m._graphs) == 0
    changed = sweep()
    assert any(not torch.equal(a, b) for a, b in zip(first, changed))
    m.train()                                                    # train() / eval() invalidate on their own
    m.eval()
    assert len(m._graphs) == 0


@pytest.mark.parametrize('farnn,B,S,R,L', [(0, 700, 300, 200, 13), (2, 520, 136, 72, 9), (0, 333, 64, 40, 14)])
def test_weight_gradient_gemm_on_tensor_cores_matches_cuda_cores(farnn, B, S, R, L):
    """The weight gradients (X^T Y over every (step, sequence) row, gemm_tn_tc.cuh: 3xTF32 with on-the-fly transposition,
    ragged split-K chunks, P / Q that are no multiples of the tile) against the fp32 CUDA-core kernel."""
    from test_gpu_parity import _random_decompose
    from re2nn_seq_b200 import _lib
    _need_tc()
    m, args, x, lens, lab = _random_decompose(31, 400, S, R, 20, 50, B, L, farnn=farnn, use_crf=1, update_nonlinear='tanh',
                                              beta=0.1, train_h0=1, train_hT=1)
    xt, lt, yt = _t(x), _t(lens), _t(lab)
    out = {}
    try:
        for on in (1, 0):
            _lib.check(_lib.fn['re2nn_debug_set_tn_tc'](on), 'tn_tc')
            m.zero_grad(set_to_none=True)
            loss, _, _ = m.forward_local(xt, yt, lt, train=True)
            loss.backward()
            torch.cuda.synchronize()
            out[on] = {k: v.grad.detach().clone() for k, v in m.named_parameters() if v.grad is not None}
    finally:
        _lib.check(_lib.fn['re2nn_debug_set_tn_tc'](1), 'tn_tc')
    checked = 0
    for k, g in out[1].items():
        ref = out[0][k]
        err = (g - ref).abs().max().item() / (ref.abs().max().item() + 1e-30)
        assert err < 5e-6, '%s: %.3e' % (k, err)
        checked += int(g.dim() == 2)
    assert checked >= 3
