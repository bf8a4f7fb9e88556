"""GPU: N-best CRF decoding and tag marginals (re2nn_crf_nbest / re2nn_crf_marginals, the CRF and model methods on
top) against the oracle restatements, the Viterbi kernels and a float64 autograd CRF."""
import numpy as np
import pytest
import torch

from helpers import rel_err
import crf_nbest_ref as ref
from oracle import re2nn_oracle as orc

pytestmark = pytest.mark.gpu


def _t(a, dev='cuda'):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _crf_case(seed, B, L, T, integer=False):
    rs = np.random.RandomState(seed)
    if integer:
        feats = rs.randint(-3, 4, size=(B, L, T)).astype(np.float32)
        trans = rs.randint(-2, 3, size=(T, T)).astype(np.float32)
    else:       # quarter steps (many exact ties) plus real-valued rows, as the Viterbi tests use
        feats = (rs.randint(-8, 9, size=(B, L, T)) * 0.25).astype(np.float32)
        feats[::3] += rs.randn(*feats[::3].shape).astype(np.float32)
        trans = (rs.randint(-4, 5, size=(T, T)) * 0.5).astype(np.float32)
    trans[:, T - 2] = -10000.0
    trans[T - 1, :] = -10000.0
    lens = rs.randint(1, L + 1, size=B).astype(np.int64)
    lens[0] = L
    return feats, trans, lens


def _check_nbest(feats, trans, lens, K, rows=None):
    from re2nn_seq_b200 import ops
    paths, scores = ops.crf_nbest(_t(feats), _t(trans), _t(lens), K)
    paths, scores = paths.cpu().numpy(), scores.cpu().numpy()
    rows = np.arange(len(lens)) if rows is None else rows
    want_p, want_s = ref.crf_nbest(feats[rows], lens[rows], trans, K)
    np.testing.assert_array_equal(paths[rows], want_p)
    np.testing.assert_array_equal(scores[rows], want_s)          # bit-identical, -inf for missing ranks
    return paths, scores


@pytest.mark.parametrize('K', [1, 2, 5, 16])
@pytest.mark.parametrize('T', [5, 34, 75, 131, 200, 260, 1024])
def test_nbest_matches_restatement(T, K):
    """Transitions in shared memory (T <= 200) and in global memory (260, and 1024 at every K); ragged lengths, an
    empty sequence, a length past L and a one-token sequence (fewer than K sequences when T < K)."""
    B, L = (4, 4) if T == 1024 else ((12, 5) if T >= 200 else (40, 6))
    feats, trans, lens = _crf_case(T + K, B, L, T)
    lens[1] = 0
    lens[2] = L + 3
    lens[-1] = 1
    paths, _ = _check_nbest(feats, trans, lens, K)
    assert (paths[1] == 0).all()
    # rank 0 is the Viterbi path at every valid position
    import re2nn_seq_b200 as r
    crf = r.CRF(T - 2, True).cuda()
    with torch.no_grad():
        crf.transitions.copy_(_t(trans))
    n = np.minimum(lens, L)
    mask = orc.length_mask(n, L)
    _, vit = crf._viterbi_decode(_t(feats), None, lengths=_t(n))
    np.testing.assert_array_equal(paths[:, :, 0][mask], vit.cpu().numpy()[mask])


@pytest.mark.parametrize('K', [4, 16])
@pytest.mark.parametrize('T', [12, 70])
def test_nbest_integer_ties(T, K):
    """Small-integer features: exact sums, many equal scores; the order of ties is the restatement's."""
    feats, trans, lens = _crf_case(3 * T + K, 200, 7, T, integer=True)
    _check_nbest(feats, trans, lens, K)


def test_nbest_large_batch():
    """B = 16384 at T = 131 (cfg5's tag set), K = 8: the whole batch runs, a sample of rows against the restatement."""
    feats, trans, lens = _crf_case(1, 16384, 10, 131)
    rows = np.concatenate([np.arange(8), np.random.RandomState(2).choice(16384, 16, replace=False)])
    _check_nbest(feats, trans, lens, 8, rows)


def test_nbest_errors():
    from re2nn_seq_b200 import ops
    feats, trans, lens = _crf_case(0, 2, 3, 7)
    for K in (0, 17):
        with pytest.raises(RuntimeError, match=r'outside \[1, 16\]'):
            ops.crf_nbest(_t(feats), _t(trans), _t(lens), K)
    T = 2000                                           # 2000 x 16 lists do not fit one sequence's shared memory
    with pytest.raises(RuntimeError, match='too large'):
        ops.crf_nbest(torch.zeros(1, 2, T, device='cuda'), torch.zeros(T, T, device='cuda'),
                      torch.tensor([2], device='cuda'), 16)
    ops.crf_nbest(torch.zeros(1, 2, T, device='cuda'), torch.zeros(T, T, device='cuda'),
                  torch.tensor([2], device='cuda'), 12)            # 2000 x 12 does


def _logz64(feats, trans, lens):
    """float64 autograd CRF (crf.py:48-99): log Z per sequence and its gradient w.r.t. the features."""
    B, L, T = feats.shape
    f64 = torch.from_numpy(feats).double().requires_grad_(True)
    t64 = torch.from_numpy(trans).double()
    n = torch.from_numpy(lens)
    part = f64[:, 0] + t64[T - 2]
    for t in range(1, L):
        nxt = torch.logsumexp(part[:, :, None] + t64, 1) + f64[:, t]
        part = torch.where((t < n)[:, None], nxt, part)
    logz = torch.logsumexp(part + t64[:, T - 1], 1)
    logz.sum().backward()
    return logz.detach().numpy(), f64.grad.numpy()


@pytest.mark.parametrize('ntag', [20, 73, 129, 151, 152, 198, 258, 598])
def test_marginals_vs_float64_gradient(ntag):
    """P(y_t = j | x) = d log Z / d feat_t[j]: against float64 autograd on spiky features with forbidden (-1e4)
    transitions (underflowing rows take the exact fallback).  T = 153 is the last scaled-exponential width; 260 and
    600 are beyond the training backward's limit."""
    import re2nn_seq_b200 as r
    rs = np.random.RandomState(ntag)
    B, L = 37, 14
    T = ntag + 2
    feats = (rs.randn(B, L, T) * 12.0).astype(np.float32)
    lens = rs.randint(2, L + 1, size=B).astype(np.int64)
    lens[0] = L
    lens[1] = 0
    trans = rs.randn(T, T).astype(np.float32)
    trans[rs.rand(T, T) < 0.4] = -10000.0
    trans[:, T - 2] = -10000.0
    trans[T - 1, :] = -10000.0
    crf = r.CRF(ntag, True).cuda()
    with torch.no_grad():
        crf.transitions.copy_(_t(trans))
    marg, log_z = crf.marginals(_t(feats), None, lengths=_t(lens))
    marg, log_z = marg.cpu().numpy(), log_z.cpu().numpy()
    keep = lens > 0
    want_z, want_m = _logz64(feats[keep], trans, lens[keep])
    # log Z is a few hundred here: fp32 keeps ~3e-5 absolute on it, which is the relative error of every marginal
    assert rel_err(marg[keep], want_m) < 3e-4, 'T = %d' % T
    assert rel_err(log_z[keep], want_z) < 1e-5
    assert log_z[1] == 0 and (marg[1] == 0).all()
    mask = orc.length_mask(lens, L)
    assert np.abs(marg.sum(2)[mask] - 1).max() < 1e-4
    assert (marg[~mask] == 0).all()


def test_marginals_match_restatement():
    from re2nn_seq_b200 import ops
    feats, trans, lens = _crf_case(4, 64, 9, 75)
    marg, log_z = ops.crf_marginals(_t(feats), _t(trans), _t(lens))
    want_m, want_z = ref.crf_marginals(feats.astype(np.float64), lens, trans.astype(np.float64))
    assert np.abs(marg.cpu().numpy() - want_m).max() < 1e-5
    assert rel_err(log_z.cpu().numpy(), want_z) < 1e-6


def test_crf_nbest_normalised_path_scores():
    """CRF._viterbi_decode_nbest: NCRF++'s softmax over the returned path scores, missing ranks at 0."""
    import re2nn_seq_b200 as r
    feats, trans, lens = _crf_case(8, 16, 5, 6)
    lens[1] = 0
    lens[2] = 1                                     # 6 sequences < K = 8
    crf = r.CRF(4, True).cuda()
    with torch.no_grad():
        crf.transitions.copy_(_t(trans))
    mask = _t(orc.length_mask(lens, 5))
    score, idx = crf._viterbi_decode_nbest(_t(feats), mask, 8)
    _, scores = ref.crf_nbest(feats, lens, trans, 8)
    with np.errstate(invalid='ignore'):                # row 1 has no sequence at all
        want = np.exp(scores.astype(np.float64) - scores.max(1, keepdims=True))
    want[1] = 0
    want[[0] + list(range(2, 16))] /= want[[0] + list(range(2, 16))].sum(1, keepdims=True)
    np.testing.assert_allclose(score.cpu().numpy(), want, rtol=0, atol=1e-6)
    assert (score[2, 6:] == 0).all() and (idx[2, 0, 6:] == -1).all()
    _, vit = crf._viterbi_decode(_t(feats), mask)
    m = orc.length_mask(lens, 5)
    np.testing.assert_array_equal(idx[:, :, 0].cpu().numpy()[m], vit.cpu().numpy()[m])


def _decompose_model(kind):
    import re2nn_seq_b200 as r
    from re2nn_seq_b200 import synth
    S, R, C, B, L, V = 120, 72, 15, 300, 9, 400
    args = synth.make_args(farnn=0, use_crf=1, update_nonlinear='tanh', beta=0.1, local_loss_func='CE1')
    f = synth.make_decompose_factors(11, V, S, R, C, 50, dtype=np.float32)
    x, lens, lab = synth.make_batch(12, B, L, V, C)
    torch.manual_seed(0)
    if kind == 'tok':
        m = r.FARNN_S_D_W_I_S(args=args, o_idx=0, **f)
        inp = x
    else:
        keep = ('S1', 'S2', 'C_output_mat', 'wildcard_mat', 'wildcard_output_vector', 'final_vector', 'start_vector')
        m = r.FARNN_S_SF(args=args, o_idx=0, is_cuda=True, priority_mat=None, **{k: f[k] for k in keep})
        inp = (np.random.RandomState(13).randn(B, L, R) * 0.3).astype(np.float32)
    with torch.no_grad():
        m.crf.transitions.copy_(torch.from_numpy(synth.crf_transitions(11, m.C)))
    return m.cuda(), _t(inp), _t(lab), _t(lens)


@pytest.mark.parametrize('kind', ['tok', 'sf'])
def test_model_forward_nbest(kind):
    """pred[..., 0] is what forward_local decodes (eager call and graph replay), under CE1 with a threshold that clamps
    column C-3; seq_prob is non-increasing, sums to at most 1, and rank 0's is exp(Viterbi score - log Z)."""
    m, inp, lab, lens = _decompose_model(kind)
    with torch.no_grad():
        sc = m.forward_scores(inp, lens)
        n = lens.cpu().numpy()
        valid = _t(orc.length_mask(n, int(n.max())))
        m.args.threshold = float(sc[:, :, m.C - 3][valid].median())     # clamps about half the valid positions
        call = m.forward_local if kind == 'tok' else m.forward
        preds = [call(inp, lab, lens, train=False)[1] for _ in range(3)]  # eager, capture, replay
    pred, seq_prob, marg = m.forward_nbest(inp, lens, nbest=4)
    assert pred.shape[2] == 4 and seq_prob.shape == (len(n), 4) and marg.shape == sc.shape
    top = pred[:, :, 0][valid]
    for p in preds:
        assert torch.equal(top, p), int((top != p).sum())
    sp = seq_prob.cpu().numpy()
    assert (np.diff(sp, axis=1) <= 0).all() and (sp.sum(1) <= 1 + 1e-6).all()
    # rank 0's probability from the Viterbi path of the clamped scores and the marginal kernels' log Z
    clamped = sc.clone()
    clamped[:, :, m.C - 3] = torch.minimum(clamped[:, :, m.C - 3], clamped.new_tensor(m.args.threshold))
    trans = m.crf.transitions.detach().cpu().numpy()
    _, want_s = ref.crf_nbest(clamped.cpu().numpy(), n, trans, 1)
    _, log_z = m.crf.marginals(clamped, None, lengths=lens)
    np.testing.assert_allclose(sp[:, 0], np.exp(want_s[:, 0] - log_z.cpu().numpy()), rtol=1e-5, atol=0)
    np.testing.assert_allclose(marg.sum(2)[valid].cpu().numpy(), 1.0, rtol=0, atol=1e-4)


def test_model_without_crf_raises():
    import re2nn_seq_b200 as r
    from re2nn_seq_b200 import synth
    args = synth.make_args(farnn=0, use_crf=0, update_nonlinear='tanh')
    f = synth.make_decompose_factors(1, 50, 16, 8, 5, 10, dtype=np.float32)
    m = r.FARNN_S_D_W_I_S(args=args, o_idx=0, **f).cuda()
    x, lens, _ = synth.make_batch(2, 4, 5, 50, 5)
    with pytest.raises(NotImplementedError, match='CRF'):
        m.forward_nbest(_t(x), _t(lens), 2)


def test_ops_registered_cuda_only():
    from re2nn_seq_b200 import _lib
    for name in ('crf_nbest', 'crf_marginals'):
        schema = str(getattr(_lib.tops, name).default._schema)
        assert schema.startswith('re2nn::' + name + '('), schema
    f, tr, ln = torch.zeros(2, 3, 5), torch.zeros(5, 5), torch.tensor([3, 2])
    with pytest.raises((RuntimeError, NotImplementedError)):
        _lib.tops.crf_nbest(f, tr, ln, 2)
    with pytest.raises((RuntimeError, NotImplementedError)):
        _lib.tops.crf_marginals(f, tr, ln)
