"""GPU: the partial-annotation CRF loss (re2nn_crf_partial_nll / _backward) and constrained decoding, from the kernels up
to the CRF and model methods, against the float64 and float32 restatements of crf_partial_ref.py and the supervised
CRF kernels."""
import numpy as np
import pytest
import torch

from helpers import rel_err
import crf_partial_ref as ref
from oracle import re2nn_oracle as orc

pytestmark = pytest.mark.gpu

TOL = 1e-5
# every forward (3-32-64-96-128-153 | 154-218 | 219-) and backward (3-96 | 97-111 | 112-159 | 160-225) range edge
WIDTHS = [3, 32, 33, 64, 65, 96, 97, 111, 112, 128, 129, 153, 154, 159, 160, 218, 219, 225]


def _t(a, dev='cuda'):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _mixed_case(T, seed=3, B=37, L=14):
    """Spiky features and forbidden (-1e4) transitions, so the scaled-exponential kernels take their exact fallback;
    ragged lengths with 0, 1 and > L; masks cycling random / one-hot / all-true over the batch, garbage at pads.
    Every mask keeps a path y* whose transitions are not forbidden, so log Z^A stays a few hundred (fp32 keeps
    ~3e-5 absolute on it, the error of every marginal)."""
    rs = np.random.RandomState(seed + T)
    feats = (rs.randn(B, L, T) * 12.0).astype(np.float32)
    trans = rs.randn(T, T).astype(np.float32)
    trans[rs.rand(T, T) < 0.4] = -10000.0
    trans[:, T - 2] = -10000.0
    trans[T - 1, :] = -10000.0
    lens = rs.randint(2, L + 1, size=B).astype(np.int64)
    lens[0], lens[1], lens[2], lens[3] = L, 0, 1, L + 5
    real = max(T - 2, 1)
    ystar = rs.randint(0, real, size=(B, L))
    for b in range(B):                      # y* avoids forbidden transitions (START -> y0 ... y_{n-1} -> STOP)
        n = min(int(lens[b]), L)
        prev = T - 2
        for t in range(n):
            if trans[prev, ystar[b, t]] < -1000:
                trans[prev, ystar[b, t]] = rs.randn()
            prev = ystar[b, t]
        if n and trans[prev, T - 1] < -1000:
            trans[prev, T - 1] = rs.randn()
    onehot = np.eye(T, dtype=bool)[ystar]
    allowed = np.ones((B, L, T), bool)
    kind = np.arange(B) % 3
    allowed[kind == 0] = (rs.rand(B, L, T) < 0.5)[kind == 0] | onehot[kind == 0]
    allowed[kind == 1] = onehot[kind == 1]
    pad = np.arange(L)[None, :] >= np.minimum(lens, L)[:, None]
    allowed[pad] = rs.rand(int(pad.sum()), T) < 0.2          # ignored by the kernels, may be empty
    return feats, trans, lens, allowed


def _crf(trans):
    import re2nn_seq_b200 as r
    T = trans.shape[0]
    crf = r.CRF(T - 2, True).cuda()
    with torch.no_grad():
        crf.transitions.copy_(_t(trans))
    return crf


@pytest.mark.parametrize('T', WIDTHS + [226])
def test_partial_loss_and_gradients_vs_float64(T):
    feats, trans, lens, allowed = _mixed_case(T)
    crf = _crf(trans)
    f = _t(feats).requires_grad_(True)
    loss = crf.partial_neg_log_likelihood_loss(f, None, _t(allowed), lengths=_t(lens))
    per_seq, want_df, want_dt = ref.crf_partial_nll(feats, lens, trans, allowed)
    # the two lattices round apart by ~1e-7 |log Z| per sequence, which is all there is when the mask only removes
    # paths of weight e^-10000 (T = 3: every START / STOP cell)
    from re2nn_seq_b200 import ops
    scale = float(ops.crf_marginals(_t(feats), _t(trans), _t(lens))[1].abs().sum())
    assert abs(loss.item() - per_seq.sum()) <= max(TOL * abs(per_seq.sum()), 1e-6 * scale), 'T = %d' % T
    if T > 225:
        with pytest.raises(RuntimeError, match='tag set too large'):
            loss.backward()
        return
    loss.backward()
    # marginal differences are at most 1 in size: measure against 1 where the float64 gradient is (near) zero (T = 3)
    for got, want in ((f.grad.cpu().numpy(), want_df), (crf.transitions.grad.cpu().numpy(), want_dt)):
        assert np.abs(got - want).max() / max(np.abs(want).max(), 1.0) < 3e-4, 'T = %d' % T
    assert np.isfinite(f.grad.cpu().numpy()).all()
    assert (f.grad[1] == 0).all()                                  # the empty sequence


def _partial(feats, trans, lens, allowed, g=1.0):
    from re2nn_seq_b200 import ops
    loss, per_seq, (part, part_a) = ops.crf_partial_nll(feats, trans, lens, allowed, save=True)
    df, dt = ops.crf_partial_nll_backward(feats, trans, lens, allowed, part, part_a,
                                          torch.tensor(g, device='cuda'))
    return loss, per_seq, df, dt


def test_partial_backward_split_same_result():
    """T = 75: the three-warps-per-sequence backward and the one-warp backward give the same gradients."""
    from re2nn_seq_b200 import _lib
    feats, trans, lens, allowed = _mixed_case(75, B=300)
    args = (_t(feats), _t(trans), _t(lens), _t(allowed))
    try:
        _lib.check(_lib.fn['re2nn_debug_set_crf_backward_split'](0), 'crf split')
        _, _, df1, dt1 = _partial(*args)
        _lib.check(_lib.fn['re2nn_debug_set_crf_backward_split'](1), 'crf split')
        _, _, df3, dt3 = _partial(*args)
    finally:
        _lib.check(_lib.fn['re2nn_debug_set_crf_backward_split'](1), 'crf split')
    np.testing.assert_allclose(df3.cpu().numpy(), df1.cpu().numpy(), rtol=0, atol=1e-6)
    assert rel_err(dt3.cpu().numpy(), dt1.cpu().numpy()) < 1e-6


@pytest.mark.parametrize('T', WIDTHS)
def test_all_true_mask_is_exactly_zero(T):
    """An all-true mask: the constrained lattice repeats the free one operation for operation, so per_seq is 0.0 and both
    gradients are exactly zero (an unlabelled sequence in a mixed batch contributes nothing at all)."""
    feats, trans, lens, _ = _mixed_case(T, seed=9)
    allowed = np.ones(feats.shape, bool)
    loss, per_seq, df, dt = _partial(_t(feats), _t(trans), _t(lens), _t(allowed), g=0.7)
    assert (per_seq == 0).all() and loss.item() == 0.0
    assert (df == 0).all() and (dt == 0).all()


@pytest.mark.parametrize('T', [5, 34, 75, 100, 131, 160, 200, 225])
def test_onehot_mask_is_the_supervised_loss(T):
    """A one-hot mask of the gold tags: per_seq and both gradients are crf_nll's, within fp32 rounding of |log Z|."""
    from re2nn_seq_b200 import ops
    rs = np.random.RandomState(T)
    B, L = 64, 11
    feats = (rs.randn(B, L, T) * 3).astype(np.float32)
    trans = rs.randn(T, T).astype(np.float32)
    lens = rs.randint(1, L + 1, size=B).astype(np.int64)
    lens[1] = 0
    tags = rs.randint(0, T, size=(B, L)).astype(np.int64)
    f, tr, ln, tg = _t(feats), _t(trans), _t(lens), _t(tags)
    g = torch.tensor(1.0, device='cuda')
    _, ps_s, part = ops.crf_nll(f, tr, ln, tg, save=True)
    df_s, dt_s = ops.crf_nll_backward(f, tr, ln, tg, part, g)
    _, ps_p, df_p, dt_p = _partial(f, tr, ln, _t(np.eye(T, dtype=bool)[tags]))
    _, log_z = ops.crf_marginals(f, tr, ln)
    scale = float(log_z.abs().max())
    assert (ps_p - ps_s).abs().max().item() <= 1e-6 * scale + 1e-5
    assert (df_p - df_s).abs().max().item() <= 1e-6 * scale + 1e-5
    assert (dt_p - dt_s).abs().max().item() <= B * (1e-6 * scale + 1e-5)


def _viterbi_seqs(ns):
    from re2nn_seq_b200 import _lib
    _lib.check(_lib.fn['re2nn_debug_set_viterbi_seqs'](ns), 'seqs')


@pytest.mark.parametrize('T', [5, 75, 160, 161, 216, 217, 260])
def test_constrained_decode(T):
    """All-true: bit-identical to _viterbi_decode (pads included).  Random masks: bit-identical to the restatement and
    every tag allowed.  One-hot: the mask itself.  Under both sequences-per-warp settings of the Viterbi kernel."""
    rs = np.random.RandomState(T)
    B, L = 96, 9
    feats = (rs.randint(-8, 9, size=(B, L, T)) * 0.25).astype(np.float32)    # many exact ties
    feats[::3] += rs.randn(*feats[::3].shape).astype(np.float32)
    trans = (rs.randint(-4, 5, size=(T, T)) * 0.5).astype(np.float32)
    trans[:, T - 2] = -10000.0
    trans[T - 1, :] = -10000.0
    lens = rs.randint(1, L + 1, size=B).astype(np.int64)
    lens[0], lens[1], lens[2] = L, 0, L + 3
    n = np.minimum(lens, L)
    valid = orc.length_mask(n, L)
    crf = _crf(trans)
    rand = rs.rand(B, L, T) < 0.3
    rand[np.arange(B)[:, None], np.arange(L)[None, :], rs.randint(0, T, size=(B, L))] = True
    gold = rs.randint(0, T, size=(B, L))
    onehot = np.eye(T, dtype=bool)[gold]
    want_r, _ = ref.crf_constrained_viterbi(feats, lens, trans, rand)
    try:
        for ns in (1, 2):
            _viterbi_seqs(ns)
            _, vit = crf._viterbi_decode(_t(feats), None, lengths=_t(lens))
            free = crf.constrained_decode(_t(feats), None, _t(np.ones_like(rand)), lengths=_t(lens))
            assert torch.equal(free, vit)
            got = crf.constrained_decode(_t(feats), None, _t(rand), lengths=_t(lens)).cpu().numpy()
            np.testing.assert_array_equal(got[valid], want_r[valid])
            b, t = np.nonzero(valid)
            assert rand[b, t, got[b, t]].all()
            got = crf.constrained_decode(_t(feats), None, _t(onehot.astype(np.uint8)), lengths=_t(lens)).cpu().numpy()
            np.testing.assert_array_equal(got[valid], gold[valid])
    finally:
        _viterbi_seqs(0)


def test_crf_rejects_bad_masks():
    feats, trans, lens, allowed = _mixed_case(7, B=6, L=5)
    crf = _crf(trans)
    f, ln = _t(feats), _t(lens)
    empty = allowed.copy()
    empty[0, 2] = False                                   # a valid position without any tag
    for bad in (_t(allowed.astype(np.float32)), _t(allowed[:, :4]), _t(allowed, 'cpu'), _t(empty)):
        with pytest.raises(ValueError):
            crf.partial_neg_log_likelihood_loss(f, None, bad, lengths=ln)
        with pytest.raises(ValueError):
            crf.constrained_decode(f, None, bad, lengths=ln)


# ---- the decompose models ---------------------------------------------------------------------------------------------
def _model(kind, farnn, loss_func, use_crf=1, seed=11):
    import re2nn_seq_b200 as r
    from re2nn_seq_b200 import synth
    S, R, C, B, L, V = 120, 72, 15, 300, 9, 400
    args = synth.make_args(farnn=farnn, use_crf=use_crf, update_nonlinear='tanh', beta=0.1, local_loss_func=loss_func)
    f = synth.make_decompose_factors(seed, V, S, R, C, 50, dtype=np.float32)
    x, lens, lab = synth.make_batch(seed + 1, B, L, V, C)
    torch.manual_seed(0)
    if kind == 'tok':
        m = r.FARNN_S_D_W_I_S(args=args, o_idx=0, **f)
        inp = x
    else:
        keep = ('S1', 'S2', 'C_output_mat', 'wildcard_mat', 'wildcard_output_vector', 'final_vector', 'start_vector')
        m = r.FARNN_S_SF(args=args, o_idx=0, is_cuda=True, priority_mat=None, **{k: f[k] for k in keep})
        inp = (np.random.RandomState(seed + 2).randn(B, L, R) * 0.3).astype(np.float32)
    if use_crf:
        with torch.no_grad():
            m.crf.transitions.copy_(torch.from_numpy(synth.crf_transitions(seed, m.C)))
    return m.cuda(), _t(inp), _t(lab), _t(lens)


def _grads(m):
    return {k: (None if p.grad is None else p.grad.detach().clone()) for k, p in m.named_parameters()}


MODELS = [(k, fa, lf) for k in ('tok', 'sf') for fa in (0, 2) for lf in ('CE', 'CE1')]


@pytest.mark.parametrize('kind,farnn,loss_func', MODELS)
def test_model_forward_partial(kind, farnn, loss_func):
    """Every label known: forward_local's CRF training loss and every parameter gradient.  None known: exactly zero."""
    from re2nn_seq_b200.crf import partial_allowed
    m, inp, lab, lens = _model(kind, farnn, loss_func)
    call = m.forward_local if kind == 'tok' else m.forward
    loss, _, _ = call(inp, lab, lens, train=True)
    loss.backward()
    want = _grads(m)
    m.zero_grad(set_to_none=True)
    got = m.forward_partial(inp, lens, partial_allowed(lab, m.C, lengths=lens))
    got.backward()
    assert rel_err(got.item(), loss.item()) < TOL
    checked = 0
    for k, g in _grads(m).items():
        if want[k] is None:
            assert g is None, k
            continue
        assert rel_err(g.cpu().numpy(), want[k].cpu().numpy()) < 1e-4, k
        checked += 1
    assert checked >= 3
    m.zero_grad(set_to_none=True)
    none = m.forward_partial(inp, lens, partial_allowed(torch.full_like(lab, -1), m.C))
    none.backward()
    assert none.item() == 0.0
    for k, g in _grads(m).items():
        assert g is None or (g == 0).all(), k


@pytest.mark.parametrize('kind,farnn,loss_func', MODELS)
def test_model_forward_constrained(kind, farnn, loss_func):
    """An all-true mask decodes what forward_local does (eager call and graph replay), under CE1 with a threshold that
    clamps column C-3; a one-hot mask of other tags decodes those tags (C-3 reported as o_idx under CE1)."""
    m, inp, lab, lens = _model(kind, farnn, loss_func)
    B = lens.shape[0]
    with torch.no_grad():
        sc = m.forward_scores(inp, lens)
        n = lens.cpu().numpy()
        L = int(n.max())
        valid = _t(orc.length_mask(n, L))
        if loss_func == 'CE1':
            m.args.threshold = float(sc[:, :, m.C - 3][valid].median())
        call = m.forward_local if kind == 'tok' else m.forward
        preds = [call(inp, lab, lens, train=False)[1] for _ in range(3)]   # eager, capture, replay
    pred = m.forward_constrained(inp, lens, torch.ones(B, L + 2, m.C, dtype=torch.bool, device='cuda'))
    assert pred.shape == (B, L)
    for p in preds:
        assert torch.equal(pred[valid], p), int((pred[valid] != p).sum())
    tags = torch.randint(0, m.C - 2, (B, L), generator=torch.Generator().manual_seed(1)).cuda()
    forced = m.forward_constrained(inp, lens, torch.nn.functional.one_hot(tags, m.C).bool())
    want = tags.clone()
    if loss_func == 'CE1':
        want[tags == m.C - 3] = m.o_idx
    assert torch.equal(forced[valid], want[valid])


def test_model_partial_errors():
    from re2nn_seq_b200.crf import partial_allowed
    m, inp, lab, lens = _model('tok', 0, 'CE', use_crf=0)
    for fn in (m.forward_partial, m.forward_constrained):
        with pytest.raises(NotImplementedError, match='CRF'):
            fn(inp, lens, partial_allowed(lab, 17))
    m, inp, lab, lens = _model('tok', 0, 'CE1')
    good = partial_allowed(lab, m.C, lengths=lens)
    empty = good.clone()
    empty[0, 0] = False
    for bad in (good.float(), good[:, :, :-1], empty):
        for fn in (m.forward_partial, m.forward_constrained):
            with pytest.raises(ValueError):
                fn(inp, lens, bad)


def test_model_partial_training_lowers_loss():
    """Twenty Adam steps on the partial loss with half of the tokens unknown lower it."""
    from re2nn_seq_b200.crf import partial_allowed
    m, inp, lab, lens = _model('tok', 0, 'CE1')
    hide = torch.rand(lab.shape, generator=torch.Generator().manual_seed(5)).cuda() < 0.5
    allowed = partial_allowed(torch.where(hide, torch.full_like(lab, -1), lab), m.C, lengths=lens)
    opt = torch.optim.Adam([p for p in m.parameters() if p.requires_grad], lr=1e-2)
    losses = []
    for _ in range(20):
        opt.zero_grad()
        loss = m.forward_partial(inp, lens, allowed)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert np.isfinite(losses).all()
    assert losses[-1] < losses[0], losses


def test_partial_ops_registered_cuda_only():
    from re2nn_seq_b200 import _lib
    for name in ('crf_partial_nll', 'crf_partial_nll_backward'):
        schema = str(getattr(_lib.tops, name).default._schema)
        assert schema.startswith('re2nn::' + name + '('), schema
    f, tr, ln, a = torch.zeros(2, 3, 5), torch.zeros(5, 5), torch.tensor([3, 2]), torch.ones(2, 3, 5, dtype=torch.bool)
    with pytest.raises((RuntimeError, NotImplementedError)):
        _lib.tops.crf_partial_nll(f, tr, ln, a, False)
