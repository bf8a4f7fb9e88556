"""GPU: the onehot recurrence and its backward (onehot.cu), max-product inference (maxprod.cu) and the batched
vector-matrix step (fst.cu) on every path they dispatch on, against plain float64 / fp32 references.

onehot_recurrence_kernel chooses (a) the cluster size: two CTAs per (sequence, direction) while 4 * B <= SMs, one
otherwise, or 1 / 2 / 4 forced through re2nn_debug_set_onehot_cluster (+8: four instead of eight rows in flight);
(b) 16-byte loads when S % 4 == 0 and the tensors are 16-byte aligned, scalar loads otherwise; (c) the sum or max
semiring.  Test IDs name those choices: c1 / c2 / c4 / auto, rows8 / rows4, vec16 / scalar, sum / max.  S = 1, 5, 13
leave some CTAs of a cluster without rows; 127-132 and 252-260 hit the tails of the 8- and 4-row unrolls and the
`j + 128 < S` split of the backward direction; 130 splits unevenly over four CTAs; 2964 is the shared-memory limit.

Bars:
- 0/1 automata (integer path counts < 2^24): bit-exact against the float64 reference, so bit-identical across
  cluster size, rows in flight and load width;
- real-valued, max semiring, none / relu: bit-exact against the fp32 restatement (one rounded product, an exact max,
  the same multiply order); tanh / relutanh: 1e-5 relative (max-norm) of float64;
- real-valued, sum semiring: 1e-5 relative (max-norm) of float64;
- onehot language_tensor gradients: 2e-5 relative (max-norm) of a float64 autograd restatement;
- max-product inference scores: 1e-5 relative of float64 orc.decompose_scores and of the differentiable dense form;
  decoded tags equal to the fp32 oracle's;
- batched_vecmat: sum within the summation-length bound (S + 1) u (|h| @ |T|) of float64; max bit-exact with
  torch.max's first-index argmax on data full of exact ties; gradients equal to float64 autograd on integer data."""
import contextlib
import functools

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import rel_err
from oracle import re2nn_oracle as orc

pytestmark = pytest.mark.gpu
NLS = ('none', 'relu', 'tanh', 'relutanh')
TOL = 1e-5
GRAD_TOL = 2e-5


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


@contextlib.contextmanager
def _onehot_path(nc, rows8=True):
    """Force the onehot cluster size (0 = chosen by batch size) and the rows in flight for one block."""
    from re2nn_seq_b200 import _lib
    _lib.check(_lib.fn['re2nn_debug_set_onehot_cluster'](nc + (0 if rows8 else 8)), 'debug_set_onehot_cluster')
    try:
        yield
    finally:
        _lib.check(_lib.fn['re2nn_debug_set_onehot_cluster'](0), 'debug_set_onehot_cluster')


def _lengths(rs, B, L):
    """Ragged lengths with a full-length row first, then 0 and 1 (as far as B allows)."""
    n = rs.randint(0, L + 1, size=B).astype(np.int64)
    n[0] = L
    n[1:3] = [0, 1][:max(0, min(2, B - 1))]
    return n


# ---- A. onehot forward ---------------------------------------------------------------------------------------------
V1 = 4      # vocabulary + pad token: few slices, so every step of every sequence streams one of the same four


@functools.lru_cache(maxsize=None)
def _fwd_case(S, B, L, kind):
    """Inputs of one forward case (numpy float32).  kind '01': a 0/1 rule automaton (o = 1); 'sum' / 'max':
    real-valued, scaled so the states stay O(1) under that semiring, with negated columns so relu has work."""
    from re2nn_seq_b200 import synth
    rs = np.random.RandomState(S * 31 + B * 7 + L + len(kind))
    if kind == '01':
        a = synth.make_onehot_automaton(S + B, V1 - 1, S, 5, lang_frac=0.7, dtype=np.float32)
        lang, W = a['language_tensor'], a['wildcard_mat']
        o, h0, hT = a['output_mat'].sum(0), a['start_vector'], a['final_vector']
    else:
        scale = 1.0 / S if kind == 'sum' else 1.0
        lang = (rs.uniform(-0.25, 2.25, (V1, S, S)) * scale).astype(np.float32)
        W = (rs.uniform(-0.1, 0.1, (S, S)) * scale).astype(np.float32)
        neg = rs.rand(S) < 0.25
        lang[:, :, neg] *= -1
        o = rs.uniform(0.5, 1.2, S).astype(np.float32)
        h0 = rs.uniform(0.2, 1.0, S).astype(np.float32)
        hT = rs.uniform(0.2, 1.0, S).astype(np.float32)
    x = rs.randint(0, V1 - 1, size=(B, L)).astype(np.int64)
    n = _lengths(rs, B, L)
    x[np.arange(L)[None, :] >= n[:, None]] = V1 - 1
    T = (lang + W).astype(np.float32)
    dev = {k: _t(v) for k, v in dict(lang=lang, W=W, T=T, o=o, h0=h0, hT=hT, x=x, n=n).items()}
    return dict(lang=lang, W=W, T=T, o=o, h0=h0, hT=hT, x=x, n=n, dev=dev)


def _states_ref(c, nl, maxp, dtype):
    """alpha, beta B x L x S in the kernels' layout, all L steps (pad rows as the reference computes them): the
    recurrence of orc.onehot_scores.  alpha[b, t] = state after token t; beta[b, t] = backward state at position t + 1
    (hT at t = n - 1)."""
    T = c['T'].astype(dtype)
    o, h0, hT, x, n = c['o'].astype(dtype), c['h0'].astype(dtype), c['hT'].astype(dtype), c['x'], c['n']
    B, L = x.shape
    semi = orc.semiring_max if maxp else orc.semiring_sum
    bx = orc.reverse_rows(x, n)
    hf, hb = np.repeat(h0[None], B, 0), np.repeat(hT[None], B, 0)
    fwd, bwd = np.zeros((B, L, len(o)), dtype), np.zeros((B, L, len(o)), dtype)
    for i in range(L):
        hf = orc.nonlinear(semi(hf, T[x[:, i]]) * o, nl)
        fwd[:, i] = hf
        hb = orc.nonlinear(semi(hb * o, T[bx[:, i]].transpose(0, 2, 1)), nl)
        bwd[:, i] = hb
    beta = orc.reverse_rows(np.concatenate([np.repeat(hT[None, None], B, 0), bwd], 1), n + 1)[:, 1:]
    return fwd, np.ascontiguousarray(beta)


@functools.lru_cache(maxsize=None)
def _fwd_refs(S, B, L, kind, nl, maxp):
    c = _fwd_case(S, B, L, kind)
    r64 = _states_ref(c, nl, maxp, np.float64)
    r32 = _states_ref(c, nl, maxp, np.float32) if maxp and nl in ('none', 'relu') and kind != '01' else None
    return r64, r32


def _check_states(got, c, key, nl, maxp, full_pad, what):
    """Kernel alpha / beta against the bar of their data kind; rows t >= n must stay zero unless full_pad."""
    S, B, L, kind = key
    r64, r32 = _fwd_refs(S, B, L, kind, nl, maxp)
    pad = ~orc.length_mask(c['n'], L)
    for g, w64, w32, name in zip(got, r64, r32 or (None, None), ('alpha', 'beta')):
        g = g.cpu().numpy()
        w64 = w64.copy()
        if w32 is not None:
            w32 = w32.copy()
        if not full_pad:
            w64[pad] = 0
            if w32 is not None:
                w32[pad] = 0
        msg = '%s %s (%s, nl=%s, full_pad=%d)' % (what, name, kind, nl, full_pad)
        if kind == '01':
            assert np.abs(w64).max() < 2 ** 24
            np.testing.assert_array_equal(g, w64.astype(np.float32), err_msg=msg)
        elif w32 is not None:
            np.testing.assert_array_equal(g, w32, err_msg=msg)
        else:
            assert rel_err(g, w64) < TOL, msg


def _run_fwd(c, nl, maxp, full_pad, T=None, presummed=True):
    from re2nn_seq_b200 import ops
    d = c['dev']
    L = c['x'].shape[1]
    if presummed:
        return ops.onehot_recurrence(d['x'], d['n'], L, d['T'] if T is None else T, None, d['o'], d['h0'], d['hT'], nl,
                                     maxp, full_pad, presummed=True)
    return ops.onehot_recurrence(d['x'], d['n'], L, d['lang'], d['W'], d['o'], d['h0'], d['hT'], nl, maxp, full_pad)


def _sweep(key, maxp, what, **kw):
    """Every data kind, nonlinearity and full_pad of one (S, B, L) through the current path."""
    S, B, L = key
    for kind in ('01', 'max' if maxp else 'sum'):
        c = _fwd_case(S, B, L, kind)
        for nl in (('none', 'relu') if kind == '01' else NLS):
            for full_pad in (False, True):
                got = _run_fwd(c, nl, maxp, full_pad, **kw)
                torch.cuda.synchronize()
                _check_states(got, c, (S, B, L, kind), nl, maxp, full_pad, what)


FWD_S = [1, 5, 13, 127, 128, 129, 130, 132, 252, 256, 260, 300, 1024]
PATHS = [(1, True), (1, False), (2, True), (2, False), (4, True), (4, False)]


def _sid(S):
    return 'S%d-%s' % (S, 'vec16' if S % 4 == 0 else 'scalar')


@pytest.mark.parametrize('semiring', ['sum', 'max'])
@pytest.mark.parametrize('S', FWD_S, ids=_sid)
@pytest.mark.parametrize('nc,rows8', PATHS, ids=['c%d-%s' % (nc, 'rows8' if r else 'rows4') for nc, r in PATHS])
def test_onehot_forward_forced_path(nc, rows8, S, semiring):
    """ops.onehot_recurrence with the cluster size and rows in flight forced, B = 5 with lengths L, 0, 1 and ragged."""
    with _onehot_path(nc, rows8):
        _sweep((S, 5, 6), semiring == 'max', 'c%d rows8=%d' % (nc, rows8))


@pytest.mark.parametrize('semiring', ['sum', 'max'])
@pytest.mark.parametrize('S', [13, 129, 300], ids=_sid)
@pytest.mark.parametrize('side', ['auto-c2', 'auto-c1'])
def test_onehot_forward_auto_cluster(side, S, semiring):
    """The batch-size heuristic on both sides of its threshold: B = SMs / 4 still runs on CTA pairs, one more sequence
    runs on single CTAs.  Also the model: FARNN_S_O_I_S.forward_score on a 0/1 automaton is bit-exact against
    orc.onehot_scores in float64."""
    import re2nn_seq_b200 as r
    from re2nn_seq_b200 import synth
    B = _sms() // 4 + (1 if side == 'auto-c1' else 0)
    maxp = semiring == 'max'
    with _onehot_path(0):
        _sweep((S, B, 6), maxp, side)
        args = synth.make_args(method='onehot', rand_constant=0.0, train_mode=semiring, update_nonlinear='relu')
        a = synth.make_onehot_automaton(S, 40, S, 9, lang_frac=0.3, dtype=np.float64)
        x, lens, lab = synth.make_batch(S, B, 7, 40, 9)
        m = r.FARNN_S_O_I_S(a['language_tensor'], a['output_mat'], a['wildcard_mat'], a['output_wildcard_vector'],
                            a['final_vector'], a['start_vector'], None, args, 0, True)
        with torch.no_grad():
            sc = m.forward_score(_t(x), _t(lab), _t(lens)).cpu().numpy()
    p = {k: v for k, v in a.items() if k != 'language_rows'}
    p.update(h0=a['start_vector'], hT=a['final_vector'])
    want = orc.onehot_scores(p, x, lens, args)
    assert np.abs(want).max() < 2 ** 24
    np.testing.assert_array_equal(sc, want.astype(np.float32))


@pytest.mark.parametrize('semiring', ['sum', 'max'])
@pytest.mark.parametrize('nc', [1, 2, 4], ids=['c1', 'c2', 'c4'])
def test_onehot_forward_smem_limit(nc, semiring):
    """S = 2964 fills the 220 KB of dynamic shared memory ((3 + 16) S floats); S = 2965 is refused before launch."""
    from re2nn_seq_b200 import ops
    S, B, L = 2964, 3, 3
    maxp = semiring == 'max'
    with _onehot_path(nc):
        for kind in ('01', semiring):
            c = _fwd_case(S, B, L, kind)
            got = _run_fwd(c, 'none', maxp, True)
            _check_states(got, c, (S, B, L, kind), 'none', maxp, True, 'S=2964 c%d' % nc)
    S = 2965
    z = torch.zeros((1, S, S), device='cuda')
    v = torch.ones((S,), device='cuda')
    x = torch.zeros((1, 1), dtype=torch.int64, device='cuda')
    with pytest.raises(RuntimeError, match='too large'):
        ops.onehot_recurrence(x, x[0] + 1, 1, z, None, v, v, v, 'none', maxp, False, presummed=True)
        torch.cuda.synchronize()


@pytest.mark.parametrize('semiring', ['sum', 'max'])
@pytest.mark.parametrize('S', [128, 260, 1024], ids=lambda S: 'S%d-offset1-scalar' % S)
def test_onehot_forward_misaligned(S, semiring):
    """A 16-byte-eligible S through a language tensor offset by one float: the scalar path, same results."""
    maxp = semiring == 'max'
    for kind in ('01', semiring):
        c = _fwd_case(S, 5, 6, kind)
        buf = torch.empty(c['T'].size + 1, device='cuda')
        Tm = buf[1:].view(c['T'].shape)
        Tm.copy_(c['dev']['T'])
        assert Tm.data_ptr() % 16 != 0
        for nl in (('none', 'relu') if kind == '01' else NLS):
            for full_pad in (False, True):
                for nc in (1, 2):
                    with _onehot_path(nc):
                        got = _run_fwd(c, nl, maxp, full_pad, T=Tm)
                        _check_states(got, c, (S, 5, 6, kind), nl, maxp, full_pad, 'offset-1 c%d' % nc)
                        if kind == '01':
                            ref = _run_fwd(c, nl, maxp, full_pad)
                            for g, w in zip(got, ref):
                                assert torch.equal(g, w)


@pytest.mark.parametrize('semiring', ['sum', 'max'])
@pytest.mark.parametrize('S', [13, 128, 130, 300], ids=_sid)
def test_onehot_forward_separate_W(S, semiring):
    """The C-ABI call with a separate W (language + W formed per load) is bit-identical to the pre-summed call."""
    maxp = semiring == 'max'
    c = _fwd_case(S, 5, 6, semiring)
    for nc in (1, 2):
        with _onehot_path(nc):
            for nl in NLS:
                for full_pad in (False, True):
                    a = _run_fwd(c, nl, maxp, full_pad, presummed=False)
                    b = _run_fwd(c, nl, maxp, full_pad)
                    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]), (nc, nl, full_pad)


# ---- B. onehot backward --------------------------------------------------------------------------------------------
def _onehot_model(S, loss, prio, nl, seed):
    """FARNN_S_O_I_S with real-valued transitions and output matrix, V = 2 (three slices: many atomics per slice)."""
    import re2nn_seq_b200 as r
    from re2nn_seq_b200 import synth
    rs = np.random.RandomState(seed)
    C = 4
    args = synth.make_args(method='onehot', rand_constant=0.0, local_loss_func=loss, use_priority=prio,
                           update_nonlinear=nl, margin=0.3)
    lang = rs.uniform(-0.25, 2.25, (3, S, S)) / S
    lang[:, :, rs.rand(S) < 0.25] *= -1
    W = rs.uniform(-0.1, 0.1, (S, S)) / S
    outm = rs.uniform(0.0, 2.0 / (C + 1), (C + 1, S))
    outw = rs.uniform(0.0, 0.3, S)
    pm = np.eye(C + 1) + 0.1 * rs.randn(C + 1, C + 1) if prio else None
    m = r.FARNN_S_O_I_S(lang, outm, W, outw, rs.uniform(0.2, 1.0, S), rs.uniform(0.2, 1.0, S), pm, args, 0, True)
    if prio:
        with torch.no_grad():
            m.priority_layer.priority_bias.copy_(torch.from_numpy(0.1 * rs.randn(C + 1)))
    return m, args


def _onehot_scores64(p, x, n, nl, ce1, prio):
    """FARNN_S_O_I_S.forward_score in float64 autograd: the recurrence of orc.onehot_scores over all L steps."""
    T = p['language_tensor'] + p['wildcard_mat']
    o = p['output_mat'].sum(0) + (0 if ce1 else p['output_wildcard_vector'])
    B, L = x.shape
    S = o.shape[0]
    pos = torch.arange(L)[None, :]
    bx = x.gather(1, torch.where(pos < n[:, None], n[:, None] - 1 - pos, pos))
    act = {'none': lambda v: v, 'relu': torch.relu, 'tanh': torch.tanh, 'relutanh': lambda v: torch.tanh(torch.relu(v))}[nl]
    hf, hb = p['h0'].expand(B, S), p['hT'].expand(B, S)
    fw, bw = [], []
    for i in range(L):
        hf = act(torch.einsum('bs,bsj->bj', hf, T[x[:, i]]) * o)
        hb = act(torch.einsum('bj,bsj->bs', hb * o, T[bx[:, i]]))
        fw.append(hf)
        bw.append(hb)
    full = torch.cat([p['hT'].expand(B, 1, S), torch.stack(bw, 1)], 1)
    beta = full.gather(1, torch.where(pos < n[:, None], n[:, None] - 1 - pos, pos + 1)[:, :, None].expand(B, L, S))
    sc = torch.einsum('bls,cs->blc', torch.stack(fw, 1) * beta, p['output_mat'])
    if prio:
        sc = sc @ p['priority_layer.priority_mat'] + p['priority_layer.priority_bias']
    return sc


def _grad_case(m, args, x, lab, n, mode, wts, nl):
    """(loss, reference loss, language_tensor.grad, reference gradient) of the CUDA path and the float64 reference for
    one way of taking the loss; mode 'score' returns the scores in place of the losses."""
    m.language_tensor.grad = None
    xt, lt, nt = _t(x), _t(lab), _t(n)
    if mode == 'score':
        scores = m.forward_score(xt, lt, nt)
        loss = (scores * _t(wts)).sum()
    else:
        m.full_pad = mode == 'local_full_pad'
        try:
            loss, _, _ = m.forward_local(xt, lt, nt, train=True)
        finally:
            m.full_pad = False
    loss.backward()
    got = m.language_tensor.grad.cpu().numpy()
    p = {k: v.detach().cpu().double() for k, v in m.state_dict().items()}
    p['language_tensor'].requires_grad_(True)
    sc = _onehot_scores64(p, torch.from_numpy(x), torch.from_numpy(n), nl, args.local_loss_func == 'CE1',
                          bool(args.use_priority))
    if mode == 'score':
        want_loss = (sc * torch.from_numpy(wts).double()).sum()
    else:
        mask = torch.from_numpy(orc.length_mask(n, x.shape[1]))
        flat, y = sc[mask], torch.from_numpy(lab)[mask]
        want_loss = (F.multi_margin_loss(flat, y, margin=args.margin) if args.local_loss_func == 'ML'
                     else F.cross_entropy(flat, y))
    want_loss.backward()
    if mode == 'score':            # a signed weighted sum cancels: compare what it sums
        return scores.detach().cpu().numpy(), sc.detach().numpy(), got, p['language_tensor'].grad.numpy()
    return loss.item(), want_loss.item(), got, p['language_tensor'].grad.numpy()


@pytest.mark.parametrize('prio', [0, 1], ids=['noprio', 'prio'])
@pytest.mark.parametrize('loss', ['CE1', 'CE', 'ML'])
@pytest.mark.parametrize('S', [11, 33, 128, 300])
def test_onehot_backward_vs_float64(S, loss, prio):
    """d loss / d language_tensor through onehot_backward_kernel for every nonlinearity, three ways: forward_local
    without and with full_pad, and a weighted sum over every position of forward_score (pad rows included, so the
    backward direction's pad steps and the state after token 0 carry gradient).  B = 7 with lengths L, 0, 1, L and
    ragged; three transition slices, so many atomics land on the same slice."""
    B, L = 7, 9
    rs = np.random.RandomState(S + 3 * prio)
    x = rs.randint(0, 2, size=(B, L)).astype(np.int64)
    n = _lengths(rs, B, L)
    n[3] = L
    x[np.arange(L)[None, :] >= n[:, None]] = 2
    lab = rs.randint(0, 5, size=(B, L)).astype(np.int64)
    wts = rs.randn(B, L, 5)
    for nl in NLS:
        m, args = _onehot_model(S, loss, prio, nl, S)
        for mode in ('local', 'local_full_pad', 'score'):
            l, wl, g, w = _grad_case(m, args, x, lab, n, mode, wts, nl)
            what = 'S=%d %s prio=%d nl=%s %s' % (S, loss, prio, nl, mode)
            assert rel_err(l, wl) < TOL, what
            assert rel_err(g, w) < GRAD_TOL, '%s: rel err %.3e' % (what, rel_err(g, w))


@pytest.mark.parametrize('full_pad,S_max', [(False, 2964), (True, 2816)], ids=['full_pad0-S2964', 'full_pad1-S2816'])
def test_onehot_backward_smem_limit(full_pad, S_max):
    """The backward keeps (3 + 16) S floats in shared memory, one more S under full_pad (the recomputed state after
    token 0): the largest S runs and matches float64, one more is refused.  The bar is 6e-5, not 2e-5: every state and
    state gradient here is an fp32 sum of ~2900 signed terms (measured on a B200 at 1000 W: 3.5e-5 at S = 2964 without
    full_pad, where the elements agree to 4-5 digits, i.e. rounding, not a misrouted term)."""
    B, L = 2, 2
    x = np.array([[0, 1], [1, 2]], dtype=np.int64)
    n = np.array([2, 1], dtype=np.int64)
    lab = np.array([[1, 2], [3, 0]], dtype=np.int64)
    wts = np.random.RandomState(0).randn(B, L, 5)
    mode = 'score' if full_pad else 'local'
    m, args = _onehot_model(S_max, 'CE', 0, 'tanh', 1)
    _, _, g, w = _grad_case(m, args, x, lab, n, mode, wts, 'tanh')
    assert rel_err(g, w) < 6e-5, rel_err(g, w)
    del m
    if not full_pad:
        return                                   # S = 2965 is refused by the forward already (test above)
    m, args = _onehot_model(S_max + 1, 'CE', 0, 'tanh', 1)
    with pytest.raises(RuntimeError, match='too large'):
        _grad_case(m, args, x, lab, n, mode, wts, 'tanh')


# ---- C. max-product inference --------------------------------------------------------------------------------------
_RENAME = {'embedding.weight': 'embedding', 'priority_layer.priority_mat': 'priority_mat',
           'priority_layer.priority_bias': 'priority_bias'}


def _maxprod_model(S, R, farnn, vmode, nl, B, L, seed):
    import re2nn_seq_b200 as r
    from re2nn_seq_b200 import synth
    args = synth.make_args(farnn=farnn, use_crf=0, update_nonlinear=nl, train_mode='max', beta=0.1,
                           local_loss_func='CE')
    f = synth.make_decompose_factors(seed, 30, S, R, 6, 16, lang_frac=0.5, dtype=np.float32)
    x, lens, lab = synth.make_batch(seed + 1, B, L, 30, 6)
    if B > 1:
        lens[1] = 1
    torch.manual_seed(seed)
    if vmode == 'token':
        m = r.FARNN_S_D_W_I_S(args=args, o_idx=0, **f)
        inp = x
    else:
        keep = ('S1', 'S2', 'C_output_mat', 'wildcard_mat', 'wildcard_output_vector', 'final_vector', 'start_vector')
        m = r.FARNN_S_SF(args=args, o_idx=0, is_cuda=True, priority_mat=None, **{k: f[k] for k in keep})
        inp = (np.random.RandomState(seed).randn(B, L, R) / np.sqrt(R) * 3).astype(np.float32)
    with torch.no_grad():
        for k in ('Wss1', 'Wrs1', 'Wss2', 'Wrs2'):
            if hasattr(m, k):
                getattr(m, k).mul_(0.05)
        if farnn:
            m.bs1.fill_(0.3)
        if farnn == 2:
            m.bs2.fill_(-0.1)
    return m.cuda(), args, inp, lens, lab


def _maxprod_check(S, R, farnn, vmode, B, L, nls=NLS):
    for nl in nls:
        m, args, inp, lens, lab = _maxprod_model(S, R, farnn, vmode, nl, B, L, S + R + farnn)
        it, lt, nt = _t(inp), _t(lab), _t(lens)
        got = {}
        with torch.no_grad():
            for fp in (False, True):
                m.full_pad = fp
                got[fp] = m.forward_scores(it, nt).cpu().numpy()
            m.full_pad = False
            if vmode == 'token':
                _, pred, _ = m.forward_local(it, lt, nt, train=False)
            else:
                _, pred, _ = m(it, lt, nt, False)
        with torch.enable_grad():
            dense = m.forward_scores(it, nt).detach().cpu().numpy()           # model_fst.ifst_decompose_max_scores
        sd = {_RENAME.get(k, k): v.detach().cpu().numpy() for k, v in m.state_dict().items()}
        p64 = {k: v.astype(np.float64) for k, v in sd.items()}
        x = inp if vmode == 'token' else np.zeros(inp.shape[:2], np.int64)
        dv = None if vmode == 'token' else inp
        want, _, _ = orc.decompose_scores(p64, x, lens, args, dense_v=None if dv is None else dv.astype(np.float64))
        mask = orc.length_mask(lens, int(lens.max()))
        what = 'S=%d R=%d farnn=%d %s nl=%s' % (S, R, farnn, vmode, nl)
        assert rel_err(got[False][mask], want[mask]) < TOL, what
        assert rel_err(got[True], want) < TOL, what + ' full_pad'
        assert rel_err(got[True], dense) < TOL, what + ' vs dense form'
        _, o_pred, _, _ = orc.decompose_forward_local(sd, x, lab, lens, args, 0, False, dense_v=dv)
        np.testing.assert_array_equal(pred.cpu().numpy(), o_pred, err_msg=what)


MAXP_SR = [(5, 3), (33, 40), (96, 72), (160, 600), (5, 600), (160, 3)]


@pytest.mark.parametrize('vmode', ['token', 'dense'])
@pytest.mark.parametrize('farnn', [0, 1, 2], ids=['farnn0', 'farnn1', 'farnn2'])
@pytest.mark.parametrize('S,R', MAXP_SR, ids=['S%d-R%d' % sr for sr in MAXP_SR])
def test_maxprod_inference(S, R, farnn, vmode):
    """decompose_max_kernel under no_grad (FARNN_S_D_W_I_S / FARNN_S_SF, train_mode='max'), every nonlinearity,
    full_pad 0 and 1: S > 32 gives a warp several output blocks, R > 512 makes the v load loop."""
    big = S * S * R > 1_000_000
    _maxprod_check(S, R, farnn, vmode, 4 if big else 6, 5 if big else 6)


def test_maxprod_smem_limit():
    """(4 + 16) S + R floats of shared memory: S = 33 with the largest R that fits 220 KB runs (B = 1, L = 2); one more
    R is refused."""
    S = 33
    R = 220 * 1024 // 4 - 20 * S
    _maxprod_check(S, R, 0, 'token', 1, 2, nls=('tanh',))
    m, args, inp, lens, lab = _maxprod_model(S, R + 1, 0, 'token', 'tanh', 1, 2, 0)
    with torch.no_grad(), pytest.raises(RuntimeError, match='too large'):
        m.forward_scores(_t(inp), _t(lens))
        torch.cuda.synchronize()


# ---- D. batched_vecmat ---------------------------------------------------------------------------------------------
def _vm_data(S, B, kind):
    """kind 'real': normal h and T; 'int': small integers (exact ties everywhere); 'ties_inf': the integers plus, with
    B >= 3, whole -inf rows and columns of T[2] under a positive h[2].  With B >= 3, h[1] = 0."""
    rs = np.random.RandomState(S * 3 + B)
    if kind == 'real':
        h = rs.randn(B, S).astype(np.float32)
        T = rs.randn(B, S, S).astype(np.float32)
    else:
        h = rs.randint(-3, 4, size=(B, S)).astype(np.float32)
        T = rs.randint(-3, 4, size=(B, S, S)).astype(np.float32)
    if B >= 3:
        h[1] = 0
        if kind == 'ties_inf':
            h[2] = rs.randint(1, 4, size=S)
            T[2, :, rs.rand(S) < 0.3] = -np.inf
            T[2, rs.rand(S) < 0.3, :] = -np.inf
    return torch.from_numpy(h), torch.from_numpy(T)


def _chunks(B, S):
    step = max(1, (1 << 25) // (S * S))
    return [(b, min(B, b + step)) for b in range(0, B, step)]


VM_CASES = [(S, B) for S in (1, 7, 31, 32, 33, 255, 256, 257, 1000) for B in (1, 3, 150)] + [(12288, 1)]


@pytest.mark.parametrize('semiring', ['sum', 'max'])
@pytest.mark.parametrize('trans', [False, True], ids=['lanes-along-s', 'transposed-warp-per-row'])
@pytest.mark.parametrize('S,B', VM_CASES, ids=['S%d-B%d' % c for c in VM_CASES])
def test_batched_vecmat(S, B, trans, semiring):
    """ops.batched_vecmat (out[b,s] = (+|max)_j h[b,j] T[b,j,s], or T[b,s,j] transposed) against torch on the CPU: the
    sum within (S + 1) u (|h| @ |T|) of float64 (any summation order of S products); the max bit-exact, its argmax
    torch.max's first maximal index."""
    from re2nn_seq_b200 import ops
    maxp = semiring == 'max'
    h, T = _vm_data(S, B, 'ties_inf' if maxp else 'real')
    hd, Td = h.cuda(), T.cuda()
    out, idx = ops.batched_vecmat(hd, Td, trans, maxp)
    out = out.cpu()
    idx = idx.cpu().long() if maxp else None
    u = 2.0 ** -24
    gam = (S + 1) * u / (1 - (S + 1) * u)
    for b0, b1 in _chunks(B, S):
        Tb = T[b0:b1].transpose(1, 2) if trans else T[b0:b1]           # [b, j, s]
        hb = h[b0:b1]
        if maxp:
            v, i = (hb[:, :, None] * Tb).max(1)
            assert torch.equal(out[b0:b1], v), (b0, b1)
            assert torch.equal(idx[b0:b1], i), (b0, b1)
        else:
            want = torch.bmm(hb.double()[:, None], Tb.double())[:, 0]
            bound = torch.bmm(hb.abs().double()[:, None], Tb.abs().double())[:, 0] * gam
            assert ((out[b0:b1].double() - want).abs() <= bound).all(), (b0, b1)
    if S * S * B > (1 << 25):
        return
    # gradients of model_fst.vecmat against float64 autograd of the same expression: exact on integer data (ties and a
    # zero h included; the max gradient follows the first maximal source, as torch.max's does)
    from re2nn_seq_b200 import model_fst
    h, T = _vm_data(S, B, 'int')
    hg, Tg = h.cuda().requires_grad_(True), T.cuda().requires_grad_(True)
    dout = torch.from_numpy(np.random.RandomState(S).randint(-2, 3, size=(B, S)).astype(np.float32))
    model_fst.vecmat(hg, Tg, trans, maxp).backward(dout.cuda())
    h64, T64 = h.double().requires_grad_(True), T.double().requires_grad_(True)
    Tt = T64.transpose(1, 2) if trans else T64
    prod = h64[:, :, None] * Tt
    ref = prod.max(1)[0] if maxp else prod.sum(1)
    ref.backward(dout.double())
    np.testing.assert_array_equal(hg.grad.cpu().numpy(), h64.grad.numpy())
    np.testing.assert_array_equal(Tg.grad.cpu().numpy(), T64.grad.numpy())


def test_batched_vecmat_refuses_large_S():
    """S floats of h live in 48 KB of shared memory: S = 12289 is refused."""
    from re2nn_seq_b200 import ops
    h = torch.zeros((1, 12289), device='cuda')
    for maxp in (False, True):
        with pytest.raises(RuntimeError, match='too large'):
            ops.batched_vecmat(h, torch.zeros((1,), device='cuda'), False, maxp)
