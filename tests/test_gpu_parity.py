"""GPU: CUDA path (through the C-ABI) vs the reference's golden fixtures and the oracle.

Tolerances (north_star): decoded tags / Viterbi paths bit-exact; scores, losses, gradients within
1e-5 relative in fp32 (rel = max|a-b| / max|b| over the tensor)."""
import numpy as np
import pytest
import torch

from conftest import golden_files
from helpers import args_of, build_module, golden_grads, load_golden, oracle_gradient_errors, oracle_params, rel_err
from oracle import re2nn_oracle as orc

pytestmark = pytest.mark.gpu
TOL = 1e-5
GRAD_TOL = 2e-5


def _t(a, dev='cuda'):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


DEC = [n for n in golden_files('dec_') + golden_files('sf_')]


@pytest.mark.parametrize('name', DEC)
def test_decompose_golden(name):
    z, meta = load_golden(name)
    m = build_module(name, z, meta).cuda()
    x, lab, lens = _t(z['x']), _t(z['labels']), _t(z['lengths'])
    inp = _t(z['dense_v']) if meta['kind'] == 'sf' else x
    re_tags = _t(z['re_tags']) if 're_tags' in z.files else None
    with torch.no_grad():
        scores = m.forward_scores(inp, lens)
        if meta['kind'] == 'sf':
            loss, pred, true = m(inp, lab, lens, True)
        else:
            loss, pred, true = m.forward_local(inp, lab, lens, train=True, re_tags=re_tags)
        m.full_pad = True                                   # reference semantics at pad positions
        full = m.forward_scores(inp, lens).cpu().numpy()
        m.full_pad = False
    assert rel_err(full, z['all_scores']) < TOL            # every position, pads included
    L = int(z['lengths'].max())
    mask = orc.length_mask(z['lengths'], L)
    got = scores.cpu().numpy()
    ref = z['all_scores']
    assert rel_err(got[mask], ref[mask]) < TOL
    assert rel_err(loss.item(), z['loss']) < TOL
    np.testing.assert_array_equal(pred.cpu().numpy(), z['pred'])
    np.testing.assert_array_equal(true.cpu().numpy(), z['true'])


@pytest.mark.parametrize('name', golden_files('one_'))
def test_onehot_golden(name):
    z, meta = load_golden(name)
    m = build_module(name, z, meta)
    x, lab, lens = torch.from_numpy(z['x']), torch.from_numpy(z['labels']), torch.from_numpy(z['lengths'])   # CPU in
    with torch.no_grad():
        scores = m.forward_score(x, lab, lens)
        loss, pred, true = m.forward_local(x, lab, lens, train=True)
        re_pred, re_scores = m.forward_RE(x, lab, lens)
    assert scores.device.type == 'cpu' and pred.device.type == 'cpu'          # results return on the caller's device
    if meta['flags']['rand_constant'] == 0:
        np.testing.assert_array_equal(scores.numpy(), z['all_scores'])          # exact path counts, pads included
    assert rel_err(scores.numpy(), z['all_scores']) < TOL                       # pad positions included
    assert rel_err(loss.item(), z['loss']) < TOL
    np.testing.assert_array_equal(pred.numpy(), z['pred'])
    np.testing.assert_array_equal(true.numpy(), z['true'])
    np.testing.assert_array_equal(re_pred.numpy(), z['re_pred'])
    assert rel_err(re_scores.numpy(), z['re_scores']) < TOL
    flat = orc.flatten_rows(z['all_scores'], z['lengths'])
    np.testing.assert_array_equal(m.local_decode(torch.from_numpy(flat)).numpy(), z['pred'])


@pytest.mark.parametrize('name', golden_files('crf_'))
def test_crf_golden(name):
    import re2nn_seq_b200 as r
    z, meta = load_golden(name)
    crf = r.CRF(meta['tagset'], True).cuda()
    with torch.no_grad():
        crf.transitions.copy_(_t(z['transitions']))
    feats = _t(z['feats']).requires_grad_(True)
    lens = z['lengths']
    mask = _t(orc.length_mask(lens, z['feats'].shape[1]))
    loss = crf.neg_log_likelihood_loss(feats, mask, _t(z['tags']))
    assert rel_err(loss.item(), z['loss']) < TOL
    _, path = crf._viterbi_decode(feats.detach(), mask)
    np.testing.assert_array_equal(path.cpu().numpy(), z['path'])                # pad quirks included
    loss.backward()
    assert rel_err(feats.grad.cpu().numpy(), z['g_feats']) < GRAD_TOL
    assert rel_err(crf.transitions.grad.cpu().numpy(), z['g_transitions']) < GRAD_TOL


def _random_decompose(seed, V, S, R, C, D, B, Lmax, **flags):
    from re2nn_seq_b200 import synth
    import re2nn_seq_b200 as r
    args = synth.make_args(**flags)
    f = synth.make_decompose_factors(seed, V, S, R, C, D, dtype=np.float32)
    x, lens, lab = synth.make_batch(seed + 1, B, Lmax, V, C)
    torch.manual_seed(seed)
    m = r.FARNN_S_D_W_I_S(args=args, o_idx=0, **f)
    with torch.no_grad():
        if args.use_crf:
            m.crf.transitions.copy_(torch.from_numpy(synth.crf_transitions(seed, m.C)))
        if args.farnn:
            for n in ('Wss1', 'Wrs1', 'Wss2', 'Wrs2'):
                if hasattr(m, n):
                    getattr(m, n).mul_(0.05)
            m.bs1.fill_(0.3)
            if hasattr(m, 'bs2'):
                m.bs2.fill_(-0.1)
    return m.cuda(), args, x, lens, lab


@pytest.mark.parametrize('farnn,crf', [(0, 1), (2, 1), (1, 0)])
def test_decompose_cfg2_shapes_vs_oracle(farnn, crf):
    """SNIPS-shaped factors (S=300, R=200, C=72, D=100) on a batch the oracle finishes in seconds."""
    m, args, x, lens, lab = _random_decompose(5, 2000, 300, 200, 72, 100, 96, 35, farnn=farnn, use_crf=crf,
                                              update_nonlinear='tanh', beta=0.1)
    with torch.no_grad():
        scores = m.forward_scores(_t(x), _t(lens)).cpu().numpy()
        loss, pred, true = m.forward_local(_t(x), _t(lab), _t(lens), train=True)
    sd = {k: v.detach().cpu().numpy() for k, v in m.state_dict().items()}
    z = {'p.' + k: v for k, v in sd.items()}

    class _Z(dict):
        files = property(lambda self: list(self.keys()))
    p32 = oracle_params(_Z(z), np.float32)
    p64 = oracle_params(_Z(z), np.float64)
    o_loss, o_pred, o_true, o_scores = orc.decompose_forward_local(p32, x, lab, lens, args, 0, True)
    t_scores, _, _ = orc.decompose_scores(p64, x, lens, args)
    mask = orc.length_mask(lens, 35)
    assert rel_err(scores[mask], t_scores[mask]) < TOL                # vs the float64 truth
    assert rel_err(scores[mask], o_scores[mask]) < TOL                # vs the fp32 restatement
    assert rel_err(loss.item(), o_loss) < TOL
    np.testing.assert_array_equal(true.cpu().numpy(), o_true)
    mism = int((pred.cpu().numpy() != o_pred).sum())
    assert mism == 0, 'decoded tags differ at %d of %d positions' % (mism, len(o_pred))


@pytest.mark.parametrize('name', DEC)
def test_decompose_gradients_golden(name):
    """loss.backward() through the CUDA backward vs the reference's autograd gradients (train_mode = 'max' included:
    its gradient follows the argmax saved by re2nn_batched_vecmat)."""
    z, meta = load_golden(name)
    m = build_module(name, z, meta).cuda()
    x, lab, lens = _t(z['x']), _t(z['labels']), _t(z['lengths'])
    if meta['kind'] == 'sf':
        loss, _, _ = m(_t(z['dense_v']), lab, lens, True)
    else:
        re_tags = _t(z['re_tags']) if 're_tags' in z.files else None      # KD / PR: scores at pads feed the loss
        loss, _, _ = m.forward_local(x, lab, lens, train=True, re_tags=re_tags)
    assert rel_err(loss.item(), z['loss']) < TOL
    loss.backward()
    gold = golden_grads(z)
    params = dict(m.named_parameters())
    assert gold, 'fixture without gradients'
    for k, ref in gold.items():
        g = params[k].grad
        assert g is not None, 'no gradient for ' + k
        if np.abs(ref).max() == 0:
            assert g.abs().max().item() < 1e-6, k
        else:
            err = rel_err(g.cpu().numpy(), ref)
            assert err < 2e-4, '%s: rel err %.3e' % (k, err)      # reference gradients are themselves fp32


@pytest.mark.parametrize('farnn,crf', [(0, 1), (2, 1), (1, 0)])
def test_decompose_gradients_cfg3_shapes_vs_oracle(farnn, crf):
    """SNIPS-shaped factors, gradients against the float64 autograd oracle within 1e-5 * max|grad| ... 1e-4."""
    m, args, x, lens, lab = _random_decompose(7, 500, 300, 200, 72, 100, 24, 20, farnn=farnn, use_crf=crf,
                                              update_nonlinear='tanh', beta=0.1, train_beta=1, train_h0=1, train_hT=1,
                                              train_V_embed=1, train_wildcard=1)
    loss, _, _ = m.forward_local(_t(x), _t(lab), _t(lens), train=True)
    loss.backward()
    loss_err, errs = oracle_gradient_errors(m, args, x, lab, lens, loss.item())
    assert loss_err < TOL
    for k, err in errs.items():
        assert err < 1e-4, '%s: rel err %.3e' % (k, err)


@pytest.mark.parametrize('name', golden_files('one_'))
def test_onehot_gradients_golden(name):
    """train_onehot.py trains language_tensor with CE: its gradient through the CUDA backward vs the reference."""
    z, meta = load_golden(name)
    m = build_module(name, z, meta)
    x, lab, lens = torch.from_numpy(z['x']), torch.from_numpy(z['labels']), torch.from_numpy(z['lengths'])
    loss, _, _ = m.forward_local(x, lab, lens, train=True)
    assert rel_err(loss.item(), z['loss']) < TOL
    loss.backward()                          # train_mode = 'max' included (argmax-routed gradient)
    gold = golden_grads(z)
    assert list(gold) == ['language_tensor']
    err = rel_err(m.language_tensor.grad.cpu().numpy(), gold['language_tensor'])
    assert err < 2e-4, err


@pytest.mark.parametrize('tp', ['tf32x3', 'fp16x3'])
@pytest.mark.parametrize('farnn,crf', [(0, 1), (2, 1)])
def test_training_with_tensor_core_forward(farnn, crf, tp):
    """train_precision: forward GEMMs on tensor cores (parity-grade split formats), backward in fp32."""
    from re2nn_seq_b200 import ops
    from oracle import re2nn_oracle_torch as ot
    if not ops.has_tcgen05():
        pytest.skip('no tcgen05')
    m, args, x, lens, lab = _random_decompose(9, 500, 300, 200, 72, 100, 40, 20, farnn=farnn, use_crf=crf,
                                              update_nonlinear='tanh', beta=0.1, train_h0=1, train_hT=1)
    m.train_precision = tp
    loss, _, _ = m.forward_local(_t(x), _t(lab), _t(lens), train=True)
    loss.backward()
    rename = {'embedding.weight': 'embedding', 'crf.transitions': 'crf_transitions',
              'priority_layer.priority_mat': 'priority_mat', 'priority_layer.priority_bias': 'priority_bias'}
    p64 = {rename.get(k, k): v.detach().cpu().numpy().astype(np.float64) for k, v in m.state_dict().items()}
    names = [rename.get(k, k) for k, v in m.named_parameters() if v.requires_grad]
    o_loss, g64 = ot.grads(p64, x, lab, lens, args, names=names)
    assert rel_err(loss.item(), o_loss) < TOL
    for k, v in m.named_parameters():
        if v.requires_grad:
            err = rel_err(v.grad.cpu().numpy(), g64[rename.get(k, k)])
            assert err < 1e-4, '%s: rel err %.3e' % (k, err)


def test_crf_hard_constraints_underflow_fallback():
    """Spiky features + forbidden (-1e4) transitions: the scaled-exponential CRF kernels underflow on some columns /
    rows and must take their exact log-domain fallback; loss and gradients against a float64 autograd CRF.  T = 22,
    100, 131, 170 and 225 land in every forward and backward kernel range of re2nn_crf_nll / _backward; at T = 226 the
    loss still works and the backward reports that the tag set is too large."""
    import re2nn_seq_b200 as r
    for ntag in (20, 98, 129, 168, 223, 224):
        rs = np.random.RandomState(3)
        B, L = 37, 14
        T = ntag + 2
        feats = (rs.randn(B, L, T) * 12.0).astype(np.float32)
        lens = rs.randint(2, L + 1, size=B).astype(np.int64)
        lens[0] = L
        tags = rs.randint(0, ntag, size=(B, L)).astype(np.int64)
        trans = rs.randn(T, T).astype(np.float32)
        trans[rs.rand(T, T) < 0.4] = -10000.0
        trans[:, T - 2] = -10000.0
        trans[T - 1, :] = -10000.0
        crf = r.CRF(ntag, True).cuda()
        with torch.no_grad():
            crf.transitions.copy_(_t(trans))
        f = _t(feats).requires_grad_(True)
        mask = _t(orc.length_mask(lens, L))
        loss = crf.neg_log_likelihood_loss(f, mask, _t(tags))
        # float64 reference (crf.py:48-99,202-251 in plain autograd), all sequences at once
        f64 = torch.from_numpy(feats).double().requires_grad_(True)
        t64 = torch.from_numpy(trans).double().requires_grad_(True)
        n = torch.from_numpy(lens)
        tg = torch.from_numpy(tags)
        part = f64[:, 0] + t64[T - 2]
        for t in range(1, L):
            nxt = torch.logsumexp(part[:, :, None] + t64, 1) + f64[:, t]
            part = torch.where((t < n)[:, None], nxt, part)
        logz = torch.logsumexp(part + t64[:, T - 1], 1)
        prev = torch.cat([torch.full((B, 1), T - 2), tg[:, :-1]], 1)
        steps = f64.gather(2, tg[:, :, None])[:, :, 0] + t64[prev, tg]
        gold = (torch.where(torch.arange(L)[None, :] < n[:, None], steps, 0.0).sum(1)
                + t64[tg[torch.arange(B), n - 1], T - 1])
        total = (logz - gold).sum()
        total.backward()
        assert rel_err(loss.item(), total.item()) < TOL, 'T = %d' % T
        if T > 225:
            with pytest.raises(RuntimeError, match='tag set too large'):
                loss.backward()
            continue
        loss.backward()
        # log Z is a few hundred here: fp32 keeps ~3e-5 absolute on it, which is the relative error of every marginal
        assert rel_err(f.grad.cpu().numpy(), f64.grad.numpy()) < 3e-4, 'T = %d' % T
        assert rel_err(crf.transitions.grad.cpu().numpy(), t64.grad.numpy()) < 3e-4, 'T = %d' % T


@pytest.mark.parametrize('B,ntag', [(2500, 12), (4801, 70)])
def test_crf_viterbi_large_batch(B, ntag):
    """Large odd batches, ragged lengths, exact ties (small-integer features): bit-exact paths against the numpy
    restatement of crf.py:102-195.  (A two-sequences-per-warp variant was measured 13 % slower at cfg2: it halves
    the warps in flight and the sweep is latency-bound, not shared-memory-bound.)"""
    import re2nn_seq_b200 as r
    rs = np.random.RandomState(B)
    L, T = 9, ntag + 2
    feats = rs.randint(-3, 4, size=(B, L, T)).astype(np.float32)
    lens = rs.randint(1, L + 1, size=B).astype(np.int64)
    lens[0] = L
    trans = rs.randint(-2, 3, size=(T, T)).astype(np.float32)
    trans[:, T - 2] = -10000.0
    trans[T - 1, :] = -10000.0
    crf = r.CRF(ntag, True).cuda()
    with torch.no_grad():
        crf.transitions.copy_(_t(trans))
    mask = orc.length_mask(lens, L)
    _, path = crf._viterbi_decode(_t(feats), _t(mask))
    want = orc.crf_viterbi(feats, mask, trans)
    np.testing.assert_array_equal(path.cpu().numpy(), want)


@pytest.mark.parametrize('seqs_per_warp', [1, 2])
@pytest.mark.parametrize('B,ntag,L', [(700, 129, 12), (500, 110, 10), (300, 198, 7), (90, 258, 6), (333, 34, 9)])
def test_crf_viterbi_wide_tagsets(B, ntag, L, seqs_per_warp):
    """T = 131 (cfg5: five target tags per lane), T = 112 (four), T = 200 (generic shared-memory sweep) and T = 260 (transition table
    beyond shared memory: global-memory kernel), real-valued features with many exact ties, one empty sequence:
    paths bit-exact against the restatement of crf.py:102-195."""
    import re2nn_seq_b200 as r
    from re2nn_seq_b200 import _lib
    _lib.check(_lib.fn['re2nn_debug_set_viterbi_seqs'](seqs_per_warp), 'seqs')
    rs = np.random.RandomState(ntag)
    T = ntag + 2
    feats = (rs.randint(-8, 9, size=(B, L, T)) * 0.25).astype(np.float32)
    feats[::3] += rs.randn(*feats[::3].shape).astype(np.float32)
    lens = rs.randint(1, L + 1, size=B).astype(np.int64)
    lens[0] = L
    trans = (rs.randint(-4, 5, size=(T, T)) * 0.5).astype(np.float32)
    trans[:, T - 2] = -10000.0
    trans[T - 1, :] = -10000.0
    crf = r.CRF(ntag, True).cuda()
    with torch.no_grad():
        crf.transitions.copy_(_t(trans))
    mask = orc.length_mask(lens, L)
    _, path = crf._viterbi_decode(_t(feats), _t(mask))
    want = orc.crf_viterbi(feats, mask, trans)
    np.testing.assert_array_equal(path.cpu().numpy(), want)
    # an empty sequence decodes to nothing and leaves its neighbours alone (the reference cannot express length 0:
    # it would index position -1; the kernels return a zero row)
    lens0 = lens.copy()
    lens0[1] = 0
    from re2nn_seq_b200 import ops
    _, p0 = ops.crf_viterbi(_t(feats), crf.transitions.detach(), _t(lens0), want_padded=True)
    p0 = p0.cpu().numpy()
    assert (p0[1] == 0).all()
    keep = np.arange(B) != 1
    np.testing.assert_array_equal(p0[keep], want[keep])
    _lib.check(_lib.fn['re2nn_debug_set_viterbi_seqs'](0), 'seqs')
