"""GPU: the reference's OWN driver code, unchanged, on the drop-in classes through the `src_seq` shadow package.

oracle/_ref holds the unmodified reference files (sha256-pinned by oracle/ref_manifest.json; they travel to the GPU
box, /root/reference does not).  Each test first runs the pure reference on the CPU, then the same reference driver
function -- val.val_onehot (src_seq/val.py:7-43) and the training loop of train_decompose.py:170-193 -- with
shim/ ahead on sys.path, so `from src_seq.farnn.model_decompose_single import FARNN_S_D_W_I_S` inside the
reference code resolves to the B200 implementation while src_seq.val / src_seq.utils / src_seq.metrics stay the
reference's files.  Tags and the metric dictionary must be identical, losses agree to 1e-5 relative.
test_reference_val_onehot_runs_on_the_dropins needs that reference checkout and skips without it; the training loop runs through the shadow package
on a stand-in reference tree and compares with stored oracle values (the repository does not contain the reference)."""
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIM = os.path.join(ROOT, 'shim')
REF = os.path.join(ROOT, 'oracle', '_ref')


def _purge():
    for k in [k for k in sys.modules if k == 'src_seq' or k.startswith('src_seq.')]:
        del sys.modules[k]
    for p in (SHIM, REF):
        while p in sys.path:
            sys.path.remove(p)


def _use_reference():
    from oracle import make_ref
    why = make_ref.verify()
    if why:
        pytest.skip(why)
    _purge()
    make_ref.import_reference()


def _use_shim(ref=REF):
    _purge()
    os.environ['RE2NN_REFERENCE_ROOT'] = ref
    sys.path.insert(0, SHIM)


def _batches(x, lens, lab, bz):
    out = []
    for i in range(0, len(lens), bz):
        l = lens[i:i + bz]
        Lm = int(l.max())
        out.append({'x': torch.from_numpy(x[i:i + bz, :Lm].copy()), 's': torch.from_numpy(lab[i:i + bz, :Lm].copy()),
                    'l': torch.from_numpy(l.copy())})
    return out


def _decompose_model(farnn, crf, seed, is_cuda):
    """Built through whatever `src_seq` currently resolves to, exactly as train_decompose.py:98-110 does."""
    from re2nn_seq_b200 import synth
    from src_seq.farnn.model_decompose_single import FARNN_S_D_W_I_S
    V, S, R, C, D = 60, 24, 16, 5, 12
    args = synth.make_args(farnn=farnn, use_crf=crf, update_nonlinear='tanh', beta=0.3, sigmoid_exponent=5, bias_init=5.0)
    f = synth.make_decompose_factors(seed, V, S, R, C, D, lang_frac=0.5)
    torch.manual_seed(seed)
    m = FARNN_S_D_W_I_S(V=f['V'], S1=f['S1'], S2=f['S2'], C_output_mat=f['C_output_mat'], wildcard_mat=f['wildcard_mat'],
                        wildcard_output_vector=f['wildcard_output_vector'], final_vector=f['final_vector'],
                        start_vector=f['start_vector'], pretrained_word_embed=f['pretrained_word_embed'],
                        priority_mat=None, args=args, o_idx=0, is_cuda=is_cuda)
    with torch.no_grad():
        if crf:
            m.crf.transitions.copy_(torch.from_numpy(synth.crf_transitions(seed, m.C)))
        if farnn:
            for n in ('Wss1', 'Wrs1', 'Wss2', 'Wrs2'):
                getattr(m, n).mul_(0.2)
    x, lens, lab = synth.make_batch(seed + 1, 37, 9, V, C)
    return m, args, x, lens, lab


@pytest.mark.parametrize('farnn,crf', [(0, 1), (2, 0)])
def test_reference_val_onehot_runs_on_the_dropins(farnn, crf):
    _use_reference()
    from src_seq.val import val_onehot
    m, args, x, lens, lab = _decompose_model(farnn, crf, 5, False)
    assert type(m).__module__ == 'src_seq.farnn.model_decompose_single' and os.path.abspath(
        sys.modules[type(m).__module__].__file__).startswith(REF)
    i2s = ['o'] + ['B-%d' % i for i in range(10)]
    want = val_onehot(_batches(x, lens, lab, 16), m, args, o_idx=0, i2s=i2s, is_cuda=False)

    _use_shim()
    from src_seq.val import val_onehot as val_shim
    import src_seq.val as val_mod
    assert os.path.abspath(val_mod.__file__).startswith(REF)           # the driver is the reference's file ...
    m2, args2, x2, lens2, lab2 = _decompose_model(farnn, crf, 5, True)
    assert type(m2).__module__.startswith('re2nn_seq_b200')           # ... the model is the B200 drop-in
    m2 = m2.cuda()
    got = val_shim(_batches(x2, lens2, lab2, 16), m2, args2, o_idx=0, i2s=i2s, is_cuda=True)
    assert got['token-level'] == want['token-level']
    assert got['entity-level'][:4] == want['entity-level'][:4]
    _purge()


def _train_like_reference(m, args, batches, steps, cuda):
    """The body of train_decompose.py:135-138,170-193 (Adam over model.parameters(), forward_local(train=True),
    loss.backward(), optimizer.step())."""
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    losses, preds = [], []
    m.train()
    for i in range(steps):
        b = batches[i % len(batches)]
        m.zero_grad()
        x, label, lengths = b['x'], b['s'], b['l']
        if cuda:
            x, label, lengths = x.cuda(), label.cuda(), lengths.cuda()
        loss, pred_label, true_label = m.forward_local(x, label, lengths, train=True)
        loss.backward()
        opt.step()
        losses.append(loss.item())
        preds.append(pred_label.cpu().numpy())
    return losses, preds


@pytest.mark.parametrize('farnn,crf', [(0, 1), (2, 1)])
def test_training_loop_through_shim_vs_oracle(farnn, crf, tmp_path):
    """The training loop above on the drop-in that the shadow package resolves (against the stand-in reference tree of
    helpers.stand_in_reference), against the same loop on the float32 torch oracle, stored by
    tests/golden/make_golden_oracle.py.  The repository does not contain the reference, so the expected values come
    from the oracle, not from the reference classes."""
    from helpers import GOLDEN, stand_in_reference
    z = np.load(os.path.join(GOLDEN, 'oracle_train_f%d_crf%d.npz' % (farnn, crf)))
    _use_shim(stand_in_reference(tmp_path))
    m, args, x, lens, lab = _decompose_model(farnn, crf, 8, True)
    assert type(m).__module__.startswith('re2nn_seq_b200')
    m = m.cuda()
    got_l, got_p = _train_like_reference(m, args, _batches(x, lens, lab, 16), 4, True)
    want_l = z['losses']
    for a, b in zip(got_l, want_l):
        assert abs(a - b) <= 2e-5 * abs(b), (got_l, want_l)
    np.testing.assert_array_equal(got_p[0], z['pred0'])                 # same parameters -> same decoded tags
    _purge()


def test_shim_off_switch_falls_through_to_reference(tmp_path):
    """Against the stand-in reference tree of helpers.stand_in_reference (the reference's layout and names)."""
    from helpers import stand_in_reference
    ref = stand_in_reference(tmp_path)
    _use_shim(ref)
    os.environ['RE2NN_SHIM'] = 'off'
    try:
        from src_seq.farnn.model_decompose_single import FARNN_S_D_W_I_S
        assert FARNN_S_D_W_I_S.__module__ == 'src_seq.farnn.model_decompose_single'
        assert os.path.abspath(sys.modules[FARNN_S_D_W_I_S.__module__].__file__).startswith(ref)
    finally:
        del os.environ['RE2NN_SHIM']
        _purge()
