"""Golden data from the ORACLE (oracle/re2nn_oracle.py, oracle/re2nn_oracle_torch.py), not from the reference.

    oracle_tags_cfg2.npz        test_gpu_configs.py::test_cfg2_benchmarked_path_vs_oracle_tags (all B=4096 rows)
    oracle_tags_cfg5.npz        test_gpu_configs.py::test_cfg5_shapes_decoded_tags_vs_oracle (the first 48 rows)
    oracle_train_f{0,2}_crf1.npz  test_gpu_shim.py::test_training_loop_through_shim_vs_oracle

    python tests/golden/make_golden_oracle.py        # host only, under a minute

These tests compared with the unmodified RE2NN-SEQ classes, run at test time from a reference checkout.  The
repository does not contain the reference, so the data here comes from the oracle instead.  The oracle restates the
reference forward, CRF loss and Viterbi decode, and tests/test_oracle_golden.py pins it to the reference's own fixtures
(tests/golden/make_golden.py).  The model parameters are those of the product's constructor, which
tests/test_host_modules.py checks against the reference's initialisation.  What the oracle and the drop-ins could get
wrong in the same way is not caught by these files.

Tag files hold `tags` (flattened in row order) and `lens` (the row lengths, so a test can check it rebuilt the same
batch).  Training files hold `losses` (one per step of the loop) and `pred0` (the tags the first step decodes).
"""
import os
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
sys.path[:0] = [ROOT, TESTS]

import re2nn_seq_b200 as r  # noqa: E402
from oracle import re2nn_oracle as orc  # noqa: E402
from oracle import re2nn_oracle_torch as ot  # noqa: E402
from re2nn_seq_b200 import synth  # noqa: E402

FLAGS = dict(farnn=0, use_crf=1, update_nonlinear='tanh', beta=0.1)
RENAME = {'embedding.weight': 'embedding', 'crf.transitions': 'crf_transitions',
          'priority_layer.priority_mat': 'priority_mat', 'priority_layer.priority_bias': 'priority_bias'}


def _params(m, dtype=np.float32):
    return {RENAME.get(k, k): v.detach().numpy().astype(dtype) for k, v in m.state_dict().items()}


def tags(factor_seed, dims, batch_seed, B, Lmax, fixed_len, model_seed, rows):
    """Constructs the module as the test does (host side) and decodes `rows` of its batch with the float32 oracle."""
    V, S, R, C, D = dims
    args = synth.make_args(**FLAGS)
    f = synth.make_decompose_factors(factor_seed, V, S, R, C, D, dtype=np.float32)
    x, lens, lab = synth.make_batch(batch_seed, B, Lmax, V, C, fixed_len=fixed_len)
    torch.manual_seed(model_seed)
    m = r.FARNN_S_D_W_I_S(args=args, o_idx=0, **f)
    with torch.no_grad():
        m.crf.transitions.copy_(torch.from_numpy(synth.crf_transitions(model_seed, m.C)))
    x, lab, lens = x[:rows], lab[:rows], lens[:rows]
    _, pred, _, _ = orc.decompose_forward_local(_params(m), x, lab, lens, args, 0, train=False)
    pred = np.asarray(pred)
    assert pred.min() >= 0 and pred.max() < 256 and lens.max() < 256
    return {'tags': pred.astype(np.uint8), 'lens': lens.astype(np.uint8)}


def training_loop(farnn, crf):
    """The loop of test_gpu_shim._train_like_reference (Adam, lr 1e-3, 4 steps) on the float32 torch oracle, from the
    module test_gpu_shim._decompose_model builds (through the shadow package, on the stand-in reference tree)."""
    import test_gpu_shim as tg
    from helpers import stand_in_reference
    with tempfile.TemporaryDirectory() as tmp:
        tg._use_shim(stand_in_reference(tmp))
        m, args, x, lens, lab = tg._decompose_model(farnn, crf, 8, False)
        tg._purge()
    assert type(m).__module__.startswith('re2nn_seq_b200')
    batches = tg._batches(x, lens, lab, 16)
    p = {k: torch.tensor(v) for k, v in _params(m).items()}
    trainable = [p[RENAME.get(k, k)].requires_grad_(True) for k, v in m.named_parameters() if v.requires_grad]
    opt = torch.optim.Adam(trainable, lr=1e-3)
    b = batches[0]
    _, pred0, _, _ = orc.decompose_forward_local({k: v.detach().numpy() for k, v in p.items()}, b['x'].numpy(),
                                                 b['s'].numpy(), b['l'].numpy(), args, 0, train=False)
    losses = []
    for i in range(4):
        b = batches[i % len(batches)]
        opt.zero_grad()
        loss, _ = ot.decompose_loss(p, b['x'], b['s'], b['l'], args)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    return {'losses': np.asarray(losses, np.float64), 'pred0': np.asarray(pred0, np.int64)}


def main():
    cases = {
        'oracle_tags_cfg2': tags(0, (12000, 300, 200, 72, 100), 1000, 4096, 35, False, 13, 4096),
        'oracle_tags_cfg5': tags(12, (900, 1024, 512, 128, 100), 13, 300, 64, True, 12, 48),
        'oracle_train_f0_crf1': training_loop(0, 1),
        'oracle_train_f2_crf1': training_loop(2, 1),
    }
    for name, z in cases.items():
        np.savez_compressed(os.path.join(HERE, name + '.npz'), **z)
        print(name, {k: v.shape for k, v in z.items()}, z['losses'] if 'losses' in z else '')


if __name__ == '__main__':
    main()
