"""Shared helpers for the parity tests (fixtures -> oracle parameter dicts)."""
import json
import os

import numpy as np

from re2nn_seq_b200 import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')

# reference state_dict key -> oracle key
_RENAME = {'embedding.weight': 'embedding', 'crf.transitions': 'crf_transitions',
           'priority_layer.priority_mat': 'priority_mat', 'priority_layer.priority_bias': 'priority_bias'}


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + '.npz'), allow_pickle=False)
    meta = json.loads(str(z['meta']))
    return z, meta


def oracle_params(z, dtype=np.float32):
    p = {}
    for k in z.files:
        if k.startswith('p.'):
            n = k[2:]
            p[_RENAME.get(n, n)] = z[k].astype(dtype)
    return p


def golden_grads(z):
    return {k[2:]: z[k] for k in z.files if k.startswith('g.')}


def args_of(meta):
    return synth.make_args(**meta['flags'])


def rel_err(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def oracle_gradient_errors(m, args, x, labels, lengths, loss, dense_v=None):
    """After loss.backward() on module `m`: its loss and every trained parameter's gradient against the float64 autograd
    oracle (oracle/re2nn_oracle_torch.py) over the same batch -> (loss rel err, {parameter name: max-norm rel err}).
    A parameter the oracle's loss does not reach must get no gradient or a zero one (error 0, else inf)."""
    from oracle import re2nn_oracle_torch as ot
    p64 = {_RENAME.get(k, k): v.detach().cpu().numpy().astype(np.float64) for k, v in m.state_dict().items()}
    names = [_RENAME.get(k, k) for k, v in m.named_parameters() if v.requires_grad]
    o_loss, g64 = ot.grads(p64, x if dense_v is None else dense_v, labels, lengths, args, dense_v=dense_v, names=names)
    errs = {}
    for k, v in m.named_parameters():
        if not v.requires_grad:
            continue
        ref = g64[_RENAME.get(k, k)]
        if ref is None:
            errs[k] = 0.0 if v.grad is None or not v.grad.any() else float('inf')
        else:
            errs[k] = rel_err(v.grad.cpu().numpy(), ref)
    return rel_err(float(loss), o_loss), errs


# ---- a stand-in reference tree for the `src_seq` shadow package (shim/) ------------------------------
# The reference's module layout and the names its drivers import, each defined in a placeholder module.  The shadow
# package's import mechanics (which name resolves to which tree) are tested against it, so those tests do not need an
# RE2NN-SEQ checkout.
_STAND_IN = {
    '__init__.py': '',
    'val.py': 'def val_onehot(*a, **k):\n    raise NotImplementedError\n',
    'utils.py': '',
    'farnn/__init__.py': '',
    'farnn/model_decompose_single.py': 'class FARNN_S_D_W_I_S:\n    pass\n\n\nclass FARNN_S_SF:\n    pass\n',
    'farnn/model_onehot.py': 'class FARNN_S_O:\n    pass\n\n\nclass FARNN_S_O_I:\n    pass\n\n\nclass FARNN_S_O_I_S:\n    pass\n',
    'farnn/model_decompose.py': 'class FARNN_S_D_W:\n    pass\n',
    'farnn/model_decompose_independent.py': 'class FARNN_S_D_W_I:\n    pass\n',
    'farnn/priority.py': 'class PriorityLayer:\n    pass\n',
    'baselines/__init__.py': '',
    'baselines/crf.py': 'class CRF:\n    pass\n',
    'baselines/KD.py': 'def KD_loss(*a, **k):\n    raise NotImplementedError\n',
}


def stand_in_reference(root):
    """Write the stand-in reference tree under `root` (root/src_seq/...) -> root."""
    for rel, text in _STAND_IN.items():
        path = os.path.join(root, 'src_seq', rel)
        os.makedirs(os.path.dirname(path), exist_ok=True)
        with open(path, 'w') as f:
            f.write(text)
    return str(root)


# ---- building product modules from fixtures --------------------------------------------------------
def golden_seed(name):
    """Seed used by tests/golden/make_golden.py for this case (see its main())."""
    order = ['dec_f0_tanh_crf', 'dec_f0_none_ce', 'dec_f1_relu_ce', 'dec_f2_tanh_crf_add', 'dec_f2_relutanh_ce_all',
             'dec_f0_tanh_max', 'dec_f0_prio_crf_sig', 'dec_f1_tanh_ce_plain', 'dec_f2_none_crf_relutanh',
             'sf_f2_tanh_crf', 'sf_f0_relu_ce', 'dec_f0_tanh_ce_kd', 'dec_f2_tanh_crf_pr', 'dec_f0_tanh_ml']
    if name in order:
        return 10 + order.index(name)
    return {'one_sum_none': 30, 'one_sum_tanh_noise': 31, 'one_max_relu': 32, 'one_sum_relutanh_ce_prio': 33, 'one_sum_relu_ml': 34}[name]


def build_module(name, z, meta, load_state=True):
    """Construct the product module exactly as make_golden.py constructed the reference one."""
    import torch
    import re2nn_seq_b200 as r
    seed = golden_seed(name)
    d = meta['dims']
    args = args_of(meta)
    kind = meta['kind']
    has_prio = bool(meta['flags'].get('use_priority')) and name in ('dec_f0_prio_crf_sig', 'one_sum_relutanh_ce_prio')
    pm = None
    if has_prio:
        rs = np.random.RandomState(seed + 2)
        pm = np.eye(d['C'] + 1) + 0.1 * rs.randn(d['C'] + 1, d['C'] + 1)
    torch.manual_seed(seed)
    if kind == 'onehot':
        a = synth.make_onehot_automaton(seed, d['V'], d['S'], d['C'], lang_frac=0.6)
        m = r.FARNN_S_O_I_S(a['language_tensor'], a['output_mat'], a['wildcard_mat'], a['output_wildcard_vector'],
                            a['final_vector'], a['start_vector'], pm, args, meta['o_idx'], False)
    else:
        f = synth.make_decompose_factors(seed, d['V'], d['S'], d['R'], d['C'], d['D'], lang_frac=0.5)
        if kind == 'sf':
            m = r.FARNN_S_SF(S1=f['S1'], S2=f['S2'], C_output_mat=f['C_output_mat'], wildcard_mat=f['wildcard_mat'],
                             wildcard_output_vector=f['wildcard_output_vector'], final_vector=f['final_vector'],
                             start_vector=f['start_vector'], priority_mat=pm, args=args, o_idx=meta['o_idx'],
                             is_cuda=False)
        else:
            m = r.FARNN_S_D_W_I_S(V=f['V'], S1=f['S1'], S2=f['S2'], C_output_mat=f['C_output_mat'],
                                  wildcard_mat=f['wildcard_mat'], wildcard_output_vector=f['wildcard_output_vector'],
                                  final_vector=f['final_vector'], start_vector=f['start_vector'],
                                  pretrained_word_embed=f['pretrained_word_embed'], priority_mat=pm, args=args,
                                  o_idx=meta['o_idx'], is_cuda=False)
    if load_state:
        sd = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith('p.')}
        m.load_state_dict(sd, strict=True)
    return m
