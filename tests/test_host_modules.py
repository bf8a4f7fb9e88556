"""CPU: the drop-in modules expose the reference's parameter surface and reproduce its initialisation."""
import numpy as np
import pytest
import torch

from conftest import golden_files
from helpers import build_module, load_golden

# parameters make_golden.py perturbs after construction
_PERTURBED = ('crf.transitions', 'beta_vec', 'wildcard_output_vector', 'output_wildcard_vector', 'bs1', 'bs2')
_SCALED = ('Wss1', 'Wrs1', 'Wss2', 'Wrs2')


@pytest.mark.parametrize('name', golden_files('dec_') + golden_files('sf_') + golden_files('one_'))
def test_state_dict_surface_and_init(name):
    z, meta = load_golden(name)
    m = build_module(name, z, meta, load_state=False).cpu()
    sd = m.state_dict()
    gold = {k[2:]: z[k] for k in z.files if k.startswith('p.')}
    assert list(sd.keys()) == list(gold)                             # same state_dict keys, in the same order
    assert [n for n, _ in m.named_parameters()] == list(gold)        # optimizers index parameters by position
    for k, g in gold.items():
        assert tuple(sd[k].shape) == g.shape, k
        if k in _PERTURBED:
            continue
        mine = sd[k].numpy() * np.float32(0.3) if k in _SCALED else sd[k].numpy()
        np.testing.assert_array_equal(mine, g, err_msg=k)            # same RNG draws, same values
    grads = {k[2:] for k in z.files if k.startswith('g.')}
    trainable = {k for k, v in m.named_parameters() if v.requires_grad}
    assert grads <= trainable


def test_forward_without_gpu_fails_loudly():
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    z, meta = load_golden('dec_f0_tanh_crf')
    m = build_module('dec_f0_tanh_crf', z, meta)
    with pytest.raises(RuntimeError, match='CUDA'):
        m.forward_local(torch.from_numpy(z['x']), torch.from_numpy(z['labels']), torch.from_numpy(z['lengths']),
                        train=False)


def test_utils_match_oracle():
    from oracle import re2nn_oracle as orc
    from re2nn_seq_b200 import utils
    rs = np.random.RandomState(0)
    a = rs.randn(5, 7, 3).astype(np.float32)
    lens = np.array([7, 1, 3, 5, 2])
    np.testing.assert_array_equal(utils.reverse(torch.from_numpy(a), torch.from_numpy(lens)).numpy(),
                                  orc.reverse_rows(a, lens))
    np.testing.assert_array_equal(utils.flatten(torch.from_numpy(a), torch.from_numpy(lens)).numpy(),
                                  orc.flatten_rows(a, lens))
    np.testing.assert_array_equal(utils.get_length_mask(torch.from_numpy(lens)).numpy(), orc.length_mask(lens))
    np.testing.assert_array_equal(utils.exclusive_offsets(torch.from_numpy(lens)).numpy(), [0, 7, 8, 11, 16])


def test_embed_aggregator_surface():
    """EmbedAggregator / FARNN_S_bert expose the reference's parameter names (bert_embeddings.py:46-80,
    model_decompose_single_with_bert.py:16-47) and its initialisation embed_r_generalized = pinv(E) @ V."""
    import re2nn_seq_b200 as r
    from re2nn_seq_b200 import synth
    args = synth.make_args(farnn=0, use_crf=0, train_V_embed=1, train_beta=0, train_word_embed=0)
    f = synth.make_decompose_factors(0, 120, 24, 16, 6, 20, dtype=np.float64)
    agg = r.EmbedAggregator(args, f['V'], f['pretrained_word_embed'])
    assert sorted(agg.state_dict()) == ['V_embed', 'beta_vec', 'embed.embedding.weight', 'embed_r_generalized']
    E = torch.from_numpy(f['pretrained_word_embed']).float()
    np.testing.assert_array_equal(agg.embed_r_generalized.detach().numpy(),
                                  torch.matmul(E.pinverse(), torch.from_numpy(f['V']).float()).numpy())
    assert agg.V_embed.requires_grad and not agg.beta_vec.requires_grad and not agg.embed.embedding.weight.requires_grad
    keep = ('S1', 'S2', 'C_output_mat', 'wildcard_mat', 'wildcard_output_vector', 'final_vector', 'start_vector')
    m = r.FARNN_S_bert(V=f['V'], static_embed=f['pretrained_word_embed'], priority_mat=None, args=args, o_idx=0,
                       is_cuda=False, **{k: f[k] for k in keep})
    keys = set(m.state_dict())
    assert {'embed.V_embed', 'embed.embed_r_generalized', 'embed.beta_vec', 'slot_filler.S1', 'slot_filler.S2',
            'slot_filler.C_output_mat'} <= keys
    args.use_bert = 1
    with pytest.raises(ValueError, match='encoder'):
        r.EmbedAggregator(args, f['V'], f['pretrained_word_embed'])


@pytest.mark.parametrize('name', golden_files('fst_'))
def test_fst_constructors_match_reference(name):
    """Host side only: same torch seed -> the FST drop-ins draw the reference's random numbers in the reference's
    order (state_dict keys, shapes and values identical; the fixture's gates / CRF transitions were edited after
    construction and are compared by key and shape only)."""
    import json
    import os
    import numpy as np
    from helpers import GOLDEN
    from test_gpu_fst import build_fst_module
    z = np.load(os.path.join(GOLDEN, name + '.npz'), allow_pickle=False)
    meta = json.loads(str(z['meta']))
    meta['name'] = name
    if meta['kind'] == 'fst_oi':
        meta['independent'] = 2 if 'ind2' in name else 1
    m = build_fst_module(z, meta, load_state=False)
    sd = m.state_dict()
    want = {k[2:]: z[k] for k in z.files if k.startswith('p.')}
    assert list(sd.keys()) == list(want)
    assert [n for n, _ in m.named_parameters()] == list(want)
    edited = ('Wss1', 'Wrs1', 'bs1', 'Wss2', 'Wrs2', 'bs2', 'crf.transitions')
    for k, v in sd.items():
        assert tuple(v.shape) == want[k].shape, k
        if k not in edited:
            np.testing.assert_array_equal(v.cpu().numpy(), want[k], err_msg=k)
    flags = {k: v.requires_grad for k, v in m.named_parameters()}
    grads = {k[2:] for k in z.files if k.startswith('g.')}
    if grads:
        assert grads <= {k for k, rg in flags.items() if rg}


def test_fst_rank_r_rejects_unknown_farnn():
    """FARNN_S_D_W / FARNN_S_D_W_I refuse farnn outside {0, 1, 2} at construction, as the other rank-R classes do."""
    import json
    import os
    from helpers import GOLDEN
    from test_gpu_fst import build_fst_module
    for name in ('fst_dw_f0_tanh_crf', 'fst_dwi_f0_tanh_crf'):
        z = np.load(os.path.join(GOLDEN, name + '.npz'), allow_pickle=False)
        meta = json.loads(str(z['meta']))
        meta['flags']['farnn'] = 3
        with pytest.raises(NotImplementedError):
            build_fst_module(z, meta, load_state=False)
