"""CPU: the partial-annotation loss and constrained Viterbi restatements (crf_partial_ref.py) against brute-force
enumeration of every tag sequence, the allowed-mask helper, and the argument checks of the C-ABI entry points."""
import itertools

import numpy as np
import pytest
import torch

import crf_partial_ref as ref
from crf_nbest_ref import crf_path_score


def _case(seed, B, L, T, kind):
    rs = np.random.RandomState(seed)
    feats = rs.randn(B, L, T)
    trans = rs.randn(T, T)
    lens = rs.randint(1, L + 1, size=B).astype(np.int64)
    lens[0] = L
    if kind == 'all':
        allowed = np.ones((B, L, T), bool)
    elif kind == 'onehot':
        allowed = np.eye(T, dtype=bool)[rs.randint(0, T, size=(B, L))]
    else:
        allowed = rs.rand(B, L, T) < 0.5
        allowed[np.arange(B)[:, None], np.arange(L)[None, :], rs.randint(0, T, size=(B, L))] = True
    return feats, trans, lens, allowed


def _enumerated(f, trans, n, allowed_b):
    """(log Z, log Z^A, dfeats n x T, dtrans T x T) of one row from all T^n sequences."""
    T = trans.shape[0]
    seqs = list(itertools.product(range(T), repeat=n))
    s = np.array([crf_path_score(f, trans, np.array(y)) for y in seqs])
    ok = np.array([all(allowed_b[t, y[t]] for t in range(n)) for y in seqs])

    def lse(v):
        m = v.max()
        return m + np.log(np.exp(v - m).sum())
    lz, lza = lse(s), lse(s[ok])
    p = np.exp(s - lz) - np.where(ok, np.exp(s - lza), 0.0)       # P - P_A per sequence
    df = np.zeros((n, T))
    dt = np.zeros((T, T))
    for w, y in zip(p, seqs):
        df[np.arange(n), list(y)] += w
        prev = [T - 2] + list(y)
        for a, b in zip(prev, list(y) + [T - 1]):
            dt[a, b] += w
    return lz, lza, df, dt


@pytest.mark.parametrize('kind', ['all', 'onehot', 'random'])
@pytest.mark.parametrize('T', [3, 4, 5])
def test_partial_loss_matches_enumeration(T, kind):
    feats, trans, lens, allowed = _case(10 * T + len(kind), 6, 5 if T < 5 else 4, T, kind)
    per_seq, dfeats, dtrans = ref.crf_partial_nll(feats, lens, trans, allowed)
    want_dt = np.zeros_like(trans)
    for b in range(len(lens)):
        n = int(lens[b])
        lz, lza, df, dt = _enumerated(feats[b], trans, n, allowed[b])
        assert abs(per_seq[b] - (lz - lza)) < 1e-10
        np.testing.assert_allclose(dfeats[b, :n], df, rtol=0, atol=1e-10)
        assert (dfeats[b, n:] == 0).all()
        want_dt += dt
    np.testing.assert_allclose(dtrans, want_dt, rtol=0, atol=1e-10)
    if kind == 'all':
        assert np.abs(per_seq).max() < 1e-12


def test_partial_loss_onehot_is_nll_and_empty_rows():
    """A one-hot mask of the gold tags gives log Z - gold score; an empty sequence gives 0 and zero rows; lengths past L
    are clamped."""
    feats, trans, lens, _ = _case(3, 5, 4, 5, 'all')
    tags = np.random.RandomState(4).randint(0, 5, size=(5, 4))
    lens = np.array([4, 0, 1, 9, 2], np.int64)
    per_seq, dfeats, dtrans = ref.crf_partial_nll(feats, lens, trans, np.eye(5, dtype=bool)[tags])
    for b in range(5):
        n = min(int(lens[b]), 4)
        if n == 0:
            assert per_seq[b] == 0 and (dfeats[b] == 0).all()
            continue
        lz = _enumerated(feats[b], trans, n, np.ones((n, 5), bool))[0]
        assert abs(per_seq[b] - (lz - crf_path_score(feats[b], trans, tags[b, :n]))) < 1e-10


@pytest.mark.parametrize('kind', ['all', 'onehot', 'random'])
@pytest.mark.parametrize('T', [3, 5])
def test_constrained_viterbi_matches_enumeration(T, kind):
    feats, trans, lens, allowed = _case(7 * T + len(kind), 8, 5, T, kind)
    lens[1] = 0
    paths, scores = ref.crf_constrained_viterbi(feats, lens, trans, allowed)
    assert (paths[1] == 0).all() and scores[1] == -np.inf
    for b in range(len(lens)):
        n = int(lens[b])
        if n == 0:
            continue
        best = max((crf_path_score(feats[b], trans, np.array(y)), y) for y in itertools.product(range(T), repeat=n)
                   if all(allowed[b, t, y[t]] for t in range(n)))
        assert abs(scores[b] - best[0]) < 1e-12
        np.testing.assert_array_equal(paths[b, :n], best[1])     # real-valued scores: the best path is unique
        assert allowed[b, np.arange(n), paths[b, :n]].all()
        assert (paths[b, n:] == 0).all()
        if kind == 'onehot':
            np.testing.assert_array_equal(paths[b, :n], allowed[b, :n].argmax(1))


def test_partial_allowed():
    from re2nn_seq_b200.crf import partial_allowed
    labels = torch.tensor([[2, -1, 0, 1], [-1, -1, -1, -1], [3, 3, 5, 5]])
    a = partial_allowed(labels, 6)
    assert a.dtype == torch.bool and a.shape == (3, 4, 6)
    assert a[0, 0].tolist() == [False, False, True, False, False, False]
    assert a[0, 1].all() and a[1].all()                    # unknown: every column, START / STOP included
    assert (a[2].sum(1) == 1).all()
    b = partial_allowed(labels, 6, lengths=torch.tensor([4, 0, 2]))
    assert b[2, 2:].all() and not b[2, :2].all() and torch.equal(b[0], a[0])   # pads are all-true
    c = partial_allowed(torch.where(labels == -1, torch.full_like(labels, 7), labels), 6, unknown=7)
    assert torch.equal(c, a)


def test_partial_entry_points_refuse_bad_arguments_before_cuda():
    """Null pointers, bad dims, a lone partition history and (backward) T > 225 fail with a message before anything is
    launched (dummy pointers: nothing is dereferenced)."""
    import ctypes
    from re2nn_seq_b200 import _lib
    p = ctypes.c_void_p(0x1000)
    fwd, bwd, err = _lib.fn['re2nn_crf_partial_nll'], _lib.fn['re2nn_crf_partial_nll_backward'], _lib.fn['re2nn_last_error']
    assert fwd(p, p, p, None, 2, 3, 7, p, p, p, p, None) != 0
    assert b'null' in err()
    assert fwd(p, p, p, p, 2, 3, 7, None, p, p, p, None) != 0
    assert b'null' in err()
    assert fwd(p, p, p, p, 2, 3, 7, p, p, p, None, None) != 0
    assert b'together' in err()
    for B, L, T in ((0, 3, 7), (2, 0, 7), (2, 3, 2)):
        assert fwd(p, p, p, p, B, L, T, p, p, None, None, None) != 0
        assert b'bad dims' in err()
    for k in range(8):                                  # each pointer argument of the backward in turn
        args = [p] * 6
        if k < 6:
            args[k] = None
        assert bwd(*args, p, 2, 3, 7, p if k != 6 else None, p if k != 7 else None, None) != 0
        assert b'null' in err()
    for B, L, T in ((0, 3, 7), (2, -1, 7), (2, 3, 1)):
        assert bwd(p, p, p, p, p, p, p, B, L, T, p, p, None) != 0
        assert b'bad dims' in err()
    assert bwd(p, p, p, p, p, p, p, 2, 3, 226, p, p, None) != 0
    assert b'tag set too large' in err()
