"""CPU: the N-best and marginal restatements (crf_nbest_ref.py) against brute-force enumeration of every tag sequence, and
the argument checks of their C-ABI entry points."""
import itertools

import numpy as np
import pytest

import crf_nbest_ref as ref
from oracle import re2nn_oracle as orc


def _case(seed, B, L, T, integer):
    rs = np.random.RandomState(seed)
    if integer:      # small integers: every sum is exact in fp32, so ties are real ties
        feats = rs.randint(-2, 3, size=(B, L, T)).astype(np.float32)
        trans = rs.randint(-2, 3, size=(T, T)).astype(np.float32)
    else:
        feats = rs.randn(B, L, T).astype(np.float32)
        trans = rs.randn(T, T).astype(np.float32)
    lens = rs.randint(1, L + 1, size=B).astype(np.int64)
    return feats, trans, lens


def _enumerate(f, trans, n):
    """[(score, tags)] of all T^n sequences of one row, best first; ties by the reversed sequence, ascending."""
    T = trans.shape[0]
    out = [(ref.crf_path_score(f, trans, np.array(y)), y) for y in itertools.product(range(T), repeat=n)]
    out.sort(key=lambda e: (-e[0], e[1][::-1]))
    return out


@pytest.mark.parametrize('K', [1, 2, 5, 16])
@pytest.mark.parametrize('T', [3, 4, 5])
def test_nbest_integer_ties_match_enumeration(T, K):
    feats, trans, lens = _case(10 * T + K, 6, 5, T, True)
    paths, scores = ref.crf_nbest(feats, lens, trans, K)
    for b in range(len(lens)):
        n = int(lens[b])
        want = _enumerate(feats[b], trans, n)[:K]
        for k, (s, y) in enumerate(want):
            assert scores[b, k] == s, (b, k)
            np.testing.assert_array_equal(paths[b, :n, k], y)      # the order of ties included
        for k in range(len(want), K):                              # fewer than K sequences exist
            assert scores[b, k] == -np.inf
            assert (paths[b, :n, k] == -1).all()
        assert (paths[b, n:] == 0).all()


@pytest.mark.parametrize('K', [1, 3, 8])
def test_nbest_real_values_match_enumeration(K):
    feats, trans, lens = _case(7 + K, 8, 5, 5, False)
    paths, scores = ref.crf_nbest(feats, lens, trans, K)
    for b in range(len(lens)):
        n = int(lens[b])
        want = _enumerate(feats[b], trans, n)[:K]
        np.testing.assert_allclose(scores[b, :len(want)], [s for s, _ in want], rtol=0, atol=1e-5)
        for k in range(len(want)):                   # each path carries the score reported for it
            assert abs(ref.crf_path_score(feats[b], trans, paths[b, :n, k]) - scores[b, k]) <= 1e-5


@pytest.mark.parametrize('integer', [True, False])
def test_nbest_rank0_is_viterbi(integer):
    feats, trans, lens = _case(3, 40, 6, 5, integer)
    paths, _ = ref.crf_nbest(feats, lens, trans, 4)
    mask = orc.length_mask(lens, 6)
    vit = orc.crf_viterbi(feats, mask, trans)
    np.testing.assert_array_equal(paths[:, :, 0][mask], vit[mask])


def test_nbest_edge_cases():
    feats, trans, lens = _case(5, 4, 4, 3, True)
    lens = np.array([0, 1, 9, 2], np.int64)          # empty, one token with T < K, longer than L (clamped)
    paths, scores = ref.crf_nbest(feats, lens, trans, 4)
    assert (paths[0] == 0).all() and (scores[0] == -np.inf).all()
    assert np.isfinite(scores[1, :3]).all() and scores[1, 3] == -np.inf and paths[1, 0, 3] == -1
    assert (paths[1, 1:] == 0).all()
    clamped, clamped_s = ref.crf_nbest(feats, np.array([0, 1, 4, 2], np.int64), trans, 4)
    np.testing.assert_array_equal(paths, clamped)
    np.testing.assert_array_equal(scores, clamped_s)


@pytest.mark.parametrize('T', [3, 5])
def test_marginals_match_enumeration(T):
    feats, trans, lens = _case(20 + T, 5, 5, T, False)
    f64, t64 = feats.astype(np.float64), trans.astype(np.float64)
    marg, log_z = ref.crf_marginals(f64, lens, t64)
    for b in range(len(lens)):
        n = int(lens[b])
        seqs = list(itertools.product(range(T), repeat=n))
        s = np.array([ref.crf_path_score(f64[b], t64, np.array(y)) for y in seqs])
        m = s.max()
        z = m + np.log(np.exp(s - m).sum())
        assert abs(log_z[b] - z) < 1e-12
        p = np.exp(s - z)
        want = np.zeros((n, T))
        for pr, y in zip(p, seqs):
            want[np.arange(n), list(y)] += pr
        np.testing.assert_allclose(marg[b, :n], want, rtol=0, atol=1e-12)
        assert (marg[b, n:] == 0).all()
    empty, lz = ref.crf_marginals(f64, np.zeros(len(lens), np.int64), t64)
    assert (empty == 0).all() and (lz == 0).all()


def test_nbest_and_marginals_refuse_bad_arguments_before_cuda():
    """Out-of-range K, a tag set too large for the lists, null pointers and a short workspace fail with a message
    before anything is launched (dummy pointers: nothing is dereferenced)."""
    import ctypes
    from re2nn_seq_b200 import _lib
    p = ctypes.c_void_p(0x1000)
    nbest, err = _lib.fn['re2nn_crf_nbest'], _lib.fn['re2nn_last_error']
    ws = _lib.fn['re2nn_crf_nbest_workspace']
    assert ws(2, 3, 7, 4) == 2 * 3 * 7 * 4 * 2
    for K in (0, 17):
        assert nbest(p, p, p, 2, 3, 7, K, p, p, p, 1 << 30, None) != 0
        assert b'outside [1, 16]' in err()
    assert nbest(p, p, p, 2, 3, 1601, 16, p, p, p, 1 << 40, None) != 0      # T * K = 25616 > 25600
    assert b'too large' in err() and b'25600' in err()
    assert nbest(p, p, p, 2, 3, 4097, 1, p, p, p, 1 << 40, None) != 0
    assert b'4096' in err()
    assert nbest(p, None, p, 2, 3, 7, 4, p, p, p, 1 << 30, None) != 0
    assert b'null' in err()
    assert nbest(p, p, p, 2, 3, 7, 4, p, p, p, ws(2, 3, 7, 4) - 1, None) != 0
    assert b'workspace too small' in err()
    assert _lib.fn['re2nn_crf_marginals'](p, p, p, 2, 3, 7, p, None, p, None) != 0
    assert b'null' in err()
