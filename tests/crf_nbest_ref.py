"""CPU restatements of N-best CRF decoding and tag marginals, the checkers of tests/test_crf_nbest_oracle.py and
tests/test_gpu_crf_nbest.py.  The reference's crf.py (and so oracle/re2nn_oracle.py) has neither; NCRF++'s CRF has
_viterbi_decode_nbest.  Arithmetic in the dtype of the arrays: float32 mirrors the kernels' rounding, float64 gives a
truth."""
import numpy as np

START_TAG = -2   # baselines/crf.py:11
STOP_TAG = -1    # baselines/crf.py:12


def crf_nbest(feats, lengths, trans, K):
    """List Viterbi over all T tags, in the dtype of `feats` with crf_viterbi's expressions:
    part_0[j] = feat_0[j] + trans[START][j]; (feat_t[j] + trans[i][j]) + part_{t-1}[i]; part_{n-1}[i] + trans[i][STOP].
    Every (t, j) keeps its K best prefixes ranked by value, then by smaller source tag, then by smaller source rank
    (so equal scores end up ordered by the reversed sequence, ascending); -inf candidates are missing.
    Returns (paths B x L x K int64: -1 at the valid positions of a missing rank, 0 at pads; scores B x K, -inf when
    missing).  Lengths are clamped to L; a sequence of length 0 has an all-zero row."""
    B, L, T = feats.shape
    dt = feats.dtype
    paths = np.zeros((B, L, K), np.int64)
    scores = np.full((B, K), -np.inf, dt)

    def top(vals):
        """vals (T*K, X): candidates in key order (source tag major, source rank minor) -> indices of the K best
        per column, stable on ties, and their values."""
        idx = np.argsort(-vals, axis=0, kind='stable')[:K]
        return idx, np.take_along_axis(vals, idx, 0)

    for b in range(B):
        n = min(int(lengths[b]), L)
        if n <= 0:
            continue
        f = feats[b]
        P = np.full((T, K), -np.inf, dt)          # P[i, r]: value of rank r at tag i
        P[:, 0] = f[0] + trans[START_TAG]
        bps = []
        for t in range(1, n):
            cand = (f[t][None, None, :] + trans[:, None, :]) + P[:, :, None]      # T x K x T (source, rank, target)
            idx, val = top(cand.reshape(T * K, T))
            bps.append(idx)                                                        # K x T
            P = val.T.copy()
        fin = (P + trans[:, STOP_TAG][:, None]).reshape(T * K, 1)
        idx, val = top(fin)
        for k in range(K):
            v = val[k, 0]
            if v == -np.inf:
                paths[b, :n, k] = -1
                continue
            scores[b, k] = v
            i, r = divmod(int(idx[k, 0]), K)
            for t in range(n - 1, -1, -1):
                paths[b, t, k] = i
                if t > 0:
                    i, r = divmod(int(bps[t - 1][r, i]), K)
    return paths, scores


def crf_path_score(feats_b, trans, tags):
    """Score of one tag sequence with the recursion crf_nbest ranks by (feats_b: n x T)."""
    T = trans.shape[0]
    s = feats_b[0, tags[0]] + trans[T - 2, tags[0]]
    for t in range(1, len(tags)):
        s = (feats_b[t, tags[t]] + trans[tags[t - 1], tags[t]]) + s
    return s + trans[tags[-1], T - 1]


def crf_marginals(feats, lengths, trans):
    """Forward-backward in the dtype of the arrays (float64 for a truth): marginals[b, t, j] = P(y_t = j | x),
    zero at pads, and log Z (0 for an empty sequence).  Lengths are clamped to L."""
    B, L, T = feats.shape
    marg = np.zeros((B, L, T), feats.dtype)
    log_z = np.zeros(B, feats.dtype)

    def lse(a, axis):
        m = a.max(axis, keepdims=True)
        return (m + np.log(np.exp(a - m).sum(axis, keepdims=True))).squeeze(axis)

    for b in range(B):
        n = min(int(lengths[b]), L)
        if n <= 0:
            continue
        f = feats[b]
        alpha = [f[0] + trans[START_TAG]]
        for t in range(1, n):
            alpha.append(lse(alpha[-1][:, None] + trans, 0) + f[t])
        beta = [trans[:, STOP_TAG]]
        for t in range(n - 1, 0, -1):
            beta.append(lse(trans + (f[t] + beta[-1])[None, :], 1))
        beta = beta[::-1]
        log_z[b] = lse(alpha[-1] + trans[:, STOP_TAG], 0)
        for t in range(n):
            marg[b, t] = np.exp(alpha[t] + beta[t] - log_z[b])
    return marg, log_z
