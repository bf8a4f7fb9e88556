"""CPU restatements of the partial-annotation CRF loss and of constrained Viterbi decoding, the checkers of
tests/test_crf_partial_oracle.py and tests/test_gpu_crf_partial.py.  Neither exists in the reference's crf.py.

allowed is a B x L x T bool mask over all T = tagset + 2 columns (START / STOP included): position t may only take the
tags j with allowed[b, t, j].  Positions at or past the (clamped) length are ignored."""
import numpy as np
import torch

START_TAG = -2   # baselines/crf.py:11
STOP_TAG = -1    # baselines/crf.py:12


def crf_partial_nll(feats, lengths, trans, allowed):
    """float64 partial-annotation loss and its gradients by autograd -> (per_seq B, dfeats B x L x T, dtrans T x T).
    per_seq[b] = log Z_b - log Z^A_b, Z^A over only the paths that satisfy the mask, with re2nn_crf_nll's path score
    (feat_0 + trans[START], then feat_t[j] + trans[i][j], then trans[i][STOP]); the gradients are those of
    sum_b per_seq[b].  An empty sequence gives 0 and zero gradient rows."""
    B, L, T = feats.shape
    n = torch.from_numpy(np.minimum(np.asarray(lengths, np.int64), L))
    valid = torch.arange(L)[None, :] < n[:, None]
    f64 = torch.from_numpy(np.asarray(feats, np.float64)).requires_grad_(True)
    t64 = torch.from_numpy(np.asarray(trans, np.float64)).requires_grad_(True)
    # pads (and every position of an empty sequence) are unconstrained, so that nothing there is -inf
    a = torch.from_numpy(np.asarray(allowed, bool)) | ~valid[:, :, None]
    fa = torch.where(a, f64, torch.tensor(-np.inf, dtype=torch.float64))

    def log_z(f):
        part = f[:, 0] + t64[START_TAG]
        for t in range(1, L):
            nxt = torch.logsumexp(part[:, :, None] + t64, 1) + f[:, t]
            part = torch.where((t < n)[:, None], nxt, part)
        return torch.logsumexp(part + t64[:, STOP_TAG], 1)

    per_seq = torch.where(n > 0, log_z(f64) - log_z(fa), torch.zeros((), dtype=torch.float64))
    per_seq.sum().backward()
    return per_seq.detach().numpy(), f64.grad.numpy(), t64.grad.numpy()


def crf_constrained_viterbi(feats, lengths, trans, allowed):
    """Viterbi over the scores with -inf in the disallowed cells, in the dtype of `feats` with the Viterbi kernels'
    expressions and first-maximal-index tie rule: part_0[j] = feat_0[j] + trans[START][j], then
    (feat_t[j] + trans[i][j]) + part_{t-1}[i], then part_{n-1}[i] + trans[i][STOP].
    Returns (paths B x L int64, tags at valid positions and 0 at pads; best scores B, -inf for an empty sequence)."""
    B, L, T = feats.shape
    f = np.where(allowed, feats, np.array(-np.inf, feats.dtype))
    paths = np.zeros((B, L), np.int64)
    scores = np.full(B, -np.inf, feats.dtype)
    for b in range(B):
        n = min(int(lengths[b]), L)
        if n <= 0:
            continue
        hist = [f[b, 0] + trans[START_TAG]]
        for t in range(1, n):
            hist.append(((f[b, t][None, :] + trans) + hist[-1][:, None]).max(0))
        fin = hist[-1] + trans[:, STOP_TAG]
        ptr = int(np.argmax(fin))
        scores[b] = fin[ptr]
        paths[b, n - 1] = ptr
        for t in range(n - 1, 0, -1):
            ptr = int(np.argmax((f[b, t, ptr] + trans[:, ptr]) + hist[t - 1]))
            paths[b, t - 1] = ptr
    return paths, scores
