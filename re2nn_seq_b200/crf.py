"""CRF with the reference's interface (src_seq/baselines/crf.py:29-260), computed by the
warp-per-sequence CUDA kernels in csrc/crf.cu."""
import torch
from torch import nn

from . import ops

START_TAG = -2
STOP_TAG = -1


class _CrfNll(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feats, transitions, lengths, tags, grad_on):
        need = grad_on and (ctx.needs_input_grad[0] or ctx.needs_input_grad[1])
        loss, _, part = ops.crf_nll(feats, transitions, lengths, tags, save=need)
        if need:
            ctx.save_for_backward(feats, transitions, lengths, tags, part)
        return loss

    @staticmethod
    def backward(ctx, g):
        feats, transitions, lengths, tags, part = ctx.saved_tensors
        dfeats, dtrans = ops.crf_nll_backward(feats, transitions, lengths, tags, part, g.contiguous().float())
        return dfeats, dtrans, None, None, None


class _CrfPartialNll(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feats, transitions, lengths, allowed, grad_on):
        need = grad_on and (ctx.needs_input_grad[0] or ctx.needs_input_grad[1])
        loss, _, parts = ops.crf_partial_nll(feats, transitions, lengths, allowed, save=need)
        if need:
            ctx.save_for_backward(feats, transitions, lengths, allowed, *parts)
        return loss

    @staticmethod
    def backward(ctx, g):
        feats, transitions, lengths, allowed, part, part_a = ctx.saved_tensors
        dfeats, dtrans = ops.crf_partial_nll_backward(feats, transitions, lengths, allowed, part, part_a,
                                                      g.contiguous().float())
        return dfeats, dtrans, None, None, None


def partial_allowed(labels, T, unknown=-1, lengths=None):
    """Allowed-tag mask (B x L x T bool) of partially labelled sequences: one-hot at a known label, every one of the
    T columns where the label is `unknown` and, given `lengths`, at the pads.  A sequence without any known label is
    the free lattice, so it adds nothing to CRF.partial_neg_log_likelihood_loss."""
    known = labels != unknown
    allowed = torch.nn.functional.one_hot(torch.where(known, labels, torch.zeros_like(labels)).long(), T).bool()
    allowed |= ~known[:, :, None]
    if lengths is not None:
        pad = torch.arange(labels.shape[1], device=labels.device)[None, :] >= lengths.to(labels.device)[:, None]
        allowed |= pad[:, :, None]
    return allowed


class CRF(nn.Module):
    def __init__(self, tagset_size, gpu):
        super().__init__()
        self.gpu = gpu
        self.tagset_size = tagset_size
        T = tagset_size + 2
        init = torch.zeros(T, T)
        init[:, START_TAG] = -10000.0      # nothing transitions into START   (crf.py:40)
        init[STOP_TAG, :] = -10000.0       # nothing leaves STOP              (crf.py:41)
        self.transitions = nn.Parameter(init, requires_grad=True)

    @staticmethod
    def _lengths(mask):
        return mask.long().sum(1)

    def _prep(self, feats):
        ops.require_cuda()
        dev = self.transitions.device
        if not self.transitions.is_cuda:
            raise RuntimeError("re2nn_b200 CRF: module must live on a CUDA device (call .cuda())")
        return feats.to(dev).float().contiguous()

    def neg_log_likelihood_loss(self, feats, mask, tags, lengths=None):
        assert feats.size(2) == self.tagset_size + 2          # crf.py:58
        feats = self._prep(feats)
        dev = feats.device
        lengths = (self._lengths(mask) if lengths is None else lengths).to(dev).contiguous()
        tags = tags.to(dev).contiguous()
        return _CrfNll.apply(feats, self.transitions, lengths, tags, torch.is_grad_enabled())

    @staticmethod
    def _check_allowed(allowed, feats, lengths):
        """allowed as the kernels take it (contiguous, bool / uint8, on feats' device, feats' B x L x T shape, at least
        one tag at every valid position), else ValueError before any kernel runs.  One reduction and one sync."""
        if not isinstance(allowed, torch.Tensor) or allowed.dtype not in (torch.bool, torch.uint8):
            raise ValueError("CRF: allowed must be a bool or uint8 tensor, got %s"
                             % (allowed.dtype if isinstance(allowed, torch.Tensor) else type(allowed).__name__))
        if allowed.device != feats.device:
            raise ValueError("CRF: allowed is on %s, the scores on %s" % (allowed.device, feats.device))
        if allowed.shape != feats.shape:
            raise ValueError("CRF: allowed has shape %s, expected the scores' B x L x T %s"
                             % (tuple(allowed.shape), tuple(feats.shape)))
        valid = torch.arange(feats.shape[1], device=feats.device)[None, :] < lengths[:, None]
        if bool((valid & ~allowed.bool().any(2)).any()):
            raise ValueError("CRF: allowed leaves a valid position without any tag")
        return allowed.contiguous()

    def partial_neg_log_likelihood_loss(self, feats, mask, allowed, lengths=None):
        """Partial-annotation loss summed over sequences: log Z - log Z^A per sequence, Z^A over only the tag sequences
        that put every valid position t of sequence b on a tag j with allowed[b, t, j] set (B x L x T, bool / uint8;
        partial_allowed builds it from labels with an unknown marker).  A one-hot mask of the gold tags gives
        neg_log_likelihood_loss; an all-true mask gives exactly 0 and a zero gradient."""
        assert feats.size(2) == self.tagset_size + 2
        feats = self._prep(feats)
        dev = feats.device
        lengths = (self._lengths(mask) if lengths is None else lengths).to(dev).contiguous()
        allowed = self._check_allowed(allowed, feats, lengths)
        return _CrfPartialNll.apply(feats, self.transitions, lengths, allowed, torch.is_grad_enabled())

    def constrained_decode(self, feats, mask, allowed, lengths=None):
        """Best tag sequence among those that keep every valid position on an allowed tag -> B x L padded path in
        _viterbi_decode's convention (pads 0, the final pointer in the last column of a short row).  The Viterbi
        kernels run on the scores with -inf in the disallowed cells, so an all-true mask gives _viterbi_decode's path."""
        assert feats.size(2) == self.tagset_size + 2
        with torch.no_grad():
            feats = self._prep(feats.detach())
            lengths = (self._lengths(mask) if lengths is None else lengths).to(feats.device).contiguous()
            allowed = self._check_allowed(allowed, feats, lengths)
            masked = feats.masked_fill(~allowed.bool(), float('-inf'))
            _, padded = ops.crf_viterbi(masked, self.transitions.detach(), lengths, want_padded=True)
        return padded

    def _viterbi_decode(self, feats, mask, lengths=None):
        assert feats.size(2) == self.tagset_size + 2          # crf.py:114
        with torch.no_grad():
            feats = self._prep(feats.detach())
            lengths = (self._lengths(mask) if lengths is None else lengths).to(feats.device).contiguous()
            _, padded = ops.crf_viterbi(feats, self.transitions.detach(), lengths, want_padded=True)
        return None, padded

    def _viterbi_decode_nbest(self, feats, mask, nbest, lengths=None):
        """NCRF++'s N-best decode -> (path_score B x K, decode_idx B x L x K): the K best distinct tag sequences, best
        first (rank 0 is _viterbi_decode's path).  path_score is NCRF++'s softmax over the K returned path scores; a
        rank that does not exist (fewer than K sequences) scores 0 and decodes to -1 at valid positions."""
        assert feats.size(2) == self.tagset_size + 2
        with torch.no_grad():
            feats = self._prep(feats.detach())
            lengths = (self._lengths(mask) if lengths is None else lengths).to(feats.device).contiguous()
            decode_idx, scores = ops.crf_nbest(feats, self.transitions.detach(), lengths, nbest)
            path_score = torch.softmax(scores, 1)       # missing ranks (-inf) get 0; a row without any sequence NaN:
            path_score = torch.where(torch.isfinite(scores), path_score, torch.zeros_like(path_score))
        return path_score, decode_idx

    def marginals(self, feats, mask, lengths=None):
        """Per-token posteriors P(y_t = j | x) (B x L x T, zero at pads) and log Z (B)."""
        assert feats.size(2) == self.tagset_size + 2
        with torch.no_grad():
            feats = self._prep(feats.detach())
            lengths = (self._lengths(mask) if lengths is None else lengths).to(feats.device).contiguous()
            return ops.crf_marginals(feats, self.transitions.detach(), lengths)

    def forward(self, feats, mask):
        return self._viterbi_decode(feats, mask)
