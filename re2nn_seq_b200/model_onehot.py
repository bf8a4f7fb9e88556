"""Drop-in exact ("onehot") i-FST module FARNN_S_O_I_S.

Same constructor signature, parameter names, requires_grad flags, state_dict keys and
forward_local / forward_RE / forward_score / local_decode contracts as
/root/reference/src_seq/farnn/model_onehot.py:310-428 (+ inherited :131-180).

The reference pins this model to the CPU (train_onehot.py:75-78, val.py:13-14) and its drivers
hand it CPU tensors.  Here the parameters live on the GPU and every call runs the CUDA kernels;
inputs on the CPU are copied to the device and the results are returned on the caller's device,
so train_onehot.py / val.py / RE.py work unchanged.
"""
import torch
from torch import nn

from . import autograd_fns, ops
from .model_decompose_single import _UPDATE_NL, _nl_name
from .priority import PriorityLayer
from .utils import exclusive_offsets, flatten


def add_random_noise(obj, amp=0.00001):
    return obj + torch.rand_like(obj) * amp          # utils.py:273-274


class _OnehotBase(nn.Module):
    """Shared pieces of the exact-FST modules (model_onehot.py:131-180): loss, decode and device handling around the
    subclass's `_scores(x, lengths, full_pad)` -> B x L x C, x and lengths on the module's device."""

    def _noisy(self, a):
        """A numpy constructor argument as float32 plus rand_constant-scaled uniform noise (one rand_like draw)."""
        return add_random_noise(torch.from_numpy(a).float(), amp=self.amp)

    def initialize(self):
        a = self.args
        self.t = 1
        if a.local_loss_func not in ('CE', 'CE1', 'ML'):
            raise NotImplementedError()
        self.full_pad = False

    def _device(self):
        ops.require_cuda()
        if not self.language_tensor.is_cuda:
            self.cuda()
        return self.language_tensor.device

    def _device_scores(self, input, lengths, full_pad):
        """(scores, lengths) with the inputs moved to the module's device."""
        dev = self._device()
        x = input.to(dev).contiguous()
        lengths = lengths.to(dev).contiguous()
        return self._scores(x, lengths, full_pad), lengths

    def forward_score(self, input, label, lengths, train=True):
        """B x L x C scores for all L = input.size(1) positions (model_onehot.py:351-428); pad positions
        are computed like the reference does (its callers may read them)."""
        out_dev = input.device
        scores, _ = self._device_scores(input, lengths, full_pad=True)
        return scores.to(out_dev)

    def forward_local(self, input, label, lengths, train=True):
        out_dev = input.device
        scores, dl = self._device_scores(input, lengths, full_pad=self.full_pad)
        dev = scores.device
        N = int(lengths.sum())
        label = label.to(dev)
        flattened_true_labels = flatten(label, dl)
        loss = None
        if train and self.args.local_loss_func == 'ML':
            from .kd import ml_loss
            loss = ml_loss(scores, dl, label, self.args.margin)
        elif train:
            loss = autograd_fns.ce_loss(scores, dl, label.contiguous(), N)
        with torch.no_grad():
            ce1 = self.args.local_loss_func == 'CE1'
            pred, _ = ops.argmax_decode(scores.detach(), dl, exclusive_offsets(dl), N,
                                        clamp_col=self.C - 1 if ce1 else -1, threshold=self.args.threshold,
                                        o_idx=self.o_idx)
        if loss is not None:
            loss = loss.to(out_dev)
        return loss, pred.to(out_dev), flattened_true_labels.to(out_dev)

    def forward_RE(self, input, label, lengths, train=False):
        """Un-flattened decode: (pred B x L, all_scores B x L x C) (model_onehot.py:148-160).  Under CE1
        the returned scores carry the clamped last column, as the reference's do."""
        out_dev = input.device
        with torch.no_grad():
            scores, dl = self._device_scores(input, lengths, full_pad=True)
            ce1 = self.args.local_loss_func == 'CE1'
            _, pred = ops.argmax_decode(scores, dl, None, 0, clamp_col=self.C - 1 if ce1 else -1,
                                        threshold=self.args.threshold, o_idx=self.o_idx, want_flat=False,
                                        want_padded=True)
            if ce1:
                scores = scores.clone()
                scores[:, :, self.C - 1].clamp_(max=float(self.args.threshold))
        return pred.to(out_dev), scores.to(out_dev)

    def local_decode(self, all_scores=None):
        """N x C flat scores -> N predictions (model_onehot.py:162-180)."""
        assert torch.is_tensor(all_scores)
        out_dev = all_scores.device
        dev = self._device()
        with torch.no_grad():
            sc = all_scores.detach().to(dev).float().contiguous().unsqueeze(1)      # N x 1 x C
            N = sc.shape[0]
            ones = torch.ones((N,), dtype=torch.int64, device=dev)
            ce1 = self.args.local_loss_func == 'CE1'
            pred, _ = ops.argmax_decode(sc, ones, torch.arange(N, dtype=torch.int64, device=dev), N,
                                        clamp_col=self.C - 1 if ce1 else -1, threshold=self.args.threshold,
                                        o_idx=self.o_idx)
        return pred.to(out_dev)


class FARNN_S_O_I_S(_OnehotBase):
    def __init__(self, language_tensor=None, output_mat=None, wildcard_mat=None, output_wildcard_vector=None,
                 final_vector=None, start_vector=None, priority_mat=None, args=None, o_idx=0, is_cuda=False):
        super().__init__()
        self.is_cuda = torch.cuda.is_available() and is_cuda
        self.args = args
        C, S = output_mat.shape
        self.S, self.C = S, C
        self.amp = args.rand_constant
        self.h0 = nn.Parameter(self._noisy(start_vector), requires_grad=False)
        self.hT = nn.Parameter(self._noisy(final_vector), requires_grad=False)
        self.language_tensor = nn.Parameter(self._noisy(language_tensor), requires_grad=True)      # (V+1) x S x S
        self.wildcard_mat = nn.Parameter(self._noisy(wildcard_mat), requires_grad=False)            # S x S
        self.output_mat = nn.Parameter(torch.from_numpy(output_mat).float(), requires_grad=False)
        self.output_wildcard_vector = nn.Parameter(torch.from_numpy(output_wildcard_vector).float(),
                                                   requires_grad=False)
        self.priority_layer = PriorityLayer(self.C, priority_mat)
        self.o_idx = o_idx
        self.initialize()
        if torch.cuda.is_available():
            self.cuda()

    def invalidate_caches(self):
        """Drop the cached language + wildcard sum.  It is keyed on (data_ptr, _version), which in-place writes
        through ``p.data`` do not bump -- call this after such writes.  Called automatically by train() / eval(),
        load_state_dict() and .to() / .cuda()."""
        self._sum_cache = {}

    def train(self, mode=True):
        self.invalidate_caches()
        return super().train(mode)

    def _apply(self, fn, *a, **k):
        self.invalidate_caches()
        return super()._apply(fn, *a, **k)

    def _load_from_state_dict(self, *a, **k):
        self.invalidate_caches()
        return super()._load_from_state_dict(*a, **k)

    def _consts(self, full_pad):
        a = self.args
        if not hasattr(self, '_sum_cache'):
            self._sum_cache = {}
        return dict(update_nonlinear=_nl_name(a.update_nonlinear, _UPDATE_NL), max_semiring=(a.train_mode == 'max'),
                    ce1=(a.local_loss_func == 'CE1'), use_priority=bool(a.use_priority), full_pad=bool(full_pad),
                    cache=self._sum_cache)

    def _scores(self, x, lengths, full_pad):
        tensors = [self.h0, self.hT, self.language_tensor, self.wildcard_mat, self.output_mat,
                   self.output_wildcard_vector]
        if self.args.train_mode == 'max' and torch.is_grad_enabled() and any(t.requires_grad for t in tensors) \
                and not full_pad:
            from .model_fst import ifst_onehot_max_scores      # max-product training: argmax-routed gradient
            return ifst_onehot_max_scores(self, x, lengths)
        pr = (self.priority_layer.priority_mat, self.priority_layer.priority_bias)
        return autograd_fns.onehot_scores(self._consts(full_pad), tensors, pr, x, lengths, x.shape[1])

    def time_recurrence(self, input, lengths):
        """Measurement hook (bench.py roofline): milliseconds of ONE onehot_recurrence_kernel launch over this batch,
        CUDA events on the launching stream."""
        dev = self._device()
        x, lengths = input.to(dev).contiguous(), lengths.to(dev).contiguous()
        c = self._consts(self.full_pad)
        with torch.no_grad():
            o = ops.output_vector_sum(self.output_mat, None if c['ce1'] else self.output_wildcard_vector)
            summed = ops.onehot_sum_tensor(self.language_tensor, self.wildcard_mat)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ops.onehot_recurrence(x, lengths, x.shape[1], summed, None, o, self.h0, self.hT, c['update_nonlinear'],
                                  c['max_semiring'], c['full_pad'], presummed=True)
            e1.record()
            torch.cuda.synchronize()
        return e0.elapsed_time(e1)
