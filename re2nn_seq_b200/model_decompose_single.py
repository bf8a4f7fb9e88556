"""Drop-in i-FST decompose modules: FARNN_S_D_W_I_S and FARNN_S_SF.

Same class names, constructor signatures, parameter names / shapes / requires_grad flags,
state_dict keys and forward_local / forward contracts as
/root/reference/src_seq/farnn/model_decompose_single.py:12-304 (FARNN_S_D_W_I_S) and :307-580
(FARNN_S_SF); shared helpers follow farnn/model_decompose.py:69-102,191-241,339-371.
All arithmetic of the hot path runs in the CUDA kernels behind re2nn_seq_b200.ops; this file
only owns parameters, picks launch-time constants from ``args`` and wires autograd.

Constructor RNG: torch random draws are made in the same order and with the same calls as the
reference constructor, so a module built after torch.manual_seed(s) is bit-identical to the
reference module built after the same seed (tests/test_host_modules.py).
"""
import numpy as np
import torch
from torch import nn

from . import autograd_fns, ops
from .crf import CRF
from .priority import PriorityLayer
from .utils import exclusive_offsets, flatten, get_length_mask

_UPDATE_NL = ('none', 'relu', 'tanh', 'relutanh')
_ADD_NL = ('none', 'relu', 'tanh', 'sigmoid', 'relutanh')


def _nl_name(name, allowed):
    return name if name in allowed else 'none'     # the reference falls through to "pass" (identity)


class _DecomposeBase(nn.Module):
    """Shared pieces of the rank-R i-FST modules."""

    def __init__(self, args, C, S, R, start_vector, final_vector, priority_mat, o_idx, fwd_params,
                 word_embed=None, is_cuda=True):
        """The construction sequence of every rank-R module; its order fixes the RNG draws and the parameter
        registration order (optimizer checkpoints index parameters by position).  C x S x R are the label / state /
        rank sizes before the CRF's two extra labels, fwd_params the subclass's init_forward_parameters arguments;
        the token-input modules pass word_embed and so own `embedding` and `beta_vec`."""
        super().__init__()
        self.is_cuda = torch.cuda.is_available() if is_cuda else False
        self.additional_states = args.additional_states
        self.args = args
        if word_embed is not None:
            self.embedding = nn.Embedding.from_pretrained(torch.from_numpy(word_embed).float(),
                                                          freeze=(not args.train_word_embed))
        self.C, self.S, self.R = C, S, R
        self.t = 1
        self.use_crf = bool(args.use_crf)
        if self.use_crf:
            self.crf = CRF(self.C, self.is_cuda)
            self.C += 2
        self.priority_layer = PriorityLayer(self.C, priority_mat)
        self.random = bool(args.random)
        self.h0 = nn.Parameter(self.pad_additional_states(torch.from_numpy(start_vector).float()),
                               requires_grad=bool(args.train_h0))
        self.hT = nn.Parameter(self.pad_additional_states(torch.from_numpy(final_vector).float()),
                               requires_grad=bool(args.train_hT))
        self.init_forward_parameters(*fwd_params)
        if word_embed is not None:
            self.beta = args.beta
            self.beta_vec = nn.Parameter(torch.tensor([self.beta] * self.R).float(), requires_grad=bool(args.train_beta))
        self.o_idx = o_idx
        self.not_o_idxs = [i for i in range(self.C) if i != self.o_idx]
        self.initialize()

    # ---- construction helpers (model_decompose.py:191-220) ------------------------------------
    def get_random(self, sizes):
        kind = self.args.random_pad_func
        if kind == 'uniform':
            return torch.rand(sizes)
        if kind == 'normal':
            return torch.randn(sizes)
        t = torch.randn(sizes)
        nn.init.xavier_normal_(t)
        return t

    def pad_additional_states(self, obj):
        """Grow every dimension equal to S by additional_states; 1-D pads with zeros, higher ranks
        with rand_constant-scaled noise (the noise tensor is drawn even when nothing grows)."""
        shape = tuple(obj.shape)
        grown = tuple(d + self.additional_states if d == self.S else d for d in shape)
        if len(shape) == 1:
            out = torch.zeros(grown)
        elif len(shape) in (2, 3, 4):
            out = self.get_random(grown) * self.args.rand_constant
        else:
            raise NotImplementedError()
        out[tuple(slice(0, d) for d in shape)] = obj
        return out

    def initialize(self):
        a = self.args
        self.additional_nonlinear = a.additional_nonlinear
        if a.train_mode not in ('sum', 'max'):
            raise NotImplementedError()
        if a.local_loss_func not in ('CE', 'CE1', 'ML'):
            raise NotImplementedError()
        if a.sigmoid_exponent <= 0 and a.farnn:
            raise AssertionError("sigmoid_exponent must be positive")
        # inference default: the fastest PARITY-GRADE mode of the device (split-fp16 / 3xTF32 tensor cores: scores within
        # 1e-5 of the reference, decoded tags identical); 'fp32' selects the CUDA-core path, 'bf16' the stated-bound mode
        self.precision = getattr(a, 'precision', 'auto')
        self._cache = {}

    def _gate_params(self, S_full):
        """Update (farnn >= 1) and reset (farnn == 2) gate parameters, model_decompose.py:137-171."""
        a = self.args
        if a.farnn not in (0, 1, 2):
            raise NotImplementedError()
        if a.farnn >= 1:
            self.Wss1 = nn.Parameter(torch.randn((S_full, S_full)).float(), requires_grad=True)
            self.Wrs1 = nn.Parameter(torch.randn((self.R, S_full)).float(), requires_grad=True)
            self.bs1 = nn.Parameter(torch.ones((1, S_full)).float() * a.bias_init, requires_grad=True)
        if a.farnn == 1 and a.xavier:
            nn.init.xavier_normal_(self.Wss1)
            nn.init.xavier_normal_(self.Wrs1)
            nn.init.xavier_normal_(self.bs1)
        if a.farnn == 2:
            self.Wss2 = nn.Parameter(torch.randn((S_full, S_full)).float(), requires_grad=True)
            self.Wrs2 = nn.Parameter(torch.randn((self.R, S_full)).float(), requires_grad=True)
            self.bs2 = nn.Parameter(torch.ones((1, S_full)).float() * a.bias_init, requires_grad=True)
            if a.xavier:
                for w in (self.Wss1, self.Wrs1, self.Wss2, self.Wrs2):
                    nn.init.xavier_normal_(w)

    def _resolved_precision(self):
        """'auto' picks the fastest parity-grade mode the device has: split-fp16 tensor cores when the state is
        bounded by the update nonlinearity (fp16 planes need |operand| < 65504), 3xTF32 otherwise, fp32 CUDA
        cores without tcgen05.  Training (grad enabled) uses `train_precision` (default fp32; 'auto', 'tf32x3' or
        'fp16x3' run the forward GEMMs on tensor cores, the backward stays fp32)."""
        training = torch.is_grad_enabled() and any(q.requires_grad for q in self.parameters())
        prec = getattr(self, 'train_precision', 'fp32') if training else self.precision
        if prec != 'auto':
            return prec
        if not ops.has_tcgen05():
            return 'fp32'
        return 'fp16x3' if self.args.update_nonlinear in ('tanh', 'relutanh') else 'tf32x3'

    def _max_needs_grad(self, tensors):
        """train_mode == 'max' with a gradient wanted: the differentiable dense-transition form (model_fst.py)."""
        return self.args.train_mode == 'max' and torch.is_grad_enabled() and any(t.requires_grad for t in tensors)

    # ---- launch-time constants -----------------------------------------------------------------
    @property
    def _S_full(self):
        return self.S + self.additional_states

    def _device(self):
        ops.require_cuda()
        dev = self.S1.device
        if dev.type != 'cuda':
            raise RuntimeError("re2nn_b200: %s must live on a CUDA device (call .cuda()); there is no CPU path"
                               % type(self).__name__)
        return dev

    def _host_shape(self, lengths):
        """(L, N) = (max length, total valid tokens) with a single device->host sync."""
        if lengths.is_cuda:
            L, N = torch.stack([lengths.max(), lengths.sum()]).tolist()
        else:
            L, N = int(lengths.max()), int(lengths.sum())
        return int(L), int(N)

    def _params_for_fn(self):
        """Ordered (name, tensor) list handed to the autograd function."""
        names = ['h0', 'hT', 'S1', 'S2', 'C_output_mat', 'wildcard_mat', 'wildcard_output_vector']
        if self.args.farnn >= 1:
            names += ['Wss1', 'Wrs1', 'bs1']
        if self.args.farnn == 2:
            names += ['Wss2', 'Wrs2', 'bs2']
        return names

    # ---- decode (model_decompose.py:339-371) ------------------------------------------------------
    def decode(self, all_scores, flattened_all_scores, mask, lengths, _shape=None, _offsets=None, _flat_out=None):
        """all_scores B x L x C -> flat predictions N (int64).  `flattened_all_scores` and `mask`
        are accepted for signature compatibility; the kernels address valid positions directly."""
        with torch.no_grad():
            dev = all_scores.device
            lengths = lengths.to(dev).contiguous()
            N = _shape[1] if _shape is not None else int(lengths.sum())
            offsets = exclusive_offsets(lengths) if _offsets is None else _offsets
            ce1 = self.args.local_loss_func == 'CE1'
            sc = all_scores.detach().contiguous()
            if self.use_crf:
                flat, _ = ops.crf_viterbi(sc, self.crf.transitions.detach(), lengths, offsets, N,
                                          clamp_col=self.C - 3 if ce1 else -1, threshold=self.args.threshold,
                                          o_idx=self.o_idx, want_flat=True, want_padded=False, flat_out=_flat_out)
            else:
                flat, _ = ops.argmax_decode(sc, lengths, offsets, N, clamp_col=self.C - 1 if ce1 else -1,
                                            threshold=self.args.threshold, o_idx=self.o_idx, flat_out=_flat_out)
        return flat

    def _crf_only(self, what):
        if not self.use_crf:
            raise NotImplementedError("%s needs a CRF head (use_crf=1); %s decodes per position"
                                      % (what, type(self).__name__))

    def _decode_scores(self, input, lengths):
        """(scores B x L x C as decode's Viterbi sees them, CE1 flag): under CE1 column C-3 clamped to the threshold."""
        sc = self.forward_scores(input, lengths).detach().contiguous()
        ce1 = self.args.local_loss_func == 'CE1'
        if ce1:
            sc = sc.clone()
            sc[:, :, self.C - 3] = torch.minimum(sc[:, :, self.C - 3], sc.new_tensor(self.args.threshold))
        return sc, ce1

    def _report_tags(self, pred, lengths, ce1):
        """decode's report: under CE1 tag C-3 at a valid position is o_idx."""
        if not ce1:
            return pred
        valid = get_length_mask(lengths, pred.shape[1])
        if pred.dim() == 3:
            valid = valid[:, :, None]
        return torch.where(valid & (pred == self.C - 3), torch.full_like(pred, self.o_idx), pred)

    @staticmethod
    def _allowed_rows(allowed, sc):
        """A caller's mask on the scores' device and cut to their L (the CRF checks it)."""
        if isinstance(allowed, torch.Tensor) and allowed.dim() == 3:
            allowed = allowed.to(sc.device)[:, :sc.shape[1]]
        return allowed

    def forward_nbest(self, input, lengths, nbest=1):
        """N-best CRF decoding with confidences -> (pred B x L x K int64, seq_prob B x K, marginals B x L x C).
        pred[..., 0] is what forward_local decodes (padded, in the caller's order; -1 marks a rank with no sequence,
        pads are 0), seq_prob[:, k] = P(path k | x) and marginals[b, t, c] = P(y_t = c | x), zero at pads.  Under CE1
        decode's clamp of column C-3 to the threshold applies to both, and tag C-3 is reported as o_idx in pred.
        Eager (no graph capture), no gradient."""
        self._crf_only('forward_nbest')
        with torch.no_grad():
            dev = self._device()
            lengths = lengths.to(dev).contiguous()
            sc, ce1 = self._decode_scores(input, lengths)
            trans = self.crf.transitions.detach()
            pred, score = ops.crf_nbest(sc, trans, lengths, nbest)
            marg, log_z = ops.crf_marginals(sc, trans, lengths)
            pred = self._report_tags(pred, lengths, ce1)
            seq_prob = torch.exp(score - log_z[:, None])
        return pred, seq_prob, marg

    def forward_partial(self, input, lengths, allowed):
        """Partial-annotation CRF loss (differentiable scalar, summed over sequences like forward_local's CRF loss):
        log Z - log Z^A per sequence, where Z^A counts only the tag sequences that keep every valid position on an
        allowed tag.  allowed: B x L' x C bool / uint8 over the CRF's C columns (START / STOP included), L' >= the
        longest length; crf.partial_allowed builds it from labels with an unknown marker.  With every label known it
        is forward_local's training loss; a sequence with none known adds nothing.  Eager."""
        self._crf_only('forward_partial')
        dev = self._device()
        lengths = lengths.to(dev).contiguous()
        sc = self.forward_scores(input, lengths)
        return self.crf.partial_neg_log_likelihood_loss(sc, None, self._allowed_rows(allowed, sc), lengths=lengths)

    def forward_constrained(self, input, lengths, allowed):
        """Constrained CRF decoding -> pred B x L int64 (padded, in the caller's order): the best tag sequence that keeps
        every valid position on a tag allowed there (allowed as in forward_partial), e.g. tokens fixed by a person or a
        rule.  CE1's clamp of column C-3 and its o_idx report apply as in forward_nbest, so an all-true mask gives what
        forward_local decodes.  Eager, no gradient."""
        self._crf_only('forward_constrained')
        with torch.no_grad():
            dev = self._device()
            lengths = lengths.to(dev).contiguous()
            sc, ce1 = self._decode_scores(input, lengths)
            pred = self.crf.constrained_decode(sc, None, self._allowed_rows(allowed, sc), lengths=lengths)
            return self._report_tags(pred, lengths, ce1)

    # ---- loss + decode tail shared by forward_local / forward (model_decompose_single.py:271-304) ---
    def _length_order(self, lengths, re_tags, L=None):
        """Process sequences longest-first so 128-row tiles finish together and are skipped once all their rows
        are done (the reference computes every pad position; only valid positions are observable).  Outputs keep
        the caller's order: flat predictions are scattered through the original offsets.
        -> (order, offsets_sorted, lengths_sorted, offsets) or (None, None, None, None)."""
        if not getattr(self, 'sort_by_length', True) or re_tags is not None or lengths.shape[0] <= 128:
            return None, None, None, None
        if L is not None and lengths.is_cuda:
            fast = ops.length_order(lengths, L)          # one launch: counting sort + offsets + gathers
            if fast is not None:
                order, ls, offs, offs_sorted = fast
                return order, offs_sorted, ls, offs
        # 16-bit keys: the radix sort needs 2 passes instead of 8.  The order is only a scheduling heuristic (any
        # permutation gives the same outputs), so lengths beyond int16 merely sort less usefully.
        _, order = torch.sort(lengths.to(torch.int16), descending=True, stable=True)
        offs = exclusive_offsets(lengths)
        return order, offs.index_select(0, order), lengths.index_select(0, order), offs

    # ---- CUDA-graph replay of the inference path --------------------------------------------------------
    # One forward_local is ~80-110 small dependent launches; on the host that is 10+ us per launch, more than
    # the kernels take.  Inference calls (no grad, no KD) are therefore captured once per (shape, precision,
    # parameter version) with static buffers and replayed: one graph launch per batch.
    def _graph_key(self, B, Lpad, L, tag):
        vers = tuple((q.data_ptr(), q._version) for q in self.parameters())
        return (tag, B, Lpad, L, self._resolved_precision(), bool(getattr(self, 'sort_by_length', True)),
                int(getattr(self, 'infer_chunks', 4)), ops.profile_enabled(), vers)

    def _infer_body(self, inp, label, lengths, L):
        """Sync-free inference body: every shape is a function of (B, Lpad, L) only."""
        B = lengths.shape[0]
        nmax = B * L
        order, offsets, ls, offs0 = self._length_order(lengths, None, L)
        if order is None:
            offs0 = exclusive_offsets(lengths)
        true = ops.flatten_i64(label.contiguous(), lengths, offs0, L, nmax)
        if order is not None:
            lengths = ls
            inp = inp.index_select(0, order)
        else:
            offsets = offs0
        chunks = self._infer_chunks(B) if order is not None else None
        if chunks is None:
            scores = self.forward_scores(inp, lengths, (L, nmax), fuse=True)      # scores feed the decoder only
            pred = self.decode(scores, None, None, lengths, _shape=(L, nmax), _offsets=offsets)
            return pred, true
        # Sequences are sorted longest-first, so the recurrence of a later chunk finishes earlier (its tiles stop at
        # their own last step) and every row tile is independent: fork one stream per chunk.  Label scoring and
        # Viterbi of the short chunks then run on the SMs their recurrence has already released while the longest
        # chunk is still iterating; only the post-processing of the LAST chunk to finish stays on the critical path.
        self._warm_tables()                                  # shared tables on the main stream, before the fork
        pred = torch.empty((nmax,), dtype=torch.int64, device=lengths.device)
        main = torch.cuda.current_stream()
        fork = torch.cuda.Event()
        fork.record(main)
        if not hasattr(self, '_chunk_streams') or len(self._chunk_streams) < len(chunks):
            self._chunk_streams = [torch.cuda.Stream() for _ in chunks]
        for st, (b0, b1) in zip(self._chunk_streams, chunks):
            st.wait_event(fork)
            with torch.cuda.stream(st):
                lc = lengths[b0:b1]
                sc = self.forward_scores(inp[b0:b1], lc, (L, nmax), fuse=True)
                self.decode(sc, None, None, lc, _shape=(L, nmax), _offsets=offsets[b0:b1], _flat_out=pred)
                done = torch.cuda.Event()
                done.record(st)
            main.wait_event(done)
        return pred, true

    def _infer_chunks(self, B):
        """[(b0, b1), ...] row ranges (multiples of the 128-row tile) for the multi-stream inference body, or None."""
        n = int(getattr(self, 'infer_chunks', 4))
        if self.args.farnn >= 1:
            n = min(n, 2)        # gated steps are bound by L2 traffic of the state / gate arrays: measured best with 1-2 chunks
        if n <= 1 or B < 256 * n:
            return None
        # only the resident recurrence kernel leaves SMs idle as its short tiles finish; with one launch per step GEMM
        # (large S / R) the chunks would just compete for the machine (measured: cfg5 shapes 10.0 -> 12.2 ms)
        S, R = self.S1.shape
        if not ops.recurrence_is_resident(S, R, self.args.farnn, self._resolved_precision()):
            return None
        per = ((B + n - 1) // n + 127) // 128 * 128
        return [(b0, min(B, b0 + per)) for b0 in range(0, B, per)]

    def _warm_tables(self):
        """Everything cached per parameter version, computed on the CURRENT stream before chunk streams fork: the
        operand-format weight copies here, the token / gate tables and the output-vector sum in the subclass."""
        names = self._params_for_fn()
        p = {n: getattr(self, n).detach().contiguous() for n in names}
        autograd_fns._weight_prep(self._recurrence_consts(), p, self._cache)

    # Capture policy.  An evaluation sweep (val.py:7-43 runs train / dev / test after every epoch) sees a new
    # (B, L) almost every batch and new parameter versions every epoch; capturing each of them would cost a warm-up
    # forward + a capture forward + instantiation per batch and pin one private memory pool per capture.  So:
    #   * a key is captured only when it is seen for the SECOND time (first sighting runs eagerly);
    #   * entries are evicted least-recently-used, entries captured under other parameter versions first;
    #   * the pools are capped by `graph_pool_bytes` (default 1/8 of the device memory).
    _GRAPH_MAX_ENTRIES = 8

    def invalidate_caches(self):
        """Drop the token / gate / output-sum tables and every captured graph.  The caches are keyed on
        (data_ptr, _version) of the parameters, which in-place writes through ``p.data`` (EMA, weight swaps, legacy
        optimisers) do NOT bump -- call this after such writes.  Called automatically by train() / eval(),
        load_state_dict() and .to() / .cuda()."""
        if getattr(self, '_cache', None) is not None:
            self._cache.clear()
        self._graphs = {}
        self._graph_seen = {}

    def train(self, mode=True):
        self.invalidate_caches()
        return super().train(mode)

    def _apply(self, fn, *a, **k):
        self.invalidate_caches()
        return super()._apply(fn, *a, **k)

    def _load_from_state_dict(self, *a, **k):
        self.invalidate_caches()
        return super()._load_from_state_dict(*a, **k)

    def _graph_evict(self, need_bytes, vers):
        cap = getattr(self, 'graph_pool_bytes', None)
        if cap is None:
            cap = torch.cuda.get_device_properties(self.S1.device).total_memory // 8
        g = self._graphs
        for k in [k for k, e in g.items() if e['vers'] != vers]:      # stale parameter versions can never hit again
            del g[k]
        def used():
            return sum(e['bytes'] for e in g.values())
        while g and (len(g) >= self._GRAPH_MAX_ENTRIES or used() + need_bytes > cap):
            del g[min(g, key=lambda k: g[k]['tick'])]
        return used() + need_bytes <= cap

    def _infer_graphed(self, inp, label, lengths, shape, tag):
        L, N = shape
        B, Lpad = lengths.shape[0], inp.shape[1]
        if not hasattr(self, '_graphs'):
            self._graphs, self._graph_seen = {}, {}
        self._graph_tick = getattr(self, '_graph_tick', 0) + 1
        key = self._graph_key(B, Lpad, L, tag)
        vers = key[-1]
        ent = self._graphs.get(key)
        if ent is None:
            seen = self._graph_seen.get(key, 0)
            if len(self._graph_seen) > 256:
                self._graph_seen.clear()
            self._graph_seen[key] = seen + 1
            S_full, C_full = self._S_full, self.C
            est = B * L * (2 * S_full + 2 * C_full + 8) * 4 + B * Lpad * 16      # alpha, beta, scores, partition history
            if seen == 0 or not self._graph_evict(est, vers):
                pred, true = self._infer_body(inp, label.contiguous(), lengths, L)   # first sighting: eager
                return None, pred[:N], true[:N]
            sx, sy, sl = inp.clone(), label.contiguous().clone(), lengths.clone()
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):                   # warm-up outside capture (lazy init, caches)
                self._infer_body(sx, sy, sl, L)
            torch.cuda.current_stream().wait_stream(side)
            l0 = ops.launches()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                pred, true = self._infer_body(sx, sy, sl, L)
            ent = dict(g=g, x=sx, y=sy, l=sl, pred=pred, true=true, launches=ops.launches() - l0, bytes=est, vers=vers)
            self._graphs[key] = ent
        ent['tick'] = self._graph_tick
        ent['x'].copy_(inp, non_blocking=True)
        ent['y'].copy_(label, non_blocking=True)
        ent['l'].copy_(lengths, non_blocking=True)
        ent['g'].replay()
        ops._count(ent['launches'])
        return None, ent['pred'][:N].clone(), ent['true'][:N].clone()

    def _can_graph(self, train, re_tags):
        return (not train) and re_tags is None and not torch.is_grad_enabled() and getattr(self, 'use_cuda_graph', True) \
            and self.args.marryup_type not in ('kd', 'pr') and not getattr(self, 'full_pad', False)

    def _forward_body(self, input, label, lengths, train, re_tags, tag):
        """forward_local / forward: a graph replay where _can_graph allows it, else the scores (longest-first when
        _length_order sorts) and the loss + decode tail.  _device_input is the subclass's forward_scores input
        conversion."""
        dev = self._device()
        lengths = lengths.to(dev).contiguous()
        shape = self._host_shape(lengths)
        if self._can_graph(train, re_tags):
            return self._infer_graphed(self._device_input(input, dev), label.to(dev), lengths, shape, tag)
        order, offsets, ls, _ = self._length_order(lengths, re_tags, shape[0])
        if order is None:
            all_scores = self.forward_scores(input, lengths, shape)
            return self._finish(all_scores, label, lengths, train, re_tags, shape)
        all_scores = self.forward_scores(input.to(dev).index_select(0, order), ls, shape)
        return self._finish(all_scores, label, ls, train, re_tags, shape, order, offsets, lengths)

    def _finish(self, all_scores, label, lengths, train, re_tags, shape, order=None, offsets=None, orig=None):
        L, N = shape
        dev = all_scores.device
        label = label.to(dev)
        if order is None:
            flattened_true_labels = ops.flatten_i64(label.contiguous(), lengths, exclusive_offsets(lengths), L, N)
        else:
            flattened_true_labels = ops.flatten_i64(label.contiguous(), orig, exclusive_offsets(orig), L, N)
            label = label.index_select(0, order)
        loss = None
        # Training: the decoder (Viterbi: one latency-bound chain per sequence, a few warps per SM) and the loss (the CRF
        # partition sweep: the same shape of work) are independent readers of the scores -> the decoder runs on a side
        # stream next to the loss and is joined before returning (cfg3: 0.13 ms of the step).
        pred = None
        side = None
        if train and all_scores.is_cuda and self.use_crf and getattr(self, 'overlap_decode', True):
            main = torch.cuda.current_stream()
            side = getattr(self, '_decode_stream', None)
            if side is None or side.device != all_scores.device:
                side = self._decode_stream = torch.cuda.Stream(device=all_scores.device)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                pred = self.decode(all_scores.detach(), None, None, lengths, _shape=shape, _offsets=offsets)
        if train:
            lab = label.contiguous()
            if self.use_crf:
                loss = self.crf.neg_log_likelihood_loss(all_scores, None, lab, lengths=lengths)
            elif self.args.local_loss_func == 'ML':
                from .kd import ml_loss
                loss = ml_loss(all_scores, lengths, lab, self.args.margin)
            else:
                # under data parallelism every rank divides by the GLOBAL token count (re2nn_seq_b200/dist.py)
                loss = autograd_fns.ce_loss(all_scores, lengths, lab, getattr(self, 'global_tokens', None) or N)
            mt = self.args.marryup_type
            if mt in ('kd', 'pr'):
                from .kd import KD_loss, PR_loss
                B, Lr, _ = re_tags.size()
                extra = 3 if self.args.use_crf else 1
                re_tags = torch.cat([re_tags.to(dev), torch.zeros(B, Lr, extra, device=dev)], dim=2)
                if mt == 'kd':
                    kl = KD_loss(all_scores, re_tags[:, :L, :], self.args)
                    loss = self.args.c2_kdpr * loss + (1 - self.args.c2_kdpr) * kl
                else:
                    kl = PR_loss(all_scores, re_tags[:, :L, :], self.args)
                    pi = max(self.args.c2_kdpr, self.args.c3_pr ** self.t)
                    loss = pi * loss + (1 - pi) * kl
        if side is not None:
            torch.cuda.current_stream().wait_stream(side)
            pred.record_stream(torch.cuda.current_stream())
        else:
            pred = self.decode(all_scores, None, None, lengths, _shape=shape, _offsets=offsets)
        return loss, pred, flattened_true_labels

    def _recurrence_consts(self):
        a = self.args
        return dict(farnn=a.farnn, max_semiring=(a.train_mode == 'max'), update_nonlinear=_nl_name(a.update_nonlinear, _UPDATE_NL),
                    sigmoid_exponent=float(a.sigmoid_exponent), precision=self._resolved_precision(),
                    ce1=(a.local_loss_func == 'CE1'), use_priority=bool(a.use_priority),
                    additional_nonlinear=_nl_name(a.additional_nonlinear, _ADD_NL),
                    full_pad=bool(getattr(self, 'full_pad', False)) or a.marryup_type in ('kd', 'pr'))


class FARNN_S_D_W_I_S(_DecomposeBase):
    def __init__(self, V=None, S1=None, S2=None, C_output_mat=None, wildcard_mat=None,
                 wildcard_output_vector=None, final_vector=None, start_vector=None,
                 pretrained_word_embed=None, priority_mat=None, args=None, o_idx=0, is_cuda=True):
        super().__init__(args, C_output_mat.shape[0], *S1.shape, start_vector, final_vector, priority_mat, o_idx,
                         (S1, S2, V, C_output_mat, wildcard_mat, wildcard_output_vector), pretrained_word_embed, is_cuda)

    def init_forward_parameters(self, S1, S2, V, C_o, W, W_o):
        a = self.args
        self.S1 = nn.Parameter(self.pad_additional_states(torch.from_numpy(S1).float()), requires_grad=True)
        self.S2 = nn.Parameter(self.pad_additional_states(torch.from_numpy(S2).float()), requires_grad=True)
        self.V_embed = nn.Parameter(torch.from_numpy(V).float(), requires_grad=bool(a.train_V_embed))
        # least-squares map from word-embedding space to rank space: G = pinv(E) @ V_embed   (D x R)
        G = torch.matmul(self.embedding.weight.data.pinverse(), self.V_embed.data)
        self.embed_r_generalized = nn.Parameter(G, requires_grad=True)
        if a.use_crf == 1:   # two extra label rows (START/STOP) of small noise
            C_o = np.concatenate((C_o, self.get_random((2, self.S)).numpy() * a.rand_constant), axis=0)
        self.C_output_mat = nn.Parameter(self.pad_additional_states(torch.from_numpy(C_o).float()),
                                         requires_grad=bool(a.train_c_output))
        self.wildcard_mat = nn.Parameter(self.pad_additional_states(torch.from_numpy(W).float()),
                                         requires_grad=bool(a.train_wildcard))
        self.wildcard_output_vector = nn.Parameter(self.pad_additional_states(torch.from_numpy(W_o).float()),
                                                   requires_grad=bool(a.train_wildcard_wildcard))
        self._gate_params(self.S + self.additional_states)
        if self.random:
            for w in (self.S1, self.S2, self.V_embed, self.C_output_mat, self.embed_r_generalized,
                      self.wildcard_mat):
                nn.init.xavier_normal_(w)
            nn.init.normal_(self.h0)
            nn.init.normal_(self.hT)

    def _fn_params(self):
        names = self._params_for_fn() + ['V_embed', 'embed_r_generalized', 'beta_vec']
        tensors = [getattr(self, n) for n in names] + [self.embedding.weight]
        return names + ['embedding'], tensors

    def forward_scores(self, input, lengths, shape=None, fuse=False):
        """all_scores B x L x C (L = max length); differentiable w.r.t. the module parameters.
        fuse=True (decode-only callers): rows past the length may hold anything -- the label-score operand then comes
        fused out of the recurrence (re2nn_decompose_recurrence ab_out) where the call allows it."""
        dev = self._device()
        x = self._device_input(input, dev)
        lengths = lengths.to(dev).contiguous()
        shape = shape or self._host_shape(lengths)
        names, tensors = self._fn_params()
        if self._max_needs_grad(tensors):
            from .model_fst import ifst_decompose_max_scores
            return ifst_decompose_max_scores(self, x, None, lengths, shape[0])
        pr = (self.priority_layer.priority_mat, self.priority_layer.priority_bias)
        return autograd_fns.decompose_scores(dict(self._recurrence_consts(), fuse_scores=bool(fuse)), names, tensors, pr, x,
                                             None, lengths, shape[0], cache=self._cache)

    def _device_input(self, input, dev):
        return input.to(dev).contiguous()

    def _warm_tables(self):
        names, tensors = self._fn_params()
        p = {n: t.detach().contiguous() for n, t in zip(names, tensors)}
        autograd_fns._prepare(self._recurrence_consts(), p, None, self._cache)
        autograd_fns._weight_prep(self._recurrence_consts(), p, self._cache)

    def forward_local(self, input, label, lengths, train=True, re_tags=None):
        return self._forward_body(input, label, lengths, train, re_tags, 'tok')


class FARNN_S_SF(_DecomposeBase):
    def __init__(self, S1=None, S2=None, C_output_mat=None, wildcard_mat=None, wildcard_output_vector=None,
                 final_vector=None, start_vector=None, priority_mat=None, args=None, o_idx=0, is_cuda=True):
        super().__init__(args, C_output_mat.shape[0], *S1.shape, start_vector, final_vector, priority_mat, o_idx,
                         (S1, S2, C_output_mat, wildcard_mat, wildcard_output_vector), is_cuda=is_cuda)

    def init_forward_parameters(self, S1, S2, C_o, W, W_o):
        a = self.args
        self.S1 = nn.Parameter(self.pad_additional_states(torch.from_numpy(S1).float()), requires_grad=True)
        self.S2 = nn.Parameter(self.pad_additional_states(torch.from_numpy(S2).float()), requires_grad=True)
        if a.use_crf == 1:
            C_o = np.concatenate((C_o, self.get_random((2, self.S)).numpy() * a.rand_constant), axis=0)
        self.C_output_mat = nn.Parameter(self.pad_additional_states(torch.from_numpy(C_o).float()),
                                         requires_grad=bool(a.train_c_output))
        self.wildcard_mat = nn.Parameter(self.pad_additional_states(torch.from_numpy(W).float()),
                                         requires_grad=bool(a.train_wildcard))
        self.wildcard_output_vector = nn.Parameter(self.pad_additional_states(torch.from_numpy(W_o).float()),
                                                   requires_grad=bool(a.train_wildcard_wildcard))
        self._gate_params(self.S + self.additional_states)
        if self.random:
            for w in (self.S1, self.S2, self.C_output_mat, self.wildcard_mat):
                nn.init.xavier_normal_(w)
            nn.init.normal_(self.h0)
            nn.init.normal_(self.hT)

    def forward_scores(self, input, lengths, shape=None, fuse=False):
        dev = self._device()
        v = self._device_input(input, dev)
        lengths = lengths.to(dev).contiguous()
        shape = shape or self._host_shape(lengths)
        names = self._params_for_fn()
        tensors = [getattr(self, n) for n in names]
        if self._max_needs_grad(tensors + [v]):
            from .model_fst import ifst_decompose_max_scores
            return ifst_decompose_max_scores(self, None, v, lengths, shape[0])
        pr = (self.priority_layer.priority_mat, self.priority_layer.priority_bias)
        return autograd_fns.decompose_scores(dict(self._recurrence_consts(), fuse_scores=bool(fuse)), names, tensors, pr, None,
                                             v, lengths, shape[0], cache=self._cache)

    def _device_input(self, input, dev):
        return input.to(dev).float().contiguous()

    def forward(self, input, label, lengths, train=True, re_tags=None):
        """input: pre-computed rank factors B x L x R (model_decompose_single.py:483-580)."""
        return self._forward_body(input, label, lengths, train, re_tags, 'sf')
