"""Drop-ins for the FST (non-independent) model family -- SURVEY.md section 8 rows a16 / f4:

    FARNN_S_D_W     farnn/model_decompose.py:10-456               4-order CP factors, wildcard factors
    FARNN_S_D_W_I   farnn/model_decompose_independent.py:12-300   language x output factorisation (independent = 1)
    FARNN_S_O       farnn/model_onehot.py:8-180                   exact FST, label-indexed transitions V x C x S x S
    FARNN_S_O_I     farnn/model_onehot.py:183-306                 exact, language x output tensors

Same class names, constructor signatures, parameter names / requires_grad flags / state_dict keys, RNG draw order and
forward_local / forward_score / forward_RE / local_decode contracts as the reference classes.

How they map onto the kernels:

* FARNN_S_D_W keeps the rank-R structure (`((h S1) * _R) S2^T + h Wsum`, model_decompose.py:278-291), so it runs on the
  i-FST recurrence kernels unchanged (tensor cores, resident kernel, gates, BPTT): token table scaled by
  sum_c C_embed[c], wildcard matrix = S1w diag(sum_c C_wildcard[c]) S2w^T + wildcard_wildcard, no output mask.  Only the
  score differs (model_decompose.py:309-324: two rank contractions against [C_embed | C_wildcard]); it is three calls
  of the library GEMM with the element-wise products between them, and its gradient reaches the recurrence through
  `re2nn_decompose_backward`'s dalpha_in / dbeta_in.
* The other three multiply a label / output mask into the transition matrix ELEMENT-WISE
  (model_decompose_independent.py:172-176, model_onehot.py:271-284), which destroys the rank structure: every
  (sequence, step) owns a dense S x S matrix.  They are built from two library primitives -- `re2nn_gemm_nt` (the
  step-GEMM mainloops) and `re2nn_batched_vecmat` (sum / max semiring, argmax routing for the max backward) -- with
  the gathers and element-wise products between them left to torch (device-side glue; autograd differentiates it).
  No shipped configuration uses these classes (SURVEY.md section 8 f4); they are complete and parity-tested, not tuned.
* train_mode = 'max' trains through `re2nn_batched_vecmat`'s saved argmax (first maximal source state, torch.max's
  tie-break) in the three dense classes; `MaxProductTrainer` below gives FARNN_S_D_W_I_S the same path.
"""
import numpy as np
import torch
from torch import nn

from . import ops
from ._lib import V_TOKEN
from .bert_embeddings import _Aggregate
from .model_decompose_single import _ADD_NL, _UPDATE_NL, _DecomposeBase, _nl_name
from .model_onehot import _OnehotBase
from .priority import PriorityLayer


# ---- differentiable wrappers of the library primitives ----------------------------------------------------------------
class _MatmulNT(torch.autograd.Function):
    """C = A @ B^T (A: M x K, B: N x K) on the library GEMM; dA = dC @ B, dB = dC^T @ A on the same kernel."""

    @staticmethod
    def forward(ctx, A, B, precision):
        A, B = A.contiguous(), B.contiguous()
        ctx.save_for_backward(A, B)
        ctx.precision = precision
        return ops.gemm_nt(A, B, precision)

    @staticmethod
    def backward(ctx, dC):
        A, B = ctx.saved_tensors
        dC = dC.contiguous()
        dA = ops.gemm_nt(dC, B.t().contiguous(), 'fp32') if ctx.needs_input_grad[0] else None
        dB = ops.gemm_nt(dC.t().contiguous(), A.t().contiguous(), 'fp32') if ctx.needs_input_grad[1] else None
        return dA, dB, None


def matmul_nt(A, B, precision='fp32'):
    return _MatmulNT.apply(A, B, precision)


class _VecMat(torch.autograd.Function):
    """out[b,s] = (+|max)_j h[b,j] T[b,j,s]  (transposed: T[b,s,j]) -- utils.py:192-199 on one dense matrix per row."""

    @staticmethod
    def forward(ctx, h, T, transposed, maxp):
        h, T = h.contiguous(), T.contiguous()
        out, idx = ops.batched_vecmat(h, T, transposed, maxp)
        ctx.save_for_backward(h, T, idx)
        ctx.transposed, ctx.maxp = transposed, maxp
        return out

    @staticmethod
    def backward(ctx, dout):
        h, T, idx = ctx.saved_tensors
        dout = dout.contiguous()
        tr = ctx.transposed
        if not ctx.maxp:
            dh, _ = ops.batched_vecmat(dout, T, not tr, False)
            dT = (dout.unsqueeze(2) * h.unsqueeze(1)) if tr else (h.unsqueeze(2) * dout.unsqueeze(1))
            return dh, dT, None, None
        ix = idx.long()                                       # B x S: the source state that won target s
        hsel = h.gather(1, ix)
        if tr:                                                # T[b, s, ix[b,s]]
            tsel = T.gather(2, ix.unsqueeze(2)).squeeze(2)
            dT = torch.zeros_like(T).scatter_(2, ix.unsqueeze(2), (dout * hsel).unsqueeze(2))
        else:                                                 # T[b, ix[b,s], s]
            tsel = T.gather(1, ix.unsqueeze(1)).squeeze(1)
            dT = torch.zeros_like(T).scatter_(1, ix.unsqueeze(1), (dout * hsel).unsqueeze(1))
        dh = torch.zeros_like(h).scatter_add_(1, ix, dout * tsel)
        return dh, dT, None, None


def vecmat(h, T, transposed=False, maxp=False):
    return _VecMat.apply(h, T, transposed, maxp)


def _apply_nl(x, name):
    if name == 'relu':
        return torch.relu(x)
    if name == 'tanh':
        return torch.tanh(x)
    if name == 'relutanh':
        return torch.tanh(torch.relu(x))
    if name == 'sigmoid':
        return torch.sigmoid(x)
    return x


def _reverse_tokens(x, lengths):
    """utils.py:183-189 `reverse` for a B x L index matrix without the Python loop over the batch."""
    L = x.shape[1]
    pos = torch.arange(L, device=x.device).unsqueeze(0)
    n = lengths.unsqueeze(1)
    return x.gather(1, torch.where(pos < n, n - 1 - pos, pos))


def _beta_rows(hT, backward_scores, lengths):
    """reversed_backward_score_x[:, i + 1] for i = 0..L-1 (e.g. model_decompose.py:420-431): row n-1-i of
    cat([hT, backward_scores]) while i < n, row i + 1 afterwards."""
    B, L, S = backward_scores.shape
    full = torch.cat([hT.view(1, 1, S).expand(B, 1, S), backward_scores], dim=1)          # B x (L+1) x S
    pos = torch.arange(L, device=full.device).unsqueeze(0)
    n = lengths.unsqueeze(1)
    idx = torch.where(pos < n, n - 1 - pos, pos + 1)
    return full.gather(1, idx.unsqueeze(2).expand(B, L, S))


def _apply_priority(m, scores):
    """scores @ priority_mat + priority_bias over the last dimension (priority.py:20-30) when args.use_priority."""
    if not m.args.use_priority:
        return scores
    Cn = scores.shape[-1]
    out = matmul_nt(scores.reshape(-1, Cn), m.priority_layer.priority_mat.t().contiguous())
    return (out + m.priority_layer.priority_bias).view(scores.shape)


def _dense_transition(m, V_vec):
    """Tr[b,j,s] = sum_r S1[j,r] V_vec[b,r] S2[s,r] + wildcard_mat[j,s]   (model_decompose_independent.py:172-175)"""
    B, S = V_vec.shape[0], m._S_full
    X = (m.S1.unsqueeze(0) * V_vec.unsqueeze(1)).reshape(B * S, m.S1.shape[1])
    return matmul_nt(X, m.S2).view(B, S, S) + m.wildcard_mat


def _gated_step(m, h, V_vec, h_init, inner):
    """One step of the gated recurrence on dense transitions: hn = nl(inner(h_bar, V_vec)) between the reset gate
    (farnn == 2: h_bar mixes h with h_init) and the update gate (farnn >= 1: hn mixes with h).  `inner` is the
    caller's semiring product with its output mask applied."""
    a = m.args
    k = float(a.sigmoid_exponent)
    h_bar = h
    if a.farnn >= 1:
        zt = torch.sigmoid(k * (matmul_nt(h, m.Wss1.t().contiguous()) + matmul_nt(V_vec, m.Wrs1.t().contiguous()) + m.bs1))
    if a.farnn == 2:
        rt = torch.sigmoid(k * (matmul_nt(h, m.Wss2.t().contiguous()) + matmul_nt(V_vec, m.Wrs2.t().contiguous()) + m.bs2))
        h_bar = (1 - rt) * h_init + rt * h
    hn = _apply_nl(inner(h_bar, V_vec), _nl_name(a.update_nonlinear, _UPDATE_NL))
    if a.farnn >= 1:
        hn = (1 - zt) * h + zt * hn
    return hn


class _FstRecurrence(torch.autograd.Function):
    """alpha, beta of the rank-R recurrence with no output mask, differentiable w.r.t. the (already scaled) token
    table, S1, S2, the wildcard matrix, h0 / hT and the gate parameters."""

    @staticmethod
    def forward(ctx, consts, x, lengths, L, vtab, S1, S2, W, h0, hT, Wss1, Wrs1, bs1, Wss2, Wrs2, bs2):
        t = [q.detach().contiguous() if q is not None else None for q in (vtab, S1, S2, W, h0, hT, Wss1, Wrs1, bs1, Wss2, Wrs2, bs2)]
        vtab, S1, S2, W, h0, hT, Wss1, Wrs1, bs1, Wss2, Wrs2, bs2 = t
        farnn = consts['farnn']
        need = consts['grad_on'] and any(ctx.needs_input_grad[4:])
        gtab = ops.gate_table(vtab, Wrs1, bs1, Wrs2, bs2, farnn) if farnn >= 1 else None
        o = torch.ones((S1.shape[0],), dtype=torch.float32, device=S1.device)
        mx = consts['max_semiring']
        if mx and need:
            raise NotImplementedError("re2nn_b200 FARNN_S_D_W: train_mode='max' is inference-only for this class")
        alpha, beta, saves = ops.decompose_recurrence(
            x, lengths, L, vtab, gtab, S1, S2, W, o, h0, hT, Wss1, Wss2, farnn, consts['update_nonlinear'],
            consts['sigmoid_exponent'], precision='fp32' if mx else consts['precision'], v_mode=V_TOKEN, full_pad=False,
            save_for_backward=need, Lpad=x.shape[1], max_semiring=mx, zero_fill=True)
        if need:
            ctx.consts, ctx.L = consts, L
            ctx.saved = (x, lengths, vtab, o, alpha, beta, saves,
                         dict(S1=S1, S2=S2, wildcard_mat=W, h0=h0, hT=hT, Wss1=Wss1, Wrs1=Wrs1, bs1=bs1, Wss2=Wss2, Wrs2=Wrs2,
                              bs2=bs2))
        return alpha, beta

    @staticmethod
    def backward(ctx, dalpha, dbeta):
        x, lengths, vtab, o, alpha, beta, saves, p = ctx.saved
        p = {k: v for k, v in p.items() if v is not None}
        names = ['vtab', 'S1', 'S2', 'wildcard_mat', 'h0', 'hT', 'Wss1', 'Wrs1', 'bs1', 'Wss2', 'Wrs2', 'bs2']
        want = {n for i, n in enumerate(names) if ctx.needs_input_grad[4 + i] and (n == 'vtab' or n in p)}
        consts = dict(ctx.consts, full_pad=False, ce1=True)
        g = ops.decompose_backward(consts, p, x, None, lengths, ctx.L, vtab, o, alpha, beta, saves, None, None, want,
                                   dalpha_in=dalpha.contiguous(), dbeta_in=dbeta.contiguous())
        out = []
        for n in names:
            v = g.get(n) if n in want else None
            if v is not None and n in ('bs1', 'bs2'):
                v = v.view_as(p[n])
            out.append(v)
        return (None, None, None, None) + tuple(out)


# ---- max-product TRAINING of the i-FST classes (SURVEY.md section 8 f4) ---------------------------------------------------
# train_mode = 'max' materialises one dense transition per sequence and step in the reference too
# (model_decompose_single.py:159-166, model_onehot.py:374-403 with utils.py:192-195); the gradient follows the argmax
# saved by re2nn_batched_vecmat.  Inference keeps the dedicated kernels (re2nn_decompose_max_recurrence, the MAXP
# onehot kernel); these differentiable forms run only when a gradient is needed.
def ifst_decompose_max_scores(m, x, dense_v, lengths, L):
    """all_scores B x L x C of FARNN_S_D_W_I_S / FARNN_S_SF under the max-product semiring, differentiable."""
    a = m.args
    S = m._S_full
    B = lengths.shape[0]
    if dense_v is None:
        vt = _Aggregate.apply(m.V_embed, m.embedding.weight, m.embed_r_generalized, m.beta_vec,
                              _nl_name(a.additional_nonlinear, _ADD_NL))
        x = x[:, :L]
        xr = _reverse_tokens(x, lengths)
        v_at = lambda i, rev: vt[(xr if rev else x)[:, i]]
    else:
        v = dense_v[:, :L]
        pos = torch.arange(L, device=v.device).unsqueeze(0)
        n = lengths.unsqueeze(1)
        ridx = torch.where(pos < n, n - 1 - pos, pos)
        vr = v.gather(1, ridx.unsqueeze(2).expand(B, L, v.shape[2]))
        v_at = lambda i, rev: (vr if rev else v)[:, i]
    o = m.C_output_mat.sum(0)
    if a.local_loss_func != 'CE1':
        o = o + m.wildcard_output_vector
    h0 = m.h0.view(1, S).expand(B, S)
    hT = m.hT.view(1, S).expand(B, S)
    fwd = lambda h_bar, V_vec: vecmat(h_bar, _dense_transition(m, V_vec), False, True) * o     # mask on the new state
    bwd = lambda h_bar, V_vec: vecmat(h_bar * o, _dense_transition(m, V_vec), True, True)      # mask on the old state
    hf, hb, fw, bw = h0, hT, [], []
    for i in range(L):
        hf = _gated_step(m, hf, v_at(i, False), h0, fwd)
        fw.append(hf)
        hb = _gated_step(m, hb, v_at(i, True), hT, bwd)
        bw.append(hb)
    alpha = torch.stack(fw, dim=1)                                          # h0_forward_score[:, i + 1]
    beta = _beta_rows(m.hT, torch.stack(bw, dim=1), lengths)                # reversed_backward_score_x[:, i + 1]
    scores = matmul_nt((alpha * beta).reshape(B * L, S), m.C_output_mat).view(B, L, m.C)
    return _apply_priority(m, scores)


def ifst_onehot_max_scores(m, x, lengths):
    """all_scores B x L x C of FARNN_S_O_I_S under the max-product semiring, differentiable (model_onehot.py:366-426)."""
    a = m.args
    B, L = x.shape
    S = m.S
    nl = _nl_name(a.update_nonlinear, _UPDATE_NL)
    T = m.language_tensor + m.wildcard_mat
    o = m.output_mat.sum(0)
    if a.local_loss_func != 'CE1':
        o = o + m.output_wildcard_vector
    xr = _reverse_tokens(x, lengths)
    hf = m.h0.view(1, S).expand(B, S)
    hb = m.hT.view(1, S).expand(B, S)
    fw, bw = [], []
    for i in range(L):
        hf = _apply_nl(vecmat(hf, T[x[:, i]], False, True) * o, nl)
        fw.append(hf)
        hb = _apply_nl(vecmat(hb * o, T[xr[:, i]], True, True), nl)
        bw.append(hb)
    alpha = torch.stack(fw, dim=1)
    beta = _beta_rows(m.hT, torch.stack(bw, dim=1), lengths)
    Cn = m.output_mat.shape[0]
    scores = matmul_nt((alpha * beta).reshape(B * L, S), m.output_mat).view(B, L, Cn)
    return _apply_priority(m, scores)


# ---- FARNN_S_D_W ------------------------------------------------------------------------------------------------------------
class FARNN_S_D_W(_DecomposeBase):
    def __init__(self, V=None, C=None, S1=None, S2=None, C_wildcard=None, S1_wildcard=None, S2_wildcard=None,
                 wildcard_wildcard=None, final_vector=None, start_vector=None, pretrained_word_embed=None,
                 priority_mat=None, args=None, o_idx=0):
        super().__init__(args, C_wildcard.shape[0], S1_wildcard.shape[0], C.shape[1], start_vector, final_vector,
                         priority_mat, o_idx, (S1, S2, C, V, S1_wildcard, S2_wildcard, C_wildcard, wildcard_wildcard),
                         pretrained_word_embed)
        self.R_W = C_wildcard.shape[1]

    def init_forward_parameters(self, S1, S2, C, V, S1_w, S2_w, C_w, W):
        a = self.args
        self.S1 = nn.Parameter(self.pad_additional_states(torch.from_numpy(S1).float()), requires_grad=True)
        self.S2 = nn.Parameter(self.pad_additional_states(torch.from_numpy(S2).float()), requires_grad=True)
        self.V_embed = nn.Parameter(torch.from_numpy(V).float(), requires_grad=bool(a.train_V_embed))
        G = torch.matmul(self.embedding.weight.data.pinverse(), self.V_embed.data)
        self.embed_r_generalized = nn.Parameter(G, requires_grad=True)
        if a.use_crf == 1:
            C = np.concatenate((C, self.get_random((2, self.R)).numpy() * a.rand_constant), axis=0)
            C_w = np.concatenate((C_w, self.get_random((2, C_w.shape[1])).numpy() * a.rand_constant), axis=0)
        self.C_wildcard = nn.Parameter(self.pad_additional_states(torch.from_numpy(C_w).float()),
                                       requires_grad=bool(a.train_wildcard))
        self.C_embed = nn.Parameter(torch.from_numpy(C).float(), requires_grad=True)
        self.S1_wildcard = nn.Parameter(self.pad_additional_states(torch.from_numpy(S1_w).float()),
                                        requires_grad=bool(a.train_wildcard))
        self.S2_wildcard = nn.Parameter(self.pad_additional_states(torch.from_numpy(S2_w).float()),
                                        requires_grad=bool(a.train_wildcard))
        self.wildcard_wildcard = nn.Parameter(self.pad_additional_states(torch.from_numpy(W).float()),
                                              requires_grad=bool(a.train_wildcard_wildcard))
        self._gate_params(self.S + self.additional_states)
        if self.random:
            for w in (self.S1, self.S2, self.C_embed, self.V_embed, self.S1_wildcard, self.S2_wildcard, self.C_wildcard,
                      self.embed_r_generalized, self.wildcard_wildcard):
                nn.init.xavier_normal_(w)
            nn.init.normal_(self.h0)
            nn.init.normal_(self.hT)

    # -- shared by FARNN_S_D_W / FARNN_S_D_W_I -----------------------------------------------------------------
    def _token_table(self):
        """get_generalized_v_embed_vec evaluated per token id (model_decompose.py:222-241): (V+1) x R."""
        return _Aggregate.apply(self.V_embed, self.embedding.weight, self.embed_r_generalized, self.beta_vec,
                                _nl_name(self.args.additional_nonlinear, _ADD_NL))

    def _gates(self):
        g = [getattr(self, n, None) for n in ('Wss1', 'Wrs1', 'bs1', 'Wss2', 'Wrs2', 'bs2')]
        return g

    def forward_scores(self, input, lengths, shape=None):
        dev = self._device()
        x = input.to(dev).contiguous()
        lengths = lengths.to(dev).contiguous()
        L, _ = shape or self._host_shape(lengths)
        B = x.shape[0]
        S = self._S_full
        consts = dict(self._recurrence_consts(), grad_on=torch.is_grad_enabled())
        vt = self._token_table()                                           # V_vec per token
        vtab_rec = vt * self.C_embed.sum(0)                                # _R = V_vec * C_vec_sum   (:255-256)
        Wsum = matmul_nt(self.S1_wildcard * self.C_wildcard.sum(0), self.S2_wildcard) + self.wildcard_wildcard   # (:326-331)
        alpha, beta = _FstRecurrence.apply(consts, x, lengths, L, vtab_rec, self.S1, self.S2, Wsum, self.h0, self.hT,
                                           *self._gates())
        # get_final_score (:309-324) at alpha index i, beta index i + 1 (:426-427)
        a_prev = torch.cat([self.h0.view(1, 1, S).expand(B, 1, S), alpha[:, :L - 1]], dim=1).reshape(B * L, S)
        aS = matmul_nt(a_prev, torch.cat([self.S1, self.S1_wildcard], dim=1).t().contiguous())
        bS = matmul_nt(beta.reshape(B * L, S), torch.cat([self.S2, self.S2_wildcard], dim=1).t().contiguous())
        prod = aS * bS
        v = vt[x[:, :L]].reshape(B * L, self.R)
        prod = torch.cat([prod[:, :self.R] * v, prod[:, self.R:]], dim=1)
        scores = matmul_nt(prod, torch.cat([self.C_embed, self.C_wildcard], dim=1)).view(B, L, self.C)
        return _apply_priority(self, scores)

    def forward_local(self, input, label, lengths, train=True):
        dev = self._device()
        lengths = lengths.to(dev).contiguous()
        shape = self._host_shape(lengths)
        all_scores = self.forward_scores(input, lengths, shape)
        return self._finish(all_scores, label, lengths, train, None, shape)


# ---- FARNN_S_D_W_I -------------------------------------------------------------------------------------------------------------
class FARNN_S_D_W_I(FARNN_S_D_W):
    def __init__(self, V=None, S1=None, S2=None, C_output=None, S1_output=None, S2_output=None, wildcard_mat=None,
                 wildcard_output=None, final_vector=None, start_vector=None, pretrained_word_embed=None, priority_mat=None,
                 args=None, o_idx=0):
        _DecomposeBase.__init__(self, args, C_output.shape[0], *S1.shape, start_vector, final_vector, priority_mat, o_idx,
                                (S1, S2, V, S1_output, S2_output, C_output, wildcard_mat, wildcard_output),
                                pretrained_word_embed)
        self.R_O = C_output.shape[1]

    def init_forward_parameters(self, S1, S2, V, S1_o, S2_o, C_o, W, W_o):
        a = self.args
        self.S1 = nn.Parameter(self.pad_additional_states(torch.from_numpy(S1).float()), requires_grad=True)
        self.S2 = nn.Parameter(self.pad_additional_states(torch.from_numpy(S2).float()), requires_grad=True)
        self.V_embed = nn.Parameter(torch.from_numpy(V).float(), requires_grad=bool(a.train_V_embed))
        G = torch.matmul(self.embedding.weight.data.pinverse(), self.V_embed.data)
        self.embed_r_generalized = nn.Parameter(G, requires_grad=True)
        if a.use_crf:
            C_o = np.concatenate((C_o, self.get_random((2, C_o.shape[1])).numpy() * a.rand_constant), axis=0)
        self.C_output = nn.Parameter(self.pad_additional_states(torch.from_numpy(C_o).float()),
                                     requires_grad=bool(a.train_wildcard))
        self.S1_output = nn.Parameter(self.pad_additional_states(torch.from_numpy(S1_o).float()),
                                      requires_grad=bool(a.train_wildcard))
        self.S2_output = nn.Parameter(self.pad_additional_states(torch.from_numpy(S2_o).float()),
                                      requires_grad=bool(a.train_wildcard))
        self.wildcard_mat = nn.Parameter(self.pad_additional_states(torch.from_numpy(W).float()),
                                         requires_grad=bool(a.train_wildcard_wildcard))
        self.wildcard_output = nn.Parameter(self.pad_additional_states(torch.from_numpy(W_o).float()),
                                            requires_grad=bool(a.train_wildcard_wildcard)) if W_o is not None else None
        self._gate_params(self.S + self.additional_states)
        if self.random:
            for w in (self.S1, self.S2, self.V_embed, self.S1_output, self.S2_output, self.C_output,
                      self.embed_r_generalized, self.wildcard_mat):
                nn.init.xavier_normal_(w)
            nn.init.normal_(self.h0)
            nn.init.normal_(self.hT)

    def forward_scores(self, input, lengths, shape=None):
        dev = self._device()
        x = input.to(dev).contiguous()
        lengths = lengths.to(dev).contiguous()
        L, _ = shape or self._host_shape(lengths)
        x = x[:, :L]
        B, S = x.shape[0], self._S_full
        maxp = self.args.train_mode == 'max'
        vt = self._token_table()
        O = matmul_nt(self.S1_output * self.C_output.sum(0), self.S2_output)               # get_output_tensor_sum (:208-215)
        if self.args.local_loss_func != 'CE1':
            O = O + self.wildcard_output
        xr = _reverse_tokens(x, lengths)
        h0 = self.h0.view(1, S).expand(B, S)
        hT = self.hT.view(1, S).expand(B, S)
        fwd = lambda h_bar, V_vec: vecmat(h_bar, _dense_transition(self, V_vec) * O, False, maxp)
        bwd = lambda h_bar, V_vec: vecmat(h_bar, _dense_transition(self, V_vec) * O, True, maxp)
        hf, hb, fw, bw = h0, hT, [], []
        for i in range(L):
            hf = _gated_step(self, hf, vt[x[:, i]], h0, fwd)
            fw.append(hf)
            hb = _gated_step(self, hb, vt[xr[:, i]], hT, bwd)
            bw.append(hb)
        fw, bw = torch.stack(fw, dim=1), torch.stack(bw, dim=1)
        alpha = torch.cat([h0.unsqueeze(1), fw[:, :L - 1]], dim=1)          # h0_forward_score[:, i]
        beta = _beta_rows(self.hT, bw, lengths)                             # reversed_backward_score_x[:, i + 1]
        s1s2_out = (self.S1_output.t().unsqueeze(2) * self.S2_output.t().unsqueeze(1)).reshape(self.R_O, S * S)
        scores = []
        for i in range(L):                                                  # get_final_score (:198-206)
            bss = _dense_transition(self, vt[x[:, i]])
            M = alpha[:, i].unsqueeze(2) * beta[:, i].unsqueeze(1) * bss
            br = matmul_nt(M.reshape(B, S * S), s1s2_out)
            scores.append(matmul_nt(br, self.C_output))
        return _apply_priority(self, torch.stack(scores, dim=1))


# ---- exact (onehot) FST classes -----------------------------------------------------------------------------------------
class FARNN_S_O(_OnehotBase):
    def __init__(self, language_tensor=None, wildcard_tensor=None, wildcard_wildcard_mat=None, final_vector=None,
                 start_vector=None, priority_mat=None, args=None, o_idx=0, is_cuda=False):
        super().__init__()
        self.is_cuda = torch.cuda.is_available() and is_cuda
        self.args = args
        C, S, S = wildcard_tensor.shape
        self.S, self.C = S, C
        self.amp = args.rand_constant
        self.h0 = nn.Parameter(self._noisy(start_vector), requires_grad=False)
        self.hT = nn.Parameter(self._noisy(final_vector), requires_grad=False)
        self.language_tensor = nn.Parameter(self._noisy(language_tensor), requires_grad=True)                  # V x C x S x S
        self.wildcard_tensor = nn.Parameter(self._noisy(wildcard_tensor), requires_grad=bool(args.train_wildcard))   # C x S x S
        self.wildcard_wildcard_mat = nn.Parameter(torch.from_numpy(wildcard_wildcard_mat).float(),
                                                  requires_grad=bool(args.train_wildcard_wildcard))
        self.priority_layer = PriorityLayer(self.C, priority_mat)
        self.o_idx = o_idx
        self.initialize()
        if torch.cuda.is_available():
            self.cuda()

    def _recurrence(self, x, lengths, sum_tensor, mask=None):
        """h <- relu(semiring(h, sum_tensor[x_t] [* mask])) in both directions (model_onehot.py:88-103, 271-290);
        -> (alpha rows i, beta rows i + 1) as the score loops index them."""
        B, L = x.shape
        S = self.S
        maxp = self.args.train_mode == 'max'
        xr = _reverse_tokens(x, lengths)
        hf = self.h0.view(1, S).expand(B, S)
        hb = self.hT.view(1, S).expand(B, S)
        fw, bw = [], []
        for i in range(L):
            Tr = sum_tensor[x[:, i]]
            Trb = sum_tensor[xr[:, i]]
            if mask is not None:
                Tr, Trb = Tr * mask, Trb * mask
            hf = torch.relu(vecmat(hf, Tr, False, maxp))
            fw.append(hf)
            hb = torch.relu(vecmat(hb, Trb, True, maxp))
            bw.append(hb)
        fw, bw = torch.stack(fw, dim=1), torch.stack(bw, dim=1)
        alpha = torch.cat([self.h0.view(1, 1, S).expand(B, 1, S), fw[:, :L - 1]], dim=1)
        return alpha, _beta_rows(self.hT, bw, lengths)

    def _scores(self, x, lengths, full_pad):
        """Every position is scored, pads included, whatever full_pad asks."""
        B, L = x.shape
        lang, wild = self.language_tensor, self.wildcard_tensor
        sum_tensor = lang.sum(1) + wild.sum(0)                                     # V x S x S   (:81-85)
        if self.args.local_loss_func != 'CE1':
            sum_tensor = sum_tensor + self.wildcard_wildcard_mat
        all_tensor = lang + wild                                                   # V x C x S x S
        alpha, beta = self._recurrence(x, lengths, sum_tensor)
        out = []
        for i in range(L):                                                         # (:119-133)
            Tr = all_tensor[x[:, i]]                                               # B x C x S x S
            sc = torch.relu(Tr * alpha[:, i].view(B, 1, self.S, 1) * beta[:, i].view(B, 1, 1, self.S)).sum(dim=(2, 3))
            out.append(_apply_priority(self, sc))
        return torch.stack(out, dim=1)


class FARNN_S_O_I(FARNN_S_O):
    def __init__(self, language_tensor=None, output_tensor=None, wildcard_mat=None, output_wildcard_mat=None,
                 final_vector=None, start_vector=None, priority_mat=None, args=None, o_idx=0, is_cuda=False):
        nn.Module.__init__(self)
        self.is_cuda = torch.cuda.is_available() and is_cuda
        self.args = args
        C, S, S = output_tensor.shape
        self.S, self.C = S, C
        self.amp = args.rand_constant
        self.h0 = nn.Parameter(self._noisy(start_vector), requires_grad=False)
        self.hT = nn.Parameter(self._noisy(final_vector), requires_grad=False)
        self.language_tensor = nn.Parameter(self._noisy(language_tensor), requires_grad=True)    # V x S x S
        self.wildcard_mat = nn.Parameter(self._noisy(wildcard_mat), requires_grad=False)         # S x S
        self.output_tensor = nn.Parameter(torch.from_numpy(output_tensor).float(), requires_grad=False)   # C x S x S
        self.output_wildcard_mat = nn.Parameter(torch.from_numpy(output_wildcard_mat).float(), requires_grad=False) \
            if output_wildcard_mat is not None else None
        self.priority_layer = PriorityLayer(self.C, priority_mat)
        self.o_idx = o_idx
        self.initialize()
        if torch.cuda.is_available():
            self.cuda()

    def _scores(self, x, lengths, full_pad):
        B, L = x.shape
        S = self.S
        sum_tensor = self.language_tensor + self.wildcard_mat                      # V x S x S   (:259)
        sum_output = self.output_tensor.sum(0)
        if self.args.local_loss_func != 'CE1':
            sum_output = sum_output + self.output_wildcard_mat
        mask = sum_output if self.args.independent == 2 else None
        alpha, beta = self._recurrence(x, lengths, sum_tensor, mask)
        out_flat = self.output_tensor.reshape(self.C, S * S)
        out = []
        for i in range(L):                                                         # get_final_score (:226-230)
            M = alpha[:, i].unsqueeze(2) * beta[:, i].unsqueeze(1) * sum_tensor[x[:, i]]
            out.append(_apply_priority(self, matmul_nt(M.reshape(B, S * S), out_flat)))
        return torch.stack(out, dim=1)
