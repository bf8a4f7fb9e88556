"""Thin Python wrappers over the C-ABI: torch owns device memory and streams, the kernels do the work.

The hot-path ops -- recurrences, label scores, decode, CRF -- are called as registered PyTorch custom ops
(`torch.ops.re2nn.*`, TORCH_LIBRARY in csrc/torch_ops.cpp, a thin C++ layer over the same C-ABI); the remaining entry
points (tables, training saves / backward, debug switches) go through ctypes.  Every function takes contiguous CUDA
tensors (fp32 / int64); outputs are allocated with torch on the tensor's device and the kernels run on the current
stream.  No computation happens in torch.
"""
import ctypes as C

import torch

from . import _lib
from ._lib import (NL, PREC, V_DENSE, V_TOKEN, BackwardArgs, OnehotArgs, OnehotBackwardArgs, RecurrenceArgs, check,
                   fn, tops)

_LAUNCHES = {'n': 0}   # launch counter read by bench.py ("gpu_launches")


def launches():
    return _LAUNCHES['n']


def _count(k):
    _LAUNCHES['n'] += k


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("re2nn_b200: expected a CUDA tensor (there is no CPU path)")
    if not t.is_contiguous():
        raise RuntimeError("re2nn_b200: expected a contiguous tensor")
    return C.c_void_p(t.data_ptr())


def _f32(t):
    if t.dtype != torch.float32:
        raise RuntimeError("re2nn_b200: expected float32, got %s" % t.dtype)
    return _p(t)


def _i64(t):
    if t.dtype != torch.int64:
        raise RuntimeError("re2nn_b200: expected int64, got %s" % t.dtype)
    return _p(t)


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("re2nn_b200 needs a CUDA device (sm_100a); there is no CPU fallback")


def _rec_args(S, R, farnn, precision, B=0, L=0, Lpad=None, x=None, update_nonlinear=None, v_mode=V_TOKEN,
              full_pad=False, save_for_backward=False, sigmoid_exponent=0.0):
    """RecurrenceArgs with the shape and configuration fields set; the tensor pointers are left to the caller.
    Lpad defaults to the row stride of x (L without x)."""
    a = RecurrenceArgs()
    a.B, a.L, a.S, a.R = B, L, S, R
    a.Lpad = Lpad if Lpad is not None else (x.shape[1] if x is not None else L)
    a.farnn, a.precision = farnn, PREC[precision]
    a.update_nonlinear = NL[update_nonlinear] if update_nonlinear is not None else 0
    a.v_mode, a.full_pad, a.save_for_backward = v_mode, int(full_pad), int(save_for_backward)
    a.sigmoid_exponent = float(sigmoid_exponent)
    return a


def token_table(V_embed, E, G, beta_vec, additional_nonlinear):
    rows, R = V_embed.shape
    D = E.shape[1]
    out = torch.empty((rows, R), dtype=torch.float32, device=V_embed.device)
    check(fn['re2nn_token_table'](_f32(V_embed), _f32(E), _f32(G), _f32(beta_vec), rows, D, R,
                                  NL[additional_nonlinear], _f32(out), _stream()), 'token_table')
    _count(1)
    return out


def gate_table(vtab, Wrs1, bs1, Wrs2, bs2, farnn):
    rows, R = vtab.shape
    S = Wrs1.shape[1]
    out = torch.empty((rows, S * farnn), dtype=torch.float32, device=vtab.device)
    check(fn['re2nn_gate_table'](_f32(vtab), rows, R, S, farnn, _f32(Wrs1), _f32(bs1),
                                 _f32(Wrs2) if farnn == 2 else None, _f32(bs2) if farnn == 2 else None,
                                 _f32(out), _stream()), 'gate_table')
    _count(farnn)
    return out


def affine(x, W, b):
    """x (M x K) @ W (K x N) + b (N): fp32 CUDA-core GEMM with the bias in the epilogue (priority.py:20-30)."""
    return gate_table(x, W, b.reshape(1, -1).contiguous(), None, None, 1)


def output_vector_sum(C_mat, wildcard_vec=None):
    Cn, S = C_mat.shape
    o = torch.empty((S,), dtype=torch.float32, device=C_mat.device)
    check(fn['re2nn_output_vector_sum'](_f32(C_mat), Cn, S, _f32(wildcard_vec) if wildcard_vec is not None else None,
                                        _f32(o), _stream()), 'output_vector_sum')
    _count(1)
    return o


def decompose_recurrence(x, lengths, L, vtab, gtab, S1, S2, W, o, h0, hT, Wss1, Wss2, farnn,
                         update_nonlinear, sigmoid_exponent, precision='fp32', v_mode=V_TOKEN,
                         full_pad=False, save_for_backward=False, Lpad=None, max_semiring=False, zero_fill=False,
                         wprep=None):
    """Returns (alpha, beta, saves): alpha/beta B x L x S (pad rows undefined); saves = per-step slabs or None."""
    B = lengths.shape[0]
    S, R = S1.shape
    dev = S1.device
    a = _rec_args(S, R, farnn, precision, B, L, Lpad, x, update_nonlinear, v_mode, full_pad, save_for_backward,
                  sigmoid_exponent)
    # pad rows are never read downstream (label_scores masks them), so no zero-fill is needed
    alloc = torch.zeros if zero_fill else torch.empty
    alpha = alloc((B, L, S), dtype=torch.float32, device=dev)
    beta = alloc((B, L, S), dtype=torch.float32, device=dev)
    saves = None
    if save_for_backward:
        z = lambda *shape: torch.zeros(shape, dtype=torch.float32, device=dev)
        saves = dict(hbar=z(2, L + 1, B, S), hst=z(2, L + 1, B, S), u=z(2, L, B, R), a=z(2, L, B, S),
                     z=z(2, L, B, S) if farnn >= 1 else None, r=z(2, L, B, S) if farnn == 2 else None)
        a.hbar_save, a.hst_save = _f32(saves['hbar']), _f32(saves['hst'])
        a.u_save, a.a_save = _f32(saves['u']), _f32(saves['a'])
        a.zsave = _f32(saves['z']) if saves['z'] is not None else None
        a.rsave = _f32(saves['r']) if saves['r'] is not None else None
    if not save_for_backward and not zero_fill:
        # inference: the registered custom op (allocates alpha / beta and the workspace itself)
        for t in (lengths, vtab, S1, S2, W, o, h0, hT):
            _p(t)
        if precision == 'fp32' or max_semiring:
            wprep = None
        alpha, beta = tops.ifst_decompose_forward(x, lengths, vtab, gtab, S1, S2, W, o, h0, hT, Wss1, Wss2, L, a.Lpad, farnn,
                                                  a.update_nonlinear, a.precision, v_mode, bool(full_pad),
                                                  float(sigmoid_exponent), bool(max_semiring), wprep)
        a.wprep = C.c_void_p(wprep.data_ptr()) if wprep is not None else None
        _count(3 if max_semiring else fn['re2nn_decompose_recurrence_launches'](C.byref(a)))
        return alpha, beta, None
    a.x = _i64(x) if x is not None else None
    a.lengths = _i64(lengths)
    a.vtab, a.gtab = _f32(vtab), (_f32(gtab) if gtab is not None else None)
    a.S1, a.S2, a.W, a.o, a.h0, a.hT = _f32(S1), _f32(S2), _f32(W), _f32(o), _f32(h0), _f32(hT)
    a.Wss1 = _f32(Wss1) if Wss1 is not None else None
    a.Wss2 = _f32(Wss2) if Wss2 is not None else None
    a.alpha, a.beta = _f32(alpha), _f32(beta)
    if max_semiring:
        need = fn['re2nn_decompose_max_workspace'](S, R)
        ws = torch.empty((need,), dtype=torch.uint8, device=dev)
        a.ws, a.ws_bytes = C.c_void_p(ws.data_ptr()), need
        check(fn['re2nn_decompose_max_recurrence'](C.byref(a), _stream()), 'decompose_max_recurrence')
        _count(3)
        return alpha, beta, saves
    need = fn['re2nn_decompose_recurrence_workspace'](C.byref(a))
    ws = torch.empty((need,), dtype=torch.uint8, device=dev)
    a.ws, a.ws_bytes = C.c_void_p(ws.data_ptr()), need
    check(fn['re2nn_decompose_recurrence'](C.byref(a), _stream()), 'decompose_recurrence')
    _count(fn['re2nn_decompose_recurrence_launches'](C.byref(a)))
    return alpha, beta, saves


def weight_prep(S1, S2, W, Wss1, Wss2, farnn, precision):
    """Operand-format copies of the recurrence weights for `wprep` (tensor-core precisions): 6-8 conversion launches
    once per parameter version instead of once per call."""
    S, R = S1.shape
    a = _rec_args(S, R, farnn, precision)
    a.S1, a.S2, a.W = _f32(S1), _f32(S2), _f32(W)
    a.Wss1 = _f32(Wss1) if Wss1 is not None else None
    a.Wss2 = _f32(Wss2) if Wss2 is not None else None
    need = fn['re2nn_decompose_weight_prep_bytes'](C.byref(a))
    buf = torch.empty((need,), dtype=torch.uint8, device=S1.device)
    check(fn['re2nn_decompose_weight_prep'](C.byref(a), C.c_void_p(buf.data_ptr()), _stream()), 'decompose_weight_prep')
    _count(6 + farnn)
    return buf


def decompose_recurrence_fused(x, lengths, L, vtab, S1, S2, W, o, h0, hT, update_nonlinear, precision, v_mode=V_TOKEN,
                               Lpad=None, wprep=None):
    """Inference without gates on the per-step tensor-core path: the backward direction runs first and the forward
    direction's state epilogue writes (alpha * beta) straight in operand format, so alpha is never materialised and
    label scoring does not re-read the states.  -> (ab operand buffer, beta) or None when the call would not fuse
    (fp32, resident kernel)."""
    B = lengths.shape[0]
    S, R = S1.shape
    dev = S1.device
    a = _rec_args(S, R, 0, precision, B, L, Lpad, x, update_nonlinear, v_mode)
    if not fn['re2nn_decompose_recurrence_fuses'](C.byref(a)):
        return None
    nbytes = fn['re2nn_label_scores_ab_bytes'](B, L, S, PREC[precision])
    ab = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    beta = torch.empty((B, L, S), dtype=torch.float32, device=dev)
    a.ab_out = C.c_void_p(ab.data_ptr())
    a.x = _i64(x) if x is not None else None
    a.lengths = _i64(lengths)
    a.vtab = _f32(vtab)
    a.S1, a.S2, a.W, a.o, a.h0, a.hT = _f32(S1), _f32(S2), _f32(W), _f32(o), _f32(h0), _f32(hT)
    a.beta = _f32(beta)
    if wprep is not None:
        a.wprep = C.c_void_p(wprep.data_ptr())
    need = fn['re2nn_decompose_recurrence_workspace'](C.byref(a))
    ws = torch.empty((need,), dtype=torch.uint8, device=dev)
    a.ws, a.ws_bytes = C.c_void_p(ws.data_ptr()), need
    check(fn['re2nn_decompose_recurrence'](C.byref(a), _stream()), 'decompose_recurrence')
    _count(fn['re2nn_decompose_recurrence_launches'](C.byref(a)))
    return ab, beta


def label_scores_ab(ab, B, L, S, C_mat, priority_mat=None, priority_bias=None, precision='bf16'):
    """scores = ab @ C^T [@ P + b] from the fused operand of decompose_recurrence_fused."""
    Cn = C_mat.shape[0]
    scores = torch.empty((B, L, Cn), dtype=torch.float32, device=C_mat.device)
    has_pr = priority_mat is not None
    need = fn['re2nn_label_scores_workspace'](B, L, S, Cn, PREC[precision], int(has_pr))
    ws = torch.empty((need,), dtype=torch.uint8, device=C_mat.device)
    check(fn['re2nn_label_scores_ab'](C.c_void_p(ab.data_ptr()), B, L, S, _f32(C_mat), Cn,
                                      _f32(priority_mat) if has_pr else None,
                                      _f32(priority_bias) if priority_bias is not None else None, PREC[precision],
                                      _f32(scores), C.c_void_p(ws.data_ptr()), need, _stream()), 'label_scores_ab')
    _count(2 + (1 if has_pr else 0))
    return scores


def recurrence_fuses(S, R, farnn, precision):
    """Would an inference call of this shape write the fused (alpha * beta) operand when asked to?"""
    return bool(fn['re2nn_decompose_recurrence_fuses'](C.byref(_rec_args(S, R, farnn, precision))))


def onehot_recurrence(x, lengths, L, language, W, o, h0, hT, update_nonlinear, max_semiring=False, full_pad=False,
                      presummed=False):
    B, Lpad = x.shape
    S = language.shape[1]
    if presummed:
        for t in (x, lengths, language, o, h0, hT):
            _p(t)
        alpha, beta = tops.ifst_onehot_forward(x, lengths, language, o, h0, hT, L, NL[update_nonlinear], bool(max_semiring),
                                               bool(full_pad))
        _count(1)
        return alpha, beta
    a = OnehotArgs()
    a.B, a.Lpad, a.L, a.S = B, Lpad, L, S
    a.update_nonlinear, a.max_semiring, a.full_pad = NL[update_nonlinear], int(max_semiring), int(full_pad)
    alpha = torch.zeros((B, L, S), dtype=torch.float32, device=language.device)
    beta = torch.zeros((B, L, S), dtype=torch.float32, device=language.device)
    a.x, a.lengths = _i64(x), _i64(lengths)
    a.language, a.W, a.o, a.h0, a.hT = _f32(language), _f32(W), _f32(o), _f32(h0), _f32(hT)
    a.alpha, a.beta = _f32(alpha), _f32(beta)
    check(fn['re2nn_onehot_recurrence'](C.byref(a), _stream()), 'onehot_recurrence')
    _count(1)
    return alpha, beta


def label_scores(alpha, beta, lengths, C_mat, priority_mat=None, priority_bias=None, full_pad=False,
                 precision='fp32'):
    for t in (alpha, beta, lengths, C_mat):
        _p(t)
    scores = tops.label_scores(alpha, beta, lengths, C_mat, priority_mat, priority_bias, bool(full_pad), PREC[precision])
    _count((1 if precision == 'fp32' else 3) + (1 if priority_mat is not None else 0))
    return scores


def argmax_decode(scores, lengths, offsets, n_flat, clamp_col, threshold, o_idx, want_flat=True, want_padded=False,
                  flat_out=None):
    """flat_out: optional shared int64 buffer the flat predictions are scattered into (through `offsets`)."""
    for t in (scores, lengths):
        _p(t)
    flat, padded = tops.argmax_decode(scores, lengths, offsets, int(n_flat), int(clamp_col), float(threshold), int(o_idx),
                                      bool(want_flat), bool(want_padded), flat_out)
    _count(1)
    return ((flat_out if flat_out is not None else flat) if want_flat else None), (padded if want_padded else None)


def crf_viterbi(feats, transitions, lengths, offsets=None, n_flat=0, clamp_col=-1, threshold=0.0, o_idx=0,
                want_flat=False, want_padded=True, flat_out=None):
    for t in (feats, transitions, lengths):
        _p(t)
    flat, padded = tops.crf_viterbi(feats, transitions, lengths, offsets, int(n_flat), int(clamp_col), float(threshold),
                                    int(o_idx), bool(want_flat), bool(want_padded), flat_out)
    _count(1)
    return ((flat_out if flat_out is not None else flat) if want_flat else None), (padded if want_padded else None)


def crf_nll(feats, transitions, lengths, tags, save=False):
    for t in (feats, transitions, lengths, tags):
        _p(t)
    loss, per_seq, part = tops.crf_nll(feats, transitions, lengths, tags, bool(save))
    _count(2)
    return loss, per_seq, (part if save else None)


def crf_nll_backward(feats, transitions, lengths, tags, part, gscale):
    dfeats, dtrans = tops.crf_nll_backward(feats, transitions, lengths, tags, part, gscale)
    _count(1)
    return dfeats, dtrans


def ce_loss(scores, lengths, labels, n_total):
    B, L, Cn = scores.shape
    per_pos = torch.empty((B * L,), dtype=torch.float32, device=scores.device)
    loss = torch.empty((), dtype=torch.float32, device=scores.device)
    check(fn['re2nn_ce_loss'](_f32(scores), _i64(lengths), _i64(labels), B, L, labels.shape[1], Cn, int(n_total),
                              _f32(per_pos), _f32(loss), _stream()), 'ce_loss')
    _count(2)
    return loss


def ce_loss_backward(scores, lengths, labels, n_total, gscale):
    B, L, Cn = scores.shape
    d = torch.empty_like(scores)
    check(fn['re2nn_ce_loss_backward'](_f32(scores), _i64(lengths), _i64(labels), _f32(gscale), B, L,
                                       labels.shape[1], Cn, int(n_total), _f32(d), _stream()), 'ce_loss_backward')
    _count(1)
    return d


def profile_enable(on):
    check(fn['re2nn_profile_enable'](int(on)), 'profile_enable')


def recurrence_is_resident(S, R, farnn, precision):
    """Would an inference call of this shape run all steps in the resident kernel?"""
    return bool(fn['re2nn_decompose_recurrence_resident'](C.byref(_rec_args(S, R, farnn, precision))))


def profile_read():
    """-> ([ms_gate, ms_gemm1, ms_gemm2, ms_resident], [n_gate, n_gemm1, n_gemm2, n_resident]) since the last read."""
    ms = (C.c_double * 4)()
    cnt = (C.c_int64 * 4)()
    check(fn['re2nn_profile_read'](ms, cnt), 'profile_read')
    return list(ms), list(cnt)


def profile_enabled():
    return bool(fn['re2nn_profile_enabled']())


def profile_intervals(cls, clear=False):
    """[(start_ms, end_ms), ...] of the launches of kernel class `cls` (3 = resident recurrence) as they last ran --
    inside a replayed CUDA graph too.  Times are relative to the earliest start of the class."""
    n = fn['re2nn_profile_count'](cls)
    s = (C.c_double * max(n, 1))()
    e = (C.c_double * max(n, 1))()
    check(fn['re2nn_profile_intervals'](cls, s, e, n, int(clear)), 'profile_intervals')
    return [(s[i], e[i]) for i in range(n)]


def has_tcgen05():
    return bool(fn['re2nn_has_tcgen05']())


def gemm_nt(A, B, precision='fp32'):
    """C = A @ B^T through the selected step-GEMM mainloop (test / calibration entry)."""
    M, K = A.shape
    N = B.shape[0]
    out = torch.empty((M, N), dtype=torch.float32, device=A.device)
    need = fn['re2nn_gemm_nt_workspace'](PREC[precision], M, N, K)
    ws = torch.empty((need,), dtype=torch.uint8, device=A.device)
    check(fn['re2nn_gemm_nt'](PREC[precision], _f32(A), _f32(B), M, N, K, _f32(out), C.c_void_p(ws.data_ptr()), need,
                              _stream()), 'gemm_nt')
    _count(1 if precision == 'fp32' else 3)
    return out


_TN_PATH = {'auto': 0, 'cuda': 1, 'tc': 2}


def gemm_tn_workspace(P, Q):
    return fn['re2nn_gemm_tn_workspace'](P, Q)


def gemm_tn_path(P, Q, rows, has_y2=False):
    """'cuda' or 'tc': the kernel the decompose backward runs a P x Q weight gradient over `rows` summed rows on."""
    return {1: 'cuda', 2: 'tc'}[fn['re2nn_gemm_tn_path'](P, Q, rows, int(has_y2))]


def gemm_tn(X0, Y0, X1=None, Y1=None, Y2=None, mask_len=None, path='auto', ws=None):
    """C = X0^T (Y0 [* Y2]) [+ X1^T Y1] through the weight-gradient GEMMs of the backward (test / calibration entry).
    Operands are 2-D fp32 CUDA tensors whose rows are the reduction index; each may be a column slice of a wider slab
    (unit column stride, any row stride).  mask_len (int64, B entries, needs Y2): row b * L + t of Y0 * Y2 counts only
    when t < mask_len[b], with L = rows / B.  path: 'auto' (the backward's choice), 'cuda' or 'tc'.  ws: optional
    uint8 scratch of gemm_tn_workspace(P, Q) bytes (the split-K partials)."""
    def ld(t):
        if t.dtype != torch.float32 or not t.is_cuda or t.dim() != 2 or (t.shape[0] > 1 and t.stride(1) != 1):
            raise RuntimeError("re2nn_b200: gemm_tn operands are 2-D fp32 CUDA tensors with unit column stride")
        return max(t.stride(0), t.shape[1])

    def ptr(t):
        return C.c_void_p(t.data_ptr()) if t is not None else None
    rows0, P = X0.shape
    Q = Y0.shape[1]
    rows1 = X1.shape[0] if X1 is not None else 0
    if Y0.shape[0] != rows0 or (X1 is not None and (Y1.shape[0] != rows1 or X1.shape[1] != P or Y1.shape[1] != Q)):
        raise RuntimeError("re2nn_b200: gemm_tn operand shapes do not match")
    if Y2 is not None and (Y2.shape != Y0.shape or ld(Y2) != ld(Y0)):
        raise RuntimeError("re2nn_b200: gemm_tn Y2 must have Y0's shape and leading dimension")
    mask_L = 0
    if mask_len is not None:
        if mask_len.numel() == 0 or rows0 % mask_len.numel() != 0:
            raise RuntimeError("re2nn_b200: gemm_tn rows must be B * L with B = len(mask_len)")
        mask_L = rows0 // mask_len.numel()
    out = torch.empty((P, Q), dtype=torch.float32, device=X0.device)
    need = gemm_tn_workspace(P, Q)
    if ws is None:
        ws = torch.empty((need,), dtype=torch.uint8, device=X0.device)
    elif ws.numel() * ws.element_size() < need or not ws.is_cuda:
        raise RuntimeError("re2nn_b200: gemm_tn workspace too small")
    check(fn['re2nn_gemm_tn'](_TN_PATH[path], P, Q, ptr(X0), ptr(Y0), ld(X0), ld(Y0), rows0,
                              ptr(X1), ptr(Y1), ld(X1) if X1 is not None else 0, ld(Y1) if Y1 is not None else 0, rows1,
                              ptr(Y2), _i64(mask_len) if mask_len is not None else None, mask_L,
                              _f32(out), C.c_void_p(ws.data_ptr()), need, _stream()), 'gemm_tn')
    _count(2)
    return out


def batched_vecmat(h, T, transposed=False, max_semiring=False):
    """out[b,s] = (+|max)_j h[b,j] * T[b,j,s] (or T[b,s,j] when transposed); -> (out, argmax int32 or None)."""
    B, S = h.shape
    out = torch.empty((B, S), dtype=torch.float32, device=h.device)
    idx = torch.empty((B, S), dtype=torch.int32, device=h.device) if max_semiring else None
    check(fn['re2nn_batched_vecmat'](_f32(h), _f32(T), B, S, int(transposed), int(max_semiring), _f32(out),
                                     _p(idx) if idx is not None else None, _stream()), 'batched_vecmat')
    _count(1)
    return out, idx


def decompose_backward(consts, p, x, dense_v, lengths, L, vtab, o, alpha, beta, saves, dscores, pr_mat, want,
                       dalpha_in=None, dbeta_in=None):
    """BPTT through both directions.  `want` = set of gradient names to produce.  Returns dict name -> tensor
    (plus 'vtab' = d loss / d token-table rows, 'o' = d loss / d output_vector_sum).
    dalpha_in / dbeta_in: gradients w.r.t. alpha / beta supplied by a caller that differentiates its own score stage
    (FST variants); dscores, C_output_mat and the priority matrix are then unused."""
    B = lengths.shape[0]
    S, R = p['S1'].shape
    direct = dalpha_in is not None
    Cn = 0 if direct else p['C_output_mat'].shape[0]
    dev = alpha.device
    farnn = consts['farnn']
    a = BackwardArgs()
    a.B, a.L, a.S, a.R, a.C = B, L, S, R, Cn
    a.Lpad = x.shape[1] if dense_v is None else dense_v.shape[1]
    a.farnn, a.update_nonlinear = farnn, NL[consts['update_nonlinear']]
    a.v_mode = V_TOKEN if dense_v is None else V_DENSE
    a.full_pad, a.ce1 = int(consts['full_pad']), int(consts['ce1'])
    a.table_rows = vtab.shape[0]
    a.sigmoid_exponent = float(consts['sigmoid_exponent'])
    a.x = _i64(x) if x is not None else None
    a.lengths = _i64(lengths)
    a.dscores = _f32(dscores) if not direct else None
    a.priority_mat = _f32(pr_mat) if (pr_mat is not None and not direct) else None
    if direct:
        a.dalpha_in, a.dbeta_in = _f32(dalpha_in), _f32(dbeta_in)
    a.vtab, a.S1, a.S2, a.W, a.o = _f32(vtab), _f32(p['S1']), _f32(p['S2']), _f32(p['wildcard_mat']), _f32(o)
    a.h0, a.hT = _f32(p['h0']), _f32(p['hT'])
    a.C_mat = _f32(p['C_output_mat']) if not direct else None
    for n in ('Wss1', 'Wss2', 'Wrs1', 'Wrs2'):
        setattr(a, n, _f32(p[n]) if n in p else None)
    a.alpha, a.beta = _f32(alpha), _f32(beta)
    a.hbar_save, a.hst_save, a.u_save, a.a_save = (_f32(saves[k]) for k in ('hbar', 'hst', 'u', 'a'))
    a.zsave = _f32(saves['z']) if saves['z'] is not None else None
    a.rsave = _f32(saves['r']) if saves['r'] is not None else None
    out = {}

    def grad(name, like, field):
        if name in want:
            out[name] = torch.empty_like(like)
            setattr(a, field, _f32(out[name]))

    grad('S1', p['S1'], 'dS1'); grad('S2', p['S2'], 'dS2'); grad('wildcard_mat', p['wildcard_mat'], 'dW')
    grad('h0', p['h0'], 'dh0'); grad('hT', p['hT'], 'dhT')
    if not direct:
        out['C_output_mat'] = torch.empty_like(p['C_output_mat']); a.dC = _f32(out['C_output_mat'])
    out['o'] = torch.empty((S,), dtype=torch.float32, device=dev); a.d_o = _f32(out['o'])
    if farnn >= 1:
        grad('Wss1', p['Wss1'], 'dWss1'); grad('Wrs1', p['Wrs1'], 'dWrs1'); grad('bs1', p['bs1'], 'dbs1')
    if farnn == 2:
        grad('Wss2', p['Wss2'], 'dWss2'); grad('Wrs2', p['Wrs2'], 'dWrs2'); grad('bs2', p['bs2'], 'dbs2')
    out['vtab'] = torch.empty_like(vtab); a.dvtab = _f32(out['vtab'])
    need = fn['re2nn_decompose_backward_workspace'](C.byref(a))
    ws = torch.empty((need,), dtype=torch.uint8, device=dev)
    a.ws, a.ws_bytes = C.c_void_p(ws.data_ptr()), need
    check(fn['re2nn_decompose_backward'](C.byref(a), _stream()), 'decompose_backward')
    # launches of the default path: without gates E1 once + (GEMM, E2, GEMM, E3+E1) per step; with gates
    # (E1, GEMM, E2, GEMM, E3, gate GEMM, scatter) per step; around the sweep: weight copies 6, label-score backward 3,
    # four to eight weight-gradient GEMMs + their ordered reductions, column sums
    _count((L * 4 + 1 if farnn == 0 else L * 7) + 22 + (12 if farnn else 0))
    return out


def token_table_backward(dvtab, V_embed, E, G, beta_vec, additional_nonlinear, want):
    rows, R = V_embed.shape
    D = E.shape[1]
    dev = dvtab.device
    out = {}
    dV = torch.empty_like(V_embed) if 'V_embed' in want else None
    dbeta = torch.empty_like(beta_vec) if 'beta_vec' in want else None
    dG = torch.empty_like(G) if 'embed_r_generalized' in want else None
    dE = torch.empty_like(E) if 'embedding' in want else None
    need = fn['re2nn_token_table_backward_workspace'](rows, D, R)
    ws = torch.empty((need,), dtype=torch.uint8, device=dev)
    check(fn['re2nn_token_table_backward'](_f32(dvtab), _f32(V_embed), _f32(E), _f32(G), _f32(beta_vec), rows, D, R,
                                           NL[additional_nonlinear], _f32(dV) if dV is not None else None,
                                           _f32(dbeta) if dbeta is not None else None,
                                           _f32(dG) if dG is not None else None, _f32(dE) if dE is not None else None,
                                           C.c_void_p(ws.data_ptr()), need, _stream()), 'token_table_backward')
    _count(5)
    for k, v in (('V_embed', dV), ('beta_vec', dbeta), ('embed_r_generalized', dG), ('embedding', dE)):
        if v is not None:
            out[k] = v
    return out


def onehot_backward(x, lengths, L, language, W, o, h0, hT, alpha, beta, dscores, C_mat, pr_mat, update_nonlinear,
                    full_pad, presummed=False):
    """d loss / d language_tensor for the sum-semiring onehot recurrence."""
    B, Lpad = x.shape
    S = language.shape[1]
    Cn = C_mat.shape[0]
    dev = language.device
    dalpha = torch.empty_like(alpha)
    dbeta = torch.empty_like(beta)
    ws = torch.empty((B, L, Cn), dtype=torch.float32, device=dev) if pr_mat is not None else None
    check(fn['re2nn_label_scores_backward'](_f32(dscores), _f32(alpha), _f32(beta), _i64(lengths), B, L, S, _f32(C_mat),
                                            Cn, _f32(pr_mat) if pr_mat is not None else None, int(full_pad),
                                            _f32(dalpha), _f32(dbeta), _f32(ws) if ws is not None else None, _stream()),
          'label_scores_backward')
    dlang = torch.zeros_like(language)
    a = OnehotBackwardArgs()
    a.B, a.Lpad, a.L, a.S = B, Lpad, L, S
    a.update_nonlinear, a.full_pad = NL[update_nonlinear], int(full_pad)
    a.x, a.lengths = _i64(x), _i64(lengths)
    a.language, a.W, a.o, a.h0, a.hT = _f32(language), (_f32(W) if not presummed else None), _f32(o), _f32(h0), _f32(hT)
    a.alpha, a.beta, a.dalpha, a.dbeta, a.dlanguage = _f32(alpha), _f32(beta), _f32(dalpha), _f32(dbeta), _f32(dlang)
    check(fn['re2nn_onehot_backward'](C.byref(a), _stream()), 'onehot_backward')
    _count(3 if pr_mat is not None else 2)
    return dlang


def length_order(lengths, L):
    """Longest-first schedule in one launch -> (order, lengths_sorted, offsets, offsets_sorted) (all int64[B]), or None
    when the batch is outside the single-CTA kernel's range (the caller then uses torch.sort / cumsum / gathers)."""
    B = lengths.shape[0]
    if not fn['re2nn_length_order_supported'](B, int(L)):
        return None
    out = torch.empty((4, B), dtype=torch.int64, device=lengths.device)
    check(fn['re2nn_length_order'](_i64(lengths), B, int(L), _i64(out[0]), _i64(out[1]), _i64(out[2]), _i64(out[3]),
                                   _stream()), 'length_order')
    _count(1)
    return out[0], out[1], out[2], out[3]


def flatten_i64(padded, lengths, offsets, L, n_flat):
    """Valid prefixes of an int64 B x Lrow tensor, batch-major (no host sync)."""
    B, Lrow = padded.shape
    flat = torch.empty((n_flat,), dtype=torch.int64, device=padded.device)
    check(fn['re2nn_flatten_i64'](_i64(padded), _i64(lengths), _i64(offsets), B, Lrow, L, _i64(flat), _stream()),
          'flatten_i64')
    _count(1)
    return flat


def onehot_sum_tensor(language, W):
    out = torch.empty_like(language)
    V1, S = language.shape[0], language.shape[1]
    check(fn['re2nn_onehot_sum_tensor'](_f32(language), _f32(W), V1, S, _f32(out), _stream()), 'onehot_sum_tensor')
    _count(1)
    return out
