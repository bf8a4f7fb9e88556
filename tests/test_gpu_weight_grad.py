"""GPU: the weight-gradient GEMMs of the decompose backward, C[P x Q] = sum_m X[m, p] Y[m, q] over every (step, sequence)
row, against float64.

Kernel level (re2nn_gemm_tn through ops.gemm_tn): every case runs the CUDA-core split-K kernel ('cuda') and the tcgen05
kernel in 3xTF32 ('tc', gemm_tn_tc.cuh: operands transposed by the loader warps, split-K, optional length mask).  The
reference is X.double().T @ Y.double() on the GPU.  Errors are reported two ways: max-norm relative
(max|C - ref| / max|ref|, the measure DESIGN.md section 2 bounds by 2e-5) and element-wise relative to |X|^T |Y|, the
scale every accumulated product and every rounding of a partial sum is bounded by, so it survives cancellation.

Training level: a shape at which every weight gradient of the backward runs on tcgen05, gradients against the float64
autograd oracle, with the GEMMs of every BPTT step on tcgen05 (the default) and on CUDA cores."""
import numpy as np
import pytest
import torch

from helpers import oracle_gradient_errors

pytestmark = pytest.mark.gpu

MAXNORM_TOL = 2e-5          # DESIGN.md section 2
# Element-wise bound relative to |X|^T |Y|, set from the measurements of this file on a B200: the largest value is
# 1.19e-5 (tcgen05, 48 k-blocks per split, uniform [0, 1) data, where element-wise and max-norm coincide); on signed
# data it stays below 3.5e-7, on the CUDA-core kernel below 7.2e-7.  The bound is the DESIGN.md one, 1.7x above that.
EW_TOL = 2e-5


def _need_tc():
    from re2nn_seq_b200 import ops
    if not ops.has_tcgen05():
        pytest.skip('no tcgen05')


def _gen(seed):
    g = torch.Generator(device='cuda')
    g.manual_seed(seed)
    return g


def _signed(rows, cols, g):
    return torch.randn(rows, cols, device='cuda', generator=g)


def _tanh(rows, cols, g):
    return torch.tanh(torch.randn(rows, cols, device='cuda', generator=g) + 0.3)


def _reference(X0, Y0, X1=None, Y1=None, Y2=None, mask_len=None):
    """(C, |X|^T |Y|) in float64; masked rows of Y0 * Y2 are zero whatever they hold."""
    Y = Y0.double()
    if Y2 is not None:
        Y = Y * Y2.double()
    if mask_len is not None:
        B = mask_len.numel()
        L = Y.shape[0] // B
        keep = (torch.arange(L, device='cuda')[None, :] < mask_len[:, None]).reshape(-1, 1)
        Y = torch.where(keep, Y, torch.zeros((), dtype=torch.float64, device='cuda'))
    X = X0.double()
    C = X.T @ Y
    if X1 is not None:
        C += X1.double().T @ Y1.double()
    if all(t is None or t.min() >= 0 for t in (X0, Y, X1, Y1)):
        return C, C
    A = X.abs().T @ Y.abs()
    if X1 is not None:
        A += X1.double().abs().T @ Y1.double().abs()
    return C, A


def _errors(C, ref, A):
    d = (C.double() - ref).abs()
    maxnorm = (d.max() / ref.abs().max().clamp_min(1e-300)).item()
    ew = torch.where(A > 0, d / A.clamp_min(1e-300), torch.where(d > 0, torch.full_like(d, float('inf')), d)).max().item()
    return maxnorm, ew


def _check(label, operands, paths=('cuda', 'tc'), maxnorm_tol=MAXNORM_TOL, ew_tol=EW_TOL, exact=False, capsys=None):
    """Run gemm_tn on every path, compare with float64 and print the errors."""
    from re2nn_seq_b200 import ops
    ref, A = _reference(**operands)
    for path in paths:
        C = ops.gemm_tn(path=path, **operands)
        torch.cuda.synchronize()
        if exact:
            d = (C.double() - ref).abs().max().item()
            line = '%s %s: %s' % (label, path, 'exact' if d == 0 else 'max |diff| %g' % d)
        else:
            mn, ew = _errors(C, ref, A)
            line = '%s %s: max-norm %.2e, element-wise %.2e' % (label, path, mn, ew)
        if capsys is not None:
            with capsys.disabled():
                print('\n' + line, end='')
        assert torch.isfinite(C).all(), line
        if exact:
            assert torch.equal(C.double(), ref), line
        else:
            assert mn <= maxnorm_tol, line
            assert ew <= ew_tol, line


# ---- tile edges: nt = cdiv(Q, 256) n-tiles of bn = round_up(cdiv(Q, nt), 16) columns, cdiv(P, 128) m-tiles --------
TILE_CASES = [
    (16, 16),       # nt 1, bn 16: the smallest tile
    (17, 17),       # bn 32 rounded up from 17, P one past the 16 bound
    (16, 1024),     # nt 4, bn 256
    (72, 200),      # cfg3 dC-like
    (127, 256),     # one m-tile short of full, nt 1 full width
    (128, 257),     # nt 2, bn 144
    (129, 300),     # two m-tiles, the second one row wide; nt 2, bn 160
    (300, 513),     # nt 3, bn 176
    (17, 513),      # nt 3 with a narrow P
    (1024, 16),     # eight m-tiles, bn 16
    (128, 17),      # bn 32
    (1024, 1024),   # 32 tiles
    (300, 200),     # cfg3 dS1
    (127, 1024),
    (129, 16),
]


@pytest.mark.parametrize('P,Q', TILE_CASES)
def test_gemm_tn_tile_edges(P, Q, capsys):
    _need_tc()
    g = _gen(P * 7919 + Q)
    rows = 5003                                  # ragged last k-block, above the 4096-row tensor-core threshold
    _check('tile P=%d Q=%d rows=%d' % (P, Q, rows), dict(X0=_signed(rows, P, g), Y0=_tanh(rows, Q, g)), capsys=capsys)


@pytest.mark.parametrize('rows', [1, 31, 32, 33, 4095, 4096, 4097, 70001])
def test_gemm_tn_row_counts(rows, capsys):
    _need_tc()
    g = _gen(rows)
    _check('rows=%d P=72 Q=200' % rows, dict(X0=_signed(rows, 72, g), Y0=_tanh(rows, 200, g)), capsys=capsys)


def test_gemm_tn_two_pairs(capsys):
    """Two pairs with different row counts (the state-weight products: forward and backward direction)."""
    _need_tc()
    g = _gen(11)
    ops_ = dict(X0=_signed(5000, 97, g), Y0=_tanh(5000, 45, g), X1=_signed(3001, 97, g), Y1=_tanh(3001, 45, g))
    _check('two pairs 5000 + 3001 rows, P=97 Q=45', ops_, capsys=capsys)


def test_gemm_tn_splits_without_k_blocks():
    """P = Q = 16 over 33 rows: two k-blocks for up to 64 splits, so most splits reduce nothing and must write zeros
    over a workspace that holds NaN.  Integer data: the result is exact."""
    from re2nn_seq_b200 import ops
    _need_tc()
    g = _gen(5)
    X = torch.randint(-3, 4, (33, 16), device='cuda', generator=g).float()
    Y = torch.randint(-3, 4, (33, 16), device='cuda', generator=g).float()
    ref = X.double().T @ Y.double()
    ws = torch.full((ops.gemm_tn_workspace(16, 16) // 4,), float('nan'), device='cuda')
    for path in ('cuda', 'tc'):
        C = ops.gemm_tn(X, Y, path=path, ws=ws)
        assert torch.equal(C.double(), ref), path


def test_gemm_tn_strided_operands(capsys):
    """ldx > P, and the layout of dWrs2: Y = dgtab[:, S:2S] inside a slab of width 2S.  S is odd, so Y starts 388 bytes
    into the slab (not 16-byte aligned) and its rows are not either."""
    _need_tc()
    g = _gen(21)
    S, R, rows = 97, 45, 4501
    xs = _signed(rows, R + 13, g)
    slab = _tanh(rows, 2 * S, g)
    X, Y = xs[:, :R], slab[:, S:]
    assert X.stride(0) == R + 13 and Y.stride(0) == 2 * S and (Y.data_ptr() % 16) != 0
    _check('strided: X ld %d (P %d), Y = slab[:, S:] ld %d (Q %d)' % (R + 13, R, 2 * S, S), dict(X0=X, Y0=Y),
           capsys=capsys)
    _check('strided: dWrs1 layout Y = slab[:, :S]', dict(X0=X, Y0=slab[:, :S]), capsys=capsys)


def _masked_operands(B, L, P, Q, seed, poison):
    """dC layout: X = draw (B*L x P), Y0 = alpha, Y2 = beta (B*L x Q); lengths include 0 and L; with `poison` the pad
    rows of alpha and beta hold NaN / Inf (they are undefined in the backward)."""
    g = _gen(seed)
    lens = torch.randint(0, L + 1, (B,), device='cuda', generator=g)
    lens[0], lens[1], lens[-1] = L, 0, 0
    lens[2] = L - 1
    X = _signed(B * L, P, g)
    Y0, Y2 = _tanh(B * L, Q, g), _tanh(B * L, Q, g)
    if poison:
        pad = (torch.arange(L, device='cuda')[None, :] >= lens[:, None]).reshape(-1)
        Y0[pad] = float('nan')
        Y2[pad] = float('inf')
        Y2[pad.nonzero()[::2, 0]] = float('-inf')
    return dict(X0=X, Y0=Y0, Y2=Y2, mask_len=lens)


def test_gemm_tn_masked_dc(capsys):
    """dC = draw^T (alpha * beta) over the valid rows, B = 141, L = 31 (4371 rows), C = 17, S = 97: NaN / Inf in the pad
    rows of both right-hand factors must not reach the result."""
    _need_tc()
    ops_ = _masked_operands(141, 31, 17, 97, 31, poison=True)
    _check('masked dC B=141 L=31 P=17 Q=97', ops_, paths=('cuda', 'tc', 'auto'), capsys=capsys)
    full = dict(ops_, mask_len=None)
    g = _gen(32)
    full['Y0'], full['Y2'] = _tanh(141 * 31, 97, g), _tanh(141 * 31, 97, g)      # full_pad: every row counts
    _check('unmasked dC (full_pad) B=141 L=31 P=17 Q=97', full, paths=('cuda', 'tc', 'auto'), capsys=capsys)


def test_gemm_tn_masked_dc_chunked(capsys):
    """More rows than one launch of the tensor-core kernel reduces (64 splits x 128 k-blocks = 262144): the rows go in
    two chunks, the second starting on sequence 8456 (262136 = 8456 * 31 rows), with its own slice of the lengths."""
    _need_tc()
    ops_ = _masked_operands(8500, 31, 24, 40, 33, poison=True)
    _check('masked dC chunked B=8500 L=31 P=24 Q=40', ops_, capsys=capsys)


def test_gemm_tn_exact_integers(capsys):
    """Small integers are exact in the tf32 hi plane (the lo planes are zero) and every partial sum stays below 2^24,
    so any transposition, swizzle, split-range, pair or mask error shows as a wrong integer."""
    _need_tc()
    g = _gen(41)

    def ints(r, c):
        return torch.randint(-3, 4, (r, c), device='cuda', generator=g).float()
    _check('exact: two pairs 70001 + 9000 rows, P=129 Q=513',
           dict(X0=ints(70001, 129), Y0=ints(70001, 513), X1=ints(9000, 129), Y1=ints(9000, 513)), exact=True,
           capsys=capsys)
    _check('exact: P=17 Q=17 rows=33', dict(X0=ints(33, 17), Y0=ints(33, 17)), exact=True, capsys=capsys)
    slab = ints(4501, 2 * 97)
    _check('exact: strided Y = slab[:, 97:]', dict(X0=ints(4501, 45), Y0=slab[:, 97:]), exact=True, capsys=capsys)
    # pad rows hold finite integers here: a row the mask wrongly lets through changes the result
    m = _masked_operands(141, 31, 17, 97, 42, poison=False)
    m.update(X0=ints(*m['X0'].shape), Y0=ints(*m['Y0'].shape), Y2=ints(*m['Y2'].shape))
    _check('exact: masked dC', m, exact=True, capsys=capsys)
    _check('exact: chunked, 300000 rows P=16 Q=24', dict(X0=ints(300000, 16), Y0=ints(300000, 24)), exact=True,
           capsys=capsys)
    m = _masked_operands(8500, 31, 16, 16, 43, poison=False)
    m.update(X0=ints(*m['X0'].shape), Y0=ints(*m['Y0'].shape), Y2=ints(*m['Y2'].shape))
    _check('exact: masked dC chunked B=8500 L=31', m, exact=True, capsys=capsys)


def test_gemm_tn_deterministic():
    from re2nn_seq_b200 import ops
    _need_tc()
    g = _gen(51)
    ops_ = dict(X0=_signed(70001, 300, g), Y0=_tanh(70001, 200, g), X1=_signed(9000, 300, g), Y1=_tanh(9000, 200, g))
    m = _masked_operands(8500, 31, 24, 40, 52, poison=True)
    for path in ('cuda', 'tc'):
        assert torch.equal(ops.gemm_tn(path=path, **ops_), ops.gemm_tn(path=path, **ops_)), path
        assert torch.equal(ops.gemm_tn(path=path, **m), ops.gemm_tn(path=path, **m)), path


# ---- long reductions: the TMEM accumulator truncates every add, so a split's error grows with its chain ------------
LONG_CASES = [
    ('P=Q=1024 rows=131072', 1024, 1024, (131072,)),
    ('P=Q=2048 rows=2x35840', 2048, 2048, (35840, 35840)),     # dW at S = 2048 over the cfg3 batch: 128 tiles
    ('P=16 Q=24 rows=300000 (chunked)', 16, 24, (300000,)),
    ('P=Q=64 rows=2x140000 (chunked)', 64, 64, (140000, 140000)),
]


@pytest.mark.parametrize('data', ['signed', 'positive'])
@pytest.mark.parametrize('label,P,Q,rows', LONG_CASES, ids=[c[0].split(' ')[0] + '_' + c[0].split(' ')[1] for c in LONG_CASES])
def test_gemm_tn_long_chains(label, P, Q, rows, data, capsys):
    """Long reductions within the DESIGN.md gradient bound: signed data (randn x tanh) and positive data (uniform [0, 1),
    where every truncation pulls the same way)."""
    _need_tc()
    g = _gen(P + Q + sum(rows) + (data == 'positive'))
    ops_ = {}
    for i, r in enumerate(rows):
        if data == 'signed':
            X, Y = _signed(r, P, g), _tanh(r, Q, g)
        else:
            X = torch.rand(r, P, device='cuda', generator=g)
            Y = torch.rand(r, Q, device='cuda', generator=g)
        ops_['X%d' % i], ops_['Y%d' % i] = X, Y
    _check('long %s %s' % (label, data), ops_, capsys=capsys)


def test_gemm_tn_path_query():
    """re2nn_gemm_tn_path follows the backward's threshold: tcgen05 from 4096 summed rows with P, Q >= 16."""
    from re2nn_seq_b200 import ops
    _need_tc()
    assert ops.gemm_tn_path(300, 200, 71680) == 'tc'
    assert ops.gemm_tn_path(16, 16, 4096) == 'tc'
    assert ops.gemm_tn_path(16, 16, 4095) == 'cuda'
    assert ops.gemm_tn_path(15, 200, 71680) == 'cuda'
    assert ops.gemm_tn_path(200, 15, 71680, True) == 'cuda'
    assert ops.gemm_tn_path(72, 300, 35840, True) == 'tc'
    with pytest.raises(RuntimeError, match='P, Q >= 16'):
        ops.gemm_tn(torch.zeros(5000, 15, device='cuda'), torch.zeros(5000, 16, device='cuda'), path='tc')


# ---- training: every weight gradient of the backward on tcgen05, against the float64 oracle ------------------------
V, S, R, D, B, L = 4500, 97, 45, 24, 141, 31
TRAIN_ALL = dict(train_beta=1, train_h0=1, train_hT=1, train_V_embed=1, train_wildcard=1, train_wildcard_wildcard=1,
                 train_word_embed=1, train_c_output=1)
TRAIN_CASES = {
    'f0_tanh_crf': dict(farnn=0, update_nonlinear='tanh', use_crf=1),
    # relu is unbounded: S1, S2 and wildcard_mat at half scale keep 31 steps from growing the states (and the fp32
    # loss) by orders of magnitude
    'f1_relu_ce': dict(farnn=1, update_nonlinear='relu', use_crf=0, local_loss_func='CE', additional_nonlinear='tanh',
                       shrink=0.5),
    'f2_tanh_crf': dict(farnn=2, update_nonlinear='tanh', use_crf=1, local_loss_func='CE'),
    'f2_relutanh_ce1': dict(farnn=2, update_nonlinear='relutanh', use_crf=0, local_loss_func='CE1'),
    # the reference has no sigmoid update nonlinearity (it falls through to identity): sigmoid is the token-table one
    'f0_sigmoid_crf_priority': dict(farnn=0, update_nonlinear='tanh', use_crf=1, use_priority=1,
                                    additional_nonlinear='sigmoid'),
    'sf_f2_tanh_crf': dict(farnn=2, update_nonlinear='tanh', use_crf=1, sf=True),
    'f0_tanh_crf_auto': dict(farnn=0, update_nonlinear='tanh', use_crf=1, train_precision='auto'),
    'f1_tanh_ce_c13': dict(farnn=1, update_nonlinear='tanh', use_crf=0, local_loss_func='CE', C=13),
}


def _train_case(name, seed):
    import re2nn_seq_b200 as r
    from re2nn_seq_b200 import synth
    flags = dict(TRAIN_CASES[name])
    sf = flags.pop('sf', False)
    tp = flags.pop('train_precision', None)
    C = flags.pop('C', 17)
    shrink = flags.pop('shrink', 1.0)
    flags.update(TRAIN_ALL, beta=0.2)
    if sf:
        for k in ('train_beta', 'train_V_embed', 'train_word_embed'):
            flags.pop(k)
    args = synth.make_args(**flags)
    f = synth.make_decompose_factors(seed, V, S, R, C, D, lang_frac=0.5, dtype=np.float32)
    for k in ('S1', 'S2', 'wildcard_mat'):
        f[k] = (f[k] * shrink).astype(np.float32)
    x, lens, lab = synth.make_batch(seed + 1, B, L, V, C)
    rs = np.random.RandomState(seed + 2)
    pm = np.eye(C + 1) + 0.1 * rs.randn(C + 1, C + 1) if args.use_priority else None
    torch.manual_seed(seed)
    common = dict(S1=f['S1'], S2=f['S2'], C_output_mat=f['C_output_mat'], wildcard_mat=f['wildcard_mat'],
                  wildcard_output_vector=f['wildcard_output_vector'], final_vector=f['final_vector'],
                  start_vector=f['start_vector'], priority_mat=pm, args=args, o_idx=0)
    if sf:
        m = r.FARNN_S_SF(**common)
    else:
        m = r.FARNN_S_D_W_I_S(V=f['V'], pretrained_word_embed=f['pretrained_word_embed'], **common)
    with torch.no_grad():
        if args.use_crf:
            m.crf.transitions.copy_(torch.from_numpy(synth.crf_transitions(seed, m.C)))
        if args.farnn:
            for n in ('Wss1', 'Wrs1', 'Wss2', 'Wrs2'):
                if hasattr(m, n):
                    getattr(m, n).mul_(0.05)
            m.bs1.fill_(0.3)
            if hasattr(m, 'bs2'):
                m.bs2.fill_(-0.1)
        if args.local_loss_func != 'CE1':
            m.wildcard_output_vector.add_(0.25)         # zero in the synthetic factors
    m = m.cuda()
    if tp is not None:
        m.train_precision = tp
    dense_v = (rs.randn(B, L, R) / np.sqrt(R)).astype(np.float32) if sf else None
    return m, args, x, lens, lab, dense_v


def _weight_gradient_products(m, args, lens, sf):
    """(P, Q, summed rows, has_y2) of every transposed GEMM the backward runs for this module's trained weights."""
    M = len(lens) * int(lens.max())
    table_rows = len(lens) * L if sf else V + 1
    prods = {'S1': (S, R, 2 * M, 0), 'S2': (S, R, 2 * M, 0)}
    if m.wildcard_mat.requires_grad:
        prods['wildcard_mat'] = (S, S, 2 * M, 0)
    if m.C_output_mat.requires_grad:
        prods['C_output_mat'] = (m.C_output_mat.shape[0], S, M, 1)
    for i in range(1, args.farnn + 1):
        prods['Wss%d' % i] = (S, S, 2 * M, 0)
        prods['Wrs%d' % i] = (R, S, table_rows, 0)
    if not sf and m.embed_r_generalized.requires_grad:
        prods['embed_r_generalized'] = (D, R, V + 1, 0)
    return prods


@pytest.mark.parametrize('name', list(TRAIN_CASES))
def test_training_gradients_on_tensor_core_backward_vs_fp64_oracle(name, capsys):
    """B = 141 (128 + 13), L = 31, S = 97, R = 45, D = 24, V = 4500: every weight gradient's transposed GEMM runs on
    tcgen05 (4371 rows for dC, 8742 for the state weights, 4501 for the token-side gate weights and dG; with C = 13 dC
    has 14 rows < 16 and stays on CUDA cores).  Odd S and R exercise the padded operand strides.

    The same step runs twice: weight-gradient GEMMs on tcgen05 (the default) and on the CUDA-core kernel.  Loss within
    1e-5 of the float64 oracle; every weight gradient of the two runs within 5e-6 of each other (what the tensor-core
    kernel alone adds); every trained gradient within 2e-5 max-norm relative of the oracle, or, where the fp32 backward
    with CUDA-core weight gradients is already further off at this small batch (relu kinks, cancellation), within
    that run's error + 5e-6."""
    from re2nn_seq_b200 import _lib, ops
    _need_tc()
    sf = TRAIN_CASES[name].get('sf', False)
    m, args, x, lens, lab, dense_v = _train_case(name, 61 + list(TRAIN_CASES).index(name))
    prods = _weight_gradient_products(m, args, lens, sf)
    for k, (P, Q, rows, y2) in prods.items():
        want = 'cuda' if min(P, Q) < 16 else 'tc'
        assert ops.gemm_tn_path(P, Q, rows, y2) == want, (k, P, Q, rows)
    assert name != 'f1_tanh_ce_c13' or ops.gemm_tn_path(*prods['C_output_mat']) == 'cuda'
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()   # noqa: E731
    grads, loss_errs, errs = {}, {}, {}
    try:
        for on in (0, 1):
            _lib.check(_lib.fn['re2nn_debug_set_tn_tc'](on), 'tn_tc')
            m.zero_grad(set_to_none=True)
            if sf:
                loss, _, _ = m(dev(dense_v), dev(lab), dev(lens), True)
            else:
                loss, _, _ = m.forward_local(dev(x), dev(lab), dev(lens), train=True)
            loss.backward()
            grads[on] = {k: v.grad.detach().clone() for k, v in m.named_parameters() if v.grad is not None}
            loss_errs[on], errs[on] = oracle_gradient_errors(m, args, x, lab, lens, loss.item(), dense_v=dense_v)
    finally:
        _lib.check(_lib.fn['re2nn_debug_set_tn_tc'](1), 'tn_tc')
    diffs = {k: ((grads[1][k] - grads[0][k]).abs().max() / grads[0][k].abs().max().clamp_min(1e-30)).item()
             for k in prods}                                   # the products are keyed by parameter name
    with capsys.disabled():
        print('\n%s: loss %.1e; gradients vs fp64 oracle (max-norm relative), tcgen05 / CUDA-core weight gradients: %s'
              % (name, loss_errs[1], ', '.join('%s %.2e / %.2e' % (k, errs[1][k], errs[0][k]) for k in sorted(errs[1]))))
        print('%s: tcgen05 vs CUDA-core weight gradients: %s' % (
            name, ', '.join('%s %.2e' % kv for kv in sorted(diffs.items()))))
    assert loss_errs[1] < 1e-5
    for k, d in diffs.items():
        assert d < 5e-6, '%s: tcgen05 vs CUDA cores %.3e' % (k, d)
    for k, e in errs[1].items():
        assert e < max(2e-5, errs[0][k] + 5e-6), '%s: %.3e (CUDA-core weight gradients: %.3e)' % (k, e, errs[0][k])


# Bounds of the CUDA-core BPTT test, from its measurements on a B200: every gradient within 1.8e-5 of the oracle except
# hT and wildcard_mat of the farnn = 0 CRF cases (2.4-3.3e-5: the same parameters the fp32 backward is furthest off on
# in the test above).  Bounds about 1.3-1.4x above that.
BPTT_CUDA_TOL = 2.5e-5
BPTT_CUDA_TOL_LOOSE = {'hT': 4.5e-5, 'wildcard_mat': 4.5e-5}


@pytest.mark.parametrize('name', list(TRAIN_CASES))
def test_training_gradients_on_cuda_core_bptt_vs_fp64_oracle(name, capsys):
    """The same eight training steps with the GEMMs of every BPTT step on the fp32 CUDA-core kernel instead of tcgen05
    (re2nn_debug_set_backward_tc(0), bench.py --backward-tc 0).  Loss within 1e-5 of the float64 oracle, every trained
    gradient within BPTT_CUDA_TOL max-norm relative of it (BPTT_CUDA_TOL_LOOSE for hT and wildcard_mat)."""
    from re2nn_seq_b200 import _lib
    sf = TRAIN_CASES[name].get('sf', False)
    m, args, x, lens, lab, dense_v = _train_case(name, 61 + list(TRAIN_CASES).index(name))
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()   # noqa: E731
    try:
        _lib.check(_lib.fn['re2nn_debug_set_backward_tc'](0), 'backward_tc')
        if sf:
            loss, _, _ = m(dev(dense_v), dev(lab), dev(lens), True)
        else:
            loss, _, _ = m.forward_local(dev(x), dev(lab), dev(lens), train=True)
        loss.backward()
        loss_err, errs = oracle_gradient_errors(m, args, x, lab, lens, loss.item(), dense_v=dense_v)
    finally:
        _lib.check(_lib.fn['re2nn_debug_set_backward_tc'](1), 'backward_tc')
    with capsys.disabled():
        print('\n%s: CUDA-core BPTT: loss %.1e; gradients vs fp64 oracle (max-norm relative): %s'
              % (name, loss_err, ', '.join('%s %.2e' % kv for kv in sorted(errs.items()))))
    assert loss_err < 1e-5
    for k, e in errs.items():
        assert e < BPTT_CUDA_TOL_LOOSE.get(k, BPTT_CUDA_TOL), '%s: %.3e' % (k, e)
