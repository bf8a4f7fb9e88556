"""Round-2 kernels under compute-sanitizer: tcgen05 weight-gradient GEMM (ragged split-K, P / Q off the tile grid, masked
dC), fused E3+E1 sweep, onehot cluster recurrence, batched vec-mat (FST family),
Viterbi with two sequences per warp, fused label-score operand."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
import numpy as np, torch
import re2nn_seq_b200 as r
from re2nn_seq_b200 import _lib, ops, synth
from test_gpu_parity import _random_decompose


def t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


for farnn in (0, 2):
    m, args, x, lens, lab = _random_decompose(3, 200, 80, 48, 10, 30, 700, 7, farnn=farnn, use_crf=1,
                                              update_nonlinear='tanh', beta=0.1, train_h0=1, train_hT=1)
    m.train_precision = 'auto'
    m.zero_grad(set_to_none=True)
    loss, _, _ = m.forward_local(t(x), t(lab), t(lens), train=True)
    loss.backward()
    torch.cuda.synchronize()
    print('train farnn', farnn, 'ok', float(loss), flush=True)

# fused label-score operand (per-step path) + Viterbi
m, args, x, lens, lab = _random_decompose(5, 200, 80, 48, 10, 30, 300, 7, farnn=0, use_crf=1, update_nonlinear='tanh', beta=0.1)
m.use_cuda_graph = False
m.precision = 'bf16'
_lib.check(_lib.fn['re2nn_debug_set_resident'](0), 'resident')
with torch.no_grad():
    m.forward_local(t(x), t(lab), t(lens), train=False)
_lib.check(_lib.fn['re2nn_debug_set_resident'](1), 'resident')
for ns in (1, 2):
    _lib.check(_lib.fn['re2nn_debug_set_viterbi_seqs'](ns), 'viterbi')
    with torch.no_grad():
        m.forward_local(t(x), t(lab), t(lens), train=False)
_lib.check(_lib.fn['re2nn_debug_set_viterbi_seqs'](0), 'viterbi')
torch.cuda.synchronize()
print('inference ok', flush=True)

# onehot: cluster of two CTAs per slice (small batch) and the plain kernel
args = synth.make_args(method='onehot', rand_constant=0.0)
a = synth.make_onehot_automaton(21, 60, 72, 9, dtype=np.float32)
oh = r.FARNN_S_O_I_S(a['language_tensor'], a['output_mat'], a['wildcard_mat'], a['output_wildcard_vector'],
                     a['final_vector'], a['start_vector'], None, args, 0, False)
for B in (8, 600):
    xx, ll, yy = synth.make_batch(7, B, 9, 60, 9)
    with torch.no_grad():
        oh.forward_local(torch.from_numpy(xx), torch.from_numpy(yy), torch.from_numpy(ll), train=False)
torch.cuda.synchronize()
print('onehot ok', flush=True)

# batched vec-mat (FST family primitive)
h = torch.rand(33, 40, device='cuda')
T = torch.rand(33, 40, 40, device='cuda')
for tr in (False, True):
    for mx in (False, True):
        ops.batched_vecmat(h, T, transposed=tr, max_semiring=mx)
torch.cuda.synchronize()
print('vecmat ok', flush=True)
