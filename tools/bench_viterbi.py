"""Viterbi kernel alone: time per launch for 1 / 2 sequences per warp at the cfg2 and cfg5 tag-set sizes."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import __graft_entry__ as ge
ge.build()
from re2nn_seq_b200 import ops, _lib, synth

for name, B, L, T, fixed in (('cfg2', 4096, 35, 75, False), ('cfg5/4', 16384, 64, 131, True)):
    rs = np.random.RandomState(0)
    feats = torch.from_numpy(rs.randn(B, L, T).astype(np.float32)).cuda()
    lens = np.full(B, L, np.int64) if fixed else np.sort(rs.randint(L // 3, L + 1, size=B))[::-1].copy()
    lt = torch.from_numpy(lens).cuda()
    offs = torch.from_numpy(np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int64)).cuda()
    tr = torch.from_numpy(synth.crf_transitions(0, T)).cuda()
    N = int(lens.sum())
    ref = None
    for ns in (1, 2):
        _lib.check(_lib.fn['re2nn_debug_set_viterbi_seqs'](ns), 'ns')
        for _ in range(2):
            flat, _ = ops.crf_viterbi(feats, tr, lt, offs, N, want_flat=True, want_padded=False)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            flat, _ = ops.crf_viterbi(feats, tr, lt, offs, N, want_flat=True, want_padded=False)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 5
        if ref is None:
            ref = flat.clone()
        print('%s B=%d L=%d T=%d ns=%d: %.3f ms  %.2f T pairs/s  same=%s' % (name, B, L, T, ns, ms, N * T * T / ms / 1e9,
                                                                         bool((flat == ref).all())))
_lib.check(_lib.fn['re2nn_debug_set_viterbi_seqs'](0), 'ns')
