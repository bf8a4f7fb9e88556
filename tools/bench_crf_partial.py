"""The partial-annotation CRF loss (forward + backward, half of the tokens unknown) against the supervised CRF loss
(forward + backward), per call, at the cfg2 (B = 4096, L = 35 ragged, T = 75) and cfg5/4 (B = 16384, L = 64, T = 131)
shapes.  CUDA events around 10 calls after 3 warm-up calls.  cfg2's features (43 MB) fit the 126 MB L2, so repeated
calls read them from there; cfg5/4's (550 MB) do not."""
import os
import subprocess
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import __graft_entry__ as ge
ge.build()
from re2nn_seq_b200 import ops, synth
from re2nn_seq_b200.crf import partial_allowed

print(torch.cuda.get_device_name(0))
print(subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv'], capture_output=True,
                     text=True).stdout.strip())


def timed(f, reps=10, warm=3):
    for _ in range(warm):
        f()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        f()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


for name, B, L, T, fixed in (('cfg2', 4096, 35, 75, False), ('cfg5/4', 16384, 64, 131, True)):
    rs = np.random.RandomState(0)
    feats = torch.from_numpy(rs.randn(B, L, T).astype(np.float32)).cuda()
    lens = np.full(B, L, np.int64) if fixed else np.sort(rs.randint(L // 3, L + 1, size=B))[::-1].copy()
    lt = torch.from_numpy(lens).cuda()
    tags = rs.randint(0, T - 2, size=(B, L)).astype(np.int64)
    tg = torch.from_numpy(tags).cuda()
    hidden = np.where(rs.rand(B, L) < 0.5, -1, tags)
    allowed = partial_allowed(torch.from_numpy(hidden).cuda(), T, lengths=lt).contiguous()
    tr = torch.from_numpy(synth.crf_transitions(0, T)).cuda()
    g = torch.ones((), device='cuda')
    N = int(lens.sum())

    def nll():
        _, _, part = ops.crf_nll(feats, tr, lt, tg, save=True)
        ops.crf_nll_backward(feats, tr, lt, tg, part, g)

    def partial():
        _, _, (part, part_a) = ops.crf_partial_nll(feats, tr, lt, allowed, save=True)
        ops.crf_partial_nll_backward(feats, tr, lt, allowed, part, part_a, g)

    res = {'nll fwd': timed(lambda: ops.crf_nll(feats, tr, lt, tg, save=True)),
           'nll fwd+bwd': timed(nll),
           'partial fwd': timed(lambda: ops.crf_partial_nll(feats, tr, lt, allowed, save=True)),
           'partial fwd+bwd': timed(partial)}
    _, ps_s, _ = ops.crf_nll(feats, tr, lt, tg)
    _, ps_p, _ = ops.crf_partial_nll(feats, tr, lt, allowed)
    print('%s B=%d L=%d T=%d (%d tokens), half unknown: partial loss %.1f <= supervised %.1f: %s'
          % (name, B, L, T, N, ps_p.sum().item(), ps_s.sum().item(), bool((ps_p <= ps_s + 1e-3).all())))
    for k, ms in res.items():
        print('  %-16s %8.3f ms  %6.2f x supervised' % (k, ms, ms / res['nll fwd+bwd' if 'bwd' in k else 'nll fwd']))
