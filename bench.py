#!/usr/bin/env python
"""bench.py -- benchmark of the RE2NN-SEQ transducer hot path on B200.

Metric (BASELINE.json): valid token positions / second of decompose i-FST inference + Viterbi decode.
The headline line is BASELINE.json configs[1] ("cfg2": V=12000, C=72, S=300, R=200, D=100, len<=35, B=4096, tanh
update, CRF, beta=0.1) in the parity-grade `auto` precision; the other BASELINE configurations ride on the same JSON
line under "extra" (each with its own value / roofline / tag-mismatch count / clocks), measured the same way at
every N:
    cfg2_gated               cfg2 with farnn = 2 (update + reset gates: what every published .res configuration uses)
    cfg4                     configs[3]: ATIS-ZH-shaped long recurrence (S=512, R=256, len<=128), B=4096
    cfg5_bf16, cfg5_parity   configs[4] north-star target: S=1024, R=512, C=128, B=65536, len=64 (bf16 with its
                             stated bound, and the parity-grade mode)
    cfg3_train               configs[2]: training step (fwd + CRF loss + bwd + gradient all-reduce), B=1024 per GPU
    cfg1_onehot, cfg5_onehot configs[0] / configs[4] exact ("onehot") i-FST: HBM-bound gather recurrence
One "step" = one forward_local over one synthetic batch (scores + decode for every sequence); training: one
fwd + loss + bwd + all-reduce.  N>1: one process per GPU (torchrun), every rank runs its own batch of the same
shape (weak scaling; sequences are independent, the only collective is the training gradient all-reduce).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--legs cfg2,cfg5_bf16,...]
                  [--dump-outputs DIR]

Both timed regions of every leg run exactly K steps: from inputs resident in HBM, then end to end from pinned host
buffers (the roofline / kernel-alone passes that follow are separate).  The inputs are seeded, so the same
arguments give the same inputs on every run; `--dump-outputs DIR` writes what the last timed step of each leg returned
to its caller (see OutputDump) so that two builds can be compared output for output.

`--impl reference` times the UNMODIFIED reference classes (oracle/_ref, vendored by oracle/make_ref.py) on the host
cores; it never imports the product package.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'token positions/sec (decompose i-FST inference + Viterbi)'
UNIT = 'tokens/s'
METRIC_TRAIN = 'token positions/sec (decompose i-FST training step: fwd + CRF loss + bwd + grad all-reduce)'
ALL_LEGS = ['cfg2', 'cfg2_gated', 'cfg4', 'cfg5_bf16', 'cfg5_parity', 'cfg3_train', 'cfg1_onehot', 'cfg5_onehot']


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--legs', default=','.join(ALL_LEGS),
                    help='comma list; the first decompose-inference leg named is the headline (default: all, cfg2 first)')
    ap.add_argument('--config', default=None, help='shorthand: headline leg only, on this synth.CONFIGS entry')
    ap.add_argument('--precision', default=os.environ.get('RE2NN_PRECISION', 'auto'))
    ap.add_argument('--farnn', type=int, default=0)
    ap.add_argument('--batch', type=int, default=0, help='override B of the headline leg')
    ap.add_argument('--mode', default='infer', choices=['infer', 'train'], help='train: headline = the cfg3 training step')
    ap.add_argument('--train-precision', default='auto', help='forward GEMMs of the training leg: auto|fp32|tf32x3|fp16x3')
    ap.add_argument('--cta-group', type=int, default=0, help='debug: force the tcgen05 CTA-group size (0 = cost model)')
    ap.add_argument('--resident', type=int, default=1, help='debug: 0 = one launch per step GEMM instead of the resident kernel')
    ap.add_argument('--backward-tc', type=int, default=1, help='debug: 0 = BPTT step GEMMs on fp32 CUDA cores')
    ap.add_argument('--infer-chunks', type=int, default=4, help='streams the graphed inference body forks into (1 = single stream)')
    ap.add_argument('--cpu-sample', type=int, default=4096, help='sequences of the batch the CPU reference runs (baseline + tag check)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', default=None, metavar='DIR',
                    help='write the outputs of the last timed step of every leg as DIR/<leg>_<name>.npy')
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    return a


def flops_per_position(S, R, D, Cp, farnn):
    """SURVEY.md section 8d: F = 8SR + 4S^2 + 2DR + 2SC' (+ 8S^2 + 8SR for farnn=2)."""
    f = 8 * S * R + 4 * S * S + 2 * D * R + 2 * S * Cp
    if farnn == 2:
        f += 8 * S * S + 8 * S * R
    elif farnn == 1:
        f += 4 * S * S + 4 * S * R
    return f


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        return {}


def load_traffic(key):
    try:
        return json.load(open(os.path.join(ROOT, 'profiles', 'r02_traffic.json'))).get(key)
    except Exception:
        return None


class ClockSampler:
    """Samples SM clock and throttle reasons through NVML every 10 ms while a timed region runs."""
    REASONS = {0x8: 'hw_slowdown', 0x40: 'hw_thermal_slowdown', 0x20: 'sw_thermal_slowdown', 0x4: 'sw_power_cap'}

    def __init__(self, index):
        self.index, self.sm, self.bits, self.stop_flag, self.th, self.max = index, [], 0, False, None, None
        self.power = []

    def _loop(self):
        nv, h = self.nv, self.h
        try:
            while not self.stop_flag:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                try:
                    self.bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
                except Exception:
                    try:
                        self.bits |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                    except Exception:
                        pass
                try:
                    self.power.append(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)
                except Exception:
                    pass
                time.sleep(0.01)
        except Exception as e:   # noqa
            self.err = str(e)

    def start(self):
        # import / nvmlInit / handle lookup HERE, before the timed region: done inside the sampling thread they held the
        # import lock and the GIL for 50-500 ms while the first timed steps were being launched (seen as a single
        # outlier step in the launch-bound training leg)
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get('CUDA_VISIBLE_DEVICES')
            idx = self.index
            if vis:
                try:
                    idx = int(vis.split(',')[self.index])
                except Exception:
                    pass
            self.nv, self.h = nv, nv.nvmlDeviceGetHandleByIndex(idx)
            self.max = float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM))
        except Exception as e:   # noqa
            self.err = str(e)
            return self
        self.th = threading.Thread(target=self._loop, daemon=True)
        self.th.start()
        return self

    def stop(self):
        self.stop_flag = True
        if self.th:
            self.th.join(timeout=2)
        reasons = sorted(n for b, n in self.REASONS.items() if self.bits & b)
        return {'sm_mhz': float(np.median(self.sm)) if self.sm else None, 'sm_max_mhz': self.max,
                'samples': len(self.sm), 'power_w_max': max(self.power) if self.power else None, 'reasons': reasons}


# ---- the reference on the host cores ------------------------------------------------------------------------------
def reference_cpu(cfg, farnn, x, lens, lab, sample, repeats, synth=None):
    """Predictions and tokens/s of the vendored, unmodified reference FARNN_S_D_W_I_S on the first `sample` sequences
    (all host threads).  Falls back to the numpy port when oracle/_ref is absent.  -> dict."""
    import torch
    from oracle import ref_runner as rr
    torch.set_num_threads(os.cpu_count())
    xs, ls, ys = x[:sample], lens[:sample], lab[:sample]
    toks = float(ls.sum())
    try:
        synth = synth or rr.load_synth()
        m, _, _ = rr.build_decompose(synth, cfg, farnn=farnn)
        pred, best, times = rr.run_forward_local(m, xs, ys, ls, repeats=repeats)
        return {'kind': 'reference', 'pred': pred, 'best_s': best, 'times': times, 'tokens': toks, 'cores': os.cpu_count(),
                'what': 'unmodified reference FARNN_S_D_W_I_S.forward_local(train=False) (oracle/_ref, sha256-pinned), torch CPU fp32'}
    except RuntimeError as e:
        why = str(e)
    # port fallback: parameters through the reference-identical host constructor of the product package
    import re2nn_seq_b200 as r
    from re2nn_seq_b200 import synth as ps
    from oracle import re2nn_oracle as orc
    c = dict(ps.CONFIGS[cfg])
    args = ps.make_args(farnn=farnn, use_crf=1, update_nonlinear='tanh', beta=0.1, sigmoid_exponent=5, bias_init=5.0)
    f = ps.make_decompose_factors(0, c['V'], c['S'], c['R'], c['C'], c['D'], dtype=np.float32)
    torch.manual_seed(0)
    mod = r.FARNN_S_D_W_I_S(args=args, o_idx=0, **f)
    with torch.no_grad():
        mod.crf.transitions.copy_(torch.from_numpy(ps.crf_transitions(0, mod.C)))
    p = oracle_params_from_module(mod)
    Lm = int(ls.max())
    times, pred = [], None
    for _ in range(repeats):
        t0 = time.perf_counter()
        _, pred, _, _ = orc.decompose_forward_local(p, xs[:, :Lm], ys[:, :Lm], ls, args, 0, train=False)
        times.append(time.perf_counter() - t0)
    return {'kind': 'port', 'pred': np.asarray(pred), 'best_s': min(times), 'times': times, 'tokens': toks,
            'cores': os.cpu_count(), 'what': 'oracle/re2nn_oracle.py numpy port (oracle/_ref unavailable: %s)' % why}


def oracle_params_from_module(m):
    rename = {'embedding.weight': 'embedding', 'crf.transitions': 'crf_transitions',
              'priority_layer.priority_mat': 'priority_mat', 'priority_layer.priority_bias': 'priority_bias'}
    return {rename.get(k, k): v.detach().cpu().numpy() for k, v in m.state_dict().items()}


def run_reference(a):
    """--impl reference: the reference's own CPU implementation of the headline path, all host threads, on a bounded
    sample of the same batch.  Rank 0 only; the product package is never imported."""
    if int(os.environ.get('RANK', '0')) != 0:
        return
    from oracle import ref_runner as rr
    synth = rr.load_synth()
    cfg = a.config or 'cfg2'
    c = dict(synth.CONFIGS[cfg])
    x, lens, lab = synth.make_batch(1000, c['B'], c['Lmax'], c['V'], c['C'], fixed_len=c.get('fixed_len', False))
    sample = min(a.cpu_sample, c['B'])
    for _ in range(min(a.warmup, 1)):
        reference_cpu(cfg, a.farnn, x, lens, lab, sample, 1, synth)
    res = reference_cpu(cfg, a.farnn, x, lens, lab, sample, a.steps, synth)
    ms = 1e3 * float(np.mean(res['times']))
    val = res['tokens'] / (ms / 1e3)
    assert 're2nn_seq_b200' not in sys.modules or res['kind'] == 'port'
    line = {'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': UNIT, 'n_gpus': a.gpus, 'steps': a.steps,
            'warmup': a.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': '%s decompose i-FST inference + Viterbi (V=%d,C=%d,S=%d,R=%d,len<=%d)'
                                   % (cfg, c['V'], c['C'], c['S'], c['R'], c['Lmax']),
                       'sample': 'first %d of B=%d sequences per step' % (sample, c['B'])},
            'cpu_baseline': {'value': val, 'unit': UNIT, 'cores': res['cores'], 'kind': res['kind'],
                             'sample': '%s on the first %d sequences of the batch' % (res['what'], sample)},
            'e2e': {'value': val, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line))


# ---- timing helpers ---------------------------------------------------------------------------------------------------
class Ctx:
    def __init__(self, a):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.a = torch, dist, a
        self.rank = int(os.environ.get('RANK', '0'))
        self.world = int(os.environ.get('WORLD_SIZE', '1'))
        self.local = int(os.environ.get('LOCAL_RANK', '0'))
        self.flush = None
        self.peaks = load_peaks()
        self.dump = OutputDump(a.dump_outputs, self.rank == 0)
        self.last_output = None

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, fn, steps):
        """K steps, each bracketed by CUDA events on the current stream, an L2 flush (256 MB write) before each, a
        barrier + synchronize on both sides.  -> per-step ms list of this rank; what the last step returned is kept in
        self.last_output (earlier steps' results are dropped as they come, as a caller looping over batches would)."""
        torch = self.torch
        if self.flush is None:
            self.flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device='cuda')   # > 126 MB L2
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        self.last_output = None
        self.barrier()
        for i in range(steps):
            self.flush.zero_()
            ev[i][0].record()
            out = fn()
            ev[i][1].record()
            if i + 1 < steps:
                out = None
        self.barrier()
        self.last_output = out
        return [s.elapsed_time(e) for s, e in ev]

    def reduce(self, total_ms, tokens):
        """max over ranks of the summed time, sum over ranks of the tokens."""
        torch = self.torch
        t = torch.tensor([total_ms], dtype=torch.float64, device='cuda')
        k = torch.tensor([float(tokens)], dtype=torch.float64, device='cuda')
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            self.dist.all_reduce(k, op=self.dist.ReduceOp.SUM)
        return t.item(), k.item()


def stats(ms):
    return {'min': float(np.min(ms)), 'median': float(np.median(ms)), 'max': float(np.max(ms)), 'argmax': int(np.argmax(ms))}


class OutputDump:
    """--dump-outputs DIR: the arrays the last timed step of a leg handed to its caller, one DIR/<leg>_<name>.npy each,
    float64 where the output is float64 and float32 otherwise (tags and labels are small integers, exact in float32).
    An array of more than CAP elements is stored as a fixed sample of its flattened values: the positions
    np.sort(np.random.RandomState(0).choice(size, CAP, replace=False)).  With CAP, the default legs write about 14 MB.
    Every rank counts the bytes (the legs have the same shapes on every rank) and only rank 0 writes, so going over
    LIMIT stops all ranks at the same leg instead of leaving the others waiting in a collective."""
    CAP = 1 << 19
    LIMIT = 64 << 20

    def __init__(self, path, writer):
        self.path, self.writer, self.bytes = path, writer, 0
        if path and writer:
            os.makedirs(path, exist_ok=True)

    def write(self, leg, arrays):
        if not self.path:
            return
        for name, t in arrays.items():
            if t is None:
                continue
            a = t.detach().cpu().numpy() if hasattr(t, 'detach') else np.asarray(t)
            a = a.astype(np.float64 if a.dtype == np.float64 else np.float32)
            if a.size > self.CAP:
                a = a.reshape(-1)[np.sort(np.random.RandomState(0).choice(a.size, self.CAP, replace=False))]
            self.bytes += a.nbytes
            if self.bytes > self.LIMIT:
                raise SystemExit('--dump-outputs: the outputs exceed %d MB' % (self.LIMIT >> 20))
            if self.writer:
                np.save(os.path.join(self.path, '%s_%s.npy' % (leg, name)), a)


# ---- decompose inference leg ------------------------------------------------------------------------------------------
def leg_decompose(ctx, name, cfg, precision, farnn, steps, warmup, batch=0, ref_sample=0, ref_repeats=1,
                  want_cpu_baseline=False):
    torch, a = ctx.torch, ctx.a
    import re2nn_seq_b200 as r
    from re2nn_seq_b200 import ops, synth
    c = dict(synth.CONFIGS[cfg])
    if batch:
        c['B'] = batch
    args = synth.make_args(farnn=farnn, use_crf=c.get('use_crf', 1), update_nonlinear=c.get('update_nonlinear', 'tanh'),
                           beta=c.get('beta', 0.1), sigmoid_exponent=5, bias_init=5.0)
    f = synth.make_decompose_factors(0, c['V'], c['S'], c['R'], c['C'], c['D'], dtype=np.float32)
    x, lens, lab = synth.make_batch(1000 + ctx.rank, c['B'], c['Lmax'], c['V'], c['C'], fixed_len=c.get('fixed_len', False))
    torch.manual_seed(0)
    m = r.FARNN_S_D_W_I_S(args=args, o_idx=0, **f)
    with torch.no_grad():
        m.crf.transitions.copy_(torch.from_numpy(synth.crf_transitions(0, m.C)))
    m.infer_chunks = a.infer_chunks
    m.precision = precision
    with torch.no_grad():
        prec = m._resolved_precision()
    m.precision = prec
    m = m.cuda().eval()
    n_tok = int(lens.sum())
    S, R, D, Cp = c['S'], c['R'], c['D'], m.C
    xd, ld, yd = torch.from_numpy(x).cuda(), torch.from_numpy(lens).cuda(), torch.from_numpy(lab).cuda()
    xh, lh, yh = torch.from_numpy(x).pin_memory(), torch.from_numpy(lens).pin_memory(), torch.from_numpy(lab).pin_memory()
    pred_host = torch.empty((n_tok,), dtype=torch.int64).pin_memory()

    def step_device():
        with torch.no_grad():
            return m.forward_local(xd, yd, ld, train=False)

    def step_e2e():
        xg, lg, yg = xh.cuda(non_blocking=True), lh.cuda(non_blocking=True), yh.cuda(non_blocking=True)
        with torch.no_grad():
            _, pred, _ = m.forward_local(xg, yg, lg, train=False)
        pred_host.copy_(pred, non_blocking=True)

    for _ in range(max(warmup, 3)):
        step_device()
    torch.cuda.synchronize()

    # ---- parity of exactly what is timed: decoded tags of this batch in this mode (graph, chunk streams) ----------
    with torch.no_grad():
        _, p_fast, _ = m.forward_local(xd, yd, ld, train=False)
        p_fast = p_fast.clone()
    mism_fp32 = None
    if prec != 'fp32':
        with torch.no_grad():
            m.precision = 'fp32'
            _, p_ref, _ = m.forward_local(xd, yd, ld, train=False)
            m.precision = prec
        mism_fp32 = int((p_fast != p_ref).sum().item())
        del p_ref
    ref = None
    mism_ref = None
    if ref_sample and ctx.rank == 0:
        ref = reference_cpu(cfg, farnn, x, lens, lab, min(ref_sample, c['B']), ref_repeats)
        n_ref = len(ref['pred'])
        mism_ref = int((p_fast[:n_ref].cpu().numpy() != ref['pred']).sum())

    # ---- timed region 1: inputs resident in HBM ----------------------------------------------------------------------
    sampler = ClockSampler(ctx.local).start()
    l0 = ops.launches()
    ms1 = ctx.timed(step_device, steps)
    launches_total = ops.launches() - l0
    loss_o, pred_o, true_o = ctx.last_output
    ctx.dump.write(name, {'loss': loss_o, 'pred': pred_o, 'true': true_o})
    del loss_o, pred_o, true_o
    ctx.last_output = None

    # ---- roofline pass: the SAME configuration (CUDA graph, chunk streams) with every recurrence launch bracketed by
    # CUDA events recorded inside the library on the launching stream (external event nodes inside the graph) ---------
    ops.profile_enable(True)
    ops.profile_read()
    for _ in range(3):          # lets the graph be re-captured with the event nodes in it (second sighting)
        step_device()
    torch.cuda.synchronize()
    graphed = bool(getattr(m, '_graphs', None))
    resident = ops.recurrence_is_resident(S, R, farnn, prec)
    dom_cls = 3 if resident else 2
    prof_steps = max(3, min(steps, 10))
    dom_ms, dom_n, cls_ms = [], 0, [0.0, 0.0, 0.0, 0.0]
    evp = []
    for _ in range(prof_steps):
        if not graphed:
            ops.profile_read()                      # eager: forget the previous step's pairs
        ctx.flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step_device()
        e1.record()
        torch.cuda.synchronize()
        evp.append(e0.elapsed_time(e1))
        for cls in range(4):
            iv = ops.profile_intervals(cls)
            if not iv:
                continue
            if cls == 3:
                # chunk streams run their resident launches concurrently: time = union of the intervals
                cls_ms[cls] += max(e for _, e in iv) - min(s for s, _ in iv)
            else:
                cls_ms[cls] += sum(e - s for s, e in iv)
            if cls == dom_cls:
                dom_n = len(iv)
                dom_ms.append((max(e for _, e in iv) - min(s for s, _ in iv)) if cls == 3 else float(np.mean([e - s for s, e in iv])))
    ops.profile_read()
    ops.profile_enable(False)
    clocks = sampler.stop()
    if hasattr(m, 'invalidate_caches'):
        m._graphs, m._graph_seen = {}, {}           # drop the profiled capture

    # ---- timed region 2: end to end from pinned host buffers ---------------------------------------------------------
    for _ in range(3):
        step_e2e()
    ms2 = ctx.timed(step_e2e, steps)

    total1, all_tok = ctx.reduce(sum(ms1), n_tok)
    total2, _ = ctx.reduce(sum(ms2), n_tok)
    ms_step = total1 / steps
    value = all_tok / (ms_step / 1e3)
    e2e = all_tok / (total2 / steps / 1e3)
    peak_tf = ctx.peaks.get('bf16_tflops_sustained') or 1400.0
    peak_src = 'MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside the step), of measured' if ctx.peaks else \
        'fallback 1.4 PFLOP/s sustained (B200_PROFILING.md), of fallback'
    rec_flops_pos = 2.0 * (2.0 * S * R + 2.0 * (R + S) * S + 2.0 * S * S * farnn)      # both directions, per valid position
    if resident:
        dom_name = 'tc_resident_kernel: all steps of both directions, G1 + G2 + fused epilogues (%s); %d launch(es) per step on ' \
                   'forked chunk streams, time = union of their intervals inside the replayed graph' % (prec, dom_n)
        dom_flops = n_tok * rec_flops_pos
    elif farnn == 0 and graphed is not None and ops.recurrence_fuses(S, R, farnn, prec) and getattr(m, 'use_cuda_graph', True):
        dom_name = 'tc_gemm_kernel<EpiH>: step GEMM2 [Q | Hbar] @ [S^T ; W] + state epilogue, ONE direction per launch (%s; the ' \
                   'forward direction writes the fused alpha*beta label-score operand)' % prec
        dom_flops = 2.0 * c['B'] * S * (R + S)
    else:
        dom_name = 'tc_gemm_kernel<EpiH>: step GEMM2 [Q | Hbar] @ [S^T ; W] + state epilogue, both directions per launch (%s)' % prec
        dom_flops = 2 * 2.0 * c['B'] * S * (R + S)
    dms = float(np.mean(dom_ms)) if dom_ms else 0.0
    achieved = dom_flops / (dms * 1e-3) / 1e12 if dms > 0 else 0.0
    prof_step_ms = float(np.mean(evp))
    rec_ms = (cls_ms[3] if resident else (cls_ms[0] + cls_ms[1] + cls_ms[2])) / prof_steps
    out = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': ctx.world, 'steps': steps, 'warmup': max(warmup, 3),
        'ms_per_step': ms_step, 'ms_per_step_stats': stats(ms1), 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': {'fp32': 'f32', 'bf16': 'bf16', 'tf32x3': 'tf32x3', 'fp16x3': 'fp16x3'}[prec], 'data': 'synthetic',
        'config': {'workload': '%s decompose i-FST inference + Viterbi (V=%d,C=%d,S=%d,R=%d,D=%d,len<=%d,B=%d per GPU)'
                               % (cfg, c['V'], c['C'], S, R, D, c['Lmax'], c['B']),
                   'mode': 'infer', 'farnn': farnn, 'precision': prec, 'tokens_per_step_per_gpu': n_tok,
                   'tag_mismatches_vs_fp32_path': mism_fp32,
                   'tag_mismatch_rate_vs_fp32_path': (mism_fp32 / n_tok) if mism_fp32 is not None else None,
                   'tag_mismatches_vs_reference_sample': mism_ref,
                   'reference_sample': ('%s, first %d sequences = %d tokens' % (ref['what'], min(ref_sample, c['B']), len(ref['pred'])))
                   if ref else None,
                   'l2': 'flushed between timed iterations (256 MB write)',
                   'cuda_graph': graphed, 'resident_kernel': bool(resident),
                   'whole_step_tflops': value / ctx.world * flops_per_position(S, R, D, Cp, farnn) / 1e12,
                   'whole_step_frac_of_peak': value / ctx.world * flops_per_position(S, R, D, Cp, farnn) / 1e12 / peak_tf,
                   'recurrence_tflops': (n_tok * rec_flops_pos / (rec_ms * 1e-3) / 1e12) if rec_ms > 0 else None},
        'roofline': {'bound': 'tensor', 'kernel': dom_name, 'achieved': achieved, 'peak': peak_tf, 'unit': 'TFLOP/s',
                     'frac': achieved / peak_tf, 'traffic': load_traffic('%s_%s' % (cfg, prec)), 'peak_source': peak_src,
                     'launches_per_step': dom_n, 'avg_launch_ms': dms,
                     'algorithmic_flops_per_launch': dom_flops,
                     'measured': 'CUDA events around the launch on its own stream, inside the timed configuration%s'
                                 % (' (external event nodes of the replayed CUDA graph)' if graphed else ''),
                     'kernel_share_of_step': (dms * (dom_n if not resident else 1)) / prof_step_ms if prof_step_ms > 0 else None,
                     'profiled_ms_per_step': prof_step_ms,
                     'class_ms_per_step': {'gate': cls_ms[0] / prof_steps, 'gemm1': cls_ms[1] / prof_steps,
                                           'gemm2': cls_ms[2] / prof_steps, 'resident': cls_ms[3] / prof_steps}},
        'e2e': {'value': e2e, 'unit': UNIT, 'ms_per_step': total2 / steps,
                'h2d_bytes_per_step': int(xh.numel() * 8 + lh.numel() * 8 + yh.numel() * 8), 'd2h_bytes_per_step': int(n_tok * 8)},
        'gpu_launches': int(launches_total), 'gpu_launches_per_step': int(launches_total // steps), 'clocks': clocks,
    }
    if want_cpu_baseline and ref is not None:
        out['cpu_baseline'] = {'value': ref['tokens'] / float(np.mean(ref['times'])), 'unit': UNIT, 'cores': ref['cores'],
                               'kind': ref['kind'],
                               'sample': '%s on the first %d of %d sequences (%d tokens), mean of %d passes, %.2f s of CPU work'
                                         % (ref['what'], min(ref_sample, c['B']), c['B'], int(ref['tokens']), len(ref['times']),
                                            sum(ref['times']))}
    del m, xd, ld, yd
    torch.cuda.empty_cache()
    return out


# ---- training leg (configs[2]) ------------------------------------------------------------------------------------------
def leg_train(ctx, cfg, farnn, steps, warmup):
    torch, a = ctx.torch, ctx.a
    import re2nn_seq_b200 as r
    from re2nn_seq_b200 import dist as rd, ops, synth
    c = dict(synth.CONFIGS[cfg])
    args = synth.make_args(farnn=farnn, use_crf=1, update_nonlinear='tanh', beta=0.1, sigmoid_exponent=5, bias_init=5.0)
    f = synth.make_decompose_factors(0, c['V'], c['S'], c['R'], c['C'], c['D'], dtype=np.float32)
    x, lens, lab = synth.make_batch(1000 + ctx.rank, c['B'], c['Lmax'], c['V'], c['C'])
    torch.manual_seed(0)
    m = r.FARNN_S_D_W_I_S(args=args, o_idx=0, **f)
    with torch.no_grad():
        m.crf.transitions.copy_(torch.from_numpy(synth.crf_transitions(0, m.C)))
    m = m.cuda().train()
    m.train_precision = a.train_precision
    prec = m._resolved_precision()
    bucket = rd.GradBucket(m)
    n_tok = int(lens.sum())
    xd, ld, yd = torch.from_numpy(x).cuda(), torch.from_numpy(lens).cuda(), torch.from_numpy(lab).cuda()
    xh, lh, yh = torch.from_numpy(x).pin_memory(), torch.from_numpy(lens).pin_memory(), torch.from_numpy(lab).pin_memory()
    loss_host = torch.empty((), dtype=torch.float32).pin_memory()

    def train_step(xg, yg, lg):
        bucket.zero_grad()
        loss, pred, true = m.forward_local(xg, yg, lg, train=True)
        loss.backward()
        bucket.all_reduce()                # one all-reduce(SUM) of the flat gradient bucket (NCCL when N>1)
        return loss, pred, true

    def step_device():
        return train_step(xd, yd, ld)

    def step_e2e():
        loss, _, _ = train_step(xh.cuda(non_blocking=True), yh.cuda(non_blocking=True), lh.cuda(non_blocking=True))
        loss_host.copy_(loss.detach(), non_blocking=True)

    for _ in range(max(warmup, 3)):
        step_device()
    torch.cuda.synchronize()
    sampler = ClockSampler(ctx.local).start()
    l0 = ops.launches()
    ms1 = ctx.timed(step_device, steps)
    launches_total = ops.launches() - l0
    clocks = sampler.stop()
    loss_o, pred_o, true_o = ctx.last_output           # the gradients of this step are still in the bucket
    ctx.dump.write('%s_train' % cfg, dict({'loss': loss_o, 'pred': pred_o, 'true': true_o},
                                          **{'grad.' + k: v.grad for k, v in m.named_parameters() if v.grad is not None}))
    del loss_o, pred_o, true_o
    ctx.last_output = None
    for _ in range(2):
        step_e2e()
    ms2 = ctx.timed(step_e2e, steps)
    total1, all_tok = ctx.reduce(sum(ms1), n_tok)
    total2, _ = ctx.reduce(sum(ms2), n_tok)
    ms_step = total1 / steps
    value = all_tok / (ms_step / 1e3)
    S, R, D, Cp = c['S'], c['R'], c['D'], m.C
    peak_tf = ctx.peaks.get('bf16_tflops_sustained') or 1400.0
    fl = 3.0 * flops_per_position(S, R, D, Cp, farnn)          # fwd + dX + dW (SURVEY section 8d)
    out = {'metric': METRIC_TRAIN, 'value': value, 'unit': UNIT, 'n_gpus': ctx.world, 'steps': steps, 'ms_per_step': ms_step,
           'ms_per_step_stats': stats(ms1), 'scaling': 'weak',
           'dtype': {'fp32': 'f32', 'tf32x3': 'tf32x3', 'fp16x3': 'fp16x3'}.get(prec, prec),
           'config': {'workload': '%s decompose i-FST training step: fwd + CRF loss + bwd + grad all-reduce + Viterbi '
                                  '(V=%d,C=%d,S=%d,R=%d,len<=%d,B=%d per GPU)' % (cfg, c['V'], c['C'], S, R, c['Lmax'], c['B']),
                      'forward_precision': prec, 'tokens_per_step_per_gpu': n_tok, 'grad_bucket_bytes': bucket.total * 4,
                      'collective': 'all-reduce(SUM) of one flat fp32 gradient bucket inside the timed step' if ctx.world > 1 else
                                    'none at N=1 (the gradients are written into the flat bucket all the same)',
                      'whole_step_tflops': value / ctx.world * fl / 1e12,
                      'whole_step_frac_of_peak': value / ctx.world * fl / 1e12 / peak_tf},
           'e2e': {'value': all_tok / (total2 / steps / 1e3), 'unit': UNIT,
                   'h2d_bytes_per_step': int(xh.numel() * 8 + lh.numel() * 8 + yh.numel() * 8), 'd2h_bytes_per_step': 4},
           'gpu_launches': int(launches_total), 'gpu_launches_per_step': int(launches_total // steps), 'clocks': clocks}
    del m, bucket
    torch.cuda.empty_cache()
    return out


# ---- onehot legs (configs[0] and the onehot half of configs[4]) -----------------------------------------------------
def leg_onehot(ctx, name, V, S, C, B, Lmax, fixed, steps, warmup, note):
    torch = ctx.torch
    import re2nn_seq_b200 as r
    from re2nn_seq_b200 import ops, synth
    args = synth.make_args(method='onehot', rand_constant=0.0)
    rs = np.random.RandomState(0)
    a8 = synth.make_onehot_automaton(0, 8, S, C, dtype=np.float32)          # small generator, tiled over the vocabulary
    lang = np.zeros((V + 1, S, S), dtype=np.float32)
    rows = rs.choice(V, size=max(1, V // 20), replace=False)                # 5 % language rows, the rest zero slices
    for i, rr_ in enumerate(rows):
        lang[rr_] = a8['language_tensor'][i % 8]
    x, lens, lab = synth.make_batch(1000 + ctx.rank, B, Lmax, V, C, fixed_len=fixed)
    m = r.FARNN_S_O_I_S(lang, a8['output_mat'], a8['wildcard_mat'], a8['output_wildcard_vector'], a8['final_vector'],
                        a8['start_vector'], None, args, 0, False)
    del lang
    xd, ld, yd = torch.from_numpy(x).cuda(), torch.from_numpy(lens).cuda(), torch.from_numpy(lab).cuda()
    xh, lh, yh = torch.from_numpy(x).pin_memory(), torch.from_numpy(lens).pin_memory(), torch.from_numpy(lab).pin_memory()
    n_tok = int(lens.sum())
    pred_host = torch.empty((n_tok,), dtype=torch.int64).pin_memory()

    def step_device():
        with torch.no_grad():
            return m.forward_local(xd, yd, ld, train=False)

    def step_e2e():
        with torch.no_grad():
            _, pred, _ = m.forward_local(xh.cuda(non_blocking=True), yh.cuda(non_blocking=True), lh.cuda(non_blocking=True), train=False)
        pred_host.copy_(pred, non_blocking=True)

    for _ in range(max(warmup, 3)):
        step_device()
    torch.cuda.synchronize()
    sampler = ClockSampler(ctx.local).start()
    l0 = ops.launches()
    ms1 = ctx.timed(step_device, steps)
    launches_total = ops.launches() - l0
    loss_o, pred_o, true_o = ctx.last_output
    ctx.dump.write(name, {'loss': loss_o, 'pred': pred_o, 'true': true_o})
    del loss_o, pred_o, true_o
    ctx.last_output = None
    # dominant kernel alone: CUDA events around the recurrence launch
    alone = []
    with torch.no_grad():
        for _ in range(min(steps, 5)):
            ctx.flush.zero_()
            t = m.time_recurrence(xd, ld) if hasattr(m, 'time_recurrence') else None
            if t is not None:
                alone.append(t)
    clocks = sampler.stop()
    for _ in range(2):
        step_e2e()
    ms2 = ctx.timed(step_e2e, steps)
    total1, all_tok = ctx.reduce(sum(ms1), n_tok)
    total2, _ = ctx.reduce(sum(ms2), n_tok)
    ms_step = total1 / steps
    peak = ctx.peaks.get('hbm_gbs') or 6650.0
    by_pos = 2.0 * S * S * 4 + 2 * S * 4 + (C + 1) * 4                     # SURVEY section 8d: dense algorithmic bytes
    k_ms = float(np.mean(alone)) if alone else ms_step
    ach = n_tok * (2.0 * S * S * 4 + 2 * S * 4) / (k_ms * 1e-3) / 1e9
    out = {'metric': 'token positions/sec (onehot i-FST inference + argmax decode)', 'value': all_tok / (ms_step / 1e3), 'unit': UNIT,
           'n_gpus': ctx.world, 'steps': steps, 'ms_per_step': ms_step, 'ms_per_step_stats': stats(ms1), 'scaling': 'weak', 'dtype': 'f32',
           'config': {'workload': '%s onehot i-FST inference (V=%d,C=%d,S=%d,len<=%d,B=%d per GPU)%s' % (name, V, C, S, Lmax, B, note),
                      'tokens_per_step_per_gpu': n_tok, 'whole_step_algorithmic_gbs': n_tok * by_pos / (ms_step * 1e-3) / 1e9},
           'roofline': {'bound': 'hbm', 'kernel': 'onehot_recurrence_kernel (both directions)', 'achieved': ach, 'peak': peak,
                        'unit': 'GB/s', 'frac': ach / peak, 'traffic': load_traffic(name), 'avg_launch_ms': k_ms,
                        'algorithmic_bytes_per_launch': n_tok * (2.0 * S * S * 4 + 2 * S * 4),
                        'peak_source': 'MEASURED_PEAKS.json hbm_gbs, of measured' if ctx.peaks else 'fallback 6.65 TB/s, of fallback'},
           'e2e': {'value': all_tok / (total2 / steps / 1e3), 'unit': UNIT,
                   'h2d_bytes_per_step': int(xh.numel() * 8 + lh.numel() * 8 + yh.numel() * 8), 'd2h_bytes_per_step': int(n_tok * 8)},
           'gpu_launches': int(launches_total), 'gpu_launches_per_step': int(launches_total // steps), 'clocks': clocks}
    del m
    torch.cuda.empty_cache()
    return out


def main():
    a = parse()
    if a.impl == 'reference':
        return run_reference(a)

    ctx = Ctx(a)
    torch, dist = ctx.torch, ctx.dist
    torch.cuda.set_device(ctx.local)
    if ctx.world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', ctx.local))
    import __graft_entry__ as ge
    if ctx.rank == 0:
        ge.build()
    if ctx.world > 1:
        dist.barrier()
    from re2nn_seq_b200 import _lib
    if not a.resident:
        _lib.check(_lib.fn['re2nn_debug_set_resident'](0), 'resident')
    if not a.backward_tc:
        _lib.check(_lib.fn['re2nn_debug_set_backward_tc'](0), 'backward_tc')
    if a.cta_group:
        _lib.check(_lib.fn['re2nn_debug_set_tc_cta_group'](a.cta_group), 'cta_group')

    legs = [s for s in a.legs.split(',') if s]
    if a.config or a.mode == 'train':
        legs = ['cfg3_train'] if a.mode == 'train' else ['custom']
    want_cpu = (not a.no_cpu_baseline) and ctx.world == 1
    ref_sample = 0 if a.no_cpu_baseline else a.cpu_sample
    results = {}
    for leg in legs:
        if leg == 'custom':
            results[leg] = leg_decompose(ctx, leg, a.config, a.precision, a.farnn, a.steps, a.warmup, batch=a.batch,
                                         ref_sample=ref_sample, ref_repeats=3, want_cpu_baseline=want_cpu)
        elif leg == 'cfg2':
            results[leg] = leg_decompose(ctx, leg, 'cfg2', a.precision, a.farnn, a.steps, a.warmup, batch=a.batch,
                                         ref_sample=ref_sample, ref_repeats=15, want_cpu_baseline=want_cpu)   # ~10-15 s of CPU work
        elif leg == 'cfg2_gated':          # farnn = 2: the configuration of every published .res file
            results[leg] = leg_decompose(ctx, leg, 'cfg2', a.precision, 2, a.steps, a.warmup, ref_sample=min(ref_sample, 256),
                                         ref_repeats=1)
        elif leg == 'cfg4':                # configs[3]: ATIS-ZH-shaped long recurrence (S=512, R=256, len<=128, B=4096)
            results[leg] = leg_decompose(ctx, leg, 'cfg4', a.precision, 0, a.steps, 3,
                                         ref_sample=min(ref_sample, 128), ref_repeats=1)
        elif leg in ('cfg5_bf16', 'cfg5_parity'):
            results[leg] = leg_decompose(ctx, leg, 'cfg5', 'bf16' if leg == 'cfg5_bf16' else 'auto', 0, a.steps, 3,
                                         ref_sample=min(ref_sample, 128), ref_repeats=1)
        elif leg == 'cfg3_train':
            results[leg] = leg_train(ctx, 'cfg3', a.farnn, a.steps, a.warmup)
        elif leg == 'cfg1_onehot':
            results[leg] = leg_onehot(ctx, leg, 900, 300, 127, 32, 46, False, a.steps, a.warmup, '')
        elif leg == 'cfg5_onehot':
            results[leg] = leg_onehot(ctx, leg, 900, 1024, 128, 1024, 64, True, a.steps, 3,
                                      ' -- B reduced from 65536: the dense gather moves 8*S^2 = 8.4 MB per position, '
                                      '65536 x 64 positions would be 35 PB per batch')
        else:
            raise SystemExit('unknown leg %r (known: %s)' % (leg, ', '.join(ALL_LEGS)))

    if ctx.rank == 0:
        head = legs[0]
        line = dict(results[head])
        line.setdefault('higher_is_better', True)
        line.setdefault('vs_baseline', None)
        line.setdefault('data', 'synthetic')
        line.setdefault('warmup', max(a.warmup, 3))
        extra = {k: v for k, v in results.items() if k != head}
        if extra:
            line['extra'] = extra
        print(json.dumps(line))
    if ctx.world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
