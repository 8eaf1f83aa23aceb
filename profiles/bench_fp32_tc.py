#!/usr/bin/env python
"""bench_fp32_tc.py -- precision='fp32-tc' (3xTF32 on tcgen05) against 'fp32' (FFMA) and 'bf16' on the state-based workloads.

  python profiles/bench_fp32_tc.py [--out FILE.json] [--rounds 5] [--steps 10]

Per workload the three precisions run in one process, each with its own agent and staged batch; after every shape has been warmed up,
the timed rounds alternate fp32 / fp32-tc / bf16, `steps` device-timed steps each (CUDA events around every FQLAgent.step, L2
overwritten with a 256 MiB write before every step, as bench.py does).  ms_per_step is the median over rounds of each round's mean.
Then the 3xTF32 GEMM alone (fql_test_gemm_f32) and the FFMA GEMM at the step's shapes of config 3 at B = 16384: achieved TFLOP/s =
ALGORITHMIC flops 2 M N K x groups (not the 3x the tensor cores execute) over the CUDA-event time of one launch, L2 overwritten
before each launch, median of 20.  The card's name and power limit are read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import WORKLOADS, make_host_batches  # noqa: E402

RUNS = [  # (workload, batch, seeds)
    ('antmaze-large', 256, 1),          # config 2
    ('humanoidmaze-medium', 1024, 1),   # config 3
    ('humanoidmaze-medium', 4096, 1),
    ('humanoidmaze-medium', 16384, 1),
    ('puzzle-4x4', 256, 8),             # config 4: 8 seeds x 256
]
PRECISIONS = ('fp32', 'fp32-tc', 'bf16')


def card():
    import torch
    info = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info['nvidia_smi'] = q
    except Exception as e:  # the numbers are still labelled with the torch device name
        info['nvidia_smi'] = repr(e)[:200]
    return info


def time_steps(agent, bufs, steps, flush):
    import torch
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for i in range(steps):
        flush.zero_()
        ev[i][0].record()
        agent.step(bufs)
        ev[i][1].record()
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in ev) / steps


def bench_workload(name, batch, seeds, rounds, steps, flush):
    import torch
    from fql_b200 import FQLAgent, get_config
    wl = WORKLOADS[name]
    F, A = wl['F'], wl['A']
    cfg = get_config()
    cfg.update(wl['cfg'])
    cfg['batch_size'] = batch
    host = make_host_batches(1, batch, F, A, seeds, seed0=77)[0]
    agents = {}
    for p in PRECISIONS:
        ag = FQLAgent.create(0, np.zeros((1, F), np.float32), np.zeros((1, A), np.float32), cfg, num_seeds=seeds, precision=p)
        bufs = ag.stage(host)
        for _ in range(5):
            info = ag.step(bufs)
        agents[p] = (ag, bufs)
    torch.cuda.synchronize()
    per = {p: [] for p in PRECISIONS}
    for _ in range(rounds):
        for p in PRECISIONS:
            per[p].append(time_steps(*agents[p], steps, flush))
    out = dict(workload=name, batch=batch, seeds=seeds)
    for p in PRECISIONS:
        info = agents[p][0].step(agents[p][1])
        loss = float(np.ravel(info['critic/critic_loss'])[0])
        out[p] = dict(ms_per_step=float(np.median(per[p])), rounds_ms=[round(x, 4) for x in per[p]],
                      samples_per_s=batch * seeds / (float(np.median(per[p])) / 1e3), finite=bool(np.isfinite(loss)))
    out['fp32_tc_speedup_over_fp32'] = out['fp32']['ms_per_step'] / out['fp32-tc']['ms_per_step']
    del agents
    torch.cuda.empty_cache()
    return out


def bench_gemm(flush, reps=20):
    """The GEMMs of config 3 (F + A = 90, hidden 512) at B = 16384 as the step launches them."""
    import torch
    from fql_b200 import _lib
    B, H, K0 = 16384, 512, 90
    shapes = [  # (name, M, N, K, P, E, trans_a, trans_b, act, mulz)
        ('critic fwd first layer (3 problems x 2 heads)', B, H, K0, 3, 2, 0, 0, 1, 0),
        ('critic fwd hidden layer (3 problems x 2 heads)', B, H, H, 3, 2, 0, 0, 1, 0),
        ('critic dgrad hidden, gelu\' fused (2 heads)', B, H, H, 1, 2, 0, 1, 0, 1),
        ('critic wgrad hidden, K = batch (2 heads)', H, H, B, 1, 2, 1, 0, 0, 0),
        ('actor wgrad first layer, K = batch', K0, H, B, 1, 1, 1, 0, 0, 0),
    ]
    res = []
    for name, M, N, K, P, E, ta, tb, act, mulz in shapes:
        ra, ca = (K, M) if ta else (M, K)
        rb, cb = (N, K) if tb else (K, N)
        g = torch.Generator(device='cuda').manual_seed(1)
        A = [torch.randn(E, ra, ca, device='cuda', generator=g) for _ in range(P)]
        Bm = [torch.randn(E, rb, cb, device='cuda', generator=g) for _ in range(P)]
        out = [torch.empty(E, M, N, device='cuda') for _ in range(P)]
        z = torch.randn(E, M, N, device='cuda', generator=g) if mulz else None

        def gp(bufs, rows, ld):
            x = _lib.FqlTestGPtr()
            for i, b in enumerate(bufs):
                x.base[i] = b.data_ptr()
            x.stride_s, x.stride_e = E * rows * ld, rows * ld
            return x
        t = _lib.FqlTestGemmF32()
        t.M, t.N, t.K, t.P, t.S, t.E = M, N, K, P, 1, E
        t.lda, t.ldb, t.ldo, t.ld_pre, t.ld_mulz = ca, cb, N, N, N
        t.trans_a, t.trans_b, t.act_gelu = ta, tb, act
        t.A, t.B, t.out = gp(A, ra, ca), gp(Bm, rb, cb), gp(out, M, N)
        if mulz:
            t.mulz = gp([z] * P, M, N)
        flops = 2.0 * M * N * K * P * E
        row = dict(gemm=name, M=M, N=N, K=K, groups=P * E, algorithmic_gflop=flops / 1e9)
        for prec, key in ((3, 'tf32x3'), (0, 'ffma')):
            stream = torch.cuda.current_stream().cuda_stream
            for _ in range(3):
                _lib.check(_lib.lib().fql_test_gemm_f32(C.byref(t), prec, C.c_void_p(stream)), 'gemm')
            ts = []
            for _ in range(reps):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                _lib.check(_lib.lib().fql_test_gemm_f32(C.byref(t), prec, C.c_void_p(stream)), 'gemm')
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            ms = float(np.median(ts))
            row[key] = dict(ms=ms, algorithmic_tflops=flops / (ms / 1e3) / 1e12)
        res.append(row)
        del A, Bm, out, z
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--steps', type=int, default=10)
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), 'bench_fp32_tc.py measures on the GPU'
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    out = dict(card=card(), method=__doc__.strip().splitlines()[2:], rounds=args.rounds, steps_per_round=args.steps)
    out['workloads'] = []
    for name, batch, seeds in RUNS:
        r = bench_workload(name, batch, seeds, args.rounds, args.steps, flush)
        print(json.dumps(r), flush=True)
        out['workloads'].append(r)
    out['gemm_config3_b16384'] = bench_gemm(flush)
    for r in out['gemm_config3_b16384']:
        print(json.dumps(r), flush=True)
    out['card_after'] = card()
    s = json.dumps(out, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(s + '\n')
    else:
        print(s)


if __name__ == '__main__':
    main()
