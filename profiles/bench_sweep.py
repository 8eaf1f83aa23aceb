#!/usr/bin/env python
"""bench_sweep.py -- an alpha sweep as vectorised seeds (FQLAgent.create(per_seed=...)) against what one could do without it.

  python profiles/bench_sweep.py [--out FILE.json] [--rounds 7] [--steps 20]

Workload: config 4's shape (puzzle-4x4: F 83, A 5, normalize_q_loss, batch 256 per agent), an alpha grid of 6 values x 8 seeds = 48
agents.  Three arms per precision ('bf16', 'fp32-tc'), each with its own agents and staged batch, in one process:
  (a) table   one 48-seed agent with per_seed={'alpha': [6 values x 8 seeds]};
  (b) shared  the same 48-seed agent with one shared alpha (no table): the cost of the table is (a) - (b);
  (c) six     six 8-seed agents, one per alpha value, stepped back to back: the sweep without per-seed hyperparameters.
After every agent has been warmed up (eager step, graph capture, replays), the timed rounds alternate (a) / (b) / (c), `steps` device-
timed units each: CUDA events around one FQLAgent.step (around all six for (c)), L2 overwritten with a 256 MiB write before every unit,
as bench.py does.  ms_per_step is the median over rounds of each round's mean.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'profiles'))

from bench import WORKLOADS, make_host_batches  # noqa: E402
from bench_fp32_tc import card  # noqa: E402

ALPHAS = (30.0, 100.0, 300.0, 1000.0, 3000.0, 10000.0)
SEEDS_PER_ALPHA = 8
PRECISIONS = ('bf16', 'fp32-tc')
ARMS = ('table', 'shared', 'six')


def time_units(units, steps, flush):
    """units: a list of (agent, bufs) stepped back to back as one timed unit."""
    import torch
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for i in range(steps):
        flush.zero_()
        ev[i][0].record()
        for agent, bufs in units:
            agent.step(bufs)
        ev[i][1].record()
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in ev) / steps


def bench_precision(precision, rounds, steps, flush):
    import torch
    from fql_b200 import FQLAgent, get_config
    wl = WORKLOADS['puzzle-4x4']
    F, A, B = wl['F'], wl['A'], 256
    S = len(ALPHAS) * SEEDS_PER_ALPHA
    cfg = get_config()
    cfg.update(wl['cfg'])
    cfg['batch_size'] = B
    host = make_host_batches(1, B, F, A, S, seed0=77)[0]
    ex = (np.zeros((1, F), np.float32), np.zeros((1, A), np.float32))
    grid = [a for a in ALPHAS for _ in range(SEEDS_PER_ALPHA)]
    arms = {}
    ag = FQLAgent.create(0, *ex, cfg, num_seeds=S, precision=precision, per_seed={'alpha': grid})
    arms['table'] = [(ag, ag.stage(host))]
    ag = FQLAgent.create(0, *ex, cfg, num_seeds=S, precision=precision)
    arms['shared'] = [(ag, ag.stage(host))]
    arms['six'] = []
    for j, alpha in enumerate(ALPHAS):
        ag = FQLAgent.create(0, *ex, dict(cfg, alpha=alpha), num_seeds=SEEDS_PER_ALPHA, precision=precision)
        part = {k: v[j * SEEDS_PER_ALPHA:(j + 1) * SEEDS_PER_ALPHA] for k, v in host.items()}
        arms['six'].append((ag, ag.stage(part)))
    for units in arms.values():
        for _ in range(5):
            for agent, bufs in units:
                agent.step(bufs)
    torch.cuda.synchronize()
    per = {a: [] for a in ARMS}
    for _ in range(rounds):
        for a in ARMS:
            per[a].append(time_units(arms[a], steps, flush))
    out = dict(precision=precision, workload='puzzle-4x4', batch=B, agents=S, alphas=list(ALPHAS), seeds_per_alpha=SEEDS_PER_ALPHA)
    for a in ARMS:
        ms = float(np.median(per[a]))
        losses = [np.ravel(agent.step(bufs)['critic/critic_loss']) for agent, bufs in arms[a]]
        out[a] = dict(ms_per_step=ms, rounds_ms=[round(x, 4) for x in per[a]], us_per_agent=ms * 1e3 / S,
                      samples_per_s=B * S / (ms / 1e3), finite=bool(all(np.isfinite(l).all() for l in losses)))
    out['table_over_shared'] = out['table']['ms_per_step'] / out['shared']['ms_per_step']
    out['six_over_table'] = out['six']['ms_per_step'] / out['table']['ms_per_step']
    del arms, ag
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--rounds', type=int, default=7)
    ap.add_argument('--steps', type=int, default=20)
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), 'bench_sweep.py measures on the GPU'
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    out = dict(card=card(), method=__doc__.strip().splitlines()[2:], rounds=args.rounds, steps_per_round=args.steps, results=[])
    for p in PRECISIONS:
        r = bench_precision(p, args.rounds, args.steps, flush)
        print(json.dumps(r), flush=True)
        out['results'].append(r)
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
