#!/usr/bin/env python
"""bench.py -- FQL update throughput on B200 (the metric BASELINE.json names), one JSON line on stdout.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload antmaze-large] [--batch 256] [--seeds 1]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...     (N > 1, one rank per GPU)
  python bench.py --impl reference ...       CPU arm: the oracle's fp32 restatement of the reference on the host cores
  python bench.py ... --dump-outputs DIR     also write the metrics and parameters of the last timed step as DIR/<name>.npy

A "step" is one FQLAgent.update (agents/fql.py:122-133) on one synthetic batch of the named OGBench shape.  The K timed steps are
steps W+1 .. W+K of one training run from the seeded initial state, so with the same arguments every run computes the same outputs.
  value   device-timed samples/s with the batch already resident in HBM (CUDA events around every step, max over ranks)
  e2e     the same through the public API `agent.update(host_batch)`: pinned H2D of the batch + D2H of the 13 metrics
N > 1 is data parallel, weak scaling: every rank holds `--batch` rows of a global batch of N*batch; the gradient buckets are
reduced by the library's own kernels over NVLink peer memory / NVLS multicast inside the step graph (FQL_DP_BACKEND=nccl: NCCL
all-reduce instead); value = global samples/s.  `--seeds S` with N > 1 shards SEEDS: every rank trains its own S independent
agents, no collective on the step.  Every line also carries `scaling_configs`: the sharded north_star configurations
(humanoidmaze-medium batch 8192/GPU data parallel; puzzle-4x4 8 seeds/GPU seed-sharded; visual-cube-single pixels batch 256/GPU data
parallel) timed in the same run at this N, and BASELINE config 1 beside the headline config 2 at N = 1.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {  # BASELINE.json configs 1-4 (state-based); SURVEY 8d hyper-parameters
    'cube-single': dict(F=28, A=5, cfg=dict(alpha=300.0)),
    'antmaze-large': dict(F=29, A=8, cfg=dict(q_agg='min', alpha=10.0)),
    'humanoidmaze-medium': dict(F=69, A=21, cfg=dict(discount=0.995, alpha=30.0)),
    'puzzle-4x4': dict(F=83, A=5, cfg=dict(normalize_q_loss=True, alpha=1000.0)),  # F=83 assumed (SURVEY 8: unverified)
    # BASELINE config 5: 64x64x3 pixels, frame_stack 3 -> 64x64x9 uint8, impala_small encoders (tcgen05 implicit-GEMM convolutions)
    'visual-cube-single': dict(F=512, A=5, image=(64, 64, 9), cfg=dict(alpha=300.0, encoder='impala_small')),
}


ENC_FWD_FLOPS = 48.10e6          # impala_small forward per 64x64x9 image (SURVEY 8d)
ENC_FIRST_DGRAD = 10.62e6        # the pixel-input gradient of the first convolution that is never needed


def flops_per_sample(F, A, H=512, pixels=False):
    """Algorithmic FLOPs of one update per sample (SURVEY 8d): MACs x2 of the Dense/Conv layers only.  Pixels: + 5 encoder
    forwards, 3 encoder backwards (2x forward minus the first conv's input gradient) and the first-layer dgrad into the features."""
    if pixels:
        return flops_per_sample(F, A, H) + 3 * 2 * F * H + 5 * ENC_FWD_FLOPS + 3 * (2 * ENC_FWD_FLOPS - ENC_FIRST_DGRAD)
    G = lambda d, o: 2 * (d * H + 3 * H * H + H * o)
    d_bc, d_os, d_c = F + A + 1, F + A, F + A
    fwd = 11 * G(d_bc, A) + 3 * G(d_os, A) + 6 * G(d_c, 1)
    bwd = (2 * G(d_bc, A) - 2 * d_bc * H) + (2 * G(d_os, A) - 2 * d_os * H) + 2 * (2 * G(d_c, 1) - 2 * d_c * H) \
        + 2 * (G(d_c, 1) - 2 * F * H)
    return fwd + bwd


def hbm_bytes_per_step(p_train, p_target, B, F, A):
    """Algorithmic HBM bytes of one update (SURVEY 8d): Adam 28 B/param, Polyak 8 B/target param (fused with Adam's read of
    the critic), every weight read once by the GEMMs (4 B), the batch."""
    return 28 * p_train + 8 * p_target + 4 * (p_train + p_target) + B * (2 * F + A + 2) * 4


def _shutdown(agent):
    """Orderly multi-rank teardown: captured graphs that hold NCCL kernels are released before the process group goes away, and a
    watchdog turns a stuck communicator teardown into a clean exit (the result line is already printed and flushed)."""
    import threading
    import torch
    import torch.distributed as dist
    sys.stdout.flush()
    threading.Thread(target=lambda: (time.sleep(30.0), os._exit(0)), daemon=True).start()
    try:
        agent.release_graphs()
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()
    except Exception:
        pass


def load_peaks():
    try:
        p = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        return dict(hbm=p['hbm_gbs'], tc=p.get('bf16_tflops_sustained', p['bf16_tflops']), tc_burst=p['bf16_tflops'],
                    src='measured (MEASURED_PEAKS.json)')
    except Exception:
        return dict(hbm=6650.0, tc=1400.0, tc_burst=1400.0, src='fallback (B200_PROFILING.md)')


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(index), f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '20'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows = [r for r in self.rows if len(r) == 6 and r[0].isdigit()]
        if not rows:
            return None
        sm = sorted(int(r[0]) for r in rows)
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith('active') for r in rows)]
        return dict(sm_mhz=sm[len(sm) // 2], sm_max_mhz=int(rows[0][1]), reasons=reasons, samples=len(rows))


def make_host_batches(n, B, F, A, seeds, seed0=0, image=None):
    import numpy as np
    out = []
    for i in range(n):
        rng = np.random.default_rng(seed0 + i)
        shp = (seeds, B) if seeds > 1 else (B,)
        rew = -(rng.random(shp) >= 0.01).astype(np.float32)
        mk = (lambda: rng.integers(0, 256, shp + tuple(image), dtype=np.uint8)) if image else (lambda: rng.standard_normal(shp + (F,), dtype=np.float32))
        out.append(dict(
            observations=mk(),
            actions=np.clip(rng.uniform(-1, 1, shp + (A,)), -1 + 1e-5, 1 - 1e-5).astype(np.float32),
            next_observations=mk(),
            rewards=rew, masks=(rew != 0).astype(np.float32), terminals=np.zeros(shp, np.float32)))
    return out


def cpu_reference_arm(wl, B, steps, warmup, budget_s=20.0):
    """The reference's CPU path: JAX is not installed (SURVEY F1), so this is oracle/fql_torch_cpu.py, the fp32 torch-CPU
    restatement of FQLAgent.update (autograd, MKL, every host core), same shapes and hyper-parameters.  kind='port'."""
    import numpy as np
    import torch
    from oracle import fql_oracle as O
    from oracle.fql_torch_cpu import TorchCpuAgent
    # every host core this process may use, also under torchrun (which exports OMP_NUM_THREADS=1 to its workers)
    try:
        torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    except Exception:
        pass
    cfg = dict(O.DEFAULT_CONFIG)
    cfg.update(wl['cfg'])
    F, A = wl['F'], wl['A']
    if wl.get('image'):
        from oracle import fql_pixel_oracle as PO
        params = PO.init_params(1, wl['image'][2], A, cfg, dtype=np.float32, hw=wl['image'][0])
    else:
        params = O.init_params(1, F, A, cfg, dtype=np.float32)
    agent = TorchCpuAgent(params, cfg)
    batches = make_host_batches(4, B, F, A, 1, image=wl.get('image'))
    noises = [O.make_noise(i, B, A, np.float32) for i in range(4)]
    for i in range(max(1, warmup)):
        agent.update(batches[i % 4], noises[i % 4])
    times = []
    t_begin = time.perf_counter()
    for i in range(steps):
        t0 = time.perf_counter()
        info, _ = agent.update(batches[i % 4], noises[i % 4])
        times.append(time.perf_counter() - t0)
        if budget_s is not None and time.perf_counter() - t_begin > budget_s and len(times) >= 3:
            break
    times.sort()
    med = times[len(times) // 2]
    return dict(ms_per_step=med * 1e3, steps_measured=len(times), cores=torch.get_num_threads(), loss=info['critic/critic_loss'])


def time_config(name, batch, seeds, mode, world, rank, pg, stream, flush, steps=20, warmup=5):
    """One more configuration timed at this N in the same run (device-timed, L2 flushed, max over ranks): mode 'dp' = rows sharded,
    gradient buckets reduced across ranks inside the step; 'seeds' = independent agents per rank, no collective; 'single' = rank-local."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from fql_b200 import FQLAgent, get_config
    wl = WORKLOADS[name]
    F, A = wl['F'], wl['A']
    cfg = get_config()
    cfg.update(wl['cfg'])
    cfg['batch_size'] = batch
    precision = 'bf16'
    ex_obs = np.zeros((1,) + tuple(wl['image']), np.uint8) if wl.get('image') else np.zeros((1, F), np.float32)
    out = dict(workload=name, batch_per_gpu=batch, seeds_per_gpu=seeds, n_gpus=world, mode=mode, precision=precision)
    try:
        with torch.cuda.stream(stream):
            agent = FQLAgent.create(rank if mode == 'seeds' else 0, ex_obs, np.zeros((1, A), np.float32), cfg, num_seeds=seeds, precision=precision,
                                    process_group=pg if (mode == 'dp' and world > 1) else None)
            bufs = agent.stage(make_host_batches(1, batch, F, A, seeds, seed0=77 + rank, image=wl.get('image'))[0])
            for _ in range(warmup):
                agent.step(bufs)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            for i in range(steps):
                flush.zero_()
                ev[i][0].record()
                info = agent.step(bufs)
                ev[i][1].record()
            torch.cuda.synchronize()
            ms = sum(a.elapsed_time(b) for a, b in ev) / steps
            loss = float(np.ravel(info['critic/critic_loss'])[0])
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device='cuda')
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        n_units = world if mode in ('dp', 'seeds') else 1
        samples = batch * seeds * n_units
        peaks = load_peaks()
        flops_gpu = flops_per_sample(F, A, pixels=bool(wl.get('image'))) * batch * seeds
        out.update(ms_per_step=ms, steps_per_sec=1e3 / ms, value=samples / (ms / 1e3), unit='samples/s', steps=steps, warmup=warmup,
                   global_batch=batch * (world if mode == 'dp' else 1), total_seeds=seeds * (world if mode == 'seeds' else 1),
                   tensor_tflops_per_gpu=flops_gpu / (ms / 1e3) / 1e12, tensor_frac=flops_gpu / (ms / 1e3) / 1e12 / peaks['tc'],
                   finite=bool(np.isfinite(loss)), transport=getattr(agent, 'dp_transport', None))
        del agent, bufs
        torch.cuda.empty_cache()
    except Exception as e:  # a scaling entry must never cost the headline line
        out['error'] = repr(e)[:300]
    return out


def euler_kernel_traffic_from_profile():
    """DRAM bytes (read + write) of one launch of the Euler cluster kernel, read from the newest committed `ncu --set full` summary under
    profiles/ (the capture is made with the same bench command; bench.py itself never runs under a profiler)."""
    import glob
    import re
    here = os.path.dirname(os.path.abspath(__file__))
    unit = {'byte': 1.0, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9}
    for path in sorted(glob.glob(os.path.join(here, 'profiles', 'r*_ncu_full_cluster_kernels.txt')), reverse=True):
        try:
            blocks = open(path).read().split('----')
        except OSError:
            continue
        for b in blocks:
            if 'euler_cluster_kernel<16, 8, 0>' not in b:
                continue
            tot = 0.0
            for name in ('dram__bytes_read.sum', 'dram__bytes_write.sum'):
                m = re.search(re.escape(name) + r' \[(\w+)\] = ([0-9.]+)', b)
                if not m:
                    break
                tot += float(m.group(2)) * unit.get(m.group(1), 1.0)
            else:
                return int(tot), 'profiles/' + os.path.basename(path)
    return None, None


def write_outputs(out_dir, arrays, limit=64 * 10 ** 6):
    """--dump-outputs: one float32 DIR/<name>.npy per array.  Past `limit` bytes in all, every array of more than 4096 elements is cut
    to the same fraction of its flattened elements, picked with a fixed seed, so two runs with the same arguments still compare
    element for element."""
    import numpy as np
    arrays = {k: np.asarray(v, np.float32) for k, v in arrays.items()}
    small = sum(a.size for a in arrays.values() if a.size <= 4096) * 4
    big = sum(a.size for a in arrays.values() if a.size > 4096) * 4
    frac = min(1.0, (limit - small - 256 * len(arrays)) / max(big, 1))    # 256 bytes: room for each .npy header
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if frac < 1.0 and a.size > 4096:
            a = a.ravel()[np.sort(np.random.default_rng(0).choice(a.size, int(a.size * frac), replace=False))]
        np.save(os.path.join(out_dir, name + '.npy'), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=20)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='antmaze-large', choices=sorted(WORKLOADS))
    ap.add_argument('--batch', type=int, default=256, help='rows per GPU (per seed)')
    ap.add_argument('--seeds', type=int, default=1, help='independent agents vectorised on each GPU')
    ap.add_argument('--precision', default='bf16', choices=['fp32', 'bf16'],
                    help='bf16: tcgen05 operands, fp32 accumulate/master weights (default); fp32: FFMA parity mode')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-fp32-leg', action='store_true')
    ap.add_argument('--no-scaling-configs', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the metrics and the parameters of the last timed step as DIR/<name>.npy (float32, at most 64 MB '
                         'in all: larger parameter sets are written as a fixed, seeded sample)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs writes what the b200 implementation computed')
    wl = WORKLOADS[args.workload]
    # pixel workloads: --precision bf16 = the ImpalaEncoders on tcgen05 in bf16 (FQL_PRECISION_BF16_ENC), MLPs behind them in fp32
    F, A = wl['F'], wl['A']
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    config = dict(workload=f'{args.workload}-shaped synthetic (obs {F}, act {A}), FQL update, batch {args.batch}/GPU, '
                           f'{args.seeds} seed(s)/GPU, 4x512 MLPs, flow_steps 10, ' + ', '.join(f'{k}={v}' for k, v in wl['cfg'].items()),
                  batch_per_gpu=args.batch, global_batch=args.batch * max(world, 1), seeds_per_gpu=args.seeds,
                  parallelism=(f'seeds sharded over {world} GPUs (no collective)' if world > 1 and args.seeds > 1 else f'dp{world}') if world > 1 else 'single',
                  l2='flushed between timed steps (256 MiB write)')

    if args.impl == 'reference':
        if rank != 0:
            return 0
        r = cpu_reference_arm(wl, args.batch, args.steps, args.warmup, budget_s=None)
        sps = 1e3 / r['ms_per_step']
        val = sps * args.batch
        sample = f"{r['steps_measured']} full updates of the same workload at batch {args.batch} (median), fp32 torch-CPU (MKL, autograd)"
        print(json.dumps(dict(
            impl='reference', metric='fql_update_samples_per_sec', value=val, unit='samples/s', steps_per_sec=sps, n_gpus=args.gpus,
            device='cpu (host cores of the box; no GPU is used by this arm)',
            steps=r['steps_measured'], warmup=max(1, args.warmup), ms_per_step=r['ms_per_step'], higher_is_better=True,
            scaling='weak', vs_baseline=None, dtype='f32', data='synthetic', config=config,
            cpu_baseline=dict(value=val, unit='samples/s', cores=r['cores'], kind='port', sample=sample),
            e2e=dict(value=val, unit='samples/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0),
            note='reference JAX is not installable here (no jax/flax/optax, no network): CPU restatement of the reference, '
                 'not JAX/XLA')))
        return 0

    import numpy as np
    import torch
    import torch.distributed as dist
    from fql_b200 import FQLAgent, get_config

    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local_rank)
    pg = None
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device(f'cuda:{local_rank}'))
        pg = dist.group.WORLD
    seed_sharded = world > 1 and args.seeds > 1       # independent agents per rank: no process group on the agent, no collective
    cfg = get_config()
    cfg.update(wl['cfg'])
    cfg['batch_size'] = args.batch
    ex_obs = np.zeros((1,) + tuple(wl['image']), np.uint8) if wl.get('image') else np.zeros((1, F), np.float32)
    agent = FQLAgent.create(rank if seed_sharded else 0, ex_obs, np.zeros((1, A), np.float32), cfg, num_seeds=args.seeds,
                            precision=args.precision, process_group=None if seed_sharded else pg)
    batches = make_host_batches(8, args.batch, F, A, args.seeds, seed0=1000 * rank, image=wl.get('image'))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    stream = torch.cuda.Stream()  # a real (non-legacy) stream: the library captures its step graph on it
    K, W = args.steps, max(args.warmup, 3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.cuda.stream(stream):
        # ---------------- device-resident leg: `value`
        bufs = agent.stage(batches[0])
        clocks = ClockSampler(local_rank) if rank == 0 else None
        for _ in range(W):
            agent.step(bufs)
        # the timed steps continue from this state: the load below runs a number of steps that depends on the clock
        warm_state = agent.state_dict()
        # keep the GPU under the same load until nvidia-smi is sampling (~0.5 s): the step count must be IDENTICAL on every rank
        # (each step contains collectives), so it is derived from a max-reduced timing, never from a per-rank clock
        torch.cuda.synchronize()
        t_probe = time.perf_counter()
        for _ in range(5):
            agent.step(bufs)
        torch.cuda.synchronize()
        per = torch.tensor([(time.perf_counter() - t_probe) / 5], dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(per, op=dist.ReduceOp.MAX)
        for _ in range(int(min(3000, max(0, 0.5 / max(float(per.item()), 1e-6))))):
            agent.step(bufs)
        barrier()
        agent.load_state_dict(warm_state)
        l0 = agent.launch_count()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        barrier()
        for i in range(K):
            flush.zero_()
            ev[i][0].record()
            info = agent.step(bufs)
            ev[i][1].record()
        barrier()
        launches = agent.launch_count() - l0
        dev_ms = sum(a.elapsed_time(b) for a, b in ev)
        if args.dump_outputs and rank == 0:
            from oracle.fql_oracle import tree_leaves
            outputs = {'info.' + k.replace('/', '.'): v for k, v in info.items()}
            outputs.update(('params.' + '.'.join(path), v) for path, v in tree_leaves(agent.export_tree('params')))
        last_loss = float(np.ravel(info['critic/critic_loss'])[0])
        assert np.isfinite(last_loss), 'non-finite loss in the timed region'
        # L2-warm variant (no flush), reported beside the headline
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            agent.step(bufs)
        e1.record()
        barrier()
        warm_ms = e0.elapsed_time(e1)
        clk = clocks.stop() if clocks else None

        # ---------------- end-to-end leg: public API, host batches, pinned H2D + D2H of the metrics every step
        for i in range(W):
            agent.update(batches[i % 8])
        barrier()
        t0 = time.perf_counter()
        for i in range(K):
            _, info = agent.update(batches[i % 8])
        _ = info['critic/critic_loss']  # materialise the last step's metrics (every step's D2H copy has been issued)
        barrier()
        e2e_s = time.perf_counter() - t0
        h2d = agent.last_h2d_bytes

    if world > 1:
        t = torch.tensor([dev_ms, warm_ms, e2e_s * 1e3], dtype=torch.float64, device='cuda')
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, warm_ms, e2e_ms = [float(x) for x in t.tolist()]
        e2e_s = e2e_ms / 1e3
    # the sharded north_star configurations at this N (every rank takes part), and BASELINE config 1 beside the headline config 2
    scaling_configs = []
    if not args.no_scaling_configs:
        scaling_configs.append(time_config('humanoidmaze-medium', 8192, 1, 'dp', world, rank, pg, stream, flush))
        scaling_configs.append(time_config('puzzle-4x4', 256, 8, 'seeds', world, rank, pg, stream, flush))
        scaling_configs.append(time_config('visual-cube-single', 256, 1, 'dp' if world > 1 else 'single', world, rank, pg, stream, flush))
        if world == 1:
            scaling_configs.append(time_config('cube-single', 256, 1, 'single', world, rank, pg, stream, flush, steps=50))
    if rank != 0:
        if world > 1:
            _shutdown(agent)
        return 0

    n = max(world, 1)
    samples_per_step = args.batch * args.seeds * n
    ms_per_step = dev_ms / K
    value = samples_per_step / (ms_per_step / 1e3)
    peaks = load_peaks()
    leaves = agent._leaves
    cnt = lambda pred: sum(l['ens'] * l['rows'] * l['cols'] for l in leaves if pred(l))
    p_train, p_target = cnt(lambda l: l['net'] != 'target_critic'), cnt(lambda l: l['net'] == 'target_critic')
    flops_gpu = flops_per_sample(F, A, pixels=bool(wl.get('image'))) * args.batch * args.seeds   # per GPU per step
    bytes_gpu = (hbm_bytes_per_step(p_train, p_target, args.batch, F, A)) * args.seeds
    if wl.get('image'):
        bytes_gpu += args.batch * 2 * int(np.prod(wl['image'])) - args.batch * 2 * F * 4   # the batch is uint8 frames, not features
    t_s = ms_per_step / 1e3
    t_tc, t_hbm = flops_gpu / (peaks['tc'] * 1e12), bytes_gpu / (peaks['hbm'] * 1e9)
    if t_hbm >= t_tc:
        roof = dict(bound='hbm', achieved=bytes_gpu / t_s / 1e9, peak=peaks['hbm'], unit='GB/s')
    else:
        roof = dict(bound='tensor', achieved=flops_gpu / t_s / 1e12, peak=peaks['tc'], unit='TFLOP/s')
    roof['frac'] = roof['achieved'] / roof['peak']
    roof.update(traffic=None, scope='whole update step (one CUDA graph); per-kernel shares in profiles/', peak_source=peaks['src'],
                algorithmic_flops_per_step_per_gpu=flops_gpu, algorithmic_bytes_per_step_per_gpu=bytes_gpu,
                tensor_tflops_achieved=flops_gpu / t_s / 1e12, tensor_frac=flops_gpu / t_s / 1e12 / peaks['tc'],
                hbm_gbs_achieved=bytes_gpu / t_s / 1e9, t_min_us=max(t_tc, t_hbm) * 1e6,
                arithmetic='fp32 FFMA (parity mode)' if args.precision == 'fp32' else
                ('bf16 tcgen05 implicit-GEMM encoders (fp32 accumulate), fp32 FFMA MLPs' if wl.get('image') else 'bf16 tcgen05, fp32 accumulate'))
    if n == 1 and args.precision == 'bf16' and not wl.get('image') and args.seeds == 1:
        # the dominant kernel, timed alone on its launching stream with CUDA events (L2 flushed between launches): the persistent
        # cluster kernel of compute_flow_actions = the longest dependent chain of the step (concat + pad + ONE cluster launch)
        try:
            with torch.cuda.stream(stream):
                obs_d = torch.randn(args.batch, F, device='cuda')
                nz_d = torch.randn(args.batch, A, device='cuda')
                for _ in range(3):
                    agent._fwd_call(agent._lib.fql_compute_flow_actions, obs_d, nz_d, to_host=False)
                kk = 20
                ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(kk)]
                for i in range(kk):
                    flush.zero_()
                    ev[i][0].record()
                    agent._fwd_call(agent._lib.fql_compute_flow_actions, obs_d, nz_d, to_host=False)
                    ev[i][1].record()
                torch.cuda.synchronize()
            k_us = 1e3 * float(np.median([x.elapsed_time(y) for x, y in ev]))
            Hh = 512
            k_flops = int(cfg['flow_steps']) * 2 * ((F + A + 1) * Hh + 3 * Hh * Hh + Hh * A) * args.batch
            k_tf = k_flops / (k_us * 1e-6) / 1e12
            default_wl = args.workload == 'antmaze-large' and args.batch == 256
            ncu_traffic = euler_kernel_traffic_from_profile()
            step_level = roof
            # the object the contract asks for: the dominant kernel against the roofline that bounds it (tensor: it is a chain of
            # dense contractions), peak = the burst figure because the kernel is timed alone; the whole-step view is kept in `step`
            roof = dict(
                bound='tensor', achieved=k_tf, peak=peaks['tc_burst'], unit='TFLOP/s', frac=k_tf / peaks['tc_burst'],
                traffic=ncu_traffic[0] if default_wl else None,
                traffic_source=(ncu_traffic[1] + ': dram__bytes_read.sum + dram__bytes_write.sum of one launch (ncu --set full; '
                                'algorithmic: 1.7 MB of bf16 weights read once + 40 KB of inputs/outputs)') if default_wl and ncu_traffic[0] else None,
                kernel='euler_cluster_kernel<16,8,EULER> = compute_flow_actions, the longest dependent chain of the step',
                us_per_launch=k_us, timed='alone through fql_compute_flow_actions (concat + bf16 pad + ONE cluster launch, ~8 us of the '
                                          'figure are the two small kernels), CUDA events on the launching stream, L2 flushed between launches',
                algorithmic_flops_per_launch=k_flops, share_of_step=k_us / (ms_per_step * 1e3), peak_source=peaks['src'],
                why_small='latency-bound by construction: flow_steps x 5 dependent layers on batch/128 = 2 row tiles (32 CTAs); one layer = '
                          'TMEM read of the 2 partial accumulators + ~1 us multicast-TMA round trip + 16 MMA issues per issuer warp (profiles/)',
                step=step_level)
        except Exception as e:  # a diagnostic, never the reason a bench line is missing
            roof['dominant_kernel_error'] = repr(e)
    out = dict(metric='fql_update_samples_per_sec', value=value, unit='samples/s', steps_per_sec=1e3 / ms_per_step, n_gpus=n,
               steps=K, warmup=W, ms_per_step=ms_per_step, higher_is_better=True, scaling='weak', vs_baseline=None,
               dtype='f32' if args.precision == 'fp32' else 'bf16', data='synthetic', config=config,
               value_l2_warm=(samples_per_step / (warm_ms / K / 1e3)) if n == 1 else None,
               ms_per_step_l2_warm=(warm_ms / K) if n == 1 else None,
               e2e=dict(value=samples_per_step * K / e2e_s, unit='samples/s', steps_per_sec=K / e2e_s, h2d_bytes_per_step=h2d,
                        d2h_bytes_per_step=13 * 4 * args.seeds, api='FQLAgent.update(host numpy batch)',
                        note='wall clock over K public-API calls, a fresh host batch each; its H2D copy runs on a copy stream under the previous step '
                             '(two input sets) and the metrics come back every step; no L2 flush in this loop: compare with value_l2_warm'),
               gpu_launches=launches, gpu_launches_per_step=launches / K, roofline=roof, clocks=clk, last_critic_loss=last_loss,
               scaling_configs=scaling_configs, dp_transport=getattr(agent, 'dp_transport', None))
    if n == 1 and not wl.get('image'):
        # online / evaluation path (main.py:225, evaluation.py:98-150): host observation in, host action out, one row and ten rows
        try:
            lat = {}
            with torch.cuda.stream(stream):
                for rows in (1, 10):
                    ob = np.random.default_rng(5).standard_normal((rows, F)).astype(np.float32)
                    for _ in range(20):
                        agent.sample_actions(ob, seed=np.array([1, 2], np.uint32))
                    ts = []
                    for _ in range(200):
                        t0 = time.perf_counter()
                        agent.sample_actions(ob, seed=np.array([1, 2], np.uint32))
                        ts.append(time.perf_counter() - t0)
                    lat[f'rows_{rows}_us_median'] = 1e6 * float(np.median(ts))
            out['sample_actions_latency'] = dict(lat, api='FQLAgent.sample_actions(host obs) -> host actions, noise drawn on the host',
                                                 note='preallocated buffers, pinned staging, one H2D + 3 kernels + one D2H + stream sync')
        except Exception as e:
            out['sample_actions_latency'] = dict(error=repr(e)[:200])
    if n == 1 and args.precision == 'bf16' and not args.no_fp32_leg and not wl.get('image'):
        with torch.cuda.stream(stream):
            a32 = FQLAgent.create(0, np.zeros((1, F), np.float32), np.zeros((1, A), np.float32), cfg, num_seeds=args.seeds, precision='fp32')
            b32 = a32.stage(batches[0])
            for _ in range(5):
                a32.step(b32)
            torch.cuda.synchronize()
            k32 = min(K, 50)
            e32 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k32)]
            for i in range(k32):
                flush.zero_()
                e32[i][0].record()
                a32.step(b32)
                e32[i][1].record()
            torch.cuda.synchronize()
            ms32 = sum(x.elapsed_time(y) for x, y in e32) / k32
        out['fp32_parity_mode'] = dict(ms_per_step=ms32, steps_per_sec=1e3 / ms32, value=samples_per_step / (ms32 / 1e3), unit='samples/s',
                                       note='FQL_PRECISION_FP32 (FFMA everywhere, 1e-5 parity vs the fp64 oracle), same workload')
    if not args.no_cpu_baseline and n == 1:
        r = cpu_reference_arm(wl, args.batch, 50, 1, budget_s=15.0)
        cv = args.batch * 1e3 / r['ms_per_step']
        out['cpu_baseline'] = dict(value=cv, unit='samples/s', steps_per_sec=1e3 / r['ms_per_step'], cores=r['cores'], kind='port',
                                   sample=f"{r['steps_measured']} full updates at batch {args.batch}, 1 seed (median), fp32 torch-CPU "
                                          f"restatement of the reference (JAX not installable)")
    if args.dump_outputs:
        write_outputs(args.dump_outputs, outputs)
    print(json.dumps(out), flush=True)
    if world > 1:
        _shutdown(agent)
    return 0


if __name__ == '__main__':
    sys.exit(main())
