"""Hyperparameter sweeps as vectorised seeds: FQLAgent.create(per_seed=...) / FqlHparams.per_seed.  Every seed of one multi-seed step
trains with its own alpha, discount, tau and lr and must equal the oracle run with ITS config; a table that repeats the shared values
is bit-identical to no table; the table reaches every entry point (graph replay, forward-only losses, target_update, data parallel)."""
import copy
import os
import socket

import numpy as np
import pytest
import torch

from oracle import fql_oracle as O
from tests.helpers import check_update_delta, f32, info_close, make_case, rel_err, stack_trees

pytestmark = pytest.mark.gpu
TOL = 1e-5
TOL_GRAD, TOL_DELTA = 4e-2, 0.9      # bf16 tolerances of tests/test_tc_gpu.py
SWEEP = dict(alpha=(3.0, 30.0, 300.0, 1000.0), discount=(0.99, 0.995, 0.9, 0.97), tau=(0.005, 0.05, 0.002, 0.02),
             lr=(3e-4, 1e-3, 1e-4, 6e-4))
SHAPES = {  # name: (cfg overrides, B, F, A, hidden)
    'small': (dict(), 32, 13, 5, 64),
    'config4': (dict(normalize_q_loss=True), 256, 83, 5, 512),
}


def seed_cfg(cfg, i, sweep=SWEEP):
    return dict(cfg, **{k: v[i] for k, v in sweep.items()})


def sweep_of(S):
    return {k: v[:S] for k, v in SWEEP.items()}


def make_seeds(over, B, F, A, hidden, S, seed0):
    cases = [make_case(over, B, F, A, seed=seed0 + i, hidden=hidden) for i in range(S)]
    return cases[0][0], [c[1:] for c in cases]          # cfg, [(state, batch, noise)]


def make_agent(cfg, B, F, A, S, precision, per_seed):
    from fql_b200 import FQLAgent
    return FQLAgent.create(0, np.zeros((1, F), np.float32), np.zeros((1, A), np.float32), dict(cfg, batch_size=B), num_seeds=S,
                           precision=precision, per_seed=per_seed)


def load(agent, seeds):
    agent.load_tree(f32(stack_trees([s[0]['params'] for s in seeds])), f32(stack_trees([s[0]['mu'] for s in seeds])),
                    f32(stack_trees([s[0]['nu'] for s in seeds])), seeds[0][0]['count'])


def stacked(seeds, j, rep=1):
    return f32({k: np.stack([np.concatenate([s[j][k]] * rep, 0) for s in seeds]) for k in seeds[0][j]})


def check_update_per_seed(agent, cfg, seeds, precision, rep=1):
    """tests/test_step_gpu.py::check_update (fp32 modes) or the bf16 checks of tests/test_tc_gpu.py, with seed i against O.update under
    seed_cfg(cfg, i).  rep > 1: the device batch is rep copies of each seed's block (means are replication-invariant)."""
    S = len(seeds)
    assert agent.seed_config(S - 1)['alpha'] == SWEEP['alpha'][S - 1]
    load(agent, seeds)
    _, info = agent.update(stacked(seeds, 1, rep), noise=stacked(seeds, 2, rep))
    got = {w: agent.export_tree(w) for w in ('params', 'mu', 'nu', 'grads')}
    worst = {}
    for si, (state, batch, noise) in enumerate(seeds):
        cfg_i = seed_cfg(cfg, si)
        assert agent.seed_config(si) == dict(agent.config, **{k: v[si] for k, v in SWEEP.items()})
        new_state, ref_info, ref_grads = O.update(copy.deepcopy(state), cfg_i, batch, noise)
        pick = lambda x: np.asarray(x)[si]
        if precision == 'bf16':
            for k in O.INFO_KEYS:
                if k.startswith('grad/'):
                    r = float(ref_info[k])
                    assert abs(info[k][si] - r) <= 0.1 * abs(r) + 1e-6, (si, k, info[k][si], r)
                else:
                    info_close(k, info[k][si], ref_info, 5e-2)
            checks = (('grads', ref_grads, TOL_GRAD), ('mu', new_state['mu'], 2e-2), ('nu', new_state['nu'], 3e-2))
        else:
            for k in O.INFO_KEYS:
                info_close(k, info[k][si], ref_info, 3 * TOL)
            checks = (('grads', ref_grads, TOL), ('params', new_state['params'], TOL), ('mu', new_state['mu'], TOL), ('nu', new_state['nu'], TOL))
        for which, ref, tol in checks:
            for (path, r), (_, g) in zip(O.tree_leaves(ref), O.tree_leaves(got[which])):
                e = rel_err(pick(g), r)
                worst[which] = max(worst.get(which, 0), e)
                assert e <= tol, (si, which, path, e)
        if precision == 'bf16':
            worst['delta'] = max(worst.get('delta', 0), check_update_delta(
                state['params'], new_state['params'], got['params'], TOL_DELTA, pick=pick, what=f'seed {si}',
                opt=dict(state=state, cfg=cfg_i, grads=got['grads'])))
        else:   # the parameter UPDATE itself (new - old), as check_update does
            for (path, new), (_, old), (_, g) in zip(O.tree_leaves(new_state['params']), O.tree_leaves(state['params']),
                                                     O.tree_leaves(got['params'])):
                d_ref = new - old
                d_got = pick(g).astype(np.float64) - old.astype(np.float32).astype(np.float64)
                if np.abs(d_ref).max() > 0:
                    assert rel_err(d_got, d_ref) <= 2e-3, (si, 'delta', path, rel_err(d_got, d_ref))
    return worst


PARITY = [('fp32', 'small', 1, None), ('fp32', 'config4', 1, None), ('fp32-tc', 'small', 1, None), ('fp32-tc', 'config4', 1, None),
          ('bf16', 'small', 1, None), ('bf16', 'config4', 1, None),
          ('bf16', 'config4', 1, '1'),      # FQL_B200_CHAIN_MIN_TILES=1: the fused per-tile chain kernels at batch 256
          ('bf16', 'config4', 16, '1')]     # B = 4096 (16 copies per seed): chain kernels and the multi-CTA loss kernels with atomics


@pytest.mark.parametrize('precision,shape,rep,chain', PARITY, ids=[f'{p}-{s}' + (f'-x{r}' if r > 1 else '') + ('-chain' if c else '')
                                                                for p, s, r, c in PARITY])
def test_per_seed_parity(precision, shape, rep, chain, monkeypatch):
    if chain:
        monkeypatch.setenv('FQL_B200_CHAIN_MIN_TILES', chain)       # read by fql_context_create
    over, B, F, A, hidden = SHAPES[shape]
    cfg, seeds = make_seeds(over, B, F, A, hidden, 4, seed0=70)
    agent = make_agent(cfg, B * rep, F, A, 4, precision, SWEEP)
    worst = check_update_per_seed(agent, cfg, seeds, precision, rep)
    print(precision, shape, rep, chain, {k: f'{v:.2e}' for k, v in worst.items()})


def _bits(agent, info):
    out = {w: agent.export_tree(w) for w in ('params', 'mu', 'nu', 'grads')}
    out['info'] = {k: np.asarray(info[k]).copy() for k in O.INFO_KEYS}
    return out


@pytest.mark.parametrize('precision', ['fp32', 'fp32-tc', 'bf16'])
def test_repeated_shared_values_are_bit_identical(precision):
    """A table whose every entry equals the shared config trains exactly like no table: three steps (eager, graph capture, replay)."""
    B, F, A, H, S = 128, 29, 8, 512, 2
    cfg, seeds = make_seeds(dict(q_agg='min', alpha=10.0), B, F, A, H, S, seed0=20)
    same = {k: [cfg[k]] * S for k in SWEEP}
    agents = [make_agent(cfg, B, F, A, S, precision, None), make_agent(cfg, B, F, A, S, precision, same)]
    assert agents[0].per_seed is None and agents[1].per_seed == {k: tuple(v) for k, v in same.items()}
    for ag in agents:
        load(ag, seeds)
    for i in range(3):
        ba = {k: np.stack([O.make_batch(30 + i + 7 * s, B, F, A)[k] for s in range(S)]) for k in seeds[0][1]}
        nz = {k: np.stack([O.make_noise(60 + i + 7 * s, B, A)[k] for s in range(S)]) for k in seeds[0][2]}
        res = [_bits(ag, ag.update(f32(ba), noise=f32(nz))[1]) for ag in agents]
        for w in ('params', 'mu', 'nu', 'grads'):
            for (path, x), (_, y) in zip(O.tree_leaves(res[0][w]), O.tree_leaves(res[1][w])):
                assert np.array_equal(x.view(np.uint32), y.view(np.uint32)), (i, w, path)
        for k in O.INFO_KEYS:
            assert np.array_equal(res[0]['info'][k].view(np.uint32), res[1]['info'][k].view(np.uint32)), (i, k)


def test_four_steps_and_graph_replay_with_a_table():
    """Step 1 eager, step 2 captures the CUDA graph, steps 3-4 replay it: every seed follows its own chained oracle run."""
    B, F, A, H, S = 64, 29, 8, 128, 4
    cfg, seeds = make_seeds(dict(q_agg='min'), B, F, A, H, S, seed0=3)
    agent = make_agent(cfg, B, F, A, S, 'fp32', SWEEP)
    load(agent, seeds)
    states = [copy.deepcopy(s[0]) for s in seeds]
    for i in range(4):
        bas = [O.make_batch(100 + i + 10 * s, B, F, A, np.float64) for s in range(S)]
        nzs = [O.make_noise(200 + i + 10 * s, B, A, np.float64) for s in range(S)]
        infos = []
        for s in range(S):
            states[s], info_ref, _ = O.update(states[s], seed_cfg(cfg, s), bas[s], nzs[s])
            infos.append(info_ref)
        _, info = agent.update(f32({k: np.stack([b[k] for b in bas]) for k in bas[0]}),
                               noise=f32({k: np.stack([n[k] for n in nzs]) for k in nzs[0]}))
        got = agent.export_tree('params')
        for s in range(S):
            for k in O.INFO_KEYS:
                info_close(k, info[k][s], infos[s], 5e-5)
            for (path, r), (_, g) in zip(O.tree_leaves(states[s]['params']), O.tree_leaves(got)):
                assert rel_err(np.asarray(g)[s], r) <= 1e-5 * (i + 1), (i, s, path)
    assert agent.network.step == seeds[0][0]['step'] + 4


@pytest.mark.parametrize('precision,tol', [('fp32', 3 * TOL), ('fp32-tc', 3 * TOL), ('bf16', 5e-2)])
def test_forward_only_losses_per_seed(precision, tol):
    """total_loss / actor_loss: actor/actor_loss = bc + alpha_s * distill + q_loss with each seed's own alpha (and its discount in the
    critic loss), against the oracle."""
    B, F, A, H, S = 48, 17, 6, 128, 4
    cfg, seeds = make_seeds(dict(normalize_q_loss=True), B, F, A, H, S, seed0=8)
    agent = make_agent(cfg, B, F, A, S, precision, SWEEP)
    load(agent, seeds)
    loss, info = agent.total_loss(stacked(seeds, 1), noise=stacked(seeds, 2))
    a_loss, a_info = agent.actor_loss(stacked(seeds, 1), noise=stacked(seeds, 2))
    for s, (state, batch, noise) in enumerate(seeds):
        ref_loss, ref_info, _ = O.total_loss(state['params'], seed_cfg(cfg, s), batch, noise, with_grads=False)
        for k in ref_info:
            info_close(k, info[k][s], ref_info, tol)
        assert abs(loss[s] - ref_loss) <= tol * max(abs(ref_loss), abs(float(ref_info['critic/q_max'])))
        parts = a_info['bc_flow_loss'][s] + SWEEP['alpha'][s] * a_info['distill_loss'][s] + a_info['q_loss'][s]
        assert abs(a_loss[s] - parts) <= 1e-5 * max(1.0, abs(parts)), (s, a_loss[s], parts)
        info_close('actor/actor_loss', a_loss[s], ref_info, tol)


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_target_update_per_seed_tau(precision):
    """target <- tau_s * critic + (1 - tau_s) * target per seed, bitwise equal to the fp32 evaluation of that expression on the host
    (one of its roundings: with or without the multiply-add contracted into one FMA); in bf16 the operand shadow follows."""
    B, F, A, H, S = 32, 13, 5, 64, 4
    cfg, seeds = make_seeds(dict(), B, F, A, H, S, seed0=40)
    agent = make_agent(cfg, B, F, A, S, precision, SWEEP)
    load(agent, seeds)
    c0, c1 = agent._net_range('critic')
    t0, t1 = agent._net_range('target_critic')
    n = min(c1 - c0, t1 - t0)
    before = agent._params.cpu().numpy()
    agent.target_update()
    torch.cuda.synchronize()
    after = agent._params.cpu().numpy()
    assert np.array_equal(after[:, :t0], before[:, :t0]) and np.array_equal(after[:, t1:], before[:, t1:])
    for s in range(S):
        h = agent._hp_table.cpu().numpy().view(np.float32).reshape(S, 12)[s]
        tau, omt = np.float32(SWEEP['tau'][s]), np.float32(1.0 - SWEEP['tau'][s])
        assert h[5] == tau and h[9] == omt                       # the uploaded entry: tau and 1 - tau rounded from double
        p, tp = before[s, c0:c0 + n], before[s, t0:t0 + n]
        x, y = p.astype(np.longdouble) * tau, tp.astype(np.longdouble) * omt
        cands = [(p * tau + tp * omt), (x + (tp * omt)).astype(np.float32), ((p * tau) + y).astype(np.float32)]
        got = after[s, t0:t0 + n]
        ok = np.zeros(got.shape, bool)
        for c in cands:
            ok |= c.view(np.uint32) == got.view(np.uint32)
        assert ok.all(), (s, int((~ok).sum()))
    if precision == 'bf16':
        sh = agent._shadow.clone()
        agent.refresh_shadow()                                   # rebuilt from the fp32 parameters: nothing may change
        torch.cuda.synchronize()
        assert torch.equal(sh, agent._shadow)


# ---- data parallel (two processes, one GPU each) ------------------------------------------------------------------------------------
def _port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _run2(target, *args):
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    ret = ctx.Queue()
    port = _port()
    procs = [ctx.Process(target=target, args=(r, 2, port, ret) + args) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(420)
        assert p.exitcode == 0
    return [ret.get(timeout=5) for _ in range(2)]


def _dp_batch_worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    os.environ['FQL_DP_BACKEND'] = 'peer'
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device(f'cuda:{rank}'))
    from fql_b200 import FQLAgent
    B, F, A, H, S = 256, 29, 8, 512, 2
    cfg, seeds = make_seeds(dict(q_agg='min'), B, F, A, H, S, seed0=6)
    sweep = sweep_of(S)
    agent = FQLAgent.create(0, np.zeros((1, F), np.float32), np.zeros((1, A), np.float32), dict(cfg, batch_size=B // world), num_seeds=S,
                            process_group=dist.group.WORLD, per_seed=sweep)
    ref = FQLAgent.create(0, np.zeros((1, F), np.float32), np.zeros((1, A), np.float32), dict(cfg, batch_size=B), num_seeds=S, per_seed=sweep)
    assert agent._dp_peer
    load(agent, seeds)
    load(ref, seeds)
    rows = lambda d: {k: v[:, rank * (B // world):(rank + 1) * (B // world)] for k, v in d.items()}
    for i in range(3):                                   # eager, graph capture, graph replay
        ba = stacked([(None, O.make_batch(40 + i + 5 * s, B, F, A), None) for s in range(S)], 1)
        nz = stacked([(None, None, O.make_noise(50 + i + 5 * s, B, A)) for s in range(S)], 2)
        _, info = agent.update(rows(ba), noise=rows(nz))
        _, info_ref = ref.update(ba, noise=nz)
        for s in range(S):
            for k in O.INFO_KEYS[:10]:
                info_close(k, info[k][s], {k2: info_ref[k2][s] for k2 in O.INFO_KEYS}, 3e-5)
        for w in ('grads', 'params', 'mu', 'nu'):
            for (path, r), (_, g) in zip(O.tree_leaves(ref.export_tree(w)), O.tree_leaves(agent.export_tree(w))):
                assert rel_err(g, r) <= TOL * (i + 1), (i, w, path, rel_err(g, r))
    mine = agent._params.view(torch.int32).sum(dtype=torch.int64).reshape(1)
    both = [torch.zeros_like(mine) for _ in range(world)]
    dist.all_gather(both, mine)
    assert all(int(x) == int(both[0]) for x in both), [int(x) for x in both]     # replicas bit-identical
    ret.put('ok')
    torch.cuda.synchronize()
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs 2 GPUs')
def test_batch_sharded_two_ranks_with_a_table():
    """Data parallel over the batch (peer-memory backend), two seeds with their own hyperparameters: every rank holds the 1-GPU step of
    the global batch (1e-5, fp32) and the replicas stay bit-identical."""
    assert _run2(_dp_batch_worker) == ['ok', 'ok']


def _seed_shard_worker(rank, world, port, ret):
    from fql_b200 import dist as fdist
    torch.cuda.set_device(rank)
    B, F, A, H, S = 64, 29, 8, 128, 4
    cfg, seeds = make_seeds(dict(q_agg='min'), B, F, A, H, S, seed0=11)
    mine = fdist.shard_seeds(S, rank, world)
    full = make_agent(cfg, B, F, A, S, 'fp32', SWEEP)
    part = make_agent(cfg, B, F, A, len(mine), 'fp32', fdist.shard_per_seed(SWEEP, rank, world))
    load(full, seeds)
    load(part, [seeds[s] for s in mine])
    bitwise = True
    for i in range(2):
        ba = stacked([(None, O.make_batch(90 + i + 3 * s, B, F, A), None) for s in range(S)], 1)
        nz = stacked([(None, None, O.make_noise(80 + i + 3 * s, B, A)) for s in range(S)], 2)
        full.update(ba, noise=nz)
        part.update({k: v[mine.start:mine.stop] for k, v in ba.items()}, noise={k: v[mine.start:mine.stop] for k, v in nz.items()})
        for w in ('grads', 'params', 'mu', 'nu'):
            for (path, r), (_, g) in zip(O.tree_leaves(full.export_tree(w)), O.tree_leaves(part.export_tree(w))):
                for j, s in enumerate(mine):
                    assert rel_err(np.asarray(g)[j], np.asarray(r)[s]) <= TOL, (i, w, s, path)
                    bitwise &= np.array_equal(np.asarray(g)[j], np.asarray(r)[s])
    for j, s in enumerate(mine):
        assert part.seed_config(j) == full.seed_config(s)
    ret.put((rank, bitwise))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs 2 GPUs')
def test_seed_sharded_sweep_over_two_ranks():
    """Four agents of a sweep over two ranks (shard_per_seed): every rank's agents equal the matching seeds of the one-GPU 4-seed run."""
    res = dict(_run2(_seed_shard_worker))
    print('seed-sharded sweep bitwise equal to the 1-GPU run:', res)


def test_a_host_table_is_refused():
    """FqlHparams.per_seed must be device memory: a host array is reported as an error before anything is enqueued."""
    from fql_b200 import _lib
    B, F, A, H, S = 32, 13, 5, 64, 2
    cfg, seeds = make_seeds(dict(), B, F, A, H, S, seed0=1)
    agent = make_agent(cfg, B, F, A, S, 'fp32', sweep_of(S))
    host = np.zeros(S * 12, np.float32)
    agent._hp.per_seed = host.ctypes.data
    with pytest.raises(_lib.FqlError, match='device memory'):
        agent.update(stacked(seeds, 1), noise=stacked(seeds, 2))
    with pytest.raises(_lib.FqlError, match='device memory'):
        agent.target_update()
