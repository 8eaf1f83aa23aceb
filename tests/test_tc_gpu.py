"""FQL_PRECISION_BF16_TC (tcgen05) path against the fp64 oracle.  Stated bf16 tolerance (north_star: "within a stated bf16
tolerance otherwise"): operands are rounded to bf16 (2^-9 relative) before every contraction, accumulation and epilogues are
fp32, master weights fp32.  Tensor-norm-relative error bounds used below:
    single 5-layer MLP output            <= 2e-2
    10-step Euler integration            <= 5e-2
    losses / metrics of one update       <= 5e-2 (relative to the scale of the quantity)
    gradients, per leaf                  <= TOL_GRAD = 4e-2  (measured worst over every case below: ~1.2e-2)
    Adam moments mu / nu, per leaf       <= 2e-2 / 3e-2
    the parameter UPDATE new - old       == the oracle's Adam/Polyak applied to the DEVICE gradients to 2e-3, and within TOL_DELTA of the
                                            reference update (tests/helpers.py::check_update_delta; an optimizer that never ran scores 1.0)
The new parameter VALUES are not compared on their own: one Adam step moves a weight by ~lr = 3e-4 against |p| ~ 0.1, so any
value-level bound a bf16 path can meet would also be met by a step that skipped the optimizer.
"""
import copy

import numpy as np
import pytest

from oracle import fql_oracle as O
from tests.helpers import check_update_delta, cuda_agent_from_state, f32, info_close, make_case, rel_err, stack_trees

pytestmark = pytest.mark.gpu
TOL_GRAD = 4e-2
TOL_DELTA = 0.9    # see check_update_delta: precision comes from (a) + TOL_GRAD; measured end-to-end 0.07-0.67


@pytest.mark.parametrize('hidden,F,A,rows', [(128, 11, 3, 40), (512, 29, 8, 256), (512, 69, 21, 300), (512, 69, 21, 1100), (512, 83, 5, 129), (256, 28, 5, 1),
                                               (128, 29, 8, 1100)])
def test_tc_forward_chains(hidden, F, A, rows):
    cfg, state, _, _ = make_case(dict(), 8, F, A, seed=hidden + rows, hidden=hidden)
    agent = cuda_agent_from_state(cfg, state, 8, F, A, precision='bf16')
    agent.load_tree(f32(state['params']))
    rng = np.random.default_rng(rows)
    obs = rng.standard_normal((rows, F))
    nz = rng.standard_normal((rows, A))
    a = agent.sample_actions(obs.astype(np.float32), noise=nz.astype(np.float32))
    ref = O.sample_actions_given_noise(state['params'], cfg, obs, nz)
    e1 = rel_err(a, ref)
    fa = agent.compute_flow_actions(obs.astype(np.float32), nz.astype(np.float32))
    ref2 = O.compute_flow_actions(state['params'], cfg, obs, nz)
    e2 = rel_err(fa, ref2)
    print(f'H={hidden} F={F} A={A} rows={rows}: sample_actions err {e1:.3e}, flow_actions err {e2:.3e}')
    assert e1 <= 2e-2 and e2 <= 5e-2


TC_CASES = [
    ('tc-small', dict(), 48, 11, 3, 128),
    ('tc-odd-batch', dict(q_agg='min'), 40, 9, 4, 128),
    ('tc-antmaze-large', dict(q_agg='min', alpha=10.0), 256, 29, 8, 512),
    ('tc-humanoidmaze', dict(discount=0.995, alpha=30.0), 256, 69, 21, 512),
    ('tc-puzzle-normq', dict(normalize_q_loss=True, alpha=1000.0), 256, 83, 5, 512),
    ('tc-ragged-512', dict(q_agg='min'), 200, 29, 8, 512),   # partial 128-row tiles in the cluster kernels
]


@pytest.mark.parametrize('name,over,B,F,A,hidden', TC_CASES, ids=[c[0] for c in TC_CASES])
def test_tc_update_step(name, over, B, F, A, hidden):
    cfg, state, batch, noise = make_case(over, B, F, A, seed=len(name), hidden=hidden)
    agent = cuda_agent_from_state(cfg, state, B, F, A, precision='bf16')
    agent.load_tree(f32(state['params']), f32(state['mu']), f32(state['nu']), state['count'])
    new_state, ref_info, ref_grads = O.update(copy.deepcopy(state), cfg, batch, noise)
    _, info = agent.update(f32(batch), noise=f32(noise))
    worst = {}
    for k in O.INFO_KEYS:
        if k.startswith('grad/'):
            r = float(ref_info[k])
            assert abs(info[k] - r) <= 0.1 * abs(r) + 1e-6, (k, info[k], r)
        else:
            info_close(k, info[k], ref_info, 5e-2)
    got = {w: agent.export_tree(w) for w in ('grads', 'params', 'mu', 'nu')}
    for which, ref, tol in (('grads', ref_grads, TOL_GRAD), ('mu', new_state['mu'], 2e-2), ('nu', new_state['nu'], 3e-2)):
        for (path, r), (_, g) in zip(O.tree_leaves(ref), O.tree_leaves(got[which])):
            e = rel_err(g, r)
            worst[which] = max(worst.get(which, 0), e)
            assert e <= tol, (which, path, e)
    worst['delta'] = check_update_delta(state['params'], new_state['params'], got['params'], TOL_DELTA, what=name,
                                        opt=dict(state=state, cfg=cfg, grads=got['grads']))
    print(name, {k: f'{v:.2e}' for k, v in worst.items()})
    # second and third step exercise graph capture / replay and the in-graph shadow refresh
    st = new_state
    for i in range(2):
        ba, nz = O.make_batch(300 + i, B, F, A, np.float64), O.make_noise(400 + i, B, A, np.float64)
        st, ref_info, _ = O.update(st, cfg, ba, nz)
        _, info = agent.update(f32(ba), noise=f32(nz))
        info_close('critic/critic_loss', info['critic/critic_loss'], ref_info, 5e-2)
        info_close('actor/distill_loss', info['actor/distill_loss'], ref_info, 8e-2)


def test_tc_unsupported_configs_fail_loudly():
    """No silent fallback: configurations the tensor-core path does not implement raise."""
    from fql_b200._lib import FqlError
    cfg, state, batch, noise = make_case(dict(actor_layer_norm=True), 32, 9, 4, seed=1, hidden=128)
    with pytest.raises(FqlError, match='actor_layer_norm'):
        agent = cuda_agent_from_state(cfg, state, 32, 9, 4, precision='bf16')
        agent.load_tree(f32(state['params']))
        agent.update(f32(batch), noise=f32(noise))
    cfg, state, batch, noise = make_case(dict(), 32, 9, 4, seed=1, hidden=96)
    with pytest.raises(FqlError, match='hidden'):
        cuda_agent_from_state(cfg, state, 32, 9, 4, precision='bf16')


def test_tc_update_two_seeds_cluster_kernels():
    """Vectorised seeds through the cluster kernels (seed strides of the activation saves, per-seed weight slices): every seed
    must match its own single-seed fp64 oracle run within the bf16 tolerance."""
    B, F, A, S = 160, 28, 5, 2
    cases = [make_case(dict(alpha=300.0), B, F, A, seed=50 + i, hidden=512) for i in range(S)]
    cfg = cases[0][0]
    agent = cuda_agent_from_state(cfg, cases[0][1], B, F, A, precision='bf16', num_seeds=S)
    cat = stack_trees
    agent.load_tree(f32(cat([c[1]['params'] for c in cases])), f32(cat([c[1]['mu'] for c in cases])), f32(cat([c[1]['nu'] for c in cases])),
                    cases[0][1]['count'])
    batch = {k: np.stack([c[2][k] for c in cases]) for k in cases[0][2]}
    noise = {k: np.stack([c[3][k] for c in cases]) for k in cases[0][3]}
    _, info = agent.update(f32(batch), noise=f32(noise))
    grads = agent.export_tree('grads')
    params = agent.export_tree('params')
    for si, (cfg_i, state, ba, nz) in enumerate(cases):
        new_state, ref_info, ref_grads = O.update(copy.deepcopy(state), cfg, ba, nz)
        for k in ('critic/critic_loss', 'actor/bc_flow_loss', 'actor/distill_loss', 'actor/q_loss'):
            info_close(k, info[k][si], ref_info, 5e-2)
        for (path, r), (_, g) in zip(O.tree_leaves(ref_grads), O.tree_leaves(grads)):
            assert rel_err(np.asarray(g)[si], r) <= TOL_GRAD, ('grads', si, path)
        check_update_delta(state['params'], new_state['params'], params, TOL_DELTA, pick=lambda x: np.asarray(x)[si], what=f'seed {si}',
                           opt=dict(state=state, cfg=cfg, grads=grads))


SWITCHES = [
    dict(FQL_B200_CLUSTER_FWD='0', FQL_B200_CLUSTER_BWD='0'),         # one-step actor layer by layer
    dict(FQL_B200_EULER_CLUSTER='0'),                                 # Euler integration layer by layer (tc_gemm Euler epilogue)
    dict(FQL_B200_CHAIN_MIN_TILES='1'),                               # large-batch routing: fused per-tile chain kernels everywhere
    dict(FQL_B200_CHAIN_MIN_TILES='1', FQL_B200_BIG_BWD='0'),         # ... with the per-layer backward (tc_gemm + LayerNorm row kernels)
    dict(FQL_B200_CHAIN_MIN_TILES='1', FQL_B200_CHAIN2_W3D='0'),      # ... with four 2-D weight boxes per stage instead of one 3-D box
    dict(FQL_B200_GRAPH='0'),                                         # every step enqueued eagerly
]


@pytest.mark.parametrize('env', SWITCHES, ids=['+'.join(f'{k[9:]}={v}' for k, v in e.items()) for e in SWITCHES])
def test_tc_alternative_schedules_match_oracle(env, monkeypatch):
    """Every alternative code path behind a schedule switch computes the same update (stated bf16 tolerance vs the fp64 oracle)."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)                                      # read by fql_context_create
    B, F, A = 256, 29, 8
    cfg, state, batch, noise = make_case(dict(q_agg='min', alpha=10.0), B, F, A, seed=31, hidden=512)
    agent = cuda_agent_from_state(cfg, state, B, F, A, precision='bf16')
    agent.load_tree(f32(state['params']), f32(state['mu']), f32(state['nu']), state['count'])
    st = copy.deepcopy(state)
    for i in range(3):                                                # eager call, graph capture, graph replay
        ba, nz = (batch, noise) if i == 0 else (O.make_batch(500 + i, B, F, A, np.float64), O.make_noise(600 + i, B, A, np.float64))
        prev = copy.deepcopy(st['params'])
        st, ref_info, ref_grads = O.update(st, cfg, ba, nz)
        _, info = agent.update(f32(ba), noise=f32(nz))
        if i == 0:
            check_update_delta(prev, st['params'], agent.export_tree('params'), TOL_DELTA, what=str(env))
        for k in ('critic/critic_loss', 'actor/bc_flow_loss', 'actor/distill_loss', 'actor/q_loss', 'actor/mse'):
            info_close(k, info[k], ref_info, 8e-2 if k == 'actor/distill_loss' else 5e-2)
        if i == 0:
            for (path, r), (_, g) in zip(O.tree_leaves(ref_grads), O.tree_leaves(agent.export_tree('grads'))):
                assert rel_err(g, r) <= TOL_GRAD, ('grads', path, rel_err(g, r))
    # after three steps the accumulated movement (3 x ~lr) against the oracle's: still a delta check, from the initial parameters
    check_update_delta(state['params'], st['params'], agent.export_tree('params'), TOL_DELTA, what=f'{env} 3 steps')
