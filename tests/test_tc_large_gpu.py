"""FQL_PRECISION_BF16_TC at the sizes north_star names (BASELINE configs 3 and 4), where the large-batch routing is reached
naturally: per-tile fused chain kernels (hidden 512, seeds x 128-row tiles >= 48), multi-CTA loss reductions with atomics, two-stage column
sums, and the clusters-of-8 fallback of the cluster kernels (more row tiles than the GPU holds clusters of 16).

The fp64 oracle cannot run 16384 rows in seconds, so the batch is R copies of one 256-row block: every loss is a batch mean, so
info, gradients and the Adam update of the big batch equal those of the block (size-independent property) -- while the kernels
see R distinct tiles and have to reduce over all of them."""
import copy

import numpy as np
import pytest

from oracle import fql_oracle as O
from tests.helpers import check_update_delta, cuda_agent_from_state, f32, info_close, make_case, rel_err, stack_trees

pytestmark = pytest.mark.gpu
TOL_GRAD, TOL_DELTA = 4e-2, 0.9


def _check(agent, agent_cfg, info, state, new_state, ref_info, ref_grads, what):
    for k in O.INFO_KEYS[:10]:
        info_close(k, info[k], ref_info, 5e-2)
    worst = 0.0
    for (path, r), (_, g) in zip(O.tree_leaves(ref_grads), O.tree_leaves(agent.export_tree('grads'))):
        e = rel_err(g, r)
        worst = max(worst, e)
        assert e <= TOL_GRAD, (what, 'grads', path, e)
    d = check_update_delta(state['params'], new_state['params'], agent.export_tree('params'), TOL_DELTA, what=what,
                           opt=dict(state=state, cfg=agent_cfg, grads=agent.export_tree('grads')))
    print(f'{what}: worst grad err {worst:.2e}, worst update err {d:.2e}')


@pytest.mark.parametrize('B,block,hidden', [(8192, 256, 512), (16384, 256, 512), (1000, 250, 512), (6144, 256, 256)],
                         ids=['B8192', 'B16384', 'B1000-ragged-nc8', 'B6144-h256'])
def test_tc_large_batch_update(B, block, hidden):
    """humanoidmaze-medium shape (config 3).  B=1000 = 7 full tiles + 104 rows: 8 row tiles > 7 clusters of 16 -> clusters of 8.
    hidden=256 at 48 row tiles: the fused chains are hidden-512 only, so the whole step runs layer by layer through tc_gemm at large M."""
    F, A = 69, 21
    cfg, state, batch, noise = make_case(dict(discount=0.995, alpha=30.0), block, F, A, seed=B % 997, hidden=hidden)
    new_state, ref_info, ref_grads = O.update(copy.deepcopy(state), cfg, batch, noise)
    rep = B // block
    big_b = {k: np.concatenate([v] * rep, 0) for k, v in batch.items()}
    big_n = {k: np.concatenate([v] * rep, 0) for k, v in noise.items()}
    agent = cuda_agent_from_state(cfg, state, B, F, A, precision='bf16')
    agent.load_tree(f32(state['params']), f32(state['mu']), f32(state['nu']), state['count'])
    _, info = agent.update(f32(big_b), noise=f32(big_n))
    _check(agent, cfg, info, state, new_state, ref_info, ref_grads, f'B={B}')
    # two more steps: graph capture and replay at this size
    st = new_state
    for i in range(2):
        ba, nz = O.make_batch(700 + i, block, F, A, np.float64), O.make_noise(800 + i, block, A, np.float64)
        st, ref_info, _ = O.update(st, cfg, ba, nz)
        _, info = agent.update(f32({k: np.concatenate([v] * rep, 0) for k, v in ba.items()}), noise=f32({k: np.concatenate([v] * rep, 0) for k, v in nz.items()}))
        info_close('critic/critic_loss', info['critic/critic_loss'], ref_info, 5e-2)
        info_close('actor/bc_flow_loss', info['actor/bc_flow_loss'], ref_info, 5e-2)


def test_tc_64_seeds_puzzle():
    """Config 4: 64 vectorised agents x batch 256, normalize_q_loss.  Four distinct (params, batch, noise) cases dealt onto the 64
    seed slots in a non-periodic pattern: a seed that read a neighbour's weights, batch or accumulators would land on another case."""
    B, F, A, S = 256, 83, 5, 64
    over = dict(normalize_q_loss=True, alpha=1000.0)
    cases = [make_case(over, B, F, A, seed=90 + i, hidden=512) for i in range(4)]
    cfg = cases[0][0]
    refs = [O.update(copy.deepcopy(c[1]), cfg, c[2], c[3]) for c in cases]
    which = [(s * s + s // 3) % 4 for s in range(S)]
    agent = cuda_agent_from_state(cfg, cases[0][1], B, F, A, precision='bf16', num_seeds=S)
    agent.load_tree(f32(stack_trees([cases[w][1]['params'] for w in which])), f32(stack_trees([cases[w][1]['mu'] for w in which])),
                    f32(stack_trees([cases[w][1]['nu'] for w in which])), cases[0][1]['count'])
    batch = {k: np.stack([cases[w][2][k] for w in which]) for k in cases[0][2]}
    noise = {k: np.stack([cases[w][3][k] for w in which]) for k in cases[0][3]}
    _, info = agent.update(f32(batch), noise=f32(noise))
    grads, params = agent.export_tree('grads'), agent.export_tree('params')
    for s in (0, 1, 2, 3, 7, 31, 32, 62, 63):
        new_state, ref_info, ref_grads = refs[which[s]]
        for k in O.INFO_KEYS[:10]:
            info_close(k, info[k][s], ref_info, 5e-2)
        for (path, r), (_, g) in zip(O.tree_leaves(ref_grads), O.tree_leaves(grads)):
            assert rel_err(np.asarray(g)[s], r) <= TOL_GRAD, ('grads', s, path, rel_err(np.asarray(g)[s], r))
        check_update_delta(cases[which[s]][1]['params'], new_state['params'], params, TOL_DELTA, pick=lambda x: np.asarray(x)[s], what=f'seed {s}',
                           opt=dict(state=cases[which[s]][1], cfg=cfg, grads=grads))
    # every seed, cheaply: the loss metrics of all 64 slots
    for s in range(S):
        for k in ('critic/critic_loss', 'actor/bc_flow_loss', 'actor/distill_loss', 'actor/q_loss'):
            info_close(k, info[k][s], refs[which[s]][1], 5e-2)

