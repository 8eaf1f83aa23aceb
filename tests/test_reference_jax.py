"""Pins the oracle to the REAL reference on a machine with jax + flax + optax + ml_collections and a checkout of the reference FQL
implementation named by FQL_REFERENCE_PATH: imports $FQL_REFERENCE_PATH/agents/fql.py unmodified, loads the oracle's parameters into
its TrainState, reproduces the five noise draws of one update with the reference's own key derivation (agents/fql.py:100,24,143,49,62,82
-- SURVEY 8a "RNG derivation"), and compares losses, gradients and the updated parameters of `agent.update(batch)` with
oracle/fql_oracle.py on the same inputs.

Without those packages or that checkout the test SKIPS: the oracle stays "parity unpinned" (DESIGN.md section 2) until this test has
run green somewhere."""
import copy
import os
import sys

import numpy as np
import pytest

jax = pytest.importorskip('jax')
pytest.importorskip('flax')
pytest.importorskip('optax')
pytest.importorskip('ml_collections')

REF = os.environ.get('FQL_REFERENCE_PATH', '')
if not REF or not os.path.isfile(os.path.join(REF, 'agents', 'fql.py')):
    pytest.skip('FQL_REFERENCE_PATH does not name a checkout of the reference FQL implementation', allow_module_level=True)

from oracle import fql_oracle as O  # noqa: E402
from tests.helpers import make_case, rel_err  # noqa: E402


def _reference_noise(key, B, A):
    """The five draws of FQLAgent.update for agent.rng == key, exactly as the reference splits its keys."""
    import jax.random as jr
    new_rng, rng = jr.split(key)                      # update(): fql.py:125
    rng, actor_rng, critic_rng = jr.split(rng, 3)     # total_loss(): fql.py:100
    _, sample_rng = jr.split(critic_rng)              # critic_loss(): fql.py:24
    k1, _ = jr.split(sample_rng)                      # sample_actions(): fql.py:143 (action_seed, noise_seed) -- noise uses the first
    z_next = jr.normal(k1, (B, A))
    rng2, x_rng, t_rng = jr.split(actor_rng, 3)       # actor_loss(): fql.py:49
    x0 = jr.normal(x_rng, (B, A))
    t = jr.uniform(t_rng, (B, 1))
    rng3, noise_rng = jr.split(rng2)                  # fql.py:62
    z = jr.normal(noise_rng, (B, A))
    k2, _ = jr.split(rng3)                            # sample_actions(seed=rng): fql.py:82 -> :143
    z_metric = jr.normal(k2, (B, A))
    return {k: np.asarray(v, np.float64) for k, v in dict(z_next=z_next, x0=x0, t=t, z=z, z_metric=z_metric).items()}


@pytest.mark.parametrize('over', [dict(), dict(q_agg='min', alpha=10.0), dict(normalize_q_loss=True, alpha=1000.0)],
                         ids=['default', 'min', 'normq'])
def test_oracle_matches_reference_update(over):
    sys.path.insert(0, REF)
    try:
        from agents.fql import FQLAgent, get_config
    finally:
        sys.path.remove(REF)
    import jax.numpy as jnp
    B, F, A, H = 32, 11, 4, 64
    cfg, state, batch, _ = make_case(over, B, F, A, seed=5, hidden=H, warm=False)
    rcfg = get_config()
    for k, v in cfg.items():
        if k in rcfg:
            rcfg[k] = v
    rcfg['actor_hidden_dims'] = rcfg['value_hidden_dims'] = (H,) * 4
    b32 = {k: np.asarray(v, np.float32) for k, v in batch.items()}
    agent = FQLAgent.create(0, b32['observations'][:1], b32['actions'][:1], rcfg)
    # same parameter tree (names and shapes must already agree: that is part of what this test pins)
    ref_params = jax.tree_util.tree_map(np.asarray, agent.network.params)
    mine = O.cast_tree(state['params'], np.float32)
    flat_ref = dict(O.tree_leaves(ref_params))
    flat_mine = dict(O.tree_leaves(mine))
    assert set(flat_ref) == set(flat_mine), set(flat_ref) ^ set(flat_mine)
    for k in flat_ref:
        assert flat_ref[k].shape == flat_mine[k].shape, (k, flat_ref[k].shape, flat_mine[k].shape)
    network = agent.network.replace(params=jax.tree_util.tree_map(jnp.asarray, mine))
    agent = agent.replace(network=network)
    noise = _reference_noise(agent.rng, B, A)
    new_agent, info = agent.update({k: jnp.asarray(v) for k, v in b32.items()})
    new_state, ref_info, _ = O.update(copy.deepcopy(state), cfg, batch, noise)
    for k in O.INFO_KEYS:
        r, g = float(ref_info[k]), float(info[k])
        assert abs(g - r) <= 2e-4 * max(abs(r), 1e-3), (k, g, r)
    got = jax.tree_util.tree_map(np.asarray, new_agent.network.params)
    for (path, r), (_, g) in zip(O.tree_leaves(new_state['params']), O.tree_leaves(got)):
        assert rel_err(g, r) <= 1e-5, (path, rel_err(g, r))
