"""CPU oracle for FQLAgent.update -- TEST INFRASTRUCTURE ONLY.

This is a NumPy restatement of the reference algorithm (zhouzypaul/fql).  It is the
*checker* for the CUDA path: only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may import it.  The
product package ``fql_b200`` never imports anything under ``oracle/``.

PARITY UNPINNED: the reference ships no tests, golden vectors or fixtures, and its
arithmetic lives in un-vendored jax/flax/optax (not installed in this image), so this
restatement cannot be pinned against the reference's own outputs.  It is instead
cross-validated (tests/test_oracle.py) by (a) central finite differences in fp64 and
(b) an independent torch-autograd transcription of the same losses.

Reference citations (relative to /root/reference):
  agents/fql.py:22-44     critic_loss
  agents/fql.py:46-92     actor_loss
  agents/fql.py:94-111    total_loss
  agents/fql.py:113-120   target_update (Polyak from the PRE-step critic)
  agents/fql.py:122-133   update
  agents/fql.py:135-153   sample_actions
  agents/fql.py:155-171   compute_flow_actions (Euler)
  utils/networks.py:34-61   MLP  (Dense -> GELU(tanh) -> LayerNorm(eps=1e-6))
  utils/networks.py:153-195 Value (2-head ensemble, params stacked on axis 0)
  utils/networks.py:198-235 ActorVectorField
  utils/flax_utils.py:120-159 apply_gradients / apply_loss_fn (grad stats, optax.adam)

Every function is dtype-parametric: pass float64 arrays for ground truth, float32 arrays
for the "reference JAX CPU" stand-in (fp32 end to end, like XLA:CPU).
Noise (z_next, x0, t, z, z_metric) is an explicit input; RNG never enters parity.
"""
from __future__ import annotations

import math

import numpy as np

NETS = ('modules_actor_bc_flow', 'modules_actor_onestep_flow', 'modules_critic', 'modules_target_critic')
INFO_KEYS = (
    'critic/critic_loss', 'critic/q_mean', 'critic/q_max', 'critic/q_min',
    'actor/actor_loss', 'actor/bc_flow_loss', 'actor/distill_loss', 'actor/q_loss', 'actor/q', 'actor/mse',
    'grad/max', 'grad/min', 'grad/norm',
)

DEFAULT_CONFIG = dict(  # agents/fql.py:249-270
    agent_name='fql', lr=3e-4, batch_size=256,
    actor_hidden_dims=(512, 512, 512, 512), value_hidden_dims=(512, 512, 512, 512),
    layer_norm=True, actor_layer_norm=False, discount=0.99, tau=0.005, q_agg='mean',
    alpha=300.0, flow_steps=10, normalize_q_loss=False, encoder=None,
)

_GELU_C = math.sqrt(2.0 / math.pi)
_GELU_A = 0.044715
LN_EPS = 1e-6  # flax.linen.LayerNorm default


# --------------------------------------------------------------------------------------
# elementwise pieces
# --------------------------------------------------------------------------------------
def gelu_tanh(x):
    """flax nn.gelu default (approximate=True); utils/networks.py:46."""
    dt = x.dtype.type
    u = dt(_GELU_C) * (x + dt(_GELU_A) * x * x * x)
    return dt(0.5) * x * (dt(1.0) + np.tanh(u))


def gelu_tanh_grad(x):
    dt = x.dtype.type
    x2 = x * x
    u = dt(_GELU_C) * (x + dt(_GELU_A) * x2 * x)
    th = np.tanh(u)
    du = dt(_GELU_C) * (dt(1.0) + dt(3.0 * _GELU_A) * x2)
    return dt(0.5) * (dt(1.0) + th) + dt(0.5) * x * (dt(1.0) - th * th) * du


def layer_norm_fwd(g, scale, bias):
    """flax nn.LayerNorm(): eps 1e-6, use_fast_variance (var = E[x^2]-E[x]^2 clamped at 0)."""
    dt = g.dtype.type
    mu = g.mean(axis=-1, keepdims=True)
    var = np.maximum(dt(0.0), (g * g).mean(axis=-1, keepdims=True) - mu * mu)
    rstd = dt(1.0) / np.sqrt(var + dt(LN_EPS))
    xhat = (g - mu) * rstd
    return xhat * scale + bias, xhat, rstd


def layer_norm_bwd(dh, xhat, rstd, scale):
    dxhat = dh * scale
    m1 = dxhat.mean(axis=-1, keepdims=True)
    m2 = (dxhat * xhat).mean(axis=-1, keepdims=True)
    dg = rstd * (dxhat - m1 - xhat * m2)
    return dg


# --------------------------------------------------------------------------------------
# MLP (utils/networks.py:34-61); `p` is {'Dense_i': {'kernel','bias'}, 'LayerNorm_i': {'scale','bias'}}
# Works for a plain MLP (kernel [in,out]) and for an ensemble (kernel [E,in,out]) via matmul broadcasting.
# --------------------------------------------------------------------------------------
def n_dense(p):
    return sum(1 for k in p if k.startswith('Dense_'))


def mlp_forward(p, x, layer_norm, save=False, q=None):
    """q: optional storage rounding of the contraction operands (e.g. to bf16), applied to every kernel and to every layer's
    input; the bias, the pre-activations and everything after them stay in the array dtype.  None (the default) rounds nothing."""
    n = n_dense(p)
    ens = p['Dense_0']['kernel'].ndim == 3
    cache = []
    h = x
    for i in range(n):
        W, b = p[f'Dense_{i}']['kernel'], p[f'Dense_{i}']['bias']
        z = (np.matmul(h, W) if q is None else np.matmul(q(h), q(W))) + (b[:, None, :] if ens else b)
        if i + 1 < n:
            g = gelu_tanh(z)
            if layer_norm:
                sc, bi = p[f'LayerNorm_{i}']['scale'], p[f'LayerNorm_{i}']['bias']
                if ens:
                    sc, bi = sc[:, None, :], bi[:, None, :]
                hn, xhat, rstd = layer_norm_fwd(g, sc, bi)
            else:
                hn, xhat, rstd = g, None, None
            if save:
                cache.append((h, z, xhat, rstd))
            h = hn
        else:
            if save:
                cache.append((h, z, None, None))
            h = z
    return (h, cache) if save else h


def mlp_backward(p, cache, dout, layer_norm, need_dx=True, need_dw=True):
    """Returns (grads-with-the-layout-of-p or None, dx or None)."""
    n = n_dense(p)
    ens = p['Dense_0']['kernel'].ndim == 3
    grads = {} if need_dw else None
    dz = dout
    dx = None
    for i in reversed(range(n)):
        h_in, z, xhat, rstd = cache[i]
        if i + 1 < n:
            # dz currently holds dL/dh_i (post-activation/LN output of layer i)
            dh = dz
            if layer_norm:
                sc = p[f'LayerNorm_{i}']['scale']
                scb = sc[:, None, :] if ens else sc
                if need_dw:
                    red = 1 if ens else 0
                    grads[f'LayerNorm_{i}'] = {'scale': (dh * xhat).sum(axis=red), 'bias': dh.sum(axis=red)}
                dg = layer_norm_bwd(dh, xhat, rstd, scb)
            else:
                dg = dh
            dz = dg * gelu_tanh_grad(z)
        W = p[f'Dense_{i}']['kernel']
        if need_dw:
            h_b = np.broadcast_to(h_in, dz.shape[:-1] + h_in.shape[-1:]) if ens and h_in.ndim == 2 else h_in
            grads[f'Dense_{i}'] = {
                'kernel': np.matmul(np.swapaxes(h_b, -1, -2), dz),
                'bias': dz.sum(axis=-2),
            }
        if i > 0 or need_dx:
            dz = np.matmul(dz, np.swapaxes(W, -1, -2))
            if i == 0:
                dx = dz
    return grads, dx


# --------------------------------------------------------------------------------------
# modules
# --------------------------------------------------------------------------------------
def actor_forward(net_p, cfg, obs, actions, times=None, save=False, q=None):
    """ActorVectorField.__call__ (utils/networks.py:216-235), state-based (no encoder)."""
    parts = [obs, actions] if times is None else [obs, actions, times]
    x = np.concatenate(parts, axis=-1)
    return mlp_forward(net_p['mlp'], x, cfg['actor_layer_norm'], save=save, q=q)


def critic_forward(net_p, cfg, obs, actions, save=False):
    """Value.__call__ (utils/networks.py:178-195): out [2,B]."""
    x = np.concatenate([obs, actions], axis=-1)
    r = mlp_forward(net_p['value_net'], x, cfg['layer_norm'], save=save)
    if save:
        return r[0][..., 0], r[1]
    return r[..., 0]


def sample_actions_given_noise(params, cfg, obs, noise, q=None):
    """agents/fql.py:135-153 with the noise draw made explicit (q: see mlp_forward)."""
    a = actor_forward(params['modules_actor_onestep_flow'], cfg, obs, noise, q=q)
    return np.clip(a, -1, 1)


def compute_flow_actions(params, cfg, obs, noises, q=None):
    """agents/fql.py:155-171.  q (see mlp_forward) rounds each step's network input, so the velocity field sees the rounded copy of
    the actions and of the time while the Euler state itself keeps the array dtype."""
    dt = obs.dtype.type
    n = cfg['flow_steps']
    a = noises
    for i in range(n):
        t = np.full(obs.shape[:-1] + (1,), i / n, dtype=obs.dtype)  # python float -> array dtype (fql.py:167)
        v = actor_forward(params['modules_actor_bc_flow'], cfg, obs, a, t, q=q)
        a = a + v / dt(n)
    return np.clip(a, -1, 1)


# --------------------------------------------------------------------------------------
# losses + manual gradient  (agents/fql.py:22-111)
# --------------------------------------------------------------------------------------
def _zeros_like_tree(t):
    if isinstance(t, dict):
        return {k: _zeros_like_tree(v) for k, v in t.items()}
    return np.zeros_like(t)


def total_loss(params, cfg, batch, noise, with_grads=True, feats=None):
    """Returns (loss, info[10 keys], grads-or-None).  grads has the full tree of `params`
    (target critic gradients are exactly zero, SURVEY F7).

    feats (pixel configs, oracle/fql_pixel_oracle.py): encoder outputs that stand in for the observations, per call site:
    {'O_next','O','T_next','C','F'} = onestep(next_obs), onestep(obs), target_critic(next_obs), critic(obs), bc_flow(obs).
    With feats the function returns a 4th value: the gradients w.r.t. feats['C'], feats['F'], feats['O']."""
    act = batch['actions']
    if feats is None:
        obs_C = obs_F = obs_O = batch['observations']
        nobs_O = nobs_T = batch['next_observations']
    else:
        obs_C, obs_F, obs_O, nobs_O, nobs_T = feats['C'], feats['F'], feats['O'], feats['O_next'], feats['T_next']
    obs, nobs = obs_C, nobs_T
    rew, masks = batch['rewards'], batch['masks']
    dt = act.dtype.type
    B, A = act.shape
    Fdim = obs.shape[-1]
    info = {}

    # ---- critic loss (fql.py:22-44)
    next_a = sample_actions_given_noise(params, cfg, nobs_O, noise['z_next'])
    next_a = np.clip(next_a, -1, 1)
    next_qs = critic_forward(params['modules_target_critic'], cfg, nobs, next_a)
    next_q = next_qs.min(axis=0) if cfg['q_agg'] == 'min' else next_qs.mean(axis=0)
    target_q = rew + dt(cfg['discount']) * masks * next_q
    q, c_cache = critic_forward(params['modules_critic'], cfg, obs, act, save=True)
    diff = q - target_q
    critic_loss = (diff * diff).mean()
    info['critic/critic_loss'] = critic_loss
    info['critic/q_mean'] = q.mean()
    info['critic/q_max'] = q.max()
    info['critic/q_min'] = q.min()

    # ---- actor loss (fql.py:46-92)
    x0, t = noise['x0'], noise['t']
    x1 = act
    x_t = (dt(1) - t) * x0 + t * x1
    vel = x1 - x0
    pred, f_cache = actor_forward(params['modules_actor_bc_flow'], cfg, obs_F, x_t, t, save=True)
    bc_diff = pred - vel
    bc_flow_loss = (bc_diff * bc_diff).mean()

    z = noise['z']
    target_flow = compute_flow_actions(params, cfg, obs_F, z)
    a_pi, o_cache = actor_forward(params['modules_actor_onestep_flow'], cfg, obs_O, z, save=True)
    d_diff = a_pi - target_flow
    distill_loss = (d_diff * d_diff).mean()

    a_clip = np.clip(a_pi, -1, 1)
    qs_pi, cpi_cache = critic_forward(params['modules_critic'], cfg, obs, a_clip, save=True)
    q_pi = qs_pi.mean(axis=0)
    q_loss = -q_pi.mean()
    lam = dt(1.0)
    if cfg['normalize_q_loss']:
        lam = dt(1.0) / np.abs(q_pi).mean()
        q_loss = lam * q_loss
    actor_loss = bc_flow_loss + dt(cfg['alpha']) * distill_loss + q_loss

    metric_a = sample_actions_given_noise(params, cfg, obs_O, noise['z_metric'])
    mse = ((metric_a - act) ** 2).mean()
    info['actor/actor_loss'] = actor_loss
    info['actor/bc_flow_loss'] = bc_flow_loss
    info['actor/distill_loss'] = distill_loss
    info['actor/q_loss'] = q_loss
    info['actor/q'] = q_pi.mean()
    info['actor/mse'] = mse
    loss = critic_loss + actor_loss
    if not with_grads:
        return (loss, info, None) if feats is None else (loss, info, None, None)

    need_dx = feats is not None
    grads = _zeros_like_tree(params)
    # critic <- critic_loss only
    dq = (dt(2.0) / dt(q.size)) * diff                              # [2,B]
    g_c, dx_C = mlp_backward(params['modules_critic']['value_net'], c_cache, dq[..., None], cfg['layer_norm'], need_dx=need_dx)
    grads['modules_critic']['value_net'] = g_c
    # bc flow <- bc_flow_loss only
    dpred = (dt(2.0) / dt(B * A)) * bc_diff
    g_f, dx_F = mlp_backward(params['modules_actor_bc_flow']['mlp'], f_cache, dpred, cfg['actor_layer_norm'], need_dx=need_dx)
    grads['modules_actor_bc_flow']['mlp'] = g_f
    # onestep <- alpha*distill + q_loss (through clip and the critic's input gradient; critic weights get nothing)
    dqs = np.full_like(qs_pi, -lam / dt(2 * B))
    _, dx_c = mlp_backward(params['modules_critic']['value_net'], cpi_cache, dqs[..., None], cfg['layer_norm'],
                           need_dx=True, need_dw=False)
    da_clip = dx_c.sum(axis=0)[:, -A:]                               # sum over the 2 heads (input was broadcast)
    inside = ((a_pi >= -1) & (a_pi <= 1)).astype(obs.dtype)
    da_pi = dt(cfg['alpha']) * (dt(2.0) / dt(B * A)) * d_diff + da_clip * inside
    g_o, dx_O = mlp_backward(params['modules_actor_onestep_flow']['mlp'], o_cache, da_pi, cfg['actor_layer_norm'], need_dx=need_dx)
    grads['modules_actor_onestep_flow']['mlp'] = g_o
    if feats is None:
        return loss, info, grads
    dfeat = {'C': dx_C.sum(axis=0)[:, :Fdim], 'F': dx_F[:, :Fdim], 'O': dx_O[:, :Fdim]}   # critic input is broadcast to both heads
    return loss, info, grads, dfeat


# --------------------------------------------------------------------------------------
# tree helpers, grad stats, Adam, Polyak, update
# --------------------------------------------------------------------------------------
def tree_leaves(t, prefix=()):
    """Leaves in jax order (dict keys sorted)."""
    if isinstance(t, dict):
        out = []
        for k in sorted(t):
            out += tree_leaves(t[k], prefix + (k,))
        return out
    return [(prefix, t)]


def tree_map(f, *ts):
    if isinstance(ts[0], dict):
        return {k: tree_map(f, *[t[k] for t in ts]) for k in ts[0]}
    return f(*ts)


def grad_stats(grads):
    """utils/flax_utils.py:139-149: max of per-leaf max, min of per-leaf min, L1 norm of per-leaf L2 norms."""
    leaves = [g for _, g in tree_leaves(grads)]
    dt = leaves[0].dtype.type
    gmax = max(l.max() for l in leaves)
    gmin = min(l.min() for l in leaves)
    norms = np.array([np.sqrt((l.astype(l.dtype) ** 2).sum()) for l in leaves], dtype=leaves[0].dtype)
    return dt(gmax), dt(gmin), dt(np.abs(norms).sum())


def adam_update(params, grads, mu, nu, count, lr, b1=0.9, b2=0.999, eps=1e-8):
    """optax.adam (scale_by_adam + scale(-lr)) then optax.apply_updates; count is the PRE-update int32.
    optax's bias_correction evaluates `1 - decay**count` with a Python-float decay and an int32 count array, i.e. in
    float32 (jax default dtype) -- pow(0.999f, t) -- and that is restated here in float32 for every oracle dtype: at
    small t it differs from the double value by ~1e-5 relative, which is the reference's arithmetic, not noise."""
    t = count + 1
    bc1 = np.float32(1) - np.power(np.float32(b1), np.float32(t))
    bc2 = np.float32(1) - np.power(np.float32(b2), np.float32(t))

    def leaf(p, g, m, v):
        dt = p.dtype.type
        m2 = dt(b1) * m + dt(1 - b1) * g
        v2 = dt(b2) * v + dt(1 - b2) * g * g
        mhat = m2 / dt(bc1)
        vhat = v2 / dt(bc2)
        upd = -dt(lr) * (mhat / (np.sqrt(vhat) + dt(eps)))
        return p + upd, m2, v2

    trip = tree_map(leaf, params, grads, mu, nu)
    return _unzip(trip, 0), _unzip(trip, 1), _unzip(trip, 2), t


def _unzip(t, i):
    if isinstance(t, dict):
        return {k: _unzip(v, i) for k, v in t.items()}
    return t[i]


def update(state, cfg, batch, noise):
    """agents/fql.py:122-133.  state = {'params','mu','nu','count','step'}; returns (new_state, info[13])."""
    params = state['params']
    loss, info, grads = total_loss(params, cfg, batch, noise, with_grads=True)
    gmax, gmin, gnorm = grad_stats(grads)
    info['grad/max'], info['grad/min'], info['grad/norm'] = gmax, gmin, gnorm
    new_p, new_m, new_v, new_count = adam_update(params, grads, state['mu'], state['nu'], state['count'], cfg['lr'])
    # Polyak from the PRE-step critic and PRE-step target (fql.py:113-120, SURVEY F6)
    dt = batch['observations'].dtype.type
    tau = dt(cfg['tau'])
    new_p['modules_target_critic'] = tree_map(
        lambda p, tp: p * tau + tp * (dt(1) - tau), params['modules_critic'], params['modules_target_critic'])
    new_state = dict(params=new_p, mu=new_m, nu=new_v, count=new_count, step=state['step'] + 1)
    return new_state, info, grads


# --------------------------------------------------------------------------------------
# construction of synthetic state / batches (shared by tests, goldens and bench's CPU leg)
# --------------------------------------------------------------------------------------
def glorot_uniform(rng, shape, dtype):
    """variance_scaling(1,'fan_avg','uniform') (utils/networks.py:9-11); ensemble axis excluded from fans."""
    fan_in, fan_out = shape[-2], shape[-1]
    lim = math.sqrt(6.0 / (fan_in + fan_out))
    return rng.uniform(-lim, lim, size=shape).astype(dtype)


def init_mlp(rng, in_dim, dims, layer_norm, ens=None, dtype=np.float32, jitter=0.0):
    p = {}
    d = in_dim
    pre = () if ens is None else (ens,)
    for i, o in enumerate(dims):
        p[f'Dense_{i}'] = {'kernel': glorot_uniform(rng, pre + (d, o), dtype),
                           'bias': (jitter * rng.standard_normal(pre + (o,))).astype(dtype)}
        if layer_norm and i + 1 < len(dims):
            p[f'LayerNorm_{i}'] = {'scale': (1.0 + jitter * rng.standard_normal(pre + (o,))).astype(dtype),
                                   'bias': (jitter * rng.standard_normal(pre + (o,))).astype(dtype)}
        d = o
    return p


def init_params(seed, obs_dim, action_dim, cfg, dtype=np.float32, jitter=0.0, target_equals_critic=True):
    """Parameter tree with the reference layout (SURVEY 8a).  jitter>0 perturbs biases / LN params away from
    their init values so that every code path is exercised in parity tests."""
    rng = np.random.default_rng(seed)
    ah, vh = tuple(cfg['actor_hidden_dims']), tuple(cfg['value_hidden_dims'])
    F, A = obs_dim, action_dim
    params = {
        'modules_actor_bc_flow': {'mlp': init_mlp(rng, F + A + 1, ah + (A,), cfg['actor_layer_norm'], None, dtype, jitter)},
        'modules_actor_onestep_flow': {'mlp': init_mlp(rng, F + A, ah + (A,), cfg['actor_layer_norm'], None, dtype, jitter)},
        'modules_critic': {'value_net': init_mlp(rng, F + A, vh + (1,), cfg['layer_norm'], 2, dtype, jitter)},
    }
    if target_equals_critic:
        params['modules_target_critic'] = tree_map(lambda x: x.copy(), params['modules_critic'])
    else:
        params['modules_target_critic'] = {'value_net': init_mlp(rng, F + A, vh + (1,), cfg['layer_norm'], 2, dtype, jitter)}
    return params


def init_state(params, warm=False, seed=0):
    if warm:
        rng = np.random.default_rng(seed + 77)
        mu = tree_map(lambda p: (1e-3 * rng.standard_normal(p.shape)).astype(p.dtype), params)
        nu = tree_map(lambda p: (1e-6 * (0.5 + rng.random(p.shape))).astype(p.dtype), params)  # |m|/sqrt(v) = O(1)
        # target-critic moments are identically zero in a real run (zero grads, SURVEY F7)
        mu['modules_target_critic'] = _zeros_like_tree(params['modules_target_critic'])
        nu['modules_target_critic'] = _zeros_like_tree(params['modules_target_critic'])
        count = 7
    else:
        mu, nu, count = _zeros_like_tree(params), _zeros_like_tree(params), 0
    return dict(params=params, mu=mu, nu=nu, count=count, step=count + 1)


def make_batch(seed, B, obs_dim, action_dim, dtype=np.float32):
    rng = np.random.default_rng(seed)
    rew = -(rng.random(B) > 0.05).astype(dtype)   # rewards in {-1, 0}
    return {
        'observations': rng.standard_normal((B, obs_dim)).astype(dtype),
        'actions': np.clip(rng.uniform(-1, 1, (B, action_dim)), -1 + 1e-5, 1 - 1e-5).astype(dtype),
        'next_observations': rng.standard_normal((B, obs_dim)).astype(dtype),
        'rewards': rew,
        'masks': (rew != 0).astype(dtype),
        'terminals': np.zeros(B, dtype),
    }


def make_noise(seed, B, action_dim, dtype=np.float32):
    rng = np.random.default_rng(seed + 10_000)
    return {
        'z_next': rng.standard_normal((B, action_dim)).astype(dtype),
        'x0': rng.standard_normal((B, action_dim)).astype(dtype),
        't': rng.random((B, 1)).astype(dtype),
        'z': rng.standard_normal((B, action_dim)).astype(dtype),
        'z_metric': rng.standard_normal((B, action_dim)).astype(dtype),
    }


def cast_tree(t, dtype):
    return tree_map(lambda x: x.astype(dtype), t)
