"""precision='fp32-tc' (FQL_PRECISION_FP32_TC): the fp32 schedule with every Dense contraction on tcgen05 as 3xTF32
(fql_b200/csrc/gemm_tf32x3.cu), held to the fp32 mode's parity tolerance.

1. The GEMM alone (fql_test_gemm_f32 on caller buffers, precision 0 = the FFMA kernel, 3 = the 3xTF32 kernel) against fp64 NumPy on
   the same fp32 operands: every orientation the step uses, every epilogue, ragged shapes, padded pitches, P x S x E groups, split-K
   and operands whose exponents span +-20.  With P[m,n] = sum_k |a_mk b_kn|, the accumulator error must be <= 2^-18 P (dropping the
   lo terms would give ~2^-11 P) and no worse than 4x the FFMA kernel's on the same inputs.
2. Determinism of the GEMM (split-K included) and of whole update steps.
3. Whole-step parity: every case of tests/test_step_gpu.py in this mode at the unchanged 1e-5 tolerance, plus a config 3 shape at
   B = 4096 (many tiles, split-K weight gradients) and three seeds; graph capture / replay; the forward entry points.
"""
import copy
import ctypes as C

import numpy as np
import pytest
import torch

from fql_b200 import _lib
from oracle import fql_oracle as O
from tests.helpers import cuda_agent_from_state, f32, info_close, make_case, rel_err
from tests.test_step_gpu import CASES, TOL, check_update

pytestmark = pytest.mark.gpu

BOUND = 2.0 ** -18


def _gptr(bufs, S, E, rows, ld):
    g = _lib.FqlTestGPtr()
    for i, b in enumerate(bufs):
        g.base[i] = b.data_ptr() if b is not None else None
    g.stride_s, g.stride_e = E * rows * ld, rows * ld
    return g


def _operand(rng, P, S, E, rows, cols, ld, spread):
    x = rng.standard_normal((P, S, E, rows, ld))
    if spread:
        x *= 2.0 ** rng.uniform(-spread, spread, x.shape)
    return x.astype(np.float32)


def run_gemm(M, N, K, P=1, S=1, E=1, trans_a=0, trans_b=0, bias=False, mulz=False, out_pre=False, act=False, pad=0, spread=0, seed=0,
             precisions=(0, 3)):
    """Returns {precision: (out, out_pre)} and the fp64 reference (acc, v_ref, out_ref, P_abs)."""
    rng = np.random.default_rng(seed)
    ra, ca = (K, M) if trans_a else (M, K)
    rb, cb = (N, K) if trans_b else (K, N)
    lda, ldb, ldo = ca + pad, cb + pad, N + pad
    A = _operand(rng, P, S, E, ra, ca, lda, spread)
    B = _operand(rng, P, S, E, rb, cb, ldb, spread)
    bias_h = rng.standard_normal((P, S, E, 1, N)).astype(np.float32) if bias else None
    mulz_h = (2 * rng.standard_normal((P, S, E, M, ldo))).astype(np.float32) if mulz else None
    opA = A[..., :ra, :ca].astype(np.float64)
    opB = B[..., :rb, :cb].astype(np.float64)
    if trans_a:
        opA = np.swapaxes(opA, -1, -2)
    if trans_b:
        opB = np.swapaxes(opB, -1, -2)
    acc = opA @ opB
    Pabs = np.abs(opA) @ np.abs(opB)
    v = acc + (bias_h.astype(np.float64) if bias else 0.0)
    out_ref = v.copy()
    gp = 1.0
    if mulz:
        z = mulz_h[..., :M, :N].astype(np.float64)
        gp = O.gelu_tanh_grad(z)
        out_ref = out_ref * gp
    if act:
        out_ref = O.gelu_tanh(out_ref)
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    dA = [dev(A[p]) for p in range(P)]
    dB = [dev(B[p]) for p in range(P)]
    dbias = [dev(bias_h[p]) for p in range(P)] if bias else [None] * P
    dmulz = [dev(mulz_h[p]) for p in range(P)] if mulz else [None] * P
    res = {}
    for prec in precisions:
        sentinel = np.float32(-12345.0)
        dout = [torch.full((S, E, M, ldo), float(sentinel), device='cuda') for _ in range(P)]
        dpre = [torch.full((S, E, M, ldo), float(sentinel), device='cuda') for _ in range(P)] if out_pre else [None] * P
        t = _lib.FqlTestGemmF32()
        t.M, t.N, t.K, t.P, t.S, t.E = M, N, K, P, S, E
        t.lda, t.ldb, t.ldo, t.ld_pre, t.ld_mulz = lda, ldb, ldo, ldo, ldo
        t.trans_a, t.trans_b, t.act_gelu = trans_a, trans_b, int(act)
        t.A, t.B = _gptr(dA, S, E, ra, lda), _gptr(dB, S, E, rb, ldb)
        t.bias = _gptr(dbias, S, E, 1, N) if bias else _lib.FqlTestGPtr()
        t.mulz = _gptr(dmulz, S, E, M, ldo) if mulz else _lib.FqlTestGPtr()
        t.out_pre = _gptr(dpre, S, E, M, ldo) if out_pre else _lib.FqlTestGPtr()
        t.out = _gptr(dout, S, E, M, ldo)
        _lib.check(_lib.lib().fql_test_gemm_f32(C.byref(t), prec, None), 'fql_test_gemm_f32')
        torch.cuda.synchronize()
        o = np.stack([d.cpu().numpy() for d in dout])
        pre = np.stack([d.cpu().numpy() for d in dpre]) if out_pre else None
        if pad:   # the pitch padding is never written
            assert (o[..., N:] == sentinel).all(), prec
            if out_pre:
                assert (pre[..., N:] == sentinel).all(), prec
        res[prec] = (o[..., :N], None if pre is None else pre[..., :N])
    return res, dict(acc=acc, v=v, out=out_ref, P=Pabs, gp=gp)


def _acc_err(got, ref):
    """max |got - exact| / (P + |bias|) over the elements (P = sum_k |a b|; the bias joins the sum in the epilogue's fp32 add)."""
    return float((np.abs(got.astype(np.float64) - ref['v']) / np.maximum(ref['P'] + np.abs(ref['v'] - ref['acc']), 1e-30)).max())


# (id, M, N, K, kwargs): the shapes the step hands launch_gemm (F + A (+1) = 37 / 38 first-layer inputs, critic head N = 1,
# actor head N = A, dgrad trans_b with the fused gelu', wgrad trans_a with K = batch)
GEMM_CASES = [
    ('fwd-first-gelu-pre', 300, 512, 37, dict(bias=True, act=True, out_pre=True, pad=3)),
    ('fwd-hidden-grouped', 130, 64, 64, dict(P=3, S=2, E=2, bias=True, act=True, out_pre=True, pad=1)),
    ('fwd-critic-head', 256, 1, 512, dict(P=3, E=2, bias=True)),
    ('fwd-actor-head', 200, 8, 96, dict(bias=True, pad=2)),
    ('dgrad-mulz', 130, 256, 64, dict(trans_b=1, mulz=True, pad=3)),
    ('dgrad-first', 256, 38, 512, dict(trans_b=1, E=2)),
    ('dgrad-from-head', 77, 96, 1, dict(trans_b=1, mulz=True)),
    ('wgrad-first', 38, 256, 256, dict(trans_a=1, pad=5)),
    ('wgrad-k16384', 512, 512, 16384, dict(trans_a=1, E=2)),
    ('wgrad-head-k16384', 37, 1, 16384, dict(trans_a=1)),
    ('wgrad-groups', 64, 21, 1000, dict(trans_a=1, P=3, S=2, E=2, pad=1)),
    ('spread-fwd', 257, 130, 200, dict(bias=True, out_pre=True, spread=20)),
    ('spread-wgrad', 70, 90, 4096, dict(trans_a=1, spread=20)),
    ('both-trans', 129, 65, 33, dict(trans_a=1, trans_b=1, pad=7)),
]


@pytest.mark.parametrize('name,M,N,K,kw', GEMM_CASES, ids=[c[0] for c in GEMM_CASES])
def test_gemm_tf32x3_against_fp64(name, M, N, K, kw):
    res, ref = run_gemm(M, N, K, seed=sum(map(ord, name)), **kw)
    errs = {}
    for prec in (0, 3):
        out, pre = res[prec]
        # the accumulator (+ bias): out_pre when the epilogue goes on, else out itself
        acc_out = pre if pre is not None else (out if not (kw.get('mulz') or kw.get('act')) else None)
        if acc_out is not None:
            errs[prec] = _acc_err(acc_out, ref)
        # the final output: the accumulator error carried through the epilogue (|gelu'| <= 1.13), plus the fp32 evaluation of
        # gelu / gelu' in fp32 (absolute error of a few 2^-24, times |v| for gelu'; the FFMA kernel reaches 2^-21 |v|) and the
        # epilogue's own rounding
        scale = (ref['P'] + np.abs(ref['v'] - ref['acc'])) * (np.abs(ref['gp']) if kw.get('mulz') else 1.0) * (1.13 if kw.get('act') else 1.0)
        nonlin = 2.0 ** -19 * np.abs(ref['v']) if (kw.get('mulz') or kw.get('act')) else 0.0
        bound = BOUND * scale + nonlin + 4e-6 * np.abs(ref['out']) + 1e-30
        worst = float((np.abs(out.astype(np.float64) - ref['out']) / bound).max())
        assert worst <= 1.0, (name, prec, worst)
    if errs:
        print(f'{name}: accumulator error / P  3xTF32 {errs[3]:.3e}  FFMA {errs[0]:.3e}  (bound {BOUND:.3e})')
        assert errs[3] <= BOUND, (name, errs)
        # 2^-24 floors the comparison where the FFMA result is exact (K = 1, or every product and sum representable)
        assert errs[3] <= 4 * errs[0] + 2.0 ** -24, (name, errs)


def test_gemm_without_lo_terms_would_fail_the_bound():
    """Calibrates the bound: the same data through a tf32-only product (hi x hi, what the kernel would compute without the lo terms)
    is ~2^-11 P, well above 2^-18 P."""
    rng = np.random.default_rng(5)
    a = rng.standard_normal((128, 256)).astype(np.float32)
    b = rng.standard_normal((256, 64)).astype(np.float32)
    hi = lambda x: (x.view(np.uint32) + np.uint32(0x1000) & np.uint32(0xFFFFE000)).view(np.float32)
    exact = a.astype(np.float64) @ b.astype(np.float64)
    Pabs = np.abs(a.astype(np.float64)) @ np.abs(b.astype(np.float64))
    e = (np.abs(hi(a).astype(np.float64) @ hi(b).astype(np.float64) - exact) / Pabs).max()
    assert e > 8 * BOUND


def test_gemm_split_k_is_deterministic():
    a, _ = run_gemm(512, 512, 16384, trans_a=1, E=2, seed=9, precisions=(3,))
    b, _ = run_gemm(512, 512, 16384, trans_a=1, E=2, seed=9, precisions=(3,))
    assert np.array_equal(a[3][0], b[3][0])


@pytest.mark.parametrize('name,over,B,F,A,hidden', CASES, ids=[c[0] for c in CASES])
def test_update_step_parity_fp32_tc(name, over, B, F, A, hidden):
    cfg, state, batch, noise = make_case(over, B, F, A, seed=sum(map(ord, name)) % 1000, hidden=hidden)
    agent = cuda_agent_from_state(cfg, state, B, F, A, precision='fp32-tc')
    worst = check_update(agent, cfg, state, batch, noise)
    print(name, {k: f'{v:.2e}' for k, v in worst.items()})


def test_update_step_parity_fp32_tc_config3_b4096():
    """BASELINE config 3 shape at B = 4096, hidden 512: many output tiles per layer and weight gradients with K = 4096 (split-K)."""
    cfg, state, batch, noise = make_case(dict(discount=0.995, alpha=30.0), 4096, 69, 21, seed=31, hidden=512)
    agent = cuda_agent_from_state(cfg, state, 4096, 69, 21, precision='fp32-tc')
    worst = check_update(agent, cfg, state, batch, noise)
    print('config3-b4096', {k: f'{v:.2e}' for k, v in worst.items()})


def test_multi_seed_fp32_tc():
    over = dict(normalize_q_loss=True, alpha=1000.0)
    seeds = []
    for s in range(3):
        cfg, state, batch, noise = make_case(over, 32, 13, 5, seed=60 + s, hidden=64)
        seeds.append((state, batch, noise))
    agent = cuda_agent_from_state(cfg, seeds[0][0], 32, 13, 5, num_seeds=3, precision='fp32-tc')
    check_update(agent, cfg, None, None, None, seeds=seeds)


def test_update_is_deterministic():
    cfg, state, batch, noise = make_case(dict(q_agg='min', alpha=10.0), 1024, 29, 8, seed=12, hidden=512)
    outs = []
    for _ in range(2):
        agent = cuda_agent_from_state(cfg, state, 1024, 29, 8, precision='fp32-tc')
        agent.load_tree(f32(state['params']), f32(state['mu']), f32(state['nu']), state['count'])
        _, info = agent.update(f32(batch), noise=f32(noise))
        outs.append((info, agent.export_tree('params'), agent.export_tree('grads')))
    for k in O.INFO_KEYS:
        assert np.array_equal(np.asarray(outs[0][0][k]), np.asarray(outs[1][0][k])), k
    for which in (1, 2):
        for (path, x), (_, y) in zip(O.tree_leaves(outs[0][which]), O.tree_leaves(outs[1][which])):
            assert np.array_equal(x, y), path


def test_two_consecutive_steps_and_graph_replay_fp32_tc():
    """Step 1 eager, step 2 captures the CUDA graph, steps 3-4 replay it: all four match the oracle."""
    cfg, state, batch, noise = make_case(dict(q_agg='min', alpha=10.0), 64, 29, 8, seed=3, hidden=128)
    agent = cuda_agent_from_state(cfg, state, 64, 29, 8, precision='fp32-tc')
    agent.load_tree(f32(state['params']), f32(state['mu']), f32(state['nu']), state['count'])
    st = copy.deepcopy(state)
    for i in range(4):
        ba = O.make_batch(100 + i, 64, 29, 8, np.float64)
        nz = O.make_noise(200 + i, 64, 8, np.float64)
        st, info_ref, _ = O.update(st, cfg, ba, nz)
        _, info = agent.update(f32(ba), noise=f32(nz))
        for k in O.INFO_KEYS:
            info_close(k, info[k], info_ref, 5e-5)
        got = agent.export_tree('params')
        for (path, r), (_, g) in zip(O.tree_leaves(st['params']), O.tree_leaves(got)):
            assert rel_err(g, r) <= 1e-5 * (i + 1), (i, path)
    assert agent.network.step == state['step'] + 4


@pytest.mark.parametrize('rows', [1, 300])
def test_forward_entry_points_fp32_tc(rows):
    cfg, state, batch, noise = make_case(dict(), 48, 29, 8, seed=21, hidden=512)
    a32 = cuda_agent_from_state(cfg, state, 48, 29, 8)
    atc = cuda_agent_from_state(cfg, state, 48, 29, 8, precision='fp32-tc')
    for ag in (a32, atc):
        ag.load_tree(f32(state['params']))
    rng = np.random.default_rng(rows)
    obs = rng.standard_normal((rows, 29)).astype(np.float32)
    nz = rng.standard_normal((rows, 8)).astype(np.float32)
    ref = O.sample_actions_given_noise(state['params'], cfg, obs.astype(np.float64), nz.astype(np.float64))
    a = atc.sample_actions(obs, noise=nz)
    assert rel_err(a, ref) <= TOL and rel_err(a, a32.sample_actions(obs, noise=nz)) <= TOL
    ref = O.compute_flow_actions(state['params'], cfg, obs.astype(np.float64), nz.astype(np.float64))
    fa = atc.compute_flow_actions(obs, nz)
    assert rel_err(fa, ref) <= TOL and rel_err(fa, a32.compute_flow_actions(obs, nz)) <= TOL
    loss, info = atc.total_loss(f32(batch), noise=f32(noise))
    ref_loss, ref_info, _ = O.total_loss(state['params'], cfg, batch, noise, with_grads=False)
    assert abs(loss - ref_loss) <= TOL * abs(ref_loss)
    for k in ref_info:
        info_close(k, info[k], ref_info, 3 * TOL)


def test_pixel_config_is_refused():
    from fql_b200 import FQLAgent
    cfg = dict(O.DEFAULT_CONFIG, encoder='impala_small')
    with pytest.raises(NotImplementedError, match='fp32-tc'):
        FQLAgent.create(0, np.zeros((1, 64, 64, 3), np.uint8), np.zeros((1, 4), np.float32), cfg, precision='fp32-tc')
    d = _lib.make_dims(64, 512, 4, precision=_lib.PRECISION_FP32_TC, image=(64, 64, 3))
    assert _lib.lib().fql_arena_floats(C.byref(d)) == -1
    assert 'FQL_PRECISION_FP32_TC' in _lib.lib().fql_last_error().decode()
