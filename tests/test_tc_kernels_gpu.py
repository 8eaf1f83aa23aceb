"""The tensor-core MLP kernels of FQL_PRECISION_BF16_TC one at a time, through the test hooks of include/fql_b200.h, against fp64
NumPy references on the same bf16 operands: tc_gemm with each of its five epilogues (fql_b200/csrc/tc_gemm.cu), split-K, groups and
operand majorness; the critic's row kernels and the bf16 column sums (tc_path.cu); and the stand-alone forward chains (the cluster
Euler kernel and the chain kernel) against an oracle that rounds the same operands to bf16.

Two operand families:
  * exact-arithmetic operands: small integers (|a|, |b| <= 8, about 20 % zeros, optionally scaled by powers of two), so every
    product and partial sum is exact in fp32 in ANY summation order.  Results must be bit-equal to the fp64 reference (rounded to
    bf16 where the output is bf16).  This is what catches indexing, tiling, K coverage, row masks, group strides and split-K.
  * Gaussian bf16 operands, checked per element against a stated bound:
      - accumulation: with P[m,n] = sum_k |a_mk b_kn|, |acc - exact| <= 2^-24 (K + 8) P (fp32 in any summation order);
      - tanh.approx.f32 (gelu_fast, gelu_grad_fast, gelu_and_grad_fast) has an absolute error <= 2^-11: the reference is evaluated
        on the interval tanh +- 2^-11 and the result may lie anywhere in it (for gelu that is 0.5 |z| 2^-11);
      - a pre-activation that is itself inexact (z = acc + bias in fp32) carries its error through gelu' (|gelu'| <= 1.13);
      - every bf16 output adds 2^-8 |ref| (round to nearest is 2^-9); fp32 epilogue arithmetic adds a few 2^-24 |terms|.
    The LayerNorm row kernels propagate the per-element gelu error through the first-order LayerNorm Jacobian (see _ln_fwd_bound
    and test_ln_bwd_rows) and add the fp32 error of the row statistics.
Measured on one B200 (power limit 1000 W), worst error / bound over all cases (the tests print theirs): bf16 outputs 0.93-0.995
(z save 0.995, h 0.93, DGRAD_GELU dZ 0.99, gelu' rows 0.99, LayerNorm(gelu) rows 0.96, LayerNorm backward 0.82; the bf16 rounding
term dominates these), fp32 outputs 0.001-0.07 (STORE_F32 0.002, DGRAD_GELU dZ 0.001, gelu' rows 0.07, LayerNorm backward 0.011,
mu / rstd 0.001).  The bounds are derived, not fitted: a ratio near 1 on a bf16 output is a value that rounds by almost half a unit.

Every output buffer is pre-filled with a finite sentinel and has a slack tail of one 128-row tile plus 64 elements beyond the
written region; elements outside that region must be bit-unchanged after the call.  Inputs the kernels read by contract never
hold the sentinel or NaN: the K padding columns of a first-layer operand are multiplied by TMA zero fill, so they must be finite
(NaN x 0 = NaN), and test_k_padding_columns_are_ignored fills them with +-1000 to check that they do not matter.
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from fql_b200 import _lib
from oracle import fql_oracle as O

pytestmark = pytest.mark.gpu

DEV = 'cuda'
EPS_TANH = 2.0 ** -11
U24 = 2.0 ** -24
SENT = {torch.float32: -12345.5, torch.bfloat16: -1232.0}     # finite sentinels of the outputs (exact in their type)
GC, GA = math.sqrt(2.0 / math.pi), 0.044715


def _stream():
    return torch.cuda.current_stream().cuda_stream


def bf16_round(x):
    """round to nearest bf16 through fp32 (what __float2bfloat16 of an fp32 value gives), back to float64"""
    return torch.as_tensor(np.asarray(x, np.float32)).to(torch.bfloat16).double().numpy()


def ints(rng, shape, lim=8, scale=1.0):
    v = rng.integers(-lim, lim + 1, shape).astype(np.float64)
    v[rng.random(shape) < 0.2] = 0.0
    return v * scale


def gauss(rng, shape, scale=1.0):
    return bf16_round(rng.standard_normal(shape) * scale)


def report(what, err, bound):
    ratio = float(np.max(err / np.maximum(bound, 1e-300))) if np.size(err) else 0.0
    print(f'{what}: max |err| {float(np.max(err)) if np.size(err) else 0.0:.3e}, worst err / bound {ratio:.3f}')
    return ratio


def assert_within(what, got, lo, hi, tol):
    """got within [lo - tol, hi + tol] element-wise (lo == hi: a point reference)"""
    err = np.maximum(np.maximum(lo - got, got - hi), 0.0)
    bad = err > tol
    assert not bad.any(), (what, int(bad.sum()), np.argwhere(bad)[:4].tolist(), float(err.max()))
    return report(what, err, tol)


def assert_exact(what, got, ref):
    bad = got != ref
    assert not bad.any(), (what, int(bad.sum()), np.argwhere(bad)[:4].tolist(), got[bad][:4].tolist(), ref[bad][:4].tolist())


# ------------------------------------------------------------------------------------------------------------------------------
# buffers
# ------------------------------------------------------------------------------------------------------------------------------
def operand(arr, ld=None):
    """bf16 TMA operand from a logical fp64 array [G1][G0][rows][inner] (bf16-exact values)"""
    G1, G0, R, inner = arr.shape
    ld = ld or inner
    buf = torch.zeros(G1, G0, R, ld, dtype=torch.bfloat16)
    buf[..., :inner] = torch.as_tensor(arr.astype(np.float32)).to(torch.bfloat16)
    buf = buf.to(DEV)
    return buf, _lib.FqlTestOperand(buf.data_ptr(), inner, R, ld, G0, R * ld, G1, G0 * R * ld)


def param(arr):
    """fp32 epilogue input [G1][G0][...] (G0 == 1: broadcast over g0, as the step passes them)"""
    t = torch.as_tensor(np.ascontiguousarray(arr, np.float32)).to(DEV)
    G1, G0 = arr.shape[:2]
    inner = int(np.prod(arr.shape[2:]))
    ld = arr.shape[-1] if arr.ndim == 4 else 0
    return t, _lib.FqlTestPtr(t.data_ptr(), inner if G0 > 1 else 0, G0 * inner, ld)


class Out:
    """output [G1][G0][M][N] with row pitch ld inside a sentinel-filled buffer with one 128-row tile + 64 elements of slack"""

    def __init__(self, G1, G0, M, N, dtype=torch.float32, ld=None, fill=None):
        self.G1, self.G0, self.M, self.N, self.dtype, self.ld = G1, G0, M, N, dtype, ld or N
        self.rows = -(-M // 128) * 128 + 128
        self.n = G1 * G0 * self.rows * self.ld
        self.buf = torch.full((self.n + 64,), SENT[dtype], dtype=dtype, device=DEV)
        if fill is not None:
            self.set(fill)
        self.snap = self.bits().clone()

    def view(self):
        return self.buf[:self.n].view(self.G1, self.G0, self.rows, self.ld)

    def set(self, arr):
        self.view()[:, :, :self.M, :self.N] = torch.as_tensor(np.broadcast_to(arr, (self.G1, self.G0, self.M, self.N)).astype(np.float32)).to(self.dtype)

    def bits(self):
        return self.buf.view(torch.int32 if self.dtype == torch.float32 else torch.int16)

    def ptr(self):
        s0 = self.rows * self.ld
        return _lib.FqlTestPtr(self.buf.data_ptr(), s0 if self.G0 > 1 else 0, self.G0 * s0, self.ld)

    def get(self):
        return self.view()[:, :, :self.M, :self.N].double().cpu().numpy()

    def get_bits(self):
        return self.view()[:, :, :self.M, :self.N].contiguous().view(torch.int32 if self.dtype == torch.float32 else torch.int16).cpu().numpy()

    def check_untouched(self, what, written=None):
        """every element outside the written region (default: [:, :, :M, :N]) is bit-unchanged"""
        keep = torch.ones(self.n + 64, dtype=torch.bool, device=DEV)
        if written is None:
            keep[:self.n].view(self.G1, self.G0, self.rows, self.ld)[:, :, :self.M, :self.N] = False
        else:
            written(keep[:self.n].view(self.G1, self.G0, self.rows, self.ld))
        changed = keep & (self.bits() != self.snap)
        n = int(changed.sum())
        assert n == 0, (what, 'elements outside the written region changed', n, torch.nonzero(changed)[:4].flatten().tolist())


def gemm(mode, M, N, K, A, B, G0=1, G1=1, a_mn=0, b_mn=0, ksplit=1, **kw):
    g = _lib.FqlTestGemm()
    g.mode, g.M, g.N, g.K, g.G0, g.G1, g.a_mn, g.b_mn, g.ksplit = mode, M, N, K, G0, G1, a_mn, b_mn, ksplit
    g.A, g.B = A, B
    for k, v in kw.items():
        setattr(g, k, v)
    _lib.check(_lib.lib().fql_test_tc_gemm(C.byref(g), _stream()), 'fql_test_tc_gemm')
    torch.cuda.synchronize()


def operands(a, b, a_mn, b_mn, a_pad=None, b_pad=None, a_fill=0.0):
    """device operands of the logical product a [G1][G0a][M][K] @ b [G1][G0b][K][N] in the requested majorness; a_pad / b_pad widen
    the inner extent (columns filled with a_fill / 0), as the zero-padded first-layer input and [H][64] last-layer weights are"""
    def pad(x, to, fill):
        if to is None or to == x.shape[-1]:
            return x
        out = np.full(x.shape[:-1] + (to,), fill)
        out[..., :x.shape[-1]] = x
        return out
    ta, oa = operand(pad(np.swapaxes(a, -1, -2) if a_mn else a, a_pad, a_fill))
    tb, ob = operand(pad(b if b_mn else np.swapaxes(b, -1, -2), b_pad, 0.0))
    return (ta, tb), oa, ob


def acc_ref(a, b):
    """exact product and the accumulation bound 2^-24 (K + 8) sum_k |a b|"""
    K = a.shape[-1]
    return a @ b, U24 * (K + 8) * (np.abs(a) @ np.abs(b))


def gelu_th(z, th):
    return 0.5 * z * (1.0 + th)


def gelu_grad_th(z, th):
    du = GC * (1.0 + 3.0 * GA * z * z)
    return 0.5 * (1.0 + th) + 0.5 * z * (1.0 - th * th) * du


def tanh_u(z):
    return np.tanh(GC * (z + GA * z ** 3))


def gelu_interval(z):
    th = tanh_u(z)
    a, b = gelu_th(z, th - EPS_TANH), gelu_th(z, th + EPS_TANH)
    return np.minimum(a, b), np.maximum(a, b)


def gelu_grad_interval(z):
    """gelu'(z) with tanh anywhere in th +- 2^-11: quadratic in th, so the ends and the clipped vertex"""
    th = tanh_u(z)
    du = GC * (1.0 + 3.0 * GA * z * z)
    lo_t, hi_t = th - EPS_TANH, th + EPS_TANH
    with np.errstate(divide='ignore', invalid='ignore'):
        tv = np.where(z * du != 0, 0.5 / (z * du), th)
    tv = np.clip(tv, lo_t, hi_t)
    vals = np.stack([gelu_grad_th(z, t) for t in (lo_t, hi_t, tv)])
    return vals.min(0), vals.max(0)


def wgrad_ksplit(Mw, N, groups, K):
    """tc_path.cu wgrad_ksplit: about two CTAs per SM, at least four K blocks per CTA"""
    base = -(-Mw // 128) * -(-N // 64) * groups
    ks = min(296 // max(base, 1), -(-K // 64) // 4)
    return max(ks, 1)


# ------------------------------------------------------------------------------------------------------------------------------
# TC_MODE_FWD_HIDDEN: z = acc + bias -> bf16 z save, h = gelu(z) -> bf16
# ------------------------------------------------------------------------------------------------------------------------------
FWD_SHAPES = [(14, 64, 128), (37, 64, 256), (38, 64, 512), (91, 128, 512), (128, 128, 128), (256, 256, 256), (512, 512, 512)]   # K, A inner, N


def _fwd_hidden(rng, M, K, Kpad, N, G1, family, a_fill=0.0):
    if family == 'int':
        a, b = ints(rng, (G1, 1, M, K), scale=2.0 ** -4), ints(rng, (G1, 1, K, N), scale=2.0 ** -4)
        bias = ints(rng, (G1, 1, N), scale=2.0 ** -8)
    else:
        a, b = gauss(rng, (G1, 1, M, K)), gauss(rng, (G1, 1, K, N), 1.0 / math.sqrt(K))
        bias = rng.standard_normal((G1, 1, N)).astype(np.float32).astype(np.float64) * 0.1
    keep, oa, ob = operands(a, b, 0, 1, a_pad=Kpad, a_fill=a_fill)
    tbias, pbias = param(bias)
    oh, oz = Out(G1, 1, M, N, torch.bfloat16), Out(G1, 1, M, N, torch.bfloat16)
    gemm(_lib.TC_MODE_FWD_HIDDEN, M, N, K, oa, ob, G1=G1, b_mn=1, bias=pbias, out_h=oh.ptr(), out_z=oz.ptr())
    oh.check_untouched('h')
    oz.check_untouched('z')
    acc, pb = acc_ref(a, b)
    return acc + bias[:, :, None, :], pb, oh, oz


@pytest.mark.parametrize('M', [1, 40, 127, 128, 129, 200, 1000])
@pytest.mark.parametrize('K,Kpad,N', FWD_SHAPES, ids=[f'K{k}-pad{p}-N{n}' for k, p, n in FWD_SHAPES])
def test_fwd_hidden(K, Kpad, N, M):
    rng = np.random.default_rng(K * 7 + N + M)
    G1 = 2 + M % 2
    # exact operands: the z save is bf16(acc + bias) bit for bit
    z, _, oh, oz = _fwd_hidden(rng, M, K, Kpad, N, G1, 'int')
    assert_exact('z save (exact operands)', oz.get(), bf16_round(z))
    lo, hi = gelu_interval(z)
    assert_within('h (exact operands)', oh.get(), lo, hi, 2.0 ** -8 * np.maximum(np.abs(lo), np.abs(hi)) + (1 + 2.0 ** -8) * U24 * 16 * np.abs(z) + 1e-30)
    # Gaussian operands: z and h within the stated bound
    z, pb, oh, oz = _fwd_hidden(rng, M, K, Kpad, N, G1, 'gauss')
    dz = pb + U24 * np.abs(z)                                   # accumulation + the fp32 bias add
    assert_within('z save (Gaussian)', oz.get(), z, z, (1 + 2.0 ** -8) * dz + 2.0 ** -8 * np.abs(z))
    lo, hi = gelu_interval(z)
    assert_within('h (Gaussian)', oh.get(), lo, hi, (1 + 2.0 ** -8) * (1.13 * dz + U24 * 16 * np.abs(z)) + 2.0 ** -8 * np.maximum(np.abs(lo), np.abs(hi)))


@pytest.mark.parametrize('K,Kpad', [(14, 64), (37, 64), (38, 64), (91, 128)])
def test_k_padding_columns_are_ignored(K, Kpad):
    """First layer: K < K0pad.  The A map's inner extent is K0pad, so columns [K, K0pad) of A are loaded and multiplied by the rows
    of B beyond K, which TMA zero-fills.  Those columns only have to be FINITE (NaN x 0 = NaN): finite garbage (+-1000) must give
    the bit-identical result of the zero-padded operand."""
    res = []
    for fill in (0.0, 1000.0, -1000.0):
        rng = np.random.default_rng(K)
        _, _, oh, oz = _fwd_hidden(rng, 200, K, Kpad, 512, 2, 'gauss', a_fill=fill)
        res.append((oh.get_bits(), oz.get_bits()))
    for r in res[1:]:
        assert_exact('h with garbage K padding', r[0], res[0][0])
        assert_exact('z with garbage K padding', r[1], res[0][1])


def test_determinism_without_split_k():
    """Two identical calls with ksplit = 1 are bit-identical (split-K and the column sums use atomics: not asserted there)."""
    outs = []
    for _ in range(2):
        rng = np.random.default_rng(5)
        _, _, oh, oz = _fwd_hidden(rng, 1000, 512, 512, 512, 2, 'gauss')
        outs.append((oh.get_bits(), oz.get_bits()))
    assert_exact('h, second call', outs[1][0], outs[0][0])
    assert_exact('z, second call', outs[1][1], outs[0][1])


# ------------------------------------------------------------------------------------------------------------------------------
# TC_MODE_STORE_F32: forward last layer (+bias, clip), critic head (N = 1, two heads, broadcast A), input gradient, fp32 Z
# ------------------------------------------------------------------------------------------------------------------------------
STORE_CASES = [
    # name, M, N, K, b_mn, B inner pad, G0 (heads), G1
    ('last-A1', 200, 1, 512, 1, 64, 1, 2),
    ('last-A3', 129, 3, 256, 1, 64, 1, 2),
    ('last-A5', 1000, 5, 512, 1, 64, 1, 1),
    ('last-A8', 127, 8, 512, 1, 64, 1, 3),
    ('last-A21', 300, 21, 512, 1, 64, 1, 2),
    ('critic-head', 257, 1, 512, 1, 64, 2, 2),
    ('input-grad-K0-38', 200, 38, 512, 0, None, 1, 2),
    ('input-grad-K0-40', 129, 40, 512, 0, None, 1, 2),       # float4 branch for columns 0..31, scalar for 32..39
    ('input-grad-K0-91', 40, 91, 512, 0, None, 2, 2),
    ('critic-Z-96', 200, 96, 128, 1, None, 2, 2),
    ('critic-Z-512', 129, 512, 512, 1, None, 2, 2),
]


@pytest.mark.parametrize('clip', [0, 1])
@pytest.mark.parametrize('with_bias', [0, 1])
@pytest.mark.parametrize('name,M,N,K,b_mn,bpad,G0,G1', STORE_CASES, ids=[c[0] for c in STORE_CASES])
def test_store_f32_exact(name, M, N, K, b_mn, bpad, G0, G1, with_bias, clip):
    rng = np.random.default_rng(M * 31 + N + 7 * with_bias + clip)
    a_bcast = name.startswith('critic-head')                     # both heads read the same first-layer input
    a = ints(rng, (G1, 1 if a_bcast else G0, M, K), scale=2.0 ** -4)
    b = ints(rng, (G1, G0, K, N), scale=2.0 ** -4)
    keep, oa, ob = operands(a, b, 0, b_mn, b_pad=bpad if b_mn else None)
    out = Out(G1, G0, M, N)
    kw = dict(out_f=out.ptr(), clip=clip)
    ref = a @ b
    if with_bias:
        bias = ints(rng, (G1, G0, N), scale=2.0 ** -8)
        tb, kw['bias'] = param(bias)
        ref = ref + bias[:, :, None, :]
    gemm(_lib.TC_MODE_STORE_F32, M, N, K, oa, ob, G0=G0, G1=G1, b_mn=b_mn, **kw)
    if clip:
        ref = np.clip(ref, -1.0, 1.0)
    assert_exact(name, out.get(), ref)
    out.check_untouched(name)


def test_store_f32_gaussian_bound():
    rng = np.random.default_rng(11)
    M, N, K, G1 = 1000, 512, 512, 2
    a, b = gauss(rng, (G1, 1, M, K)), gauss(rng, (G1, 1, K, N), 1.0 / math.sqrt(K))
    keep, oa, ob = operands(a, b, 0, 1)
    bias = rng.standard_normal((G1, 1, N)).astype(np.float32).astype(np.float64)
    tb, pb = param(bias)
    out = Out(G1, 1, M, N)
    gemm(_lib.TC_MODE_STORE_F32, M, N, K, oa, ob, G1=G1, b_mn=1, bias=pb, out_f=out.ptr())
    acc, bnd = acc_ref(a, b)
    ref = acc + bias[:, :, None, :]
    assert_within('store_f32 (Gaussian)', out.get(), ref, ref, bnd + U24 * np.abs(ref))
    out.check_untouched('store_f32 (Gaussian)')


# ------------------------------------------------------------------------------------------------------------------------------
# weight gradients: a_mn = b_mn = 1, K = batch, split-K into a zeroed output
# ------------------------------------------------------------------------------------------------------------------------------
WGRAD_SHAPES = [(38, 64, 512, 512), (512, 512, 512, 512), (512, 512, 8, 64)]   # M (= in), A inner, N, B inner


@pytest.mark.parametrize('K', [40, 129, 256, 1000, 8192, 16384])
@pytest.mark.parametrize('M,Apad,N,Bpad', WGRAD_SHAPES, ids=[f'M{m}-N{n}' for m, _, n, _ in WGRAD_SHAPES])
def test_wgrad_split_k_exact(M, Apad, N, Bpad, K):
    rng = np.random.default_rng(M + N + K)
    G1 = 2
    x = ints(rng, (G1, 1, K, M))                                  # [batch][in] activations
    dz = ints(rng, (G1, 1, K, N))                                 # [batch][out] upstream gradient
    keep, oa, ob = operands(np.swapaxes(x, -1, -2), dz, 1, 1, a_pad=Apad, b_pad=Bpad)
    ref = np.swapaxes(x, -1, -2) @ dz
    nkb = -(-K // 64)
    for ks in sorted({1, 2, 3, 7, wgrad_ksplit(M, N, G1, K), nkb + 1}):
        out = Out(G1, 1, M, N, fill=0.0)
        gemm(_lib.TC_MODE_STORE_F32, M, N, K, oa, ob, G1=G1, a_mn=1, b_mn=1, ksplit=ks, out_f=out.ptr())
        assert_exact(f'wgrad ksplit={ks}', out.get(), ref)
        out.check_untouched(f'wgrad ksplit={ks}')


def test_split_k_rejects_bias_and_non_accumulating_epilogues():
    """host-side validation: split-K only with an accumulating fp32 epilogue and without a bias (nothing is launched)"""
    rng = np.random.default_rng(0)
    keep, oa, ob = operands(ints(rng, (1, 1, 128, 512)), ints(rng, (1, 1, 512, 512)), 0, 1)
    bias, pb = param(np.zeros((1, 1, 512)))
    out, oh = Out(1, 1, 128, 512), Out(1, 1, 128, 512, torch.bfloat16)
    with pytest.raises(_lib.FqlError, match='split-K with a bias'):
        gemm(_lib.TC_MODE_STORE_F32, 128, 512, 512, oa, ob, b_mn=1, ksplit=2, bias=pb, out_f=out.ptr())
    with pytest.raises(_lib.FqlError, match='split-K needs'):
        gemm(_lib.TC_MODE_FWD_HIDDEN, 128, 512, 512, oa, ob, b_mn=1, ksplit=2, out_h=oh.ptr())
    with pytest.raises(_lib.FqlError, match='N % 64'):
        gemm(_lib.TC_MODE_FWD_HIDDEN, 128, 500, 512, oa, ob, b_mn=1, out_h=oh.ptr())
    out.check_untouched('rejected calls')
    oh.check_untouched('rejected calls')


# ------------------------------------------------------------------------------------------------------------------------------
# TC_MODE_DGRAD_GELU: dZ = acc * gelu'(zin), bf16 + optional fp32
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('family', ['int', 'gauss'])
@pytest.mark.parametrize('M', [1, 129, 1000])
@pytest.mark.parametrize('K,N', [(64, 512), (512, 512), (64, 256)])
def test_dgrad_gelu(K, N, M, family):
    rng = np.random.default_rng(K + N + M)
    G1 = 2
    if family == 'int':
        dy, w = ints(rng, (G1, 1, M, K), scale=2.0 ** -4), ints(rng, (G1, 1, K, N), scale=2.0 ** -4)
    else:
        dy, w = gauss(rng, (G1, 1, M, K)), gauss(rng, (G1, 1, K, N), 1.0 / math.sqrt(K))
    if K == 64:                                                   # padded dOut [M][64] x last-layer weights [H][64] (only A columns)
        dy[..., 8:] = 0.0
    zin = gauss(rng, (G1, 1, M, N), 1.5)
    keep, oa, ob = operands(dy, w, 0, 0)                          # B K-major: the row-major weights [n = in][k = out]
    zb = Out(G1, 1, M, N, torch.bfloat16, fill=zin)              # read by row: the same slack as the outputs
    oh, of = Out(G1, 1, M, N, torch.bfloat16), Out(G1, 1, M, N)
    gemm(_lib.TC_MODE_DGRAD_GELU, M, N, K, oa, ob, G1=G1, b_mn=0, zin=zb.ptr(), out_h=oh.ptr(), out_f=of.ptr())
    acc, bnd = acc_ref(dy, w)
    glo, ghi = gelu_grad_interval(zin)
    cands = np.stack([acc * glo, acc * ghi])
    lo, hi = cands.min(0), cands.max(0)
    tol = bnd * np.maximum(np.abs(glo), np.abs(ghi)) + U24 * 4 * np.maximum(np.abs(lo), np.abs(hi))
    assert_within(f'dZ fp32 ({family})', of.get(), lo, hi, tol)
    assert_within(f'dZ bf16 ({family})', oh.get(), lo, hi, tol * (1 + 2.0 ** -8) + 2.0 ** -8 * np.maximum(np.abs(lo), np.abs(hi)))
    oh.check_untouched('dZ bf16')
    of.check_untouched('dZ fp32')


# ------------------------------------------------------------------------------------------------------------------------------
# TC_MODE_EULER: act += (acc + bias) / n; xb[F + n] = bf16(act); xb[F + A] = bf16((step + 1) / n); target = clip(act) at the end
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('step', [0, 9])
@pytest.mark.parametrize('M', [1, 129, 200])
@pytest.mark.parametrize('F,A', [(11, 1), (69, 8), (69, 21), (11, 21)])
def test_euler_epilogue_exact(F, A, M, step):
    rng = np.random.default_rng(F * A + M + step)
    G1, H, n_steps = 2, 512, 10
    K0 = F + A + 1
    K0pad = -(-K0 // 64) * 64
    h = ints(rng, (G1, 1, M, H), scale=2.0 ** -4)
    w = ints(rng, (G1, 1, H, A), scale=2.0 ** -4)
    bias = ints(rng, (G1, 1, A), scale=2.0 ** -8)
    keep, oa, ob = operands(h, w, 0, 1, b_pad=64)
    tb, pb = param(bias)
    act0 = rng.standard_normal((G1, 1, M, A)).astype(np.float32)
    act = Out(G1, 1, M, A, fill=act0)
    target = Out(G1, 1, M, A)
    xb0 = gauss(rng, (G1, 1, M, K0pad))
    xb = Out(G1, 1, M, K0pad, torch.bfloat16, fill=xb0)
    gemm(_lib.TC_MODE_EULER, M, A, H, oa, ob, G1=G1, b_mn=1, bias=pb, act=act.ptr(), xb=xb.ptr(), target=target.ptr(),
         F=F, Adim=A, step=step, n_steps=n_steps)
    v = (h @ w + bias[:, :, None, :]).astype(np.float32)         # exact in fp32
    a_new = act0 + v / np.float32(n_steps)                        # the kernel's fp32 division and add, both round to nearest
    assert_exact('act', act.get(), a_new.astype(np.float64))
    act.check_untouched('act')
    xb_ref = xb0.copy()
    xb_ref[..., F:F + A] = bf16_round(a_new)
    xb_ref[..., F + A] = bf16_round(np.float32((step + 1) / n_steps))
    assert_exact('xb', xb.get(), xb_ref)
    xb.check_untouched('xb')
    if step == n_steps - 1:
        assert_exact('target', target.get(), np.clip(a_new, -1, 1).astype(np.float64))
        target.check_untouched('target')
    else:
        target.check_untouched('target before the last step', written=lambda keep: None)


# ------------------------------------------------------------------------------------------------------------------------------
# TC_MODE_WGRAD_LN: dW = gamma_m G + beta_m db_n, dgamma_m = sum_n W G, dbeta_m = sum_n W db (once over the K splits)
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('K', [256, 1000, 16384])
@pytest.mark.parametrize('G1', [2, 3])
def test_wgrad_ln_exact(G1, K):
    """entries in {-1, 0, 1}: |G| <= K = 2^14 and |dgamma| <= 512 K = 2^23, so every partial sum is exact in any order"""
    rng = np.random.default_rng(K + G1)
    E, H, N = 2, 512, 512
    xhat = ints(rng, (G1, E, K, H), lim=1)
    dz = ints(rng, (G1, E, K, N), lim=1)
    gam, bet = ints(rng, (G1, E, H), lim=1), ints(rng, (G1, E, H), lim=1)
    db = ints(rng, (G1, E, N), lim=1)
    W = ints(rng, (G1, E, H, N), lim=1)
    keep, oa, ob = operands(np.swapaxes(xhat, -1, -2), dz, 1, 1)
    tg, pg = param(gam)
    tbe, pbe = param(bet)
    tdb, pdb = param(db)
    tW, pW = param(W)
    pW.ld = 0
    G = np.swapaxes(xhat, -1, -2) @ dz
    ref_dw = gam[..., None] * G + bet[..., None] * db[:, :, None, :]
    ref_dg = (W * G).sum(-1)
    ref_dbt = (W * db[:, :, None, :]).sum(-1)
    for ks in sorted({1, 3, wgrad_ksplit(H, N, G1 * E, K), -(-K // 64) + 1}):
        dw = Out(G1, E, H, N, fill=0.0)
        dg = Out(G1, E, 1, H, fill=0.0)
        dbt = Out(G1, E, 1, H, fill=0.0)
        flat = lambda o: _lib.FqlTestPtr(o.buf.data_ptr(), o.rows * o.ld, E * o.rows * o.ld, 0)
        gemm(_lib.TC_MODE_WGRAD_LN, H, N, K, oa, ob, G0=E, G1=G1, a_mn=1, b_mn=1, ksplit=ks, out_f=dw.ptr(), ln_s=pg, ln_b=pbe, dbias=pdb,
             wmaster=pW, dln_s=flat(dg), dln_b=flat(dbt))
        assert_exact(f'dW ksplit={ks}', dw.get(), ref_dw)
        assert_exact(f'dgamma ksplit={ks}', dg.get()[:, :, 0], ref_dg)
        assert_exact(f'dbeta ksplit={ks}', dbt.get()[:, :, 0], ref_dbt)
        for o, nm in ((dw, 'dW'), (dg, 'dgamma'), (dbt, 'dbeta')):
            o.check_untouched(f'{nm} ksplit={ks}')


# ------------------------------------------------------------------------------------------------------------------------------
# row kernels of the critic chain and the bf16 column sums
# ------------------------------------------------------------------------------------------------------------------------------
def _gelu_err(z):
    return 0.5 * np.abs(z) * EPS_TANH + U24 * 16 * (np.abs(z) + 1e-30)


def _ln_fwd_bound(g, e):
    """first-order bound on xhat, mu and rstd/rstd from per-element errors e of g (rows on the last axis), plus the fp32 statistics"""
    mu = g.mean(-1, keepdims=True)
    var = np.maximum((g * g).mean(-1, keepdims=True) - mu * mu, 0)
    sig = np.sqrt(var + O.LN_EPS)
    xh = (g - mu) / sig
    stat = 64 * U24 * (g * g).mean(-1, keepdims=True) / (var + O.LN_EPS)      # fp32 E[g^2] - mu^2 (cancellation) relative to var
    d_rstd = (np.abs(xh) * e).mean(-1, keepdims=True) / sig + stat            # relative
    d_mu = e.mean(-1, keepdims=True) + 64 * U24 * np.abs(g).mean(-1, keepdims=True)
    d_xh = (e + d_mu) / sig + np.abs(xh) * d_rstd
    return xh, sig, d_xh, d_mu, d_rstd


@pytest.mark.parametrize('ln', [0, 1])
@pytest.mark.parametrize('M', [1, 37, 200])
@pytest.mark.parametrize('N', [128, 256, 512])
def test_act_ln_rows(N, M, ln):
    rng = np.random.default_rng(N + M + ln)
    S, E = 2, 2
    z = rng.standard_normal((S, E, M, N)).astype(np.float32).astype(np.float64) * 1.5
    sc = rng.standard_normal((S, E, N)).astype(np.float32).astype(np.float64)
    bi = rng.standard_normal((S, E, N)).astype(np.float32).astype(np.float64) * 0.1
    tz = torch.as_tensor(z.astype(np.float32)).to(DEV)
    tsc, tbi = torch.as_tensor(sc.astype(np.float32)).to(DEV), torch.as_tensor(bi.astype(np.float32)).to(DEV)
    # the row kernels address dense [S][E][M][N] rows: flat buffers with a sentinel tail
    hd = torch.full((S * E * M * N + 64,), SENT[torch.bfloat16], dtype=torch.bfloat16, device=DEV)
    mud = torch.full((S * E * M + 64,), SENT[torch.float32], device=DEV)
    rsd = torch.full((S * E * M + 64,), SENT[torch.float32], device=DEV)
    _lib.check(_lib.lib().fql_test_act_ln_bf16(tz.data_ptr(), tsc.data_ptr() if ln else None, tbi.data_ptr() if ln else None, E * N, N,
                                               hd.data_ptr(), mud.data_ptr() if ln else None, rsd.data_ptr() if ln else None, M, N, S, E, ln,
                                               _stream()), 'act_ln')
    torch.cuda.synchronize()
    assert (hd[S * E * M * N:].float() == SENT[torch.bfloat16]).all()
    got = hd[:S * E * M * N].double().cpu().numpy().reshape(S, E, M, N)
    glo, ghi = gelu_interval(z)
    g = 0.5 * (glo + ghi)
    e = 0.5 * (ghi - glo) + _gelu_err(z)
    if not ln:
        assert_within(f'gelu rows N={N}', got, glo, ghi, (1 + 2.0 ** -8) * _gelu_err(z) + 2.0 ** -8 * np.maximum(np.abs(glo), np.abs(ghi)))
        assert (mud.cpu() == SENT[torch.float32]).all() and (rsd.cpu() == SENT[torch.float32]).all()
        return
    xh, sig, d_xh, d_mu, d_rstd = _ln_fwd_bound(g, e)
    ref = xh * sc[:, :, None, :] + bi[:, :, None, :]
    tol = (1 + 2.0 ** -8) * (np.abs(sc[:, :, None, :]) * d_xh + 8 * U24 * (np.abs(xh * sc[:, :, None, :]) + np.abs(bi[:, :, None, :]))) \
        + 2.0 ** -8 * np.abs(ref)
    assert_within(f'LayerNorm(gelu) rows N={N}', got, ref, ref, tol)
    gm = mud[:S * E * M].double().cpu().numpy().reshape(S, E, M)
    gr = rsd[:S * E * M].double().cpu().numpy().reshape(S, E, M)
    assert_within('mu', gm, g.mean(-1), g.mean(-1), d_mu[..., 0])
    assert_within('rstd', gr, 1 / sig[..., 0], 1 / sig[..., 0], (d_rstd[..., 0] + 4 * U24) / sig[..., 0])
    assert (mud[S * E * M:].cpu() == SENT[torch.float32]).all() and (rsd[S * E * M:].cpu() == SENT[torch.float32]).all()


def _z_rows(rng, S, E, M, N, Mcap, scale=1.5):
    """Z rows of group (s, e) at (s * z_rows_s + e * z_rows_e + r) * N inside a larger buffer (the grouped pass layout with Mcap
    rows per group and a problem offset), NOT contiguous with dH"""
    zbuf = rng.standard_normal((S * E * Mcap + 3) * N).astype(np.float32).astype(np.float64) * scale
    off = 3 * N
    z = np.stack([np.stack([zbuf[off + (s * E * Mcap + e * Mcap) * N: off + (s * E * Mcap + e * Mcap + M) * N].reshape(M, N)
                            for e in range(E)]) for s in range(S)])
    return zbuf, off, z, Mcap, E * Mcap


@pytest.mark.parametrize('M', [1, 37, 200])
@pytest.mark.parametrize('N', [128, 256, 512])
def test_ln_bwd_rows(N, M):
    rng = np.random.default_rng(N * 3 + M)
    S, E = 2, 2
    zbuf, off, z, ze, zs = _z_rows(rng, S, E, M, N, M + 5)
    dh = rng.standard_normal((S, E, M, N)).astype(np.float32).astype(np.float64)
    sc = rng.standard_normal((S, E, N)).astype(np.float32).astype(np.float64)
    tzb = torch.as_tensor(zbuf.astype(np.float32)).to(DEV)
    tdh = torch.as_tensor(dh.astype(np.float32)).to(DEV)
    tsc = torch.as_tensor(sc.astype(np.float32)).to(DEV)
    n = S * E * M * N
    dzf = torch.full((n + 64,), SENT[torch.float32], device=DEV)
    dzb = torch.full((n + 64,), SENT[torch.bfloat16], dtype=torch.bfloat16, device=DEV)
    _lib.check(_lib.lib().fql_test_ln_bwd_bf16(tdh.data_ptr(), tzb.data_ptr() + 4 * off, tsc.data_ptr(), E * N, N, dzf.data_ptr(), dzb.data_ptr(),
                                               M, N, S, E, ze, zs, _stream()), 'ln_bwd')
    torch.cuda.synchronize()
    th = tanh_u(z)
    g = gelu_th(z, th)
    e = 0.5 * np.abs(z) * EPS_TANH + _gelu_err(z)
    dlo, dhi = gelu_grad_interval(z)
    dg = gelu_grad_th(z, th)
    f = np.maximum(dhi - dg, dg - dlo) + 16 * U24 * (1 + np.abs(z))
    xh, sig, d_xh, _, d_rstd = _ln_fwd_bound(g, e)
    dx = dh * sc[:, :, None, :]
    m1 = dx.mean(-1, keepdims=True)
    m2 = (dx * xh).mean(-1, keepdims=True)
    v = (dx - m1 - xh * m2) / sig
    ref = v * dg
    dv = np.abs(v) * d_rstd + (d_xh * np.abs(m2) + np.abs(xh) * (np.abs(dx) * d_xh).mean(-1, keepdims=True)) / sig \
        + 64 * U24 * (np.abs(dx) + np.abs(m1) + np.abs(xh * m2) + np.abs(dx).mean(-1, keepdims=True) + np.abs(xh) * np.abs(dx * xh).mean(-1, keepdims=True)) / sig
    tol = dv * np.abs(dg) + np.abs(v) * f
    assert_within(f'LayerNorm bwd fp32 N={N}', dzf[:n].double().cpu().numpy().reshape(S, E, M, N), ref, ref, tol)
    assert_within(f'LayerNorm bwd bf16 N={N}', dzb[:n].double().cpu().numpy().reshape(S, E, M, N), ref, ref, tol * (1 + 2.0 ** -8) + 2.0 ** -8 * np.abs(ref))
    assert (dzf[n:].cpu() == SENT[torch.float32]).all() and (dzb[n:].float().cpu() == SENT[torch.bfloat16]).all()


@pytest.mark.parametrize('M', [1, 37, 200])
@pytest.mark.parametrize('N', [128, 512])
def test_gelu_bwd_rows(N, M):
    rng = np.random.default_rng(N * 5 + M)
    S, E = 2, 2
    zbuf, off, z, ze, zs = _z_rows(rng, S, E, M, N, M + 3)
    dh = rng.standard_normal((S, E, M, N)).astype(np.float32).astype(np.float64)
    tzb = torch.as_tensor(zbuf.astype(np.float32)).to(DEV)
    tdh = torch.as_tensor(dh.astype(np.float32)).to(DEV)
    n = S * E * M * N
    dzf = torch.full((n + 64,), SENT[torch.float32], device=DEV)
    dzb = torch.full((n + 64,), SENT[torch.bfloat16], dtype=torch.bfloat16, device=DEV)
    _lib.check(_lib.lib().fql_test_gelu_bwd_bf16(tdh.data_ptr(), tzb.data_ptr() + 4 * off, dzf.data_ptr(), dzb.data_ptr(), M, N, S, E, ze, zs,
                                                 _stream()), 'gelu_bwd')
    torch.cuda.synchronize()
    dlo, dhi = gelu_grad_interval(z)
    cands = np.stack([dh * dlo, dh * dhi])
    lo, hi = cands.min(0), cands.max(0)
    tol = np.abs(dh) * 16 * U24 * (1 + np.abs(z)) + U24 * np.abs(hi)
    assert_within(f'gelu bwd fp32 N={N}', dzf[:n].double().cpu().numpy().reshape(S, E, M, N), lo, hi, tol)
    assert_within(f'gelu bwd bf16 N={N}', dzb[:n].double().cpu().numpy().reshape(S, E, M, N), lo, hi,
                  tol * (1 + 2.0 ** -8) + 2.0 ** -8 * np.maximum(np.abs(lo), np.abs(hi)))
    assert (dzf[n:].cpu() == SENT[torch.float32]).all() and (dzb[n:].float().cpu() == SENT[torch.bfloat16]).all()


@pytest.mark.parametrize('M', [1, 7, 255, 256, 257, 16384])
def test_colsum_bf16_exact(M):
    """bias gradients from the bf16 dZ saves: column sums ADDED into the output ([g1][g0] strides of the grouped critic)"""
    rng = np.random.default_rng(M)
    G0, G1, N = 2, 3, 512
    x = ints(rng, (G1 * G0, M, N))
    tx = torch.as_tensor(x.astype(np.float32)).to(torch.bfloat16).to(DEV)
    os0, os1 = N + 64, 3 * (N + 64)                               # leaves apart, as in the gradient arena
    out = torch.full((G1 * os1 + 64,), SENT[torch.float32], device=DEV)
    init = ints(rng, (G1, G0, N), lim=100)
    ov = out[:G1 * os1].view(G1, 3, N + 64)
    ov[:, :G0, :N] = torch.as_tensor(init.astype(np.float32)).to(DEV)
    snap = out.clone()
    _lib.check(_lib.lib().fql_test_colsum_bf16(tx.data_ptr(), G1 * G0, M, N, out.data_ptr(), os0, G0, os1, _stream()), 'colsum')
    torch.cuda.synchronize()
    ref = init + x.reshape(G1, G0, M, N).sum(2)
    assert_exact('colsum', ov[:, :G0, :N].double().cpu().numpy(), ref)
    keep = torch.ones_like(out, dtype=torch.bool)
    keep[:G1 * os1].view(G1, 3, N + 64)[:, :G0, :N] = False
    assert int((keep & (out.view(torch.int32) != snap.view(torch.int32))).sum()) == 0


# ------------------------------------------------------------------------------------------------------------------------------
# forward chains through the public ABI against a same-rounding oracle
# ------------------------------------------------------------------------------------------------------------------------------
# Per-element absolute bounds (actions are O(1) and clipped to [-1, 1]).  Measured worst on one B200 (power limit 1000 W) over
# every case below: sample_actions 4.1e-3, compute_flow_actions 1.3e-3; the bounds sit about 2.4x above.  Dropping the bias of one
# 32-column slice of layer 1 in one CTA of the cluster Euler kernel moves compute_flow_actions by 7e-2 or more.
CHAIN_TOL_SAMPLE, CHAIN_TOL_FLOW = 1e-2, 3e-3


@pytest.mark.parametrize('env', [{}, {'FQL_B200_CHAIN_MIN_TILES': '1'}], ids=['default', 'CHAIN_MIN_TILES=1'])
@pytest.mark.parametrize('pseed', [0, 1])
@pytest.mark.parametrize('rows', [1, 127, 128, 129, 1000, 6144])
def test_forward_chains_same_rounding(rows, pseed, env, monkeypatch):
    """fql_sample_actions (chain kernel, chain2_tc.cu) and fql_compute_flow_actions (cluster Euler kernel at hidden 512,
    euler_cluster.cu) per row against the fp64 oracle with the kernels' storage rounding: bf16 weights and layer inputs, fp32
    Euler state, bf16 action / time columns.  The stand-alone entry points choose their kernel from the hidden width alone, so the
    6144-row case (48 row tiles, where the step switches to the per-tile chain kernels) and FQL_B200_CHAIN_MIN_TILES run the same
    kernels at more clusters."""
    from tests.helpers import cuda_agent_from_state, f32, make_case
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    F, A = 29, 8
    cfg, state, _, _ = make_case(dict(), 8, F, A, seed=100 + pseed, hidden=512, jitter=0.5)   # biases large enough that losing one shows
    agent = cuda_agent_from_state(cfg, state, 8, F, A, precision='bf16')
    params = f32(state['params'])
    agent.load_tree(params)
    rng = np.random.default_rng(rows + 10 * pseed)
    obs = rng.standard_normal((rows, F)).astype(np.float32)
    nz = rng.standard_normal((rows, A)).astype(np.float32)
    p64 = O.cast_tree(params, np.float64)
    o64, n64 = obs.astype(np.float64), nz.astype(np.float64)
    a = agent.sample_actions(obs, noise=nz)
    ref = O.sample_actions_given_noise(p64, cfg, o64, n64, q=bf16_round)
    e1 = np.abs(np.asarray(a, np.float64) - ref).max(-1)
    fa = agent.compute_flow_actions(obs, nz)
    ref2 = O.compute_flow_actions(p64, cfg, o64, n64, q=bf16_round)
    e2 = np.abs(np.asarray(fa, np.float64) - ref2).max(-1)
    print(f'rows={rows} seed={pseed} {env}: worst row error sample_actions {e1.max():.3e}, compute_flow_actions {e2.max():.3e}')
    assert e1.max() <= CHAIN_TOL_SAMPLE, (int(np.argmax(e1)), e1.max())
    assert e2.max() <= CHAIN_TOL_FLOW, (int(np.argmax(e2)), e2.max())
