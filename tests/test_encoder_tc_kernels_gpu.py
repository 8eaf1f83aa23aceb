"""The tensor-core ImpalaEncoder (fql_b200/csrc/encoder_tc.cu) kernel by kernel, through the test hooks of include/fql_b200.h, against
oracle/encoder_oracle.py: the max pool and its gradient, the frame layer (enc_image + the first convolution at 1/255), the convolution
epilogues and geometries the public fql_conv3x3_* entry points cannot reach, and whole encoder passes checked against references that
are fed the device's OWN saved activations (teacher forcing).  Teacher forcing is what makes tight checks possible: when the device
and an independent reference round differently, a relu or max-pool decision can come out differently and re-route one element's
gradient completely (tests/test_pixels_gpu.py documents this); fed the device's saved tensors, the reference takes the same decisions
and only arithmetic is left to compare.

Exact checks (bit-equal, or equal as values where only the sign of a zero could differ):
  * pool forward: out, relu(out) and the argmax byte ky * 3 + kx against encoder_oracle.pool_fwd (first maximum in row-major order,
    -inf SAME padding) on tie-heavy, all-negative and Gaussian inputs;
  * pool backward: small-integer upstream gradients against pool_bwd (exact in any summation order); Gaussian ones against an fp32 sum
    in the kernel's fixed window order (yo, then xo ascending) rounded to nearest-even bf16; pixels no window routes to are +0;
  * the frames as bf16 (img): the integers 0..255 of the real channels, zeros above;
  * convolutions of an exact family -- activations small integers, weights and biases small integers x 2^-3, so that every product
    and partial sum is exact in fp32 in any order (|partial sums| <= 9 * 32 * 8 * 8 * 2^-3 + |bias| << 2^21, on a 2^-3 grid) and
    the bf16 outputs must be bf16_round of the fp64 reference; weight gradients use activations in [-2, 2] and gradients in [-1, 1],
    so that the sums over up to 2^20 pixels stay integers below 2^21 and gw / gb are exact as well;
  * whole forward pass: r1 == relu(p), flat == relu(xs[2]), stack 2's p / arg == pool_fwd(y0) (after a forward-only pass y0 still
    holds stack 2's pre-pool output; the backward reuses y0 for the pooling gradients, so after it stack 2's pool is checked like
    those of stacks 0 and 1), the prepared bf16 weight matrices and Dense kernel; whole backward pass: dzb == bf16(dz).

Bounded checks (u = 2^-24; P = the same contraction on absolute values, K = its depth; all derived, not fitted):
  * fp32 accumulation in any order: |acc - exact| <= u (K + 8) P.  The epilogue fmaf(acc, scale, bias) adds u |v| (one rounding; the
    reference uses the same fp32 scale, so 1/255 itself adds nothing), a skip addend one more u |v|.
  * a bf16 output must lie in the bf16 bracket [bf16(v - tol), bf16(v + tol)] of the fp64 reference v widened by that tol (round to
    nearest is monotone); relu is applied to both ends where the kernel applies it.  The printed ratio is |got - v| over tol plus half
    a bf16 unit at the output, which the bracket keeps <= 1.
  * max pool of bracketed convolution outputs (stacks 0 and 1, whose pre-pool output is overwritten by the next stack): p lies in
    [pool(lo), pool(hi)]; arg points at an element whose bracket holds p, and at the unique maximum wherever one window element's lower
    end exceeds every other element's upper end.
  * z = flat @ bf16(Wd) + bd and the Dense gradients (fp32 outputs of tc_gemm / the column sum): u (K + 8) P + u |v|.
  * feat = gelu(z) with accurate tanhf and dz = dfeat gelu'(z): u = C (z + A z^3) is five fp32 roundings (bounded by 7 u C (|z| +
    A |z|^3) with the rounded constant), tanhf <= 2 ulp (CUDA C Programming Guide), the remaining products and sums a few u of their
    value: |feat - gelu(z)| <= 0.5 |z| (du + 2^-21) + 2^-22 |gelu(z)| and |dz - dfeat gelu'(z)| <= |dfeat| ((0.5 + |z| u'(z)) (du +
    2^-21) + 2^-21 (1 + |z| u'(z))) + 2^-23 |dz|, u'(z) = C (1 + 3 A z^2).
  * every convolution leaf of the whole backward pass, tensor-norm relative (max |g - r| / max |r|) against an fp64 backward that takes
    the relu masks and argmaxes from the device's saved r1, r2, p, arg and flat, starts from the device's dzb and rounds to bf16 where
    the device stores (dx, dc1, dpool, dc0): 2e-3.  What is left is an fp32 value that lands on the other side of a bf16 rounding
    boundary from its fp64 reference (a one-unit storage flip), propagated linearly.  The bound is an estimate of that, not a
    measurement.

Every output buffer starts full of a finite sentinel and has a slack tail of one 128-pixel tile of 32 channels plus 64 elements; what
lies outside the written region must come back bit-unchanged (for the encoder pass: every float of the gradient arena outside this
network's encoder leaves, including the padding of those leaves, and the workspace beyond the size the pass reports).
Every test prints its worst error / bound.
"""
import ctypes as C
import math
import time

import numpy as np
import pytest
import torch

from fql_b200 import _lib
from oracle import encoder_oracle as E

pytestmark = pytest.mark.gpu

DEV = 'cuda'
U24 = 2.0 ** -24
S255 = float(np.float32(1.0 / 255.0))          # the fp32 scale the kernels apply to the frame layer
GC, GA = math.sqrt(2.0 / math.pi), 0.044715
SENT = {torch.bfloat16: -1232.0, torch.float32: -12345.5, torch.uint8: 0xEE}
SLACK = 128 * 32 + 64
BITS = {torch.bfloat16: torch.int16, torch.float32: torch.int32, torch.uint8: torch.uint8}
TOL_LEAF = 2e-3


def _stream():
    return torch.cuda.current_stream().cuda_stream


def bfr(x):
    """round to nearest-even bf16 (through fp32, as the device stores an fp32 value), as float64"""
    return E.bf16_round(np.asarray(x, np.float32)).astype(np.float64)


def ints(rng, shape, lim, scale=1.0):
    v = rng.integers(-lim, lim + 1, shape).astype(np.float64)
    v[rng.random(shape) < 0.2] = 0.0
    return v * scale


def gauss(rng, shape, scale=1.0):
    return bfr(rng.standard_normal(shape) * scale)


def to_dev(a, dtype):
    return torch.as_tensor(np.ascontiguousarray(a, np.float32)).to(dtype).to(DEV) if dtype != torch.uint8 else \
        torch.as_tensor(np.ascontiguousarray(a, np.uint8)).to(DEV)


def report(what, err, bound):
    ratio = float(np.max(err / np.maximum(bound, 1e-300))) if np.size(err) else 0.0
    print(f'{what}: max |err| {float(np.max(err)) if np.size(err) else 0.0:.3e}, worst err / bound {ratio:.3f}')
    return ratio


def assert_exact(what, got, ref):
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    bad = got != ref
    assert not bad.any(), (what, int(bad.sum()), np.argwhere(bad)[:4].tolist(), got[bad][:4].tolist(), ref[bad][:4].tolist())
    print(f'{what}: exact ({got.size} elements)')


def assert_within(what, got, ref, tol):
    err = np.abs(got - ref)
    bad = ~(err <= tol)
    assert not bad.any(), (what, int(bad.sum()), np.argwhere(bad)[:4].tolist(), got[bad][:4].tolist(), ref[bad][:4].tolist())
    return report(what, err, tol)


def half_unit(x):
    """half a bf16 unit in the last place at |x|"""
    x = np.maximum(np.abs(x), 2.0 ** -126)
    return np.exp2(np.floor(np.log2(x)) - 8)


def assert_bracket(what, got, v, tol, relu=False):
    """got (bf16 values) inside [bf16(v - tol), bf16(v + tol)] (relu of both ends when the kernel applies relu before rounding)"""
    lo, hi = v - tol, v + tol
    if relu:
        lo, hi = np.maximum(lo, 0), np.maximum(hi, 0)
    lo, hi = bfr(lo), bfr(hi)
    bad = (got < lo) | (got > hi)
    assert not bad.any(), (what, int(bad.sum()), np.argwhere(bad)[:4].tolist(), got[bad][:4].tolist(), v[bad][:4].tolist(), tol[bad][:4].tolist())
    ref = np.maximum(v, 0) if relu else v
    return report(what, np.abs(got - ref), tol + half_unit(np.maximum(np.abs(got), np.abs(ref))))


def rel_err(g, r):
    den = np.abs(r).max()
    return float(np.abs(g - r).max() / den) if den > 0 else float(np.abs(g).max())


class Buf:
    """device output of n elements followed by SLACK, all holding the sentinel of its type"""

    def __init__(self, n, dtype):
        self.n, self.dtype = n, dtype
        self.t = torch.full((n + SLACK,), SENT[dtype], dtype=dtype, device=DEV)
        self.snap = self.t.view(BITS[dtype]).clone()

    def ptr(self):
        return self.t.data_ptr()

    def get(self, shape, n=None):
        v = self.t[:self.n if n is None else n]
        return (v.cpu().numpy() if self.dtype == torch.uint8 else v.double().cpu().numpy()).reshape(shape)

    def bits(self, shape):
        return self.t[:self.n].view(BITS[self.dtype]).cpu().numpy().reshape(shape)

    def check_untouched(self, what, written=None):
        """elements [written, n + SLACK) are bit-unchanged (written defaults to n)"""
        w = self.n if written is None else written
        changed = self.t.view(BITS[self.dtype])[w:] != self.snap[w:]
        n = int(changed.sum())
        assert n == 0, (what, 'elements outside the written region changed', n, (torch.nonzero(changed)[:4].flatten() + w).tolist())


def chunked(fn, *arrays, chunk=8):
    """fn over batch chunks of the arrays, results concatenated on the batch axis (keeps the fp64 im2col of the oracle small)"""
    B = arrays[0].shape[0]
    return np.concatenate([fn(*[a[i:i + chunk] for a in arrays]) for i in range(0, B, chunk)])


def conv_ref(x, w, b):
    """encoder_oracle.conv_fwd and the same contraction on absolute values (the accumulation bound's P)"""
    v = chunked(lambda xc: E.conv_fwd(xc, w, b), x)
    P = chunked(lambda xc: E.conv_fwd(np.abs(xc), np.abs(w), 0.0), x)
    return v, P


def wgrad_ref(x, dy, cout):
    """(dW, db) of encoder_oracle.conv_bwd summed over batch chunks, and the same sums on absolute values"""
    cin = x.shape[-1]
    w0 = np.zeros((3, 3, cin, cout))
    gw, gb, pw, pb = 0.0, 0.0, 0.0, 0.0
    for i in range(0, x.shape[0], 8):
        _, dw, db = E.conv_bwd(x[i:i + 8], w0, dy[i:i + 8])
        _, adw, adb = E.conv_bwd(np.abs(x[i:i + 8]), w0, np.abs(dy[i:i + 8]))
        gw, gb, pw, pb = gw + dw, gb + db, pw + adw, pb + adb
    return gw, gb, pw, pb


def dgrad_ref(dy, w):
    """input gradient of encoder_oracle.conv_bwd"""
    B, H, W, _ = dy.shape
    return chunked(lambda d: E.conv_bwd(np.zeros(d.shape[:3] + (w.shape[2],)), w, d)[0], dy)


# ------------------------------------------------------------------------------------------------------------------------------
# hooks
# ------------------------------------------------------------------------------------------------------------------------------
def pool_fwd_dev(x, B, H, W, Cc):
    Ho, Wo = (H + 1) // 2, (W + 1) // 2
    n = B * Ho * Wo * Cc
    out, orl, arg = Buf(n, torch.bfloat16), Buf(n, torch.bfloat16), Buf(n, torch.uint8)
    xin = to_dev(x, torch.bfloat16)
    _lib.check(_lib.lib().fql_test_pool_bf16(xin.data_ptr(), out.ptr(), orl.ptr(), arg.ptr(), B, H, W, Cc, _stream()), 'fql_test_pool_bf16')
    torch.cuda.synchronize()
    return out, orl, arg


def pool_bwd_dev(dout, arg, B, H, W, Cc):
    din = Buf(B * H * W * Cc, torch.bfloat16)
    d, a = to_dev(dout, torch.bfloat16), to_dev(arg, torch.uint8)
    _lib.check(_lib.lib().fql_test_pool_bwd_bf16(d.data_ptr(), a.data_ptr(), din.ptr(), B, H, W, Cc, _stream()), 'fql_test_pool_bwd_bf16')
    torch.cuda.synchronize()
    return din


_WS = {}


def conv_dev(mode, B, H, W, cin, cin_p, cout, *, x=None, w=None, dy=None, bias=None, mask=None, add=None, relu_out=0, scale=1.0,
             out_relu=False):
    """one fql_test_conv_bf16 call; array arguments are uploaded (x may also be a device pointer).  Returns the output Bufs."""
    if 'ws' not in _WS:
        nb = int(_lib.lib().fql_conv3x3_workspace_bytes())
        _WS['ws'], _WS['nb'] = torch.empty(nb, dtype=torch.uint8, device=DEV), nb
    keep = []

    def up(a, dtype):
        if a is None:
            return None
        if isinstance(a, int):
            return a
        t = to_dev(a, dtype)
        keep.append(t)
        return t.data_ptr()
    c = _lib.FqlTestConv()
    c.mode, c.B, c.H, c.W, c.cin, c.cin_p, c.cout, c.scale, c.relu_out = mode, B, H, W, cin, cin_p, cout, scale, relu_out
    c.x, c.w, c.dy, c.bias = up(x, torch.bfloat16), up(w, torch.float32), up(dy, torch.bfloat16), up(bias, torch.float32)
    c.mask, c.add = up(mask, torch.bfloat16), up(add, torch.bfloat16)
    c.workspace, c.ws_bytes = _WS['ws'].data_ptr(), _WS['nb']
    npix = B * H * W
    res = {}
    if mode == _lib.TEST_CONV_WGRAD:
        res['gw'], res['gb'] = Buf(9 * cin_p * cout, torch.float32), Buf(cout, torch.float32)
        c.gw, c.gb = res['gw'].ptr(), res['gb'].ptr()
    else:
        res['out'] = Buf(npix * (cout if mode == _lib.TEST_CONV_FWD else cin), torch.bfloat16)
        c.out = res['out'].ptr()
        if out_relu:
            res['out_relu'] = Buf(npix * cout, torch.bfloat16)
            c.out_relu = res['out_relu'].ptr()
    _lib.check(_lib.lib().fql_test_conv_bf16(C.byref(c), _stream()), 'fql_test_conv_bf16')
    torch.cuda.synchronize()
    return res


# ------------------------------------------------------------------------------------------------------------------------------
# max pool 3x3 / 2 SAME
# ------------------------------------------------------------------------------------------------------------------------------
# (B, H, W, C): the three stack inputs of config 5 at B = 256; the odd 20 -> 10 -> 5 -> 3 chain; 1x1, 2x2, 1x9, 5x7.  The small ones
# launch B Ho Wo C / 8 threads, not a multiple of the 256-thread block (e.g. 5 x 3 x 3 x 2 = 90).
POOL_SHAPES = [(256, 64, 64, 16), (256, 32, 32, 32), (256, 16, 16, 32), (5, 20, 20, 16), (5, 10, 10, 32), (5, 5, 5, 32), (5, 3, 3, 32),
               (3, 1, 1, 16), (3, 2, 2, 32), (4, 1, 9, 16), (2, 5, 7, 32), (7, 5, 7, 16)]


def pool_input(rng, family, shape):
    if family == 'ties':       # a handful of bf16 levels (no -0), every third image constant per channel: windows of equal values
        x = rng.choice(np.array([-3.0, -1.0, -0.5, 0.0, 0.5, 1.0, 2.0, 3.0]), shape)
        x[::3] = x[::3, :1, :1, :]
        return x
    if family == 'negative':   # the -inf padding must never win, the argmax must point inside the image
        return -bfr(np.abs(rng.standard_normal(shape)) + 2.0 ** -4)
    return gauss(rng, shape)


@pytest.mark.parametrize('B,H,W,Cc', POOL_SHAPES)
def test_pool_forward_exact(B, H, W, Cc):
    rng = np.random.default_rng(B * 100 + H * 10 + W)
    Ho, Wo = (H + 1) // 2, (W + 1) // 2
    for family in ('ties', 'negative', 'gauss'):
        x = pool_input(rng, family, (B, H, W, Cc))
        ref, arg, pad = E.pool_fwd(x.astype(np.float32))
        out, orl, ga = pool_fwd_dev(x, B, H, W, Cc)
        shp = (B, Ho, Wo, Cc)
        assert_exact(f'pool {family} {B}x{H}x{W}x{Cc} out', out.get(shp), ref.astype(np.float64))
        assert_exact(f'pool {family} out_relu', orl.get(shp), np.maximum(ref, 0).astype(np.float64))
        assert_exact(f'pool {family} argmax', ga.get(shp), arg.astype(np.uint8))
        if family == 'negative':   # a pointer into the padding would name a tap outside the image
            ky, kx = ga.get(shp) // 3, ga.get(shp) % 3
            iy = 2 * np.arange(Ho)[None, :, None, None] + ky - pad[0]
            ix = 2 * np.arange(Wo)[None, None, :, None] + kx - pad[1]
            assert ((iy >= 0) & (iy < H) & (ix >= 0) & (ix < W)).all()
        for b, w in ((out, 'out'), (orl, 'out_relu'), (ga, 'arg')):
            b.check_untouched(f'pool {family} {w}')


def pool_bwd_fixed_order(dout, arg, H, W):
    """fp32 sum of the routed upstream gradients in pool_bwd_bf16_kernel's order: windows yo = (y + lo) / 2 - 1, (y + lo) / 2, each
    over xo likewise (a zero is added where a window does not route to the pixel: adding +0 leaves an fp32 sum unchanged)"""
    B, Ho, Wo, Cc = dout.shape
    lo_h, lo_w = ((Ho - 1) * 2 + 3 - H) // 2, ((Wo - 1) * 2 + 3 - W) // 2
    y, x = np.arange(H), np.arange(W)
    s = np.zeros((B, H, W, Cc), np.float32)
    for a in (0, 1):
        yo = (y + lo_h) // 2 - 1 + a
        ky = y + lo_h - 2 * yo
        vy = (yo >= 0) & (yo < Ho) & (ky >= 0) & (ky <= 2)
        for b in (0, 1):
            xo = (x + lo_w) // 2 - 1 + b
            kx = x + lo_w - 2 * xo
            vx = (xo >= 0) & (xo < Wo) & (kx >= 0) & (kx <= 2)
            yc, xc = np.clip(yo, 0, Ho - 1), np.clip(xo, 0, Wo - 1)
            d = dout[:, yc][:, :, xc].astype(np.float32)
            g = arg[:, yc][:, :, xc]
            me = ky[:, None] * 3 + kx[None, :]
            take = (vy[:, None] & vx[None, :])[None, :, :, None] & (g == me[None, :, :, None])
            s = s + np.where(take, d, np.float32(0.0))
    return s


@pytest.mark.parametrize('B,H,W,Cc', POOL_SHAPES)
def test_pool_backward_exact(B, H, W, Cc):
    rng = np.random.default_rng(B * 101 + H * 10 + W)
    Ho, Wo = (H + 1) // 2, (W + 1) // 2
    x = pool_input(rng, 'ties', (B, H, W, Cc))
    _, arg, pad = E.pool_fwd(x.astype(np.float32))
    arg = arg.astype(np.uint8)
    routes = E.pool_bwd(np.ones((B, Ho, Wo, Cc)), arg, x.shape, pad)
    shp = (B, H, W, Cc)
    # small integers: exact in any summation order
    dout = ints(rng, (B, Ho, Wo, Cc), 8)
    din = pool_bwd_dev(dout, arg, B, H, W, Cc)
    assert_exact(f'pool backward integers {B}x{H}x{W}x{Cc}', din.get(shp), bfr(E.pool_bwd(dout, arg, x.shape, pad)))
    din.check_untouched('pool backward integers')
    # Gaussian: the fp32 sum in the kernel's window order, rounded once
    dout = gauss(rng, (B, Ho, Wo, Cc))
    din = pool_bwd_dev(dout, arg, B, H, W, Cc)
    ref = pool_bwd_fixed_order(dout, arg, H, W)
    assert_exact('pool backward Gaussian (bits)', din.bits(shp), (E.bf16_round(ref).view(np.int32) >> 16).astype(np.int16))
    # a pixel no window routes to gets exactly +0
    unrouted = routes == 0
    assert unrouted.any() or H * W <= 2
    assert_exact('pool backward unrouted pixels (bits)', din.bits(shp)[unrouted], np.zeros(int(unrouted.sum()), np.int16))
    din.check_untouched('pool backward Gaussian')


# ------------------------------------------------------------------------------------------------------------------------------
# convolutions the public entry points cannot reach (exact family)
# ------------------------------------------------------------------------------------------------------------------------------
def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.mark.parametrize('B,H,W', [(256, 8, 8), (5, 3, 3)])   # stack 2's last convolution of config 5 and of the 20-pixel chain
def test_conv_out_relu_with_skip_exact(B, H, W):
    """xs = conv(r2) + b + p and flat = relu(xs) from ONE epilogue (relu_out = 0, out_relu set): both bit-equal"""
    rng = np.random.default_rng(B + H)
    cc = 32
    x, w, b, skip = ints(rng, (B, H, W, cc), 8), ints(rng, (3, 3, cc, cc), 8, 2.0 ** -3), ints(rng, cc, 16, 2.0 ** -3), ints(rng, (B, H, W, cc), 8)
    r = conv_dev(_lib.TEST_CONV_FWD, B, H, W, cc, cc, cc, x=x, w=w, bias=b, add=skip, relu_out=0, out_relu=True)
    ref = chunked(lambda xc: E.conv_fwd(xc, w, b), x) + skip
    shp = (B, H, W, cc)
    assert (ref < 0).any() and (ref > 0).any()
    assert_exact(f'conv + skip {B}x{H}x{W} out', r['out'].get(shp), bfr(ref))
    assert_exact('conv + skip out_relu', r['out_relu'].get(shp), bfr(np.maximum(ref, 0)))
    r['out'].check_untouched('out')
    r['out_relu'].check_untouched('out_relu')


# (name, B, H, W, cin, cin_p, cout): config 5's stack-0 geometry at B = 256 (8192 pixel tiles = 55-56 per persistent CTA on 148 SMs;
# an odd operand-buffer count once aliased a barrier parity at exactly this count) with the 9 real channels of the frame layer in
# a 16-channel tensor, and stack 1's 16 -> 32 first convolution at 32 x 32
SCALE_CASES = [('stack0', 256, 64, 64, 9, 16, 16), ('stack1-conv0', 256, 32, 32, 16, 16, 32)]


@pytest.mark.parametrize('mode', ['forward', 'input-gradient', 'weight-gradient'])
@pytest.mark.parametrize('name,B,H,W,cin,cin_p,cout', SCALE_CASES)
def test_conv_exact_at_scale(name, B, H, W, cin, cin_p, cout, mode):
    rng = np.random.default_rng([B, H, cin, cout, ('forward', 'input-gradient', 'weight-gradient').index(mode)])
    t0 = time.time()
    tiles = -(-B * H * W // 128)
    print(f'{name} {mode}: {tiles} pixel tiles, {-(-tiles // min(tiles, sm_count()))} per CTA')
    w = ints(rng, (3, 3, cin, cout), 8, 2.0 ** -3)
    if mode == 'forward':
        x = ints(rng, (B, H, W, cin_p), 8)        # channels >= cin are finite garbage: the prepared weights must zero them
        b = ints(rng, cout, 16, 2.0 ** -3)
        r = conv_dev(_lib.TEST_CONV_FWD, B, H, W, cin, cin_p, cout, x=x, w=w, bias=b, out_relu=True)
        ref = conv_ref(x[..., :cin], w, b)[0]
        assert_exact(f'{name} forward', r['out'].get((B, H, W, cout)), bfr(ref))
        assert_exact(f'{name} forward out_relu', r['out_relu'].get((B, H, W, cout)), bfr(np.maximum(ref, 0)))
        r['out'].check_untouched('out')
        r['out_relu'].check_untouched('out_relu')
    elif mode == 'input-gradient':
        if cin != cin_p:
            cin = cin_p
            w = ints(rng, (3, 3, cin, cout), 8, 2.0 ** -3)
        dy, mask, add = ints(rng, (B, H, W, cout), 8), gauss(rng, (B, H, W, cin)), ints(rng, (B, H, W, cin), 8)
        mask[rng.random(mask.shape) < 0.1] = 0.0
        r = conv_dev(_lib.TEST_CONV_DGRAD, B, H, W, cin, cin, cout, x=dy, w=w, mask=mask, add=add)
        ref = dgrad_ref(dy, w) * (mask > 0) + add
        assert_exact(f'{name} input gradient', r['out'].get((B, H, W, cin)), bfr(ref))
        r['out'].check_untouched('out')
    else:
        x, dy = ints(rng, (B, H, W, cin_p), 2), ints(rng, (B, H, W, cout), 1)
        r = conv_dev(_lib.TEST_CONV_WGRAD, B, H, W, cin, cin_p, cout, x=x, dy=dy)
        gw, gb, pw, pb = wgrad_ref(x[..., :cin], dy, cout)
        assert pw.max() < 2 ** 21 and pb.max() < 2 ** 21          # every partial sum is an integer below 2^21: exact in fp32
        assert_exact(f'{name} weight gradient', r['gw'].get((3, 3, cin, cout), n=9 * cin * cout), gw)
        assert_exact(f'{name} bias gradient', r['gb'].get(cout), gb)
        r['gw'].check_untouched('gw', 9 * cin * cout)
        r['gb'].check_untouched('gb')
    print(f'{name} {mode}: {time.time() - t0:.1f} s')


# ------------------------------------------------------------------------------------------------------------------------------
# whole encoder passes
# ------------------------------------------------------------------------------------------------------------------------------
def enc_leaves(dims, net):
    leaves, arena = _lib.layout(dims)
    return [l for l in leaves if l['net'] == net and l['path'][0] == 'encoder'], arena


def encoder_params(dims, rng, Cimg, hw):
    """an fp32 arena of noise with every network's encoder leaves set from encoder_oracle.init_encoder (a wrong offset reads noise)"""
    leaves, arena = _lib.layout(dims)
    params = (rng.standard_normal(arena) * 0.05).astype(np.float32)
    trees = {}
    for l in leaves:
        if l['path'][0] != 'encoder':
            continue
        tree = trees.setdefault(l['net'], E.init_encoder(rng, Cimg, hw=hw, jitter=0.05))
        a = np.asarray(tree[l['path'][1]][l['path'][2]][l['name']], np.float32)
        assert a.size == l['rows'] * l['cols'] * l['ens'], (l['path'], a.shape)
        params[l['offset']:l['offset'] + a.size] = a.ravel()
    return params, trees


def frames(rng, B, H, W, Cimg):
    obs = rng.integers(0, 256, (B, H, W, Cimg)).astype(np.uint8)
    if B >= 3:
        obs[0], obs[1] = 0, 255
    return obs


class EncoderPass:
    """fql_test_encoder_bf16 on one network: forward (+ backward when dfeat is given); the carved buffers read back by name"""

    def __init__(self, dims, net, params, obs, dfeat=None):
        lib = _lib.lib()
        B = obs.shape[0]
        self.B = B
        off = (C.c_int64 * _lib.TEST_ENC_NOFF)()
        dptr = C.c_void_p(1) if dfeat is not None else None
        _lib.check(lib.fql_test_encoder_bf16(C.byref(dims), _lib.NET_NAMES.index(net), None, None, B, dptr, None, None, None, 0, off, None),
                   'fql_test_encoder_bf16 size')
        self.need = int(off[_lib.TEST_ENC_NOFF - 1])
        self.ws = torch.full((self.need + SLACK,), 0xEE, dtype=torch.uint8, device=DEV)     # finite bf16 / fp32 bit pattern
        self.ws_tail = self.ws[self.need:].clone()
        p, o = torch.as_tensor(params).to(DEV), to_dev(obs, torch.uint8)
        self.feat = Buf(B * 512, torch.float32)
        self.grads = None
        df = None
        if dfeat is not None:
            df = torch.as_tensor(np.ascontiguousarray(dfeat, np.float32)).to(DEV)
            self.grads = torch.full((params.size + 64,), SENT[torch.float32], dtype=torch.float32, device=DEV)
        _lib.check(lib.fql_test_encoder_bf16(C.byref(dims), _lib.NET_NAMES.index(net), p.data_ptr(), o.data_ptr(), B,
                                             df.data_ptr() if df is not None else None, self.feat.ptr(),
                                             self.grads.data_ptr() if self.grads is not None else None, self.ws.data_ptr(), self.need + SLACK,
                                             off, _stream()), 'fql_test_encoder_bf16')
        torch.cuda.synchronize()
        self.off = {k: int(off[i]) for i, k in enumerate(_lib.TEST_ENC_BUFS)}
        assert int(off[_lib.TEST_ENC_NOFF - 1]) == self.need
        assert torch.equal(self.ws[self.need:], self.ws_tail), 'the encoder pass wrote past the workspace size it reports'

    def get(self, name, shape, dtype=torch.bfloat16):
        o = self.off[name]
        assert o >= 0, name
        n = int(np.prod(shape)) * torch.tensor([], dtype=dtype).element_size()
        t = self.ws[o:o + n].view(dtype)
        return (t.cpu().numpy() if dtype == torch.uint8 else t.double().cpu().numpy()).reshape(shape)


def geometry(H, W):
    Hs, Ws = [H], [W]
    for _ in range(3):
        Hs.append((Hs[-1] + 1) // 2)
        Ws.append((Ws[-1] + 1) // 2)
    return Hs, Ws


def windows(x):
    """[9, B, Ho, Wo, C] windows of encoder_oracle.pool_fwd (the same -inf SAME padding)"""
    B, H, W, Cc = x.shape
    Ho, Wo = (H + 1) // 2, (W + 1) // 2
    ph, pw = max((Ho - 1) * 2 + 3 - H, 0), max((Wo - 1) * 2 + 3 - W, 0)
    xp = np.pad(x, ((0, 0), (ph // 2, ph - ph // 2), (pw // 2, pw - pw // 2), (0, 0)), constant_values=-np.inf)
    return np.stack([xp[:, ky:ky + 2 * Ho:2, kx:kx + 2 * Wo:2, :] for ky in range(3) for kx in range(3)], axis=0)


def conv_bracket(xin, w, b, scale, cin_p=None):
    """fp64 pre-activation v = scale * conv(xin, w) + b and its fp32 tolerance (accumulation over the K = 9 cin_p products the kernel
    forms, + the fmaf rounding)"""
    acc, P = conv_ref(xin, w, 0.0)
    v = scale * acc + b
    return v, scale * U24 * (9 * (cin_p or w.shape[2]) + 8) * P + U24 * np.abs(v)


def check_pool_of_bracket(what, p, arg, v, tol):
    """p / arg of a max pool whose input is only known to lie in the bf16 bracket of v +- tol"""
    lo, hi = bfr(v - tol).astype(np.float32), bfr(v + tol).astype(np.float32)
    wl, wh = windows(lo), windows(hi)
    plo, phi = wl.max(0), wh.max(0)
    bad = (p < plo) | (p > phi)
    assert not bad.any(), (what, 'p outside [pool(lo), pool(hi)]', int(bad.sum()), np.argwhere(bad)[:4].tolist())
    a = arg.astype(np.int64)[None]
    sl, sh = np.take_along_axis(wl, a, 0)[0], np.take_along_axis(wh, a, 0)[0]
    bad = (sl > p) | (sh < p)
    assert not bad.any(), (what, 'arg points at an element that cannot hold the maximum', int(bad.sum()), np.argwhere(bad)[:4].tolist())
    j = wl.argmax(0)
    wh_other = wh.copy()
    np.put_along_axis(wh_other, j[None], -np.inf, 0)
    uniq = np.take_along_axis(wl, j[None], 0)[0] > wh_other.max(0)
    assert_exact(f'{what} arg at the unique maxima ({int(uniq.sum())} of {uniq.size})', arg[uniq], j[uniq].astype(np.uint8))
    return report(f'{what} p in [pool(lo), pool(hi)]', np.maximum(np.maximum(plo - p, p - phi), 0), np.maximum(phi - plo, 1e-30))


def gelu_du(z):
    return 7 * U24 * GC * (np.abs(z) + GA * np.abs(z) ** 3)


def check_forward(ep, trees_net, obs, Cimg, y0_kept=True):
    """every saved activation of the forward pass against references fed the device's own inputs (see the module docstring).
    y0_kept: y0 still holds stack 2's pre-pool output -- false after a backward pass, which reuses y0 for the pooling gradients."""
    B, H, W = obs.shape[:3]
    Hs, Ws = geometry(H, W)
    img = ep.get('img', (B, H, W, 16))
    ref_img = np.zeros((B, H, W, 16))
    ref_img[..., :Cimg] = obs
    assert_exact('img', img, ref_img)
    xin, scale = img[..., :Cimg], S255
    for i, f in enumerate(E.STACKS):
        blk = trees_net[f'stack_blocks_{i}']
        H1, W1 = Hs[i + 1], Ws[i + 1]
        shp = (B, H1, W1, f)
        p, r1, r2, xs = (ep.get(f'{k}{i}', shp) for k in ('p', 'r1_', 'r2_', 'xs'))
        arg = ep.get(f'arg{i}', shp, torch.uint8)
        v, tol = conv_bracket(xin, bfr(blk['Conv_0']['kernel']), blk['Conv_0']['bias'].astype(np.float64), scale, 16 if i == 0 else None)
        if i == 2 and y0_kept:
            y0 = ep.get('y0', (B, Hs[i], Ws[i], f))
            assert_bracket(f'stack {i} conv0 (y0)', y0, v, tol)
            ref, ref_arg, _ = E.pool_fwd(y0)
            assert_exact(f'stack {i} p == pool(y0)', p, ref)
            assert_exact(f'stack {i} arg == argmax(y0)', arg, ref_arg.astype(np.uint8))
        else:
            check_pool_of_bracket(f'stack {i} pool(conv0)', p, arg, v, tol)
        assert_exact(f'stack {i} r1 == relu(p)', r1, np.maximum(p, 0))
        v, tol = conv_bracket(r1, bfr(blk['Conv_1']['kernel']), blk['Conv_1']['bias'].astype(np.float64), 1.0)
        assert_bracket(f'stack {i} r2 = relu(conv1(r1))', r2, v, tol, relu=True)
        v, tol = conv_bracket(r2, bfr(blk['Conv_2']['kernel']), blk['Conv_2']['bias'].astype(np.float64), 1.0)
        assert_bracket(f'stack {i} xs = conv2(r2) + p', xs, v + p, tol + U24 * np.abs(v + p))
        xin, scale = xs, 1.0
    flat_dim = Hs[3] * Ws[3] * 32
    flat = ep.get('flat', (B, flat_dim))
    assert_exact('flat == relu(xs[2])', flat, np.maximum(xin, 0).reshape(B, flat_dim))
    d = trees_net['MLP_0']['Dense_0']
    wd = bfr(d['kernel'])
    z = ep.get('z', (B, 512), torch.float32)
    zr = flat @ wd + d['bias']
    assert_within('z = flat @ bf16(Wd) + bd', z, zr, U24 * (flat_dim + 8) * (np.abs(flat) @ np.abs(wd)) + U24 * np.abs(zr))
    feat = ep.feat.get((B, 512))
    g = E.gelu_tanh(z)
    assert_within('feat = gelu(z)', feat, g, 0.5 * np.abs(z) * (gelu_du(z) + 2.0 ** -21) + 2.0 ** -22 * np.abs(g))
    ep.feat.check_untouched('feat')
    # the prepared operands: bf16 forward [k = tap * cin_p + ci][co] and input-gradient [k = tap * cout + co][ci] (flipped taps)
    # matrices of the nine convolutions in [320][64] slots, zero elsewhere; the Dense kernel
    wf, wdg = ep.get('wf', (9, 320, 64)), ep.get('wd', (9, 320, 64))
    cin = Cimg
    for i, f in enumerate(E.STACKS):
        for j in range(3):
            k = bfr(trees_net[f'stack_blocks_{i}'][f'Conv_{j}']['kernel'])
            ci = cin if j == 0 else f
            cp = 16 if (i == 0 and j == 0) else ci
            ref = np.zeros((320, 64))
            kp = np.zeros((3, 3, cp, f))
            kp[:, :, :ci] = k
            ref[:9 * cp, :f] = kp.reshape(9 * cp, f)
            assert_exact(f'prepared forward matrix {i}.{j}', wf[3 * i + j], ref)
            ref = np.zeros((320, 64))
            ref[:9 * f, :ci] = np.flip(k, (0, 1)).transpose(0, 1, 3, 2).reshape(9 * f, ci)
            assert_exact(f'prepared input-gradient matrix {i}.{j}', wdg[3 * i + j], ref)
        cin = f
    assert_exact('prepared Dense kernel', ep.get('wdense', (flat_dim, 512)), wd)


FWD_CASES = [(64, 64, 9, 1), (64, 64, 9, 256), (16, 16, 6, 6), (20, 20, 3, 5)]


@pytest.mark.parametrize('H,W,Cimg,B', FWD_CASES)
def test_encoder_forward_teacher_forced(H, W, Cimg, B):
    t0 = time.time()
    rng = np.random.default_rng(H * 1000 + B)
    dims = _lib.make_dims(B, 512, 5, hidden=64, precision=_lib.PRECISION_BF16_ENC, image=(H, W, Cimg))
    params, trees = encoder_params(dims, rng, Cimg, H)
    obs = frames(rng, B, H, W, Cimg)
    ep = EncoderPass(dims, 'critic', params, obs)
    check_forward(ep, trees['critic'], obs, Cimg)
    print(f'forward {H}x{W}x{Cimg} B={B}: {time.time() - t0:.1f} s')


def backward_reference(ep, tree, obs, Cimg, dzb):
    """fp64 backward with the device's masks / argmaxes / saved activations, bf16 rounding where the device stores"""
    B, H, W = obs.shape[:3]
    Hs, Ws = geometry(H, W)
    flat_dim = Hs[3] * Ws[3] * 32
    flat = ep.get('flat', (B, flat_dim))
    wd = bfr(tree['MLP_0']['Dense_0']['kernel'])
    g = {}
    dx = bfr((dzb @ wd.T) * (flat > 0)).reshape(B, Hs[3], Ws[3], 32)
    for i in reversed(range(3)):
        f = E.STACKS[i]
        blk = tree[f'stack_blocks_{i}']
        shp = (B, Hs[i + 1], Ws[i + 1], f)
        p, r1, r2 = (ep.get(f'{k}{i}', shp) for k in ('p', 'r1_', 'r2_'))
        arg = ep.get(f'arg{i}', shp, torch.uint8)
        gi = {}
        dr2, gi['Conv_2/kernel'], gi['Conv_2/bias'] = E.conv_bwd(r2, bfr(blk['Conv_2']['kernel']), dx)
        dc1 = bfr(dr2 * (r2 > 0))
        dr1, gi['Conv_1/kernel'], gi['Conv_1/bias'] = E.conv_bwd(r1, bfr(blk['Conv_1']['kernel']), dc1)
        dpool = bfr(dx + dr1 * (r1 > 0))
        pad = (((Hs[i + 1] - 1) * 2 + 3 - Hs[i]) // 2, ((Ws[i + 1] - 1) * 2 + 3 - Ws[i]) // 2)
        dc0 = bfr(E.pool_bwd(dpool, arg, (B, Hs[i], Ws[i], f), pad))
        if i > 0:
            xin = ep.get(f'xs{i - 1}', (B, Hs[i], Ws[i], E.STACKS[i - 1]))
            dxin, gi['Conv_0/kernel'], gi['Conv_0/bias'] = E.conv_bwd(xin, bfr(blk['Conv_0']['kernel']), dc0)
            dx = bfr(dxin)
        else:
            xin = ep.get('img', (B, H, W, 16))[..., :Cimg]
            _, gw, gi['Conv_0/bias'] = E.conv_bwd(xin, bfr(blk['Conv_0']['kernel']), dc0)
            gi['Conv_0/kernel'] = gw * S255
        g[f'stack_blocks_{i}'] = gi
    return g


def check_backward(ep, dims, net, tree, obs, Cimg, dfeat):
    B, H, W = obs.shape[:3]
    Hs, Ws = geometry(H, W)
    flat_dim = Hs[3] * Ws[3] * 32
    z = ep.get('z', (B, 512), torch.float32)
    dz = ep.get('dz', (B, 512), torch.float32)
    du = 0.0 + GC * (1 + 3 * GA * z * z)
    ref = dfeat * E.gelu_tanh_grad(z)
    tol = np.abs(dfeat) * ((0.5 + np.abs(z) * du) * (gelu_du(z) + 2.0 ** -21) + 2.0 ** -21 * (1 + np.abs(z) * du)) + 2.0 ** -23 * np.abs(ref)
    ratios = [assert_within('dz = dfeat gelu\'(z)', dz, ref, tol)]
    dzb = ep.get('dzb', (B, 512))
    assert_exact('dzb == bf16(dz)', dzb, bfr(dz))
    flat = ep.get('flat', (B, flat_dim))
    wd = bfr(tree['MLP_0']['Dense_0']['kernel'])
    dflat = ep.get('dflat', (B, flat_dim), torch.float32)
    ref = dzb @ wd.T
    ratios.append(assert_within('dflat = dzb @ bf16(Wd)^T', dflat, ref, U24 * (512 + 8) * (np.abs(dzb) @ np.abs(wd).T) + U24 * np.abs(ref)))
    leaves, arena = enc_leaves(dims, net)
    grads = ep.grads.cpu().numpy().astype(np.float64)
    ref_g = backward_reference(ep, tree, obs, Cimg, dzb)
    written = np.zeros(grads.size, bool)
    worst = 0.0
    for l in leaves:
        n = l['rows'] * l['cols'] * l['ens']
        got = grads[l['offset']:l['offset'] + n]
        written[l['offset']:l['offset'] + n] = True
        name = '/'.join(l['path'][1:]) + '/' + l['name']
        if l['path'][1] == 'MLP_0':
            if l['name'] == 'kernel':
                r = flat.T @ dzb
                ratios.append(assert_within(f'{net} {name}', got.reshape(flat_dim, 512), r, U24 * (B + 8) * (np.abs(flat).T @ np.abs(dzb)) + U24 * np.abs(r)))
            else:
                r = dz.sum(0)
                ratios.append(assert_within(f'{net} {name}', got, r, U24 * (B + 8) * np.abs(dz).sum(0) + U24 * np.abs(r)))
            continue
        r = np.asarray(ref_g[l['path'][1]][f"{l['path'][2]}/{l['name']}"]).ravel()
        e = rel_err(got, r)
        assert e <= TOL_LEAF, (net, name, e)
        worst = max(worst, e)
    print(f'{net}: convolution leaves, worst tensor-norm-relative error {worst:.2e}, worst err / bound {worst / TOL_LEAF:.3f}')
    untouched = ep.grads.view(torch.int32).cpu().numpy()
    keep = ~written
    sent = np.array([SENT[torch.float32]], np.float32).view(np.int32)[0]
    changed = keep & (untouched != sent)
    assert not changed.any(), (net, 'gradient floats outside the encoder leaves changed', int(changed.sum()), np.argwhere(changed)[:4].ravel().tolist())
    return max(ratios + [worst / TOL_LEAF])


BWD_CASES = [(16, 16, 6, 6), (20, 20, 3, 5)]


@pytest.mark.parametrize('precision', ['bf16-enc', 'bf16'])
@pytest.mark.parametrize('H,W,Cimg,B', BWD_CASES)
def test_encoder_backward_teacher_forced(H, W, Cimg, B, precision):
    """every network's encoder (all four carry one) in both tensor-core modes"""
    t0 = time.time()
    prec = {'bf16-enc': _lib.PRECISION_BF16_ENC, 'bf16': _lib.PRECISION_BF16_TC}[precision]
    rng = np.random.default_rng(H * 1000 + B + prec)
    dims = _lib.make_dims(B, 512, 5, hidden=64, precision=prec, image=(H, W, Cimg))
    params, trees = encoder_params(dims, rng, Cimg, H)
    obs = frames(rng, B, H, W, Cimg)
    for net in _lib.NET_NAMES:
        dfeat = rng.standard_normal((B, 512)).astype(np.float32)
        ep = EncoderPass(dims, net, params, obs, dfeat)
        check_forward(ep, trees[net], obs, Cimg, y0_kept=False)
        check_backward(ep, dims, net, trees[net], obs, Cimg, dfeat.astype(np.float64))
    print(f'backward {H}x{W}x{Cimg} B={B} {precision}: {time.time() - t0:.1f} s')


def test_encoder_backward_teacher_forced_config5():
    """config 5 (64 x 64 x 9 frames) at its batch size 256, the critic's encoder"""
    t0 = time.time()
    H, W, Cimg, B = 64, 64, 9, 256
    rng = np.random.default_rng(5)
    dims = _lib.make_dims(B, 512, 5, hidden=64, precision=_lib.PRECISION_BF16_ENC, image=(H, W, Cimg))
    params, trees = encoder_params(dims, rng, Cimg, H)
    obs = frames(rng, B, H, W, Cimg)
    dfeat = rng.standard_normal((B, 512)).astype(np.float32)
    ep = EncoderPass(dims, 'critic', params, obs, dfeat)
    check_backward(ep, dims, 'critic', trees['critic'], obs, Cimg, dfeat.astype(np.float64))
    print(f'backward 64x64x9 B=256: {time.time() - t0:.1f} s')


# ------------------------------------------------------------------------------------------------------------------------------
# the frame layer: enc_image + the first convolution (16-channel tensor, cin real channels, scale 1/255, bias)
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('Cimg', [3, 6, 9, 16])
def test_frame_layer(Cimg):
    B, H, W = 4, 64, 64                       # image 0 all 0, image 1 all 255, two random
    rng = np.random.default_rng(Cimg)
    dims = _lib.make_dims(B, 512, 5, hidden=64, precision=_lib.PRECISION_BF16_ENC, image=(H, W, Cimg))
    params, trees = encoder_params(dims, rng, Cimg, H)
    obs = frames(rng, B, H, W, Cimg)
    ep = EncoderPass(dims, 'critic', params, obs)
    img = ep.get('img', (B, H, W, 16))
    ref_img = np.zeros((B, H, W, 16))
    ref_img[..., :Cimg] = obs
    assert_exact(f'img C={Cimg}', img, ref_img)
    img_ptr = ep.ws.data_ptr() + ep.off['img']
    w = trees['critic']['stack_blocks_0']['Conv_0']['kernel'].astype(np.float64)
    b = trees['critic']['stack_blocks_0']['Conv_0']['bias'].astype(np.float64)
    r = conv_dev(_lib.TEST_CONV_FWD, B, H, W, Cimg, 16, 16, x=img_ptr, w=w, bias=b, scale=S255)
    v, tol = conv_bracket(img[..., :Cimg], bfr(w), b, S255, 16)
    ratio = assert_bracket(f'frame layer forward C={Cimg}', r['out'].get((B, H, W, 16)), v, tol)
    r['out'].check_untouched('frame layer forward')
    dy = gauss(rng, (B, H, W, 16))
    r = conv_dev(_lib.TEST_CONV_WGRAD, B, H, W, Cimg, 16, 16, x=img_ptr, dy=dy, scale=S255)
    gw, gb, pw, pb = wgrad_ref(img[..., :Cimg], dy, 16)
    n = B * H * W
    ratio = max(ratio, assert_within(f'frame layer weight gradient C={Cimg}', r['gw'].get((3, 3, Cimg, 16), n=9 * Cimg * 16), S255 * gw,
                                     S255 * U24 * (n + 8) * pw + U24 * S255 * np.abs(gw)))
    ratio = max(ratio, assert_within(f'frame layer bias gradient (not scaled) C={Cimg}', r['gb'].get(16), gb, U24 * (n + 8) * pb))
    r['gw'].check_untouched('gw: exactly 9 C cout weights are written', 9 * Cimg * 16)
    r['gb'].check_untouched('gb')
