"""CPU-side checks of the 3xTF32 tensor-core mode (FQL_PRECISION_FP32_TC, precision='fp32-tc'): the shipped SASS of its GEMM kernel
and the host-side validation of the mode.  No GPU needed."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, 'fql_b200', 'libfql_b200.so')


@pytest.fixture(scope='module')
def L():
    import __graft_entry__ as g
    g.build()
    from fql_b200 import _lib
    return _lib


def test_tf32x3_kernel_is_tcgen05_and_warp_uniform(L):
    """UTCHMMA (tcgen05.mma kind::tf32), UTCBAR (commit) and LDTM (TMEM load) present; the MMA issuer compiled warp-uniform (the same
    R2UR.BROADCAST bound tests/test_sass.py applies to the other tensor-core kernels)."""
    cuobjdump = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(cuobjdump):
        pytest.skip('cuobjdump not available')
    out = subprocess.run([cuobjdump, '-sass', LIB], capture_output=True, text=True, check=True).stdout
    counts, name = {}, None
    for line in out.splitlines():
        m = re.search(r'Function : (\S+)', line)
        if m:
            name = m.group(1)
            counts[name] = dict(mma=0, bcast=0, ldtm=0, commit=0)
        elif name is not None:
            c = counts[name]
            for key, op in (('mma', 'UTCHMMA'), ('bcast', 'R2UR.BROADCAST'), ('ldtm', 'LDTM'), ('commit', 'UTCBAR')):
                if op in line:
                    c[key] += 1
    ks = {k: v for k, v in counts.items() if 'gemm_tf32x3_kernel' in k}
    assert len(ks) == 1, list(counts)
    c = next(iter(ks.values()))
    assert c['mma'] >= 12 and c['commit'] > 0 and c['ldtm'] > 0, c      # 4 k-steps x 3 products per K block
    assert c['bcast'] <= max(12, c['mma'] // 4), c


def test_fp32_tc_dims_validate_for_state_configs(L):
    lib = L.lib()
    for kw in (dict(), dict(actor_layer_norm=True, hidden=96), dict(num_seeds=8, hidden=32)):
        d = L.make_dims(256, 29, 8, precision=L.PRECISION_FP32_TC, **kw)
        assert lib.fql_workspace_bytes(C.byref(d)) > 0, lib.fql_last_error().decode()
        assert lib.fql_shadow_bytes(C.byref(d)) == 0           # fp32 master weights only: no bf16 shadow
        d32 = L.make_dims(256, 29, 8, precision=L.PRECISION_FP32, **kw)
        assert lib.fql_workspace_bytes(C.byref(d)) == lib.fql_workspace_bytes(C.byref(d32))   # the fp32 schedule's workspace
        assert L.layout(d) == L.layout(d32)


def test_fp32_tc_refuses_pixel_dims(L):
    lib = L.lib()
    d = L.make_dims(64, 512, 4, precision=L.PRECISION_FP32_TC, image=(64, 64, 3))
    assert lib.fql_workspace_bytes(C.byref(d)) == 0
    assert lib.fql_arena_floats(C.byref(d)) == -1
    msg = lib.fql_last_error().decode()
    assert 'FQL_PRECISION_FP32_TC' in msg and 'fp32-tc' in msg, msg


def test_agent_refuses_fp32_tc_with_an_encoder():
    """Refused in FQLAgent.create before any library call (no GPU needed to reach the check)."""
    pytest.importorskip('torch')
    from fql_b200.agent import FQLAgent
    from fql_b200.config import get_config
    cfg = dict(get_config(), encoder='impala_small')
    with pytest.raises(NotImplementedError, match='fp32-tc'):
        FQLAgent.create(0, np.zeros((1, 64, 64, 3), np.uint8), np.zeros((1, 4), np.float32), cfg, precision='fp32-tc', device='cpu')
