"""CPU-side check of the shipped SASS (no GPU needed: cuobjdump reads the cross-compiled library).

1. The contractions really are tcgen05 / TMEM / TMA code (UTCHMMA, UTMALDG, LDTM, UTCBAR present).
2. The single-thread roles (TMA producer, MMA issuer) are compiled warp-uniform: with their loops under `if (lane == 0)` ptxas wraps EVERY
   tcgen05.mma / tcgen05.commit / TMA instruction in an ELECT + R2UR.BROADCAST waterfall (measured: 178 instead of 139 ns per two MMAs +
   commit, profiles/micro/mma_dual_bench.cu; DESIGN.md section 5).  A kernel whose R2UR.BROADCAST count approaches its UTCHMMA count has
   fallen back into that pattern.
"""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, 'fql_b200', 'libfql_b200.so')


@pytest.fixture(scope='module')
def sass_counts():
    cuobjdump = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(cuobjdump):
        pytest.skip('cuobjdump not available')
    if not os.path.exists(LIB):
        pytest.skip('libfql_b200.so not built (python -c "import __graft_entry__ as g; g.build()")')
    out = subprocess.run([cuobjdump, '-sass', LIB], capture_output=True, text=True, check=True).stdout
    counts, name = {}, None
    for line in out.splitlines():
        m = re.search(r'Function : (\S+)', line)
        if m:
            name = m.group(1)
            counts[name] = dict(mma=0, bcast=0, tma=0, ldtm=0, commit=0)
            continue
        if name is None:
            continue
        c = counts[name]
        if 'UTCHMMA' in line:
            c['mma'] += 1
        elif 'R2UR.BROADCAST' in line:
            c['bcast'] += 1
        elif 'UTMALDG' in line:
            c['tma'] += 1
        elif 'LDTM' in line:
            c['ldtm'] += 1
        elif 'UTCBAR' in line:
            c['commit'] += 1
    return counts


def _family(counts, key):
    return {k: v for k, v in counts.items() if key in k}


def test_contractions_are_tcgen05_tmem_tma(sass_counts):
    for fam in ('euler_cluster_kernel', 'mlp_chain2_kernel', 'tc_gemm_kernel', 'conv_tc_kernel'):
        ks = _family(sass_counts, fam)
        assert ks, fam
        for name, c in ks.items():
            assert c['mma'] > 0 and c['tma'] > 0 and c['ldtm'] > 0 and c['commit'] > 0, (name, c)


def test_single_thread_roles_are_warp_uniform(sass_counts):
    for fam in ('euler_cluster_kernel', 'mlp_chain2_kernel', 'tc_gemm_kernel', 'conv_tc_kernel'):
        for name, c in _family(sass_counts, fam).items():
            assert c['bcast'] <= max(12, c['mma'] // 4), (name, c)
