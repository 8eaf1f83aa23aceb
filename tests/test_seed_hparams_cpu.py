"""Hyperparameter sweeps as vectorised seeds, host side (no GPU): the FqlHparams.per_seed layout in the header and in ctypes,
FQLAgent.create(per_seed=...) validation before any library call, seed_config, and dist.shard_per_seed."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_ctypes_layout_of_the_table_pointer():
    from fql_b200 import _lib
    assert C.sizeof(_lib.FqlHparams) == 48
    assert _lib.FqlHparams.per_seed.offset == 40 and C.alignment(_lib.FqlHparams) == 8
    assert _lib.make_hparams().per_seed is None


def test_header_layout_of_the_table_pointer(tmp_path):
    cc = shutil.which('cc') or shutil.which('gcc')
    if cc is None:
        pytest.skip('no C compiler')
    src = tmp_path / 'layout.c'
    src.write_text('#include <stddef.h>\n#include "fql_b200.h"\n'
                   '_Static_assert(sizeof(FqlHparams) == 48, "size");\n'
                   '_Static_assert(offsetof(FqlHparams, per_seed) == 40, "offset");\n'
                   '_Static_assert(_Alignof(FqlHparams) == 8, "alignment");\n')
    r = subprocess.run([cc, '-std=c11', '-fsyntax-only', '-I', os.path.join(ROOT, 'include'), str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


@pytest.fixture
def no_library(monkeypatch):
    """Any call into libfql_b200 fails the test: validation must happen before the library is touched."""
    from fql_b200 import _lib

    def boom():
        raise AssertionError('library called')
    monkeypatch.setattr(_lib, 'lib', boom)


def _create(per_seed, num_seeds=3, **cfg_over):
    pytest.importorskip('torch')
    from fql_b200.agent import FQLAgent
    from fql_b200.config import get_config
    cfg = dict(get_config(), **cfg_over)
    return FQLAgent.create(0, np.zeros((1, 9), np.float32), np.zeros((1, 3), np.float32), cfg, num_seeds=num_seeds, per_seed=per_seed,
                           device='cpu')


@pytest.mark.parametrize('key', ['q_agg', 'flow_steps', 'normalize_q_loss', 'batch_size', 'beta1', 'Alpha'])
def test_create_rejects_keys_that_cannot_vary(no_library, key):
    with pytest.raises(ValueError) as e:
        _create({'alpha': [1.0, 2.0, 3.0], key: [1, 2, 3]})
    msg = str(e.value)
    assert repr(key) in msg and all(k in msg for k in ('alpha', 'discount', 'tau', 'lr')) and 'shared' in msg, msg


@pytest.mark.parametrize('bad', [[1.0, 2.0], [1.0, 2.0, 3.0, 4.0], [[1.0, 2.0, 3.0]], 5.0])
def test_create_rejects_wrong_lengths(no_library, bad):
    with pytest.raises(ValueError, match="per_seed\\['alpha'\\]: expected 3 values"):
        _create({'alpha': bad})


@pytest.mark.parametrize('bad', [float('nan'), float('inf'), -float('inf')])
def test_create_rejects_non_finite_values(no_library, bad):
    with pytest.raises(ValueError, match='finite'):
        _create({'tau': [0.005, bad, 0.01]})


def test_create_rejects_a_non_dict(no_library):
    with pytest.raises(ValueError, match='dict'):
        _create([('alpha', [1.0, 2.0, 3.0])])


def test_a_valid_table_passes_validation(no_library):
    """Valid input gets as far as the first library call (which the fixture turns into an AssertionError)."""
    with pytest.raises(AssertionError, match='library called'):
        _create({'alpha': [30, 300, 3000], 'discount': (0.99, 0.995, 0.9), 'tau': np.array([0.005, 0.01, 0.02]), 'lr': [3e-4] * 3})


def test_seed_config():
    from fql_b200.agent import FQLAgent, _check_per_seed
    from fql_b200.config import get_config
    a = FQLAgent.__new__(FQLAgent)
    a.config, a.num_seeds = dict(get_config()), 3
    a._per_seed = _check_per_seed({'alpha': [30, 300, 3000], 'lr': np.array([1e-4, 3e-4, 1e-3])}, 3)
    assert a.per_seed == {'alpha': (30.0, 300.0, 3000.0), 'lr': (1e-4, 3e-4, 1e-3)}
    for i in range(3):
        c = a.seed_config(i)
        assert c['alpha'] == a.per_seed['alpha'][i] and c['lr'] == a.per_seed['lr'][i]
        assert c['discount'] == a.config['discount'] and c['tau'] == a.config['tau']
        assert {k: v for k, v in c.items() if k not in ('alpha', 'lr')} == {k: v for k, v in a.config.items() if k not in ('alpha', 'lr')}
    assert a.config['alpha'] == 300.0                           # the shared config is untouched
    with pytest.raises(IndexError):
        a.seed_config(3)
    a._per_seed = _check_per_seed(None, 3)
    assert a.per_seed is None and a.seed_config(2) == a.config
    assert _check_per_seed({}, 3) is None


@pytest.mark.parametrize('S,world', [(4, 1), (4, 2), (8, 4), (6, 3), (48, 8)])
def test_shard_per_seed_slices_like_shard_seeds(S, world):
    from fql_b200 import dist as fdist
    sweep = {'alpha': [float(10 * i) for i in range(S)], 'tau': tuple(0.001 * (i + 1) for i in range(S)), 'lr': np.arange(S) * 1e-4}
    got = []
    for rank in range(world):
        mine = fdist.shard_seeds(S, rank, world)
        part = fdist.shard_per_seed(sweep, rank, world)
        assert set(part) == set(sweep)
        for k in sweep:
            assert list(part[k]) == [sweep[k][i] for i in mine], (k, rank)
        got += list(part['alpha'])
    assert got == sweep['alpha']


def test_shard_per_seed_errors_and_none():
    from fql_b200 import dist as fdist
    assert fdist.shard_per_seed(None, 1, 2) is None
    with pytest.raises(ValueError, match='differ in length'):
        fdist.shard_per_seed({'alpha': [1, 2], 'tau': [1, 2, 3, 4]}, 0, 2)
    with pytest.raises(ValueError, match='divide'):
        fdist.shard_per_seed({'alpha': [1, 2, 3]}, 0, 2)
