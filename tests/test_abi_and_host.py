"""CPU-only checks (-m "not gpu"): the C-ABI library loads and exports every symbol the header declares, the
ctypes table matches it, and the host-side logic that needs no device behaves like the reference."""
import os
import re
import subprocess

import numpy as np
import pytest

import pufferlib_b200.vector as pvec
from pufferlib_b200 import _native, spaces
from pufferlib_b200.environments import ocean, resolve
from pufferlib_b200.exceptions import APIUsageError

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    src = open(os.path.join(REPO, 'include', 'pufferlib_b200.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(pb_[a-z0-9_]+)\s*\(', src)))


def test_library_exports_every_declared_symbol():
    assert os.path.exists(_native.SO_PATH), 'run `python -m pufferlib_b200.build` (done by __graft_entry__.build())'
    out = subprocess.check_output(['nm', '-D', '--defined-only', _native.SO_PATH], text=True)
    exported = set(re.findall(r' T (pb_[a-z0-9_]+)', out))
    declared = header_functions()
    assert len(declared) >= 18
    missing = [f for f in declared if f not in exported]
    assert not missing, f'declared in include/pufferlib_b200.h but not exported: {missing}'


def test_ctypes_table_matches_header():
    assert sorted(_native.SIGNATURES) == header_functions()
    lib = _native.lib()                      # loads without a GPU
    assert lib.pb_abi_version() == 1
    for name in _native.SIGNATURES:
        assert hasattr(lib, name)


def test_calls_fail_loudly_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip('a GPU is present')
    with pytest.raises(RuntimeError):
        pvec.make(ocean.env_creator('squared'), num_envs=4, backend=pvec.B200)
    import ctypes as C
    cfg = _native.EnvConfig(kind=0, num_envs=4, device=0)
    h = C.c_void_p()
    rc = _native.lib().pb_env_create(C.byref(cfg), C.byref(h))
    assert rc == _native.PB_ERR_CUDA and 'CUDA' in _native.last_error() or 'cuda' in _native.last_error()


def test_mlp_update_fused_rejects_dpre_out():
    """The fused update always forms dW_enc inside the kernel: a non-null dpre_out is refused before anything touches the
    device, so this holds with or without a GPU."""
    import ctypes as C
    p = C.c_void_p(1 << 20)                  # never dereferenced: the argument check comes first
    rc = _native.lib().pb_mlp_update_fused(p, 128, 128, 128, 1, *[p] * 10, 128, 4, 0.1, 1, 0.1, 0.5, 0.01, p, p, p, 1 << 30,
                                           p, None, None, None, None)
    assert rc == _native.PB_ERR_UNSUPPORTED
    assert 'dpre_out' in _native.last_error()


def test_sm100a_only_cubin():
    out = subprocess.check_output(['cuobjdump', '--list-elf', _native.SO_PATH], text=True)
    archs = set(re.findall(r'sm_\d+a?', out))
    assert archs == {'sm_100a'}, archs


class _Recorder:
    def __init__(self, creators, args, kwargs, num_envs, **kw):
        self.creators, self.args, self.kwargs, self.num_envs, self.kw = creators, args, kwargs, num_envs, kw


def test_make_validation_matches_reference_messages():
    c = ocean.env_creator('squared')
    with pytest.raises(APIUsageError, match='num_envs must be at least 1'):
        pvec.make(c, num_envs=0, backend=_Recorder)
    with pytest.raises(APIUsageError, match='num_envs must be an integer'):
        pvec.make(c, num_envs=1.5, backend=_Recorder)
    with pytest.raises(APIUsageError, match='divisible by num_workers'):
        pvec.make(c, num_envs=5, num_workers=2, backend=_Recorder)
    with pytest.raises(APIUsageError, match='batch_size must be divisible'):
        pvec.make(c, num_envs=8, num_workers=2, batch_size=6, backend=_Recorder)
    with pytest.raises(APIUsageError, match='Invalid argument'):
        pvec.make(c, num_envs=2, backend=_Recorder, nope=1)
    with pytest.raises(APIUsageError, match='list of callables'):
        pvec.make([1, 2], env_args=[[], []], env_kwargs=[{}, {}], num_envs=2, backend=_Recorder)
    with pytest.raises(APIUsageError, match='list of length num_envs'):
        pvec.make([c], env_args=[[]], env_kwargs=[{}], num_envs=2, backend=_Recorder)
    r = pvec.make(c, env_kwargs={'distance_to_target': 2}, num_envs=3, backend=_Recorder, num_workers=1)
    assert r.num_envs == 3 and len(r.creators) == 3 and r.kwargs[0] == {'distance_to_target': 2}
    assert r.kw == {'num_workers': 1}


def test_env_creator_registry():
    assert resolve(ocean.env_creator('squared'), [], {}) == ('squared', [3, 0, 0, 0, 0, 0, 0, 0])
    assert resolve(ocean.env_creator('squared'), [5], {})[1][0] == 5
    assert resolve(ocean.env_creator('squared'), [], {'distance_to_target': 2})[1][0] == 2

    def make_squared():     # the reference's creator is recognised by name (ocean/environment.py:28)
        pass
    assert resolve(make_squared, [], {})[0] == 'squared'
    with pytest.raises(APIUsageError):
        resolve(lambda: None, [], {})
    with pytest.raises(APIUsageError):
        resolve(ocean.env_creator('squared'), [], {'num_targets': 2})
    with pytest.raises(APIUsageError):
        ocean.env_creator('squared')()       # no CPU instantiation
    with pytest.raises(ValueError):
        ocean.env_creator('nope')


def test_spaces_and_joint_space():
    d = spaces.Discrete(8)
    j = pvec.joint_space(d, 5)
    assert isinstance(j, spaces.MultiDiscrete) and j.contains(np.array([0, 7, 3, 2, 1]))
    assert not j.contains(np.array([0, 8, 3, 2, 1])) and not j.contains(np.zeros(4, dtype=np.int64))
    b = spaces.Box(-1, 1, (7, 7), np.float32)
    jb = pvec.joint_space(b, 3)
    assert jb.shape == (3, 7, 7) and jb.dtype == np.float32
    assert pvec.make_seeds(10, 3) == [10, 11, 12]
    with pytest.raises(APIUsageError):
        pvec.make_seeds([1, 2], 3)


def test_sorted_permutation_is_arithmetic():
    from pufferlib_b200.clean_pufferl import _LazyIdxs
    n, h = 6, 8
    keys = [(e, t) for t in range(h) for e in range(n)]
    ref = np.asarray(sorted(range(len(keys)), key=keys.__getitem__))      # clean_pufferl.py:453-454
    assert np.array_equal(np.asarray(_LazyIdxs(n, h)), ref)
