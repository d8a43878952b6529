"""Pin the oracle (oracle/) against outputs of the reference itself (tests/golden/*.npz, generate.py)."""
import random

import numpy as np
import pytest

from oracle import gae as ogae
from oracle import experience as oexp
from oracle.mt19937 import MT19937
from oracle.squared import SquaredSerial, reward_table

SQUARED_CASES = ['squared_c1', 'squared_n5_seed42', 'squared_n1_seed7', 'squared_d2_n33', 'squared_d5_n8']


@pytest.mark.parametrize('seed', [0, 1, 42, 2**31 + 5, 2**32 + 7, 123456789012345])
def test_mt19937_matches_cpython_random(seed):
    mt = MT19937(seed)
    random.seed(seed)
    for _ in range(1500):   # crosses two twists
        assert mt.getrandbits(32) == random.getrandbits(32)
    for n in (24, 16, 40, 7):
        for _ in range(50):
            assert mt.randbelow(n) == random.sample(range(n), 1)[0]


def run_oracle_squared(g):
    n, seed, h = int(g['num_envs']), int(g['seed']), int(g['horizon'])
    vec = SquaredSerial(n, distance_to_target=int(g['distance_to_target']))
    vec.async_reset(seed)
    rows, infos = [], []
    for t in range(h + 1):
        o, r, d, tr, info, ids, m = vec.recv()
        rows.append((o.copy(), r.copy(), d.copy(), tr.copy(), m.copy()))
        for k, i in enumerate(info):
            infos.append((t, k, i['episode_return'], i['episode_length'], i['score']))
        if t < h:
            vec.send(g['actions'][t])
    return rows, np.asarray(infos, dtype=np.float64).reshape(-1, 5)


@pytest.mark.parametrize('case', SQUARED_CASES)
def test_squared_oracle_bit_exact(golden, case):
    g = golden(case)
    rows, infos = run_oracle_squared(g)
    for t, (o, r, d, tr, m) in enumerate(rows):
        assert np.array_equal(o, g['obs_i8'][t].astype(np.float32)), f'obs step {t}'
        assert np.array_equal(r.view(np.uint32), g['rewards'][t].view(np.uint32)), f'reward bits step {t}'
        assert np.array_equal(d, g['terminals'][t]) and np.array_equal(tr, g['truncations'][t])
        assert np.array_equal(m, g['masks'][t])
    assert np.array_equal(infos, g['infos'])   # episode_return is a python-double sum: exact


def test_reward_table_values():
    assert np.array_equal(reward_table(3), np.float32([1, 1 - 1 / 3, 1 - 2 / 3, 0, 1 - 4 / 3, 1 - 5 / 3, -1]))


def gae_inputs(n, seed, p_done):
    rng = np.random.default_rng(seed)
    rewards = rng.standard_normal(n).astype(np.float32)
    values = rng.standard_normal(n).astype(np.float32)
    dones = (rng.random(n) < p_done).astype(np.float32)
    return dones, values, rewards


def test_gae_oracle_bit_exact(golden):
    g = golden('gae')
    for k in range(int(g['num_cases'])):
        n, seed, p, gamma, lam = g[f'case{k}_meta']
        d, v, r = gae_inputs(int(n), int(seed), p)
        adv = ogae.compute_gae(d, v, r, gamma, lam)
        assert np.array_equal(adv.view(np.uint32), g[f'case{k}_adv'].view(np.uint32)), f'case {k}'
        if n <= 8192:
            assert np.array_equal(ogae.compute_gae_np(d, v, r, gamma, lam), adv)


def test_gae_oracle_empty_and_single():
    z = np.zeros(0, dtype=np.float32)
    assert ogae.compute_gae(z, z, z, 0.99, 0.95).shape == (0,)
    one = np.ones(1, dtype=np.float32)
    assert np.array_equal(ogae.compute_gae(one, one, one, 0.99, 0.95), np.zeros(1, dtype=np.float32))


@pytest.mark.parametrize('case', ['experience_c1', 'experience_small', 'experience_one_mb'])
def test_experience_oracle(golden, case):
    g = golden(case)
    n, h = int(g['num_envs']), int(g['horizon'])
    exp = oexp.Experience(n * h, int(g['bptt']), int(g['minibatch_size']), (7, 7), np.float32)
    vec = SquaredSerial(n)
    vec.async_reset(int(g['seed']))
    t = 0
    while not exp.full:
        o, r, d, tr, infos, env_id, mask = vec.recv()
        exp.store(o, g['values_in'][t], g['tape'][t], g['logprobs_in'][t], r, d, env_id, mask)
        vec.send(g['tape'][t])
        t += 1
    assert np.array_equal(exp.obs, g['stored_obs_i8'].astype(np.float32))
    for k in ('actions', 'logprobs', 'rewards', 'dones', 'values'):
        assert np.array_equal(getattr(exp, k), g['stored_' + k]), k
    idxs = exp.sort_training_data()
    assert np.array_equal(idxs, g['idxs'])
    # arithmetic form used on the device: sorted position e*H+t holds arrival row t*N+e
    e, tt = np.divmod(np.arange(n * h), h)
    assert np.array_equal(idxs, tt * n + e)
    adv = ogae.compute_gae(exp.dones[idxs], exp.values[idxs], exp.rewards[idxs], float(g['gamma']),
                           float(g['gae_lambda']))
    assert np.array_equal(adv, g['advantages'])
    exp.flatten_batch(adv)
    assert np.array_equal(exp.b_idxs_obs, g['b_idxs_obs'])
    assert np.array_equal(exp.b_obs, g['b_obs_i8'].astype(np.float32))
    for k in ('b_actions', 'b_logprobs', 'b_dones', 'b_values', 'b_advantages', 'b_returns', 'returns_np'):
        assert np.array_equal(getattr(exp, k), g[k]), k
    for mb in range(exp.num_minibatches):
        ref = g['b_advantages_normalized'][mb]
        got = oexp.normalize_advantages(exp.b_advantages[mb])
        assert np.allclose(got, ref, rtol=1e-5, atol=1e-6)


def test_experience_validation_errors():
    with pytest.raises(ValueError):
        oexp.Experience(100, 4, 30, (7, 7), np.float32)
    with pytest.raises(ValueError):
        oexp.Experience(100, 3, 50, (7, 7), np.float32)


@pytest.mark.parametrize('n,p_done,gamma,lam', [(2, 0.0, 0.99, 0.95), (1000, 0.02, 0.99, 0.95), (50000, 0.1, 0.9, 0.5),
                                                (4096, 1.0, 0.99, 0.95), (4096, 0.0, 1.0, 1.0)])
def test_gae_oracle_vs_reference_compiled_c_gae(golden, n, p_done, gamma, lam):
    """The oracle's C restatement against the reference's own c_gae.pyx (its outputs on these inputs are stored in
    c_gae_cases.npz by generate.py): bit for bit, at sizes gae.npz does not hold."""
    ref = golden('c_gae_cases')[f'cpu_{n}_{p_done}_{gamma}_{lam}']
    d, v, r = gae_inputs(n, seed=n, p_done=p_done)
    got = ogae.compute_gae(d, v, r, gamma, lam)
    assert np.array_equal(ref.view(np.uint32), got.view(np.uint32))


@pytest.mark.parametrize('case', ['squared_mp_n8_w2', 'squared_mp_n12_w4'])
def test_squared_multiprocessing_oracle_bit_exact(golden, case):
    """vector.Multiprocessing (reference run with real worker processes, tests/golden/generate.py): per-worker
    process-global MT19937 streams (vector.py:168-190) -- the oracle restates it as one SquaredSerial per worker."""
    from oracle.squared import SquaredMultiprocessing
    g = golden(case)
    assert bool(g['differs_from_serial'])       # the golden really exercises the per-worker stream consequence
    n, w, seed, h = int(g['num_envs']), int(g['num_workers']), int(g['seed']), int(g['horizon'])
    vec = SquaredMultiprocessing(n, w)
    vec.async_reset(seed)
    infos = []
    for t in range(h + 1):
        o, r, d, tr, info, ids, m = vec.recv()
        assert np.array_equal(o, g['obs_i8'][t].astype(np.float32)), f'obs step {t}'
        assert np.array_equal(r.view(np.uint32), g['rewards'][t].view(np.uint32)), f'reward bits step {t}'
        assert np.array_equal(d, g['terminals'][t]) and not tr.any() and m.all()
        for k, i in enumerate(info):
            infos.append((t, k, i['episode_return'], i['episode_length'], i['score']))
        if t < h:
            vec.send(g['actions'][t])
    assert np.array_equal(np.asarray(infos, dtype=np.float64).reshape(-1, 5), g['infos'])
