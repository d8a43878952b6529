"""CPU checks of the MultiDiscrete path (-m "not gpu"): the `spaces` oracle against the reference's own rollout
(tests/golden/spaces_serial.npz), the env registry and spaces, the list form of sample_logits, models.Default's heads
and the C-ABI table entries of the multi-head kernels."""
import os

import numpy as np
import torch
from torch.distributions import Categorical

import pufferlib_b200.vector as pvec
from oracle import spaces as ospaces
from pufferlib_b200 import _native, models, spaces
from pufferlib_b200.environments import OBS_RECORD_DTYPE, ocean, resolve
from pufferlib_b200.frameworks import cleanrl

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = np.load(os.path.join(HERE, 'golden', 'spaces_serial.npz'))


def golden_source(g):
    """obs_source for oracle.spaces.SpacesSerial: the native observations the reference drew, in reset order."""
    n = int(g['num_envs'])
    return lambda ids, k: (g['reset_flat'][k * n + ids], g['reset_image'][k * n + ids])


def test_oracle_packs_reference_observations():
    g = GOLDEN
    n = int(g['num_envs'])
    rec = ospaces.pack(g['reset_flat'], g['reset_image'])
    assert rec.shape[1] == ospaces.RECORD_BYTES == int(g['obs_space_shape'][0])
    # reset rows of the rollout: recv 0, 2, 4, ... (every step is terminal, the next send resets)
    for t in range(0, int(g['horizon']) + 1, 2):
        assert np.array_equal(g['obs'][t], rec[(t // 2) * n:(t // 2 + 1) * n])
    # the record layout is the emulated dtype of the reference (sorted Dict keys, align=True)
    dt = OBS_RECORD_DTYPE['spaces']
    assert dt.itemsize == ospaces.RECORD_BYTES and str(g['obs_space_dtype']) == 'uint8'
    assert list(dt.names) == list(g['obs_field_names']) == ['flat', 'image']
    assert [dt.fields[k][1] for k in dt.names] == list(g['obs_field_offsets']) == [0, 8]
    assert list(g['action_names']) == ['flat', 'image'] and list(g['action_nvec']) == list(ospaces.NVEC)


def test_oracle_replays_reference_rollout():
    g = GOLDEN
    n, h = int(g['num_envs']), int(g['horizon'])
    ora = ospaces.SpacesSerial(n, obs_source=golden_source(g))
    ora.async_reset(int(g['seed']))
    info_rows = []
    for t in range(h + 1):
        o, r, d, tr, infos, env_id, m = ora.recv()
        assert np.array_equal(o, g['obs'][t]), t
        assert np.array_equal(r.view(np.uint32), g['rewards'][t].view(np.uint32)), t
        assert np.array_equal(d, g['terminals'][t]) and np.array_equal(tr, g['truncations'][t])
        assert np.array_equal(m, g['masks'][t])
        assert d.all() == (t % 2 == 1) and d.any() == (t % 2 == 1)      # reset rows and step rows alternate
        if t % 2 == 1:
            assert np.array_equal(o, g['obs'][t - 1])                   # a step shows the observation of its reset
        for k, i in enumerate(infos):
            info_rows.append((t, k, i['episode_return'], i['episode_length'], i['score']))
        if t < h:
            ora.send(g['actions'][t])
    assert np.array_equal(np.asarray(info_rows, dtype=np.float64).reshape(-1, 5), g['infos'])


def test_oracle_draws_are_exact_in_fp32():
    flat, image = ospaces.draw_observation(np.arange(4096, dtype=np.uint64) + 17, np.arange(4096) % 5)
    assert flat.min() == -1 and flat.max() == 1
    steps = image.astype(np.float64) * 128
    assert np.array_equal(steps, np.round(steps)) and np.abs(steps).max() <= 510
    fwd = image.reshape(-1, 25).sum(1, dtype=np.float32)
    rev = image.reshape(-1, 25)[:, ::-1].sum(1, dtype=np.float32)
    assert np.array_equal(fwd, rev) and np.array_equal(fwd.astype(np.float64), steps.reshape(-1, 25).sum(1) / 128)


def test_registry_and_spaces():
    assert _native.ENV_KINDS['spaces'] == 4
    assert resolve(ocean.env_creator('spaces'), [], {}) == ('spaces', [0] * 8)

    def make_spaces():      # the reference's creator is recognised by name (ocean/environment.py)
        pass
    assert resolve(make_spaces, [], {})[0] == 'spaces'
    md = spaces.MultiDiscrete([2, 2])
    j = pvec.joint_space(md, 5)
    assert isinstance(j, spaces.Box) and j.shape == (5, 2)
    assert j.contains(np.array([[0, 1]] * 5)) and not j.contains(np.array([[0, 2]] * 5))
    assert not j.contains(np.zeros((5,), dtype=np.int64))


def correct_sample_logits(logits, action=None):
    """The reference test's formulation (tests/test_cleanrl_utils.py), one Categorical per head."""
    dists = [Categorical(logits=lg) for lg in logits]
    if action is None:
        action = torch.stack([d.sample() for d in dists], 1)
    logprob = torch.stack([d.log_prob(a) for d, a in zip(dists, action.T)], 1).sum(1)
    ent = torch.stack([d.entropy() for d in dists], 1).sum(1)
    return action, logprob, ent


def test_sample_logits_list_matches_categorical():
    torch.manual_seed(0)
    batch, nvec = 8, [3, 7, 4]
    logits = [torch.randn(batch, n) for n in nvec]
    action = torch.stack([torch.randint(0, n, (batch,)) for n in nvec], 1)
    a1, l1, e1 = cleanrl.sample_logits(logits, action=action)
    a2, l2, e2 = correct_sample_logits(logits, action)
    assert a1.shape == a2.shape == (batch, 3) and torch.equal(a1, action)
    assert torch.allclose(l1, l2, atol=1e-6) and torch.allclose(e1, e2, atol=1e-6)
    a3, l3, e3 = cleanrl.sample_logits(logits)
    assert a3.shape == (batch, 3) and l3.shape == e3.shape == (batch,)
    assert all(int(a3[:, h].max()) < n for h, n in enumerate(nvec))
    _, l4, e4 = correct_sample_logits(logits, a3)
    assert torch.allclose(l3, l4, atol=1e-6) and torch.allclose(e3, e4, atol=1e-6)
    # [rows, bptt, k] actions of a minibatch are read as action.view(batch, -1).T
    a5, l5, _ = cleanrl.sample_logits(logits, action=action.view(2, 4, 3))
    assert torch.equal(a5, action) and torch.allclose(l5, l2, atol=1e-6)


class _Env:
    single_observation_space = spaces.Box(0, 255, (108,), np.uint8)
    single_action_space = spaces.MultiDiscrete([2, 2])


def test_default_heads_match_reference_names_and_shapes():
    m = models.Default(_Env())
    sd = m.state_dict()
    names = [str(x) for x in GOLDEN['param_names']]
    shapes = [tuple(int(d) for d in s if d) for s in GOLDEN['param_shapes']]
    assert list(sd.keys()) == names
    assert [tuple(v.shape) for v in sd.values()] == shapes
    assert isinstance(m.decoder, torch.nn.ModuleList) and m.n_logits == 4
    hidden = torch.randn(5, 128)
    logits, value = m.decode_actions(hidden, None)
    assert isinstance(logits, list) and [tuple(x.shape) for x in logits] == [(5, 2), (5, 2)] and value.shape == (5, 1)
    for d, lg in zip(m.decoder, logits):
        assert torch.allclose(lg, d(hidden), atol=1e-5)
    assert torch.allclose(value, m.value_head(hidden), atol=1e-5)
    w, b = m.decoder_params()
    assert torch.equal(w, torch.cat([m.decoder[0].weight, m.decoder[1].weight])) and b.shape == (4,)


def test_abi_table_has_multihead_entry_points():
    from test_abi_and_host import header_functions
    declared = header_functions()
    for name in ('pb_env_action_nvec', 'pb_sample_logits_multi', 'pb_ppo_loss_multi'):
        assert name in declared and name in _native.SIGNATURES
        assert hasattr(_native.lib(), name)
    assert sorted(_native.SIGNATURES) == declared
