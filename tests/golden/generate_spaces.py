"""Generate the MultiDiscrete golden vectors by running the UNMODIFIED reference (/root/reference) in this container.

    python tests/golden/generate_spaces.py      # writes tests/golden/spaces_serial.npz and experience_md.npz

  spaces_serial.npz  pufferlib.vector.make(ocean.env_creator('spaces'), backend=Serial) with np.random.seed fixed, driven
                     by a seeded [H, N, 2] action tape: the native observation of every reset, every recv() row, the
                     infos, the emulated spaces and record layout, and the reference models.Default parameter names /
                     shapes for this env.                        [ocean.py:356-404, emulation.py:68-120, models.py:12-62]
  experience_md.npz  clean_pufferl.Experience with atn_shape = (2,): store -> sort_training_data -> compute_gae ->
                     flatten_batch, including the [nm, rows, bptt, 2] b_actions.

Uses the gymnasium stand-ins of ``oracle/shim`` through generate.py.  gymnasium 0.29 sorts the keys of a plain-dict
``spaces.Dict`` (and keeps insertion order when they do not compare); the stand-in keeps insertion order, which no other
fixture depends on, so this script applies gymnasium's rule to it for the run.  The Dict layout of the emulated
observation and the MultiDiscrete action columns follow that order.
"""
import os
import sys
from collections import OrderedDict

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from generate import HERE, load_c_gae  # noqa: E402  (sets up the shim and the reference on sys.path)

import gymnasium.spaces  # noqa: E402
import numpy as np  # noqa: E402
import torch  # noqa: E402

import pufferlib  # noqa: E402
import pufferlib.vector  # noqa: E402
from pufferlib.environments import ocean  # noqa: E402


def _sorted_dict_init(init):
    def __init__(self, spaces=None, **kw):
        if isinstance(spaces, dict) and not isinstance(spaces, OrderedDict):
            try:
                spaces = dict(sorted(spaces.items()))
            except TypeError:
                pass
        init(self, spaces, **kw)
    return __init__


gymnasium.spaces.Dict.__init__ = _sorted_dict_init(gymnasium.spaces.Dict.__init__)


def run_spaces(num_envs, seed, horizon, np_seed):
    """The reference's ocean `spaces` env (ocean.py:356-404: Dict obs, Dict({'image', 'flat'}) of Discrete(2) actions
    that emulation turns into MultiDiscrete([2, 2])) behind Serial, driven by a seeded [H, N, 2] action tape.  The env
    draws from numpy's process-global stream, so np.random.seed is fixed; the native observation of every reset is
    recorded (in reset order) so that a restatement with another RNG can be fed the same observations."""
    from pufferlib.environments.ocean import ocean as ocean_envs
    resets = []
    orig_reset = ocean_envs.Spaces.reset

    def recording_reset(self, seed=None):
        out = orig_reset(self, seed)
        resets.append((self.observation['flat'].copy(), self.observation['image'].copy()))
        return out
    ocean_envs.Spaces.reset = recording_reset
    try:
        np.random.seed(np_seed)
        vec = pufferlib.vector.make(ocean.env_creator('spaces'), num_envs=num_envs, backend=pufferlib.vector.Serial)
        resets.clear()          # construction resets (EpisodeStats.__init__) are not part of the rollout
        tape = np.random.default_rng(seed).integers(0, 2, size=(horizon, num_envs, 2), dtype=np.int64)
        obs, rew, term, trunc, mask, info_rows = [], [], [], [], [], []
        vec.async_reset(seed)
        for t in range(horizon + 1):
            o, r, d, tr, infos, env_id, m = vec.recv()
            assert np.array_equal(env_id, np.arange(num_envs))
            obs.append(o.copy()); rew.append(r.copy()); term.append(d.copy()); trunc.append(tr.copy()); mask.append(m.copy())
            for k, i in enumerate(infos):
                info_rows.append((t, k, i['episode_return'], i['episode_length'], i['score']))
            if t < horizon:
                vec.send(tape[t])
        drv = vec.driver_env
        out = dict(
            num_envs=num_envs, seed=seed, np_seed=np_seed, horizon=horizon, actions=tape,
            obs=np.stack(obs), rewards=np.stack(rew), terminals=np.stack(term), truncations=np.stack(trunc),
            masks=np.stack(mask), infos=np.asarray(info_rows, dtype=np.float64).reshape(-1, 5),
            reset_flat=np.stack([f for f, _ in resets]), reset_image=np.stack([i for _, i in resets]),
            action_nvec=np.asarray(drv.single_action_space.nvec, dtype=np.int64),
            obs_space_shape=np.asarray(drv.single_observation_space.shape, dtype=np.int64),
            obs_space_dtype=str(drv.single_observation_space.dtype),
            obs_record_descr=repr(drv.emulated.emulated_observation_dtype.descr),
            obs_field_offsets=np.asarray([drv.emulated.emulated_observation_dtype.fields[k][1]
                                          for k in drv.emulated.emulated_observation_dtype.names], dtype=np.int64),
            obs_field_names=np.asarray(drv.emulated.emulated_observation_dtype.names),
            action_names=np.asarray(list(drv.env.action_space.keys())),
        )
        vec.close()
        return out
    finally:
        ocean_envs.Spaces.reset = orig_reset


def gen_spaces():
    """spaces_serial.npz: the Serial rollout above plus the reference models.Default parameter names / shapes for this
    env; experience_md.npz: the reference Experience with atn_shape = (2,) (store -> sort -> GAE -> flatten_batch)."""
    import clean_pufferl
    import pufferlib.models
    out = run_spaces(num_envs=7, seed=3, horizon=12, np_seed=11)
    vec = pufferlib.vector.make(ocean.env_creator('spaces'), num_envs=1, backend=pufferlib.vector.Serial)
    model = pufferlib.models.Default(vec.driver_env)
    sd = model.state_dict()
    out['param_names'] = np.asarray(list(sd.keys()))
    out['param_shapes'] = np.asarray([list(v.shape) + [0] * (2 - v.dim()) for v in sd.values()], dtype=np.int64)
    vec.close()
    np.savez_compressed(os.path.join(HERE, 'spaces_serial.npz'), **out)
    print('spaces_serial', out['obs'].shape, 'resets', out['reset_flat'].shape, 'infos', out['infos'].shape)

    compute_gae = load_c_gae()
    n, h, mbs, bptt, seed = 6, 8, 16, 4, 2
    np.random.seed(5)
    vec = pufferlib.vector.make(ocean.env_creator('spaces'), num_envs=n, backend=pufferlib.vector.Serial)
    exp = clean_pufferl.Experience(n * h, bptt, mbs, vec.single_observation_space.shape,
                                   vec.single_observation_space.dtype, vec.single_action_space.shape,
                                   cpu_offload=False, device='cpu')
    tape = np.random.default_rng(seed).integers(0, 2, size=(h, n, 2), dtype=np.int64)
    rng = np.random.default_rng(100 + seed)
    values = rng.standard_normal((h, n)).astype(np.float32)
    logprobs = -rng.random((h, n)).astype(np.float32)
    vec.async_reset(seed)
    t = 0
    while not exp.full:
        o, r, d, tr, infos, env_id, mask = vec.recv()
        exp.store(torch.as_tensor(o), torch.as_tensor(values[t]), tape[t], torch.as_tensor(logprobs[t]),
                  torch.as_tensor(r), torch.as_tensor(d), env_id.tolist(), torch.as_tensor(mask))
        vec.send(tape[t])
        t += 1
    stored = dict(obs=exp.obs.numpy().copy(), actions=exp.actions_np.copy(), logprobs=exp.logprobs_np.copy(),
                  rewards=exp.rewards_np.copy(), dones=exp.dones_np.copy(), values=exp.values_np.copy())
    idxs = exp.sort_training_data()
    gamma, lam = 0.99, 0.95
    adv = compute_gae(exp.dones_np[idxs], exp.values_np[idxs], exp.rewards_np[idxs], gamma, lam)
    exp.flatten_batch(adv)
    vec.close()
    np.savez_compressed(
        os.path.join(HERE, 'experience_md.npz'),
        num_envs=n, horizon=h, minibatch_size=mbs, bptt=bptt, seed=seed, gamma=gamma, gae_lambda=lam, tape=tape,
        values_in=values, logprobs_in=logprobs, idxs=idxs, advantages=adv, returns_np=exp.returns_np,
        b_obs=exp.b_obs.numpy(), b_actions=exp.b_actions.numpy(), b_logprobs=exp.b_logprobs.numpy(),
        b_dones=exp.b_dones.numpy(), b_values=exp.b_values.numpy(), b_advantages=exp.b_advantages.numpy(),
        b_returns=exp.b_returns.numpy(), **{'stored_' + k: v for k, v in stored.items()})
    print('experience_md', 'actions', tuple(exp.actions.shape), 'b_actions', tuple(exp.b_actions.shape))


if __name__ == '__main__':
    gen_spaces()
