"""Generate golden vectors by running the UNMODIFIED reference (/root/reference) in this container.

    python tests/golden/generate.py        # writes tests/golden/*.npz

The reference cannot travel to the GPU box, so its outputs are committed here as small fixtures:

  squared_*.npz     pufferlib.vector.make(ocean.env_creator('squared'), backend=Serial) driven by a fixed
                    action tape (np.random.default_rng(0)); every recv() row (obs/reward/terminal/trunc/mask)
                    and every info dict.                        [vector.py:70-166, ocean.py:406-513]
  gae.npz           c_gae.compute_gae (the reference's Cython, built by pyximport) on seeded inputs.
  c_gae_cases.npz   c_gae.compute_gae on the inputs of the tests that compare against it at larger sizes
                    (``python tests/golden/generate.py c_gae_cases`` writes this file alone).
  experience_*.npz  clean_pufferl.Experience store -> sort_training_data -> compute_gae -> flatten_batch and
                    the per-minibatch advantage normalisation of clean_pufferl.train (torch CPU fp32).

gymnasium / gym / pettingzoo are not installed in this image; ``oracle/shim`` provides stand-ins for the
handful of classes the reference touches on this path (the reference source itself is not modified).
"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [os.path.join(REPO, 'oracle', 'shim'), '/root/reference']

import warnings
warnings.filterwarnings('ignore')
import numpy as np
import torch

import pufferlib
import pufferlib.vector
from pufferlib.environments import ocean


def action_tape(horizon, num_envs, n_act=8, seed=0):
    return np.random.default_rng(seed).integers(0, n_act, size=(horizon, num_envs), dtype=np.int64)


def run_squared(num_envs, seed, horizon, env_kwargs=None):
    vec = pufferlib.vector.make(ocean.env_creator('squared'), env_kwargs=env_kwargs or {},
                                num_envs=num_envs, backend=pufferlib.vector.Serial)
    tape = action_tape(horizon, num_envs)
    obs, rew, term, trunc, mask = [], [], [], [], []
    info_rows = []   # (recv index, position in infos list, episode_return, episode_length, score)
    vec.async_reset(seed)
    for t in range(horizon + 1):
        o, r, d, tr, infos, env_id, m = vec.recv()
        assert np.array_equal(env_id, np.arange(num_envs))
        obs.append(o.copy()); rew.append(r.copy()); term.append(d.copy()); trunc.append(tr.copy()); mask.append(m.copy())
        for k, i in enumerate(infos):
            info_rows.append((t, k, i['episode_return'], i['episode_length'], i['score']))
        if t < horizon:
            vec.send(tape[t])
    obs = np.stack(obs)
    assert np.array_equal(obs, obs.astype(np.int8).astype(np.float32))
    vec.close()
    return dict(
        num_envs=num_envs, seed=seed, horizon=horizon, actions=tape,
        obs_i8=obs.astype(np.int8), obs_dtype=str(obs.dtype), rewards=np.stack(rew), terminals=np.stack(term),
        truncations=np.stack(trunc), masks=np.stack(mask),
        infos=np.asarray(info_rows, dtype=np.float64).reshape(-1, 5),
        distance_to_target=(env_kwargs or {}).get('distance_to_target', 3),
    )


def gen_squared():
    cases = {
        'squared_c1': dict(num_envs=64, seed=1, horizon=128),          # BASELINE config C1
        'squared_n5_seed42': dict(num_envs=5, seed=42, horizon=41),
        'squared_n1_seed7': dict(num_envs=1, seed=7, horizon=17),
        'squared_d2_n33': dict(num_envs=33, seed=123456789, horizon=30, env_kwargs={'distance_to_target': 2}),
        'squared_d5_n8': dict(num_envs=8, seed=2**31 + 5, horizon=36, env_kwargs={'distance_to_target': 5}),
    }
    for name, kw in cases.items():
        out = run_squared(**kw)
        np.savez_compressed(os.path.join(HERE, name + '.npz'), **out)
        print(name, out['obs_i8'].shape, 'infos', out['infos'].shape)


def gae_inputs(n, seed, p_done=0.01):
    rng = np.random.default_rng(seed)
    rewards = rng.standard_normal(n).astype(np.float32)
    values = rng.standard_normal(n).astype(np.float32)
    dones = (rng.random(n) < p_done).astype(np.float32)
    return dones, values, rewards


def load_c_gae():
    import pyximport
    pyximport.install(setup_args={'include_dirs': np.get_include()})
    from c_gae import compute_gae
    return compute_gae


def gen_gae():
    compute_gae = load_c_gae()
    out = {}
    cases = [(1, 0, 0.01, 0.99, 0.95), (2, 1, 0.5, 0.99, 0.95), (7, 2, 0.3, 0.9, 0.8), (129, 3, 0.05, 0.99, 0.95),
             (8192, 0, 0.01, 0.99, 0.95), (8192, 4, 0.0, 1.0, 1.0), (4096, 5, 1.0, 0.99, 0.95),
             (65536, 6, 0.01, 0.99, 0.95)]
    for k, (n, seed, p, gamma, lam) in enumerate(cases):
        d, v, r = gae_inputs(n, seed, p)
        adv = compute_gae(d, v, r, gamma, lam)
        out[f'case{k}_meta'] = np.asarray([n, seed, p, gamma, lam], dtype=np.float64)
        out[f'case{k}_adv'] = adv
    out['num_cases'] = np.asarray(len(cases))
    np.savez_compressed(os.path.join(HERE, 'gae.npz'), **out)
    print('gae cases', len(cases))
    return compute_gae


# (n, p_done, gamma, lambda) of tests/test_oracle_golden.py::test_gae_oracle_vs_reference_compiled_c_gae
C_GAE_CPU_CASES = [(2, 0.0, 0.99, 0.95), (1000, 0.02, 0.99, 0.95), (50000, 0.1, 0.9, 0.5), (4096, 1.0, 0.99, 0.95),
                   (4096, 0.0, 1.0, 1.0)]
# (h, n, p_done, gamma, lambda) of tests/test_gpu_gae.py::test_gae_vs_reference_compiled_c_gae
C_GAE_GPU_CASES = [(128, 64, 0.02, 0.99, 0.95), (256, 1024, 0.01, 0.99, 0.95), (4096, 1, 0.05, 0.9, 0.8),
                   (16, 333, 0.2, 1.0, 1.0), (128, 16384, 0.01, 0.99, 0.95)]
C_GAE_SAMPLE = 16384


def gen_c_gae_cases(compute_gae):
    """c_gae.compute_gae on the inputs of the two reference-comparison tests above.  The CPU cases are stored whole (the
    test is bit-exact); a GPU case longer than C_GAE_SAMPLE keeps a fixed, seeded sample of positions (gpu_*_idx)."""
    out = {}
    for n, p, gamma, lam in C_GAE_CPU_CASES:
        d, v, r = gae_inputs(n, seed=n, p_done=p)
        out[f'cpu_{n}_{p}_{gamma}_{lam}'] = np.asarray(compute_gae(d, v, r, gamma, lam))
    for h, n, p, gamma, lam in C_GAE_GPU_CASES:
        rng = np.random.default_rng(7 * h + n)                      # make_inputs of tests/test_gpu_gae.py
        r = rng.standard_normal((h, n)).astype(np.float32)
        v = rng.standard_normal((h, n)).astype(np.float32)
        d = (rng.random((h, n)) < p).astype(np.float32)
        r, v, d = (np.ascontiguousarray(x.T).reshape(-1) for x in (r, v, d))   # arrival [H, N] -> sorted e*H + t
        adv = np.asarray(compute_gae(d, v, r, gamma, lam))
        idx = np.arange(adv.size)
        if adv.size > C_GAE_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(adv.size, C_GAE_SAMPLE, replace=False))
        out[f'gpu_{h}x{n}_idx'] = idx.astype(np.int32)
        out[f'gpu_{h}x{n}_adv'] = adv[idx]
    np.savez_compressed(os.path.join(HERE, 'c_gae_cases.npz'), **out)
    print('c_gae_cases', len(C_GAE_CPU_CASES), 'cpu +', len(C_GAE_GPU_CASES), 'gpu')


def gen_experience(compute_gae):
    import clean_pufferl
    cases = {
        # C1: squared N=64 H=128, batch 8192, minibatch 2048, bptt 16
        'experience_c1': dict(num_envs=64, horizon=128, minibatch_size=2048, bptt=16, seed=1),
        'experience_small': dict(num_envs=6, horizon=8, minibatch_size=12, bptt=4, seed=3),
        'experience_one_mb': dict(num_envs=4, horizon=16, minibatch_size=64, bptt=8, seed=5),
    }
    for name, c in cases.items():
        n, h = c['num_envs'], c['horizon']
        batch = n * h
        vec = pufferlib.vector.make(ocean.env_creator('squared'), num_envs=n, backend=pufferlib.vector.Serial)
        exp = clean_pufferl.Experience(batch, c['bptt'], c['minibatch_size'], vec.single_observation_space.shape,
                                       vec.single_observation_space.dtype, vec.single_action_space.shape,
                                       cpu_offload=False, device='cpu')
        tape = action_tape(h, n)
        rng = np.random.default_rng(100 + c['seed'])
        values = rng.standard_normal((h, n)).astype(np.float32)
        logprobs = -rng.random((h, n)).astype(np.float32)
        vec.async_reset(c['seed'])
        t = 0
        while not exp.full:
            o, r, d, tr, infos, env_id, mask = vec.recv()
            exp.store(torch.as_tensor(o), torch.as_tensor(values[t]), tape[t], torch.as_tensor(logprobs[t]),
                      torch.as_tensor(r), torch.as_tensor(d), env_id.tolist(), torch.as_tensor(mask))
            vec.send(tape[t])
            t += 1
        assert t == h
        stored = dict(obs_i8=exp.obs.numpy().astype(np.int8), actions=exp.actions_np.copy(),
                      logprobs=exp.logprobs_np.copy(), rewards=exp.rewards_np.copy(), dones=exp.dones_np.copy(),
                      values=exp.values_np.copy())
        idxs = exp.sort_training_data()
        gamma, lam = 0.99, 0.95
        adv = compute_gae(exp.dones_np[idxs], exp.values_np[idxs], exp.rewards_np[idxs], gamma, lam)
        exp.flatten_batch(adv)
        norm = torch.stack([(a - a.mean()) / (a.std() + 1e-8) for a in exp.b_advantages])
        np.savez_compressed(
            os.path.join(HERE, name + '.npz'),
            num_envs=n, horizon=h, minibatch_size=c['minibatch_size'], bptt=c['bptt'], seed=c['seed'],
            gamma=gamma, gae_lambda=lam, tape=tape, values_in=values, logprobs_in=logprobs,
            idxs=idxs, advantages=adv, returns_np=exp.returns_np,
            b_idxs_obs=exp.b_idxs_obs.numpy(), b_obs_i8=exp.b_obs.numpy().astype(np.int8),
            b_actions=exp.b_actions.numpy(), b_logprobs=exp.b_logprobs.numpy(), b_dones=exp.b_dones.numpy(),
            b_values=exp.b_values.numpy(), b_advantages=exp.b_advantages.numpy(), b_returns=exp.b_returns.numpy(),
            b_advantages_normalized=norm.numpy(),
            **{'stored_' + k: v for k, v in stored.items()})
        vec.close()
        print(name, 'B', batch, 'b_obs', tuple(exp.b_obs.shape))




def run_squared_multiprocessing(num_envs, num_workers, seed, horizon):
    """The reference's Multiprocessing backend in its synchronous mode (batch_size == num_envs: every recv() returns
    all workers' rows in worker order, vector.py:360-369), so the golden is deterministic.  Each worker process runs a
    Serial over its envs with its OWN process-global `random` stream (vector.py:168-190): the outputs differ from the
    Serial golden of the same seed from the first auto-reset on."""
    vec = pufferlib.vector.make(ocean.env_creator('squared'), num_envs=num_envs, num_workers=num_workers,
                                batch_size=num_envs, backend=pufferlib.vector.Multiprocessing)
    tape = action_tape(horizon, num_envs)
    obs, rew, term, info_rows = [], [], [], []
    vec.async_reset(seed)
    for t in range(horizon + 1):
        o, r, d, tr, infos, env_id, m = vec.recv()
        assert np.array_equal(env_id, np.arange(num_envs)) and m.all() and not tr.any()
        obs.append(o.copy()); rew.append(r.copy()); term.append(d.copy())
        for k, i in enumerate(infos):
            info_rows.append((t, k, i['episode_return'], i['episode_length'], i['score']))
        if t < horizon:
            vec.send(tape[t])
    vec.close()
    obs = np.stack(obs)
    return dict(num_envs=num_envs, num_workers=num_workers, seed=seed, horizon=horizon, actions=tape,
                obs_i8=obs.astype(np.int8), rewards=np.stack(rew), terminals=np.stack(term),
                infos=np.asarray(info_rows, dtype=np.float64).reshape(-1, 5))


def gen_squared_multiprocessing():
    for name, kw in {'squared_mp_n8_w2': dict(num_envs=8, num_workers=2, seed=11, horizon=40),
                     'squared_mp_n12_w4': dict(num_envs=12, num_workers=4, seed=5, horizon=33)}.items():
        out = run_squared_multiprocessing(**kw)
        serial = run_squared(kw['num_envs'], kw['seed'], kw['horizon'])
        out['differs_from_serial'] = np.asarray(not np.array_equal(serial['obs_i8'], out['obs_i8']))
        np.savez_compressed(os.path.join(HERE, name + '.npz'), **out)
        print(name, out['obs_i8'].shape, 'differs from Serial:', bool(out['differs_from_serial']))


def gen_lstm():
    """The reference's recurrent path end to end on CPU: create -> evaluate (lstm_h[:, env_id] state carry,
    clean_pufferl.py:100-105) -> train (bptt segments [rows, bptt, *obs], state carried ACROSS minibatches inside an
    epoch and reset per epoch, :176-191) with models.LSTMWrapper (models.py:64-111) around models.Default."""
    import clean_pufferl
    import pufferlib.models
    import pufferlib.frameworks.cleanrl
    n, h, bptt, mbs, hid = 8, 16, 4, 64, 32
    vec = pufferlib.vector.make(ocean.env_creator('squared'), num_envs=n, backend=pufferlib.vector.Serial)
    torch.manual_seed(3)
    base = pufferlib.models.Default(vec.driver_env, hidden_size=hid)
    wrapper = pufferlib.models.LSTMWrapper(vec.driver_env, base, input_size=hid, hidden_size=hid)
    policy = pufferlib.frameworks.cleanrl.RecurrentPolicy(wrapper)
    init = {k: v.detach().clone().numpy() for k, v in policy.state_dict().items()}
    cfg = dict(seed=1, torch_deterministic=True, env='squared', batch_size=n * h, bptt_horizon=bptt, minibatch_size=mbs,
               cpu_offload=False, device='cpu', compile=False, compile_mode='default', learning_rate=2.5e-3, gamma=0.99,
               gae_lambda=0.95, update_epochs=2, norm_adv=True, clip_coef=0.1, clip_vloss=True, vf_clip_coef=0.1,
               vf_coef=0.5, ent_coef=0.01, max_grad_norm=0.5, target_kl=None, anneal_lr=False,
               total_timesteps=10 ** 9, checkpoint_interval=10 ** 9, data_dir='/tmp/golden_lstm', exp_id='lstm')
    data = clean_pufferl.create(pufferlib.namespace(**cfg), vec, policy)
    clean_pufferl.evaluate(data)
    exp = data.experience
    out = dict(num_envs=n, horizon=h, bptt=bptt, minibatch_size=mbs, hidden=hid, seed=1,
               learning_rate=cfg['learning_rate'], update_epochs=cfg['update_epochs'],
               obs_i8=exp.obs.numpy().astype(np.int8), actions=exp.actions_np.copy(), logprobs=exp.logprobs_np.copy(),
               values=exp.values_np.copy(), rewards=exp.rewards_np.copy(), dones=exp.dones_np.copy(),
               lstm_h=exp.lstm_h.numpy().copy(), lstm_c=exp.lstm_c.numpy().copy())
    clean_pufferl.train(data)
    for k in ('policy_loss', 'value_loss', 'entropy', 'old_approx_kl', 'approx_kl', 'clipfrac', 'explained_variance'):
        out['loss_' + k] = np.asarray(getattr(data.losses, k), dtype=np.float64)
    out['b_obs_i8'] = exp.b_obs.numpy().astype(np.int8)
    out['advantages'] = exp.b_advantages.numpy().copy()
    for k, v in init.items():
        out['init/' + k] = v
    for k, v in policy.state_dict().items():
        out['after/' + k] = v.detach().numpy().copy()
    data.utilization.stop()
    vec.close()
    np.savez_compressed(os.path.join(HERE, 'lstm_squared.npz'), **out)
    print('lstm_squared', {k: float(out['loss_' + k]) for k in ('policy_loss', 'value_loss', 'entropy')},
          'params', sum(v.size for k, v in out.items() if k.startswith('init/')))


if __name__ == '__main__':
    if sys.argv[1:] == ['c_gae_cases']:       # only c_gae_cases.npz
        gen_c_gae_cases(load_c_gae())
        sys.exit()
    gen_squared()
    gen_squared_multiprocessing()
    cg = gen_gae()
    gen_experience(cg)
    gen_c_gae_cases(cg)
    gen_lstm()
