"""MultiDiscrete on the device: the `spaces` env kernel vs oracle/spaces.py (bit-exact obs, reward bits, terminals,
infos) through every vecenv mode, pb_sample_logits_multi and pb_ppo_loss_multi vs torch, Experience with [B, 2]
actions vs the reference (tests/golden/experience_md.npz), and create / evaluate / train on `spaces`."""
import ctypes as C

import numpy as np
import pytest
import torch

import pufferlib_b200
import pufferlib_b200.vector as pvec
from oracle import gae as ogae
from oracle import spaces as ospaces
from pufferlib_b200 import _native, clean_pufferl, models, spaces
from pufferlib_b200.environments import ocean
from pufferlib_b200.frameworks import cleanrl

pytestmark = pytest.mark.gpu


def cpu(x):
    return x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


def check_row(t, got, want, infos=None, want_infos=None):
    o, r, term, trunc, mask = got
    oo, orr, ot = want
    assert np.array_equal(cpu(o), oo), f'obs differ at step {t}'
    assert np.array_equal(cpu(r).view(np.uint32), orr.view(np.uint32)), f'reward bits differ at step {t}'
    assert np.array_equal(cpu(term), ot), f'terminals differ at step {t}'
    assert not cpu(trunc).any() and cpu(mask).all()
    if want_infos is not None:
        assert infos == want_infos, f'infos differ at step {t}'


def tape(h, n, seed=0):
    return np.random.default_rng(seed).integers(0, 2, size=(h, n, 2), dtype=np.int64)


# -- the env ------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize('n', [1, 37, 4096])
@pytest.mark.parametrize('mode', ['own', 'offset', 'host'])
def test_spaces_env_matches_oracle(n, mode):
    offset = 1000003 if mode == 'offset' else 0
    vec = pvec.make(ocean.env_creator('spaces'), num_envs=n,
                    backend=pvec.B200.options(exact_infos=True, env_index_offset=offset, host_buffers=mode == 'host'))
    assert vec.single_action_space == spaces.MultiDiscrete([2, 2])
    assert vec.single_observation_space.shape == (108,) and vec.single_observation_space.dtype == np.uint8
    assert vec.action_space.shape == (n, 2)
    ora = ospaces.SpacesSerial(n, env_index_offset=offset)
    seed, h = 7, 9
    acts = tape(h, n, seed)
    vec.async_reset(seed)
    ora.async_reset(seed)
    ret_sum, episodes = 0.0, 0
    for t in range(h + 1):
        o, r, term, trunc, infos, _, mask = vec.recv()
        oo, orr, ot, _, oinf, _, _ = ora.recv()
        check_row(t, (o, r, term, trunc, mask), (oo, orr, ot), infos, oinf)
        ret_sum, episodes = ret_sum + float(orr[ot].sum()), episodes + int(ot.sum())
        if t < h:
            vec.send(acts[t] if mode == 'host' else torch.as_tensor(acts[t], device='cuda'))
            ora.send(acts[t])
    means, cnt = vec.episode_stats()           # the device-side EpisodeStats reduction
    assert cnt == episodes == n * ((h + 1) // 2)
    assert np.isclose(means['episode_return'], ret_sum / episodes) and means['episode_length'] == 1.0
    assert np.isclose(means['score'], ret_sum / episodes)
    vec.close()


def test_spaces_env_shards_by_global_index():
    """Two handles with env_index_offset = 0 and n/2 produce the rows of one n-env handle."""
    n, h, seed = 64, 5, 3
    whole = ospaces.SpacesSerial(n)
    halves = [pvec.make(ocean.env_creator('spaces'), num_envs=n // 2,
                        backend=pvec.B200.options(env_index_offset=k * n // 2)) for k in range(2)]
    whole.async_reset(seed)
    for v in halves:
        v.async_reset(seed)
    acts = tape(h, n, 1)
    for t in range(h + 1):
        rows = [v.recv() for v in halves]
        oo, orr, ot = whole.recv()[:3]
        check_row(t, tuple(torch.cat([cpu_t[i] for cpu_t in rows]) for i in (0, 1, 2, 3, 6)), (oo, orr, ot))
        if t < h:
            for k, v in enumerate(halves):
                v.send(torch.as_tensor(acts[t, k * n // 2:(k + 1) * n // 2], device='cuda'))
            whole.send(acts[t])


@pytest.mark.parametrize('n,batch', [(2, 1), (74, 37), (4096, 1024)])
def test_spaces_pool_mode_matches_oracle(n, batch):
    vec = pvec.make(ocean.env_creator('spaces'), num_envs=n, batch_size=batch, backend=pvec.B200)
    ora = ospaces.SpacesSerial(n)
    seed, h = 5, 6
    acts = tape(h, n, 2)
    vec.async_reset(seed)
    ora.async_reset(seed)
    for t in range(h):
        oo, orr, ot = (x.copy() for x in ora.recv()[:3])
        for g in range(n // batch):                  # groups come round-robin, each stepped on its own stream
            o, r, term, trunc, _, ids, mask = vec.recv()
            lo = int(ids[0])
            assert lo == g * batch
            check_row(t, (o, r, term, trunc, mask), (oo[lo:lo + batch], orr[lo:lo + batch], ot[lo:lo + batch]))
            vec.send(torch.as_tensor(acts[t, lo:lo + batch], device='cuda'))
        ora.send(acts[t])
    vec.close()


@pytest.mark.parametrize('n', [1, 37, 4096])
def test_spaces_bound_rollout_rows_match_oracle(n):
    """Step outputs written straight into Experience rows (bind_rollout) with [B, 2] actions."""
    vec = pvec.make(ocean.env_creator('spaces'), num_envs=n, backend=pvec.B200)
    h = 8
    exp = clean_pufferl.Experience(n * h, 4, n * h, (108,), np.uint8, (2,))
    vec.bind_rollout(exp)
    ora = ospaces.SpacesSerial(n)
    acts = tape(2 * h, n, 9)
    vec.async_reset(11)
    ora.async_reset(11)
    want = []
    for t in range(2 * h):
        o, r, term, trunc, _, ids, mask = vec.recv()
        oo, orr, ot = (x.copy() for x in ora.recv()[:3])
        check_row(t, (o, r, term, trunc, mask), (oo, orr, ot))
        want.append((oo, orr, ot))
        a = torch.as_tensor(acts[t], device='cuda')
        z = torch.zeros(n, device='cuda')
        exp.store(o, z, a, z, r, term, ids, mask)
        if exp.full:
            rows = [(cpu(exp.obs).reshape(h, n, 108), cpu(exp.rewards).reshape(h, n), cpu(exp.dones).reshape(h, n),
                     cpu(exp.actions).reshape(h, n, 2))]
            for k in range(h):
                oo, orr, ot = want[t - h + 1 + k]
                assert np.array_equal(rows[0][0][k], oo) and np.array_equal(rows[0][1][k], orr)
                assert np.array_equal(rows[0][2][k], ot.astype(np.float32))
                assert np.array_equal(rows[0][3][k], acts[t - h + 1 + k])
            exp.sort_training_data()
        vec.send(a)
        ora.send(acts[t])


def test_spaces_env_full_size():
    n, h, seed = 65536, 4, 123
    vec = pvec.make(ocean.env_creator('spaces'), num_envs=n, backend=pvec.B200.options(exact_infos=True))
    ora = ospaces.SpacesSerial(n)
    acts = tape(h, n, 4)
    vec.async_reset(seed)
    ora.async_reset(seed)
    for t in range(h + 1):
        o, r, term, trunc, infos, _, mask = vec.recv()
        oo, orr, ot, _, oinf, _, _ = ora.recv()
        check_row(t, (o, r, term, trunc, mask), (oo, orr, ot), infos, oinf)
        if t < h:
            vec.send(torch.as_tensor(acts[t], device='cuda'))
            ora.send(acts[t])


def test_spaces_actions_are_checked_and_clamped():
    vec = pvec.make(ocean.env_creator('spaces'), num_envs=4, backend=pvec.B200)
    vec.async_reset(1)
    vec.recv()
    with pytest.raises(pufferlib_b200.exceptions.APIUsageError):
        vec.send(torch.full((4, 2), 2, dtype=torch.int64, device='cuda'))       # first send: action_space check
    vec = pvec.make(ocean.env_creator('spaces'), num_envs=4, backend=pvec.B200)
    ora = ospaces.SpacesSerial(4)
    vec.async_reset(1)
    ora.async_reset(1)
    vec.recv()
    vec.send(torch.zeros(4, 2, dtype=torch.int64, device='cuda'))
    ora.send(np.zeros((4, 2), dtype=np.int64))
    vec.recv()
    vec.send(torch.zeros(4, 2, dtype=torch.int64, device='cuda'))            # reset step
    ora.send(np.zeros((4, 2), dtype=np.int64))
    vec.recv()
    bad = np.array([[5, -3], [1, 7], [-1, 0], [0, 1]], dtype=np.int64)          # device clamps each column
    vec.send(torch.as_tensor(bad, device='cuda'))
    ora.send(bad)
    o, r, term = vec.recv()[:3]
    assert np.array_equal(cpu(r), ora.recv()[1])
    nvec, heads = (C.c_int32 * 8)(), C.c_int32()
    _native.check(_native.lib().pb_env_action_nvec(vec._handle, nvec, C.byref(heads)))
    assert heads.value == 2 and list(nvec) == [2, 2, 0, 0, 0, 0, 0, 0]
    sq = pvec.make(ocean.env_creator('squared'), num_envs=2, backend=pvec.B200)
    _native.check(_native.lib().pb_env_action_nvec(sq._handle, nvec, C.byref(heads)))
    assert heads.value == 0 and isinstance(sq.single_action_space, spaces.Discrete)


# -- pb_sample_logits_multi -------------------------------------------------------------------------------------------

def sample_multi(logits, nvec, seed=3, offset=0, value=None, rows=None):
    n = logits.shape[0]
    dev = logits.device
    a = torch.empty(n, len(nvec), dtype=torch.int64, device=dev)
    lp = torch.empty(n, device=dev)
    ent = torch.empty(n, device=dev)
    nv = (C.c_int32 * len(nvec))(*nvec)
    vr, lr, ar = rows if rows is not None else (None, None, None)
    _native.check(_native.lib().pb_sample_logits_multi(
        _native.ptr(logits), logits.stride(0), n, nv, len(nvec), C.c_uint64(seed), C.c_uint64(offset), None,
        _native.ptr(a), _native.ptr(lp), _native.ptr(ent), _native.ptr(value), 0 if value is None else value.stride(0),
        _native.ptr(vr), _native.ptr(lr), _native.ptr(ar), _native.stream_ptr()))
    return a, lp, ent


@pytest.mark.parametrize('nvec', [[2, 2], [3, 7, 4], [1, 5], [7]])
def test_sample_multi_logprob_entropy_match_fp64(nvec):
    torch.manual_seed(len(nvec) * 10 + sum(nvec))
    n, total = 70001, sum(nvec)
    base = torch.randn(n, total + 3, device='cuda') * 3           # strided rows, like a packed head output
    logits = base[:, :total]
    a, lp, ent = sample_multi(logits, nvec)
    assert a.shape == (n, len(nvec))
    heads = list(logits.double().split(nvec, dim=1))
    for h, k in enumerate(nvec):
        assert int(a[:, h].min()) >= 0 and int(a[:, h].max()) < k
    _, ref_lp, ref_ent = cleanrl.sample_logits(heads, a)
    assert float((lp.double() - ref_lp).abs().max()) <= 1e-5 * max(1.0, float(ref_lp.abs().max()))
    assert float((ent.double() - ref_ent).abs().max()) <= 1e-5 * max(1.0, float(ref_ent.abs().max()))


@pytest.mark.parametrize('n_act', [2, 4, 7, 18])
def test_sample_multi_single_head_is_pb_sample_logits(n_act):
    torch.manual_seed(n_act)
    n = 50000
    logits = torch.randn(n, n_act + 1, device='cuda')[:, :n_act]
    value = torch.randn(n, 1, device='cuda')
    counter = torch.tensor([5], dtype=torch.int64, device='cuda')
    outs = []
    for multi in (False, True):
        a = torch.empty((n, 1) if multi else (n,), dtype=torch.int64, device='cuda')
        lp, ent = torch.empty(n, device='cuda'), torch.empty(n, device='cuda')
        args = (C.c_uint64(9), C.c_uint64(2), _native.ptr(counter), _native.ptr(a), _native.ptr(lp), _native.ptr(ent),
                _native.ptr(value), 1, None, None, None, _native.stream_ptr())
        if multi:
            _native.check(_native.lib().pb_sample_logits_multi(_native.ptr(logits), logits.stride(0), n,
                                                               (C.c_int32 * 1)(n_act), 1, *args))
        else:
            _native.check(_native.lib().pb_sample_logits(_native.ptr(logits), logits.stride(0), n, n_act, *args))
        outs.append((a.reshape(-1), lp, ent))
    for x, y in zip(*outs):
        assert torch.equal(x, y)


def test_sample_multi_chi_square_per_head():
    from scipy.stats import chisquare
    nvec = [3, 7, 4]
    n = 1_000_000
    torch.manual_seed(1)
    row = torch.randn(1, sum(nvec), device='cuda')
    logits = row.expand(n, -1).contiguous()
    a, _, _ = sample_multi(logits, nvec, seed=12345, offset=7)
    for h, lg in enumerate(row.double()[0].split(nvec)):
        p = torch.softmax(lg, 0).cpu().numpy()
        counts = torch.bincount(a[:, h], minlength=nvec[h]).cpu().numpy()
        stat, pval = chisquare(counts, p * n)
        assert pval > 1e-4, (h, counts, pval)
    # heads draw independent uniforms: the joint of heads 0 and 2 factorises (independence test, (3-1)(4-1) dof)
    joint = torch.bincount(a[:, 0] * 4 + a[:, 2], minlength=12).cpu().numpy().reshape(3, 4)
    expect = np.outer(joint.sum(1), joint.sum(0)) / n
    stat, pval = chisquare(joint.ravel(), expect.ravel(), ddof=12 - 1 - (3 - 1) * (4 - 1))
    assert pval > 1e-4


def test_sample_multi_row_stores():
    nvec = [2, 2]
    n = 4099
    torch.manual_seed(2)
    out = torch.randn(n, 8, device='cuda')
    values, logprobs = torch.full((n,), float('nan'), device='cuda'), torch.full((n,), float('nan'), device='cuda')
    actions = torch.full((n, 2), -1, dtype=torch.int64, device='cuda')
    a, lp, ent = sample_multi(out, nvec, value=out[:, 4:5], rows=(values, logprobs, actions))
    assert torch.equal(values, out[:, 4]) and torch.equal(logprobs, lp) and torch.equal(actions, a)


# -- pb_ppo_loss_multi ------------------------------------------------------------------------------------------------

def reference_loss(logits, value, actions, old_lp, adv, ret, old_v, cfg):
    _, newlogprob, entropy = cleanrl.sample_logits(logits, actions)
    logratio = newlogprob - old_lp
    ratio = logratio.exp()
    old_kl = (-logratio).mean()
    kl = ((ratio - 1) - logratio).mean()
    clipfrac = ((ratio - 1.0).abs() > cfg.clip_coef).to(ratio.dtype).mean()
    pg = torch.max(-adv * ratio, -adv * torch.clamp(ratio, 1 - cfg.clip_coef, 1 + cfg.clip_coef)).mean()
    nv = value.view(-1)
    if cfg.clip_vloss:
        vc = old_v + torch.clamp(nv - old_v, -cfg.vf_clip_coef, cfg.vf_clip_coef)
        vl = 0.5 * torch.max((nv - ret) ** 2, (vc - ret) ** 2).mean()
    else:
        vl = 0.5 * ((nv - ret) ** 2).mean()
    ent = entropy.mean()
    loss = pg - cfg.ent_coef * ent + vl * cfg.vf_coef
    return loss, torch.stack([pg, vl, ent, old_kl, kl, clipfrac]).detach()


def loss_inputs(m, nvec, seed):
    dev = torch.device('cuda')
    torch.manual_seed(seed)
    total = sum(nvec)
    out = torch.randn(m, 8 if total < 8 else total + 3, device=dev)
    actions = torch.stack([torch.randint(0, k, (m,), device=dev) for k in nvec], 1)
    with torch.no_grad():
        _, nlp, _ = cleanrl.sample_logits(list(out[:, :total].split(nvec, 1)), actions)
    old_lp = nlp + 0.2 * torch.randn(m, device=dev)
    old_lp[::3] = nlp[::3]                       # exact ties: ratio == 1
    adv, ret = torch.randn(m, device=dev), torch.randn(m, device=dev)
    old_v = out[:, total] + 0.15 * torch.randn(m, device=dev)
    return out, actions, old_lp, adv, ret, old_v


@pytest.mark.parametrize('m,nvec', [(1, [2, 2]), (1000, [3, 7, 4]), (4097, [1, 5]), (524288, [2, 2]), (333, [9, 11, 2])])
@pytest.mark.parametrize('clip_vloss', [True, False])
def test_ppo_loss_multi_matches_fp64_autograd(m, nvec, clip_vloss):
    cfg = pufferlib_b200.namespace(clip_coef=0.1, clip_vloss=clip_vloss, vf_clip_coef=0.1, vf_coef=0.5, ent_coef=0.01)
    out, actions, old_lp, adv, ret, old_v = loss_inputs(m, nvec, m + sum(nvec))
    total = sum(nvec)
    ref_in = out.detach().double().requires_grad_(True)
    loss_ref, st_ref = reference_loss(list(ref_in[:, :total].split(nvec, 1)), ref_in[:, total:total + 1], actions,
                                      old_lp.double(), adv.double(), ret.double(), old_v.double(), cfg)
    loss_ref.backward()
    got_in = out.detach().clone().requires_grad_(True)
    packed = total + 1 <= 8
    if packed:
        loss, st = clean_pufferl.fused_ppo_loss_packed_multi(got_in, nvec, actions, old_lp, adv, ret, old_v, cfg)
    else:
        loss, st = clean_pufferl.fused_ppo_loss_multi(list(got_in[:, :total].split(nvec, 1)),
                                                      got_in[:, total:total + 1], actions, old_lp, adv, ret, old_v, cfg)
    loss.backward()
    assert abs(float(loss) - float(loss_ref)) <= 1e-5 * abs(float(loss_ref)) + 1e-6
    assert torch.allclose(st.double(), st_ref, rtol=1e-5, atol=1e-6)
    g, gr = got_in.grad[:, :total + 1].double(), ref_in.grad[:, :total + 1]
    assert float((g - gr).abs().max()) <= 1e-5 * float(gr.abs().max()) + 1e-10
    if packed:
        assert float(got_in.grad[:, total + 1:].abs().sum()) == 0.0


@pytest.mark.parametrize('n_act', [2, 4, 7])
def test_ppo_loss_multi_single_head_matches_pb_ppo_loss(n_act):
    cfg = pufferlib_b200.namespace(clip_coef=0.2, clip_vloss=True, vf_clip_coef=0.2, vf_coef=0.5, ent_coef=0.01)
    out, actions, old_lp, adv, ret, old_v = loss_inputs(20000, [n_act], n_act)
    a = out.detach().clone().requires_grad_(True)
    b = out.detach().clone().requires_grad_(True)
    la, sa = clean_pufferl.fused_ppo_loss_packed(a, n_act, actions.view(-1), old_lp, adv, ret, old_v, cfg)
    lb, sb = clean_pufferl.fused_ppo_loss_packed_multi(b, [n_act], actions, old_lp, adv, ret, old_v, cfg)
    la.backward()
    lb.backward()
    assert torch.allclose(la, lb, rtol=1e-6, atol=0) and torch.allclose(sa, sb, rtol=1e-6, atol=1e-9)
    assert float((a.grad - b.grad).abs().max()) <= 1e-6 * float(a.grad.abs().max())


# -- Experience with [B, 2] actions ----------------------------------------------------------------------------------

def test_experience_md_matches_reference(golden):
    g = golden('experience_md')
    n, h, mbs, bptt = int(g['num_envs']), int(g['horizon']), int(g['minibatch_size']), int(g['bptt'])
    exp = clean_pufferl.Experience(n * h, bptt, mbs, (108,), np.uint8, (2,))
    dev = 'cuda'
    obs = g['stored_obs'].reshape(h, n, 108)
    for t in range(h):
        exp.store(torch.as_tensor(obs[t], device=dev), torch.as_tensor(g['values_in'][t], device=dev),
                  torch.as_tensor(g['tape'][t], device=dev), torch.as_tensor(g['logprobs_in'][t], device=dev),
                  torch.as_tensor(g['stored_rewards'][t * n:(t + 1) * n], device=dev),
                  torch.as_tensor(g['stored_dones'][t * n:(t + 1) * n], device=dev), np.arange(n), np.ones(n, bool))
    assert np.array_equal(cpu(exp.actions), g['stored_actions']) and exp.actions.shape == (n * h, 2)
    assert np.array_equal(np.asarray(exp.sort_training_data()), g['idxs'])
    exp.compute_gae(float(g['gamma']), float(g['gae_lambda']))
    adv = cpu(exp.advantages)
    assert np.max(np.abs(adv - g['advantages']) / np.maximum(1, np.abs(g['advantages']))) <= 1e-5
    exp.flatten_batch(torch.as_tensor(g['advantages'], device=dev))
    assert exp.b_actions.shape == g['b_actions'].shape
    assert np.array_equal(cpu(exp.b_actions), g['b_actions'])
    assert np.array_equal(cpu(exp.b_obs), g['b_obs'])
    for k in ('b_logprobs', 'b_dones', 'b_values', 'b_advantages', 'b_returns'):
        assert np.array_equal(cpu(getattr(exp, k)), g[k]), k


def test_experience_md_slab_and_gathered_minibatches_agree():
    n, h, bptt, nm = 16, 16, 4, 2
    exp = clean_pufferl.Experience(n * h, bptt, n * h // nm, (108,), np.uint8, (2,))
    torch.manual_seed(0)
    for t in range(h):
        exp.store(torch.randint(0, 255, (n, 108), dtype=torch.uint8, device='cuda'), torch.randn(n, device='cuda'),
                  torch.randint(0, 2, (n, 2), device='cuda'), torch.rand(n, device='cuda'),
                  torch.randn(n, device='cuda'), (torch.rand(n, device='cuda') < 0.1).float(), np.arange(n),
                  np.ones(n, bool))
    exp.sort_training_data()
    exp.compute_gae(0.99, 0.95)
    exp.flatten_batch()
    assert exp.flatten_batch_slabs()
    sl = exp._slabs
    idx = clean_pufferl.slab_row_index(n, h, nm, bptt)
    acts, lps = cpu(exp.actions), cpu(exp.logprobs)
    for mb in range(nm):
        assert np.array_equal(cpu(sl.actions[mb]), acts[idx[mb]])
        gathered = sorted(zip(cpu(exp.b_logprobs[mb]).ravel(), map(tuple, cpu(exp.b_actions[mb]).reshape(-1, 2))))
        slab = sorted(zip(lps[idx[mb]], map(tuple, cpu(sl.actions[mb]))))
        assert gathered == slab


# -- create / evaluate / train on `spaces` --------------------------------------------------------------------------------

def ppo_config(n, h, **kw):
    cfg = dict(seed=1, torch_deterministic=True, env='spaces', batch_size=n * h, bptt_horizon=8, minibatch_size=n * h // 2,
               cpu_offload=False, device='cuda', compile=False, learning_rate=2.5e-3, gamma=0.99, gae_lambda=0.95,
               update_epochs=1, norm_adv=True, clip_coef=0.1, clip_vloss=True, vf_clip_coef=0.1, vf_coef=0.5,
               ent_coef=0.01, max_grad_norm=0.5, target_kl=None, anneal_lr=False, total_timesteps=10 ** 9)
    cfg.update(kw)
    return pufferlib_b200.namespace(**cfg)


def make_run(n, h, mode='eager', fused_sample=True, seed=0, **cfg_kw):
    opts = {}
    if mode == 'host':
        opts['host_buffers'] = True
    kw = dict(batch_size=n // 4) if mode == 'pool' else {}
    vec = pvec.make(ocean.env_creator('spaces'), num_envs=n, backend=pvec.B200.options(**opts) if opts else pvec.B200, **kw)
    torch.manual_seed(seed)
    base = models.Default(vec.driver_env)
    if mode == 'lstm':
        policy = cleanrl.RecurrentPolicy(models.LSTMWrapper(vec.driver_env, base)).cuda()
    else:
        policy = cleanrl.Policy(base, fused_sample=fused_sample, seed=seed + 1).cuda()
    cfg = ppo_config(n, h, cuda_graph=mode == 'graph', **cfg_kw)
    return clean_pufferl.create(cfg, vec, policy), cfg


def replay_rollout(exp, n, h, ora):
    obs, rew = cpu(exp.obs).reshape(h, n, 108), cpu(exp.rewards).reshape(h, n)
    done, acts = cpu(exp.dones).reshape(h, n), cpu(exp.actions).reshape(h, n, 2)
    for t in range(h):
        o, r, d = ora.recv()[:3]
        assert np.array_equal(o, obs[t]) and np.array_equal(r.view(np.uint32), rew[t].view(np.uint32)), t
        assert np.array_equal(d.astype(np.float32), done[t]), t
        ora.send(acts[t])


@pytest.mark.parametrize('mode', ['eager', 'graph', 'host', 'pool', 'lstm'])
def test_spaces_create_evaluate_train(mode):
    n, h = 256, 16
    data, cfg = make_run(n, h, mode)
    assert data.fused_loss == (mode != 'lstm') and data.action_nvec == [2, 2]
    assert not clean_pufferl._DefaultMLPUpdate.eligible(data)
    assert not data.vecenv.fused_rollout_ok(data.experience, data.policy) if hasattr(data.vecenv, 'fused_rollout_ok') else True
    if mode != 'lstm':
        x = torch.zeros(4, 108, device='cuda')
        assert data.policy._policy_step_fused(x) is None
    ora = ospaces.SpacesSerial(n)
    ora.async_reset(cfg.seed)
    for it in range(3):
        clean_pufferl.evaluate(data)
        replay_rollout(data.experience, n, h, ora)
        clean_pufferl.train(data)
        assert np.isfinite(data.losses.policy_loss) and np.isfinite(data.losses.value_loss)
        assert data.losses.entropy > 0
    if mode == 'graph':
        assert data.graph_replays >= 1 and data.train_graph_replays >= 1
    clean_pufferl.close(data)


def test_spaces_graphed_training_equals_eager():
    n, h = 512, 16
    params = []
    for mode in ('eager', 'graph'):
        data, _ = make_run(n, h, mode)
        for _ in range(3):
            clean_pufferl.evaluate(data)
            clean_pufferl.train(data)
        params.append([p.detach().clone() for p in data.policy.parameters()])
        clean_pufferl.close(data)
    for a, b in zip(*params):
        assert torch.allclose(a, b, rtol=0, atol=1e-5), float((a - b).abs().max())


def test_spaces_train_matches_pure_torch_restatement():
    """One train() (one minibatch, two epochs) vs the reference's update written in plain torch: GAE, advantage
    normalisation, sample_logits on the list of head logits, the loss of clean_pufferl.py:202-238, clip_grad_norm_ and
    Adam(eps=1e-5)."""
    n, h = 256, 16
    data, cfg = make_run(n, h, 'eager', minibatch_size=n * h, update_epochs=2, learning_rate=2.5e-4)
    clean_pufferl.evaluate(data)
    exp = data.experience
    ref = models.Default(data.vecenv.driver_env).cuda()
    ref.fast_path = False
    ref.load_state_dict(data.policy.policy.state_dict())
    obs, acts = exp.obs.clone(), exp.actions.clone()
    logprobs, values = exp.logprobs.clone(), exp.values.clone()
    rew, done = cpu(exp.rewards), cpu(exp.dones)
    clean_pufferl.train(data)

    idx = np.asarray(clean_pufferl._LazyIdxs(n, h))
    adv = torch.as_tensor(ogae.compute_gae(done[idx], cpu(values)[idx], rew[idx], cfg.gamma, cfg.gae_lambda),
                          device='cuda')
    ii = torch.as_tensor(idx, device='cuda')
    x, a, old_lp, old_v = obs[ii], acts[ii], logprobs[ii], values[ii]
    ret = adv + old_v
    advn = (adv - adv.mean()) / (adv.std() + 1e-8)
    opt = torch.optim.Adam(ref.parameters(), lr=cfg.learning_rate, eps=1e-5)
    for _ in range(cfg.update_epochs):
        logits, v = ref(x)
        loss, _ = reference_loss(logits, v, a, old_lp, advn, ret, old_v, cfg)
        opt.zero_grad()
        loss.backward()
        torch.nn.utils.clip_grad_norm_(ref.parameters(), cfg.max_grad_norm)
        opt.step()
    got = dict(data.policy.policy.named_parameters())
    for name, p in ref.named_parameters():
        err = float((got[name] - p).abs().max())
        assert err <= 2.5e-4, (name, err)
    clean_pufferl.close(data)


# measured on a B200 (1000 W): mean episode return over the last 5 of 150 iterations 0.684, rising from 0.506; the best
# observation-independent policy gets 0.55 (sum(flat) > 0 has probability ~0.4), higher lr plateaus there
LEARN_ITERS = 150
LEARN_THRESHOLD = 0.65


def test_spaces_learns():
    """A short seeded run lifts the mean episode return above the uniform policy's 0.5 and above the 0.55 of always
    answering the more likely sign: the flat head is learnable from the raw observation bytes."""
    n, h = 1024, 16
    data, _ = make_run(n, h, 'eager', learning_rate=3e-4, update_epochs=4)
    returns = []
    for _ in range(LEARN_ITERS):
        stats, _ = clean_pufferl.evaluate(data)
        returns.append(stats.get('episode_return', float('nan')))
        clean_pufferl.train(data)
    print('spaces episode_return every 10 iterations:', np.round(returns[::10], 3).tolist())
    assert abs(returns[0] - 0.5) < 0.05
    assert np.mean(returns[-5:]) >= LEARN_THRESHOLD, returns
    clean_pufferl.close(data)
