#!/usr/bin/env python
"""bench.py -- agent-steps/sec of the env-step + PPO-rollout hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A "step" is one full PPO iteration over one batch: H vectorised env steps with the policy in the loop (obs /
reward / done / value / logprob / action rows written into the device rollout), then GAE, minibatch construction,
advantage normalisation and update_epochs x num_minibatches optimizer steps.  Workload = BASELINE.json configs[1]:
breakout, num_envs=16384 per GPU, horizon=128, MLP policy (hidden 128); multi-GPU = configs[4] (env shards per
rank, one NCCL gradient all-reduce per optimizer step, weak scaling).  PPO hyper-parameters are the reference's
defaults (config.yaml:12-42) with its batch:minibatch ratio of 4.

`value`  : everything device-resident (CUDA-graphed rollout, no per-step host traffic).
`e2e`    : the same step through the public vector/clean_pufferl API with HOST buffers (recv() returns pinned numpy
           arrays, send() takes numpy actions; obs H2D for the policy and action D2H every env step, like the
           reference's evaluate loop).
`--impl reference` / `cpu_baseline`: the oracle's CPU restatement of the same path (oracle/: C vectoriser + env with
           OpenMP over all host cores, Python sort_training_data, C GAE, numpy flatten, torch-CPU policy and PPO
           update) on a bounded sample of the workload.  /root/reference itself cannot travel to the GPU box.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

import numpy as np
import torch

METRIC = 'agent-steps/sec (env step + PPO rollout/update hot path)'
UNIT = 'agent-steps/s'


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--env', default='breakout')
    ap.add_argument('--num-envs', type=int, default=16384, help='per GPU')
    ap.add_argument('--horizon', type=int, default=128)
    ap.add_argument('--hidden', type=int, default=128)
    ap.add_argument('--no-graph', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extra-configs', action='store_true', help='skip the C3 / C4 per-kernel rooflines')
    ap.add_argument('--minibatches', type=int, default=4, help='batch_size / minibatch_size (reference ratio: 4)')
    ap.add_argument('--epochs', type=int, default=4)
    ap.add_argument('--kernels-only', action='store_true', help='skip the PPO loop; report the per-kernel rooflines')
    ap.add_argument('--ref-horizon', type=int, default=8, help='bounded sample: env steps per reference-arm step')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step computed to DIR/<name>.npy (see dump_outputs)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'b200' or args.kernels_only):
        ap.error('--dump-outputs needs the timed PPO steps of --impl b200')
    return args


def ppo_config(num_envs, horizon, device, seed=1, cuda_graph=True, minibatches=4, epochs=4, env='breakout'):
    import pufferlib_b200
    batch = num_envs * horizon
    return pufferlib_b200.namespace(
        seed=seed, torch_deterministic=True, env=env, batch_size=batch, bptt_horizon=16,
        minibatch_size=batch // minibatches, cpu_offload=False, device=device, compile=False, learning_rate=2.5e-4,
        gamma=0.99, gae_lambda=0.95, update_epochs=epochs, norm_adv=True, clip_coef=0.1, clip_vloss=True,
        vf_clip_coef=0.1, vf_coef=0.5, ent_coef=0.01, max_grad_norm=0.5, target_kl=None, anneal_lr=False,
        total_timesteps=10_000_000_000, cuda_graph=cuda_graph)


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms from the start of the timed region; when that region is shorter
    than ~0.6 s (K steps of 3.6 ms) the same steps keep running, untimed, until at least that long has been sampled under load
    (`window` in the JSON says so)."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', f'--id={self.index}', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                 '-lms', '50'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.06)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for nm, v in zip(names, r[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(nm)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


# ------------------------------------------------------------------------------------------------ B200 arm
def make_b200(args, rank, world, host_buffers, cuda_graph):
    import pufferlib_b200.vector as pvec
    from pufferlib_b200 import clean_pufferl, models, distributed as pdist
    from pufferlib_b200.environments import ocean
    from pufferlib_b200.frameworks import cleanrl
    n = args.num_envs
    vec = pvec.make(ocean.env_creator(args.env), num_envs=n,
                    backend=pvec.B200.options(host_buffers=host_buffers, exact_infos=False,
                                              env_index_offset=rank * n))
    torch.manual_seed(1)
    net = models.Convolutional(vec.driver_env) if args.env == 'pong' else models.Default(vec.driver_env, hidden_size=args.hidden)
    policy = cleanrl.Policy(net, fused_sample=True, seed=1 + rank)
    policy = policy.cuda()
    pdist.broadcast_parameters(policy)
    cfg = ppo_config(n, args.horizon, 'cuda', seed=1, cuda_graph=cuda_graph, minibatches=args.minibatches,
                     epochs=args.epochs, env=args.env)
    data = clean_pufferl.create(cfg, vec, policy)
    return data, clean_pufferl


def timed_steps(data, cp, steps, world):
    """K steps bracketed by barrier + synchronize, timed with CUDA events; returns max-over-ranks milliseconds."""
    import torch.distributed as dist
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        cp.evaluate(data)
        cp.train(data)
    if getattr(data.vecenv, 'host_buffers', False):
        data.vecenv.host_sync()      # e2e: every device->host copy of the timed steps has landed before the clock stops
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device='cuda')
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.barrier()
    return float(ms.item())


DUMP_ROWS = 1 << 16              # rollout rows sampled for the per-row arrays
DUMP_OBS_BYTES = 32 << 20        # float32 bytes of sampled observation rows
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(data, out_dir):
    """Write what the last PPO step handed its caller to out_dir/<name>.npy (float32, or float64 for statistics), so that
    two builds run with the same arguments -- hence the same seeded inputs -- can be compared array by array:
      param_<name>   the policy parameters after the update;
      loss_<name>    the loss statistics of train(); stat_<name> the episode statistics of evaluate();
      rows           the sampled rollout row positions (a fixed, seeded sample of DUMP_ROWS rows); <field> the rollout
                     tensors of the Experience at those positions (actions, logprobs, rewards, dones, values,
                     advantages, returns);
      obs_rows, obs  an evenly spaced subset of `rows` and their observations (at most DUMP_OBS_BYTES)."""
    exp = data.experience
    out = {}
    for name, p in data.policy.named_parameters():
        out['param_' + name] = p.detach().float().cpu().numpy()
    for k, v in data.losses.items():
        out['loss_' + k] = np.float64(v)
    for k, v in data.stats.items():
        out['stat_' + k.replace('/', '_')] = np.float64(v)
    b = exp.batch_size
    rows = np.sort(np.random.default_rng(0).choice(b, min(b, DUMP_ROWS), replace=False))
    idx = torch.as_tensor(rows, device=exp.obs.device)
    out['rows'] = rows.astype(np.float64)
    for k in ('actions', 'logprobs', 'rewards', 'dones', 'values', 'advantages', 'returns'):
        out[k] = getattr(exp, k).index_select(0, idx).float().cpu().numpy()
    k = min(len(rows), max(1, DUMP_OBS_BYTES // (4 * int(np.prod(exp.obs_shape)))))
    sel = np.arange(k) * len(rows) // k
    out['obs_rows'] = rows[sel].astype(np.float64)
    out['obs'] = exp.obs.index_select(0, idx[torch.as_tensor(sel, device=idx.device)]).float().cpu().numpy()
    total = sum(np.asarray(v).nbytes for v in out.values())
    if total > DUMP_MAX_BYTES:
        raise ValueError(f'--dump-outputs: {total} bytes exceed {DUMP_MAX_BYTES}')
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + '.npy'), np.asarray(v))


def kernel_rooflines(data, args, peak_gbs, peak_src):
    """Per-kernel achieved HBM GB/s from ALGORITHMIC bytes / average launch duration (CUDA events on the launch
    stream, back-to-back launches, working sets larger than L2: the 1 GiB rollout rotates under the env kernel)."""
    import ctypes as C
    from pufferlib_b200 import _native
    exp, vec = data.experience, data.vecenv
    n, h, o = args.num_envs, args.horizon, vec.obs_bytes
    lib, s = _native.lib(), _native.stream_ptr()
    out = {}

    def time_launches(fn, reps):
        """Average device time of one launch: `reps` launches captured into a CUDA graph (no Python / ctypes gaps
        between them) and replayed between two events on the launching stream."""
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for i in range(reps):
                fn(i)
        g.replay()                                   # warm-up replay
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        best = float('inf')
        for _ in range(3):
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return best / reps * 1e-3     # seconds per launch

    # env step + obs/reward/done row write (one launch = one vectorised step of N envs)
    actions = torch.randint(0, vec.single_action_space.n, (n,), device='cuda')
    rows = [vec._env_out(t) for t in range(h)]

    def env_step(i):
        _native.check(lib.pb_env_step(vec._handle, _native.ptr(actions), C.byref(rows[i % h]), _native.stream_ptr()))
    for i in range(h):
        env_step(i)
    t_env = time_launches(env_step, h)
    # algorithmic bytes per agent-step (DESIGN.md §3): obs row + reward + done + action; snake also reads the
    # previous row (the obs is the state), pong reads the three surviving frames of it
    extra = {'snake': o, 'pong': 3 * (o // 4)}.get(args.env, 0)
    bytes_env = n * (o + 16 + extra)
    env_kernel = {'snake': 'k_snake4<1> (4 lanes / env)'}.get(args.env, f'k_{args.env}<1>')
    out['env_step'] = dict(kernel=env_kernel, bytes_per_launch=bytes_env, seconds=t_env, launches_per_step=h)
    if args.env == 'snake':      # A/B: the 16-lanes-per-env kernel of round 1
        try:
            _native.check(lib.pb_snake_set_variant(16))
            env_step(0)
            out['env_step_round1_kernel'] = dict(kernel='k_snake<1> (16 lanes / env, round 1)', bytes_per_launch=bytes_env,
                                                 seconds=time_launches(env_step, h), launches_per_step=0)
        finally:
            lib.pb_snake_set_variant(4)

    # GAE (+returns): 20 B per agent-step.  8 rotating input/output sets (8 x 42 MB > the 126 MB L2) so every launch
    # streams from HBM like it does after a 1 GiB rollout has passed through the cache.
    exp.num_envs, exp.horizon = n, h
    exp.compute_gae(0.99, 0.95)                     # allocates the workspace, sets kernel attributes
    torch.cuda.synchronize()
    sets = []
    for k in range(8):
        r = torch.randn(n * h, device='cuda')
        v = torch.randn(n * h, device='cuda')
        d = (torch.rand(n * h, device='cuda') < 0.01).float()
        sets.append((r, v, d, torch.empty(n * h, device='cuda'), torch.empty(n * h, device='cuda')))

    def gae(i):
        r, v, d, a, rt = sets[i % len(sets)]
        _native.check(lib.pb_gae(_native.ptr(r), _native.ptr(v), _native.ptr(d), _native.ptr(a), _native.ptr(rt), n, h,
                                 C.c_float(0.99), C.c_float(0.95), _native.ptr(exp._gae_ws), exp._gae_ws.numel(),
                                 _native.stream_ptr()))
    t_gae = time_launches(gae, 16)
    t_gae_v1 = t_gae_v3 = t_gae_v2 = None
    if h in (128, 256, 512) and n % 4 == 0:      # A/B: the other tile-kernel variants on the same inputs
        try:
            _native.check(lib.pb_gae_set_variant(1))
            gae(0)
            t_gae_v1 = time_launches(gae, 16)
            _native.check(lib.pb_gae_set_variant(3))
            gae(0)
            t_gae_v3 = time_launches(gae, 16)
            _native.check(lib.pb_gae_set_variant(2))
            gae(0)
            t_gae_v2 = time_launches(gae, 16)
        finally:
            lib.pb_gae_set_variant(0)
    del sets
    # pb_gae's dispatch (csrc/gae.cu): the single-pass tile kernel for H in {128, 256, 512} and N % 4 == 0, else the general one
    gae_kernel = 'k_gae_fast' if (h in (128, 256, 512) and n % 4 == 0) else 'k_gae'
    gae_kernel = 'k_gae_tile' if gae_kernel == 'k_gae_fast' else gae_kernel
    if gae_kernel == 'k_gae_tile':
        gae_kernel += ' (double-buffered)' if h <= 128 else ' (single-buffered)'       # pb_gae's choice by horizon (csrc/gae.cu)
    out['gae'] = dict(kernel=gae_kernel, bytes_per_launch=n * h * 20, seconds=t_gae, launches_per_step=1)
    if t_gae_v2 is not None:
        out['gae_double_buffered'] = dict(kernel='k_gae_tile, NBUF = 2 (for comparison)', bytes_per_launch=n * h * 20,
                                          seconds=t_gae_v2, launches_per_step=0)
    if t_gae_v3 is not None:
        out['gae_single_buffered'] = dict(kernel='k_gae_tile, NBUF = 1 (for comparison)', bytes_per_launch=n * h * 20,
                                          seconds=t_gae_v3, launches_per_step=0)
    if t_gae_v1 is not None:
        out['gae_round1_kernel'] = dict(kernel='k_gae_fast (round 1, for comparison)', bytes_per_launch=n * h * 20,
                                        seconds=t_gae_v1, launches_per_step=0)

    # minibatch gather of the observations: read + write of every row
    def gather(i):
        _native.check(lib.pb_minibatch_gather(_native.ptr(exp.obs), _native.ptr(exp.b_obs), exp.obs_row_bytes, n, h,
                                              exp.num_minibatches, exp.minibatch_rows, exp.bptt_horizon, 0,
                                              exp.num_minibatches, _native.stream_ptr()))
    gather(0)
    t_g = time_launches(gather, 5)
    # with zero-copy slab minibatches (the default for the non-LSTM path) the gather is not on the step path at all
    on_path = 0 if getattr(exp, '_slabs', None) is not None else 1
    out['obs_gather'] = dict(kernel='k_minibatch_gather<uint4,8>', bytes_per_launch=2 * n * h * o, seconds=t_g,
                             launches_per_step=on_path)
    # fused rollout-time policy step (encoder + ReLU + heads + sampling), launched on the rollout rows
    pol = data.policy
    if hasattr(pol, '_policy_step_fused') and args.env == 'breakout':
        obs_rows = [exp.obs[t * n:(t + 1) * n] for t in range(h)]
        outs3 = (torch.empty(n, device='cuda'), torch.empty(n, device='cuda'), torch.empty(n, dtype=torch.int64, device='cuda'))

        def pstep(i):
            with torch.no_grad():
                pol._policy_step_fused(obs_rows[i % h], outs3)
        pstep(0)
        t_pol = time_launches(pstep, h)
        out['policy_step'] = dict(kernel='k_policy_mlp_sample', seconds=t_pol,
                                  bytes_per_launch=n * (o + 16) + 128 * 128 * 4, launches_per_step=h)
    # the persistent rollout kernel (H env steps + policy in ONE launch): when evaluate() uses it, the per-step kernels above
    # are off the step path.  Algorithmic bytes per agent-step: obs row + reward + done + value + logprob + action (int64).
    if getattr(data, 'fused_rollouts', 0) > 0 and vec.fused_rollout_ok(exp, pol):
        def roll(i):
            with torch.no_grad():
                vec.fused_rollout(exp, pol)
        roll(0)
        t_roll = time_launches(roll, 4)
        out['rollout'] = dict(kernel='k_breakout_rollout (tcgen05 policy + env, persistent)', seconds=t_roll,
                              bytes_per_launch=n * h * (o + 4 + 4 + 4 + 4 + 8), launches_per_step=1)
        exp.ptr = 0
        for k_ in ('env_step', 'policy_step'):
            if k_ in out:
                out[k_]['launches_per_step'] = 0
    # train-side kernels at the minibatch size of the workload (rotating buffers > L2 where the working set is small)
    if args.env != 'pong' and args.hidden == 128:
        mb = n * h // args.minibatches
        n_act = vec.single_action_space.n
        hid = torch.relu(torch.randn(mb, 128, device='cuda'))
        douts = [torch.randn(mb, 8, device='cuda') for _ in range(4)]
        w_cat = torch.randn(8, 128, device='cuda')
        dpre = torch.empty_like(hid)
        grads = torch.empty(8 * 128 + 128 + 8, device='cuda')
        ws = torch.empty(lib.pb_mlp_tail_workspace_bytes(mb, 128), dtype=torch.uint8, device='cuda')

        def tail(i):
            d = douts[i % 4]
            _native.check(lib.pb_mlp_tail_backward(_native.ptr(d), 8, _native.ptr(w_cat), _native.ptr(hid), mb, 128,
                                                   _native.ptr(dpre), _native.ptr(grads), _native.ptr(ws), ws.numel(),
                                                   _native.stream_ptr()))
        tail(0)
        t_tail = time_launches(tail, 4)
        out['mlp_tail_bwd'] = dict(kernel='k_mlp_tail_bwd_tma<128> + k_reduce_partials', seconds=t_tail,
                                   bytes_per_launch=mb * (2 * 128 * 4 + 32), launches_per_step=args.minibatches * args.epochs)
        outs = [torch.randn(mb, 8, device='cuda') for _ in range(4)]
        gouts = torch.zeros(mb, 8, device='cuda')
        acts = torch.randint(0, n_act, (mb,), device='cuda')
        f32 = [torch.randn(mb, device='cuda') for _ in range(4)]
        stats = torch.zeros(8, dtype=torch.float64, device='cuda')

        def loss(i):
            o = outs[i % 4]
            _native.check(lib.pb_ppo_loss(_native.ptr(o), 8, C.c_void_p(o.data_ptr() + 4 * n_act), 8, _native.ptr(acts),
                                          _native.ptr(f32[0]), _native.ptr(f32[1]), _native.ptr(f32[2]), _native.ptr(f32[3]),
                                          mb, n_act, C.c_float(0.1), 1, C.c_float(0.1), C.c_float(0.5), C.c_float(0.01),
                                          _native.ptr(gouts), 8, C.c_void_p(gouts.data_ptr() + 4 * n_act), 8,
                                          _native.ptr(stats), _native.stream_ptr()))
        loss(0)
        t_loss = time_launches(loss, 8)
        out['ppo_loss'] = dict(kernel='k_ppo_loss', seconds=t_loss, bytes_per_launch=mb * (8 * n_act + 32 + 4),
                               launches_per_step=args.minibatches * args.epochs)
        del hid, douts, dpre, outs, gouts
        # the fused tcgen05 minibatch update (forward + loss + backward in one kernel): algorithmic bytes = the observation
        # rows (read once) + 24 B of per-row scalars; launched on zero-copy slab views of the rollout like train() does
        mu = getattr(data, 'manual_update', None)
        if mu is not None and getattr(mu, 'used_fused', False) and o == 512:
            from pufferlib_b200 import clean_pufferl as cp_
            nm = args.minibatches
            layout = cp_.slab_layout(n, h, nm, 16)
            if layout is not None:
                g_, r_ = layout
                xs = [exp.obs.view(g_, nm, r_, 128)[:, k] for k in range(nm)]
                ws = torch.empty(lib.pb_mlp_update_workspace_bytes(), dtype=torch.uint8, device='cuda')
                gfl = torch.empty(128 * 128 + 8 * 128 + 128 + 8, device='cuda')
                st8 = torch.zeros(8, dtype=torch.float64, device='cuda')
                model = data.policy.policy
                w_cat, b_cat = model.head_matrix()

                def upd(i):
                    x = xs[i % nm]
                    _native.check(lib.pb_mlp_update_fused(
                        _native.ptr(x), 128, r_, x.stride(0) // 128 if g_ > 1 else r_, g_, _native.ptr(model.encoder.weight),
                        _native.ptr(model.encoder.bias), _native.ptr(w_cat), _native.ptr(b_cat), _native.ptr(acts),
                        _native.ptr(f32[0]), _native.ptr(f32[1]), _native.ptr(f32[2]), _native.ptr(f32[3]), None, r_, n_act,
                        C.c_float(0.1), 1,
                        C.c_float(0.1), C.c_float(0.5), C.c_float(0.01), _native.ptr(gfl), _native.ptr(st8), _native.ptr(ws),
                        ws.numel(), _native.ptr(dpre_b) if dpre_b is not None else None, None, None, None, _native.stream_ptr()))
                dw_mode = str(getattr(data.config, 'fused_update_dw', cp_.FUSED_UPDATE_DW_DEFAULT))
                dpre_b = None if dw_mode == 'kernel' else torch.empty(mb, 128, device='cuda')
                with torch.no_grad():
                    upd(0)
                    t_upd = time_launches(upd, 8)
                out['mlp_update'] = dict(kernel=('k_mlp_update_xt (tcgen05 forward / x^T / dW + mma.sync epilogue)' if dw_mode == 'kernel' else
                                                 'k_mlp_update_fused (tcgen05, dPre to HBM, dW: cuBLAS)') + ' + k_update_reduce', seconds=t_upd,
                                         bytes_per_launch=mb * (512 + 28 + (512 if dpre_b is not None else 0)),
                                         launches_per_step=nm * args.epochs,
                                         tf32_tflops=round(2 * 2 * mb * 128 * 128 / t_upd / 1e12, 1))
    for k, v in out.items():
        v['achieved'] = v['bytes_per_launch'] / v['seconds'] / 1e9
        v['frac'] = v['achieved'] / peak_gbs
        v['share_s'] = v['seconds'] * v['launches_per_step']
    dom = max(out, key=lambda k: out[k]['share_s'])
    d = out[dom]
    # DRAM traffic per launch from the committed `ncu --set full` capture of this workload (profiles/), else null
    traffic = None
    try:
        tr = json.load(open(os.path.join(REPO, 'profiles', 'ncu_traffic_r02.json')))['bytes_per_launch']
        if args.env == 'breakout' and n == 16384 and h == 128:
            traffic = tr.get({'env_step': 'breakout', 'obs_gather': 'gather'}.get(dom, dom))
    except Exception:
        pass
    roof = {'bound': 'hbm', 'kernel': d['kernel'], 'achieved': round(d['achieved'], 1), 'peak': peak_gbs,
            'peak_source': peak_src, 'unit': 'GB/s', 'frac': round(d['frac'], 4), 'traffic': traffic,
            'algorithmic_bytes_per_launch': d['bytes_per_launch'], 'avg_launch_us': round(d['seconds'] * 1e6, 2)}
    others = {k: {'kernel': v['kernel'], 'achieved': round(v['achieved'], 1), 'frac': round(v['frac'], 4),
                  'avg_launch_us': round(v['seconds'] * 1e6, 2), 'algorithmic_bytes_per_launch': v['bytes_per_launch'],
                  'launches_per_step': v['launches_per_step'], **({'tf32_tflops': v['tf32_tflops']} if 'tf32_tflops' in v else {})}
              for k, v in out.items()}
    return roof, others


def load_peak():
    p = os.path.join(REPO, 'MEASURED_PEAKS.json')
    try:
        return float(json.load(open(p))['hbm_gbs']), 'MEASURED_PEAKS.json (measured copy bandwidth)'
    except Exception:
        return 6650.0, 'fallback 6.65 TB/s (B200_PROFILING.md)'


def run_b200(args):
    from pufferlib_b200 import distributed as pdist, _native
    rank, local, world = pdist.init()
    assert world == args.gpus, f'launched with WORLD_SIZE={world} but --gpus {args.gpus}'
    torch.cuda.set_device(local)
    n, h = args.num_envs, args.horizon
    data, cp = make_b200(args, rank, world, host_buffers=False, cuda_graph=not args.no_graph)
    if args.kernels_only:   # per-kernel HBM rooflines of another config (C3 snake, C4 pong) without the PPO loop
        peak, peak_src = load_peak()
        roof, roof_all = kernel_rooflines(data, args, peak, peak_src)
        if rank == 0:
            print(json.dumps({'kernels_only': True, 'config': {'workload': f'{args.env} num_envs={n} horizon={h}'},
                              'roofline': roof, 'roofline_kernels': roof_all}))
        cp.close(data)
        return
    for _ in range(max(args.warmup, 3)):
        cp.evaluate(data)
        cp.train(data)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    launches0, replays0, treplays0 = _native.lib().pb_launch_count(), data.graph_replays, data.train_graph_replays
    seg0 = getattr(data.train_segments, 'replayed_launches', 0)
    ms = timed_steps(data, cp, args.steps, world)
    if args.dump_outputs and rank == 0:
        dump_outputs(data, args.dump_outputs)
    launches = ((_native.lib().pb_launch_count() - launches0) + (data.graph_replays - replays0) * data.graph_launches
                + (data.train_graph_replays - treplays0) * data.train_graph_launches
                + (getattr(data.train_segments, 'replayed_launches', 0) - seg0))
    # clocks under load: keep the same steps running (untimed) until the sampler has had 0.6 s of them
    # (the count comes from the rank-maximum step time, so every rank runs the same number of exchanges)
    extra = max(0, int(np.ceil((600.0 - ms) / max(ms / args.steps, 1e-3)))) if ms < 600.0 else 0
    extra = min(extra, 2000)
    for i in range(extra):
        cp.evaluate(data)
        cp.train(data)
        if i % 8 == 7:
            torch.cuda.synchronize()
    torch.cuda.synchronize()
    clk = clocks.stop() if rank == 0 else None
    if clk is not None:
        clk['window'] = f'{args.steps} timed steps' + (f' + {extra} more of the same steps, untimed' if extra else '')
    value = world * n * h * args.steps / (ms * 1e-3)
    prof = {k: round(v, 4) for k, v in dict(data.profile).items() if k.endswith('_time')}
    stats = {k: float(v) for k, v in data.stats.items()}

    peak, peak_src = load_peak()
    roof, roof_all = kernel_rooflines(data, args, peak, peak_src)

    # ---- e2e: same step through the public API with host buffers
    e2e = None
    if not args.no_e2e:
        # host buffers: the rollout loop talks to the host every env step (no rollout graph); the update has no host
        # interaction, so it is still captured (first train() eager, second captures: two warm-up steps)
        hdata, _ = make_b200(args, rank, world, host_buffers=True, cuda_graph=not args.no_graph)
        for _ in range(2):
            cp.evaluate(hdata); cp.train(hdata)
        hv = hdata.vecenv
        io0 = (hdata.io.h2d + hv.h2d_bytes, hdata.io.d2h + hv.d2h_bytes)
        k_e2e = args.steps
        ms_e = timed_steps(hdata, cp, k_e2e, world)
        io1 = (hdata.io.h2d + hv.h2d_bytes, hdata.io.d2h + hv.d2h_bytes)
        e2e = {'value': world * n * h * k_e2e / (ms_e * 1e-3), 'unit': UNIT, 'steps': k_e2e,
               'h2d_bytes_per_step': int((io1[0] - io0[0]) / k_e2e), 'd2h_bytes_per_step': int((io1[1] - io0[1]) / k_e2e),
               'api': 'pufferlib_b200.vector.make(backend=B200.options(host_buffers=True)) + clean_pufferl.evaluate/train'}
        cp.close(hdata)

    # ---- the other single-GPU configs of BASELINE.json (C3 snake: the GAE / obs-write HBM roofline config; C4 pong: the
    # TMA image pack): per-kernel rooflines only (their full PPO loops are covered by tests/test_gpu_configs.py)
    extra = {}
    if world == 1 and not args.no_extra_configs:
        import copy
        for key, kw in (('c3_snake', dict(env='snake', num_envs=65536, horizon=256)),
                        ('c4_pong', dict(env='pong', num_envs=8192, horizon=128))):
            try:
                a2 = copy.copy(args)
                for k_, v_ in kw.items():
                    setattr(a2, k_, v_)
                d2, _ = make_b200(a2, rank, world, host_buffers=False, cuda_graph=False)
                r2, all2 = kernel_rooflines(d2, a2, peak, peak_src)
                extra[key] = {'workload': f"{kw['env']} num_envs={kw['num_envs']} horizon={kw['horizon']}", 'roofline_kernels': all2}
                cp.close(d2)
                del d2
                torch.cuda.empty_cache()
            except Exception as e:           # never lose the headline line to an auxiliary measurement
                extra[key] = {'error': f'{type(e).__name__}: {e}'}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = reference_arm(args, steps=5, warmup=1)

    if rank == 0:
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
            'warmup': max(args.warmup, 3), 'ms_per_step': ms / args.steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32 (env state int32; policy GEMMs tf32 like the reference)',
            'data': 'synthetic (fixed-seed envs, random-init policy)',
            'config': {'workload': f'{args.env} num_envs={n}/GPU horizon={h} MLP hidden={args.hidden} '
                                   f'(BASELINE.json configs[1]; x{world} ranks = configs[4])',
                       'global_batch': world * n * h, 'minibatch_size': n * h // args.minibatches, 'update_epochs': args.epochs,
                       'bptt_horizon': 16, 'parallelism': f'dp{world} (env shards; one 68.6 KB gradient exchange per optimizer step over NVLink peer memory, inside the update graph)',
                       'l2': 'inputs larger than L2 (1 GiB rollout rotates; no flush needed)',
                       'cuda_graph_rollout': not args.no_graph,
                       'cuda_graph_train': 'whole' if data.train_graph_state == 2 else ('segments' if data.train_segments else False), 'zero_copy_minibatches': getattr(data.experience, '_slabs', None) is not None, 'note': data.msg},
            'e2e': e2e, 'gpu_launches': int(launches), 'roofline': roof, 'roofline_kernels': roof_all,
            'roofline_other_configs': extra,
            'cpu_baseline': cpu, 'clocks': clk, 'profile_s': prof, 'env_stats': stats,
        }
        print(json.dumps(line))
    cp.close(data)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ reference arm
def reference_arm(args, steps, warmup):
    """The reference path's CPU implementation, restated by the oracle, on all host cores, on a bounded sample."""
    import psutil
    from oracle.envs import OracleVec, NUM_ACTIONS, OBS
    from oracle import experience as oexp
    from oracle import gae as ogae
    cores = psutil.cpu_count(logical=False) or os.cpu_count()
    n, h = args.num_envs, args.ref_horizon
    batch = n * h
    shape, dtype = OBS[args.env]
    vec = OracleVec(args.env, n, threads=cores)       # env stepping: OpenMP over all physical cores
    vec.collect_infos = False
    torch.manual_seed(1)
    in_dim, n_act = int(np.prod(shape)), NUM_ACTIONS[args.env]
    enc, dec, vh = torch.nn.Linear(in_dim, args.hidden), torch.nn.Linear(args.hidden, n_act), torch.nn.Linear(args.hidden, 1)
    params = list(enc.parameters()) + list(dec.parameters()) + list(vh.parameters())
    opt = torch.optim.Adam(params, lr=2.5e-4, eps=1e-5)

    def policy(obs, action=None):
        hid = torch.relu(enc(obs.reshape(obs.shape[0], -1).float()))
        logits, value = dec(hid), vh(hid)
        norm = logits - logits.logsumexp(-1, keepdim=True)
        if action is None:
            action = torch.multinomial(norm.exp(), 1).squeeze(-1)
        logprob = norm.gather(-1, action.reshape(-1, 1)).squeeze(-1)
        ent = -(norm * norm.exp()).sum(-1)
        return action, logprob, ent, value

    vec.async_reset(1)

    def one_step():
        exp = oexp.Experience(batch, 16, batch // 4, shape, dtype)
        while not exp.full:                                           # clean_pufferl.evaluate (:84-124)
            o, r, d, t, info, env_id, mask = vec.recv()
            with torch.no_grad():
                a, lp, _, v = policy(torch.as_tensor(o))
            exp.store(o, v.flatten().numpy(), a.numpy(), lp.numpy(), r, d, env_id, mask)
            vec.send(a.numpy())
        idxs = exp.sort_training_data()                               # clean_pufferl.train (:163-170)
        adv = ogae.compute_gae(exp.dones[idxs], exp.values[idxs], exp.rewards[idxs], 0.99, 0.95)
        exp.flatten_batch(adv)
        for epoch in range(4):
            for mb in range(exp.num_minibatches):
                obs = torch.as_tensor(exp.b_obs[mb]).reshape(-1, *shape)
                atn = torch.as_tensor(exp.b_actions[mb]).reshape(-1)
                _, nlp, ent, nv = policy(obs, atn)
                logratio = nlp - torch.as_tensor(exp.b_logprobs[mb]).reshape(-1)
                ratio = logratio.exp()
                a_ = torch.as_tensor(exp.b_advantages[mb]).reshape(-1)
                a_ = (a_ - a_.mean()) / (a_.std() + 1e-8)
                pg = torch.max(-a_ * ratio, -a_ * torch.clamp(ratio, 0.9, 1.1)).mean()
                nv = nv.view(-1)
                ret, val = torch.as_tensor(exp.b_returns[mb]), torch.as_tensor(exp.b_values[mb])
                v_clipped = val + torch.clamp(nv - val, -0.1, 0.1)
                vl = 0.5 * torch.max((nv - ret) ** 2, (v_clipped - ret) ** 2).mean()
                loss = pg - 0.01 * ent.mean() + 0.5 * vl
                opt.zero_grad()
                loss.backward()
                torch.nn.utils.clip_grad_norm_(params, 0.5)
                opt.step()

    # torch's CPU thread count: all cores is not always fastest for these small GEMMs -- take the best of a few
    # settings, measured, so the baseline is as strong as the host allows
    best_threads, best_dt = cores, float('inf')
    for th in sorted({cores, max(1, cores // 2), max(1, cores // 4), min(cores, 16), min(cores, 8)}, reverse=True):
        torch.set_num_threads(th)
        one_step()
        t0 = time.perf_counter()
        one_step()
        dt_th = time.perf_counter() - t0
        if dt_th < best_dt:
            best_threads, best_dt = th, dt_th
    torch.set_num_threads(best_threads)
    for _ in range(warmup):
        one_step()
    t0 = time.perf_counter()
    for _ in range(steps):
        one_step()
    dt = time.perf_counter() - t0
    value = batch * steps / dt
    return {'value': value, 'unit': UNIT, 'cores': int(cores), 'torch_threads': int(best_threads), 'kind': 'port',
            'sample': f'{args.env} num_envs={n} x {h} env steps of the {args.horizon}-step rollout per step '
                      f'({batch} agent-steps), full PPO update on it (4 epochs x 4 minibatches), {steps} steps',
            'seconds': dt}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    res = reference_arm(args, steps=args.steps, warmup=max(1, min(args.warmup, 2)))
    n, h = args.num_envs, args.ref_horizon
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': res['value'], 'unit': UNIT, 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': max(1, min(args.warmup, 2)), 'ms_per_step': res['seconds'] / args.steps * 1e3,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': f'{args.env} num_envs={n} horizon={args.horizon} MLP hidden={args.hidden} '
                               f'(bounded sample: {h} env steps per step)', 'parallelism': 'host cores (OpenMP + torch CPU)'},
        'cpu_baseline': {k: res[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')},
        'e2e': {'value': res['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line))


if __name__ == '__main__':
    a = parse_args()
    if a.impl == 'reference':
        run_reference(a)
    else:
        run_b200(a)
