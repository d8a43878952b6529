"""``clean_pufferl`` create / evaluate / train / close with the reference signatures, device-resident.

Mirrors /root/reference/clean_pufferl.py: ``create`` (:30-73), ``evaluate`` (:75-154), ``train`` (:156-292),
``close`` (:294-304), ``Experience`` (:380-482), ``make_losses`` (:369-378), ``seed_everything``.  What changes:

* ``Experience`` tensors all live in HBM in arrival order (row t*N + e) -- the same memory layout the reference
  gives them -- and the env-step kernel writes obs / reward / done rows into them directly
  (``vecenv.bind_rollout``).  ``store`` is one fused kernel for value / logprob / action (pb_rollout_store).
* ``sort_training_data`` is arithmetic (sorted position e*H+t <-> arrival row t*N+e): no Python sort, no index
  tensor.  GAE is one launch (pb_gae) reading the arrival-order tensors transposed; ``flatten_batch`` is one
  launch for the scalars (pb_flatten_batch) + one gather for the observations (pb_minibatch_gather); the
  per-minibatch advantage normalisation of train (:211-213) is done for all minibatches at once (pb_adv_norm).
* No per-step device<->host traffic in evaluate; losses are accumulated on the device and read once per train.
* Multi-GPU: if torch.distributed is initialised, gradients are summed with ONE all-reduce over a flat bucket
  per optimizer step (NCCL over NVLink) -- the reference has no distributed path (SURVEY §8e).

The policy stays a torch ``nn.Module`` with the reference's call convention
(``policy(obs) -> actions, logprob, entropy, value``; ``policy(obs, action=a)`` in train).
"""
import ctypes as C
import random
import time
from collections import defaultdict

import numpy as np
import torch

import pufferlib_b200
from pufferlib_b200 import _native
from pufferlib_b200.exceptions import APIUsageError

torch.set_float32_matmul_precision('high')   # clean_pufferl.py:22

numpy_to_torch_dtype_dict = {
    np.dtype('float64'): torch.float64, np.dtype('float32'): torch.float32, np.dtype('float16'): torch.float16,
    np.dtype('uint8'): torch.uint8, np.dtype('int8'): torch.int8, np.dtype('int16'): torch.int16,
    np.dtype('int32'): torch.int32, np.dtype('int64'): torch.int64, np.dtype('bool'): torch.bool,
}


def seed_everything(seed, torch_deterministic):
    random.seed(seed)
    np.random.seed(seed)
    if seed is not None:
        torch.manual_seed(seed)
    torch.backends.cudnn.deterministic = torch_deterministic


def make_losses():
    return pufferlib_b200.namespace(policy_loss=0, value_loss=0, entropy=0, old_approx_kl=0, approx_kl=0,
                                    clipfrac=0, explained_variance=0)


class Profile:
    """Wall-clock buckets with the reference's names (clean_pufferl.py:306-367); device work is asynchronous, so
    a bucket is only exact where the caller synchronises (end of evaluate / end of train)."""
    BUCKETS = ('env', 'eval_forward', 'eval_misc', 'train_forward', 'learn', 'train_misc')

    class _Timer:
        def __init__(self):
            self.elapsed = 0.0
            self._t0 = 0.0

        def __enter__(self):
            self._t0 = time.perf_counter()
            return self

        def __exit__(self, *a):
            self.elapsed += time.perf_counter() - self._t0

    def __init__(self):
        for b in self.BUCKETS:
            setattr(self, b, Profile._Timer())
        self.start = time.time()
        self.SPS = 0
        self.uptime = 0
        self._last_step = 0
        self._last_time = time.time()

    def __iter__(self):
        yield 'SPS', self.SPS
        yield 'uptime', self.uptime
        for b in self.BUCKETS:
            yield b + '_time', getattr(self, b).elapsed

    def update(self, data, interval_s=1):
        now = time.time()
        if now - self._last_time < interval_s:
            return False
        self.SPS = (data.global_step - self._last_step) / (now - self._last_time)
        self._last_step, self._last_time = data.global_step, now
        self.uptime = now - self.start
        return True


class _FusedPPOLoss(torch.autograd.Function):
    """clean_pufferl.py:202-238 as ONE kernel (pb_ppo_loss): forward returns (loss, stats[6]) and stashes the analytic
    gradients w.r.t. logits / value that backward hands to autograd for the network backward."""

    @staticmethod
    def forward(ctx, logits, value, actions, old_logprobs, adv, returns, old_values, cfg, packed_n_act):
        """packed_n_act > 0: `logits` is the packed head output [M, 8] (logits | value | zero pad) and `value` is
        ignored; the gradient comes back as ONE [M, 8] tensor (no slice/cat nodes in the autograd graph)."""
        clip_coef, clip_vloss, vf_clip_coef, vf_coef, ent_coef = cfg
        dev = logits.device
        if packed_n_act:
            out, n_act = logits, packed_n_act
            m = out.shape[0]
            assert out.stride(1) == 1 and out.dtype == torch.float32
            l_ptr, l_stride = out.data_ptr(), out.stride(0)
            v_ptr, v_stride = out.data_ptr() + 4 * n_act, out.stride(0)
            # [M, 8] rows: the kernel writes whole rows (zero padding included); other widths need the memset
            grad = torch.empty_like(out) if out.shape[1] == 8 and n_act <= 7 else torch.zeros_like(out)
            gl_ptr, gl_stride, gv_ptr, gv_stride = grad.data_ptr(), grad.stride(0), grad.data_ptr() + 4 * n_act, grad.stride(0)
            ctx.packed = True
            ctx.save_for_backward(grad)
        else:
            m, n_act = logits.shape
            v2 = value.reshape(m, -1)
            if logits.stride(1) != 1 or logits.dtype != torch.float32:
                logits = logits.float().contiguous()
            grad_logits = torch.empty(m, n_act, dtype=torch.float32, device=dev)
            grad_value = torch.empty(m, dtype=torch.float32, device=dev)
            l_ptr, l_stride, v_ptr, v_stride = logits.data_ptr(), logits.stride(0), v2.data_ptr(), v2.stride(0)
            gl_ptr, gl_stride, gv_ptr, gv_stride = grad_logits.data_ptr(), n_act, grad_value.data_ptr(), 1
            ctx.packed = False
            ctx.save_for_backward(grad_logits, grad_value)
            ctx.value_shape = value.shape
        stats = torch.empty(8, dtype=torch.float64, device=dev)
        cp = C.c_void_p
        _native.check(_native.lib().pb_ppo_loss(
            cp(l_ptr), l_stride, cp(v_ptr), v_stride,
            _native.ptr(actions.reshape(-1).contiguous()), _native.ptr(old_logprobs.reshape(-1).contiguous()),
            _native.ptr(adv.reshape(-1).contiguous()), _native.ptr(returns.reshape(-1).contiguous()),
            _native.ptr(old_values.reshape(-1).contiguous()), m, n_act, C.c_float(clip_coef), int(bool(clip_vloss)),
            C.c_float(vf_clip_coef), C.c_float(vf_coef), C.c_float(ent_coef), cp(gl_ptr), gl_stride, cp(gv_ptr),
            gv_stride, _native.ptr(stats), _native.stream_ptr()))
        means = stats[:6] / m
        means[1] *= 0.5                                  # v_loss = 0.5 * mean(max(...))
        loss = (means[0] - ent_coef * means[2] + vf_coef * means[1]).float()
        return loss, means.float()

    @staticmethod
    def backward(ctx, g_loss, g_stats):
        if ctx.packed:
            (grad,) = ctx.saved_tensors
            return g_loss * grad, None, None, None, None, None, None, None, None
        grad_logits, grad_value = ctx.saved_tensors
        return (g_loss * grad_logits, (g_loss * grad_value).view(ctx.value_shape), None, None, None, None, None, None,
                None)


class _FusedPPOLossMulti(torch.autograd.Function):
    """_FusedPPOLoss for a MultiDiscrete space (pb_ppo_loss_multi): `logits` holds every head's columns, head after head
    ([M, sum(nvec)], or the packed [M, 8] head output with the value in column sum(nvec) when packed).  The gradient
    comes back in the same layout, so the packed form hands ONE [M, 8] gradient to pb_mlp_tail_backward."""

    @staticmethod
    def forward(ctx, logits, value, actions, old_logprobs, adv, returns, old_values, cfg, nvec, packed):
        clip_coef, clip_vloss, vf_clip_coef, vf_coef, ent_coef = cfg
        total, m = sum(nvec), logits.shape[0]
        if logits.stride(1) != 1 or logits.dtype != torch.float32:
            logits = logits.float().contiguous()
        grad = torch.empty_like(logits)
        if packed:
            l_ptr, v_ptr, v_stride = logits.data_ptr(), logits.data_ptr() + 4 * total, logits.stride(0)
            grad_value = None
            gv_ptr, gv_stride = grad.data_ptr() + 4 * total, grad.stride(0)
            if grad.shape[1] != 8:          # the kernel writes whole rows only for [M, 8]
                grad.zero_()
        else:
            v2 = value.reshape(m, -1)
            l_ptr, v_ptr, v_stride = logits.data_ptr(), v2.data_ptr(), v2.stride(0)
            grad_value = torch.empty(m, dtype=torch.float32, device=logits.device)
            gv_ptr, gv_stride = grad_value.data_ptr(), 1
            ctx.value_shape = value.shape
        stats = torch.empty(8, dtype=torch.float64, device=logits.device)
        cp = C.c_void_p
        nv = (C.c_int32 * len(nvec))(*nvec)
        _native.check(_native.lib().pb_ppo_loss_multi(
            cp(l_ptr), logits.stride(0), cp(v_ptr), v_stride,
            _native.ptr(actions.reshape(m, len(nvec)).contiguous()), _native.ptr(old_logprobs.reshape(-1).contiguous()),
            _native.ptr(adv.reshape(-1).contiguous()), _native.ptr(returns.reshape(-1).contiguous()),
            _native.ptr(old_values.reshape(-1).contiguous()), m, nv, len(nvec), C.c_float(clip_coef),
            int(bool(clip_vloss)), C.c_float(vf_clip_coef), C.c_float(vf_coef), C.c_float(ent_coef), cp(grad.data_ptr()),
            grad.stride(0), cp(gv_ptr), gv_stride, _native.ptr(stats), _native.stream_ptr()))
        ctx.packed = packed
        ctx.save_for_backward(grad, *(() if grad_value is None else (grad_value,)))
        means = stats[:6] / m
        means[1] *= 0.5
        loss = (means[0] - ent_coef * means[2] + vf_coef * means[1]).float()
        return loss, means.float()

    @staticmethod
    def backward(ctx, g_loss, g_stats):
        none = (None,) * 8
        if ctx.packed:
            (grad,) = ctx.saved_tensors
            return (g_loss * grad, None) + none
        grad, grad_value = ctx.saved_tensors
        return (g_loss * grad, (g_loss * grad_value).view(ctx.value_shape)) + none


def _loss_cfg(config):
    return (float(config.clip_coef), bool(config.clip_vloss), float(config.vf_clip_coef), float(config.vf_coef),
            float(config.ent_coef))


def fused_ppo_loss_multi(logits, value, actions, old_logprobs, adv, returns, old_values, config):
    """fused_ppo_loss for a list of head logits (MultiDiscrete); actions [M, k]."""
    nvec = [lg.shape[1] for lg in logits]
    return _FusedPPOLossMulti.apply(torch.cat(logits, dim=1), value, actions, old_logprobs, adv, returns, old_values,
                                    _loss_cfg(config), nvec, False)


def fused_ppo_loss_packed_multi(out, nvec, actions, old_logprobs, adv, returns, old_values, config):
    """fused_ppo_loss_packed for a MultiDiscrete models.Default: out = [M, 8] (all heads | value | zero padding)."""
    return _FusedPPOLossMulti.apply(out, None, actions, old_logprobs, adv, returns, old_values, _loss_cfg(config),
                                    list(nvec), True)


def fused_ppo_loss(logits, value, actions, old_logprobs, adv, returns, old_values, config):
    """-> (loss, stats) with stats = [pg_loss, v_loss, entropy, old_approx_kl, approx_kl, clipfrac] (detached)."""
    cfg = (float(config.clip_coef), bool(config.clip_vloss), float(config.vf_clip_coef), float(config.vf_coef),
           float(config.ent_coef))
    return _FusedPPOLoss.apply(logits, value, actions, old_logprobs, adv, returns, old_values, cfg, 0)


def fused_ppo_loss_packed(out, n_act, actions, old_logprobs, adv, returns, old_values, config):
    """Same, on the packed head output [M, 8] of models.Default.forward_packed (one [M, 8] gradient back)."""
    cfg = (float(config.clip_coef), bool(config.clip_vloss), float(config.vf_clip_coef), float(config.vf_coef),
           float(config.ent_coef))
    return _FusedPPOLoss.apply(out, None, actions, old_logprobs, adv, returns, old_values, cfg, int(n_act))


def slab_layout(num_envs, horizon, num_minibatches, bptt_horizon):
    """(G, R) of the zero-copy minibatch form, or None when the reference minibatches are not unions of whole time
    windows.  Minibatch mb of clean_pufferl.py:452-482 holds the bptt segments s = r*n_mb + mb of the (env, step)
    sorted batch; segment s = e*S + k (S = horizon / bptt segments per env) lies in minibatch (e*S + k) % n_mb, which is
    k % n_mb for every env iff S % n_mb == 0.  Then minibatch mb = time windows k = mb, mb + n_mb, ... of ALL envs =
    G = S / n_mb slabs of R = bptt * num_envs consecutive rows of the time-major rollout buffer."""
    if horizon % bptt_horizon != 0:
        return None
    s_per_env = horizon // bptt_horizon
    if s_per_env % num_minibatches != 0:
        return None
    return s_per_env // num_minibatches, bptt_horizon * num_envs


def slab_row_index(num_envs, horizon, num_minibatches, bptt_horizon):
    """[n_mb, G*R] arrival-order row of every slab-major minibatch position (numpy; for tests and documentation --
    the device path never materialises it): position (g, j, e) of minibatch mb is row ((g*n_mb + mb)*bptt + j)*N + e."""
    g_, r_ = slab_layout(num_envs, horizon, num_minibatches, bptt_horizon)
    rows = np.arange(num_envs * horizon, dtype=np.int64).reshape(g_, num_minibatches, r_)
    return rows.transpose(1, 0, 2).reshape(num_minibatches, g_ * r_)


# the fused tcgen05 minibatch-update kernel (csrc/mlp_update.cu) is the default where it applies; config.fused_update
# overrides
FUSED_UPDATE_DEFAULT = True
FUSED_UPDATE_DW_DEFAULT = 'kernel'      # the fused kernel forms dW_enc itself (the only mode); bench.py reads this name
# the persistent rollout kernel (pb_rollout_breakout_mlp) likewise; config.fused_rollout overrides
FUSED_ROLLOUT_DEFAULT = True


class _DefaultMLPUpdate:
    """The minibatch update of clean_pufferl.py:186-244 for models.Default + the fused PPO loss, written out by hand
    instead of through autograd: with 17k parameters and 524k-row minibatches the update is a fixed chain of seven
    large kernels, and everything autograd, clip_grad_norm_ and the optimizer add around it (gradient scaling by the
    upstream 1.0, AccumulateGrad copies, ~12 norm/clip/Adam launches, 6 launches to re-pack the heads, 8 to fold the
    statistics) is ~120 us of 3-us launches per minibatch.  Chain per minibatch:
        encoder GEMM (+bias+ReLU epilogue, one per slab) -> 8-column head GEMM -> pb_ppo_loss (loss statistics +
        analytic dLoss/dOut) -> pb_mlp_tail_backward (dPre, dW_heads, db_heads, db_enc) -> split-K dW_enc GEMM + sum
        [-> gradient all-reduce over ONE flat buffer when world_size > 1] -> pb_clip_adam -> pb_pack_heads.
    Same math as the autograd path (tests/test_gpu_experience.py::test_manual_update_matches_autograd_update); the
    optimizer's own state tensors are updated in place, so state_dict() and optimizer.step() keep working."""

    @staticmethod
    def eligible(data):
        config, model, opt = data.config, getattr(data.policy, 'policy', None), data.optimizer
        if not (data.fused_loss and data.experience.lstm_h is None and bool(getattr(config, 'manual_update', True))):
            return False
        if not (hasattr(model, 'forward_packed_slabs') and getattr(model, 'fast_path', False)):
            return False
        if config.target_kl is not None or not getattr(data, 'own_optimizer', False):
            return False
        if not bool(getattr(config, 'manual_update_multi_gpu', True)):
            world = torch.distributed.get_world_size() if (torch.distributed.is_available() and
                                                            torch.distributed.is_initialized()) else 1
            if world > 1:
                return False      # opt-out: ranks > 1 on the autograd + GradBucket (NCCL) path
        if not isinstance(model.decoder, torch.nn.Linear):
            return False          # MultiDiscrete heads: the fused update kernel and this chain handle one Discrete head
        n_act, hid = model.decoder.weight.shape
        if hid != 128 or n_act > 7 or model.encoder.weight.dtype != torch.float32 or not model.encoder.weight.is_cuda:
            return False
        g = opt.param_groups[0]
        if len(opt.param_groups) != 1 or g.get('amsgrad') or g.get('weight_decay') or g.get('maximize'):
            return False
        params = [model.encoder.weight, model.encoder.bias, model.decoder.weight, model.decoder.bias,
                  model.value_head.weight, model.value_head.bias]
        mine = {id(p) for p in params}
        return {id(p) for p in g['params']} == mine and sum(p.numel() for p in params) <= (1 << 20)

    def __init__(self, data):
        model, opt = data.policy.policy, data.optimizer
        self.model, self.opt = model, opt
        dev = model.encoder.weight.device
        self.n_act, self.hid = model.decoder.weight.shape
        self.features = model.encoder.weight.shape[1]
        hid, f_, n_act = self.hid, self.features, self.n_act
        z = dict(dtype=torch.float32, device=dev)
        # ONE flat gradient buffer: dW_enc | dW_heads (8 x hid) | db_enc | db_heads (8)  (also the all-reduce bucket)
        self.gflat = torch.zeros(hid * f_ + 8 * hid + hid + 8, **z)
        self.dw_enc = self.gflat[:hid * f_].view(hid, f_)
        self.tail = self.gflat[hid * f_:]
        dw_cat = self.tail[:8 * hid].view(8, hid)
        db_enc, db_cat = self.tail[8 * hid:9 * hid], self.tail[9 * hid:]
        self.w_cat, self.b_cat = torch.zeros(8, hid, **z), torch.zeros(8, **z)
        params = [model.encoder.weight, model.encoder.bias, model.decoder.weight, model.decoder.bias,
                  model.value_head.weight, model.value_head.bias]
        grads = [self.dw_enc, db_enc, dw_cat[:n_act], db_cat[:n_act], dw_cat[n_act:n_act + 1], db_cat[n_act:n_act + 1]]
        self.tensors = (_native.AdamTensor * len(params))()
        for k, (p, g) in enumerate(zip(params, grads)):
            st = opt.state[p]
            if len(st) == 0:          # what torch.optim.Adam._init_group creates for fused / capturable parameters
                st['step'] = torch.zeros((), **z)
                st['exp_avg'] = torch.zeros_like(p, memory_format=torch.preserve_format)
                st['exp_avg_sq'] = torch.zeros_like(p, memory_format=torch.preserve_format)
            assert st['step'].is_cuda and st['step'].dtype == torch.float32 and p.is_contiguous() and g.is_contiguous()
            self.tensors[k] = _native.AdamTensor(p.data_ptr(), st['exp_avg'].data_ptr(), st['exp_avg_sq'].data_ptr(),
                                                 st['step'].data_ptr(), g.data_ptr(), p.numel())
        self._keep = (params, grads)
        self._state_ptrs = self._current_state_ptrs()
        self.fused_ws, self.used_fused, self.part = None, False, None
        self.rows = 0
        self.stats = None
        self.world = torch.distributed.get_world_size() if (torch.distributed.is_available() and
                                                            torch.distributed.is_initialized()) else 1
        # multi-GPU: the gradient sum is fused into pb_clip_adam_peer over NVLink peer memory (distributed.PeerComm); the
        # NCCL all-reduce is only the fallback when peer mapping is unavailable (config.peer_allreduce=False, or IPC failed)
        self.peer = None
        self.peer_parts = None
        self.head_pack = None
        if self.world > 1 and bool(getattr(data.config, 'peer_allreduce', True)):
            from pufferlib_b200.distributed import PeerComm
            ok = torch.ones(1, device=dev)
            try:
                self.peer = PeerComm(self.gflat.numel())
            except Exception as e:           # every rank must take the same path: agree on it below
                data.msg = f'peer all-reduce unavailable ({type(e).__name__}: {e}); using NCCL'
                ok.zero_()
            torch.distributed.all_reduce(ok, op=torch.distributed.ReduceOp.MIN)
            if float(ok.item()) == 0.0:
                if self.peer is not None:
                    self.peer.close()
                self.peer = None

    def _current_state_ptrs(self):
        out = []
        for p in self._keep[0]:
            st = self.opt.state.get(p, {})
            out.append(tuple(st[k].data_ptr() if k in st else 0 for k in ('exp_avg', 'exp_avg_sq', 'step')) + (p.data_ptr(),))
        return out

    def stale(self):
        """True when the optimizer's state tensors are no longer the ones whose addresses pb_clip_adam was given
        (optimizer.load_state_dict() replaces them): the caller rebuilds the update object."""
        return self._current_state_ptrs() != self._state_ptrs

    def _buffers(self, m, n_stats):
        if self.rows != m:
            z = dict(dtype=torch.float32, device=self.gflat.device)
            self.hidden, self.dpre = torch.empty(m, self.hid, **z), torch.empty(m, self.hid, **z)
            self.out, self.dout = torch.empty(m, 8, **z), torch.empty(m, 8, **z)
            self.ws = torch.empty(_native.lib().pb_mlp_tail_workspace_bytes(m, self.hid), dtype=torch.uint8,
                                  device=self.gflat.device)
            self.part = None
            self.rows = m
        if self.stats is None or self.stats.shape[0] != n_stats:
            self.stats = torch.zeros(n_stats, 8, dtype=torch.float64, device=self.gflat.device)

    def pack_heads(self):
        m = self.model
        _native.check(_native.lib().pb_pack_heads(
            _native.ptr(m.decoder.weight), _native.ptr(m.decoder.bias), _native.ptr(m.value_head.weight),
            _native.ptr(m.value_head.bias), self.n_act, self.hid, _native.ptr(self.w_cat), _native.ptr(self.b_cat),
            None, None, 0, _native.stream_ptr()))

    def _fused_ok(self, x, config):
        """pb_mlp_update_fused (csrc/mlp_update.cu): fp32 observations with exactly 128 features in equally spaced row
        slabs -- the C2 / C5 workload.  Everything else takes the kernel chain below."""
        return (bool(getattr(config, 'fused_update', FUSED_UPDATE_DEFAULT)) and x.dtype == torch.float32 and x.shape[2] == 128
                and self.hid == 128 and x.stride(2) == 1 and x.stride(1) % 4 == 0 and x.data_ptr() % 16 == 0
                and (x.shape[0] == 1 or (x.stride(0) % x.stride(1) == 0 and x.stride(0) >= x.shape[1] * x.stride(1))))

    @torch.no_grad()
    def forward_backward(self, k, n_stats, obs, slab_form, atn, log_probs, adv, ret, val, config, row_slab_stride=None,
                         adv_norm=None):
        """obs: slab view [G, R, *obs] (slab_form) or [M, *obs]; the rest [M] in slab-major order -- or, with
        row_slab_stride (fused kernel only), arrival-order tensors whose slab s starts at element s * row_slab_stride;
        adv_norm: device (mean, 1/(std+1e-8)) applied to `adv` inside the kernel; ret None: adv + val.  Statistics of this
        minibatch go to row k of self.stats."""
        x = obs if slab_form else obs.reshape(1, atn.numel(), -1)
        x = x.flatten(2)
        assert row_slab_stride is None or self._fused_ok(x, config)
        if self._fused_ok(x, config):
            # ONE tcgen05 kernel: x read once, hidden / dPre stay on the SM, gradients land in self.gflat
            g_, r_, _ = x.shape
            lib = _native.lib()
            if self.stats is None or self.stats.shape[0] != n_stats:
                self.stats = torch.zeros(n_stats, 8, dtype=torch.float64, device=self.gflat.device)
            if self.fused_ws is None:
                self.fused_ws = torch.empty(lib.pb_mlp_update_workspace_bytes(), dtype=torch.uint8, device=self.gflat.device)
            self.mb_rows = g_ * r_
            m_ = self.model
            _native.check(lib.pb_mlp_update_fused(
                _native.ptr(x), x.stride(1), r_, (x.stride(0) // x.stride(1)) if g_ > 1 else r_, g_,
                _native.ptr(m_.encoder.weight), _native.ptr(m_.encoder.bias), _native.ptr(self.w_cat), _native.ptr(self.b_cat),
                _native.ptr(atn.reshape(-1)), _native.ptr(log_probs.reshape(-1)), _native.ptr(adv.reshape(-1)),
                _native.ptr(ret.reshape(-1)) if ret is not None else None, _native.ptr(val.reshape(-1)),
                _native.ptr(adv_norm) if adv_norm is not None else None, r_ if row_slab_stride is None else int(row_slab_stride),
                self.n_act, C.c_float(config.clip_coef),
                int(bool(config.clip_vloss)), C.c_float(config.vf_clip_coef), C.c_float(config.vf_coef),
                C.c_float(config.ent_coef), _native.ptr(self.gflat), C.c_void_p(self.stats.data_ptr() + 64 * k),
                _native.ptr(self.fused_ws), self.fused_ws.numel(), None, None, None, None, _native.stream_ptr()))
            self.used_fused = True
            return
        x = x.float()
        g_, r_, f_ = x.shape
        m, hid = g_ * r_, self.hid
        self._buffers(m, n_stats)
        self.mb_rows = m
        model, lib, s = self.model, _native.lib(), _native.stream_ptr()
        w_enc, b_enc = model.encoder.weight, model.encoder.bias
        for g in range(g_):
            torch._addmm_activation(b_enc, x[g], w_enc.t(), use_gelu=False, out=self.hidden[g * r_:(g + 1) * r_])
        torch.addmm(self.b_cat, self.hidden, self.w_cat.t(), out=self.out)
        cp = C.c_void_p
        o_ptr, d_ptr, n_act = self.out.data_ptr(), self.dout.data_ptr(), self.n_act
        _native.check(lib.pb_ppo_loss(
            cp(o_ptr), 8, cp(o_ptr + 4 * n_act), 8, _native.ptr(atn.reshape(-1)), _native.ptr(log_probs.reshape(-1)),
            _native.ptr(adv.reshape(-1)), _native.ptr(ret.reshape(-1)), _native.ptr(val.reshape(-1)), m, n_act,
            C.c_float(config.clip_coef), int(bool(config.clip_vloss)), C.c_float(config.vf_clip_coef),
            C.c_float(config.vf_coef), C.c_float(config.ent_coef), cp(d_ptr), 8, cp(d_ptr + 4 * n_act), 8,
            cp(self.stats.data_ptr() + 64 * k), s))
        _native.check(lib.pb_mlp_tail_backward(_native.ptr(self.dout), 8, _native.ptr(self.w_cat),
                                               _native.ptr(self.hidden), m, hid, _native.ptr(self.dpre),
                                               _native.ptr(self.tail), _native.ptr(self.ws), self.ws.numel(), s))
        sp = max(1, 64 // g_)
        while r_ % sp:
            sp //= 2
        if self.part is None or self.part.shape != (g_ * sp, hid, f_):
            self.part = torch.empty(g_ * sp, hid, f_, dtype=torch.float32, device=x.device)
        for g in range(g_):
            torch.bmm(self.dpre[g * r_:(g + 1) * r_].view(sp, r_ // sp, hid).transpose(1, 2),
                      x[g].view(sp, r_ // sp, f_), out=self.part[g * sp:(g + 1) * sp])
        torch.sum(self.part, 0, out=self.dw_enc)

    def all_reduce(self):
        if self.world > 1 and self.peer is None:
            torch.distributed.all_reduce(self.gflat)

    @torch.no_grad()
    def optimizer_step(self, config):
        g = self.opt.param_groups[0]
        lr = g['lr']
        lr_dev = _native.ptr(lr) if isinstance(lr, torch.Tensor) else None
        b1, b2 = g['betas']
        lib = _native.lib()
        hyper = (C.c_float(float(config.max_grad_norm)), C.c_float(1.0 / self.world),
                 C.c_float(0.0 if lr_dev is not None else float(lr)), lr_dev, C.c_float(b1), C.c_float(b2), C.c_float(g['eps']), None)
        if self.used_fused and (self.world == 1 or self.peer is not None):
            # the fused update's reduce step left the gradient's sum of squares as partial sums: multi-CTA clip + Adam without a
            # norm pass; several ranks: sliced peer all-reduce first, which leaves its own partial sums of squares
            m = self.model
            if self.head_pack is None:      # the head matrix is rebuilt by the last CTA of the optimizer kernel
                self.head_pack = _native.HeadPack(m.decoder.weight.data_ptr(), m.decoder.bias.data_ptr(), m.value_head.weight.data_ptr(),
                                                  m.value_head.bias.data_ptr(), self.w_cat.data_ptr(), self.b_cat.data_ptr(),
                                                  self.n_act, self.hid)
            if self.peer is not None:       # exchange + clip + Adam: one kernel
                if self.peer_parts is None:
                    self.peer_parts = torch.zeros(lib.pb_peer_slices(), dtype=torch.float64, device=self.gflat.device)
                _native.check(lib.pb_clip_adam_peer_parts(
                    self.tensors, len(self.tensors), *hyper, C.byref(self.peer.struct), _native.ptr(self.gflat), self.gflat.numel(),
                    _native.ptr(self.peer_parts), C.byref(self.head_pack), _native.stream_ptr()))
            else:
                parts = C.c_void_p(self.fused_ws.data_ptr() + lib.pb_mlp_update_sumsq_offset())
                _native.check(lib.pb_clip_adam_parts(self.tensors, len(self.tensors), *hyper, parts, lib.pb_mlp_update_sumsq_parts(),
                                                     None, C.byref(self.head_pack), _native.stream_ptr()))
            return
        else:
            _native.check(lib.pb_clip_adam_peer(
                self.tensors, len(self.tensors), *hyper, C.byref(self.peer.struct) if self.peer is not None else None,
                _native.ptr(self.gflat), self.gflat.numel(), _native.stream_ptr()))
        self.pack_heads()

    def loss_means(self, n_mb):
        """[policy, value, entropy, old_kl, kl, clipfrac]: per-minibatch means / n_mb, summed over all minibatches
        (the accumulation of clean_pufferl.py:249-254)."""
        tot = self.stats.sum(0)[:6] / (self.mb_rows * n_mb)
        tot[1] *= 0.5
        return tot.float()


class Experience:
    """Flat tensor storage in arrival order, on the device (reference: clean_pufferl.py:380-482)."""

    def __init__(self, batch_size, bptt_horizon, minibatch_size, obs_shape, obs_dtype, atn_shape,
                 cpu_offload=False, device='cuda', lstm=None, lstm_total_agents=0):
        if minibatch_size is None:
            minibatch_size = batch_size
        if cpu_offload:
            raise NotImplementedError('cpu_offload: the B200 rollout is device-resident by design')
        atn_shape = tuple(atn_shape)
        if len(atn_shape) > 1:
            raise NotImplementedError('only Discrete and MultiDiscrete action spaces are on the device path')
        obs_dtype = numpy_to_torch_dtype_dict[np.dtype(obs_dtype)]
        dev = torch.device(device)
        if dev.type != 'cuda':
            raise RuntimeError('pufferlib_b200.Experience needs a CUDA device (no CPU fallback)')
        self.device = dev
        z = dict(device=dev)
        self.obs = torch.zeros(batch_size, *obs_shape, dtype=obs_dtype, **z)
        self.actions = torch.zeros(batch_size, *atn_shape, dtype=torch.int64, **z)     # clean_pufferl.py:392
        self.atn_shape = atn_shape
        self.atn_row_bytes = 8 * int(np.prod(atn_shape, dtype=np.int64))
        self.logprobs = torch.zeros(batch_size, **z)
        self.rewards = torch.zeros(batch_size, **z)
        self.dones = torch.zeros(batch_size, **z)
        self.truncateds = torch.zeros(batch_size, **z)   # never written, as in the reference
        self.values = torch.zeros(batch_size, **z)
        self.lstm_h = self.lstm_c = None
        if lstm is not None:     # clean_pufferl.py:407-412
            assert lstm_total_agents > 0
            shape = (lstm.num_layers, lstm_total_agents, lstm.hidden_size)
            self.lstm_h = torch.zeros(shape, **z)
            self.lstm_c = torch.zeros(shape, **z)

        num_minibatches = batch_size / minibatch_size
        self.num_minibatches = int(num_minibatches)
        if self.num_minibatches != num_minibatches:
            raise ValueError('batch_size must be divisible by minibatch_size')
        minibatch_rows = minibatch_size / bptt_horizon
        self.minibatch_rows = int(minibatch_rows)
        if self.minibatch_rows != minibatch_rows:
            raise ValueError('minibatch_size must be divisible by bptt_horizon')

        self.batch_size = batch_size
        self.bptt_horizon = bptt_horizon
        self.minibatch_size = minibatch_size
        self.obs_shape = tuple(obs_shape)
        self.obs_row_bytes = int(np.prod(obs_shape, dtype=np.int64)) * self.obs.element_size()
        self.ptr = 0
        self.step = 0
        self.num_envs = None      # agents per step, fixed by the first store()
        # train-side tensors, allocated once and reused every epoch
        nm, mb = self.num_minibatches, self.minibatch_size
        self.advantages = torch.zeros(batch_size, **z)        # sorted order (== advantages_np)
        self.returns_sorted = torch.zeros(batch_size, **z)
        self.returns = torch.zeros(batch_size, **z)           # returns_np of clean_pufferl.py:476
        shape3 = (nm, self.minibatch_rows, bptt_horizon)
        self._b_obs = None        # [nm, minibatch_rows, bptt, *obs]: allocated by the first flatten_batch() that gathers
        self._slabs = None        # zero-copy minibatch form (flatten_batch_slabs)
        self.b_actions = torch.zeros(*shape3, *atn_shape, dtype=torch.int64, **z)
        self.b_logprobs = torch.zeros(shape3, **z)
        self.b_dones = torch.zeros(shape3, **z)
        self.b_values = torch.zeros(nm, mb, **z)
        self.b_advantages = torch.zeros(nm, mb, **z)
        self.b_returns = torch.zeros(nm, mb, **z)
        self.b_advantages_normalized = torch.zeros(nm, mb, **z)
        lib = _native.lib()
        self._advnorm_ws = torch.zeros(max(16, lib.pb_adv_norm_workspace_bytes(nm, mb)), dtype=torch.uint8, **z)
        self._gae_ws = None
        self.advantages_tm = None     # arrival-order advantages (pb_gae_tm) for the in-place (direct slab) update
        self.adv_norm = None          # [nm, 2]: (mean, 1 / (std + 1e-8)) per minibatch

    @property
    def b_obs(self):
        if self._b_obs is None:
            self._b_obs = torch.zeros(self.num_minibatches, self.minibatch_rows, self.bptt_horizon, *self.obs_shape,
                                      dtype=self.obs.dtype, device=self.device)
        return self._b_obs

    @property
    def full(self):
        return self.ptr >= self.batch_size

    # numpy views of the reference become explicit device->host copies here
    @property
    def values_np(self):
        return self.values.cpu().numpy()

    @property
    def returns_np(self):
        return self.returns.cpu().numpy()

    @property
    def rewards_np(self):
        return self.rewards.cpu().numpy()

    @property
    def dones_np(self):
        return self.dones.cpu().numpy()

    @property
    def actions_np(self):
        return self.actions.cpu().numpy()

    @property
    def logprobs_np(self):
        return self.logprobs.cpu().numpy()

    def store(self, obs, value, action, logprob, reward, done, env_id, mask):
        """clean_pufferl.py:436-450 for an all-True mask with env_id == arange(N) (what the B200 backend
        produces): rows ptr:ptr+N.  Tensors already living in their rollout row (bound vecenv) are not copied."""
        n = value.shape[0]
        if self.num_envs is None:            # total agents (create() sets it; pool mode stores batch_size-row chunks)
            self.num_envs = n
        # the arithmetic sort needs arange-ordered, fully valid blocks (what the B200 backends produce); anything else
        # would be trained on in the wrong order, so refuse it (the reference filters by mask and sorts by (env_id, step))
        if env_id is not None and (len(env_id) != n or int(env_id[0]) != self.ptr % self.num_envs
                                   or int(env_id[-1]) - int(env_id[0]) != n - 1):
            raise APIUsageError('store(): env_id must be the contiguous block of agents expected at this rollout position')
        if isinstance(mask, np.ndarray) and not mask.all():
            raise APIUsageError('store(): padded agents (mask False) are not supported on the device path')
        if self.batch_size % n != 0 or self.num_envs % n != 0:
            raise APIUsageError('batch_size / num_envs must be multiples of the agents per store()')
        ptr, end = self.ptr, self.ptr + n
        if end > self.batch_size:
            raise APIUsageError('store(): rollout buffer is full')
        lib, s = _native.lib(), _native.stream_ptr()
        obs_row = self.obs.data_ptr() + ptr * self.obs_row_bytes
        if obs.data_ptr() != obs_row:
            obs = obs.to(self.device)
            _native.check(lib.pb_copy_rows(_native.ptr(obs.contiguous()), self.obs_row_bytes, C.c_void_p(obs_row),
                                           self.obs_row_bytes, self.obs_row_bytes, n, s))
        if reward.data_ptr() != self.rewards.data_ptr() + ptr * 4:
            self.rewards[ptr:end] = torch.as_tensor(reward).to(self.device, torch.float32)
            self.dones[ptr:end] = torch.as_tensor(done).to(self.device, torch.float32)
        if isinstance(value, torch.Tensor) and value.data_ptr() == self.values.data_ptr() + ptr * 4 and \
                isinstance(action, torch.Tensor) and action.data_ptr() == self.actions.data_ptr() + ptr * self.atn_row_bytes and \
                logprob.data_ptr() == self.logprobs.data_ptr() + ptr * 4:
            self.ptr = end          # the fused sampling epilogue already wrote value / logprob / action in place
            self.step += 1
            return
        value = value.reshape(-1).to(self.device, torch.float32).contiguous()
        logprob = logprob.reshape(-1).to(self.device, torch.float32).contiguous()
        action = torch.as_tensor(action).reshape(n, *self.atn_shape).to(self.device, torch.int64).contiguous()
        multi = len(self.atn_shape) > 0
        _native.check(lib.pb_rollout_store(
            _native.ptr(value), _native.ptr(logprob), None if multi else _native.ptr(action),
            C.c_void_p(self.values.data_ptr() + ptr * 4), C.c_void_p(self.logprobs.data_ptr() + ptr * 4),
            None if multi else C.c_void_p(self.actions.data_ptr() + ptr * 8), n, s))
        if multi:               # [n, k] action rows: one row copy of 8k bytes each
            _native.check(lib.pb_copy_rows(_native.ptr(action), self.atn_row_bytes,
                                           C.c_void_p(self.actions.data_ptr() + ptr * self.atn_row_bytes),
                                           self.atn_row_bytes, self.atn_row_bytes, n, s))
        self.ptr = end
        self.step += 1

    def rows(self):
        """(values, logprobs, actions) views of the rollout rows the next store() will fill."""
        n = self.num_envs
        lo, hi = self.ptr, self.ptr + n
        return self.values[lo:hi], self.logprobs[lo:hi], self.actions[lo:hi]

    def sort_training_data(self):
        """clean_pufferl.py:452-464.  The permutation is arithmetic on the device; the index array is only
        materialised (on the host) for callers that ask for the reference's return value."""
        n = self.num_envs
        h = self.batch_size // n
        self.horizon = h
        self.ptr = 0
        self.step = 0
        return _LazyIdxs(n, h)

    def compute_gae(self, gamma, gae_lambda, time_major=False):
        """c_gae.compute_gae on the sorted batch (clean_pufferl.py:164-169) -> self.advantages (sorted order).
        time_major: ALSO self.advantages_tm in arrival order (row t*N + e) and no sorted returns (pb_gae_tm)."""
        n, h = self.num_envs, self.horizon
        lib = _native.lib()
        need = lib.pb_gae_workspace_bytes(n, h)
        if self._gae_ws is None or self._gae_ws.numel() < need:
            self._gae_ws = torch.zeros(need, dtype=torch.uint8, device=self.device)
        if time_major:
            if self.advantages_tm is None:
                self.advantages_tm = torch.zeros(self.batch_size, device=self.device)
            _native.check(lib.pb_gae_tm(_native.ptr(self.rewards), _native.ptr(self.values), _native.ptr(self.dones),
                                        _native.ptr(self.advantages), None, _native.ptr(self.advantages_tm), n, h,
                                        C.c_float(gamma), C.c_float(gae_lambda), _native.ptr(self._gae_ws),
                                        self._gae_ws.numel(), _native.stream_ptr()))
            return self.advantages
        _native.check(lib.pb_gae(_native.ptr(self.rewards), _native.ptr(self.values), _native.ptr(self.dones),
                                 _native.ptr(self.advantages), _native.ptr(self.returns_sorted), n, h,
                                 C.c_float(gamma), C.c_float(gae_lambda), _native.ptr(self._gae_ws),
                                 self._gae_ws.numel(), _native.stream_ptr()))
        return self.advantages

    def direct_slabs_ok(self, manual, config):
        """Can the update read the rollout tensors in place (zero-copy observations AND zero-copy per-row tensors)?  Needs
        the slab layout, the GAE tile kernel's time-major output and the fused update kernel for these observations."""
        n, h, nm, bptt = self.num_envs, self.horizon, self.num_minibatches, self.bptt_horizon
        layout = slab_layout(n, h, nm, bptt)
        if layout is None or not _native.lib().pb_gae_time_major_supported(n, h):
            return False
        g_, r_ = layout
        x0 = self.obs.view(g_, nm, r_, *self.obs_shape)[:, 0].flatten(2)
        return manual._fused_ok(x0, config)

    def prepare_direct_slabs(self, norm_adv):
        """After compute_gae(time_major=True): the returns of clean_pufferl.py:476 (for the explained variance) and the
        per-minibatch advantage-normalisation constants of :211-213, straight from the arrival-order advantages."""
        n, h, nm, bptt = self.num_envs, self.horizon, self.num_minibatches, self.bptt_horizon
        g_, r_ = slab_layout(n, h, nm, bptt)
        torch.add(self.advantages, self.values, out=self.returns)       # sorted + arrival, same flat index (the reference's)
        if self._slabs is None:
            self._slabs = pufferlib_b200.namespace()
        self._slabs.shape = (g_, r_)
        if norm_adv:
            if self.adv_norm is None:
                self.adv_norm = torch.zeros(nm, 2, device=self.device)
            _native.check(_native.lib().pb_adv_stats_slabs(
                _native.ptr(self.advantages_tm), r_, g_, nm, _native.ptr(self.adv_norm), _native.ptr(self._advnorm_ws),
                self._advnorm_ws.numel(), _native.stream_ptr()))

    def direct_minibatch(self, mb, norm_adv):
        """Minibatch mb as views of the rollout tensors: slab s of the minibatch = rows (s*nm + mb)*R .. +R."""
        g_, r_ = self._slabs.shape
        lo = mb * r_
        return pufferlib_b200.namespace(
            obs=self.slab_obs(mb), actions=self.actions[lo:], logprobs=self.logprobs[lo:], old_values=self.values[lo:],
            advantages=self.advantages_tm[lo:], row_slab_stride=self.num_minibatches * r_,
            adv_norm=self.adv_norm[mb] if norm_adv else None)

    def flatten_batch(self, advantages=None):
        """clean_pufferl.py:466-482 (advantages: sorted-order device tensor, default self.advantages)."""
        adv = self.advantages if advantages is None else advantages
        n, h = self.num_envs, self.horizon
        lib, s = _native.lib(), _native.stream_ptr()
        multi = len(self.atn_shape) > 0
        _native.check(lib.pb_flatten_batch(
            None if multi else _native.ptr(self.actions), _native.ptr(self.logprobs), _native.ptr(self.dones),
            _native.ptr(self.values), _native.ptr(adv), None if multi else _native.ptr(self.b_actions),
            _native.ptr(self.b_logprobs), _native.ptr(self.b_dones),
            _native.ptr(self.b_values), _native.ptr(self.b_advantages), _native.ptr(self.b_returns),
            _native.ptr(self.returns), n, h, self.num_minibatches, self.minibatch_rows, self.bptt_horizon, s))
        if multi:               # b_actions [nm, rows, bptt, k] = actions[b_idxs]: the observation gather on 8k-byte rows
            _native.check(lib.pb_minibatch_gather(
                _native.ptr(self.actions), _native.ptr(self.b_actions), self.atn_row_bytes, n, h, self.num_minibatches,
                self.minibatch_rows, self.bptt_horizon, 0, self.num_minibatches, s))
        _native.check(lib.pb_minibatch_gather(
            _native.ptr(self.obs), _native.ptr(self.b_obs), self.obs_row_bytes, n, h, self.num_minibatches,
            self.minibatch_rows, self.bptt_horizon, 0, self.num_minibatches, s))

    def flatten_batch_slabs(self, advantages=None):
        """flatten_batch without the observation gather, for policies whose loss does not depend on the row order
        inside a minibatch (no LSTM).  Minibatch mb of clean_pufferl.py:466-482 holds the bptt segments s = r*nm + mb;
        when the segments per env S = H/bptt are a multiple of nm these are, for EVERY env, the time windows
        k = mb, mb+nm, ... -- in the time-major rollout buffer that is G = S/nm contiguous slabs of bptt*N rows.  So
        the minibatch observations are a strided view [G, bptt*N, *obs] of self.obs (slab_obs) and only the small
        per-row tensors are re-ordered (slab-major: s_x[mb][g][j*N + e] = x[((g*nm + mb)*bptt + j)*N + e]).  Same
        row SETS as the reference, so the minibatch means, the advantage normalisation and the gradients agree up to
        summation order.  Returns False (nothing done) when the shape condition does not hold."""
        adv = self.advantages if advantages is None else advantages
        n, h, nm, bptt = self.num_envs, self.horizon, self.num_minibatches, self.bptt_horizon
        layout = slab_layout(n, h, nm, bptt)
        if layout is None:
            return False
        g_, r_ = layout
        if self._slabs is None or getattr(self._slabs, 'actions', None) is None:
            z = dict(device=self.device)
            mb = self.minibatch_size
            self._slabs = pufferlib_b200.namespace(
                actions=torch.zeros(nm, mb, *self.atn_shape, dtype=torch.int64, **z), logprobs=torch.zeros(nm, mb, **z),
                values=torch.zeros(nm, mb, **z), advantages=torch.zeros(nm, mb, **z), returns=torch.zeros(nm, mb, **z),
                advantages_normalized=torch.zeros(nm, mb, **z))
        sl = self._slabs
        for dst, src in ((sl.actions, self.actions), (sl.logprobs, self.logprobs), (sl.values, self.values)):
            tail = tuple(src.shape[1:])          # (k,) for MultiDiscrete actions
            dst.view(nm, g_, r_, *tail).copy_(src.view(g_, nm, r_, *tail).transpose(0, 1))
        sl.advantages.view(nm, g_, bptt, n).copy_(adv.view(n, g_, nm, bptt).permute(2, 1, 3, 0))   # sorted -> slab-major
        torch.add(sl.advantages, sl.values, out=sl.returns)
        torch.add(adv, self.values, out=self.returns)            # returns_np of clean_pufferl.py:476 (sorted + arrival)
        sl.shape = (g_, r_)
        return True

    def slab_obs(self, mb):
        """Observations of minibatch mb as a zero-copy view [G, bptt*N, *obs] of the rollout buffer."""
        g_, r_ = self._slabs.shape
        return self.obs.view(g_, self.num_minibatches, r_, *self.obs_shape)[:, mb]

    def normalize_advantages(self, slabs=False):
        """clean_pufferl.py:211-213 for every minibatch at once -> self.b_advantages_normalized."""
        src, dst = (self._slabs.advantages, self._slabs.advantages_normalized) if slabs else \
            (self.b_advantages, self.b_advantages_normalized)
        _native.check(_native.lib().pb_adv_norm(
            _native.ptr(src), _native.ptr(dst), self.num_minibatches,
            self.minibatch_size, _native.ptr(self._advnorm_ws), self._advnorm_ws.numel(), _native.stream_ptr()))
        return dst


class _LazyIdxs:
    """Return value of sort_training_data: the (env_id, step) argsort, computed only if someone looks."""

    def __init__(self, n, h):
        self.n, self.h = n, h

    def __array__(self, dtype=None, copy=None):
        e, t = np.divmod(np.arange(self.n * self.h), self.h)
        idxs = t * self.n + e
        return idxs if dtype is None else idxs.astype(dtype)

    def __len__(self):
        return self.n * self.h


def _set_lr(optimizer, lr):
    """The learning rate is a device tensor when the optimizer is capturable (graph replays read it in place)."""
    cur = optimizer.param_groups[0]['lr']
    if isinstance(cur, torch.Tensor):
        cur.fill_(lr)
    else:
        optimizer.param_groups[0]['lr'] = lr


def create(config, vecenv, policy, optimizer=None, wandb=None):
    seed_everything(config.seed, config.torch_deterministic)
    profile = Profile()
    losses = make_losses()
    n_params = sum(p.numel() for p in policy.parameters() if p.requires_grad)
    msg = f'Model Size: {n_params} parameters'

    vecenv.async_reset(config.seed)
    obs_shape = vecenv.single_observation_space.shape
    obs_dtype = vecenv.single_observation_space.dtype
    atn_shape = vecenv.single_action_space.shape
    total_agents = vecenv.num_agents

    lstm = policy.lstm if hasattr(policy, 'lstm') else None
    experience = Experience(config.batch_size, config.bptt_horizon, config.minibatch_size, obs_shape, obs_dtype,
                            atn_shape, config.cpu_offload, config.device, lstm, total_agents)
    experience.num_envs = total_agents      # rows arrive in arrival order t*N + e (also in pool mode: (t, group) blocks)
    if hasattr(vecenv, 'bind_rollout'):
        vecenv.bind_rollout(experience)     # env-step kernels write rollout rows directly (host_buffers mode too: the
                                            # host arrays are filled FROM the rows, the policy reads the rows)

    uncompiled_policy = policy
    if getattr(config, 'compile', False):
        raise NotImplementedError('torch.compile is not used on the B200 path (no Triton); set compile=False')

    own_optimizer = optimizer is None
    if optimizer is None:
        # same update rule as the reference's Adam (clean_pufferl.py:54-55); fused=True applies it in one kernel
        graphed = any(bool(getattr(config, k, False)) for k in ('cuda_graph', 'cuda_graph_train', 'cuda_graph_rollout'))
        lr = torch.tensor(float(config.learning_rate), device=config.device) if graphed else config.learning_rate
        optimizer = torch.optim.Adam(policy.parameters(), lr=lr, eps=1e-5, fused=True, capturable=graphed)

    model = getattr(policy, 'policy', None)
    if hasattr(model, 'invalidate_cache'):      # cached head matrix of models.Default: stale after every optimizer step
        optimizer.register_step_post_hook(lambda *a, **k: model.invalidate_cache())

    grad_bucket = None
    if torch.distributed.is_available() and torch.distributed.is_initialized() and \
            torch.distributed.get_world_size() > 1:
        from pufferlib_b200.distributed import GradBucket
        grad_bucket = GradBucket(policy)

    return pufferlib_b200.namespace(
        config=config, vecenv=vecenv, policy=policy, uncompiled_policy=uncompiled_policy, optimizer=optimizer,
        experience=experience, profile=profile, losses=losses, wandb=wandb, global_step=0, epoch=0, stats={},
        msg=msg, last_log_time=0, utilization=None, grad_bucket=grad_bucket,
        io=pufferlib_b200.namespace(h2d=0, d2h=0), graph_state=0, rollout_graph=None, graph_steps=0,
        graph_launches=0, graph_replays=0, train_graph_state=0, train_graph=None, train_result=None, train_graph_launches=0, train_graph_replays=0, train_segments=None, train_acc=None, own_optimizer=own_optimizer, manual_update=None,
        fused_rows=bool(getattr(policy, 'fused_sample', False)) and hasattr(vecenv, 'bind_rollout'),
        # one-kernel PPO loss (pb_ppo_loss, or pb_ppo_loss_multi for MultiDiscrete heads): needs a wrapper exposing
        # .policy(obs) -> (logits, value)
        fused_loss=bool(getattr(config, 'fused_loss', True)) and hasattr(policy, 'policy')
        and not hasattr(policy, 'lstm') and len(tuple(vecenv.single_action_space.shape)) <= 1,
        action_nvec=([int(x) for x in vecenv.single_action_space.nvec]
                     if len(tuple(vecenv.single_action_space.shape)) == 1 else None),
    )


def _rollout_loop(data, infos):
    """The body of evaluate (clean_pufferl.py:84-124): recv -> policy -> store -> send until the buffer is full.
    On the device path it contains no host synchronisation, so it can be captured in a CUDA graph."""
    config, profile, experience = data.config, data.profile, data.experience
    policy, vecenv = data.policy, data.vecenv
    on_device = not getattr(vecenv, 'host_buffers', False)
    io = data.io
    # the whole horizon as ONE persistent kernel (env state in registers, tcgen05 policy, csrc/env_breakout.cu) where it applies
    if bool(getattr(config, 'fused_rollout', FUSED_ROLLOUT_DEFAULT)) and hasattr(vecenv, 'fused_rollout_ok') and \
            data.fused_rows and vecenv.fused_rollout_ok(experience, policy):
        with profile.env:
            vecenv.fused_rollout(experience, policy)
        data.global_step += experience.batch_size
        experience.ptr = experience.batch_size
        experience.step = experience.batch_size // experience.num_envs
        data.fused_rollouts = getattr(data, 'fused_rollouts', 0) + 1
        return
    device_feed = not on_device and hasattr(vecenv, 'recv_device')
    while not experience.full:
        with profile.env:
            # host_buffers mode: the step as DEVICE tensors; its copy into the pinned host arrays (what recv() returns to
            # a host-side caller) runs on the copy stream beside the policy forward and is awaited once, before send()
            o, r, d, t, info, env_id, mask = vecenv.recv_device() if device_feed else vecenv.recv()

        with profile.eval_misc:
            # sum(mask) of clean_pufferl.py:90; count_nonzero instead of the Python-level sum over a numpy array, which
            # costs 1 ms per env step at N = 16384
            data.global_step += len(env_id) if (on_device or device_feed) else int(np.count_nonzero(mask))
            if on_device or device_feed:
                o_device = o      # the device copy of the observations already exists: no H2D (clean_pufferl.py:92-95)
            else:   # a host-only vecenv: the reference's H2D of the observation batch
                o_device = vecenv.pinned(o).to(config.device, non_blocking=True)
                r = vecenv.pinned(r).to(config.device, non_blocking=True)
                d = vecenv.pinned(d).to(config.device, non_blocking=True)
                io.h2d += o.nbytes + r.nbytes + d.nbytes

        with profile.eval_forward, torch.no_grad():
            if experience.lstm_h is not None:
                # clean_pufferl.py:100-105: h = lstm_h[:, env_id] -> policy -> lstm_h[:, env_id] = h.  env_id is a
                # contiguous range here (every env, or one pool group): slices instead of index gathers
                lo, hi = int(env_id[0]), int(env_id[0]) + len(env_id)
                if lo == 0 and hi == experience.lstm_h.shape[1]:
                    h_in, c_in = experience.lstm_h, experience.lstm_c
                else:
                    h_in, c_in = experience.lstm_h[:, lo:hi].contiguous(), experience.lstm_c[:, lo:hi].contiguous()
                actions, logprob, _, value, (h, c) = policy(o_device, (h_in, c_in))
                experience.lstm_h[:, lo:hi].copy_(h)
                experience.lstm_c[:, lo:hi].copy_(c)
            elif data.fused_rows and experience.num_envs is not None:
                actions, logprob, _, value = policy(o_device, out=experience.rows())
            else:
                actions, logprob, _, value = policy(o_device)

        with profile.eval_misc:
            value = value.flatten()
            experience.store(o_device, value, actions, logprob, r, d, env_id, mask)
            if device_feed:   # the reference's D2H of the actions (clean_pufferl.py:114) + the ONE host wait of this env step
                a_host = vecenv.actions_to_host(actions)
                if getattr(vecenv, 'exact_infos', False) or vecenv._rollout is None:
                    info = vecenv.host_sync()[4]          # per-step info dicts need the terminal flags on the host
                elif torch.cuda.is_current_stream_capturing():
                    # captured rollout (host_graph): the action round trip device -> pinned host array -> device is stream-ordered
                    # inside the graph (store kernel, then the H2D copy node of send()); the host is not in the loop
                    info = []
                else:
                    # nothing on the host side reads this step's observations: wait for the actions only and let the big
                    # copies stream behind (each reads its own rollout row); they are awaited when the rollout ends
                    vecenv.host_sync(actions_only=True)
                    info = []
            for i in info:
                for k, v in i.items():
                    infos[k].append(v)

        with profile.env:
            if on_device:
                vecenv.send(actions)
            elif device_feed:
                vecenv.send(a_host)
            else:
                a_host = actions.cpu().numpy()
                io.d2h += a_host.nbytes
                vecenv.send(a_host)
    if device_feed and torch.cuda.is_current_stream_capturing():
        vecenv.join_copies()     # the copy stream rejoins the captured stream: the graph ends when every host copy has landed
    elif device_feed and not bool(getattr(config, 'host_copy_defer', True)):
        vecenv.host_sync()       # every device->host copy of the rollout has landed
    # (default: the observation blocks keep streaming to the pinned host arrays while train() runs -- it only reads the
    #  rollout tensors; the next rollout's first write waits for them on the device, and any host-side reader (recv(),
    #  host_sync(), close()) waits for them as before)
    if hasattr(vecenv, 'join'):
        vecenv.join()            # pool mode: side-stream env steps rejoin the caller's stream (and any graph capture)


def _invalidate_policy_cache(data):
    model = getattr(data.policy, 'policy', None)
    if hasattr(model, 'invalidate_cache'):
        model.invalidate_cache()


def evaluate(data):
    """Collect one rollout.  With ``config.cuda_graph`` (device path only) the whole H-step loop -- env-step
    kernels, policy forward, sampling, rollout stores -- is captured once and replayed as ONE graph launch; the
    first call runs eagerly (warm-up and allocations), the second captures."""
    config, profile, experience = data.config, data.profile, data.experience
    infos = defaultdict(list)
    vecenv = data.vecenv
    on_device = not getattr(vecenv, 'host_buffers', False)
    _invalidate_policy_cache(data)          # parameters may have changed since the last rollout
    # host_buffers mode: the loop is capturable when nothing on the host reads a step while it runs (no per-step info dicts,
    # rollout rows bound): every env step still moves its observation block to the pinned host arrays and takes its actions
    # from the pinned host action array, as copy nodes of the graph
    host_graph = not on_device and hasattr(vecenv, 'recv_device') and getattr(vecenv, '_rollout', None) is not None and \
        bool(getattr(config, 'cuda_graph_host_rollout', True))
    use_graph = bool(getattr(config, 'cuda_graph_rollout', getattr(config, 'cuda_graph', False))) and \
        (on_device or host_graph) and not getattr(vecenv, 'exact_infos', False)

    if not use_graph or data.graph_state == 0:
        _rollout_loop(data, infos)
        if use_graph:
            data.graph_state = 1
    else:
        if data.graph_state == 1:
            torch.cuda.synchronize()
            step0, launches0 = data.global_step, _native.lib().pb_launch_count()
            io0 = (data.io.h2d + getattr(vecenv, 'h2d_bytes', 0), data.io.d2h + getattr(vecenv, 'd2h_bytes', 0))
            _invalidate_policy_cache(data)       # anything cached eagerly must be rebuilt inside the capture
            if not on_device:
                vecenv.host_sync()               # outstanding eager copies (their events are not part of the capture)
                vecenv.graph_mode = True
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                _rollout_loop(data, infos)       # python-side state advances exactly as in an eager rollout
            data.rollout_graph = graph
            # host <-> device bytes one replay moves (the byte counters only advance while Python runs the loop)
            data.graph_io = (data.io.h2d + getattr(vecenv, 'h2d_bytes', 0) - io0[0], data.io.d2h + getattr(vecenv, 'd2h_bytes', 0) - io0[1])
            if not on_device:
                vecenv.h2d_bytes -= data.graph_io[0]     # capture executes nothing: the replay below adds them back
                vecenv.d2h_bytes -= data.graph_io[1]
            data.graph_steps = data.global_step - step0
            data.graph_launches = _native.lib().pb_launch_count() - launches0
            data.graph_state = 2
            data.global_step = step0
        with profile.env:
            data.rollout_graph.replay()
        data.global_step += data.graph_steps
        data.graph_replays += 1
        if not on_device:
            vecenv.h2d_bytes += data.graph_io[0]
            vecenv.d2h_bytes += data.graph_io[1]
        experience.ptr = experience.batch_size    # what the captured loop leaves behind
        experience.step = experience.batch_size // experience.num_envs

    with profile.eval_misc:
        data.stats = {}
        if hasattr(vecenv, 'episode_stats') and not getattr(vecenv, 'exact_infos', False):
            means, count = vecenv.episode_stats(clear=True)    # device-side EpisodeStats reduction, one D2H
            data.io.d2h += 256 * 32
            for k, v in means.items():
                infos[k].append(v)
        for k, v in infos.items():
            try:
                data.stats[k] = np.mean(v)
            except Exception:
                continue

    return data.stats, infos


class _SegmentGraphs:
    """Per-segment CUDA graphs for the multi-GPU update loop: each (forward + loss + backward) minibatch segment and the
    (clip + Adam) segment is captured once and replayed; the NCCL all-reduce between them stays an ordinary call."""

    def __init__(self):
        self.graphs = {}
        self.launches = {}
        self.replays = 0

    def run(self, key, fn):
        g = self.graphs.get(key)
        if g is None:
            torch.cuda.synchronize()
            l0 = _native.lib().pb_launch_count()
            g = torch.cuda.CUDAGraph()
            # thread_local: the NCCL watchdog thread may poll events while we capture
            with torch.cuda.graph(g, capture_error_mode='thread_local'):
                fn()
            self.graphs[key] = g
            self.launches[key] = _native.lib().pb_launch_count() - l0
        g.replay()
        self.replays += 1
        self.replayed_launches = getattr(self, 'replayed_launches', 0) + self.launches[key]


def _train_device_part(data, seg=None):
    """Everything of train() that runs on the device without touching the host: GAE, minibatch construction, the
    update_epochs x num_minibatches optimizer steps, the loss statistics.  No synchronisation inside, so the whole
    thing can be captured in ONE CUDA graph (single GPU, see train) or, with ``seg``, as per-segment graphs around
    the gradient all-reduce (multi-GPU)."""
    config, profile, experience = data.config, data.profile, data.experience
    device = experience.device
    _invalidate_policy_cache(data)     # nothing cached by the rollout (eager or captured) may leak into an update graph

    # zero-copy minibatches (Experience.flatten_batch_slabs): order-free loss only, i.e. the fused non-LSTM path
    model = getattr(data.policy, 'policy', None)
    want_slabs = data.fused_loss and experience.lstm_h is None and hasattr(model, 'forward_packed_slabs') and \
        bool(getattr(config, 'zero_copy_minibatches', True))
    manual = None
    if _DefaultMLPUpdate.eligible(data):
        if getattr(data, 'manual_update', None) is None or data.manual_update.stale():
            data.manual_update = _DefaultMLPUpdate(data)
        manual = data.manual_update
    with profile.train_misc:
        experience.sort_training_data()
        # the fused update kernel reads the ARRIVAL-order rollout tensors through slab strides: no minibatch copies at all
        # (GAE writes the advantages in arrival order as well; the advantage normalisation constants are applied on the fly)
        direct = want_slabs and manual is not None and experience.direct_slabs_ok(manual, config)
        if direct:
            experience.compute_gae(config.gamma, config.gae_lambda, time_major=True)
            experience.prepare_direct_slabs(config.norm_adv)
            slabs = True
        else:
            experience.compute_gae(config.gamma, config.gae_lambda)
            slabs = want_slabs and experience.flatten_batch_slabs()
            if not slabs:
                experience.flatten_batch()
            if config.norm_adv:
                experience.normalize_advantages(slabs=slabs)

    n_mb = experience.num_minibatches
    if seg is not None:                        # persistent accumulator: the segment graphs update it in place
        if data.train_acc is None:
            data.train_acc = torch.zeros(6, device=device)
        acc = data.train_acc
        acc.zero_()
    else:
        acc = torch.zeros(6, device=device)    # policy, value, entropy, old_kl, kl, clipfrac
    obs_shape = data.vecenv.single_observation_space.shape
    fused = data.fused_loss and experience.lstm_h is None
    carry = {'lstm_state': None, 'approx_kl': None}
    if manual is not None:
        manual.pack_heads()                      # the parameters may have changed since the last train() (checkpoints)
    n_stats = config.update_epochs * n_mb

    def forward_backward(mb, k=0):              # k = epoch * n_mb + mb: the manual path's statistics row
        if direct:
            with profile.train_forward:
                d = experience.direct_minibatch(mb, config.norm_adv)
                manual.forward_backward(k, n_stats, d.obs, True, d.actions, d.logprobs, d.advantages, None, d.old_values, config,
                                        row_slab_stride=d.row_slab_stride, adv_norm=d.adv_norm)
            return
        if slabs:
            sl = experience._slabs
            obs = experience.slab_obs(mb)
            atn, log_probs, val, ret = sl.actions[mb], sl.logprobs[mb], sl.values[mb], sl.returns[mb]
            adv = sl.advantages_normalized[mb] if config.norm_adv else sl.advantages[mb]
        else:
            obs = experience.b_obs[mb]
            atn = experience.b_actions[mb]
            log_probs = experience.b_logprobs[mb]
            val = experience.b_values[mb]
            adv = experience.b_advantages_normalized[mb] if config.norm_adv else experience.b_advantages[mb]
            ret = experience.b_returns[mb]

        if manual is not None:
            with profile.train_forward:
                manual.forward_backward(k, n_stats, obs, bool(slabs), atn, log_probs, adv, ret, val, config)
            return

        with profile.train_forward:
            packed = None
            if fused:          # logits / value straight from the model; loss + its gradient in one kernel
                model = data.policy.policy
                if slabs:
                    packed = model.forward_packed_slabs(obs)
                elif hasattr(model, 'forward_packed'):
                    packed = model.forward_packed(obs.reshape(-1, *obs_shape))
                if packed is None:
                    logits, newvalue = model(obs.reshape(-1, *obs_shape))
            elif experience.lstm_h is not None:       # clean_pufferl.py:188-191: [rows, bptt, *obs] segments
                _, newlogprob, entropy, newvalue, st_ = data.policy(obs, state=carry['lstm_state'], action=atn)
                carry['lstm_state'] = (st_[0].detach(), st_[1].detach())
            else:
                _, newlogprob, entropy, newvalue = data.policy(obs.reshape(-1, *obs_shape), action=atn)

        with profile.train_misc:
            if fused and data.action_nvec is not None:
                if packed is not None:
                    loss, st = fused_ppo_loss_packed_multi(packed[0], data.action_nvec, atn, log_probs, adv, ret, val,
                                                           config)
                else:
                    loss, st = fused_ppo_loss_multi(logits, newvalue, atn, log_probs, adv, ret, val, config)
                pg_loss, v_loss, entropy_loss, old_approx_kl, approx_kl, clipfrac = st.unbind(0)
            elif fused:
                if packed is not None:
                    loss, st = fused_ppo_loss_packed(packed[0], packed[1], atn, log_probs, adv, ret, val, config)
                else:
                    loss, st = fused_ppo_loss(logits, newvalue, atn, log_probs, adv, ret, val, config)
                pg_loss, v_loss, entropy_loss, old_approx_kl, approx_kl, clipfrac = st.unbind(0)
            else:
                logratio = newlogprob - log_probs.reshape(-1)
                ratio = logratio.exp()
                with torch.no_grad():
                    old_approx_kl = (-logratio).mean()
                    approx_kl = ((ratio - 1) - logratio).mean()
                    clipfrac = ((ratio - 1.0).abs() > config.clip_coef).float().mean()

                adv = adv.reshape(-1)
                pg_loss1 = -adv * ratio
                pg_loss2 = -adv * torch.clamp(ratio, 1 - config.clip_coef, 1 + config.clip_coef)
                pg_loss = torch.max(pg_loss1, pg_loss2).mean()

                newvalue = newvalue.view(-1)
                if config.clip_vloss:
                    v_loss_unclipped = (newvalue - ret) ** 2
                    v_clipped = val + torch.clamp(newvalue - val, -config.vf_clip_coef, config.vf_clip_coef)
                    v_loss_clipped = (v_clipped - ret) ** 2
                    v_loss = 0.5 * torch.max(v_loss_unclipped, v_loss_clipped).mean()
                else:
                    v_loss = 0.5 * ((newvalue - ret) ** 2).mean()

                entropy_loss = entropy.mean()
                loss = pg_loss - config.ent_coef * entropy_loss + v_loss * config.vf_coef

        with profile.learn:
            if data.grad_bucket is not None:
                data.grad_bucket.zero()                     # grads are views into one flat buffer
            else:
                data.optimizer.zero_grad()
            loss.backward()

        with profile.train_misc, torch.no_grad():
            acc.add_(torch.stack([pg_loss.detach(), v_loss.detach(), entropy_loss.detach(), old_approx_kl,
                                  approx_kl, clipfrac]) / n_mb)
        carry['approx_kl'] = approx_kl

    def optimizer_step():
        with profile.learn:
            if manual is not None:
                manual.optimizer_step(config)
                return
            torch.nn.utils.clip_grad_norm_(data.policy.parameters(), config.max_grad_norm)
            data.optimizer.step()

    for epoch in range(config.update_epochs):
        carry['lstm_state'] = None
        for mb in range(n_mb):
            if seg is not None:       # the manual path writes its statistics to a per-(epoch, minibatch) row
                seg.run(('fb', mb) if manual is None else ('fb', epoch, mb),
                        lambda: forward_backward(mb, epoch * n_mb + mb))
            else:
                forward_backward(mb, epoch * n_mb + mb)
            if manual is not None:
                with profile.learn:
                    manual.all_reduce()                         # ONE NCCL all-reduce (sum; 1/world folded into the step)
            elif data.grad_bucket is not None:
                with profile.learn:
                    data.grad_bucket.all_reduce_mean()          # ONE NCCL all-reduce per optimizer step
            if seg is not None:
                seg.run('opt', optimizer_step)
            else:
                optimizer_step()

        if config.target_kl is not None:
            if carry['approx_kl'].item() > config.target_kl:
                break

    with profile.train_misc:
        # explained variance on the device, same quantities as clean_pufferl.py:266-270
        y_pred, y_true = experience.values, experience.returns
        var_y = y_true.var(unbiased=False)
        ev = 1 - (y_true - y_pred).var(unbiased=False) / var_y
        if manual is not None:
            acc = manual.loss_means(n_mb)
        return torch.cat([acc, torch.stack([ev, var_y])])


def train(data):
    """One PPO update (reference: clean_pufferl.py:156-292).  With ``config.cuda_graph`` (no target_kl, no
    LSTM) the device part is captured once -- after an eager first call that initialises the optimizer state -- and
    replayed as ONE graph launch; the learning rate lives in a device tensor so annealing works under replay."""
    config, profile, experience = data.config, data.profile, data.experience
    data.losses = make_losses()
    losses = data.losses
    if getattr(data, 'manual_update', None) is not None and data.manual_update.stale():
        # optimizer.load_state_dict() (try_load_checkpoint) replaced the Adam state tensors: the hand-written update
        # and any captured graph hold the old addresses -- rebuild both (eager call now, re-capture on the next one)
        if getattr(data.manual_update, 'peer', None) is not None:
            data.manual_update.peer.close()          # collective: every rank loaded the same checkpoint
        data.manual_update = None
        if data.train_graph_state > 0:
            data.train_graph, data.train_segments, data.train_graph_state = None, None, 0
    # multi-GPU: capturing the NCCL all-reduce inside one big graph hung on this stack (torch 2.11 / NCCL 2.28); ranks > 1
    # use per-segment graphs around an ordinary all-reduce call instead (see `segmented`)
    want_graph = bool(getattr(config, 'cuda_graph_train', getattr(config, 'cuda_graph', False)))
    # an NCCL call inside the update loop (autograd path on several ranks, or the hand-written update without peer
    # memory) keeps the update out of ONE graph; with the peer all-reduce fused into pb_clip_adam_peer there is none
    mu = getattr(data, 'manual_update', None)
    nccl_in_loop = data.grad_bucket is not None and not (mu is not None and (mu.world == 1 or mu.peer is not None))
    graphable = want_graph and not nccl_in_loop and \
        config.target_kl is None and experience.lstm_h is None and data.train_graph_state >= 0
    segmented = want_graph and nccl_in_loop and \
        config.target_kl is None and experience.lstm_h is None and data.train_graph_state >= 0
    if segmented and data.train_graph_state >= 1:
        if data.train_segments is None:
            data.train_segments = _SegmentGraphs()
        result = _train_device_part(data, seg=data.train_segments)
    elif not graphable or data.train_graph_state == 0:
        result = _train_device_part(data)
        if graphable or segmented:
            data.train_graph_state = 1
    else:
        if data.train_graph_state == 1:
            try:
                torch.cuda.synchronize()
                launches0 = _native.lib().pb_launch_count()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    data.train_result = _train_device_part(data)
                data.train_graph = graph
                data.train_graph_launches = _native.lib().pb_launch_count() - launches0
                data.train_graph_state = 2
            except Exception as e:          # capture is an optimisation: fall back to eager for good
                data.train_graph_state = -1
                data.msg = f'train graph capture failed ({type(e).__name__}: {e}); running eager'
                torch.cuda.synchronize()
                result = _train_device_part(data)
        if data.train_graph_state == 2:
            with profile.learn:
                data.train_graph.replay()
            data.train_graph_replays += 1
            experience.ptr = 0            # what sort_training_data leaves behind (clean_pufferl.py:461-463)
            experience.step = 0
            result = data.train_result

    _invalidate_policy_cache(data)          # graph replays update the parameters without running python hooks
    with profile.train_misc:
        if config.anneal_lr:
            frac = 1.0 - data.global_step / config.total_timesteps
            _set_lr(data.optimizer, frac * config.learning_rate)
        host = result.cpu().numpy()    # the one D2H of train()
        data.io.d2h += host.nbytes
        # like the reference the per-minibatch means are divided by num_minibatches and summed over ALL epochs
        # (clean_pufferl.py:249-254)
        losses.policy_loss, losses.value_loss, losses.entropy = float(host[0]), float(host[1]), float(host[2])
        losses.old_approx_kl, losses.approx_kl, losses.clipfrac = float(host[3]), float(host[4]), float(host[5])
        losses.explained_variance = float('nan') if host[7] == 0 else float(host[6])
        data.epoch += 1
        profile.update(data)
        interval = getattr(config, 'checkpoint_interval', None)        # clean_pufferl.py:288-290
        if interval and hasattr(config, 'data_dir') and \
                (data.epoch % interval == 0 or data.global_step >= config.total_timesteps):
            save_checkpoint(data)
            data.msg = f'Checkpoint saved at update {data.epoch}'


def save_checkpoint(data):
    """clean_pufferl.py:509-530: model_<epoch>.pt (the whole module) + trainer_state.pt (optimizer state, counters)."""
    import os
    config = data.config
    path = os.path.join(config.data_dir, config.exp_id)
    os.makedirs(path, exist_ok=True)
    model_name = f'model_{data.epoch:06d}.pt'
    model_path = os.path.join(path, model_name)
    torch.save(data.uncompiled_policy, model_path)
    state = {'optimizer_state_dict': data.optimizer.state_dict(), 'global_step': data.global_step,
             'agent_step': data.global_step, 'update': data.epoch, 'model_name': model_name, 'exp_id': config.exp_id}
    state_path = os.path.join(path, 'trainer_state.pt')
    torch.save(state, state_path + '.tmp')
    os.rename(state_path + '.tmp', state_path)
    return model_path


def try_load_checkpoint(data):
    """clean_pufferl.py:532-546.  The parameters are loaded IN PLACE (their addresses are captured in CUDA graphs);
    the optimizer state tensors are replaced by load_state_dict, which train() detects (_DefaultMLPUpdate.stale)."""
    import os
    config = data.config
    path = os.path.join(config.data_dir, config.exp_id)
    if not os.path.exists(path):
        print('No checkpoints found. Assuming new experiment')
        return
    resume_state = torch.load(os.path.join(path, 'trainer_state.pt'), weights_only=False)
    data.global_step = resume_state['global_step']
    data.epoch = resume_state['update']
    model_path = os.path.join(path, resume_state['model_name'])
    data.uncompiled_policy.load_state_dict(torch.load(model_path, weights_only=False).state_dict())
    data.optimizer.load_state_dict(resume_state['optimizer_state_dict'])
    _invalidate_policy_cache(data)
    if data.train_graph_state > 0:      # captured updates hold the old optimizer-state addresses: capture again
        data.train_graph, data.train_segments, data.train_graph_state = None, None, 0
    print(f'Loaded checkpoint {resume_state["model_name"]}')


def close(data):
    mu = getattr(data, 'manual_update', None)
    if mu is not None and getattr(mu, 'peer', None) is not None:
        mu.peer.close()            # collective: every rank closes (unmaps the peers' buffers, then frees its own)
        mu.peer = None
    data.vecenv.close()
