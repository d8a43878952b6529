"""``pufferlib.vector`` surface for device-resident envs: make / reset / step / send / recv.

Mirrors /root/reference/pufferlib/vector.py: ``make`` (:577-637) with the same validation and error
messages, module-level ``reset``/``step`` (:44-53), the RESET/SEND/RECV flag protocol and prechecks (:17-42),
``joint_space`` (:55-68), ``make_seeds`` (:639-650) and the ``Serial`` object surface (:70-166).  The backend
class ``B200`` replaces Serial/Multiprocessing: instead of N Python env objects stepped in a loop it owns one
``pb_env`` handle (N env instances on one GPU) and every send() is one kernel launch that writes obs / reward /
done rows where they are needed -- its own buffers, or straight into a bound rollout (``bind_rollout``).

recv() returns torch CUDA tensors (aliasing internal buffers across calls, as the reference aliases its numpy
buffers, vector.py:158-162).  With ``host_buffers=True`` it returns pinned-host numpy arrays exactly like Serial
(D2H copy per step), which is what an unmodified ``clean_pufferl.evaluate`` consumes.
"""
import ctypes as C
import functools

import numpy as np
import torch

from pufferlib_b200 import _native, spaces
from pufferlib_b200.environments import OBS_RECORD_DTYPE, resolve
from pufferlib_b200.exceptions import APIUsageError
from pufferlib_b200.namespace import Namespace, namespace

RESET = 0
STEP = 1
SEND = 2
RECV = 3
CLOSE = 4
MAIN = 5
INFO = 6


def recv_precheck(vecenv):
    if vecenv.flag != RECV:
        raise APIUsageError('Call reset before stepping')
    vecenv.flag = SEND


def send_precheck(vecenv, actions):
    if vecenv.flag != SEND:
        raise APIUsageError('Call (async) reset + recv before sending')
    if not vecenv.initialized:
        vecenv.initialized = True
        if isinstance(actions, torch.Tensor):
            space = vecenv.single_action_space
            if isinstance(space, spaces.MultiDiscrete):     # [N, k], column h in [0, nvec[h])
                shape = (vecenv.num_agents, len(space))
                bound = torch.as_tensor(space.nvec, device=actions.device)
            else:
                shape, bound = (vecenv.num_agents,), space.n
            ok = (tuple(actions.shape) == shape and not actions.dtype.is_floating_point
                  and bool(((actions >= 0) & (actions < bound)).all()))
        else:
            ok = vecenv.action_space.contains(np.asarray(actions))
        if not ok:
            raise APIUsageError('Actions do not match action space')
    vecenv.flag = RECV
    return actions


def reset(vecenv, seed=42):
    vecenv.async_reset(seed)
    obs, rewards, terminals, truncations, infos, env_ids, masks = vecenv.recv()
    return obs, infos


def step(vecenv, actions):
    vecenv.send(actions)
    obs, rewards, terminals, truncations, infos, env_ids, masks = vecenv.recv()
    return obs, rewards, terminals, truncations, infos


def joint_space(space, n):
    if isinstance(space, spaces.Discrete):
        return spaces.MultiDiscrete([space.n] * n)
    elif isinstance(space, spaces.MultiDiscrete):
        return spaces.Box(low=0, high=np.repeat(space.nvec[None] - 1, n, axis=0),
                          shape=(n, len(space)), dtype=space.dtype)
    elif isinstance(space, spaces.Box):
        return spaces.Box(low=np.repeat(space.low[None], n, axis=0), high=np.repeat(space.high[None], n, axis=0),
                          shape=(n, *space.shape), dtype=space.dtype)
    else:
        raise ValueError(f'Unsupported space: {space}')


def make_seeds(seed, num_envs):
    if isinstance(seed, int):
        return [seed + i for i in range(num_envs)]
    err = f'seed {seed} must be an integer or a list of integers'
    if isinstance(seed, (list, tuple)):
        if len(seed) != num_envs:
            raise APIUsageError(err)
        return seed
    raise APIUsageError(err)


_NP_DTYPES = {_native.DTYPE_F32: np.float32, _native.DTYPE_U8: np.uint8}
_TORCH_DTYPES = {_native.DTYPE_F32: torch.float32, _native.DTYPE_U8: torch.uint8}


class _DriverEnv:
    """What ``vecenv.driver_env`` must expose (SURVEY §8b): spaces, emulated, render()."""

    def __init__(self, vec):
        self.single_observation_space = vec.single_observation_space
        self.single_action_space = vec.single_action_space
        self.observation_space = vec.single_observation_space
        self.action_space = vec.single_action_space
        self.emulated = vec.emulated
        self.num_agents = 1
        self.render_mode = 'ansi'
        self._vec = vec

    def render(self):
        obs = self._vec.buf.observations[0].detach().cpu().numpy()
        return np.array2string(obs, max_line_width=200)


class B200:
    """Device-resident vectorised env backend (pass as ``backend=`` to ``make``)."""
    reset = reset
    step = step

    @classmethod
    def options(cls, **opts):
        """``backend=B200.options(host_buffers=True, exact_infos=True, device=0, env_index_offset=...)``:
        ``make`` forwards only num_workers / batch_size / zero_copy (vector.py:631-633), so backend options are
        bound here."""
        return functools.partial(cls, **opts)

    @property
    def num_envs(self):
        return self.agents_per_batch

    def __new__(cls, env_creators=None, env_args=None, env_kwargs=None, num_envs=None, **kwargs):
        # batch_size < num_envs: the reference's pool mode (vector.py:345-390) -> round-robin groups on side streams
        bs = kwargs.get('batch_size')
        if cls is B200 and bs is not None and num_envs is not None and bs != num_envs:
            return B200Pool(env_creators, env_args, env_kwargs, num_envs, **kwargs)
        return super().__new__(cls)

    def __init__(self, env_creators, env_args, env_kwargs, num_envs, host_buffers=False, exact_infos=None,
                 device=None, env_index_offset=0, **kwargs):
        for k in kwargs:
            if k not in ('num_workers', 'batch_size', 'zero_copy', 'backend'):
                raise APIUsageError(f'Invalid argument: {k}')
        kind, iparam = resolve(env_creators[0], env_args[0], env_kwargs[0])
        for c, a, k in zip(env_creators, env_args, env_kwargs):
            if resolve(c, a, k) != (kind, iparam):
                raise APIUsageError('B200 backend: all env creators / args must be identical')
        if not torch.cuda.is_available():
            raise RuntimeError('pufferlib_b200 needs a CUDA device (no CPU fallback)')
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device('cuda', self.device_index)
        self.kind = kind
        self.host_buffers = bool(host_buffers)
        self.exact_infos = self.host_buffers if exact_infos is None else bool(exact_infos)
        lib = _native.lib()
        # num_workers (the reference's Multiprocessing argument): every worker PROCESS there runs a Serial over its envs
        # with its own process-global `random` stream (vector.py:168-190, seeds sliced per worker at :424-428).  Only envs
        # that draw from that global stream depend on it (ocean.Squared); for them the envs are split into one pb_env
        # shard per worker, each with its own MT19937 stream, writing into the same contiguous buffers.  The other
        # kinds key their counter-based RNG by global env index, so the worker split cannot change their results.
        workers = kwargs.get('num_workers') or 1
        if kind != 'squared' or workers <= 1:
            workers = 1
        if num_envs % workers != 0:
            raise APIUsageError('num_envs must be divisible by num_workers')
        per = num_envs // workers
        self._shards = []          # (handle, first env, envs)
        for w in range(workers):
            cfg = _native.EnvConfig(kind=_native.ENV_KINDS[kind], num_envs=per, device=self.device_index,
                                    reserved=0, env_index_offset=int(env_index_offset) + w * per,
                                    iparam=(C.c_int32 * 8)(*iparam))
            handle = C.c_void_p()
            _native.check(lib.pb_env_create(C.byref(cfg), C.byref(handle)))
            self._shards.append((handle, w * per, per))
        self._handle = self._shards[0][0]
        info = _native.EnvInfo()
        _native.check(lib.pb_env_get_info(self._handle, C.byref(info)))
        self.obs_bytes = int(info.obs_bytes)
        self._obs_torch_dtype = _TORCH_DTYPES[info.obs_dtype]
        obs_shape = tuple(info.obs_shape[i] for i in range(info.obs_ndim))
        self.single_observation_space = spaces.Box(low=info.obs_low, high=info.obs_high, shape=obs_shape,
                                                   dtype=_NP_DTYPES[info.obs_dtype])
        nvec, heads = (C.c_int32 * 8)(), C.c_int32()
        _native.check(lib.pb_env_action_nvec(self._handle, nvec, C.byref(heads)))
        # MultiDiscrete kinds (emulation.py:115-120): actions are [N, k] int64 rows, column h in [0, nvec[h])
        self.atn_heads = int(heads.value)
        self.single_action_space = spaces.MultiDiscrete(list(nvec)[:self.atn_heads]) if self.atn_heads else \
            spaces.Discrete(info.num_actions)
        atn_shape = (num_envs, self.atn_heads) if self.atn_heads else (num_envs,)
        self._atn_row_bytes = 8 * max(1, self.atn_heads)
        self.emulated = namespace(observation_dtype=self.single_observation_space.dtype,
                                  emulated_observation_dtype=OBS_RECORD_DTYPE.get(kind, self.single_observation_space.dtype))
        self.agents_per_batch = num_envs
        self.num_agents = num_envs
        self.action_space = joint_space(self.single_action_space, num_envs)
        self.observation_space = joint_space(self.single_observation_space, num_envs)
        self.agent_ids = np.arange(num_envs)
        self.initialized = False
        self.flag = RESET
        self.infos = []
        with torch.cuda.device(self.device):
            self.buf = namespace(
                observations=torch.zeros((num_envs, *obs_shape), dtype=self._obs_torch_dtype, device=self.device),
                rewards=torch.zeros(num_envs, dtype=torch.float32, device=self.device),
                terminals=torch.zeros(num_envs, dtype=torch.bool, device=self.device),
                truncations=torch.zeros(num_envs, dtype=torch.bool, device=self.device),
                masks=torch.ones(num_envs, dtype=torch.bool, device=self.device),
                dones_f32=torch.zeros(num_envs, dtype=torch.float32, device=self.device),
            )
            self._actions_dev = torch.zeros(atn_shape, dtype=torch.int64, device=self.device)
        self.driver_env = _DriverEnv(self)
        # rollout binding (clean_pufferl.create): step outputs go straight into Experience rows
        self._rollout = None
        self._cursor = 0            # rollout row of the observation recv() returns next
        self._pending_own = True    # latest step output lives in self.buf (not yet in a rollout row)
        if self.host_buffers:
            self._host = namespace(
                observations=torch.zeros((num_envs, *obs_shape), dtype=self._obs_torch_dtype).pin_memory(),
                rewards=torch.zeros(num_envs, dtype=torch.float32).pin_memory(),
                terminals=torch.zeros(num_envs, dtype=torch.bool).pin_memory(),
                truncations=torch.zeros(num_envs, dtype=torch.bool).pin_memory(),
                masks=torch.ones(num_envs, dtype=torch.bool).pin_memory(),
                actions=torch.zeros(atn_shape, dtype=torch.int64).pin_memory(),
            )
            self._host_np = namespace(**{k: v.numpy() for k, v in self._host.items()})
            with torch.cuda.device(self.device):
                # device->host copies run on their own stream, behind the env kernel and beside the policy forward
                self._copy_stream = torch.cuda.Stream()
                self._ev_step, self._ev_copy, self._ev_act = torch.cuda.Event(), torch.cuda.Event(), torch.cuda.Event()
            self._host_pending = False
            self.graph_mode = False
        self.h2d_bytes = 0
        self.d2h_bytes = 0

    # -- rollout binding --------------------------------------------------------------------------------------
    def bind_rollout(self, experience):
        """Let send() write obs / reward / done rows directly into ``experience`` (time-major [H][N] tensors).
        Row 0 of each rollout is filled from the carry-over buffers at the first recv()."""
        if experience.batch_size % self.num_agents != 0:
            raise APIUsageError('batch_size must be a multiple of num_envs to bind a rollout')
        self._rollout = experience
        self._horizon = experience.batch_size // self.num_agents
        self._cursor = 0
        self._pending_own = True

    def _env_out(self, row, lo=0):
        """pb_env_out for rollout row `row`, or for the vecenv's own buffers when row is None; `lo` = first env of the
        shard the outputs belong to."""
        b = self.buf
        if row is None:
            return _native.EnvOut(obs=b.observations.data_ptr() + lo * self.obs_bytes, obs_stride=self.obs_bytes,
                                  rewards=b.rewards.data_ptr() + lo * 4, terminals=b.terminals.data_ptr() + lo,
                                  truncations=b.truncations.data_ptr() + lo, masks=b.masks.data_ptr() + lo,
                                  dones_f32=b.dones_f32.data_ptr() + lo * 4)
        x, n = self._rollout, self.num_agents
        return _native.EnvOut(obs=x.obs.data_ptr() + (row * n + lo) * self.obs_bytes, obs_stride=self.obs_bytes,
                              rewards=x.rewards.data_ptr() + (row * n + lo) * 4, terminals=b.terminals.data_ptr() + lo,
                              truncations=b.truncations.data_ptr() + lo, masks=b.masks.data_ptr() + lo,
                              dones_f32=x.dones.data_ptr() + (row * n + lo) * 4)

    # -- vector.Serial surface ---------------------------------------------------------------------------------
    def async_reset(self, seed=42):
        if not isinstance(seed, int):
            # list form of make_seeds (vector.py:639-650) -- what Multiprocessing hands each worker is the slice
            # [seed + lo, ..., seed + hi - 1] (:424-428).  Env i is seeded with seed + i on the device, so a list is
            # accepted when it is such a run of consecutive integers; arbitrary per-env seeds have no device form.
            seeds = make_seeds(seed, self.num_agents)
            if not all(isinstance(x, (int, np.integer)) for x in seeds) or \
                    any(int(seeds[i]) != int(seeds[0]) + i for i in range(len(seeds))):
                raise APIUsageError(f'seed {seed} must be an integer or a list of consecutive integers')
            seed = int(seeds[0])
        self.flag = RECV
        with torch.cuda.device(self.device):
            for handle, lo, _ in self._shards:
                out = self._env_out(None, lo)
                _native.check(_native.lib().pb_env_reset(handle, C.c_uint64(seed % (1 << 64)), C.byref(out),
                                                         _native.stream_ptr()))
        self._pending_own = True
        self._cursor = 0
        self.infos = []

    def send(self, actions):
        actions = send_precheck(self, actions)
        with torch.cuda.device(self.device):
            if isinstance(actions, torch.Tensor) and actions.is_cuda:
                a = actions if (actions.dtype == torch.int64 and actions.is_contiguous()) else \
                    actions.to(torch.int64).contiguous()
            else:
                a_np = np.ascontiguousarray(np.asarray(actions), dtype=np.int64)
                if self.host_buffers:
                    if a_np.ctypes.data != self._host_np.actions.ctypes.data:     # else: already in the pinned array
                        self._host_np.actions[:] = a_np
                    self._actions_dev.copy_(self._host.actions, non_blocking=True)
                else:
                    self._actions_dev.copy_(torch.from_numpy(a_np), non_blocking=False)
                self.h2d_bytes += a_np.nbytes
                a = self._actions_dev
            row = None
            if self._rollout is not None and not self._pending_own and self._cursor + 1 < self._horizon:
                row = self._cursor + 1
            for handle, lo, _ in self._shards:
                out = self._env_out(row, lo)
                _native.check(_native.lib().pb_env_step(handle, C.c_void_p(a.data_ptr() + self._atn_row_bytes * lo), C.byref(out),
                                                        _native.stream_ptr()))
            if self._rollout is not None:
                if row is None:
                    self._pending_own = True
                    self._cursor = 0
                else:
                    self._cursor = row
        self._stepped = True

    def recv(self, _device=False):
        recv_precheck(self)
        b = self.buf
        with torch.cuda.device(self.device):
            if self._rollout is not None:
                x, n, t = self._rollout, self.num_agents, self._cursor
                lo, hi = t * n, (t + 1) * n
                if self._pending_own:   # carry-over rows (reset, or the step that closed the previous rollout)
                    lib = _native.lib()
                    if self.host_buffers and self._host_pending and not self.graph_mode:
                        # copies of the previous rollout's rows may still be streaming to the host (host_defer): the first
                        # write into the rollout tensors waits for them on the device, the host does not block
                        torch.cuda.current_stream().wait_event(self._ev_copy)
                    _native.check(lib.pb_copy_rows(_native.ptr(b.observations), self.obs_bytes,
                                                   C.c_void_p(x.obs.data_ptr() + lo * self.obs_bytes),
                                                   self.obs_bytes, self.obs_bytes, n, _native.stream_ptr()))
                    x.rewards[lo:hi].copy_(b.rewards)
                    x.dones[lo:hi].copy_(b.dones_f32)
                    self._pending_own = False
                obs, rewards = x.obs[lo:hi], x.rewards[lo:hi]
            else:
                obs, rewards = b.observations, b.rewards
            if self.host_buffers:
                # the step's rows go to the pinned host arrays on the copy stream (ordered behind the env kernel that
                # produced them); recv() waits for them, recv_device() leaves the wait to host_sync()
                h, cs = self._host, self._copy_stream
                self._ev_step.record()
                cs.wait_event(self._ev_step)
                with torch.cuda.stream(cs):
                    h.observations.copy_(obs, non_blocking=True)
                    h.rewards.copy_(rewards, non_blocking=True)
                    h.terminals.copy_(b.terminals, non_blocking=True)
                    h.truncations.copy_(b.truncations, non_blocking=True)
                    self._ev_copy.record(cs)
                self._host_pending = True
                self.d2h_bytes += (h.observations.numel() * h.observations.element_size()
                                   + 4 * self.num_agents + 2 * self.num_agents)
                self._device_view = (obs, rewards, b.terminals, b.truncations, [], self.agent_ids, b.masks)
                return self.host_sync() if not _device else self._device_view
            infos = self._collect_infos() if self.exact_infos else []
            self.infos = infos
        return (obs, rewards, b.terminals, b.truncations, infos, self.agent_ids, b.masks)

    def recv_device(self):
        """host_buffers mode, for callers that keep computing on the device (clean_pufferl.evaluate): the same step as
        recv(), returned as DEVICE tensors, while the copies into the pinned host arrays are still in flight on the copy
        stream.  host_sync() completes the step on the host side (one wait per env step)."""
        if not self.host_buffers:
            return self.recv()
        return self.recv(_device=True)

    def actions_to_host(self, actions):
        """Device actions -> the pinned host action array (async, on the caller's stream); valid after host_sync()."""
        # a kernel store into the pinned (UVA-mapped) host array, not a DMA copy: the copy engine is busy with the 8 MB
        # observation blocks of this and earlier steps, and a 128 KB cudaMemcpyAsync would queue behind them (150 us per step)
        a = actions.reshape(-1)
        if a.dtype != torch.int64 or not a.is_contiguous():
            a = a.to(torch.int64).contiguous()
        nbytes = 8 * a.numel()
        _native.check(_native.lib().pb_copy_rows(_native.ptr(a), nbytes, C.c_void_p(self._host.actions.data_ptr()), nbytes, nbytes, 1,
                                                 _native.stream_ptr()))
        self._ev_act.record()
        self._act_pending = True
        self.d2h_bytes += self._atn_row_bytes * self.num_agents
        return self._host_np.actions

    def join_copies(self):
        """Inside a stream capture: the copy stream's work becomes a predecessor of whatever the caller's stream does next
        (the captured graph then ends only when every host copy has landed)."""
        torch.cuda.current_stream().wait_event(self._ev_copy)

    def host_sync(self, actions_only=False):
        """Wait for the step's device->host copies (and an outstanding actions_to_host); returns what recv() returns in
        host_buffers mode: pinned numpy arrays + the info dicts.  actions_only: wait for the action copy alone -- the
        observation / reward / flag copies keep streaming on the copy stream (they are ordered among themselves, each reads
        its own rollout row) and are awaited by the next full host_sync(); for callers that do not read them every step."""
        if self.graph_mode:
            # the rollout runs as a captured graph whose last node joins the copy stream: the caller's stream is the one
            # thing to wait for (events recorded during a capture cannot be waited on from the host)
            if not torch.cuda.is_current_stream_capturing():
                torch.cuda.current_stream().synchronize()
            self._host_pending = self._act_pending = False
            if actions_only:
                return None
        elif actions_only:
            if getattr(self, '_act_pending', False):
                self._ev_act.synchronize()
                self._act_pending = False
            return None
        else:
            if self._host_pending:
                self._ev_copy.synchronize()
                self._host_pending = False
            if getattr(self, '_act_pending', False):
                self._ev_act.synchronize()
                self._act_pending = False
        hn = self._host_np
        # the terminal flags are on the host already: no second D2H for the info dicts
        infos = self._collect_infos(hn.terminals) if self.exact_infos else []
        self.infos = infos
        return (hn.observations, hn.rewards, hn.terminals, hn.truncations, infos, self.agent_ids, hn.masks)

    def fused_rollout_ok(self, experience, policy):
        """Can the whole rollout run as ONE persistent kernel (pb_rollout_breakout_mlp)?  breakout, one RNG shard, device
        path, rollout bound to `experience` and standing at a rollout boundary, models.Default 128 -> 128 -> <= 4 actions
        behind a cleanrl.Policy with the fused sampler."""
        model = getattr(policy, 'policy', None)
        if not isinstance(self.single_action_space, spaces.Discrete):
            return False          # the persistent kernel samples one Discrete head
        if not (self.kind == 'breakout' and not self.host_buffers and not self.exact_infos and len(self._shards) == 1
                and self._rollout is experience and self._pending_own and self._cursor == 0 and self.flag == RECV
                and self.num_agents % 128 == 0 and experience.ptr == 0 and experience.lstm_h is None):
            return False
        if not (getattr(policy, 'fused_sample', False) and hasattr(model, 'head_matrix') and getattr(model, 'fast_path', False)):
            return False
        n_act, hid = model.decoder.weight.shape
        w = model.encoder.weight
        return (hid == 128 and tuple(w.shape) == (128, 128) and n_act == 4 and w.is_cuda and w.dtype == torch.float32
                and w.is_contiguous() and experience.obs.dtype == torch.float32)

    def fused_rollout(self, experience, policy):
        """evaluate's recv -> policy -> store -> send loop for the whole horizon in one launch; leaves the vecenv exactly
        where the loop would: the closing step's outputs in its own buffers, waiting for recv()."""
        x, model = experience, policy.policy
        if policy._counter is None:
            policy._counter = torch.zeros(1, dtype=torch.int64, device=self.device)
        with torch.no_grad():
            w_cat, b_cat = model.head_matrix()
        carry = self._env_out(None)
        with torch.cuda.device(self.device):
            _native.check(_native.lib().pb_rollout_breakout_mlp(
                self._handle, self._horizon, _native.ptr(x.obs), _native.ptr(x.rewards), _native.ptr(x.dones),
                _native.ptr(x.values), _native.ptr(x.logprobs), _native.ptr(x.actions), C.byref(carry),
                _native.ptr(model.encoder.weight), _native.ptr(model.encoder.bias), _native.ptr(w_cat), _native.ptr(b_cat),
                model.decoder.weight.shape[0], C.c_uint64(policy._seed), _native.ptr(policy._counter), _native.stream_ptr()))
        self._pending_own, self._cursor = True, 0
        self.initialized = True
        self.flag = RECV

    def pinned(self, array):
        """The pinned torch tensor behind one of the numpy arrays recv() returned in host_buffers mode (so the
        caller's H2D copy is a true async pinned transfer)."""
        for k, v in self._host_np.items():
            if v is array:
                return self._host[k]
        return torch.as_tensor(array)

    def _collect_infos(self, term=None):
        """Per-env info dicts for rows that just ended an episode (EpisodeStats, postprocess.py:36-52), in env
        order like Serial.send (vector.py:153-154).  Costs one D2H of the terminal flags per recv unless the caller
        already has them on the host (``term``)."""
        if term is None:
            term = self.buf.terminals.cpu().numpy()
            self.d2h_bytes += term.nbytes
        idx = np.nonzero(term)[0]
        if len(idx) == 0:
            return []
        lib = _native.lib()
        n = self.num_agents
        # the three per-env arrays through ONE staging tensor and ONE device->host copy (one sync instead of three)
        stage = torch.empty(16 * n, dtype=torch.uint8, device=self.buf.terminals.device)
        base, s_ = stage.data_ptr(), _native.stream_ptr()
        for handle, lo, cnt in self._shards:
            p_ret, p_len, p_score = C.c_void_p(), C.c_void_p(), C.c_void_p()
            _native.check(lib.pb_env_episode_rows(handle, C.byref(p_ret), C.byref(p_len), C.byref(p_score)))
            for src, off, nbytes in ((p_ret.value, 8 * lo, 8 * cnt), (p_len.value, 8 * n + 4 * lo, 4 * cnt),
                                     (p_score.value, 12 * n + 4 * lo, 4 * cnt)):
                _native.check(lib.pb_copy_rows(C.c_void_p(src), nbytes, C.c_void_p(base + off), nbytes, nbytes, 1, s_))
        host = stage.cpu().numpy()
        ret, length, score = host[:8 * n].view(np.float64), host[8 * n:12 * n].view(np.int32), \
            host[12 * n:].view(np.float32)
        self.d2h_bytes += n * 16
        return [{'episode_return': float(ret[i]), 'episode_length': int(length[i]), 'score': float(score[i])}
                for i in idx]

    def episode_stats(self, clear=True):
        """Device-side EpisodeStats reduction: {episode_return, episode_length, score} means over the episodes
        finished since the last call, plus their count (one 32-byte D2H)."""
        out = [0.0] * 4
        with torch.cuda.device(self.device):
            for handle, _, _ in self._shards:
                part = (C.c_double * 4)()
                _native.check(_native.lib().pb_env_stats_read(handle, part, int(clear), _native.stream_ptr()))
                out = [a + b for a, b in zip(out, part)]
                self.d2h_bytes += 256 * 32
        cnt = out[0]
        if cnt <= 0:
            return {}, 0
        return {'episode_return': out[1] / cnt, 'episode_length': out[2] / cnt, 'score': out[3] / cnt}, int(cnt)

    def close(self):
        for handle, _, _ in getattr(self, '_shards', []):
            _native.lib().pb_env_destroy(handle)
        self._shards, self._handle = [], None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class B200Pool:
    """``batch_size < num_envs``: the pool / double-buffering mode of the reference's Multiprocessing backend
    (vector.py:345-390).  The N envs are split into G = N / batch_size groups (contiguous env ranges, one pb_env handle
    each, seeded by global env index).  recv() returns the groups round-robin (deterministically, unlike the reference's
    first-ready order); send() steps the group just received on that group's own CUDA stream, so its env-step kernel
    overlaps the policy forward of the next group on the caller's stream.  Rows therefore arrive as
    (step t, group g) blocks = arrival index t*N + e, the layout Experience expects."""
    reset = reset
    step = step

    @property
    def num_envs(self):
        return self.agents_per_batch

    def __init__(self, env_creators, env_args, env_kwargs, num_envs, host_buffers=False, exact_infos=None,
                 device=None, env_index_offset=0, **kwargs):
        b = int(kwargs.pop('batch_size'))
        for k in kwargs:
            if k not in ('num_workers', 'zero_copy', 'backend'):
                raise APIUsageError(f'Invalid argument: {k}')
        if b < 1 or num_envs % b != 0:
            raise APIUsageError('num_envs must be divisible by batch_size')
        g = num_envs // b
        # num_workers given: a batch is workers_per_batch = batch_size / envs_per_worker whole workers (vector.py:244-246),
        # each with its own RNG stream; not given: one stream per group
        nw = kwargs.get('num_workers')
        wpb = {}
        if nw:
            epw = num_envs // nw
            if epw < 1 or b % epw != 0:
                raise APIUsageError('batch_size must be divisible by (num_envs / num_workers)')
            wpb = {'num_workers': b // epw}
        self.groups = [B200(env_creators[i * b:(i + 1) * b], env_args[i * b:(i + 1) * b], env_kwargs[i * b:(i + 1) * b], b,
                            host_buffers=host_buffers, exact_infos=exact_infos, device=device,
                            env_index_offset=env_index_offset + i * b, **wpb) for i in range(g)]
        first = self.groups[0]
        self.device = first.device
        self.host_buffers, self.exact_infos = first.host_buffers, first.exact_infos
        self.single_observation_space, self.single_action_space = first.single_observation_space, first.single_action_space
        self.emulated, self.driver_env, self.obs_bytes = first.emulated, first.driver_env, first.obs_bytes
        self.agents_per_batch, self.num_agents = b, num_envs
        self.action_space, self.observation_space = first.action_space, first.observation_space
        self.agent_ids = np.arange(num_envs)
        self._ids = [np.arange(i * b, (i + 1) * b) for i in range(g)]
        self.initialized = False
        self.flag = RESET
        self.infos = []
        with torch.cuda.device(self.device):
            self._streams = [torch.cuda.Stream() for _ in range(g)]
            self._events = [torch.cuda.Event() for _ in range(g)]
        self._next = 0          # group recv() returns next
        self._pending = None    # group whose actions send() expects

    @property
    def h2d_bytes(self):
        return sum(v.h2d_bytes for v in self.groups)

    @property
    def d2h_bytes(self):
        return sum(v.d2h_bytes for v in self.groups)

    def pinned(self, array):
        for v in self.groups:
            t = v.pinned(array)
            if t.is_pinned():
                return t
        return torch.as_tensor(array)

    def async_reset(self, seed=42):
        for v in self.groups:
            v.async_reset(seed)
        with torch.cuda.device(self.device):
            for ev in self._events:
                ev.record()
        self.flag = RECV
        self._next, self._pending = 0, None

    def recv(self):
        recv_precheck(self)
        g = self._next
        v = self.groups[g]
        with torch.cuda.device(self.device):
            torch.cuda.current_stream().wait_event(self._events[g])      # group g's last step has finished
        v.flag = RECV
        o, r, d, t, infos, _, m = v.recv()
        self.infos = infos
        self._pending = g
        return o, r, d, t, infos, self._ids[g], m

    def send(self, actions):
        if self.flag != SEND:
            raise APIUsageError('Call (async) reset + recv before sending')
        g = self._pending
        v = self.groups[g]
        with torch.cuda.device(self.device):
            side = self._streams[g]
            side.wait_stream(torch.cuda.current_stream())                # the actions were produced on the caller's stream
            with torch.cuda.stream(side):
                v.flag = SEND
                v.send(actions)
                self._events[g].record(side)
        self.initialized = v.initialized
        self.flag = RECV
        self._next = (g + 1) % len(self.groups)

    def join(self):
        """Make the caller's stream wait for every group's outstanding step (needed before graph capture ends)."""
        with torch.cuda.device(self.device):
            for ev in self._events:
                torch.cuda.current_stream().wait_event(ev)

    def episode_stats(self, clear=True):
        self.join()
        tot, cnt = {}, 0
        for v in self.groups:
            means, c = v.episode_stats(clear)
            for k, x in means.items():
                tot[k] = tot.get(k, 0.0) + x * c
            cnt += c
        return ({k: x / cnt for k, x in tot.items()}, cnt) if cnt else ({}, 0)

    def close(self):
        for v in self.groups:
            v.close()


def make(env_creator_or_creators, env_args=None, env_kwargs=None, backend=B200, num_envs=1, **kwargs):
    """Same contract and error behaviour as the reference ``pufferlib.vector.make`` (vector.py:577-637)."""
    if num_envs < 1:
        raise APIUsageError('num_envs must be at least 1')
    if num_envs != int(num_envs):
        raise APIUsageError('num_envs must be an integer')

    if 'num_workers' in kwargs:
        num_workers = kwargs['num_workers']
        envs_per_worker = num_envs / num_workers
        if envs_per_worker != int(envs_per_worker):
            raise APIUsageError('num_envs must be divisible by num_workers')
        if 'batch_size' in kwargs:
            batch_size = kwargs['batch_size']
            if batch_size is None:
                batch_size = num_envs
            if batch_size % envs_per_worker != 0:
                raise APIUsageError('batch_size must be divisible by (num_envs / num_workers)')

    if env_args is None:
        env_args = []
    if env_kwargs is None:
        env_kwargs = {}

    if not isinstance(env_creator_or_creators, (list, tuple)):
        env_creators = [env_creator_or_creators] * num_envs
        env_args = [env_args] * num_envs
        env_kwargs = [env_kwargs] * num_envs
    else:
        env_creators = env_creator_or_creators

    if len(env_creators) != num_envs:
        raise APIUsageError('env_creators must be a list of length num_envs')
    if len(env_args) != num_envs:
        raise APIUsageError('env_args must be a list of length num_envs')
    if len(env_kwargs) != num_envs:
        raise APIUsageError('env_kwargs must be a list of length num_envs')

    # per-entry validation: identical objects are checked once (N can be 131072)
    seen = set()
    for i in range(num_envs):
        key = (id(env_creators[i]), id(env_args[i]), id(env_kwargs[i]))
        if key in seen:
            continue
        seen.add(key)
        if not callable(env_creators[i]):
            raise APIUsageError('env_creators must be a list of callables')
        if not isinstance(env_args[i], (list, tuple)):
            raise APIUsageError('env_args must be a list of lists or tuples')
        if not isinstance(env_kwargs[i], (dict, Namespace)):
            raise APIUsageError('env_kwargs must be a list of dictionaries')

    for k in kwargs:
        if k not in ['num_workers', 'batch_size', 'zero_copy', 'backend']:
            raise APIUsageError(f'Invalid argument: {k}')

    return backend(env_creators, env_args, env_kwargs, num_envs, **kwargs)
