"""``pufferlib.frameworks.cleanrl`` equivalent: logits -> action / logprob / entropy, and the Policy wrapper.

Reference: /root/reference/pufferlib/frameworks/cleanrl.py:25-47 (sample_logits), :50-66 (Policy).
``sample_logits`` is the plain torch formulation (used in train, where actions are given);
``Policy(fused_sample=True)`` routes the sampling case through the fused CUDA epilogue pb_sample_logits.
"""
import ctypes as C

import torch

from pufferlib_b200 import _native


def log_prob(logits, value):
    value = value.long().unsqueeze(-1)
    value, log_pmf = torch.broadcast_tensors(value, logits)
    value = value[..., :1]
    return log_pmf.gather(-1, value).squeeze(-1)


def entropy(logits):
    min_real = torch.finfo(logits.dtype).min
    logits = torch.clamp(logits, min=min_real)
    p_log_p = logits * torch.softmax(logits, dim=-1)
    return -p_log_p.sum(-1)


def sample_logits(logits, action=None):
    """Returns (action, logprob, entropy).  `logits` is one tensor (Discrete) or a list with one tensor per head
    (MultiDiscrete, the reference's semantics and shapes): action [N, k] (given actions are read as
    action.view(N, -1).T), logprob and entropy summed over the heads."""
    if isinstance(logits, torch.Tensor):
        normalized = logits - logits.logsumexp(dim=-1, keepdim=True)
        if action is None:
            action = torch.multinomial(torch.softmax(normalized, dim=-1), 1).squeeze(-1)
        else:
            action = action.reshape(-1)
        return action, log_prob(normalized, action), entropy(normalized)
    normalized = [lg - lg.logsumexp(dim=-1, keepdim=True) for lg in logits]
    if action is None:
        action = torch.stack([torch.multinomial(torch.softmax(nl, dim=-1), 1).squeeze(-1) for nl in normalized])
    else:
        action = action.view(logits[0].shape[0], -1).T
    assert len(normalized) == len(action)
    logprob = torch.stack([log_prob(nl, a) for nl, a in zip(normalized, action)]).T.sum(1)
    ent = torch.stack([entropy(nl) for nl in normalized]).T.sum(1)
    return action.T, logprob, ent


class Policy(torch.nn.Module):
    """Wrap a non-recurrent model: forward(x, action=None) -> (action, logprob, entropy, value)."""

    def __init__(self, policy, fused_sample=False, seed=0):
        super().__init__()
        self.policy = policy
        self.fused_sample = fused_sample
        self._seed = int(seed)
        self._counter = None     # device-side draw counter: CUDA-graph replays keep drawing fresh numbers
        self._ticket = None      # exit ticket of pb_policy_mlp_sample (its last CTA advances the counter)

    def get_value(self, x, state=None):
        _, value = self.policy(x)
        return value

    def get_action_and_value(self, x, action=None, out=None):
        """``out`` (optional, sampling only): (values_row, logprobs_row, actions_row) rollout row views the fused
        epilogue writes into directly -- the policy-output part of Experience.store without a copy kernel."""
        if action is None and self.fused_sample and not torch.is_grad_enabled():
            fused = self._policy_step_fused(x, out)
            if fused is not None:
                return fused
        logits, value = self.policy(x)
        if action is None and self.fused_sample and not torch.is_grad_enabled():
            if not isinstance(logits, torch.Tensor):
                return self._sample_fused_multi(logits, value, out)
            return self._sample_fused(logits, value, out)
        action, logprob, ent = sample_logits(logits, action)
        return action, logprob, ent, value

    def _policy_step_fused(self, x, out=None):
        """models.Default with 128 fp32 features / 128 hidden / <= 7 actions: the whole rollout-time policy step (encoder,
        ReLU, heads, sampling, row stores) as ONE kernel (pb_policy_mlp_sample).  Returns None if it does not apply."""
        model = self.policy
        if not (hasattr(model, 'head_matrix') and getattr(model, 'fast_path', False) and x.is_cuda
                and x.dtype == torch.float32):
            return None
        if not isinstance(model.decoder, torch.nn.Linear):
            return None           # the one-kernel policy step samples one Discrete head
        x2 = x.view(x.shape[0], -1)
        n_act, hid = model.decoder.weight.shape
        if x2.shape[1] != 128 or hid != 128 or n_act > 7 or x2.stride(1) != 1 or x2.stride(0) % 4 != 0:
            return None
        n, dev = x2.shape[0], x2.device
        if out is None:
            value = torch.empty(n, dtype=torch.float32, device=dev)
            logprob = torch.empty(n, dtype=torch.float32, device=dev)
            actions = torch.empty(n, dtype=torch.int64, device=dev)
        else:
            value, logprob, actions = out
        ent = torch.empty(n, dtype=torch.float32, device=dev)
        if self._counter is None:
            self._counter = torch.zeros(1, dtype=torch.int64, device=dev)
        if self._ticket is None:
            self._ticket = torch.zeros(1, dtype=torch.int32, device=dev)
        w_cat, b_cat = model.head_matrix()
        w_enc = model.encoder_weight_tf32()
        _native.check(_native.lib().pb_policy_mlp_sample(
            _native.ptr(x2), x2.stride(0), _native.ptr(w_enc), _native.ptr(model.encoder.bias),
            _native.ptr(w_cat), _native.ptr(b_cat), n, 128, hid, n_act, C.c_uint64(self._seed),
            _native.ptr(self._counter), _native.ptr(self._ticket), _native.ptr(actions), _native.ptr(logprob),
            _native.ptr(value), _native.ptr(ent), _native.stream_ptr()))   # the kernel's last CTA advances the counter
        return actions, logprob, ent, value

    def _sample_fused(self, logits, value, out=None):
        if logits.dtype != torch.float32 or logits.stride(1) != 1:
            logits = logits.float().contiguous()
        n, a = logits.shape
        dev = logits.device
        if out is None:
            actions = torch.empty(n, dtype=torch.int64, device=dev)
            logprob = torch.empty(n, dtype=torch.float32, device=dev)
            rows = (None, None, None)
            value_out = value
        else:
            value_out, logprob, actions = out
            rows = (_native.ptr(value_out), None, None)     # logprob / action rows ARE the primary outputs
        ent = torch.empty(n, dtype=torch.float32, device=dev)
        if self._counter is None:
            self._counter = torch.zeros(1, dtype=torch.int64, device=dev)
        v2 = value.reshape(n, -1)
        _native.check(_native.lib().pb_sample_logits(
            _native.ptr(logits), logits.stride(0), n, a, C.c_uint64(self._seed), C.c_uint64(0),
            _native.ptr(self._counter), _native.ptr(actions), _native.ptr(logprob), _native.ptr(ent),
            _native.ptr(v2), v2.stride(0), rows[0], rows[1], rows[2], _native.stream_ptr()))
        self._counter.add_(1)
        return actions, logprob, ent, value_out

    def _sample_fused_multi(self, logits, value, out=None):
        """pb_sample_logits_multi on a list of head logits.  Heads that are consecutive column blocks of one row-major
        tensor (models.Default's packed [M, 8] output) are read in place; otherwise they are concatenated once."""
        n, dev = logits[0].shape[0], logits[0].device
        nvec = [lg.shape[1] for lg in logits]
        base, stride = logits[0], logits[0].stride(0)
        in_place = base.dtype == torch.float32 and all(
            lg.dtype == torch.float32 and lg.stride(1) == 1 and lg.stride(0) == stride
            and lg.data_ptr() == base.data_ptr() + 4 * sum(nvec[:h]) for h, lg in enumerate(logits))
        if not in_place:
            base = torch.cat([lg.float() for lg in logits], dim=1).contiguous()
            stride = base.stride(0)
        if out is None:
            actions = torch.empty(n, len(nvec), dtype=torch.int64, device=dev)
            logprob = torch.empty(n, dtype=torch.float32, device=dev)
            values_row = None
            value_out = value
        else:
            value_out, logprob, actions = out
            values_row = _native.ptr(value_out)
        ent = torch.empty(n, dtype=torch.float32, device=dev)
        if self._counter is None:
            self._counter = torch.zeros(1, dtype=torch.int64, device=dev)
        v2 = value.reshape(n, -1)
        nv = (C.c_int32 * len(nvec))(*nvec)
        _native.check(_native.lib().pb_sample_logits_multi(
            _native.ptr(base), stride, n, nv, len(nvec), C.c_uint64(self._seed), C.c_uint64(0),
            _native.ptr(self._counter), _native.ptr(actions), _native.ptr(logprob), _native.ptr(ent),
            _native.ptr(v2), v2.stride(0), values_row, None, None, _native.stream_ptr()))
        self._counter.add_(1)
        return actions, logprob, ent, value_out

    def forward(self, x, action=None, out=None):
        return self.get_action_and_value(x, action, out)


class RecurrentPolicy(torch.nn.Module):
    """Wrap a recurrent model (reference: pufferlib/frameworks/cleanrl.py:69-93):
    forward(x, state=None, action=None) -> (action, logprob, entropy, value, state)."""

    def __init__(self, policy):
        super().__init__()
        self.policy = policy

    @property
    def lstm(self):
        if hasattr(self.policy, 'recurrent'):
            return self.policy.recurrent
        if hasattr(self.policy, 'lstm'):
            return self.policy.lstm
        raise ValueError('Policy must have a subnetwork named lstm or recurrent')

    def get_action_and_value(self, x, state=None, action=None):
        logits, value, state = self.policy(x, state)
        action, logprob, ent = sample_logits(logits, action)
        return action, logprob, ent, value, state

    def forward(self, x, state=None, action=None):
        return self.get_action_and_value(x, state, action)
