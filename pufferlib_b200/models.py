"""Policies for the configs in BASELINE.json: PyTorch modules, dense GEMMs on cuBLAS/cuDNN (tensor cores).

Same architecture and call convention as the reference (adjacent to the hot path, not rewritten):
  Default        /root/reference/pufferlib/models.py:12-62   Linear(prod(obs)->hidden)+ReLU; heads hidden->n_act, ->1
  Convolutional  /root/reference/pufferlib/models.py:113-157 NatureCNN for (4,84,84) uint8 (atari/torch.py:8-18)
  layer_init     /root/reference/pufferlib/pytorch.py:193-199
"""
import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional  # noqa: F401


class _DefaultMLPFunction(torch.autograd.Function):
    """models.Default as one autograd node on the device fast path.

    forward : hidden = relu(x @ W_enc^T + b_enc)  -- bias + ReLU fused into the cuBLASLt GEMM epilogue;
              out    = hidden @ W_cat^T + b_cat    -- both heads in ONE 8-column GEMM (n_act logits, value, zero pad).
    backward: pb_mlp_tail_backward reads `hidden` once and produces dPre (heads dX + ReLU backward), dW_heads, db_heads
              and db_enc; the dense dW_enc = dPre^T @ x stays on cuBLAS tensor cores.  x (the observations) has no grad.
    """

    @staticmethod
    def forward(ctx, x, w_enc, b_enc, w_dec, b_dec, w_val, b_val, cache):
        n_act, hid = w_dec.shape
        if x.dim() == 3:
            # slab form [G, R, F]: G equally spaced row slabs of the rollout buffer (a strided VIEW, see
            # Experience.flatten_batch_slabs) -- one GEMM per slab writes its part of the contiguous hidden layer,
            # the observations are never gathered into a minibatch copy
            g_, r_, _ = x.shape
            hidden = x.new_empty(g_ * r_, hid)
            for g in range(g_):
                torch._addmm_activation(b_enc, x[g], w_enc.t(), use_gelu=False, out=hidden[g * r_:(g + 1) * r_])
        else:
            try:
                hidden = torch._addmm_activation(b_enc, x, w_enc.t(), use_gelu=False)
            except (AttributeError, RuntimeError):
                hidden = torch.relu(torch.addmm(b_enc, x, w_enc.t()))
        # the 8-row head matrix: rebuilt on every forward that records gradients (the parameters change every optimizer
        # step, and fused optimizers do NOT bump tensor._version, so it cannot be cached across steps); under no_grad
        # (the rollout: 128 forwards with frozen parameters) it is built once and reused until invalidate_cache()
        # (torch.is_grad_enabled() is always False inside Function.forward: decide from the inputs that need gradients)
        use_cache = not any(ctx.needs_input_grad[1:7])
        key = (w_dec.data_ptr(), torch.cuda.is_current_stream_capturing())
        if use_cache and cache.get('key') == key:
            w_cat, b_cat = cache['w'], cache['b']
        else:
            w_cat = x.new_zeros(8, hid)
            w_cat[:n_act] = w_dec
            w_cat[n_act] = w_val[0]
            b_cat = x.new_zeros(8)
            b_cat[:n_act] = b_dec
            b_cat[n_act] = b_val[0]
            if use_cache:
                cache['key'], cache['w'], cache['b'] = key, w_cat, b_cat
        out = torch.addmm(b_cat, hidden, w_cat.t())
        ctx.save_for_backward(x, hidden, w_cat)
        ctx.n_act = n_act
        return out

    @staticmethod
    def backward(ctx, dout):
        from pufferlib_b200 import _native
        x, hidden, w_cat = ctx.saved_tensors
        n_act, (m, hid) = ctx.n_act, hidden.shape
        dout = dout.contiguous()
        dpre = torch.empty_like(hidden)
        grads = torch.empty(8 * hid + hid + 8, dtype=torch.float32, device=x.device)
        lib = _native.lib()
        ws = torch.empty(lib.pb_mlp_tail_workspace_bytes(m, hid), dtype=torch.uint8, device=x.device)
        _native.check(lib.pb_mlp_tail_backward(_native.ptr(dout), dout.stride(0), _native.ptr(w_cat), _native.ptr(hidden),
                                               m, hid, _native.ptr(dpre), _native.ptr(grads), _native.ptr(ws),
                                               ws.numel(), _native.stream_ptr()))
        dw_cat = grads[:8 * hid].view(8, hid)
        db_enc = grads[8 * hid:9 * hid]
        db_cat = grads[9 * hid:]
        # dW_enc = dPre^T @ x is one 128x128 output tile with K = M: as a batched GEMM over 64 K-slices (+ a 64-way sum)
        # the library GEMM runs at the HBM roofline (91 us vs 193 us at M = 524288; profiles/tools/gemm_variants.py)
        split = 64
        if x.dim() == 3:            # slab form: the K-slices tile each slab, partial products into one buffer
            g_, r_, f_ = x.shape
            sp = max(1, split // g_)
            while r_ % sp:
                sp //= 2
            part = x.new_empty(g_ * sp, hid, f_)
            for g in range(g_):
                torch.bmm(dpre[g * r_:(g + 1) * r_].view(sp, r_ // sp, hid).transpose(1, 2),
                          x[g].view(sp, r_ // sp, f_), out=part[g * sp:(g + 1) * sp])
            dw_enc = part.sum(0)
        elif m % split == 0 and m // split >= 256:
            dw_enc = torch.bmm(dpre.view(split, m // split, hid).transpose(1, 2), x.view(split, m // split, -1)).sum(0)
        else:
            dw_enc = dpre.t() @ x
        return (None, dw_enc, db_enc, dw_cat[:n_act], db_cat[:n_act], dw_cat[n_act:n_act + 1],
                db_cat[n_act:n_act + 1], None)


def layer_init(layer, std=np.sqrt(2), bias_const=0.0):
    torch.nn.init.orthogonal_(layer.weight, std)
    torch.nn.init.constant_(layer.bias, bias_const)
    return layer


class Default(nn.Module):
    def __init__(self, env, hidden_size=128):
        super().__init__()
        self.encoder = nn.Linear(int(np.prod(env.single_observation_space.shape)), hidden_size)
        # MultiDiscrete: one decoder per head (models.py:29-38), state-dict keys decoder.0.weight, ...
        nvec = getattr(env.single_action_space, 'nvec', None)
        self.is_multidiscrete = nvec is not None
        if self.is_multidiscrete:
            self.nvec = [int(n) for n in nvec]
            self.decoder = nn.ModuleList([layer_init(nn.Linear(hidden_size, n), std=0.01) for n in self.nvec])
        else:
            self.decoder = layer_init(nn.Linear(hidden_size, env.single_action_space.n), std=0.01)
        self.value_head = nn.Linear(hidden_size, 1)
        self.fast_path = True     # fused forward epilogues + pb_mlp_tail_backward (CUDA, hidden 128, <= 7 actions)
        self._head_cache = {}

    def invalidate_cache(self):
        """Call after the parameters changed (clean_pufferl does: optimizer post-step hook, start of evaluate, end of
        train)."""
        self._head_cache.clear()

    def decoder_params(self):
        """(weight [n_logits, H], bias [n_logits]) of all action heads, head after head (a differentiable cat for a
        MultiDiscrete decoder)."""
        if self.is_multidiscrete:
            return torch.cat([d.weight for d in self.decoder]), torch.cat([d.bias for d in self.decoder])
        return self.decoder.weight, self.decoder.bias

    @property
    def n_logits(self):
        return sum(self.nvec) if self.is_multidiscrete else self.decoder.out_features

    def split_logits(self, logits):
        """[M, n_logits] -> the reference's decode_actions output: one tensor, or a list of views per head."""
        return list(logits.split(self.nvec, dim=1)) if self.is_multidiscrete else logits

    def head_matrix(self):
        """(w_cat [8, H], b_cat [8]): logit rows of every head | value row | zero padding; cached under no_grad."""
        cache = self._head_cache
        w0 = self.decoder[0].weight if self.is_multidiscrete else self.decoder.weight
        key = (w0.data_ptr(), torch.cuda.is_current_stream_capturing())
        if not torch.is_grad_enabled() and cache.get('key') == key:
            return cache['w'], cache['b']
        with torch.no_grad():
            w_dec, b_dec = self.decoder_params()
            n_act, hid = w_dec.shape
            w_cat = w_dec.new_zeros(8, hid)
            w_cat[:n_act] = w_dec
            w_cat[n_act] = self.value_head.weight[0]
            b_cat = w_dec.new_zeros(8)
            b_cat[:n_act] = b_dec
            b_cat[n_act] = self.value_head.bias[0]
        if not torch.is_grad_enabled():
            cache['key'], cache['w'], cache['b'] = key, w_cat, b_cat
        return w_cat, b_cat

    def encoder_weight_tf32(self):
        """The encoder weight rounded to TF32 (round-to-nearest, ties away: cvt.rna) for pb_policy_mlp_sample, which
        feeds the bits straight to the tensor cores; cached with the head matrix (same invalidation)."""
        cache = self._head_cache
        key = (self.encoder.weight.data_ptr(), torch.cuda.is_current_stream_capturing())
        if not torch.is_grad_enabled() and cache.get('ekey') == key:
            return cache['wenc']
        with torch.no_grad():
            bits = self.encoder.weight.detach().contiguous().view(torch.int32)
            w = ((bits + 0x1000) & ~0x1FFF).view(torch.float32)
        if not torch.is_grad_enabled():
            cache['ekey'], cache['wenc'] = key, w
        return w

    def _fast_ok(self, x):
        hid = self.encoder.out_features
        return self.fast_path and x.is_cuda and hid == 128 and self.n_logits + 1 <= 8 and not x.requires_grad

    def forward_packed(self, observations):
        """-> (out [M, 8], n_act) with logits = out[:, :n_act] (every head, head after head), value = out[:, n_act]
        (zero padding after), or None when the fast path does not apply.  Lets the fused PPO loss hand back ONE [M, 8]
        gradient."""
        x = observations.view(observations.shape[0], -1)
        if not self._fast_ok(x):
            return None
        w_dec, b_dec = self.decoder_params()
        out = _DefaultMLPFunction.apply(x.float().contiguous(), self.encoder.weight, self.encoder.bias,
                                        w_dec, b_dec, self.value_head.weight,
                                        self.value_head.bias, self._head_cache)
        return out, self.n_logits

    def forward_packed_slabs(self, slabs):
        """forward_packed for a minibatch given as [G, R, features] row slabs (a strided view of the rollout
        observations; Experience.slab_obs): rows of the result are slab-major.  None when the fast path does not apply."""
        if slabs.dim() > 3:
            slabs = slabs.flatten(2)          # [G, R, *obs] -> [G, R, features] (a view: obs dims are contiguous)
        if slabs.dim() != 3 or not self._fast_ok(slabs) or slabs.stride(2) != 1 or slabs.stride(1) != slabs.shape[2]:
            return None
        w_dec, b_dec = self.decoder_params()
        out = _DefaultMLPFunction.apply(slabs.float(), self.encoder.weight, self.encoder.bias,
                                        w_dec, b_dec, self.value_head.weight,
                                        self.value_head.bias, self._head_cache)
        return out, self.n_logits

    def forward(self, observations):
        packed = self.forward_packed(observations)
        if packed is not None:
            out, n_act = packed
            return self.split_logits(out[:, :n_act]), out[:, n_act:n_act + 1]
        hidden, lookup = self.encode_observations(observations)
        return self.decode_actions(hidden, lookup)

    def encode_observations(self, observations):
        batch_size = observations.shape[0]
        observations = observations.view(batch_size, -1)
        return torch.relu(self.encoder(observations.float())), None

    def decode_actions(self, hidden, lookup, concat=True):
        # both heads out of ONE GEMM (same parameters, same math as two nn.Linear calls): the value head is a
        # 1-column GEMV that would otherwise re-read `hidden`
        w_dec, b_dec = self.decoder_params()
        n_act = w_dec.shape[0]
        pad = (-(n_act + 1)) % 8          # zero rows up to a multiple of 8 columns: keeps the aligned GEMM kernels
        w = torch.cat([w_dec, self.value_head.weight, hidden.new_zeros(pad, hidden.shape[1])], dim=0)
        b = torch.cat([b_dec, self.value_head.bias, hidden.new_zeros(pad)], dim=0)
        out = torch.nn.functional.linear(hidden, w, b)
        return self.split_logits(out[:, :n_act]), out[:, n_act:n_act + 1]


class LSTMWrapper(nn.Module):
    """Recurrent wrapper around a policy that defines encode_observations / decode_actions (reference:
    pufferlib/models.py:64-111): obs [B, *obs] or [B, T, *obs] -> encode -> nn.LSTM (cuDNN) over T -> decode.
    Returns (logits, value, state)."""

    def __init__(self, env, policy, input_size=128, hidden_size=128, num_layers=1):
        super().__init__()
        self.obs_shape = tuple(env.single_observation_space.shape)
        self.policy = policy
        self.input_size = input_size
        self.hidden_size = hidden_size
        self.recurrent = nn.LSTM(input_size, hidden_size, num_layers)
        for name, param in self.recurrent.named_parameters():
            if 'bias' in name:
                nn.init.constant_(param, 0)
            elif 'weight' in name:
                nn.init.orthogonal_(param, 1.0)

    def forward(self, x, state):
        nd = len(self.obs_shape)
        if tuple(x.shape[-nd:]) != self.obs_shape or x.dim() not in (nd + 1, nd + 2):
            raise ValueError('Invalid input tensor shape', x.shape)
        batch, steps = (x.shape[0], 1) if x.dim() == nd + 1 else (x.shape[0], x.shape[1])
        if state is not None:
            assert state[0].shape[1] == state[1].shape[1] == batch
        hidden, lookup = self.policy.encode_observations(x.reshape(batch * steps, *self.obs_shape))
        assert hidden.shape == (batch * steps, self.input_size)
        seq = hidden.reshape(batch, steps, self.input_size).transpose(0, 1)       # [T, B, F] for nn.LSTM
        seq, state = self.recurrent(seq, state)
        flat = seq.transpose(0, 1).reshape(batch * steps, self.hidden_size)
        logits, value = self.policy.decode_actions(flat, lookup)
        return logits, value, state


class Convolutional(nn.Module):
    def __init__(self, env, *args, framestack=4, flat_size=64 * 7 * 7, input_size=512, hidden_size=512,
                 output_size=512, channels_last=False, downsample=1, **kwargs):
        super().__init__()
        self.channels_last = channels_last
        self.downsample = downsample
        self.network = nn.Sequential(
            layer_init(nn.Conv2d(framestack, 32, 8, stride=4)), nn.ReLU(),
            layer_init(nn.Conv2d(32, 64, 4, stride=2)), nn.ReLU(),
            layer_init(nn.Conv2d(64, 64, 3, stride=1)), nn.ReLU(),
            nn.Flatten(),
            layer_init(nn.Linear(flat_size, hidden_size)), nn.ReLU(),
        )
        self.actor = layer_init(nn.Linear(output_size, env.single_action_space.n), std=0.01)
        self.value_fn = layer_init(nn.Linear(output_size, 1), std=1)

    def forward(self, observations):
        hidden, lookup = self.encode_observations(observations)
        return self.decode_actions(hidden, lookup)

    def encode_observations(self, observations):
        if self.channels_last:
            observations = observations.permute(0, 3, 1, 2)
        if self.downsample > 1:
            observations = observations[:, :, ::self.downsample, ::self.downsample]
        return self.network(observations.float() / 255.0), None

    def decode_actions(self, flat_hidden, lookup, concat=None):
        return self.actor(flat_hidden), self.value_fn(flat_hidden)
