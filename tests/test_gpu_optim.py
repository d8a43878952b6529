"""pb_clip_adam / pb_pack_heads and the hand-written minibatch update vs their torch formulations (GPU)."""
import ctypes as C

import numpy as np
import pytest
import torch

from pufferlib_b200 import _native

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize('max_norm,world,lr_on_device', [(0.5, 1, True), (0.5, 2, False), (100.0, 1, False), (0.0, 1, True)])
def test_clip_adam_matches_torch_clip_and_adam(max_norm, world, lr_on_device):
    """clean_pufferl.py:240-244: clip_grad_norm_ + Adam(eps=1e-5).step(), five steps, six tensors of a models.Default."""
    dev = torch.device('cuda')
    torch.manual_seed(3)
    shapes = [(128, 128), (128,), (4, 128), (4,), (1, 128), (1,)]
    ours = [torch.randn(s, device=dev) * 0.1 for s in shapes]
    ref = [p.clone().requires_grad_(True) for p in ours]
    lr = 2.5e-4
    opt = torch.optim.Adam(ref, lr=torch.tensor(lr, device=dev), eps=1e-5, fused=True, capturable=True)
    state = [dict(step=torch.zeros((), device=dev), m=torch.zeros_like(p), v=torch.zeros_like(p)) for p in ours]
    lr_t = torch.tensor(lr, device=dev)
    norm_out = torch.zeros(1, device=dev)
    for it in range(5):
        grads = [torch.randn(s, device=dev) * (10.0 if it == 2 else 0.05) for s in shapes]   # it 2: clipping is active
        for p, g in zip(ref, grads):
            p.grad = (g / world).clone()
        if max_norm > 0:
            ref_norm = torch.nn.utils.clip_grad_norm_(ref, max_norm)
        else:
            ref_norm = torch.linalg.vector_norm(torch.cat([p.grad.flatten() for p in ref]))
        opt.step()
        arr = (_native.AdamTensor * 6)()
        for k in range(6):
            arr[k] = _native.AdamTensor(ours[k].data_ptr(), state[k]['m'].data_ptr(), state[k]['v'].data_ptr(),
                                        state[k]['step'].data_ptr(), grads[k].data_ptr(), ours[k].numel())
        _native.check(_native.lib().pb_clip_adam(
            arr, 6, C.c_float(max_norm), C.c_float(1.0 / world), C.c_float(0.0 if lr_on_device else lr),
            _native.ptr(lr_t) if lr_on_device else None, C.c_float(0.9), C.c_float(0.999), C.c_float(1e-5),
            _native.ptr(norm_out), _native.stream_ptr()))
        torch.cuda.synchronize()
        assert abs(float(norm_out) - float(ref_norm)) <= 1e-5 * float(ref_norm)
        for k in range(6):
            assert float(state[k]['step']) == it + 1 == float(opt.state[ref[k]]['step'])
            assert torch.allclose(state[k]['m'], opt.state[ref[k]]['exp_avg'], rtol=1e-5, atol=1e-9)
            assert torch.allclose(state[k]['v'], opt.state[ref[k]]['exp_avg_sq'], rtol=1e-5, atol=1e-12)
            # one Adam step moves a parameter by at most ~lr; agreement to 1e-3 of that
            assert float((ours[k] - ref[k].detach()).abs().max()) <= 1e-3 * lr * (it + 1), (it, k)


@pytest.mark.parametrize('world,n_parts', [(1, 275), (2, 16), (1, 1)])
def test_clip_adam_parts_matches_single_cta_kernel(world, n_parts):
    """pb_clip_adam_parts (multi-CTA, norm from partial sums of squares of the unscaled gradient) vs pb_clip_adam on the same
    gradients, several steps with and without clipping: same step counters, moments and parameters."""
    dev = torch.device('cuda')
    torch.manual_seed(3)
    shapes = [(128, 128), (128,), (4, 128), (4,), (1, 128), (1,)]
    pa = [torch.randn(s, device=dev) * 0.1 for s in shapes]
    pb = [p.clone() for p in pa]
    mk = lambda ps: [dict(step=torch.zeros((), device=dev), m=torch.zeros_like(p), v=torch.zeros_like(p)) for p in ps]
    sa, sb = mk(pa), mk(pb)
    lib = _native.lib()
    na, nb = torch.zeros(1, device=dev), torch.zeros(1, device=dev)
    for it in range(4):
        flat = torch.randn(sum(int(np.prod(s)) for s in shapes), device=dev) * (10.0 if it == 1 else 0.05)
        grads, off = [], 0
        for s in shapes:
            k = int(np.prod(s))
            grads.append(flat[off:off + k])
            off += k
        chunks = torch.tensor_split(flat.double(), n_parts)
        parts = torch.stack([(c * c).sum() for c in chunks])
        for ps, st, norm, use_parts in ((pa, sa, na, False), (pb, sb, nb, True)):
            arr = (_native.AdamTensor * 6)()
            for k in range(6):
                arr[k] = _native.AdamTensor(ps[k].data_ptr(), st[k]['m'].data_ptr(), st[k]['v'].data_ptr(),
                                            st[k]['step'].data_ptr(), grads[k].data_ptr(), ps[k].numel())
            hyper = (C.c_float(0.5), C.c_float(1.0 / world), C.c_float(2.5e-4), None, C.c_float(0.9), C.c_float(0.999),
                     C.c_float(1e-5), _native.ptr(norm))
            if use_parts:
                _native.check(lib.pb_clip_adam_parts(arr, 6, *hyper, _native.ptr(parts), n_parts, None, None, _native.stream_ptr()))
            else:
                _native.check(lib.pb_clip_adam(arr, 6, *hyper, _native.stream_ptr()))
        torch.cuda.synchronize()
        assert abs(float(na) - float(nb)) <= 1e-6 * float(na)
        for k in range(6):
            assert float(sa[k]['step']) == float(sb[k]['step']) == it + 1
            assert torch.allclose(sa[k]['m'], sb[k]['m'], rtol=1e-5, atol=1e-10)
            assert torch.allclose(sa[k]['v'], sb[k]['v'], rtol=1e-5, atol=1e-12)
            assert float((pa[k] - pb[k]).abs().max()) <= 1e-7


@pytest.mark.parametrize('n_act,features', [(4, 128), (7, 49), (1, 300)])
def test_pack_heads_matches_torch_construction(n_act, features):
    dev = torch.device('cuda')
    torch.manual_seed(n_act)
    hid = 128
    w_dec, b_dec = torch.randn(n_act, hid, device=dev), torch.randn(n_act, device=dev)
    w_val, b_val = torch.randn(1, hid, device=dev), torch.randn(1, device=dev)
    w_enc = torch.randn(hid, features, device=dev) * 3
    w_cat, b_cat = torch.full((8, hid), 9.0, device=dev), torch.full((8,), 9.0, device=dev)
    w_tf = torch.empty_like(w_enc)
    _native.check(_native.lib().pb_pack_heads(_native.ptr(w_dec), _native.ptr(b_dec), _native.ptr(w_val),
                                              _native.ptr(b_val), n_act, hid, _native.ptr(w_cat), _native.ptr(b_cat),
                                              _native.ptr(w_enc), _native.ptr(w_tf), w_enc.numel(), _native.stream_ptr()))
    ref_w = torch.zeros(8, hid, device=dev)
    ref_w[:n_act], ref_w[n_act] = w_dec, w_val[0]
    ref_b = torch.zeros(8, device=dev)
    ref_b[:n_act], ref_b[n_act] = b_dec, b_val[0]
    assert torch.equal(w_cat, ref_w) and torch.equal(b_cat, ref_b)
    bits = w_enc.view(torch.int32)
    assert torch.equal(w_tf, ((bits + 0x1000) & ~0x1FFF).view(torch.float32))      # round to nearest, ties away


def test_manual_update_matches_autograd_update():
    """train() through the hand-written update chain (_DefaultMLPUpdate: pb_ppo_loss -> pb_mlp_tail_backward -> split-K
    dW -> pb_clip_adam) vs the autograd + clip_grad_norm_ + torch.optim.Adam path: same rollout, parameters after the
    first update agree to 2e-5, the reported losses to 1e-4."""
    import pufferlib_b200.vector as pvec
    from pufferlib_b200 import clean_pufferl, models
    from pufferlib_b200.environments import ocean
    from pufferlib_b200.frameworks import cleanrl
    from test_gpu_experience import make_config
    n, h = 64, 32
    params, losses, used, states = {}, {}, {}, {}
    for manual in (True, False):
        vec = pvec.make(ocean.env_creator('breakout'), num_envs=n, backend=pvec.B200)
        torch.manual_seed(0)
        pol = cleanrl.Policy(models.Default(vec.driver_env), fused_sample=True, seed=7).cuda()
        data = clean_pufferl.create(make_config(n, h, env='breakout', manual_update=manual, fused_update=False), vec, pol)
        clean_pufferl.evaluate(data)
        clean_pufferl.train(data)
        params[manual] = [p.detach().cpu().clone() for p in pol.parameters()]
        losses[manual] = np.array([data.losses.policy_loss, data.losses.value_loss, data.losses.entropy,
                                   data.losses.approx_kl, data.losses.clipfrac, data.losses.explained_variance])
        used[manual] = data.manual_update is not None
        states[manual] = [float(data.optimizer.state[p]['step']) for p in pol.parameters()]
        clean_pufferl.evaluate(data)              # the rollout after the update runs on the updated heads
        clean_pufferl.train(data)
        assert np.isfinite(data.losses.policy_loss)
        clean_pufferl.close(data)
    assert used[True] and not used[False]
    assert states[True] == states[False] == [4.0] * 6            # update_epochs 2 x 2 minibatches
    diff = max(float((a - b).abs().max()) for a, b in zip(params[True], params[False]))
    assert diff <= 2e-5, diff
    assert np.allclose(losses[True], losses[False], rtol=1e-4, atol=1e-6), (losses[True], losses[False])


def test_fused_update_kernel_matches_kernel_chain():
    """train() through pb_mlp_update_fused (ONE tcgen05 kernel per minibatch: csrc/mlp_update.cu) vs the kernel chain it
    replaces (cuBLAS GEMMs + pb_ppo_loss + pb_mlp_tail_backward + split-K dW): same rollout, same minibatches.  Both
    compute the dense products in TF32 (operands truncated by the tensor core), so gradients agree to TF32 noise; the
    statistics come from the same row math."""
    import pufferlib_b200.vector as pvec
    from pufferlib_b200 import clean_pufferl, models
    from pufferlib_b200.environments import ocean
    from pufferlib_b200.frameworks import cleanrl
    from test_gpu_experience import make_config
    n, h = 256, 32          # 2 minibatches of 4096 rows = 32 tiles of 128 rows; slabs of bptt * n = 2048 rows
    grads, losses, params, used = {}, {}, {}, {}
    for fused in (True, False):
        vec = pvec.make(ocean.env_creator('breakout'), num_envs=n, backend=pvec.B200)
        torch.manual_seed(0)
        pol = cleanrl.Policy(models.Default(vec.driver_env), fused_sample=True, seed=7).cuda()
        cfg = make_config(n, h, env='breakout', manual_update=True, fused_update=fused)
        cfg.update_epochs = 1
        cfg.minibatch_size = n * h          # ONE minibatch: gflat after train() is its gradient
        data = clean_pufferl.create(cfg, vec, pol)
        clean_pufferl.evaluate(data)
        clean_pufferl.train(data)
        mu = data.manual_update
        used[fused] = mu.used_fused
        grads[fused] = mu.gflat.detach().cpu().clone()
        params[fused] = torch.cat([p.detach().reshape(-1).cpu() for p in pol.parameters()])
        losses[fused] = np.array([data.losses.policy_loss, data.losses.value_loss, data.losses.entropy,
                                  data.losses.approx_kl, data.losses.clipfrac])
        clean_pufferl.evaluate(data)
        clean_pufferl.train(data)
        assert np.isfinite(data.losses.policy_loss)
        clean_pufferl.close(data)
    assert used[True] and not used[False]
    ga, gb = grads[True], grads[False]
    sections = {'dW_enc': slice(0, 128 * 128), 'dW_heads': slice(128 * 128, 128 * 128 + 1024),
                'db_enc': slice(128 * 128 + 1024, 128 * 128 + 1152), 'db_heads': slice(128 * 128 + 1152, None)}
    for name, sl in sections.items():
        err = float((ga[sl] - gb[sl]).abs().max()) / (float(gb[sl].abs().max()) + 1e-30)
        # both paths take TF32 operands in every product (torch 'high' precision, clean_pufferl.py:22) but round at different
        # places (cuBLAS rounds, the tensor core truncates), and a TF32-sized change of a logit moves a few of the 8192 rows
        # across the clipping boundaries of the loss
        assert err < 1.5e-2, (name, err)
    # the value loss of a freshly initialised policy differs by ~1 % for the same reason
    assert np.allclose(losses[True], losses[False], rtol=3e-2, atol=1e-6), (losses[True], losses[False])
    # one Adam step of size lr = 2.5e-4 from nearly identical gradients
    assert float((params[True] - params[False]).abs().max()) < 2.5e-4
    assert float((params[True] - params[False]).abs().mean()) < 2e-6


def test_fused_update_kernel_inside_train_graph():
    """The fused update inside the captured train graph (tensor-map kernel parameters) replays to the same parameters as
    eager execution."""
    import pufferlib_b200.vector as pvec
    from pufferlib_b200 import clean_pufferl, models
    from pufferlib_b200.environments import ocean
    from pufferlib_b200.frameworks import cleanrl
    from test_gpu_experience import make_config
    n, h = 128, 32
    out = {}
    for graph in (False, True):
        vec = pvec.make(ocean.env_creator('breakout'), num_envs=n, backend=pvec.B200)
        torch.manual_seed(0)
        pol = cleanrl.Policy(models.Default(vec.driver_env), fused_sample=True, seed=7).cuda()
        cfg = make_config(n, h, env='breakout', manual_update=True, fused_update=True, cuda_graph_train=graph,
                          cuda_graph_rollout=False)
        data = clean_pufferl.create(cfg, vec, pol)
        for _ in range(3):
            clean_pufferl.evaluate(data)
            clean_pufferl.train(data)
        assert data.manual_update.used_fused
        assert (data.train_graph_state == 2) == graph
        out[graph] = torch.cat([p.detach().reshape(-1).cpu() for p in pol.parameters()])
        clean_pufferl.close(data)
    # same program, eager vs replayed: identical up to the GAE look-back's run-to-run fp32 noise (see
    # test_graphed_training_matches_eager_training)
    assert float((out[True] - out[False]).abs().max()) < 1e-4
