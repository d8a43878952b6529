"""pb_gae (CUDA affine suffix scan) vs the oracle restatement of c_gae.compute_gae and the reference's goldens.

Tolerance (north_star): fp32 GAE/returns within 1e-5 relative; the scan reorders the fp32 chain, nothing else."""
import numpy as np
import pytest

from oracle import gae as ogae
from util_gpu import gae_device, gae_tolerance_check, sorted_from_time_major

pytestmark = pytest.mark.gpu


def make_inputs(h, n, seed, p_done=0.01):
    rng = np.random.default_rng(seed)
    r = rng.standard_normal((h, n)).astype(np.float32)
    v = rng.standard_normal((h, n)).astype(np.float32)
    d = (rng.random((h, n)) < p_done).astype(np.float32)
    return r, v, d


def check_case(h, n, seed, p_done, gamma, lam):
    r, v, d = make_inputs(h, n, seed, p_done)
    adv, ret = gae_device(r, v, d, gamma, lam)
    rs, vs, ds = (sorted_from_time_major(x) for x in (r, v, d))
    ref32 = ogae.compute_gae(ds, vs, rs, gamma, lam)
    ref64 = ogae.compute_gae_f64(ds, vs, rs, gamma, lam)
    gae_tolerance_check(adv, ref32, ref64)
    assert adv[-1] == 0.0                                   # A[B-1] = 0 (c_gae.pyx:15,24)
    assert np.allclose(ret, adv + vs, rtol=0, atol=1e-6)


def gae_golden_inputs(n, seed, p_done):
    rng = np.random.default_rng(seed)
    rewards = rng.standard_normal(n).astype(np.float32)
    values = rng.standard_normal(n).astype(np.float32)
    dones = (rng.random(n) < p_done).astype(np.float32)
    return dones, values, rewards


def test_gae_golden_flat(golden):
    """The reference's own outputs (flat signature: one env, horizon = batch)."""
    g = golden('gae')
    for k in range(int(g['num_cases'])):
        n, seed, p, gamma, lam = g[f'case{k}_meta']
        n = int(n)
        d, v, r = gae_golden_inputs(n, int(seed), p)
        adv, _ = gae_device(r.reshape(n, 1), v.reshape(n, 1), d.reshape(n, 1), gamma, lam)
        ref = g[f'case{k}_adv']
        ref64 = ogae.compute_gae_f64(d, v, r, gamma, lam)
        gae_tolerance_check(adv, ref, ref64)


@pytest.mark.parametrize('h,n', [(128, 64), (128, 16384), (1, 1), (1, 7), (5, 1), (3, 64), (41, 5), (17, 33),
                                 (256, 96), (100, 200), (2048, 3), (1024, 16), (4, 70000), (5000, 1), (8, 513),
                                 (128, 33), (256, 17), (512, 40), (128, 2), (512, 1000), (128, 15), (256, 16)])
def test_gae_shapes(h, n):
    check_case(h, n, seed=h * 1000 + n, p_done=0.02, gamma=0.99, lam=0.95)


@pytest.mark.parametrize('p_done,gamma,lam', [(0.0, 0.99, 0.95), (1.0, 0.99, 0.95), (0.0, 1.0, 1.0), (0.3, 0.9, 0.5),
                                              (0.001, 0.999, 0.99)])
def test_gae_chain_regimes(p_done, gamma, lam):
    """gamma = lambda = 1 with no dones never zeroes the slope: the look-back must walk every tile."""
    check_case(128, 4096, seed=11, p_done=p_done, gamma=gamma, lam=lam)


def test_gae_cross_env_chain_matters():
    """The reference chain crosses env boundaries (clean_pufferl.py:167 TODO): env e's last row bootstraps from
    env e+1's first row.  A per-env scan would differ; ours must not."""
    h, n = 4, 3
    r, v, d = make_inputs(h, n, seed=5, p_done=0.0)
    adv, _ = gae_device(r, v, d, 1.0, 1.0)
    rs, vs, ds = (sorted_from_time_major(x) for x in (r, v, d))
    ref = ogae.compute_gae_np(ds, vs, rs, 1.0, 1.0)
    assert np.allclose(adv, ref, rtol=1e-5, atol=1e-5)
    per_env_last = np.zeros(n)                      # what an independent per-env scan would give at t = H-1
    assert not np.allclose(adv.reshape(n, h)[:-1, -1], per_env_last[:-1])


def test_gae_c2_full_size():
    check_case(128, 16384, seed=0, p_done=0.01, gamma=0.99, lam=0.95)


def test_gae_c3_full_size_properties():
    """C3 size (B = 16.7M): oracle comparison plus size-independent properties (linearity in rewards with dones
    and values fixed at 0: A(r1 + r2) = A(r1) + A(r2))."""
    h, n = 256, 65536
    check_case(h, n, seed=3, p_done=0.01, gamma=0.99, lam=0.95)
    rng = np.random.default_rng(9)
    r1 = rng.standard_normal((h, n)).astype(np.float32)
    r2 = rng.standard_normal((h, n)).astype(np.float32)
    z = np.zeros((h, n), dtype=np.float32)
    d = (rng.random((h, n)) < 0.01).astype(np.float32)
    a1, _ = gae_device(r1, z, d, 0.99, 0.95, want_returns=False)
    a2, _ = gae_device(r2, z, d, 0.99, 0.95, want_returns=False)
    a12, _ = gae_device(r1 + r2, z, d, 0.99, 0.95, want_returns=False)
    assert np.allclose(a12, a1 + a2, rtol=1e-4, atol=1e-4)


def test_gae_argument_errors():
    import ctypes as C
    import torch
    from pufferlib_b200 import _native
    from pufferlib_b200.exceptions import APIUsageError
    x = torch.zeros(16, device='cuda')
    with pytest.raises(APIUsageError):
        _native.check(_native.lib().pb_gae(_native.ptr(x), _native.ptr(x), _native.ptr(x), _native.ptr(x), None, 4, 4,
                                           C.c_float(0.99), C.c_float(0.95), None, 0, _native.stream_ptr()))
    # empty batch is a no-op
    _native.check(_native.lib().pb_gae(None, None, None, None, None, 0, 0, C.c_float(0.99), C.c_float(0.95), None, 0,
                                       _native.stream_ptr()))


def test_gae_vs_reference_compiled_c_gae(golden):
    """pb_gae against the reference's OWN c_gae.pyx: its outputs on these inputs are stored in c_gae_cases.npz by
    generate.py, whole or, for the two larger cases, at a fixed sample of positions (idx)."""
    g = golden('c_gae_cases')
    for h, n, p_done, gamma, lam in ((128, 64, 0.02, 0.99, 0.95), (256, 1024, 0.01, 0.99, 0.95), (4096, 1, 0.05, 0.9, 0.8),
                                     (16, 333, 0.2, 1.0, 1.0), (128, 16384, 0.01, 0.99, 0.95)):
        r, v, d = make_inputs(h, n, seed=7 * h + n, p_done=p_done)
        adv, ret = gae_device(r, v, d, gamma, lam)
        rs, vs, ds = (sorted_from_time_major(x) for x in (r, v, d))
        idx, ref = g[f'gpu_{h}x{n}_idx'], g[f'gpu_{h}x{n}_adv']
        ref64 = ogae.compute_gae_f64(ds, vs, rs, gamma, lam)
        gae_tolerance_check(adv[idx], ref, ref64[idx])


@pytest.mark.parametrize('h,n', [(128, 64), (128, 36), (256, 1024), (512, 40), (128, 16384)])
def test_gae_time_major_output_and_slab_statistics(h, n):
    """pb_gae_tm: the arrival-order (time-major) advantages are the sorted-order ones transposed, bit for bit; and
    pb_adv_stats_slabs gives the (mean, 1/(std+1e-8)) of clean_pufferl.py:211-213 for the zero-copy slab minibatches."""
    import ctypes as C
    import torch
    from pufferlib_b200 import _native, clean_pufferl
    lib = _native.lib()
    assert lib.pb_gae_time_major_supported(n, h) == 1 and lib.pb_gae_time_major_supported(n, h + 1) == 0
    r, v, d = make_inputs(h, n, seed=h + n, p_done=0.02)
    dev = torch.device('cuda')
    tr, tv, td = (torch.as_tensor(x, device=dev) for x in (r, v, d))
    adv = torch.full((n * h,), float('nan'), device=dev)
    adv_tm = torch.full((n * h,), float('nan'), device=dev)
    ws = torch.zeros(lib.pb_gae_workspace_bytes(n, h), dtype=torch.uint8, device=dev)
    for sorted_out in (adv, None):       # with and without the sorted output
        adv_tm.fill_(float('nan'))
        _native.check(lib.pb_gae_tm(_native.ptr(tr), _native.ptr(tv), _native.ptr(td), _native.ptr(sorted_out), None,
                                    _native.ptr(adv_tm), n, h, C.c_float(0.99), C.c_float(0.95), _native.ptr(ws), ws.numel(),
                                    _native.stream_ptr()))
        torch.cuda.synchronize()
        a_sorted = adv.cpu().numpy().reshape(n, h)
        assert np.array_equal(adv_tm.cpu().numpy().reshape(h, n).view(np.uint32), a_sorted.T.view(np.uint32))
    ref = ogae.compute_gae(sorted_from_time_major(d), sorted_from_time_major(v), sorted_from_time_major(r), 0.99, 0.95)
    ref64 = ogae.compute_gae_f64(sorted_from_time_major(d), sorted_from_time_major(v), sorted_from_time_major(r), 0.99, 0.95)
    gae_tolerance_check(adv.cpu().numpy(), ref, ref64)
    # slab statistics: minibatch mb = time windows k = mb, mb + nm, ... of bptt steps (all envs)
    bptt, nm = 16, 4
    g_, r_ = clean_pufferl.slab_layout(n, h, nm, bptt)
    norm = torch.zeros(nm, 2, device=dev)
    ws2 = torch.zeros(max(16, lib.pb_adv_norm_workspace_bytes(nm, g_ * r_)), dtype=torch.uint8, device=dev)
    _native.check(lib.pb_adv_stats_slabs(_native.ptr(adv_tm), r_, g_, nm, _native.ptr(norm), _native.ptr(ws2), ws2.numel(),
                                         _native.stream_ptr()))
    torch.cuda.synchronize()
    rows = clean_pufferl.slab_row_index(n, h, nm, bptt)
    a = adv_tm.cpu().numpy().astype(np.float64)
    got = norm.cpu().numpy()
    for mb in range(nm):
        x = a[rows[mb]]
        assert np.isclose(got[mb, 0], x.mean(), rtol=1e-5, atol=1e-7)
        assert np.isclose(got[mb, 1], 1.0 / (x.std(ddof=1) + 1e-8), rtol=1e-5)


@pytest.mark.parametrize('h,n', [(128, 64), (128, 36), (128, 16384), (256, 96), (256, 4096), (512, 40), (512, 1000)])
def test_gae_tile_kernel_variants_agree(h, n):
    """k_gae_tile (double-buffered, coalesced outputs; default) and the round-1 k_gae_fast are the same arithmetic: the
    element maps are identical, only the tile look-back may compose in a different order run to run -> compare to 1e-6."""
    from pufferlib_b200 import _native
    lib = _native.lib()
    r, v, d = make_inputs(h, n, seed=3 * h + n, p_done=0.02)
    out = {}
    try:
        for variant in (1, 2):
            _native.check(lib.pb_gae_set_variant(variant))
            out[variant] = gae_device(r, v, d, 0.99, 0.95)
    finally:
        lib.pb_gae_set_variant(0)
    for k in (0, 1):
        assert np.allclose(out[1][k], out[2][k], rtol=1e-6, atol=1e-6)
    rs, vs, ds = (sorted_from_time_major(x) for x in (r, v, d))
    gae_tolerance_check(out[2][0], ogae.compute_gae(ds, vs, rs, 0.99, 0.95), ogae.compute_gae_f64(ds, vs, rs, 0.99, 0.95))
