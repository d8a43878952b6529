"""Hardware check of the fused tcgen05 minibatch-update kernel (csrc/mlp_update.cu).

Stage-wise: every stage's reference is computed from the kernel's OWN previous-stage dump (hidden -> dOut -> dPre ->
gradients), so a mismatch names the stage that is wrong; then an end-to-end comparison against the validated chain
(cuBLAS GEMMs + pb_ppo_loss + pb_mlp_tail_backward + dW GEMM), then timing at the bench minibatch.  Not collected by
pytest; run on a B200 box under a timeout:

    gpurun --timeout 300 -- 'timeout 200 python tests/experimental/check_mlp_update_fused.py'
"""
import ctypes as C
import os
import sys

import torch

REPO = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, REPO)
from pufferlib_b200 import _native  # noqa: E402

lib = _native.lib()
CFG = (0.1, 1, 0.1, 0.5, 0.01)      # clip, clip_vloss, vclip, vf_coef, ent_coef


def ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def trunc_tf32(t):
    return (t.contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)


def rna_tf32(t):
    return ((t.contiguous().view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)


def fused(xbuf, ldx, slab_rows, slab_stride, n_slabs, w_enc, b_enc, w_cat, b_cat, act, olp, adv, ret, oval, n_act, debug):
    dev = xbuf.device
    m = slab_rows * n_slabs
    gflat = torch.full((128 * 128 + 8 * 128 + 128 + 8,), float('nan'), device=dev)
    stats = torch.zeros(8, dtype=torch.float64, device=dev)
    ws = torch.empty(lib.pb_mlp_update_workspace_bytes(), dtype=torch.uint8, device=dev)
    dh = dp = do = None
    if debug:
        dh = torch.full((m, 128), float('nan'), device=dev)
        dp = torch.full((m, 128), float('nan'), device=dev)
        do = torch.full((m, 8), float('nan'), device=dev)
    _native.check(lib.pb_mlp_update_fused(ptr(xbuf), ldx, slab_rows, slab_stride, n_slabs, ptr(w_enc), ptr(b_enc), ptr(w_cat), ptr(b_cat),
                                  ptr(act), ptr(olp), ptr(adv), ptr(ret), ptr(oval), None, slab_rows, n_act, CFG[0], CFG[1], CFG[2], CFG[3],
                                  CFG[4], ptr(gflat), ptr(stats), ptr(ws), ws.numel(), None, ptr(dh), ptr(dp), ptr(do),
                                  C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return gflat, stats, dh, dp, do


def ppo_loss(out, act, olp, adv, ret, oval, n_act):
    lib, s = _native.lib(), _native.stream_ptr()
    m = out.shape[0]
    dout = torch.empty_like(out)
    stats = torch.empty(8, dtype=torch.float64, device=out.device)
    o, d = out.data_ptr(), dout.data_ptr()
    _native.check(lib.pb_ppo_loss(C.c_void_p(o), 8, C.c_void_p(o + 4 * n_act), 8, ptr(act), ptr(olp), ptr(adv), ptr(ret),
                                  ptr(oval), m, n_act, C.c_float(CFG[0]), CFG[1], C.c_float(CFG[2]), C.c_float(CFG[3]),
                                  C.c_float(CFG[4]), C.c_void_p(d), 8, C.c_void_p(d + 4 * n_act), 8, ptr(stats), s))
    return dout, stats


def rel(a, b):
    return float((a.double() - b.double()).abs().max()) / (float(b.double().abs().max()) + 1e-30)


def check(name, a, b, tol):
    e = rel(a, b)
    print(f'    {name:34s} max err / max|ref| = {e:.3e}  {"ok" if e <= tol else "MISMATCH"}', flush=True)
    return e <= tol


def case(slab_rows, n_slabs, slab_stride, n_act, seed):
    dev = torch.device('cuda')
    torch.manual_seed(seed)
    m = slab_rows * n_slabs
    total_rows = (n_slabs - 1) * slab_stride + slab_rows
    xbuf = torch.randn(total_rows + 64, 128, device=dev)          # rows between / after the slabs hold unrelated data
    w_enc = torch.randn(128, 128, device=dev) * 0.1
    b_enc = torch.randn(128, device=dev) * 0.1
    w_cat = torch.zeros(8, 128, device=dev)
    w_cat[:n_act + 1] = torch.randn(n_act + 1, 128, device=dev) * 0.1
    b_cat = torch.zeros(8, device=dev)
    b_cat[:n_act + 1] = torch.randn(n_act + 1, device=dev) * 0.1
    act = torch.randint(0, n_act, (m,), device=dev)
    olp = -torch.rand(m, device=dev) - 0.5
    adv, ret, oval = torch.randn(m, device=dev), torch.randn(m, device=dev), torch.randn(m, device=dev)
    x = torch.cat([xbuf[s * slab_stride:s * slab_stride + slab_rows] for s in range(n_slabs)])       # slab-major rows
    print(f'case slab_rows={slab_rows} n_slabs={n_slabs} stride={slab_stride} n_act={n_act} (M={m})', flush=True)
    gflat, stats, dh, dp, do = fused(xbuf, 128, slab_rows, slab_stride, n_slabs, w_enc, b_enc, w_cat, b_cat, act, olp, adv,
                                     ret, oval, n_act, debug=True)
    torch.cuda.synchronize()
    ok = True
    # stage 1: forward UMMA (TF32 = truncated operands, fp32 accumulate) + bias + ReLU
    h_ref = torch.relu(trunc_tf32(x).double() @ trunc_tf32(w_enc).double().t() + b_enc.double())
    ok &= check('hidden (forward UMMA)', dh, h_ref, 2e-5)
    # stage 2: heads + loss from the kernel's own hidden.  The epilogue's products (mma.sync) take TF32 operands like torch
    # 'high': hidden / dOut truncated (the raw fp32 bits), W_heads rounded to nearest (cvt.rna), fp32 accumulation
    out = (trunc_tf32(dh).double() @ rna_tf32(w_cat).double().t() + b_cat.double()).float()
    dout_ref, stats_ref = ppo_loss(out, act, olp, adv, ret, oval, n_act)
    ok &= check('dOut (heads + PPO loss)', do, dout_ref, 2e-4)
    ok &= check('loss statistics', stats[:6], stats_ref[:6], 2e-3)
    # stage 3: dPre from the kernel's own dOut and hidden
    dpre_ref = (trunc_tf32(do).double() @ rna_tf32(w_cat).double()) * (dh > 0)
    ok &= check('dPre', dp, dpre_ref, 1e-5)
    # stage 4: gradients from the kernel's own dPre / dOut / hidden
    dw_enc = gflat[:128 * 128].view(128, 128)
    tail = gflat[128 * 128:]
    dw_heads, db_enc, db_heads = tail[:1024].view(8, 128), tail[1024:1152], tail[1152:]
    ok &= check('dW_enc (TS UMMA on x^T)', dw_enc, trunc_tf32(dp).double().t() @ trunc_tf32(x).double(), 2e-5)
    ok &= check('dW_heads (mma.sync)', dw_heads, trunc_tf32(do).double().t() @ trunc_tf32(dh).double(), 2e-5)
    ok &= check('db_enc', db_enc, dp.double().sum(0), 2e-5)
    ok &= check('db_heads', db_heads, do.double().sum(0), 2e-5)
    # end to end against plain fp32 math (TF32-level agreement)
    h32 = torch.relu(x.double() @ w_enc.double().t() + b_enc.double())
    out32 = (h32 @ w_cat.double().t() + b_cat.double()).float()
    dout32, _ = ppo_loss(out32, act, olp, adv, ret, oval, n_act)
    dpre32 = (dout32.double() @ w_cat.double()) * (h32 > 0)
    ok &= check('dW_enc vs fp64 chain (TF32 tol)', dw_enc, dpre32.t() @ x.double(), 5e-3 if m > 30000 else 5e-2)
    ok &= check('dW_heads vs fp64 chain (TF32 tol)', dw_heads, dout32.double().t() @ h32, 5e-3)
    # the same launch without the debug dumps must give the same gradients
    g2, s2, _, _, _ = fused(xbuf, 128, slab_rows, slab_stride, n_slabs, w_enc, b_enc, w_cat, b_cat, act, olp, adv, ret, oval,
                            n_act, debug=False)
    torch.cuda.synchronize()
    ok &= check('repeat launch (no dumps)', g2, gflat, 1e-6)
    return ok


def timing():
    dev = torch.device('cuda')
    m, n_act = 524288, 4
    torch.manual_seed(0)
    xbuf = torch.randn(4 * m, 128, device=dev)      # the 1 GiB rollout: two slabs of a minibatch are 2 M rows apart
    w_enc = torch.randn(128, 128, device=dev) * 0.1
    b_enc = torch.randn(128, device=dev) * 0.1
    w_cat = torch.zeros(8, 128, device=dev)
    w_cat[:n_act + 1] = torch.randn(n_act + 1, 128, device=dev) * 0.1
    b_cat = torch.zeros(8, device=dev)
    act = torch.randint(0, n_act, (m,), device=dev)
    olp = -torch.rand(m, device=dev) - 0.5
    adv, ret, oval = torch.randn(m, device=dev), torch.randn(m, device=dev), torch.randn(m, device=dev)
    for name, (rows, slabs, stride) in (('1 slab of 524288 rows', (m, 1, m)), ('2 slabs of 262144 rows', (m // 2, 2, 2 * m))):
        def fn(k):
            off = (k % 4) * (m // 2) if slabs == 2 else (k % 4) * m
            return fused(xbuf[off:], 128, rows, stride, slabs, w_enc, b_enc, w_cat, b_cat, act, olp, adv, ret, oval, n_act, False)
        for k in range(3):
            fn(k)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(16):
            fn(k)
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1000 / 16
        print(f'fused update, {name}: {us:8.1f} us / minibatch   x read at {m * 512 / us / 1e3:7.1f} GB/s', flush=True)


def main():
    ok = True
    for args in ((128, 1, 128, 4, 1), (1000, 1, 1000, 4, 2), (148 * 128 * 2 + 77, 1, 148 * 128 * 2 + 77, 7, 3),
                 (300, 2, 1000, 1, 4), (4096, 4, 16384, 4, 5)):
        ok &= case(*args)
    print('ALL OK' if ok else 'SOME MISMATCH', flush=True)
    timing()
    print('done')


if __name__ == '__main__':
    main()
