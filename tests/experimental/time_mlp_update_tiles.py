"""Per-phase SM-clock stamps of the fused update kernel (pb_mlp_update_debug_clock): where does a tile's time go?

    python tests/experimental/time_mlp_update_tiles.py
"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import check_mlp_update_fused as cf      # noqa: E402

lib = cf.lib
dev = torch.device('cuda')
m, n_act = 524288, 4
torch.manual_seed(0)
x = torch.randn(m, 128, device=dev)
w_enc, b_enc = torch.randn(128, 128, device=dev) * 0.1, torch.randn(128, device=dev) * 0.1
w_cat = torch.zeros(8, 128, device=dev)
w_cat[:5] = torch.randn(5, 128, device=dev) * 0.1
b_cat = torch.zeros(8, device=dev)
act = torch.randint(0, n_act, (m,), device=dev)
olp = -torch.rand(m, device=dev) - 0.5
adv, ret, oval = torch.randn(m, device=dev), torch.randn(m, device=dev), torch.randn(m, device=dev)
clk = torch.zeros(148 * 18 * 4 * 8, dtype=torch.int64, device=dev)
for k in range(2):
    cf.fused(x, 128, m, m, 1, w_enc, b_enc, w_cat, b_cat, act, olp, adv, ret, oval, n_act, False)
lib.pb_mlp_update_debug_clock(cf.ptr(clk))
cf.fused(x, 128, m, m, 1, w_enc, b_enc, w_cat, b_cat, act, olp, adv, ret, oval, n_act, False)
torch.cuda.synchronize()
lib.pb_mlp_update_debug_clock(None)
c = clk.cpu().numpy().reshape(148, 18, 4, 8).astype(np.float64)
for cta in (0, 73, 147):
    t0 = c[cta, 2:, 0, 0].min()
    print(f'--- CTA {cta}: clocks relative to the first epilogue warp entering tile 8')
    print('TMA  [tile][wait xk_empty from, until]           ', np.round(c[cta, 0, :, :2] - t0).astype(int).tolist())
    print('MMA  [tile][fwd: enter, h_empty ok, xk_full ok | dp_full q0..q3 | transpose issued]')
    for it in range(4):
        print('     ', np.round(c[cta, 1, it] - t0).astype(int).tolist())
    print('EPI  warp (q,c): [enter, h_full, dp_empty, staged+heads, bar1, loss done, bar2, dp_full arrive]')
    for w in (2, 3, 4, 5, 6, 10, 14):
        q, cc = w & 3, (w - 2) >> 2
        for it in range(2):
            print(f'      w{w:2d} (q{q},c{cc}) tile {8 + it}:', np.round(c[cta, w, it] - t0).astype(int).tolist())
per = c[:, 2:, 1:, 0] - c[:, 2:, :-1, 0]
print('mean tile period (clocks) over all CTAs / epilogue warps:', per.mean(), ' min', per.min(), ' max', per.max())
seg = np.diff(c[:, 2:, :, :], axis=-1)
names = ['wait h_full', 'tmem ld + wait dp_empty', 'relu + stage + heads mma', 'bar 1', 'loss (4 lanes per row)', 'bar 2', 'g^T + dW_heads + mask + store']
for i, n in enumerate(names):
    print(f'{n:34s} mean {seg[..., i].mean():8.0f}   c==0 warps {seg[:, [2, 3, 0, 1], :, i].mean():8.0f}   others {seg[:, 4:, :, i].mean():8.0f}')
print('tail: arrive -> next tile enter', (c[:, 2:, 1:, 0] - c[:, 2:, :-1, 7]).mean())
