"""CUDA-event timings of the MultiDiscrete path: pb_sample_logits_multi (M = 16384 rows, the rollout-step size of a
16k-env run), pb_ppo_loss_multi (M = 524288, a C2-size minibatch) and the `spaces` env step (N = 65536), each with the
bytes it moves (from shapes) and the time a device-to-device copy of the same byte count takes in the same run.

    python profiles/tools/time_multidiscrete.py --out profiles/multidiscrete_b200.json

Needs a CUDA device; the card name and power limit are read in the same run and stored with the numbers."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import pufferlib_b200.vector as pvec  # noqa: E402
from pufferlib_b200 import _native  # noqa: E402
from pufferlib_b200.environments import ocean  # noqa: E402


def time_ms(fn, iters):
    for _ in range(10):
        fn()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for _ in range(iters):
        fn()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / iters


def copy_ms(nbytes, iters):
    """A D2D copy that moves nbytes in total (nbytes / 2 read + nbytes / 2 written)."""
    half = max(16, nbytes // 2)
    src = torch.empty(half, dtype=torch.uint8, device='cuda')
    dst = torch.empty_like(src)
    return time_ms(lambda: dst.copy_(src), iters)


def entry(name, ms, nbytes, iters, **shape):
    c = copy_ms(nbytes, iters)
    return dict(name=name, ms=ms, bytes=nbytes, gb_per_s=nbytes / ms / 1e6, copy_ms=c, fraction_of_copy=c / ms,
                iters=iters, **shape)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--iters', type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device')
    lib, dev, it = _native.lib(), torch.device('cuda'), args.iters
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()
    results = []
    nvec = [2, 2]
    k, s_ = len(nvec), sum(nvec)
    nv = (C.c_int32 * k)(*nvec)

    # sampling: packed [M, 8] head output (2 + 2 logits | value | pad), rollout-row stores as in Policy
    m = 16384
    out = torch.randn(m, 8, device=dev)
    acts = torch.empty(m, k, dtype=torch.int64, device=dev)
    lp, ent, vrow = (torch.empty(m, device=dev) for _ in range(3))
    counter = torch.zeros(1, dtype=torch.int64, device=dev)

    def sample():
        _native.check(lib.pb_sample_logits_multi(
            _native.ptr(out), 8, m, nv, k, C.c_uint64(1), C.c_uint64(0), _native.ptr(counter), _native.ptr(acts),
            _native.ptr(lp), _native.ptr(ent), C.c_void_p(out.data_ptr() + 4 * s_), 8, _native.ptr(vrow), None, None,
            _native.stream_ptr()))
    results.append(entry('pb_sample_logits_multi', time_ms(sample, it), m * (4 * s_ + 4) + m * (8 * k + 12), it,
                         rows=m, nvec=nvec))

    # loss: packed rows, gradient back into a packed [M, 8] buffer
    m = 524288
    out = torch.randn(m, 8, device=dev)
    acts = torch.randint(0, 2, (m, k), device=dev)
    old_lp, adv, ret, old_v = (torch.randn(m, device=dev) for _ in range(4))
    grad = torch.empty_like(out)
    stats = torch.empty(8, dtype=torch.float64, device=dev)

    def loss():
        _native.check(lib.pb_ppo_loss_multi(
            _native.ptr(out), 8, C.c_void_p(out.data_ptr() + 4 * s_), 8, _native.ptr(acts), _native.ptr(old_lp),
            _native.ptr(adv), _native.ptr(ret), _native.ptr(old_v), m, nv, k, C.c_float(0.1), 1, C.c_float(0.1),
            C.c_float(0.5), C.c_float(0.01), _native.ptr(grad), 8, C.c_void_p(grad.data_ptr() + 4 * s_), 8,
            _native.ptr(stats), _native.stream_ptr()))
    results.append(entry('pb_ppo_loss_multi', time_ms(loss, it), m * (32 + 8 * k + 16) + m * 32, it, rows=m, nvec=nvec))

    # env step: reset and step rows alternate, so one timed unit is a (reset send, step send) pair
    n = 65536
    vec = pvec.make(ocean.env_creator('spaces'), num_envs=n, backend=pvec.B200)
    vec.async_reset(1)
    vec.recv()
    a = torch.randint(0, 2, (n, k), device=dev)

    def two_steps():
        for _ in range(2):
            vec.flag = pvec.SEND
            vec.send(a)
    per_env = (8 * k + 4 + 1) + (108 + 4 + 1 + 1 + 1 + 1 + 4 + 4)   # read actions/k/done; write obs..dones_f32, k, done
    ms = time_ms(two_steps, it) / 2
    results.append(entry('spaces env step', ms, n * per_env, it, envs=n,
                         note='mean of a reset send and a step send; episode-stat stores not counted'))
    vec.close()

    doc = dict(gpu=smi, torch=torch.__version__, results=results)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(doc, indent=1))


if __name__ == '__main__':
    main()
