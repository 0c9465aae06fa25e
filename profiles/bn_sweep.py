"""Sweep of the run-time knobs of the fused BatchNorm(train)+SiLU kernels (fused_mlp.cu):
CTAs per SM of the partial reductions, rows in flight per thread of the backward passes,
elements in flight of the forward apply.  CUDA events over ITERS launches on rotating buffers
(working set > L2).  Prints a table; the best setting becomes the default.

    python profiles/bn_sweep.py > gpurun_out/bn_sweep.txt
"""
import itertools
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pygho_b200  # noqa: E402,F401
from pygho_b200 import _lib, ops  # noqa: E402,F401

O = torch.ops.pygho_b200
dev = torch.device("cuda", 0)
ROWS = int(os.environ.get("ROWS", "230147"))
ITERS = int(os.environ.get("ITERS", "24"))


def tune(key, val):
    _lib.call("pgh_set_tuning", key, val)


def timeit(fn):
    for i in range(3):
        fn(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(ITERS):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / ITERS


for C in (384, 128):
    g = torch.Generator(device=dev).manual_seed(0)
    nset = 3 if C == 384 else 4
    ys = [torch.randn((ROWS, C), device=dev, generator=g) for _ in range(nset)]
    dzs = [torch.randn((ROWS, C), device=dev, generator=g) for _ in range(nset)]
    gam = torch.rand(C, device=dev) + 0.5
    bet = torch.randn(C, device=dev)
    rm, rv = torch.zeros(C, device=dev), torch.ones(C, device=dev)
    fwd_bytes = 4 * ROWS * C * 3
    bwd_bytes = 4 * ROWS * C * 5
    # reference result (default knobs) for a bit-for-bit / tolerance check of every variant
    for k in (2, 3, 5):
        tune(k, 0)
    m0, r0 = O.bn_stats(ys[0], 1e-5, 0.1, rm.clone(), rv.clone())
    z0 = O.bn_act_fwd(ys[0], m0, r0, gam, bet, 1)
    def bwd(dz, y):
        sums, dg, db = O.bn_act_bwd_reduce(dz, y, m0, r0, gam, bet, 1, None, None, None)
        dy, dbias = O.bn_act_bwd_apply(dz, y, m0, r0, gam, bet, sums, None, 1, None, True, None)
        return dy, dg, db, dbias
    dy0, dg0, db0, dbias0 = bwd(dzs[0], ys[0])
    print(f"# rows={ROWS} C={C}: fwd {fwd_bytes / 1e6:.0f} MB, bwd {bwd_bytes / 1e6:.0f} MB algorithmic")
    for bps, un in itertools.product((4, 8), (1, 2, 4)):
        tune(2, bps); tune(5, un)

        def fwd(i):
            m, r = O.bn_stats(ys[i % nset], 1e-5, 0.1, rm, rv)
            return O.bn_act_fwd(ys[i % nset], m, r, gam, bet, 1)

        z = fwd(0)
        err = float((z - z0).abs().max())
        us = timeit(fwd)
        print(f"fwd C={C} ctas/sm={bps} un={un}: {us:7.1f} us {fwd_bytes / us / 1e3:6.0f} GB/s  maxdiff {err:.1e}")
    tune(5, 0)
    for bps, un in itertools.product((4, 8), (2, 4)):
        tune(2, bps); tune(3, un)

        def bwd(i):
            return bwd(dzs[i % nset], ys[i % nset])

        dy, dg, db, dbias = bwd(0)
        err = max(float((dy - dy0).abs().max()), float((dg - dg0).abs().max() / dg0.abs().max()),
                  float((dbias - dbias0).abs().max()))
        us = timeit(bwd)
        print(f"bwd C={C} ctas/sm={bps} un={un}: {us:7.1f} us {bwd_bytes / us / 1e3:6.0f} GB/s  maxdiff {err:.1e}")
    for k in (2, 3, 5):
        tune(k, 0)
    del ys, dzs
    torch.cuda.empty_cache()
