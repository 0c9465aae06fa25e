"""Time evaluation (BatchNorm in eval mode, no autograd) of the tuplewise MLP and of the model.

Per block, at 230 147 rows (the tuple count of 1024 ZINC-shaped graphs), with TF32 allowed as in
the reference: the module path (``nn.Linear`` -> ``nn.BatchNorm1d`` in eval -> ``nn.SiLU``), the
fallback of ``ops.linear_bn_eval`` (cuBLAS + the BatchNorm-apply kernel) and the one-pass kernel
(``pgh_linear_bn_eval_f32``).  CUDA events over many calls after warm-up; every call reads one of
four distinct inputs, so the working set (>= 470 MB) exceeds the 126 MB L2.  Share of peak:
algorithmic bytes 4 (M K + N K + M N) (+ 4 M N with a residual) over time, against the measured
HBM peak of ``MEASURED_PEAKS.json`` if present, else the 6531.6 GB/s of DESIGN.md section 4.

Whole model, SSWL+ 6 x 128 on 1024 and 128 graphs: eager eval on the module path, eager eval on
the fused path as ``ops`` selects it and with the one-pass kernel forced wherever it fits (all on
device-resident batches with cached plans), and ``StaticPredictor`` replay (host batches fed by
its loader), in graphs/s.

    python profiles/run_eval.py [--iters 50]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from examples.zinc_models import SpModel  # noqa: E402
from pygho_b200 import ops, static as ST  # noqa: E402
from pygho_b200.honn import utils as U  # noqa: E402
from pygho_b200.hodata.device import attach_host_plans, prefetch_plans, sp_datadict  # noqa: E402
from pygho_b200.hodata.synthetic import make_batch  # noqa: E402
from pygho_b200.honn.SpOperator import parse_precomputekey  # noqa: E402

ROWS = 230147


def events_us(fn, iters):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for i in range(iters):
        fn(i)
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop) * 1e3 / iters


def block(K, N, residual, iters, peak, dev):
    torch.manual_seed(K + N)
    lin = torch.nn.Linear(K, N).to(dev)
    bn = torch.nn.BatchNorm1d(N).to(dev).eval()
    with torch.no_grad():
        bn.weight.uniform_(0.5, 1.5)
        bn.bias.uniform_(-0.5, 0.5)
        bn.running_mean.normal_(0.0, 0.5)
        bn.running_var.uniform_(0.1, 10.0)
    act = torch.nn.SiLU()
    xs = [torch.randn(ROWS, K, device=dev) for _ in range(4)]
    rs = [torch.randn(ROWS, N, device=dev) for _ in range(4)] if residual else [None] * 4

    def module(i):
        z = act(bn(lin(xs[i & 3])))
        return z if rs[i & 3] is None else z + rs[i & 3]

    def fallback(i):
        y = torch.nn.functional.linear(xs[i & 3], lin.weight, lin.bias)
        rstd = torch.rsqrt(bn.running_var + bn.eps)
        return ops._ops.bn_act_fwd(y, bn.running_mean, rstd, bn.weight, bn.bias, 1, rs[i & 3], None)

    def kernel(i):
        return ops._ops.linear_bn_eval(xs[i & 3], lin.weight, lin.bias, bn.weight, bn.bias,
                                       bn.running_mean, bn.running_var, bn.eps, 1, rs[i & 3], None)

    nbytes = 4 * (ROWS * K + N * K + ROWS * N) + (4 * ROWS * N if residual else 0)
    res = {}
    with torch.no_grad():
        ref = module(0)
        for name, fn in (("module", module), ("fallback", fallback), ("kernel", kernel)):
            diff = float((fn(0) - ref).abs().max())
            for i in range(5):
                fn(i)
            torch.cuda.synchronize()
            us = min(events_us(fn, iters) for _ in range(3))
            res[name] = (us, nbytes / (us * 1e-6) / 1e9 / peak, diff)
    line = f"block {K}->{N} silu{' +residual' if residual else ''}, {ROWS} rows, {nbytes / 1e6:.0f} MB |"
    for name, (us, frac, diff) in res.items():
        line += f" {name} {us:.1f} us ({frac:.2f} of peak, max|d| vs module {diff:.1e}) |"
    win = "kernel" if res["kernel"][0] < res["fallback"][0] else "fallback"
    print(line + f" faster: {win}", flush=True)


def model_eval(graphs, iters, dev):
    torch.manual_seed(0)
    model = SpModel("SSWL", num_layer=6, hiddim=128).to(dev)
    keys = parse_precomputekey(model)
    tables = {"x": model.x_encoder.num_embeddings, "A": model.ea_encoder.num_embeddings,
              "X": model.tuplefeat_encoder.num_embeddings}
    hbs = [make_batch(graphs, seed=1000 + i) for i in range(4)]
    dds = []
    for hb in hbs:
        dd = sp_datadict(hb, dev, keys)
        attach_host_plans(hb, dd, keys)
        prefetch_plans(dd, keys, embeddings=tables)
        dds.append(dd)
    n_graphs = sum(hb.num_graphs for hb in hbs)
    model.eval()

    def eager():
        with torch.no_grad():
            return torch.cat([model(dd) for dd in dds])

    def rate(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(iters):
            out = fn()
        torch.cuda.synchronize()
        return n_graphs * iters / (time.perf_counter() - t0), out

    real = U._match_eval_block
    U._match_eval_block = lambda mods, i: None            # the stock modules, block by block
    try:
        g_module, p_module = rate(eager)
    finally:
        U._match_eval_block = real
    g_fused, p_fused = rate(eager)
    widths = ops._EVAL_GEMM_WIDTHS
    ops._EVAL_GEMM_WIDTHS = (128, 256, 384)              # the one-pass kernel wherever it fits
    try:
        g_kernel, _p = rate(eager)
    finally:
        ops._EVAL_GEMM_WIDTHS = widths
    pred = ST.StaticPredictor(hbs, ST.capacities(hbs, keys), dev, keys, model)
    g_replay, p_replay = rate(pred)
    pred.close()
    print(f"SSWL+ 6x128 eval, 4 batches of {graphs} graphs | module path {g_module:.0f} graphs/s | "
          f"fused path (selection rule) {g_fused:.0f} graphs/s | fused path, one-pass kernel forced "
          f"{g_kernel:.0f} graphs/s | StaticPredictor replay {g_replay:.0f} graphs/s | "
          f"max|fused - module| {float((p_fused - p_module).abs().max()):.1e}, "
          f"max|replay - fused| {float((p_replay - p_fused).abs().max()):.1e}", flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("run_eval.py measures the GPU path: no CUDA device")
    dev = torch.device("cuda", 0)
    torch.backends.cuda.matmul.allow_tf32 = True          # like the reference (zinc.py:30)
    smi = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                          "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print(f"device: {torch.cuda.get_device_name(dev)} | nvidia-smi name, power.limit, "
          f"clocks.max.sm: {smi}")
    peak, source = 6531.6, "6531.6 GB/s (DESIGN.md section 4)"
    try:
        measured = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs")
        if measured:
            peak, source = float(measured), f"MEASURED_PEAKS.json hbm_gbs {float(measured):.1f} GB/s"
    except (OSError, ValueError):
        pass
    print(f"HBM peak for the shares: {source}")
    for K, N in ((384, 128), (128, 128), (384, 384), (384, 256)):
        for residual in (False, True):
            block(K, N, residual, args.iters, peak, dev)
    for graphs in (1024, 128):
        model_eval(graphs, max(3, args.iters // 10), dev)


if __name__ == "__main__":
    main()
