#!/usr/bin/env python
"""Benchmark: training throughput (graphs/s) of the pygho.backend hot path on synthetic batches.

    python bench.py --gpus N --steps K --warmup W            # this repo (CUDA kernels)
    python bench.py --impl reference --gpus N --steps K ...  # reference CPU path (oracle port)

Workloads (``--workload``; BASELINE.json ``configs``):

* ``sswl`` (default, configs[1] / [4]): 6-layer SSWL+ sparse model of the reference's
  ``example/zinc.py`` (hidden 128, mlplayer 2, outlayer 4, bn/silu, npool sum, lpool mean) on
  synthetic ZINC-shaped k-hop(3) batches, GLOBAL batch 1024 graphs.  With N GPUs the global
  batch is sharded 1024/N graphs per rank (``"scaling": "strong"``, SURVEY.md 8e);
  ``--scaling weak`` keeps 1024 graphs per GPU instead.
* ``ppgn_dd`` (configs[2]): dense PPGN / 2-FWL MaskedTensor model (mamamm), 128 graphs.
* ``dssgnn_sr25`` / ``i2_sr25`` (configs[3]): DSSGNN (2-D tuples) / I2-GNN (3-D tuples) on
  sr25-shaped strongly regular graphs, 64 graphs.

One "step" is one full optimisation step (forward, L1 loss, backward, gradient all-reduce when
N > 1, AdamW).  Prints ONE JSON line (rank 0).

* ``value``: graphs/s with batches and plans resident in HBM (device-timed, max over ranks).
* ``e2e``: the same step driven from pinned HOST buffers in the reference's datadict format:
  host->device copies, SparseTensor wrapping, CSR regrouping of the plans and a device->host
  read of the loss are inside the timed region.
* ``roofline``: the dominant kernel of the workload's hot path timed alone with CUDA events on
  rotating operand sets larger than L2; achieved = algorithmic bytes (SURVEY.md 8d) / duration.
* ``cpu_baseline``: the oracle port of the reference (torch CPU ops) on the host cores, on a
  bounded sample of the same workload; ``stock_gpu_baseline``: the same ATen op chain the
  reference would run, moved to this GPU (the "kernel to beat" of BASELINE.md).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

# batches differ in size from step to step: growable segments keep the caching allocator from
# falling back to cudaMalloc/cudaFree (device-synchronising) when a block does not fit, and
# size classes of 1/8 power of two let batches of slightly different sizes reuse each other's
# blocks instead of fragmenting the pool
os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF",
                      "expandable_segments:True,roundup_power2_divisions:8")

# NCCL prints its version banner (NCCL_DEBUG=VERSION/INFO) to stdout by default: keep stdout
# for the one JSON line
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

import numpy as np  # noqa: E402
import torch  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (metric, default global batch, conv, mode, graph shape, tuple sampler)
    "sswl": ("sswl_plus_zinc_shape_train_graphs_per_s", 1024, "SSWL", "sparse", "zinc", "khop"),
    "ppgn_dd": ("ppgn_dense_zinc_shape_train_graphs_per_s", 128, "PPGN", "dense", "zinc", "khop"),
    "dssgnn_sr25": ("dssgnn_sr25_shape_train_graphs_per_s", 64, "DSSGNN", "sparse", "sr25", "khop"),
    "i2_sr25": ("i2gnn_sr25_shape_train_graphs_per_s", 64, "I2GNN", "sparse", "sr25", "i2"),
}
ORACLE_KEYS = {"SSWL": ["X___X___1___A___0", "X___A___1___X___0"], "NGNN": ["X___X___1___A___0"],
               "DSSGNN": ["X___X___1___A___0"], "PPGN": ["X___X___1___X___0"],
               "I2GNN": ["X___X___2___A___0"]}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="sswl", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0,
                    help="GLOBAL batch in graphs (default: the workload's; 1024 for sswl)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong: --batch is sharded over the GPUs; weak: --batch graphs per GPU")
    ap.add_argument("--conv", default="", help="override the workload's conv layer (sparse mode)")
    ap.add_argument("--hidden", type=int, default=128)
    ap.add_argument("--layers", type=int, default=6)
    ap.add_argument("--num-batches", type=int, default=3, help="distinct batches rotated")
    ap.add_argument("--ref-batch", type=int, default=0,
                    help="graphs per CPU reference step (default: the global batch)")
    ap.add_argument("--ref-budget-s", type=float, default=240.0,
                    help="the reference arm trims its step count to finish within this time")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-stock-gpu", action="store_true")
    ap.add_argument("--torch-adamw", action="store_true",
                    help="torch.optim.AdamW(fused, capturable) instead of the one-launch FlatAdamW")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-static", action="store_true",
                    help="host-fed path: eager steps on exact-size batches instead of graph "
                         "replay on capacity-padded batches")
    ap.add_argument("--no-graph", action="store_true",
                    help="launch the resident-batch steps eagerly instead of replaying CUDA graphs")
    ap.add_argument("--syncbn", action="store_true",
                    help="BatchNorm statistics all-reduced over the ranks (equals single-process "
                         "training on the global batch)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the last one computed (loss, "
                         "predictions, parameters, gradients, BatchNorm statistics of rank 0) as "
                         "DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm only")
    metric, batch, conv, mode, shape, tuples = WORKLOADS[args.workload]
    args.metric, args.mode, args.shape, args.tuples = metric, mode, shape, tuples
    args.batch = args.batch or batch
    args.conv = args.conv or conv
    args.ref_batch = args.ref_batch or args.batch
    return args


def split(args, world):
    """(graphs per GPU, global batch)."""
    if args.scaling == "weak":
        return args.batch, args.batch * world
    if args.batch % world:
        raise SystemExit(f"--batch {args.batch} is not divisible by {world} GPUs")
    return args.batch // world, args.batch


def config_of(args, world, stats):
    """The `config` object: identical for the own arm and the reference arm of one workload
    at one N (so the driver can match them); arm-specific notes live in other keys."""
    per_gpu, glob = split(args, world)
    model = {"sparse": "SpModel", "dense": "MaModel"}[args.mode]
    cfg = {
        "workload": (f"{args.conv}{'+' if args.conv == 'SSWL' else ''} {model} {args.layers}x{args.hidden} "
                     f"(example/zinc.py, work.sh flags) on synthetic {args.shape}-shape "
                     f"{args.tuples} batches, global batch {glob} graphs"),
        "global_batch": glob, "per_gpu_batch": per_gpu, "n_gpus": world,
        "matmul": "tf32 on the GPU (reference: set_float32_matmul_precision('high')), fp32 on the CPU",
        "l2": "step working set >> L2 at 1024 graphs/GPU; distinct batches rotated",
        "parallelism": f"dp{world}: graphs sharded {per_gpu}/GPU (balanced by tuple count), "
                       "flat-bucket NCCL all-reduce"
                       + (", SyncBN" if getattr(args, "syncbn", False) else ""),
    }
    cfg.update(stats)
    return cfg


# ------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi sampled every 50 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.lines, self.proc = index, [], None

    def __enter__(self):
        if self.index < 0:
            return self
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "50", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def __exit__(self, *a):
        if self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, smax, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = max(smax, float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": smax,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------- host batches
def host_batches(args, per_gpu, rank, count, world=1):
    """`count` distinct host batches of `per_gpu` graphs for this rank.

    Strong scaling (world > 1): every rank generates the SAME global batch i (one seed stream, so
    the N-GPU job trains on exactly the graphs the 1-GPU job would see) and takes its shard.  The
    shard is balanced by cost: graphs sorted by tuple count and dealt to the ranks in snake order
    (equal graph counts, near-equal tuple / triple counts), because the step ends with an
    all-reduce and therefore runs at the pace of the largest shard (SURVEY.md 8e "greedy balance
    by sum of T per graph")."""
    from pygho_b200.hodata.synthetic import collate, make_batch, make_graphs
    if world == 1 or args.scaling == "weak":
        return [make_batch(per_gpu, seed=1000 * rank + i, tuples=args.tuples, shape=args.shape)
                for i in range(count)]
    out = []
    for i in range(count):
        graphs = make_graphs(per_gpu * world, seed=i, tuples=args.tuples, shape=args.shape)
        order = sorted(range(len(graphs)), key=lambda g: (-graphs[g].tupleid.shape[1], g))
        mine = []
        for pos, g in enumerate(order):
            rnd, k = divmod(pos, world)
            owner = k if rnd % 2 == 0 else world - 1 - k
            if owner == rank:
                mine.append(g)
        out.append(collate([graphs[g] for g in sorted(mine)]))
    return out


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays, budget=DUMP_BYTES):
    """Write every named array as ``out_dir/<name>.npy`` in float32 (float64 stays float64).
    When the files would exceed `budget` bytes together, every array keeps the same fraction of
    its elements: a sample of flat positions drawn with a fixed seed and kept in ascending order,
    so two runs with the same arguments write the same positions."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    arrays = {k: a if a.dtype == np.float64 else a.astype(np.float32, copy=False)
              for k, a in arrays.items()}
    header = 256                                   # upper bound of one .npy header here
    data = sum(a.nbytes for a in arrays.values())
    room = budget - header * len(arrays)
    frac = 1.0 if data <= room else room / data
    for name, a in arrays.items():
        if frac < 1.0:
            keep = int(a.size * frac)
            pos = np.random.default_rng(0).choice(a.size, keep, replace=False)
            a = a.reshape(-1)[np.sort(pos)]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def batch_stats(args, hb, keys):
    st = {"nodes": int(hb.num_nodes), "edges": int(hb.edge_index.shape[1]),
          "tuples": int(hb.tupleid.shape[1])}
    if args.mode == "dense":
        n = int(np.diff(hb.node_ptr).max())
        st.update(padded_n=n, dense_positions=int(hb.num_graphs * n * n))
    elif keys and keys[0] in hb.plans:
        st["triples_per_key"] = int(hb.plans[keys[0]].shape[1])
    return st


def host_plans(hb, conv):
    """The reference precomputes the ``acd`` plans per graph on the CPU (hodata/SpData.py:115-172);
    here with the numpy oracle (reference arm / CPU baseline only)."""
    from oracle import pygho_oracle as O
    plans = {}
    for key in ORACLE_KEYS[conv]:
        _o0, o1, d1, o2, d2 = key.split("___")
        pick = lambda op: hb.edge_index if op == "A" else hb.tupleid  # noqa: E731
        plans[key + "___acd"] = torch.from_numpy(
            O.filterind(hb.tupleid, *O.spspmm_ind(pick(o1), int(d1), pick(o2), int(d2))))
    return plans


# ----------------------------------------------------------------- reference arm
def oracle_step_fn(args, batch_graphs, device="cpu", seed=1000):
    """(step(), stats) of the CPU restatement of the reference (oracle/model_oracle.py) on one
    batch of `batch_graphs` graphs made by the same generator as the GPU arm's."""
    from oracle import model_oracle as MO
    from pygho_b200.hodata.synthetic import make_batch
    torch.manual_seed(0)
    hb = make_batch(batch_graphs, seed=seed, tuples=args.tuples, shape=args.shape)
    if args.mode == "dense":
        g = MO.host_dense_dict(hb)
        model = MO.OMaModel(num_layer=args.layers, hiddim=args.hidden)
        stats = batch_stats(args, hb, [])
    else:
        plans = host_plans(hb, args.conv)
        g = MO.host_graph_dict(hb, plans)
        model = MO.OSpModel(conv=args.conv, num_layer=args.layers, hiddim=args.hidden)
        stats = batch_stats(args, hb, [])
        stats["triples_per_key"] = int(next(iter(plans.values())).shape[1])
    if device != "cpu":
        g = {k: (v.to(device) if isinstance(v, torch.Tensor) else v) for k, v in g.items()}
        model = model.to(device)
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3)

    def step():
        opt.zero_grad()
        loss = torch.nn.functional.l1_loss(g["y"].unsqueeze(-1), model(g))
        loss.backward()
        opt.step()
        return loss

    return step, stats


def oracle_cpu_throughput(args, steps, warmup, batch_graphs, budget_s=None):
    """graphs/s of the oracle port on all host threads; trims `steps` to `budget_s`."""
    try:   # all host threads the process may use (torchrun pins OMP_NUM_THREADS=1 by default)
        torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    except Exception:
        pass
    step, stats = oracle_step_fn(args, batch_graphs)
    t_w = time.perf_counter()
    for _ in range(warmup):
        float(step())
    per = (time.perf_counter() - t_w) / max(warmup, 1)
    if budget_s is not None and warmup and per * (steps + warmup) > budget_s:
        steps = max(2, int(budget_s / per) - warmup)
    t0 = time.perf_counter()
    for _ in range(steps):
        float(step())
    dt = time.perf_counter() - t0
    return batch_graphs * steps / dt, dt / steps * 1e3, torch.get_num_threads(), steps, stats


def run_reference(args):
    """Reference arm: the reference's CPU implementation of the path (oracle port, all host
    threads) on the own arm's workload: the GLOBAL batch per step, same steps and warm-up
    (trimmed only if the run would exceed --ref-budget-s).  Rank 0 alone runs."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    steps, warmup = max(1, args.steps), max(1, args.warmup)
    val, ms, cores, ran, stats = oracle_cpu_throughput(args, steps, warmup, args.ref_batch,
                                                      args.ref_budget_s)
    _per_gpu, glob = split(args, world)
    sample = (f"{ran} steps (+{warmup} warm-up) of {args.ref_batch} graphs = "
              f"{'the global batch' if args.ref_batch == glob else 'a sample of the global batch'}"
              f" of the GPU arm, same generator and model, {cores} host threads")
    cfg = config_of(args, world, stats if args.ref_batch == glob else {})
    print(json.dumps({
        "impl": "reference", "metric": args.metric, "value": val, "unit": "graphs/s",
        "n_gpus": args.gpus, "steps": ran, "warmup": warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": cfg,
        "reference_kind": "oracle_port_cpu (oracle/model_oracle.py: the reference's own torch "
                          "CPU op chain, pinned to the real reference's layer outputs/gradients; "
                          "/root/reference needs torch_geometric and cannot travel)",
        "cpu_baseline": {"value": val, "unit": "graphs/s", "cores": cores, "kind": "port",
                         "sample": sample},
        "e2e": {"value": val, "unit": "graphs/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }), flush=True)


def stock_gpu_throughput(args, device, batch_graphs, steps=8, warmup=3):
    """The reference's ATen op chain (index_select / mul / scatter_reduce_ / cuBLAS / cuDNN BN)
    run on THIS GPU: the oracle model moved to `device`.  This is what a PygHO user gets on a
    B200 today (BASELINE.md "kernel to beat"); none of this repo's kernels are on that path."""
    step, _ = oracle_step_fn(args, batch_graphs, device=device)
    for _ in range(warmup):
        step()
    torch.cuda.synchronize(device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize(device)
    ms = e0.elapsed_time(e1) / steps
    return {"value": batch_graphs / (ms * 1e-3), "unit": "graphs/s", "ms_per_step": ms,
            "steps": steps, "warmup": warmup, "graphs_per_step": batch_graphs,
            "what": "oracle/model_oracle.py on cuda: stock torch ops (index_select, mul, "
                    "scatter_reduce_, addmm, batch_norm), eager, TF32 matmuls"}


# ---------------------------------------------------------------------- rooflines
def _l2_bytes():
    try:
        from pygho_b200 import _lib
        import ctypes
        info = (ctypes.c_int32 * 5)()
        _lib.call("pgh_device_info", info)
        return int(info[2]) << 10
    except Exception:
        return 128 << 20


def _time_launches(launch, iters, device):
    """Mean device time (us) of `iters` back-to-back launches: captured into one CUDA graph and
    replayed (no Python / launch gaps); eager fallback if capture fails."""
    torch.cuda.synchronize(device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    try:
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for i in range(iters):
                launch(i)
        graph.replay()
        torch.cuda.synchronize(device)
        best = float("inf")
        for _ in range(3):
            e0.record()
            graph.replay()
            e1.record()
            torch.cuda.synchronize(device)
            best = min(best, e0.elapsed_time(e1))
        del graph
        return best * 1e3 / iters, "cuda graph replay of the launches"
    except Exception:  # noqa: BLE001
        torch.cuda.synchronize(device)
        e0.record()
        for i in range(iters):
            launch(i)
        e1.record()
        torch.cuda.synchronize(device)
        return e0.elapsed_time(e1) * 1e3 / iters, "eager launches"


def _roofline_obj(kernel, alg_bytes, us, timing, peaks, traffic_key, extra):
    peak = peaks.get("hbm_gbs")
    achieved = alg_bytes / (us * 1e-6) / 1e9
    traffic = None
    try:  # dram bytes of this launch from the committed ncu --set full capture
        traffic = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))[traffic_key]
    except Exception:
        pass
    out = {"bound": "hbm", "kernel": kernel, "achieved": achieved,
           "peak": peak if peak else 6650.0, "unit": "GB/s",
           "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst, kernel timed alone)" if peak
           else "fallback 6650 GB/s (B200_PROFILING.md)",
           "frac": achieved / (peak if peak else 6650.0), "traffic": traffic,
           "us_per_launch": us, "algorithmic_bytes": alg_bytes, "timing": timing}
    out.update(extra)
    return out


def roofline_spspmm(dd, hidden, device, peaks, key="X___X___1___A___0"):
    """The fused spspmm forward (SSWL / DSSGNN / NGNN key ``X x A``) alone."""
    from pygho_b200 import plans as P
    ops = torch.ops.pygho_b200
    nX, nA = dd["X"].nnz, dd["A"].nnz
    plan = P.plan_from_acd(dd[key + "___acd"], nX, nX, nA)
    g = plan.group("a")
    T = plan.T
    alg_bytes = 4 * hidden * (nX + nA + nX) + 4 * (2 * T + nX + 1)
    l2 = _l2_bytes()
    per_set = 4 * hidden * (2 * nX + nA)
    nsets = max(4, int(np.ceil(2.5 * l2 / per_set)))
    gen = torch.Generator(device=device).manual_seed(0)
    sets = [(torch.randn((nX, hidden), device=device, generator=gen),
             torch.randn((nA, hidden), device=device, generator=gen)) for _ in range(nsets)]

    def launch(i):
        xv, av = sets[i % nsets]
        ops.seg_gmr(xv, g.first, None, av, g.second, g.rowptr, nX, 0)

    for i in range(3):
        launch(i)
    us, timing = _time_launches(launch, 5 * nsets, device)
    return _roofline_obj(f"seg_gmr_lean_kernel<sum,B> (spspmm fwd, key {key})", alg_bytes, us,
                         timing, peaks, "spspmm_fwd",
                         {"rows": nX, "triples": T, "operand_sets": nsets, "l2_bytes": l2})


def roofline_mamamm(dd, hidden, device, peaks):
    """The dense 2-FWL contraction (PPGNConv DD) alone: the default kernel (algo 4, exact fp32 from
    a TMA-fed shared-memory ring) and, beside it, the tcgen05 TF32 pipeline (algo 2)."""
    from pygho_b200.backend.Mamamm import default_algo, mamamm
    from pygho_b200 import MaskedTensor
    X = dd["X"]
    mask = X.mask
    b, n = mask.shape[0], mask.shape[1]
    l2 = _l2_bytes()
    per_set = 4 * hidden * b * n * n * 3
    nsets = max(3, int(np.ceil(2.5 * l2 / per_set)))
    gen = torch.Generator(device=device).manual_seed(0)
    m = mask.unsqueeze(-1)
    sets = [(MaskedTensor(torch.randn((b, n, n, hidden), device=device, generator=gen) * m, mask, 0.0, True),
             MaskedTensor(torch.randn((b, n, n, hidden), device=device, generator=gen) * m, mask, 0.0, True))
            for _ in range(nsets)]

    def launch(i):
        a, c = sets[i % nsets]
        mamamm(a, 2, c, 1, mask)

    for i in range(3):
        launch(i)
    us, timing = _time_launches(launch, 5 * nsets, device)
    import os
    keep = os.environ.get("PYGHO_B200_MAMAMM_ALGO")
    os.environ["PYGHO_B200_MAMAMM_ALGO"] = "2"
    try:
        for i in range(3):
            launch(i)
        us_tc, _ = _time_launches(launch, 5 * nsets, device)
    finally:
        if keep is None:
            del os.environ["PYGHO_B200_MAMAMM_ALGO"]
        else:
            os.environ["PYGHO_B200_MAMAMM_ALGO"] = keep
    sizes = mask[:, :, 0].sum(1).double()
    alg_bytes = 4 * hidden * b * 3 * n * n + b * n * n            # SURVEY 8d (padded tensors)
    moved = int(4 * hidden * float((2 * sizes * sizes).sum() + b * n * n) + b * n * n)
    useful = 2.0 * hidden * float((sizes ** 3).sum())
    names = {4: "mamamm_smem_kernel (algo 4; exact fp32 FMAs from a TMA-fed shared-memory ring, largest graph first)",
             2: "mamamm_tc_pipe_kernel (algo 2; tcgen05 kind::tf32, TMEM accumulators)"}
    return _roofline_obj(names.get(default_algo(), f"mamamm algo {default_algo()}"),
                         alg_bytes, us, timing, peaks, "mamamm",
                         {"graphs": b, "padded_n": n, "operand_sets": nsets, "l2_bytes": l2,
                          "moved_bytes_valid_extents": moved,
                          "moved_frac_of_peak": moved / (us * 1e-6) / 1e9 / (peaks.get("hbm_gbs") or 6650.0),
                          "useful_tflops": useful / (us * 1e-6) / 1e12,
                          "tcgen05_algo2_us_per_launch": us_tc,
                          "tcgen05_algo2_useful_tflops": useful / (us_tc * 1e-6) / 1e12,
                          "tcgen05_algo2_tensor_pipe_util_vs_tf32_dense_1100": useful / (us_tc * 1e-6) / 1e12 / 1100.0})


def roofline_pool(dd, hidden, device, peaks, three_d):
    """Pooling kernels of cfg4: 2-D tuples pooled over dim 0 (key = indices[1], unsorted: needs
    the CSC permutation) or 3-D tuples pooled over dim 2 into the sparse (i, j) pattern."""
    X = dd["X"]
    nX = X.nnz
    l2 = _l2_bytes()
    nsets = max(4, int(np.ceil(2.5 * l2 / (4 * hidden * nX))))
    gen = torch.Generator(device=device).manual_seed(0)
    from pygho_b200 import SparseTensor
    sets = [SparseTensor(X.indices, torch.randn((nX, hidden), device=device, generator=gen),
                         tuple(X.shape[:X.sparse_dim]) + (hidden,), True) for _ in range(nsets)]
    if three_d:
        n_out = sets[0].mean([2], return_sparse=True).nnz
        launch = lambda i: sets[i % nsets].mean([2], return_sparse=True)  # noqa: E731
        name = "seg_gmr ring kernel (3-D tuples -> sparse (i,j) pattern, mean)"
        alg = 4 * hidden * (nX + n_out) + 4 * (n_out + 1)
    else:
        n_out = X.shape[1]
        launch = lambda i: sets[i % nsets].mean([0])  # noqa: E731
        name = "seg_gmr ring kernel (pool over dim 0, unsorted key, mean)"
        alg = 4 * hidden * (nX + n_out) + 4 * (n_out + 1) + 4 * nX
    for i in range(3):
        launch(i)
    us, timing = _time_launches(launch, 5 * nsets, device)
    return _roofline_obj(name, alg, us, timing, peaks, "pool3d" if three_d else "pool_cross",
                         {"rows_in": nX, "rows_out": int(n_out), "operand_sets": nsets, "l2_bytes": l2})


# ------------------------------------------------------------------------ own arm
def run_b200(args):
    import torch.distributed as dist
    from examples.zinc_models import MaModel, SpModel
    from pygho_b200 import _lib
    from pygho_b200.dist import FlatGradBucket, broadcast_parameters
    from pygho_b200.hodata.device import (DeferredScalar, DevicePrefetcher, attach_host_plans,
                                          ma_datadict, pin_host_batch, sp_datadict)
    from pygho_b200.honn.SpOperator import parse_precomputekey

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl b200) needs a CUDA device: the kernels have no CPU path")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    torch.backends.cuda.matmul.allow_tf32 = True      # reference: set_float32_matmul_precision('high')
    torch.backends.cudnn.allow_tf32 = True
    _lib.load()
    per_gpu, glob = split(args, world)
    sparse = args.mode == "sparse"

    torch.manual_seed(0)
    if sparse:
        model = SpModel(args.conv, num_layer=args.layers, hiddim=args.hidden).to(device)
        keys = parse_precomputekey(model)
    else:
        model = MaModel(args.conv, num_layer=args.layers, hiddim=args.hidden).to(device)
        keys = []
    broadcast_parameters(model)
    if args.syncbn and world > 1:
        from pygho_b200.dist import enable_sync_batchnorm
        enable_sync_batchnorm(model)
    bucket = FlatGradBucket(model.parameters())
    # both keep the step counter on the device, so the optimizer can be graph-captured.
    # FlatAdamW: the whole AdamW update (torch.optim.AdamW's rule, 1 / world of the gradient
    # average folded in) as ONE launch over flat parameter / gradient / moment buffers
    if args.torch_adamw:
        opt = torch.optim.AdamW(model.parameters(), lr=1e-3, fused=True, capturable=True)
    else:
        from pygho_b200.dist import FlatAdamW
        opt = FlatAdamW(bucket, lr=1e-3)

    hbs = host_batches(args, per_gpu, rank, args.num_batches, world)
    pinned = {}
    dds = []
    for hb in hbs:
        if sparse:
            dd = sp_datadict(hb, device, keys, pinned)
            attach_host_plans(hb, dd, keys)
        else:
            dd = ma_datadict(hb, device, pinned=pinned)
        dds.append(dd)
    if sparse:   # pin the host plans too (they are what the reference's loader would ship)
        for hb in hbs:
            pin_host_batch(hb, pinned)
    h2d_bytes = int(np.mean([hb.nbytes() for hb in hbs]))

    def step_outputs(dd):
        """(loss, predictions) of one optimisation step on `dd`."""
        bucket.zero()
        pred, y = model(dd), dd["y"].unsqueeze(-1)
        nv = dd.get("num_valid_graphs")           # capacity-padded batch: drop the dummy graph
        if nv is not None:
            pred, y = pred[:nv], y[:nv]
        loss = torch.nn.functional.l1_loss(y, pred)
        loss.backward()
        if args.torch_adamw:
            bucket.allreduce_mean()
            opt.step()
        else:
            opt.step(1.0 / bucket.allreduce_sum())
        return loss, pred.detach()

    def train_step(dd):
        return step_outputs(dd)[0]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    def timed(fn, steps, finish=None, per_step=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = _lib.launches()
        e0.record()
        for i in range(steps):
            last = fn(i)
            if per_step is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                per_step.append(ev)
        if finish is not None:
            finish()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        if per_step is not None:
            evs = [e0] + per_step
            per_step[:] = [a.elapsed_time(b) for a, b in zip(evs[:-1], evs[1:])]
        return float(ms.item()), _lib.launches() - l0, last

    warm = max(3, args.warmup)
    for i in range(warm):
        train_step(dds[i % len(dds)])
    # Resident batches: the whole step (fwd, loss, bwd, all-reduce, AdamW) of each batch is
    # captured into one CUDA graph and replayed (pygho_b200/graph.py).  If capture fails on this
    # rank the eager step is used (it issues the same collectives).
    graphs, graph_note = None, "eager (--no-graph)"
    if not args.no_graph:
        try:
            from pygho_b200.graph import StepGraph
            graphs = [StepGraph(lambda dd=dd: step_outputs(dd), warmup=1) for dd in dds]
            graph_note = f"cuda graph replay, one graph per resident batch ({len(graphs)})"
        except Exception as e:  # noqa: BLE001
            graphs = None
            graph_note = f"eager (graph capture failed: {type(e).__name__}: {str(e)[:120]})"
            print(f"[bench] rank {rank}: {graph_note}", file=sys.stderr, flush=True)
            torch.cuda.synchronize(device)
    if graphs is not None:
        run_step = lambda i: graphs[i % len(graphs)].replay()  # noqa: E731
    else:
        run_step = lambda i: step_outputs(dds[i % len(dds)])  # noqa: E731
    for i in range(warm):
        run_step(i)
    # clocks / throttle reasons are sampled by rank 0 only (its own GPU): eight nvidia-smi pollers
    # contend for the driver lock and slow the graph launches of every rank
    with ClockSampler(local if rank == 0 else -1) as clocks:
        ms_total, launches, (last_loss, last_pred) = timed(run_step, args.steps)
    if graphs is not None:                                # replays do not pass through Python
        launches = sum(graphs[i % len(graphs)].launches for i in range(args.steps))
    if args.dump_outputs and rank == 0:
        named = dict(model.named_parameters())
        arrays = {"loss": last_loss.reshape(1), "pred": last_pred}
        arrays.update({f"param.{k}": p for k, p in named.items()})
        arrays.update({f"grad.{k}": p.grad for k, p in named.items() if p.grad is not None})
        arrays.update({f"buffer.{k}": b for k, b in model.named_buffers() if b.is_floating_point()})
        dump_outputs(args.dump_outputs, {k: v.detach().cpu().numpy() for k, v in arrays.items()})
    clock_summary = clocks.summary()
    ms_step = ms_total / args.steps
    value = glob / (ms_step * 1e-3)

    # ---- end to end: pinned host buffers in, loss out -------------------------------
    e2e = None
    if not args.no_e2e:
        reader = DeferredScalar()
        losses = []
        static_ok = sparse and hbs[0].tupleid.shape[0] == 2 and not args.no_graph and not args.no_static
        e2e_mode = "eager step, threaded side-stream prefetch (DevicePrefetcher)"
        if static_ok:
            # Host-fed steps as CUDA-graph replays: the host batches are padded to fixed
            # capacities at collate time (pygho_b200/static.py), so ONE captured graph per slot
            # serves every batch; per step the host enqueues the H2D copies + plan regrouping of
            # the next batch on a side stream and one graph launch.
            from pygho_b200 import static as ST
            caps = ST.capacities(hbs, keys)
            padded = [ST.pad_host_batch(hb, caps, keys) for hb in hbs]
            for hb in padded:
                pin_host_batch(hb, pinned)
            h2d_bytes = int(np.mean([hb.nbytes() for hb in padded]))
            feeder = ST.StaticFeeder(padded, caps, device, keys, train_step, pinned)
            e2e_mode = (f"cuda graph replay on capacity-padded batches (2 static slots, capacities "
                        f"{ {k: v for k, v in caps.items() if len(k) < 3} }), threaded side-stream loader")

            def e2e_step(i):
                loss = feeder.step()
                prev = reader.push(loss)                 # loss of the step before this one
                if prev is not None:
                    losses.append(prev)
        elif sparse:
            # every step's inputs come from pinned host memory (reference datadict format incl.
            # the acd plans); the copies + CSR regrouping of batch i+1 are issued on a side
            # stream right after step i has been launched, the loss is read back every step
            tables = {"x": model.x_encoder.num_embeddings, "A": model.ea_encoder.num_embeddings}
            if hasattr(model.tuplefeat_encoder, "num_embeddings") and hbs[0].tuplefeat.ndim == 1:
                tables["X"] = model.tuplefeat_encoder.num_embeddings
            feeder = DevicePrefetcher(hbs, device, keys, pinned, embeddings=tables)

            def e2e_step(i):
                dd = feeder.get()
                loss = train_step(dd)
                prev = reader.push(loss)                 # loss of the step before this one
                if prev is not None:
                    losses.append(prev)
                feeder.advance()                         # next batch's H2D + plans, side stream
        else:
            feeder = None
            e2e_mode = "eager step, H2D + device-side padding on the compute stream"

            def e2e_step(i):
                dd = ma_datadict(hbs[i % len(hbs)], device, pinned=pinned)   # H2D + device padding
                loss = train_step(dd)
                prev = reader.push(loss)
                if prev is not None:
                    losses.append(prev)

        def read_pending():
            v = reader.flush()
            if v is not None:
                losses.append(v)                         # D2H read of the result

        def e2e_steps(n):
            for i in range(n):
                e2e_step(i)
            read_pending()

        # two full cycles over the host batches: every allocation size of both streams was seen
        e2e_steps(max(args.warmup, 2 * len(hbs) + 1))
        losses.clear()
        if os.environ.get("PYGHO_B200_PROFILE_LOADER") and static_ok:
            # launch list of ONE batch load (H2D, plan regrouping, copy into the static slot) for
            # `ncu --profile-from-start off`: profiles/r2_loader_launches_*.csv
            torch.cuda.synchronize(device)
            torch.cuda.profiler.start()
            feeder._load(feeder.pos + 1)
            torch.cuda.synchronize(device)
            torch.cuda.profiler.stop()
        import gc
        gc.collect()
        gc.freeze()    # long-lived objects out of the collector's way: no multi-ms gen-2 pauses
        per_step = []
        e2e_ms, _, _ = timed(e2e_step, args.steps, finish=read_pending, per_step=per_step)
        assert len(losses) == args.steps and all(np.isfinite(losses)), "e2e: every step's loss is read"
        if os.environ.get("PYGHO_B200_BENCH_TRACE"):
            print(f"[trace] rank {rank} e2e device ms per step: {[round(v, 2) for v in per_step]}",
                  file=sys.stderr)
            if hasattr(feeder, "load_ms"):
                print(f"[trace] loader host ms: {[round(v, 2) for v in feeder.load_ms[-args.steps:]]}; "
                      f"arrays mirrored per load: {feeder.copies}", file=sys.stderr)
            ms_ = torch.cuda.memory_stats(device)
            print(f"[trace] allocator: device_alloc {ms_['num_device_alloc']} device_free "
                  f"{ms_['num_device_free']} retries {ms_['num_alloc_retries']}", file=sys.stderr)
        e2e = {"value": glob / (e2e_ms / args.steps * 1e-3), "unit": "graphs/s",
               "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
               "ms_per_step": e2e_ms / args.steps, "mode": e2e_mode,
               "step_ms": {"min": float(np.min(per_step)), "median": float(np.median(per_step)),
                           "max": float(np.max(per_step))}}
        if feeder is not None:
            feeder.close()                               # no stray side-stream work below
        torch.cuda.synchronize(device)

    out = None
    peaks = {}
    if rank == 0:
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        out = {
            "metric": args.metric, "value": value, "unit": "graphs/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": config_of(args, world, batch_stats(args, hbs[0], keys)),
            "launch": graph_note,
            "e2e": e2e, "gpu_launches": launches, "clocks": clock_summary,
        }
    if rank == 0 and not args.no_roofline:
        try:
            if args.workload == "ppgn_dd":
                out["roofline"] = roofline_mamamm(dds[0], args.hidden, device, peaks)
            elif args.workload == "dssgnn_sr25":
                out["roofline"] = roofline_pool(dds[0], args.hidden, device, peaks, False)
                out["roofline_spspmm"] = roofline_spspmm(dds[0], args.hidden, device, peaks)
            elif args.workload == "i2_sr25":
                out["roofline"] = roofline_pool(dds[0], args.hidden, device, peaks, True)
                out["roofline_spspmm"] = roofline_spspmm(dds[0], args.hidden, device, peaks,
                                                         "X___X___2___A___0")
            else:
                out["roofline"] = roofline_spspmm(dds[0], args.hidden, device, peaks)
        except Exception as e:  # noqa: BLE001
            out["roofline"] = {"error": f"{type(e).__name__}: {str(e)[:200]}"}
    if world > 1:
        dist.barrier()
    if rank == 0 and world == 1:
        del dds
        graphs = None
        run_step = None
        torch.cuda.empty_cache()
        if not args.no_stock_gpu:
            try:
                out["stock_gpu_baseline"] = stock_gpu_throughput(args, device, per_gpu)
                out["stock_gpu_baseline"]["own_over_stock"] = value / out["stock_gpu_baseline"]["value"]
            except Exception as e:  # noqa: BLE001
                out["stock_gpu_baseline"] = {"error": f"{type(e).__name__}: {str(e)[:200]}"}
            torch.cuda.empty_cache()
        if not args.no_cpu_baseline:
            v, ms, cores, ran, _ = oracle_cpu_throughput(args, 3, 1, args.ref_batch)
            out["cpu_baseline"] = {"value": v, "unit": "graphs/s", "cores": cores, "kind": "port",
                                   "sample": f"{ran} steps (+1 warm-up) of {args.ref_batch} graphs, "
                                             "oracle port of the reference (torch CPU ops), same "
                                             "model and generator as the GPU arm"}
    if rank == 0:
        print(json.dumps(out), flush=True)
    # Orderly teardown: prefetch thread first (closed above), then the CUDA graphs (they hold
    # captured NCCL kernels and must go before the communicator), then the process group.  If the
    # shutdown hangs, fail LOUDLY (non-zero status) instead of waiting for the driver's limit.
    sys.stdout.flush()
    sys.stderr.flush()

    def _hung():
        print(f"[bench] rank {rank}: teardown did not finish within 120 s", file=sys.stderr, flush=True)
        os._exit(3)

    killer = threading.Timer(120.0, _hung)
    killer.daemon = True
    killer.start()
    run_step = None
    graphs = None
    import gc
    gc.collect()
    torch.cuda.synchronize(device)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    killer.cancel()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
