"""Time ``rdsampler`` on the device against the host path it replaces.

Device: CUDA events around ``rdsampler`` calls (host node_ptr, the usual loader case; includes
the Python glue, the per-graph layout ops and the two kernels), and around the two kernel
launches alone with the layout precomputed.  Host: per graph ``numpy.linalg.pinv`` of the
Laplacian, R from it, padding into a (B, nmax, nmax) float32 array and the copy to the device
-- the reference's way (hodata/MaTupleSampler.py:34-57 + to_dense_tuplefeat).  Every input fits
in L2 after the first pass; these are the sizes a loader hands over per batch.

    python profiles/run_rdsampler.py [--iters 200]
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from pygho_b200 import _lib  # noqa: E402
from pygho_b200._lib import call, ptr, stream_ptr  # noqa: E402
from pygho_b200.hodata.MaTupleSampler import rdsampler  # noqa: E402
from pygho_b200.hodata.SpTupleSampler import _batch_layout  # noqa: E402
from pygho_b200.hodata.synthetic import make_batch  # noqa: E402


def host_rdsampler(edge_index, node_ptr, dev):
    B = node_ptr.shape[0] - 1
    sizes = np.diff(node_ptr)
    nmax = int(sizes.max())
    out = np.zeros((B, nmax, nmax), dtype=np.float32)
    graph_of = np.searchsorted(node_ptr[1:], edge_index[0], side="right")
    for g in range(B):
        n0, n = int(node_ptr[g]), int(sizes[g])
        e = edge_index[:, graph_of == g] - n0
        A = np.zeros((n, n))
        A[e[0], e[1]] = 1.0
        A[e[1], e[0]] = 1.0
        np.fill_diagonal(A, 0.0)
        P = np.linalg.pinv(np.diag(A.sum(1)) - A, hermitian=True)
        d = np.diag(P)
        out[g, :n, :n] = d[:, None] + d[None, :] - 2.0 * P
    t = torch.from_numpy(out).to(dev)
    torch.cuda.synchronize(dev)
    return t


def events_ms(fn, iters, dev):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        fn()
    stop.record()
    torch.cuda.synchronize(dev)
    return start.elapsed_time(stop) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--host-reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("run_rdsampler.py measures the GPU path: no CUDA device")
    dev = torch.device("cuda", 0)
    smi = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                          "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print(f"device: {torch.cuda.get_device_name(dev)} | nvidia-smi name, power.limit, "
          f"clocks.max.sm: {smi}")
    for label, hb in (("zinc x1024", make_batch(1024, seed=0)),
                      ("sr25 x64", make_batch(64, seed=0, shape="sr25"))):
        ei = torch.from_numpy(hb.edge_index).to(dev)
        node_ptr = hb.node_ptr
        for _ in range(10):
            X = rdsampler(ei, node_ptr)
        torch.cuda.synchronize(dev)
        full = events_ms(lambda: rdsampler(ei, node_ptr), args.iters, dev)

        src, dst, dptr, edge_ptr, sq_ptr, node_graph, nmax = _batch_layout(ei, node_ptr, True)
        B, N = dptr.numel() - 1, node_graph.numel()
        R = torch.empty((N * nmax,), dtype=torch.float32, device=dev)
        out = torch.empty((B, nmax, nmax), dtype=torch.float32, device=dev)
        mask = torch.empty((B, nmax, nmax), dtype=torch.bool, device=dev)
        s = stream_ptr(dev)

        def resistance():
            call("pgh_resistance_f32", ptr(src), ptr(dst), ptr(dptr), ptr(edge_ptr), ptr(sq_ptr),
                 B, nmax, ptr(R), s)

        def dense():
            call("pgh_rd_dense_f32", ptr(R), ptr(dptr), ptr(sq_ptr), B, nmax, 0.0, ptr(out),
                 ptr(mask), s)

        for _ in range(10):
            resistance()
            dense()
        k_res = events_ms(resistance, args.iters, dev)
        k_dense = events_ms(dense, args.iters, dev)

        host = []
        for _ in range(args.host_reps):
            t0 = time.perf_counter()
            ref = host_rdsampler(hb.edge_index, hb.node_ptr, dev)
            host.append((time.perf_counter() - t0) * 1e3)
        diff = float((ref - X.data).abs().max())
        print(f"{label}: {B} graphs, {N} nodes, nmax {nmax} | rdsampler {full * 1e3:.1f} us/call "
              f"(events, {args.iters} calls) | kernels: resistance {k_res * 1e3:.1f} us, "
              f"rd_dense {k_dense * 1e3:.1f} us | host pinv loop + pad + copy "
              f"{float(np.median(host)):.1f} ms (median of {args.host_reps}) | "
              f"speed-up {float(np.median(host)) / full:.0f}x | max |device - host| {diff:.2e}")


if __name__ == "__main__":
    main()
