"""Train the SSWL+ model of the reference's ``example/zinc.py`` on synthetic ZINC-shaped batches
with pygho_b200: host batches -> ``DevicePrefetcher`` (worker thread + side stream) -> eager
steps, or, with ``--resident``, one CUDA-graph replay per step on device-resident batches.

    python examples/train_zinc.py --steps 50 [--resident] [--conv SSWL|NGNN|DSSGNN] [--batch 1024]
                                  [--eval-batches K --eval-every 10]

``--eval-batches K`` holds out K more batches (seeds distinct from the training batches) and every
``--eval-every`` steps prints their MAE, predicted by graph replay (``static.StaticPredictor``: eval
mode, no autograd, one-pass BatchNorm blocks), and the evaluation rate.
"""
from __future__ import annotations

import argparse
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from examples.zinc_models import SpModel  # noqa: E402
from pygho_b200 import static as ST  # noqa: E402
from pygho_b200.dist import FlatGradBucket  # noqa: E402
from pygho_b200.graph import StepGraph  # noqa: E402
from pygho_b200.hodata.device import (DeferredScalar, DevicePrefetcher, attach_host_plans,  # noqa: E402
                                      prefetch_plans, sp_datadict)
from pygho_b200.hodata.synthetic import make_batch  # noqa: E402
from pygho_b200.honn.SpOperator import parse_precomputekey  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--conv", default="SSWL")
    ap.add_argument("--hidden", type=int, default=128)
    ap.add_argument("--layers", type=int, default=6)
    ap.add_argument("--num-batches", type=int, default=4)
    ap.add_argument("--resident", action="store_true", help="batches stay in HBM, steps replay CUDA graphs")
    ap.add_argument("--eval-batches", type=int, default=0, help="held-out batches evaluated during training")
    ap.add_argument("--eval-every", type=int, default=10)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.backends.cuda.matmul.allow_tf32 = True          # like the reference (zinc.py:30)
    torch.manual_seed(0)
    model = SpModel(args.conv, num_layer=args.layers, hiddim=args.hidden).to(dev)
    keys = parse_precomputekey(model)
    tables = {"x": model.x_encoder.num_embeddings, "A": model.ea_encoder.num_embeddings,
              "X": model.tuplefeat_encoder.num_embeddings}
    bucket = FlatGradBucket(model.parameters())
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3, fused=True, capturable=True)
    hbs = [make_batch(args.batch, seed=i) for i in range(args.num_batches)]
    print(f"{args.conv}: {sum(p.numel() for p in model.parameters())} parameters, "
          f"{len(hbs)} batches of {args.batch} graphs ({hbs[0].tupleid.shape[1]} tuples)")

    def train_step(dd):
        bucket.zero()
        loss = torch.nn.functional.l1_loss(dd["y"].unsqueeze(-1), model(dd))
        loss.backward()
        opt.step()
        return loss.detach()

    # plans are built on the device the first time a batch is seen and shipped from the host
    # afterwards, like the reference's pre-transformed datasets
    dds = []
    for hb in hbs:
        dd = sp_datadict(hb, dev, keys)
        attach_host_plans(hb, dd, keys)
        prefetch_plans(dd, keys, embeddings=tables)
        dds.append(dd)
    evaluate = None
    if args.eval_batches:
        eval_hbs = [make_batch(args.batch, seed=100000 + i) for i in range(args.eval_batches)]
        for hb in eval_hbs:
            attach_host_plans(hb, sp_datadict(hb, dev, keys), keys)
        eval_y = torch.cat([torch.from_numpy(hb.y) for hb in eval_hbs]).to(dev).float().unsqueeze(-1)
        predictor = ST.StaticPredictor(eval_hbs, ST.capacities(eval_hbs, keys), dev, keys, model)

        def evaluate(step):
            torch.cuda.synchronize()
            t = time.perf_counter()
            mae = float((predictor() - eval_y).abs().mean())
            rate = len(eval_y) / (time.perf_counter() - t)
            print(f"step {step:4d} validation MAE {mae:.6f} ({len(eval_y)} graphs, {rate:.0f} graphs/s)")
            return mae
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    if args.resident:
        graphs = [StepGraph(lambda dd=dd: train_step(dd), warmup=1) for dd in dds]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(args.steps):
            loss = graphs[i % len(graphs)].replay()
            if i % 10 == 0:
                print(f"step {i:4d} loss {float(loss):.4f}")
            if evaluate and (i + 1) % args.eval_every == 0:
                evaluate(i)
    else:
        feeder = DevicePrefetcher(hbs, dev, keys, embeddings=tables)
        reader = DeferredScalar()
        for i in range(args.steps):
            dd = feeder.get()
            loss = train_step(dd)
            prev = reader.push(loss)            # loss of step i-1; waits for that step only
            if prev is not None and (i - 1) % 10 == 0:
                print(f"step {i - 1:4d} loss {prev:.4f}")
            feeder.advance()                    # H2D + plans of the next batch, side stream
            if evaluate and (i + 1) % args.eval_every == 0:
                evaluate(i)
        print(f"step {args.steps - 1:4d} loss {reader.flush():.4f}")
        feeder.close()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    print(f"{args.steps} steps in {dt:.2f} s = {args.batch * args.steps / dt:.0f} graphs/s"
          + (" (incl. evaluation)" if evaluate else ""))
    if evaluate:
        mae = evaluate(args.steps - 1)
        model.eval()                            # the same batches, eager and unpadded
        with torch.no_grad():
            pred = torch.cat([model(sp_datadict(hb, dev, keys)) for hb in eval_hbs])
        model.train()
        eager = float((pred - eval_y).abs().mean())
        print(f"eager no-grad evaluation MAE {eager:.6f} (|replay - eager| = {abs(mae - eager):.1e})")
        predictor.close()


if __name__ == "__main__":
    main()
