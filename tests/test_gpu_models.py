"""GPU parity at layer and model level: product layers (CUDA kernels) against the golden
outputs of the real reference layers and against the CPU oracle model."""
import copy

import numpy as np
import pytest
import torch

from oracle import model_oracle as MO

pytestmark = pytest.mark.gpu
DEV = "cuda"


def T(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def close(a, b, rtol):
    a = a.detach().cpu().double().numpy() if isinstance(a, torch.Tensor) else np.asarray(a, np.float64)
    b = b.detach().cpu().double().numpy() if isinstance(b, torch.Tensor) else np.asarray(b, np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    scale = max(1.0, float(np.abs(b).max()) if b.size else 1.0)
    err = float(np.abs(a - b).max(initial=0.0))
    assert err <= rtol * scale, (err, scale)


MLP = {"numlayer": 2, "tailact": True, "norm": "bn", "act": "silu", "dp": 0.0}


def test_convs_match_reference_golden(golden):
    from pygho_b200 import SparseTensor
    from pygho_b200.honn import Conv
    g = golden("conv")
    ei, tid, N = T(g["edge_index"]), T(g["tupleid"]), int(g["N"])
    dd = {k: T(v) for k, v in g.items() if k.endswith("___acd")}
    mk = {"NGNN": lambda: Conv.NGNNConv(8, 8, "sum", "SS", dict(MLP)),
          "SSWL": lambda: Conv.SSWLConv(8, 8, "sum", "SS", dict(MLP)),
          "SSWLmax": lambda: Conv.SSWLConv(8, 8, "max", "SS", dict(MLP)),
          "DSSGNN": lambda: Conv.DSSGNNConv(8, 8, "sum", "sum", "mean", "SS", dict(MLP)),
          "PPGN": lambda: Conv.PPGNConv(8, 8, "sum", "SS", dict(MLP))}
    for name, fn in mk.items():
        conv = fn()
        sd = {k[len(name) + 4:]: torch.from_numpy(v) for k, v in g.items()
              if k.startswith(name + ".sd.")}
        conv.load_state_dict(sd)
        conv = conv.to(DEV)
        A = SparseTensor(ei, T(g["Av"]), (N, N, 8), True)
        xv = T(g["Xv"]).requires_grad_(True)
        X = SparseTensor(tid, xv, (N, N, 8), True)
        Y = conv(A, X, dd)
        assert Y.indices is tid
        (Y.values ** 2).mean().backward()
        close(Y.values, g[f"{name}.out"], 2e-5)
        close(xv.grad, g[f"{name}.gradX"], 5e-5)
        for k, p in conv.named_parameters():
            close(p.grad, g[f"{name}.grad.{k}"], 1e-4)


@pytest.mark.parametrize("conv,aggr,lpool,npool", [("SSWL", "sum", "mean", "sum"),
                                                   ("SSWL", "max", "max", "mean"),
                                                   ("NGNN", "mean", "sum", "max"),
                                                   ("DSSGNN", "sum", "mean", "sum"),
                                                   ("PPGN", "sum", "mean", "sum"),
                                                   ("I2GNN", "sum", "mean", "sum"),
                                                   ("I2GNN", "max", "max", "mean")])
def test_sp_model_matches_oracle_model(conv, aggr, lpool, npool):
    """Whole model, forward + backward, device-built plans: loss and every parameter
    gradient against the CPU oracle model with identical weights."""
    from examples.zinc_models import SpModel
    from pygho_b200.hodata.device import attach_host_plans, sp_datadict
    from pygho_b200.hodata.synthetic import make_batch
    from pygho_b200.honn.SpOperator import parse_precomputekey
    torch.manual_seed(0)
    hb = make_batch(6, seed=3, tuples="i2" if conv == "I2GNN" else "khop")
    kw = dict(conv=conv, num_layer=2, hiddim=32, aggr=aggr, npool=npool, lpool=lpool,
              mlplayer=2, outlayer=2)
    model = SpModel(**kw)
    oracle = MO.OSpModel(**{k: v for k, v in kw.items()})
    oracle.load_state_dict(copy.deepcopy(model.state_dict()))
    model = model.to(DEV)
    keys = parse_precomputekey(model)
    dd = sp_datadict(hb, DEV, keys)
    attach_host_plans(hb, dd, keys)
    g = MO.host_graph_dict(hb, {k + "___acd": torch.from_numpy(v) for k, v in hb.plans.items()})
    pred = model(dd)
    loss = torch.nn.functional.l1_loss(dd["y"].unsqueeze(-1), pred)
    loss.backward()
    opred = oracle(g)
    oloss = torch.nn.functional.l1_loss(g["y"].unsqueeze(-1), opred)
    oloss.backward()
    close(pred, opred, 1e-4)
    close(loss, oloss, 1e-4)
    ograds = dict(oracle.named_parameters())
    for k, p in model.named_parameters():
        if ograds[k].grad is None:          # e.g. the edge encoder of PPGN (A is unused)
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, k
            continue
        close(p.grad, ograds[k].grad, 2e-3)


def test_i2conv_matches_reference_golden(golden):
    """I2Conv on 3-D tuples, the 3-D tupleinit (zinc.py:270-273) and the read-out chain
    OpPoolingSubg3D -> OpPoolingSubg2D (zinc.py:258) against the REAL reference
    (tests/golden/conv_i2.npz): layer output, read-out, input and parameter gradients."""
    from pygho_b200 import SparseTensor
    from pygho_b200.honn import Conv
    from pygho_b200.honn.TensorOp import OpPoolingSubg2D, OpPoolingSubg3D
    g = golden("conv_i2")
    ei, tid, N = T(g["edge_index"]), T(g["tupleid"]), int(g["N"])
    dd = {k: T(v) for k, v in g.items() if k.endswith("___acd")}
    for name, aggr, pool in (("I2", "sum", "mean"), ("I2max", "max", "max")):
        conv = Conv.I2Conv(8, 8, aggr, "SS", dict(MLP))
        conv.load_state_dict({k[len(name) + 4:]: torch.from_numpy(v) for k, v in g.items()
                              if k.startswith(name + ".sd.")})
        conv = conv.to(DEV)
        lins = [torch.nn.Linear(8, 8) for _ in range(3)]
        for i, lin in enumerate(lins):
            lin.load_state_dict({"weight": torch.from_numpy(g[f"{name}.init{i}.weight"]),
                                 "bias": torch.from_numpy(g[f"{name}.init{i}.bias"])})
            lin.to(DEV)
        lpool = torch.nn.Sequential(OpPoolingSubg3D("S", pool), OpPoolingSubg2D("S", pool))
        A = SparseTensor(ei, T(g["Av"]), (N, N, 8), True)
        xv = T(g["Xv"]).requires_grad_(True)
        xn = T(g["xn"]).requires_grad_(True)
        X = SparseTensor(tid, xv, (N, N, N, 8), True)
        root = X.unpooling_fromdense1dim(0, lins[0](xn)).values
        node = X.unpooling_fromdense1dim(1, lins[1](xn)).values
        third = X.unpooling_fromdense1dim(1, lins[2](xn)).values
        X = X.tuplewiseapply(lambda val: root * node * third * val)
        Y = conv(A, X, dd)
        h = lpool(X.add(Y, True))
        ((h ** 2).mean() + (Y.values ** 2).mean()).backward()
        close(Y.values, g[f"{name}.out"], 2e-5)
        close(h, g[f"{name}.readout"], 2e-5)
        close(xv.grad, g[f"{name}.gradX"], 1e-4)
        close(xn.grad, g[f"{name}.gradx"], 1e-4)
        for k, p in conv.named_parameters():
            close(p.grad, g[f"{name}.grad.{k}"], 1e-4)
        for i, lin in enumerate(lins):
            close(lin.weight.grad, g[f"{name}.init{i}.gweight"], 1e-4)
            close(lin.bias.grad, g[f"{name}.init{i}.gbias"], 1e-4)


@pytest.mark.parametrize("aggr", ("sum", "mean"))
def test_bench_path_sswl_6x128_matches_oracle_model(aggr):
    """The configuration bench.py times -- SpModel("SSWL", 6 layers, hidden 128, residual folded
    into the MLP's last kernel), i.e. the fused SswlAggregate epilogue + lean streaming kernel +
    residual-in-BatchNorm + EmbeddingGather path (all need d % 128 == 0) -- on a 64-graph batch
    against the CPU oracle model with identical weights: prediction, loss, every gradient."""
    from examples.zinc_models import SpModel
    from pygho_b200.hodata.device import attach_host_plans, sp_datadict
    from pygho_b200.hodata.synthetic import make_batch
    from pygho_b200.honn.SpOperator import parse_precomputekey
    torch.manual_seed(0)
    hb = make_batch(64, seed=17)
    kw = dict(conv="SSWL", num_layer=6, hiddim=128, aggr=aggr)
    model = SpModel(**kw)
    oracle = MO.OSpModel(**kw)
    oracle.load_state_dict(copy.deepcopy(model.state_dict()))
    model = model.to(DEV)
    keys = parse_precomputekey(model)
    dd = sp_datadict(hb, DEV, keys)
    attach_host_plans(hb, dd, keys)
    g = MO.host_graph_dict(hb, {k + "___acd": torch.from_numpy(v) for k, v in hb.plans.items()})
    from pygho_b200 import _lib
    n0 = _lib.launches()
    pred = model(dd)
    loss = torch.nn.functional.l1_loss(dd["y"].unsqueeze(-1), pred)
    loss.backward()
    assert _lib.launches() - n0 > 100            # the CUDA kernels ran (no silent fallback)
    opred = oracle(g)
    oloss = torch.nn.functional.l1_loss(g["y"].unsqueeze(-1), opred)
    oloss.backward()
    close(pred, opred, 5e-4)
    close(loss, oloss, 5e-4)
    ograds = dict(oracle.named_parameters())
    for k, p in model.named_parameters():
        close(p.grad, ograds[k].grad, 5e-3)
    # running statistics of every BatchNorm were updated identically
    obuf = dict(oracle.named_buffers())
    for k, b in model.named_buffers():
        if b.dtype.is_floating_point:
            close(b, obuf[k], 1e-4)


@pytest.mark.parametrize("algo,tol", [(0, 1.0), (2, 200.0)])
def test_ppgn_dense_conv_matches_reference_golden(golden, monkeypatch, algo, tol):
    """PPGNConv DD (mamamm kernels) against the REAL reference on equal-size graphs
    (tests/golden/conv_dd.npz); exact-fp32 kernel at 5e-5, TF32 tensor-core kernel at 1e-2."""
    monkeypatch.setenv("PYGHO_B200_MAMAMM_ALGO", str(algo))
    from pygho_b200 import MaskedTensor
    from pygho_b200.honn import Conv
    g = golden("conv_dd")
    conv = Conv.PPGNConv(8, 8, "sum", "DD", dict(MLP))
    conv.load_state_dict({k[3:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("sd.")})
    conv = conv.to(DEV)
    xd = T(g["X"]).requires_grad_(True)
    Y = conv(None, MaskedTensor(xd, T(g["mask"])), {})
    (Y.data ** 2).mean().backward()
    close(Y.data, g["out"], 5e-5 * tol)
    close(xd.grad, g["gradX"], 5e-5 * tol)
    for k, p in conv.named_parameters():
        close(p.grad, g[f"grad.{k}"], 1e-4 * tol)


@pytest.mark.parametrize("algo,tol", [(0, 1.0), (2, 50.0), (4, 1.0)])
def test_ma_model_matches_oracle_model(monkeypatch, algo, tol):
    """Dense PPGN model (example/zinc.py:155-219; bench.py --workload ppgn_dd) on ragged graphs:
    prediction, loss and every parameter gradient against the CPU oracle model."""
    monkeypatch.setenv("PYGHO_B200_MAMAMM_ALGO", str(algo))
    from examples.zinc_models import MaModel
    from pygho_b200.hodata.device import ma_datadict
    from pygho_b200.hodata.synthetic import make_batch
    torch.manual_seed(3)
    hb = make_batch(7, seed=5)
    kw = dict(num_layer=2, hiddim=32, npool="sum", lpool="mean", mlplayer=2, outlayer=2)
    model = MaModel("PPGN", **kw)
    oracle = MO.OMaModel(**kw)
    oracle.load_state_dict(copy.deepcopy(model.state_dict()))
    model = model.to(DEV)
    dd = ma_datadict(hb, DEV)
    g = MO.host_dense_dict(hb)
    assert torch.equal(dd["X"].data.cpu(), g["X"]) and torch.equal(dd["A"].data.cpu(), g["A"])
    pred = model(dd)
    loss = torch.nn.functional.l1_loss(dd["y"].unsqueeze(-1), pred)
    loss.backward()
    opred = oracle(g)
    oloss = torch.nn.functional.l1_loss(g["y"].unsqueeze(-1), opred)
    oloss.backward()
    close(pred, opred, 1e-4 * tol)
    close(loss, oloss, 1e-4 * tol)
    ograds = dict(oracle.named_parameters())
    for k, p in model.named_parameters():
        if ograds[k].grad is None:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, k
            continue
        close(p.grad, ograds[k].grad, 2e-3 * tol)


def test_sp_model_host_plans_equal_device_plans():
    """Shipping precomputed (host) plans gives bit-identical predictions to building
    them on the device."""
    from examples.zinc_models import SpModel
    from pygho_b200.hodata.device import attach_host_plans, sp_datadict
    from pygho_b200.hodata.synthetic import make_batch
    from pygho_b200.honn.SpOperator import parse_precomputekey
    torch.manual_seed(1)
    hb = make_batch(5, seed=9)
    model = SpModel("SSWL", num_layer=2, hiddim=16).to(DEV).eval()
    keys = parse_precomputekey(model)
    dd = sp_datadict(hb, DEV, keys)
    p1 = model(dd)
    attach_host_plans(hb, dd, keys)
    p2 = model(sp_datadict(hb, DEV, keys))
    assert torch.equal(p1, p2)


def test_i2_and_gnnak_models_run():
    from examples.zinc_models import SpModel
    from pygho_b200.hodata.device import sp_datadict
    from pygho_b200.hodata.synthetic import make_batch
    from pygho_b200.honn.SpOperator import parse_precomputekey
    torch.manual_seed(2)
    for conv, tuples in (("I2GNN", "i2"), ("GNNAK", "khop")):
        hb = make_batch(3, seed=4, tuples=tuples)
        model = SpModel(conv, num_layer=2, hiddim=16).to(DEV)
        dd = sp_datadict(hb, DEV, parse_precomputekey(model))
        pred = model(dd)
        assert pred.shape == (3, 1) and bool(torch.isfinite(pred).all())
        pred.sum().backward()
        assert all(p.grad is not None and bool(torch.isfinite(p.grad).all())
                   for p in model.parameters() if p.requires_grad and p.grad is not None)


@pytest.mark.parametrize("algo,tol", [(0, 1.0), (1, 500.0), (2, 500.0)])
def test_ppgn_dense_conv_matches_einsum(monkeypatch, algo, tol):
    """PPGNConv in DD mode (mamamm) against a torch restatement with the same weights
    (exact-fp32 kernel at 2e-5; TF32 tensor-core kernel at 1e-2)."""
    monkeypatch.setenv("PYGHO_B200_MAMAMM_ALGO", str(algo))
    from pygho_b200 import MaskedTensor
    from pygho_b200.honn import Conv
    torch.manual_seed(3)
    b, n, d = 4, 9, 16
    sizes = torch.tensor([9, 5, 7, 3])
    ar = torch.arange(n)
    mask = (ar[None, :, None] < sizes[:, None, None]) & (ar[None, None, :] < sizes[:, None, None])
    data = torch.randn(b, n, n, d) * mask.unsqueeze(-1)
    conv = Conv.PPGNConv(d, d, "sum", "DD", dict(MLP))
    ref = copy.deepcopy(conv)
    xr = data.clone().requires_grad_(True)
    m = mask.unsqueeze(-1)
    h1, h2 = ref.lin1(xr * m) * m, ref.lin2(xr * m) * m
    oref = torch.einsum("bijd,bjkd->bikd", h1, h2) * m
    (oref ** 2).mean().backward()
    conv = conv.to(DEV)
    xg = data.to(DEV).requires_grad_(True)
    X = MaskedTensor(xg, mask.to(DEV))
    out = conv(None, X, {})
    (out.data ** 2).mean().backward()
    close(out.data, oref, 2e-5 * tol)
    close(xg.grad, xr.grad, 1e-4 * min(tol, 100.0))
    for (k, p), (_, q) in zip(conv.named_parameters(), ref.named_parameters()):
        close(p.grad, q.grad, 2e-4 * min(tol, 50.0))


def test_ma_model_runs_and_masks():
    from examples.zinc_models import MaModel
    from pygho_b200.hodata.device import ma_datadict
    from pygho_b200.hodata.synthetic import make_batch
    torch.manual_seed(4)
    hb = make_batch(4, seed=8)
    for conv in ("PPGN", "SSWL", "NGNN"):
        model = MaModel(conv, num_layer=2, hiddim=16).to(DEV)
        pred = model(ma_datadict(hb, DEV))
        assert pred.shape == (4, 1) and bool(torch.isfinite(pred).all())
        pred.sum().backward()


@pytest.mark.parametrize("rows,cin,cout,act", [(1000, 24, 8, "silu"), (4097, 128, 128, "silu"),
                                               (3001, 384, 384, "silu"), (777, 16, 12, "relu")])
def test_fused_linear_bn_act_matches_torch(rows, cin, cout, act):
    """MLP block through the fused kernels vs the same modules run one by one by torch:
    output, running statistics and every gradient."""
    from pygho_b200.honn.utils import MLP
    torch.manual_seed(rows)
    mlp = MLP(cin, cout, 2, True, norm="bn", act=act, normparam=0.3).to(DEV)
    with torch.no_grad():
        for m in mlp.modules():
            if isinstance(m, torch.nn.BatchNorm1d):
                m.weight.uniform_(0.5, 1.5)
                m.bias.uniform_(-0.5, 0.5)
    ref = copy.deepcopy(mlp)
    x = torch.randn(rows, cin, device=DEV) * 2 + 0.7
    xr = x.clone().requires_grad_(True)
    xf = x.clone().requires_grad_(True)
    w = torch.randn(rows, cout, device=DEV)
    out_ref = ref.lins(xr)                    # plain torch path (Sequential, module by module)
    (out_ref * w).sum().backward()
    out = mlp(xf)                             # fused path
    (out * w).sum().backward()
    close(out, out_ref, 2e-5)
    close(xf.grad, xr.grad, 5e-5)
    for (k, p), (_, q) in zip(mlp.named_parameters(), ref.named_parameters()):
        if k.endswith("bias") and "norm" not in k:
            # a Linear bias in front of a training-mode BatchNorm has gradient sum(dy) == 0
            # exactly; both implementations return rounding noise of the size of one ulp of
            # sum(|dy|), which cannot agree digit by digit
            assert float(p.grad.abs().max()) < 2e-3 and float(q.grad.abs().max()) < 2e-3
            continue
        close(p.grad, q.grad, 1e-4)
    for (k, p), (_, q) in zip(mlp.named_buffers(), ref.named_buffers()):
        close(p.float(), q.float(), 1e-5)
    # eval mode falls back to the stock modules and agrees
    mlp.eval(), ref.eval()
    close(mlp(x), ref.lins(x), 1e-5)


def test_step_graph_replay_matches_eager_training():
    """A CUDA-graph replay of the whole training step (pygho_b200/graph.py) updates the model
    exactly like the eager step: same kernels, same order, deterministic reductions."""
    from examples.zinc_models import SpModel
    from pygho_b200.dist import FlatGradBucket
    from pygho_b200.graph import StepGraph
    from pygho_b200.hodata.device import prefetch_plans, sp_datadict
    from pygho_b200.hodata.synthetic import make_batch
    from pygho_b200.honn.SpOperator import parse_precomputekey
    hb = make_batch(24, seed=21)

    def build():
        torch.manual_seed(5)
        model = SpModel("SSWL", num_layer=2, hiddim=32).to(DEV)
        keys = parse_precomputekey(model)
        dd = sp_datadict(hb, DEV, keys)
        prefetch_plans(dd, keys)
        bucket = FlatGradBucket(model.parameters())
        opt = torch.optim.AdamW(model.parameters(), lr=1e-3, fused=True, capturable=True)

        def step():
            bucket.zero()
            loss = torch.nn.functional.l1_loss(dd["y"].unsqueeze(-1), model(dd))
            loss.backward()
            opt.step()
            return loss.detach()
        return model, step

    m_eager, step_eager = build()
    eager_losses, eager_state = [], None
    for i in range(4):
        eager_losses.append(float(step_eager()))
        if i == 1:
            eager_state = {k: v.detach().clone().float() for k, v in m_eager.state_dict().items()}
    m_graph, step_graph = build()
    sg = StepGraph(step_graph, warmup=1)                 # 1 eager step, then capture
    assert sg.launches > 10                              # our kernels are inside the graph
    graph_losses = [float(sg.replay())]
    # after two updates the two models agree to rounding.  (Later states are compared through
    # the loss only: Linear biases in front of a BatchNorm have a mathematically zero gradient,
    # Adam normalises the ~1e-9 atomics noise of torch's embedding backward to +-lr steps.)
    for k, q in m_graph.state_dict().items():
        close(q.float(), eager_state[k], 1e-6)
    graph_losses += [float(sg.replay()) for _ in range(2)]
    for a, b in zip(eager_losses[1:], graph_losses):
        assert abs(a - b) <= 1e-5 * max(1.0, abs(a)), (eager_losses, graph_losses)


@pytest.mark.parametrize("threaded", [False, True])
def test_device_prefetcher_feeds_identical_batches(threaded):
    from pygho_b200.hodata.device import DevicePrefetcher, sp_datadict
    from pygho_b200.hodata.synthetic import make_batch
    keys = ["X___X___1___A___0", "X___A___1___X___0"]
    hbs = [make_batch(6 + i, seed=30 + i) for i in range(3)]
    want = [sp_datadict(hb, DEV, keys) for hb in hbs]
    feeder = DevicePrefetcher(hbs, torch.device(DEV, 0), keys, threaded=threaded)
    for i in range(7):
        dd = feeder.get()
        w = want[i % 3]
        assert torch.equal(dd["X"].indices, w["X"].indices) and torch.equal(dd["x"], w["x"])
        for k in keys:
            a = dd[k + "___acd"]
            b = w[k + "___acd"]
            ka = torch.sort((a[0] * (1 << 40)) + (a[1] << 20) + a[2]).values
            kb = torch.sort((b[0] * (1 << 40)) + (b[1] << 20) + b[2]).values
            assert torch.equal(ka, kb)
        torch.cuda.synchronize()
        feeder.advance()
    feeder.close()
