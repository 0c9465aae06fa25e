"""GPU tests of evaluation on the fused path: the eval epilogue of the Linear GEMM
(ops.linear_bn_eval, csrc/linear_stats.cu), its dispatch from the tuplewise MLP, eval-mode
model parity with the oracle models, and graph-replayed prediction (static.StaticPredictor)."""
import contextlib
import copy

import numpy as np
import pytest
import torch

from oracle import model_oracle as MO

pytestmark = pytest.mark.gpu
DEV = "cuda"
ACTS = {"none": 0, "silu": 1, "relu": 2}


def close(a, b, rtol):
    a = a.detach().cpu().double().numpy() if isinstance(a, torch.Tensor) else np.asarray(a, np.float64)
    b = b.detach().cpu().double().numpy() if isinstance(b, torch.Tensor) else np.asarray(b, np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    scale = max(1.0, float(np.abs(b).max()) if b.size else 1.0)
    err = float(np.abs(a - b).max(initial=0.0))
    assert err <= rtol * scale, (err, scale)


@contextlib.contextmanager
def tf32(flag):
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = flag
    try:
        yield
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


@contextlib.contextmanager
def c_calls(monkeypatch):
    """Names of the C entry points pygho_b200.ops calls inside the block."""
    from pygho_b200 import ops
    names = []
    real = ops.call

    def spy(name, *args):
        names.append(name)
        return real(name, *args)
    monkeypatch.setattr(ops, "call", spy)
    try:
        yield names
    finally:
        monkeypatch.setattr(ops, "call", real)


def _kernel():
    """The one-pass kernel's op, whatever the dispatch rule selects."""
    from pygho_b200 import ops
    return ops._ops.linear_bn_eval


def _operands(M, K, N, bias, affine, residual, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn(M, K, device=DEV, generator=g)
    w = torch.randn(N, K, device=DEV, generator=g) / K ** 0.5
    b = torch.randn(N, device=DEV, generator=g) if bias else None
    gamma = torch.rand(N, device=DEV, generator=g) + 0.5 if affine else None
    beta = torch.randn(N, device=DEV, generator=g) if affine else None
    rm = torch.randn(N, device=DEV, generator=g) * 0.5
    rv = 10.0 ** (torch.rand(N, device=DEV, generator=g) * 4 - 2)        # 1e-2 .. 1e2
    res = torch.randn(M, N, device=DEV, generator=g) if residual else None
    return x, w, b, gamma, beta, rm, rv, res


def _reference(x, w, b, gamma, beta, rm, rv, eps, act, res):
    d = lambda t: None if t is None else t.double()  # noqa: E731
    y = d(x) @ d(w).t()
    if b is not None:
        y = y + d(b)
    z = (y - d(rm)) / torch.sqrt(d(rv) + eps)
    if gamma is not None:
        z = z * d(gamma) + d(beta)
    z = {"none": z, "silu": torch.nn.functional.silu(z), "relu": torch.relu(z)}[act]
    return z if res is None else z + d(res)


FLAGS = [(True, True, True), (False, False, False), (True, False, True), (False, True, False)]
CASES = [(M, K, N, act, f) for N in (128, 256, 384) for K in (128, 384) for M in (4096, 4097)
         for act in ACTS for f in FLAGS]
CASES += [(230147, 384, 128, "silu", (True, True, True)), (230147, 384, 384, "silu", (True, True, True))]


@pytest.mark.parametrize("M,K,N,act,flags", CASES)
def test_linear_bn_eval_kernel_matches_fp64(M, K, N, act, flags):
    """One pass of act((x W^T + b - rm) / sqrt(rv + eps) * gamma + beta) (+ r) against fp64 torch,
    with non-trivial running statistics; TF32 tolerance as for linear_stats."""
    residual, bias, affine = flags
    x, w, b, gamma, beta, rm, rv, res = _operands(M, K, N, bias, affine, residual, M + K + N)
    rm0, rv0 = rm.clone(), rv.clone()
    z = _kernel()(x, w, b, gamma, beta, rm, rv, 1e-5, ACTS[act], res, None)
    want = _reference(x, w, b, gamma, beta, rm, rv, 1e-5, act, res)
    assert z.shape == (M, N) and bool(torch.isfinite(z).all())
    assert float((z.double() - want).abs().max()) <= 2e-3 * float(want.abs().max())
    assert torch.equal(rm, rm0) and torch.equal(rv, rv0)


@pytest.mark.parametrize("N,residual", [(128, True), (384, False)])
def test_linear_bn_eval_pad_rows(N, residual):
    """rows_dev = n < M: rows >= n are exactly 0, rows < n equal the call on the first n rows bit
    for bit."""
    M, K, n = 8192, 256, 5000
    x, w, b, gamma, beta, rm, rv, res = _operands(M, K, N, True, True, residual, 7)
    rows = torch.tensor([n], dtype=torch.int32, device=DEV)
    op = _kernel()
    z = op(x, w, b, gamma, beta, rm, rv, 1e-5, 1, res, rows)
    z_n = op(x[:n].contiguous(), w, b, gamma, beta, rm, rv, 1e-5, 1,
             None if res is None else res[:n].contiguous(), None)
    assert float(z[n:].abs().max()) == 0.0
    assert torch.equal(z[:n], z_n)


def _mlp(rows, cin, cout, act="silu", seed=0):
    """An MLP whose BatchNorms have non-trivial parameters and running statistics."""
    from pygho_b200.honn.utils import MLP
    torch.manual_seed(seed)
    mlp = MLP(cin, cout, 2, True, norm="bn", act=act, normparam=0.3).to(DEV)
    with torch.no_grad():
        for m in mlp.modules():
            if isinstance(m, torch.nn.BatchNorm1d):
                m.weight.uniform_(0.5, 1.5)
                m.bias.uniform_(-0.5, 0.5)
                m.running_mean.normal_(0.0, 0.5)
                m.running_var.copy_(10.0 ** (torch.rand_like(m.running_var) * 4 - 2))
                m.num_batches_tracked.fill_(7)
    return mlp.eval()


def _buffers(m):
    return {k: b.clone() for k, b in m.named_buffers()}


def _same_buffers(m, before):
    for k, b in m.named_buffers():
        assert torch.equal(b, before[k]), k


@pytest.mark.parametrize("rows,cin,cout,act", [(5000, 128, 128, "silu"), (777, 16, 12, "relu"),
                                               (4097, 384, 384, "silu")])
def test_fallback_path_matches_module_path(rows, cin, cout, act, monkeypatch):
    """Without TF32 the eval blocks run cuBLAS fp32 + the BatchNorm-apply kernel: the module
    path's GEMM, so they agree to 1e-5 (residual folded in too)."""
    mlp = _mlp(rows, cin, cout, act, seed=rows)
    before = _buffers(mlp)
    x = torch.randn(rows, cin, device=DEV) * 2 + 0.7
    r = torch.randn(rows, cout, device=DEV)
    with tf32(False), torch.no_grad(), c_calls(monkeypatch) as names:
        out = mlp(x)
        out_r = mlp(x, residual=r)
        ref = mlp.lins(x)
    assert "pgh_bn_act_res_fwd_f32" in names and "pgh_linear_bn_eval_f32" not in names
    close(out, ref, 1e-5)
    close(out_r, ref + r, 1e-5)
    _same_buffers(mlp, before)


@pytest.mark.parametrize("K,N", [(128, 128), (384, 128), (384, 384), (48, 128), (128, 192)])
@pytest.mark.parametrize("select", [False, True])
def test_linear_bn_eval_dispatch(K, N, select, monkeypatch):
    """ops.linear_bn_eval runs the one-pass kernel exactly where the selection rule lists the width
    and the kernel supports the shape (K % 32 == 0, N in {128, 256, 384}); everything else takes
    cuBLAS + the BatchNorm-apply kernel.  Both give the block's result."""
    from pygho_b200 import ops
    if select:
        monkeypatch.setattr(ops, "_EVAL_GEMM_WIDTHS", (128, 256, 384))
    M = 5000
    x, w, b, gamma, beta, rm, rv, res = _operands(M, K, N, True, True, True, K * N)
    bn = torch.nn.BatchNorm1d(N).to(DEV).eval()
    with torch.no_grad():
        bn.weight.copy_(gamma), bn.bias.copy_(beta), bn.running_mean.copy_(rm), bn.running_var.copy_(rv)
    want = _reference(x, w, b, gamma, beta, rm, rv, bn.eps, "silu", res)
    with tf32(True), torch.no_grad(), c_calls(monkeypatch) as names:
        z = ops.linear_bn_eval(x, w, b, bn, "silu", res)
    kernel = select and K % 32 == 0 and N in (128, 256, 384)
    assert names == (["pgh_linear_bn_eval_f32"] if kernel else ["pgh_bn_act_res_fwd_f32"])
    assert float((z.double() - want).abs().max()) <= 2e-3 * float(want.abs().max())


def test_linear_bn_eval_rejects_mismatched_shapes():
    op = _kernel()
    x = torch.randn(4096, 128, device=DEV)
    w = torch.randn(128, 128, device=DEV)
    v = torch.ones(128, device=DEV)
    with pytest.raises(ValueError, match="weight"):
        op(x, torch.randn(128, 96, device=DEV), None, None, None, v, v, 1e-5, 1)
    with pytest.raises(ValueError, match="running_var"):
        op(x, w, None, None, None, v, torch.ones(64, device=DEV), 1e-5, 1)


def test_eval_dispatch_and_no_side_effects(monkeypatch):
    """no_grad + eval: the selected one-pass kernel runs (one launch per block, residual folded);
    with gradients enabled the stock modules run, bit for bit; no running statistic ever changes."""
    from pygho_b200 import _lib, ops
    monkeypatch.setattr(ops, "_EVAL_GEMM_WIDTHS", (128,))
    mlp = _mlp(5000, 128, 128, seed=1)
    before = _buffers(mlp)
    x = torch.randn(5000, 128, device=DEV)
    r = torch.randn(5000, 128, device=DEV)
    with tf32(True):
        with torch.no_grad(), c_calls(monkeypatch) as names:
            n0 = _lib.launches()
            out = mlp(x, residual=r)
            assert _lib.launches() - n0 == 2
        assert names == ["pgh_linear_bn_eval_f32"] * 2
        with torch.no_grad():
            ref = mlp.lins(x) + r
        close(out, ref, 2e-3)
        xg = x.clone().requires_grad_(True)
        with c_calls(monkeypatch) as names:
            got = mlp(xg)
        assert names == []
        assert torch.equal(got, mlp.lins(xg))
    _same_buffers(mlp, before)


def _sp_model(conv="SSWL", layers=6, hidden=128, aggr="sum", seed=0):
    from examples.zinc_models import SpModel
    torch.manual_seed(seed)
    kw = dict(conv=conv, num_layer=layers, hiddim=hidden, aggr=aggr)
    return SpModel(**kw), kw


def _sp_batch(graphs, seed, keys):
    from pygho_b200.hodata.device import attach_host_plans, sp_datadict
    from pygho_b200.hodata.synthetic import make_batch
    hb = make_batch(graphs, seed=seed)
    dd = sp_datadict(hb, DEV, keys)
    attach_host_plans(hb, dd, keys)
    return hb, dd


def _train(model, dd, steps=3):
    model.train()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3)
    for _ in range(steps):
        opt.zero_grad()
        loss = torch.nn.functional.l1_loss(dd["y"].unsqueeze(-1), model(dd))
        loss.backward()
        opt.step()
    return float(loss)


def test_training_step_after_evaluation_is_unchanged():
    """Evaluating on a datadict (plans cached under no_grad) leaves the next training step on
    that datadict exactly as it would be without the evaluation."""
    from pygho_b200.honn.SpOperator import parse_precomputekey
    model, _kw = _sp_model(layers=2, seed=5)
    model = model.to(DEV)
    keys = parse_precomputekey(model)
    _hb, dd_a = _sp_batch(32, 21, keys)
    _hb, dd_b = _sp_batch(32, 21, keys)
    twin = copy.deepcopy(model)
    before = _buffers(model)
    with tf32(True):
        model.eval()
        with torch.no_grad():
            model(dd_a)
        _same_buffers(model, before)
        la = _train(model, dd_a, steps=1)
        lb = _train(twin, dd_b, steps=1)
    assert la == lb
    for (k, p), (_, q) in zip(model.named_parameters(), twin.named_parameters()):
        assert torch.equal(p, q), k
    for (k, p), (_, q) in zip(model.named_buffers(), twin.named_buffers()):
        assert torch.equal(p, q), k


@pytest.mark.parametrize("aggr,allow_tf32,tol", [("sum", False, 5e-4), ("mean", False, 5e-4),
                                                 ("sum", True, 1e-2)])
def test_sp_model_eval_matches_oracle_model(aggr, allow_tf32, tol, monkeypatch):
    """SSWL+ 6 x 128 trained for three steps (running statistics away from (0, 1)), then eval-mode
    predictions on another batch against the oracle model with the same state dict.  fp32 GEMMs
    (fallback) at the model-parity tolerance; the TF32 one-pass kernel (selected for N = 128
    here) at a TF32 tolerance."""
    from pygho_b200 import ops
    from pygho_b200.honn.SpOperator import parse_precomputekey
    monkeypatch.setattr(ops, "_EVAL_GEMM_WIDTHS", (128,))
    model, kw = _sp_model(aggr=aggr)
    model = model.to(DEV)
    keys = parse_precomputekey(model)
    _hb, dd = _sp_batch(64, 17, keys)
    _train(model, dd)
    oracle = MO.OSpModel(**kw)
    oracle.load_state_dict({k: v.cpu() for k, v in model.state_dict().items()})
    assert all(float((m.running_var - 1).abs().max()) > 1e-4
               for m in model.modules() if isinstance(m, torch.nn.BatchNorm1d))
    hb, dd = _sp_batch(64, 99, keys)
    model.eval(), oracle.eval()
    before = _buffers(model)
    with tf32(allow_tf32), torch.no_grad(), c_calls(monkeypatch) as names:
        pred = model(dd)
    assert ("pgh_linear_bn_eval_f32" in names) == allow_tf32
    _same_buffers(model, before)
    g = MO.host_graph_dict(hb, {k + "___acd": torch.from_numpy(v) for k, v in hb.plans.items()})
    with torch.no_grad():
        opred = oracle(g)
    close(pred, opred, tol)


def test_ma_model_eval_matches_oracle_model():
    """Dense PPGN model, trained for three steps, eval-mode predictions against the oracle."""
    from examples.zinc_models import MaModel
    from pygho_b200.hodata.device import ma_datadict
    from pygho_b200.hodata.synthetic import make_batch
    torch.manual_seed(3)
    kw = dict(num_layer=2, hiddim=32, npool="sum", lpool="mean", mlplayer=2, outlayer=2)
    model = MaModel("PPGN", **kw).to(DEV)
    _train(model, ma_datadict(make_batch(7, seed=5), DEV))
    oracle = MO.OMaModel(**kw)
    oracle.load_state_dict({k: v.cpu() for k, v in model.state_dict().items()})
    hb = make_batch(9, seed=6)
    dd = ma_datadict(hb, DEV)
    g = MO.host_dense_dict(hb)
    assert torch.equal(dd["X"].data.cpu(), g["X"]) and torch.equal(dd["A"].data.cpu(), g["A"])
    model.eval(), oracle.eval()
    before = _buffers(model)
    with tf32(False), torch.no_grad():
        pred = model(dd)
        opred = oracle(g)
    _same_buffers(model, before)
    close(pred, opred, 5e-4)


def test_static_predictor_matches_eager_eval():
    """Graph-replayed prediction over three batches of different graph counts equals eager eval
    of the unpadded batches; it follows an optimizer step; the training flag is restored."""
    from pygho_b200 import static as ST
    from pygho_b200.honn.SpOperator import parse_precomputekey
    model, _kw = _sp_model(layers=2, seed=8)
    model = model.to(DEV)
    keys = parse_precomputekey(model)
    batches = [_sp_batch(n, 50 + n, keys) for n in (40, 32, 48)]
    hbs = [hb for hb, _dd in batches]
    caps = ST.capacities(hbs, keys)

    def eager():
        model.eval()
        with torch.no_grad():
            out = torch.cat([model(dd) for _hb, dd in batches])
        model.train()
        return out

    with tf32(True):
        _train(model, batches[0][1], steps=1)
        model.train()
        pred = ST.StaticPredictor(hbs, caps, torch.device(DEV, 0), keys, model)
        assert model.training
        before = _buffers(model)
        got = pred()
        assert got.shape == (120, 1)
        close(got, eager(), 1e-5)
        _same_buffers(model, before)
        _train(model, batches[1][1], steps=1)          # in-place parameter / statistics updates
        got2 = pred()
        assert float((got2 - got).abs().max()) > 0
        close(got2, eager(), 1e-5)
        pred.close()
