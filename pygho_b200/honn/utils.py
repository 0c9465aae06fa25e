"""MLP and normalisation blocks used around the tensor operators (reference
``pygho/honn/utils.py``: ``NormMomentumScheduler`` :10, ``NoneNorm`` :36, ``BatchNorm`` :46,
``LayerNorm`` :65, ``MLP`` :85-142).  Stock torch modules: the dense GEMM / norm kernels
are out of the hot-path scope (SURVEY.md section 2, row 12) and are reused as they are."""
from __future__ import annotations

from typing import Callable

import torch.nn as nn
from torch import Tensor


class NormMomentumScheduler:
    """Scales the momentum of every norm layer of type ``normtype`` by ``mfunc(epoch)``."""

    def __init__(self, mfunc: Callable, initmomentum: float, normtype=nn.BatchNorm1d) -> None:
        self.normtype, self.mfunc = normtype, mfunc
        self.epoch, self.initmomentum = 0, initmomentum

    def step(self, model: nn.Module):
        ratio = self.mfunc(self.epoch)
        if abs(ratio - 1) < 1e-6:
            return self.initmomentum
        momentum = self.initmomentum * ratio
        self.epoch += 1
        for mod in model.modules():
            if type(mod) is self.normtype:
                mod.momentum = momentum
        return momentum


class NoneNorm(nn.Module):
    def __init__(self, dim=0, normparam=0) -> None:
        super().__init__()
        self.num_features = dim

    def forward(self, x):
        return x


class BatchNorm(nn.Module):
    """BatchNorm1d over all leading dims flattened (all tuples of the batch)."""

    def __init__(self, dim, normparam=0.1) -> None:
        super().__init__()
        self.num_features = dim
        self.norm = nn.BatchNorm1d(dim, momentum=normparam)

    def forward(self, x: Tensor):
        if x.dim() < 2:
            raise NotImplementedError
        if x.dim() == 2:
            return self.norm(x)
        return self.norm(x.flatten(0, -2)).reshape(x.shape)


class LayerNorm(nn.Module):
    def __init__(self, dim, normparam=0.1) -> None:
        super().__init__()
        self.num_features = dim
        self.norm = nn.LayerNorm(dim)

    def forward(self, x: Tensor):
        return self.norm(x)


class Embedding(nn.Embedding):
    """``nn.Embedding`` whose CUDA path gathers with the seg_gmr kernel and computes the weight
    gradient deterministically from a per-batch plan cached on the index tensor (the integer
    node / edge / tuple labels of a batch never change).  Same parameters and state dict;
    ``padding_idx`` / ``max_norm`` / ``sparse`` tables and non-fp32 weights use torch's path."""

    def forward(self, input: Tensor) -> Tensor:
        import torch
        if (input.is_cuda and self.weight.dtype == torch.float32 and self.padding_idx is None
                and self.max_norm is None and not self.sparse and not self.scale_grad_by_freq
                and input.dtype in (torch.int64, torch.int32) and input.numel() > 0
                and self.embedding_dim % 4 == 0):
            from .. import plans as P
            from ..ops import EmbeddingGather
            return EmbeddingGather.apply(self.weight, input,
                                         P.embedding_plan(input, self.num_embeddings))
        return super().forward(input)


normdict = {"bn": BatchNorm, "ln": LayerNorm, "none": NoneNorm}
act_dict = {"relu": nn.ReLU(inplace=True), "ELU": nn.ELU(inplace=True),
            "silu": nn.SiLU(inplace=True)}


class MLP(nn.Module):
    """``numlayer`` x [Linear, norm, (Dropout), act]; the last block keeps norm/act only
    when ``tailact``.  Hidden blocks are hiddim->hiddim, the last one hiddim->outdim."""

    def __init__(self, hiddim: int, outdim: int, numlayer: int, tailact: bool, dp: float = 0,
                 norm: str = "bn", act: str = "relu", tailbias=True, normparam: float = 0.1) -> None:
        super().__init__()
        assert numlayer >= 0
        if numlayer == 0:
            assert hiddim == outdim
            self.lins = NoneNorm()
            return

        def tail(width):
            blk = [normdict[norm](width, normparam)]
            if dp > 0:
                blk.append(nn.Dropout(dp, inplace=True))
            blk.append(act_dict[act])
            return blk

        layers = []
        for _ in range(numlayer - 1):
            layers += [nn.Linear(hiddim, hiddim)] + tail(hiddim)
        layers.append(nn.Linear(hiddim, outdim, bias=tailbias))
        if tailact:
            layers += tail(outdim)
        self.lins = nn.Sequential(*layers)

    def forward(self, x: Tensor, residual: Tensor = None):
        """``residual`` (same shape as the output) is added to the result; when the MLP ends
        with a fused Linear-BatchNorm-activation block the addition happens inside that
        block's kernel instead of a separate pass."""
        if not _fusable(self.lins, x):
            out = self.lins(x)
            return out if residual is None else out + residual
        # Linear -> BatchNorm(train) -> SiLU/ReLU blocks go through the fused kernels
        # (pygho_b200/csrc/fused_mlp.cu), inference blocks (BatchNorm in eval mode, no autograd)
        # through ops.linear_bn_eval; anything else runs module by module.
        from .. import static
        from ..ops import ACT_CODE, LinearBNAct, linear_bn_eval
        mods = list(self.lins)
        shape = x.shape
        h = x.reshape(-1, shape[-1])
        i = 0
        while i < len(mods):
            m = mods[i]
            blk = _match_block(mods, i)
            if blk is not None:
                bn, act = blk
                res = None
                if residual is not None and i + 3 == len(mods):
                    res, residual = residual.reshape(-1, residual.shape[-1]), None
                h = LinearBNAct.apply(h, m.weight, m.bias, bn.weight, bn.bias, bn.running_mean,
                                      bn.running_var, bn.momentum, bn.eps, ACT_CODE[act], res,
                                      static.rows_dev_for(h.shape[0]),
                                      getattr(bn, "_pgh_sync_group", None),
                                      bn.num_batches_tracked if bn.track_running_stats else None)
                i += 3
                continue
            blk = _match_eval_block(mods, i)
            if blk is not None:
                bn, act, n = blk
                res = None
                if residual is not None and i + n == len(mods):
                    res, residual = residual.reshape(-1, residual.shape[-1]), None
                h = linear_bn_eval(h, m.weight, m.bias, bn, act, res, static.rows_dev_for(h.shape[0]))
                i += n
            else:
                h = m(h)
                i += 1
        h = h.reshape(shape[:-1] + (h.shape[-1],))
        return h if residual is None else h + residual


def _match_block(mods, i):
    """(BatchNorm1d, act name) if mods[i:i+3] is Linear, BatchNorm(train, affine), SiLU/ReLU."""
    if i + 2 >= len(mods) or not isinstance(mods[i], nn.Linear) or type(mods[i + 1]) is not BatchNorm:
        return None
    bn = mods[i + 1].norm
    act = {nn.SiLU: "silu", nn.ReLU: "relu"}.get(type(mods[i + 2]))
    if act is None or not bn.training or bn.momentum is None or bn.num_features % 4 \
            or bn.num_features > 1024:
        return None
    return bn, act


def _match_eval_block(mods, i):
    """(BatchNorm1d, act name, block length) if mods[i:] starts with Linear, BatchNorm(eval, running
    statistics), [Dropout(eval)], SiLU/ReLU and autograd is off: an inference block that needs no
    backward, so the BatchNorm folds into the GEMM epilogue.  With gradients enabled (e.g. fine-
    tuning with a frozen BatchNorm) the block stays on the stock modules."""
    import torch
    if torch.is_grad_enabled() or i + 2 >= len(mods) or not isinstance(mods[i], nn.Linear) \
            or type(mods[i + 1]) is not BatchNorm:
        return None
    bn = mods[i + 1].norm
    j = i + 2
    if isinstance(mods[j], nn.Dropout) and not mods[j].training and j + 1 < len(mods):
        j += 1
    act = {nn.SiLU: "silu", nn.ReLU: "relu"}.get(type(mods[j]))
    if act is None or bn.training or not bn.track_running_stats or bn.running_mean is None \
            or bn.num_features % 4 or bn.num_features > 1024:
        return None
    return bn, act, j + 1 - i


def _fusable(lins, x: Tensor) -> bool:
    import torch
    return (isinstance(lins, nn.Sequential) and x.is_cuda and x.dtype == torch.float32
            and x.numel() > 0 and torch.is_grad_enabled() is not None
            and any(_match_block(list(lins), i) is not None or _match_eval_block(list(lins), i)
                    is not None for i in range(len(lins))))
