"""The inference-block matcher of the tuplewise MLP (honn/utils.py): which eval-mode
Linear -> BatchNorm -> activation blocks go to ops.linear_bn_eval.  Module lists only: no GPU."""
import pytest
import torch
import torch.nn as nn


def _mlp(width=128, act="silu", dp=0.0, norm="bn"):
    from pygho_b200.honn.utils import MLP
    return MLP(width, width, 2, True, dp=dp, norm=norm, act=act)


def _match(mlp, i=0):
    from pygho_b200.honn.utils import _match_eval_block
    return _match_eval_block(list(mlp.lins), i)


@pytest.mark.parametrize("act,dp,length", [("silu", 0.0, 3), ("relu", 0.0, 3), ("silu", 0.2, 4)])
def test_eval_blocks_are_accepted(act, dp, length):
    mlp = _mlp(act=act, dp=dp).eval()
    with torch.no_grad():
        blk = _match(mlp)
        assert blk is not None
        bn, name, n = blk
        assert bn is mlp.lins[1].norm and name == act and n == length
        assert _match(mlp, length) is not None               # the second block too
        assert _match(mlp, 1) is None                        # not at a BatchNorm


def test_training_batchnorm_is_rejected():
    mlp = _mlp()
    with torch.no_grad():
        assert _match(mlp) is None
        mlp.eval()
        mlp.lins[1].norm.train()
        assert _match(mlp) is None


def test_untracked_running_statistics_are_rejected():
    mlp = _mlp().eval()
    mlp.lins[1].norm = nn.BatchNorm1d(128, track_running_stats=False).eval()
    with torch.no_grad():
        assert _match(mlp) is None


def test_layernorm_is_rejected():
    mlp = _mlp(norm="ln").eval()
    with torch.no_grad():
        assert _match(mlp) is None


@pytest.mark.parametrize("width", [126, 1028])
def test_unsupported_width_is_rejected(width):
    mlp = _mlp(width=width).eval()
    with torch.no_grad():
        assert _match(mlp) is None


def test_gradients_enabled_keep_the_module_path():
    mlp = _mlp().eval()
    assert torch.is_grad_enabled()
    assert _match(mlp) is None


def test_training_dropout_is_rejected():
    mlp = _mlp(dp=0.2).eval()
    mlp.lins[2].train()
    with torch.no_grad():
        assert _match(mlp) is None
