"""Node BatchNorm of a padded batch: ``nn.BatchNorm1d`` in training mode over the real nodes only.

A captured training step pads every batch with one dummy graph (``train.pad_batch``); a BatchNorm over all node rows would
mix the dummy nodes into the batch statistics and train a different model than the eager step on the same graphs.
``batch_norm_rows`` normalises with the statistics of the first ``cnt`` rows, ``cnt`` read on the device
(``graph_ptr[real_graphs]``), through the two-launch kernels of ``gnnml3_bn_rows_fwd`` / ``_bwd``: no host sync, capturable.
The module's own parameters and running buffers are used and updated as ``nn.BatchNorm1d`` would on ``x[:cnt]``.

Under data parallelism every rank normalises with the statistics of its own shard, as DDP does without SyncBatchNorm."""
import torch

from . import ops


class _BNRowsFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, cnt, bn):
        y, mean, invstd = ops.bn_rows_fwd(x, cnt, weight, bias, bn.running_mean, bn.running_var, bn.num_batches_tracked, bn.eps,
                                          bn.momentum)
        ctx.save_for_backward(x, weight, mean, invstd)
        ctx.cnt = cnt
        return y

    @staticmethod
    def backward(ctx, gy):
        x, weight, mean, invstd = ctx.saved_tensors
        dx, dw, db = ops.bn_rows_bwd(x, gy, ctx.cnt, weight, mean, invstd)
        return dx, dw, db, None, None


def check_bn_module(bn):
    """The configuration of the presets' node BatchNorm (mutag.py:283-285) is the one this path implements: ValueError otherwise."""
    if not isinstance(bn, torch.nn.BatchNorm1d):
        raise ValueError("batch_norm_rows: expected an nn.BatchNorm1d, got %s" % type(bn).__name__)
    if not bn.affine or not bn.track_running_stats:
        raise ValueError("batch_norm_rows: needs affine=True and track_running_stats=True")
    if not isinstance(bn.momentum, float):
        raise ValueError("batch_norm_rows: needs a float momentum (got %r; None is the cumulative average)" % (bn.momentum,))


def batch_norm_rows(x, cnt, bn):
    """``bn(x[:cnt])`` in training mode for the first ``cnt`` rows of x [N, F] and the same affine map on the rest; ``cnt`` is a
    one-element int32 CUDA tensor.  Gradients reach x (zero on rows >= cnt) and ``bn``'s weight and bias."""
    check_bn_module(bn)
    return _BNRowsFn.apply(x, bn.weight, bn.bias, cnt, bn)
