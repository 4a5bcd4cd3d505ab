"""The paper's isomorphism test (Table 1): how many graph pairs a model cannot tell apart.

The reference runs it in three scripts -- ``graph8c.py:281-302`` (11,117 graphs, 100 seeds), ``sr25.py`` (15 strongly regular
graphs, 105 pairs) and ``exp_iso.py`` (600 listed pairs, ``E[0::2]`` against ``E[1::2]``).  Every seed is a freshly initialised
model under ``torch.manual_seed(seed)``; a pair counts as distinguished once the L1 distance of its two embeddings exceeds
the threshold (1e-3) under any seed so far.

    tracker = PairTracker(n, device)                # the cross-seed state: one bit per pair, on the device
    tracker.update(emb)                             # OR one seed's embeddings [n, d] in
    tracker.count()                                 # device int64 scalar: pairs not distinguished so far

    res = isomorphism_test(lambda: GNNML3("graph8c", ne=6, ninp=2), dataset, seeds=range(100))
    res["counts"]                                   # undistinguished pairs after each seed

Distances are FP32 sums over the embedding dimension in a fixed order (``gnnml3_pairs_mark``), so the counts are
deterministic.  A pair whose distance is NaN is not distinguished, as with the reference's ``cdist > thr``.  Single GPU: sharding
the seeds over ranks would need a bitwise-OR all-reduce of the bitmap, which NCCL does not offer.
"""
import math
import numbers

import numpy as np
import torch

from . import ops


def _check_threshold(threshold):
    if isinstance(threshold, bool) or not isinstance(threshold, numbers.Real) or not math.isfinite(threshold) or threshold < 0:
        raise ValueError("threshold must be a finite number >= 0, got %r" % (threshold,))
    return float(threshold)


def _check_n(n):
    if isinstance(n, bool) or not isinstance(n, numbers.Integral) or n < 0:
        raise ValueError("n must be an integer >= 0, got %r" % (n,))
    return int(n)


def _check_device(device):
    device = torch.device(device)
    if device.type != "cuda":
        raise ValueError("the isomorphism test runs on a CUDA device, got %s (there is no CPU path)" % device)
    return device


def _check_pairs(pairs, n):
    """Host array or CUDA tensor [P, 2] of row ids in [0, n), P >= 1 -> (host int64 array or None, CUDA tensor or None).  The
    range check of a CUDA tensor reads one flag back from the device."""
    if isinstance(pairs, torch.Tensor) and pairs.is_cuda:
        if pairs.dim() != 2 or pairs.size(1) != 2 or pairs.size(0) == 0:
            raise ValueError("pairs must have shape [P, 2] with P >= 1, got %s" % (tuple(pairs.shape),))
        if pairs.dtype.is_floating_point or pairs.dtype.is_complex or pairs.dtype == torch.bool:
            raise ValueError("pairs must hold integer ids, got %s" % pairs.dtype)
        if bool(((pairs < 0) | (pairs >= n)).any()):
            raise ValueError("pairs hold ids outside [0, %d)" % n)
        return None, pairs
    arr = np.asarray(pairs.numpy() if isinstance(pairs, torch.Tensor) else pairs)
    if arr.ndim != 2 or arr.shape[1] != 2 or arr.shape[0] == 0:
        raise ValueError("pairs must have shape [P, 2] with P >= 1, got %s" % (arr.shape,))
    if not np.issubdtype(arr.dtype, np.integer):
        raise ValueError("pairs must hold integer ids, got %s" % arr.dtype)
    if arr.min() < 0 or arr.max() >= n:
        raise ValueError("pairs hold ids outside [0, %d)" % n)
    return arr.astype(np.int64), None


class PairTracker(object):
    """Which pairs of ``n`` embeddings have been distinguished so far: a zeroed device bitmap, one bit per pair.

    ``pairs=None`` tracks every pair i < j (n (n - 1) / 2 bits in ``n`` rows of ``wpr`` words); ``pairs`` [P, 2] (host array or
    CUDA tensor of row ids, range-checked here, once) tracks the listed pairs only.  ``update(emb)`` marks the pairs whose L1
    distance exceeds ``threshold``; ``count()`` returns the pairs not yet marked as a device int64 scalar; ``reset()`` clears
    the bitmap.  ``update`` and ``count`` launch one kernel each and never synchronise, so they can be captured in a CUDA graph."""

    def __init__(self, n, device, threshold=1e-3, pairs=None):
        self.n = _check_n(n)
        self.threshold = _check_threshold(threshold)
        self.device = _check_device(device)
        host, dev_pairs = (None, None) if pairs is None else _check_pairs(pairs, self.n)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        if pairs is None:
            self.P = 0
            self.wpr = (self.n + 127) // 128 * 4                   # whole 128-bit rows: the count kernel reads 16 bytes at a time
            self.pairs = None
            self.bits = torch.zeros(self.n, self.wpr, dtype=torch.int32, device=self.device)
        else:
            self.P = int(host.shape[0] if host is not None else dev_pairs.size(0))
            self.wpr = 0
            self.pairs = (torch.from_numpy(host) if host is not None else dev_pairs).to(self.device, torch.int64).contiguous()
            self.bits = torch.zeros((self.P + 31) // 32, dtype=torch.int32, device=self.device)

    def update(self, emb):
        """OR the pairs that the embeddings ``emb`` [n, d] (float32 on the tracker's device; row-strided views are fine)
        distinguish into the bitmap."""
        if not isinstance(emb, torch.Tensor):
            raise TypeError("emb must be a tensor")
        if emb.dim() != 2 or emb.size(0) != self.n or emb.size(1) < 1:
            raise ValueError("emb must have shape [%d, d >= 1], got %s" % (self.n, tuple(emb.shape)))
        if emb.dtype != torch.float32:
            raise ValueError("emb must be float32, got %s" % emb.dtype)
        if not emb.is_cuda or emb.device != self.device:
            raise ValueError("emb must be on %s, got %s (there is no CPU path)" % (self.device, emb.device))
        ops.pairs_mark(emb, self.bits, self.wpr, self.threshold, self.pairs)

    def count(self, out=None):
        """Pairs not distinguished so far -> device int64 scalar (written into ``out`` when given)."""
        if out is None:
            out = torch.empty((), dtype=torch.int64, device=self.device)
        elif out.dtype != torch.int64 or out.numel() != 1 or out.device != self.device:
            raise ValueError("out must be a one-element int64 tensor on %s" % self.device)
        return ops.pairs_count(self.bits, self.n, self.wpr, self.P, out)

    def reset(self):
        self.bits.zero_()


def isomorphism_test(make_model, dataset, seeds=range(100), batch_size=100, threshold=1e-3, pairs=None, ids=None,
                     return_embeddings=False):
    """The reference's multi-seed protocol over the graphs ``ids`` (default: all) of a resident ``synthetic.DeviceDataset``.

    For each seed: ``torch.manual_seed(seed)``, then ``make_model()`` builds a fresh model on the CPU (the reference's RNG
    order).  The first model is moved to the dataset's device and captured once in a ``train.GraphedEvaluator`` (``metric=None``,
    ``batch_size`` graphs per batch); every later model's ``state_dict`` is loaded in place into the captured one and the graph is
    replayed.  The embeddings of each seed are OR-ed into a ``PairTracker`` (all pairs, or the listed ``pairs`` [P, 2] of
    positions in ``ids``) and its count is stored on the device; the counts are read once, at the end.

    -> {"graphs": len(ids), "pairs": pairs tracked, "counts": [undistinguished pairs after each seed]} (+ "embeddings": the
    [len(ids), d] device tensor of every seed with ``return_embeddings=True``)."""
    from .train import GraphedEvaluator
    if not callable(make_model):
        raise TypeError("make_model must be a callable that returns a fresh model")
    seeds = [int(s) for s in seeds]
    if not seeds:
        raise ValueError("seeds is empty")
    if isinstance(batch_size, bool) or not isinstance(batch_size, numbers.Integral) or batch_size < 1:
        raise ValueError("batch_size must be a positive integer, got %r" % (batch_size,))
    threshold = _check_threshold(threshold)
    G = len(dataset.n_h)
    ids = np.arange(G, dtype=np.int64) if ids is None else np.asarray(ids).reshape(-1)
    if len(ids) == 0:
        raise ValueError("ids is empty")
    if not np.issubdtype(ids.dtype, np.integer) or ids.min() < 0 or ids.max() >= G:
        raise ValueError("ids must be integer graph ids in [0, %d)" % G)
    device = _check_device(dataset.x.device)

    tracker = PairTracker(len(ids), device, threshold, pairs)
    counts = torch.zeros(len(seeds), dtype=torch.int64, device=device)
    model, ev, embeddings = None, None, []
    for s, seed in enumerate(seeds):
        torch.manual_seed(seed)
        fresh = make_model()
        if ev is None:
            model = fresh.to(device)
            ev = GraphedEvaluator(model, dataset, ids, batch_size, metric=None)
        else:
            model.load_state_dict(fresh.state_dict())
        emb = ev.run(outputs=True)["outputs"]
        tracker.update(emb)
        tracker.count(out=counts[s])
        if return_embeddings:
            embeddings.append(emb)
    res = {"graphs": len(ids), "pairs": tracker.P if tracker.pairs is not None else len(ids) * (len(ids) - 1) // 2,
           "counts": counts.tolist()}
    if return_embeddings:
        res["embeddings"] = embeddings
    return res
