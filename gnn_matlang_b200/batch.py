"""Batching of per-graph records into one disjoint-union batch -- the semantics of PyG's
``Batch.from_data_list`` for the attributes GNNML3 reads (``DataLoader`` at graph8c.py:18, Zinc12k.py:20-22,
exp_classify.py:19-21, counting.py:29-31).  Integer work, bit-exact with the reference:

* ``x``, ``edge_attr2``, ``y`` are concatenated along dim 0;
* ``edge_index2`` (name contains "index") is concatenated along the last dim and shifted by the running
  node count, so the batched edge list stays sorted by (src, dst);
* ``batch[n]`` = index of the graph that owns node n; graphs stay contiguous and in input order.

In addition the batch carries ``graph_ptr`` (int32 node offsets) so that the readout and the CSR build never
have to rediscover the block structure.
"""
import numpy as np
import torch


class Batch(object):
    """Attribute bag with the reference's field names (``x``, ``edge_index2``, ``edge_attr2``, ``batch``, ``y``)."""

    def __init__(self, **kw):
        self.__dict__.update(kw)

    def to(self, device, non_blocking=True):
        out = Batch()
        for k, v in self.__dict__.items():
            out.__dict__[k] = v.to(device, non_blocking=non_blocking) if isinstance(v, torch.Tensor) else v
        if getattr(out, "batch", None) is not None and getattr(out, "graph_ptr", None) is not None and out.batch.is_cuda:
            out.batch._gnnml3_ptr = (out.batch._version, out.graph_ptr)
        return out

    def fresh(self):
        """New tensor objects over the same storage: drops the per-tensor caches (graph plan, sorted edge
        features), i.e. what a training loop sees when every step brings a new batch."""
        out = Batch()
        for k, v in self.__dict__.items():
            out.__dict__[k] = v.detach() if isinstance(v, torch.Tensor) else v
        if getattr(out, "batch", None) is not None and getattr(out, "graph_ptr", None) is not None and out.batch.is_cuda:
            out.batch._gnnml3_ptr = (out.batch._version, out.graph_ptr)
        return out

    def pin_memory(self):
        out = Batch()
        for k, v in self.__dict__.items():
            out.__dict__[k] = v.pin_memory() if isinstance(v, torch.Tensor) else v
        return out

    def nbytes(self):
        return sum(v.numel() * v.element_size() for v in self.__dict__.values() if isinstance(v, torch.Tensor))


def collate(graphs, adjacency=False):
    """``graphs``: sequence of dicts / objects with ``x [n,f]``, ``edge_index2 [2,e]``, ``edge_attr2 [e,K]``
    and optionally ``y``.  Returns a host ``Batch``.  ``adjacency=True``: the records also carry the graph's plain
    ``edge_index [2, m]`` (what GNNML1 reads), concatenated and shifted by the running node count like ``edge_index2``; records
    without ``edge_index2`` (GNNML1 needs no SpectralDesign supports) then give a batch without ``edge_index2`` / ``edge_attr2``."""
    def get(g, k):
        return g.get(k) if isinstance(g, dict) else getattr(g, k, None)

    ns = np.array([int(get(g, "x").shape[0]) for g in graphs], dtype=np.int64)
    off = np.zeros(len(graphs) + 1, dtype=np.int64)
    np.cumsum(ns, out=off[1:])
    x = torch.cat([torch.as_tensor(get(g, "x"), dtype=torch.float32) for g in graphs], 0)
    kw = dict(x=x)
    if not adjacency or all(get(g, "edge_index2") is not None for g in graphs):
        kw["edge_index2"] = torch.cat([torch.as_tensor(get(g, "edge_index2"), dtype=torch.int64) + int(o) for g, o in zip(graphs, off[:-1])], 1)
        kw["edge_attr2"] = torch.cat([torch.as_tensor(get(g, "edge_attr2"), dtype=torch.float32) for g in graphs], 0)
    batch = torch.from_numpy(np.repeat(np.arange(len(graphs), dtype=np.int64), ns))
    kw.update(batch=batch, num_graphs=len(graphs), graph_ptr=torch.from_numpy(off.astype(np.int32)))
    out = Batch(**kw)
    ys = [get(g, "y") for g in graphs]
    if all(y is not None for y in ys) and len(ys) > 0:
        ys = [torch.as_tensor(y) for y in ys]
        out.y = torch.cat([y.reshape(1, -1) if y.dim() < 2 else y for y in ys], 0)
    if adjacency:
        out.edge_index = torch.cat([torch.as_tensor(get(g, "edge_index"), dtype=torch.int64).reshape(2, -1) + int(o)
                                    for g, o in zip(graphs, off[:-1])], 1)
    return out


class CompactBatch(object):
    """Wire format of a batch for the host -> device link (the reference ships every attribute of the PyG batch as it sits in
    host memory: int64 ``edge_index2``, int64 ``batch``, FP32 one-hot ``x`` -- Zinc12k.py:360 ``data.to(device)``):

    * ``n [B]``, ``e [B]`` int32      nodes / support entries per graph (instead of ``batch [N]`` int64)
    * ``el [2, E]`` uint8 / int16     edge_index2 with node ids LOCAL to their graph (instead of int64 global ids)
    * ``xc [N, C]`` uint8 + ``widths``  class codes of a concatenation of one-hot blocks (ZINC: atom type | degree code),
                                       or ``x [N, F]`` float32 when the features are not one-hot
    * ``ea [E, K]`` float32, ``y``    unchanged

    ``expand(device)`` rebuilds the reference's batch attributes ON THE DEVICE, bit-exact (integer work) -- tested against
    ``collate``.  For the ZINC-shaped bench batches this is 36 bytes per support entry + 2 per node instead of 48 + 108."""

    def __init__(self, **kw):
        self.__dict__.update(kw)

    @staticmethod
    def from_batch(b, onehot_widths=None):
        """Host ``Batch`` -> ``CompactBatch`` (numpy work on the host; exact)."""
        gp = b.graph_ptr.numpy().astype(np.int64)
        n = np.diff(gp)
        ei = b.edge_index2.numpy()
        eg = np.searchsorted(gp, ei[0], side="right") - 1            # graph of every entry (by its source node)
        e = np.bincount(eg, minlength=len(n))
        loc = ei - gp[eg][None, :]
        if not (np.all(loc >= 0) and np.all(loc[1] < n[eg])):
            raise ValueError("edge_index2 crosses graph boundaries")
        if len(eg) and np.any(np.diff(eg) < 0):
            raise ValueError("edge_index2 is not grouped by graph")
        dt = np.uint8 if (n.max() if len(n) else 0) <= 256 else np.int16 if n.max() <= 32768 else np.int32
        kw = dict(n=torch.from_numpy(n.astype(np.int32)), e=torch.from_numpy(e.astype(np.int32)), el=torch.from_numpy(np.ascontiguousarray(loc.astype(dt))),
                  ea=b.edge_attr2, y=getattr(b, "y", None), num_graphs=len(n), widths=None, x=None, xc=None)
        x = b.x.numpy()
        if onehot_widths is not None:
            codes, off = [], 0
            for w in onehot_widths:
                blk = x[:, off:off + w]
                if not (np.all((blk == 0) | (blk == 1)) and np.all(blk.sum(1) == 1)):
                    raise ValueError("x is not a concatenation of one-hot blocks of widths %s" % (onehot_widths,))
                codes.append(blk.argmax(1).astype(np.uint8))
                off += w
            kw["xc"], kw["widths"] = torch.from_numpy(np.stack(codes, 1)), tuple(int(w) for w in onehot_widths)
        else:
            kw["x"] = b.x
        return CompactBatch(**kw)

    def _tensors(self):
        return {k: v for k, v in self.__dict__.items() if isinstance(v, torch.Tensor)}

    def pin_memory(self):
        out = CompactBatch(**self.__dict__)
        for k, v in self._tensors().items():
            out.__dict__[k] = v.pin_memory()
        return out

    def nbytes(self):
        return sum(v.numel() * v.element_size() for v in self._tensors().values())

    def to(self, device, non_blocking=True):
        out = CompactBatch(**self.__dict__)
        for k, v in self._tensors().items():
            out.__dict__[k] = v.to(device, non_blocking=non_blocking)
        return out

    def _out(self, Np, Ep, padded):
        dev = self.n.device
        F = sum(self.widths) if self.xc is not None else self.x.size(1)
        B = self.num_graphs
        return Batch(x=torch.empty(Np, F, dtype=torch.float32, device=dev), edge_index2=torch.empty(2, Ep, dtype=torch.int64, device=dev),
                     edge_attr2=torch.empty(Ep, self.ea.size(1), dtype=torch.float32, device=dev),
                     batch=torch.empty(Np, dtype=torch.int64, device=dev),
                     graph_ptr=torch.empty(B + (2 if padded else 1), dtype=torch.int32, device=dev), num_graphs=B)

    def expand_into(self, out):
        """Device ``CompactBatch`` -> the preallocated device ``Batch`` ``out`` (its tensors may be larger than the batch: the rest
        receives the neutral padding of ``train.pad_batch``).  Two library launches (``gnnml3_collate``), no host sync; integer
        work, bit-exact with host ``collate``."""
        from . import ops
        ops.collate_device(self.n, self.e, self.el, self.ea, self.num_graphs, out, xc=self.xc, widths=self.widths, x=self.x)
        if self.y is not None and getattr(out, "y", None) is not None and out.y is not self.y:
            out.y.copy_(self.y.reshape(out.y.shape), non_blocking=True)
        return out

    def expand(self):
        """Device ``CompactBatch`` -> device ``Batch`` with the reference's attributes (``x``, ``edge_index2`` int64 global ids,
        ``edge_attr2``, ``batch`` int64, ``y``) + ``graph_ptr``; integer work, bit-exact with host ``collate``."""
        N, E = (self.xc if self.xc is not None else self.x).size(0), self.el.size(1)
        out = self._out(N, E, False)
        if self.y is not None:
            out.y = self.y
        self.expand_into(out)
        out.batch._gnnml3_ptr = (out.batch._version, out.graph_ptr)
        return out
