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


def _local_ids(ei, gp, n, name):
    """Global [2, E] edge ids of a collated batch -> (edges per graph, graph-local ids in the smallest integer dtype that holds
    the largest graph's ids).  The edges must stay inside their graph and be grouped by graph in batch order."""
    eg = np.searchsorted(gp, ei[0], side="right") - 1            # graph of every edge (by its source node)
    cnt = np.bincount(eg, minlength=len(n))
    loc = ei - gp[eg][None, :]
    if not (np.all(loc >= 0) and np.all(loc[1] < n[eg])):
        raise ValueError("%s crosses graph boundaries" % name)
    if len(eg) and np.any(np.diff(eg) < 0):
        raise ValueError("%s is not grouped by graph" % name)
    dt = np.uint8 if (n.max() if len(n) else 0) <= 256 else np.int16 if n.max() <= 32768 else np.int32
    return cnt, np.ascontiguousarray(loc.astype(dt))


class CompactBatch(object):
    """Wire format of a batch for the host -> device link (the reference ships every attribute of the PyG batch as it sits in
    host memory: int64 ``edge_index2``, int64 ``batch``, FP32 one-hot ``x`` -- Zinc12k.py:360 ``data.to(device)``):

    * ``n [B]``, ``e [B]`` int32      nodes / support entries per graph (instead of ``batch [N]`` int64)
    * ``el [2, E]`` uint8 / int16     edge_index2 with node ids LOCAL to their graph (instead of int64 global ids)
    * ``xc [N, C]`` uint8 + ``widths``  class codes of a concatenation of one-hot blocks (ZINC: atom type | degree code),
                                       or ``x [N, F]`` float32 when the features are not one-hot
    * ``ea [E, K]`` float32, ``y``    unchanged
    * ``m [B]`` int32, ``al [2, M]``  for batches of ``collate(..., adjacency=True)``: plain edges per graph and the plain
                                       ``edge_index`` (what GNNML1 reads) with graph-local ids, like ``e`` / ``el``

    A batch without supports (GNNML1 records) has ``e`` / ``el`` / ``ea`` = None; one without the plain list has ``m`` / ``al``
    = None.  ``expand(device)`` rebuilds the reference's batch attributes ON THE DEVICE, bit-exact (integer work) -- tested
    against ``collate``.  For the ZINC-shaped bench batches this is 36 bytes per support entry + 2 per node instead of 48 + 108,
    and 2 bytes per plain edge instead of 16."""

    def __init__(self, **kw):
        self.__dict__.update(kw)

    @staticmethod
    def from_batch(b, onehot_widths=None):
        """Host ``Batch`` -> ``CompactBatch`` (numpy work on the host; exact)."""
        gp = b.graph_ptr.numpy().astype(np.int64)
        n = np.diff(gp)
        kw = dict(n=torch.from_numpy(n.astype(np.int32)), e=None, el=None, ea=None, m=None, al=None, y=getattr(b, "y", None),
                  num_graphs=len(n), widths=None, x=None, xc=None)
        if getattr(b, "edge_index2", None) is not None:
            e, el = _local_ids(b.edge_index2.numpy(), gp, n, "edge_index2")
            kw.update(e=torch.from_numpy(e.astype(np.int32)), el=torch.from_numpy(el), ea=b.edge_attr2)
        if getattr(b, "edge_index", None) is not None:
            m, al = _local_ids(b.edge_index.numpy(), gp, n, "edge_index")
            kw.update(m=torch.from_numpy(m.astype(np.int32)), al=torch.from_numpy(al))
        if kw["el"] is None and kw["al"] is None:
            raise ValueError("the batch has neither edge_index2 nor edge_index")
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

    def sizes(self):
        """(nodes, support entries, plain edges) of the batch; None for a list it does not carry."""
        return ((self.xc if self.xc is not None else self.x).size(0), None if self.el is None else self.el.size(1),
                None if getattr(self, "al", None) is None else self.al.size(1))

    def _out(self, Np, Ep, padded, Mp=None):
        dev = self.n.device
        F = sum(self.widths) if self.xc is not None else self.x.size(1)
        B = self.num_graphs
        out = Batch(x=torch.empty(Np, F, dtype=torch.float32, device=dev))
        if self.el is not None:
            out.edge_index2 = torch.empty(2, Ep, dtype=torch.int64, device=dev)
            out.edge_attr2 = torch.empty(Ep, self.ea.size(1), dtype=torch.float32, device=dev)
        out.batch = torch.empty(Np, dtype=torch.int64, device=dev)
        out.graph_ptr = torch.empty(B + (2 if padded else 1), dtype=torch.int32, device=dev)
        out.num_graphs = B
        if Mp is not None:
            out.edge_index = torch.empty(2, Mp, dtype=torch.int64, device=dev)
        return out

    def expand_into(self, out):
        """Device ``CompactBatch`` -> the preallocated device ``Batch`` ``out`` (its tensors may be larger than the batch: the rest
        receives the neutral padding of ``train.pad_batch``).  Two library launches (``gnnml3_collate``, or
        ``gnnml3_collate_graphs`` with the plain list), no host sync; integer work, bit-exact with host ``collate``.  ``out.edge_index``
        is filled when both carry the plain list."""
        from . import ops
        al = getattr(self, "al", None)
        if al is not None and getattr(out, "edge_index", None) is not None:
            N, _, M = self.sizes()
            if out.edge_index.size(1) > M and out.x.size(0) <= N:
                raise ValueError("expand_into: padding edge_index (%d > %d edges) needs dummy nodes (out.x has %d rows for %d nodes)"
                                 % (out.edge_index.size(1), M, out.x.size(0), N))
            ops.collate_device(self.n, self.e, self.el, self.ea, self.num_graphs, out, xc=self.xc, widths=self.widths, x=self.x,
                               m=self.m, al=al)
        else:
            ops.collate_device(self.n, self.e, self.el, self.ea, self.num_graphs, out, xc=self.xc, widths=self.widths, x=self.x)
        if self.y is not None and getattr(out, "y", None) is not None and out.y is not self.y:
            out.y.copy_(self.y.reshape(out.y.shape), non_blocking=True)
        return out

    def expand(self):
        """Device ``CompactBatch`` -> device ``Batch`` with the reference's attributes (``x``, ``edge_index2`` int64 global ids,
        ``edge_attr2``, ``edge_index`` when the batch carries the plain list, ``batch`` int64, ``y``) + ``graph_ptr``; integer work,
        bit-exact with host ``collate``."""
        N, E, M = self.sizes()
        out = self._out(N, E, False, M)
        if self.y is not None:
            out.y = self.y
        self.expand_into(out)
        out.batch._gnnml3_ptr = (out.batch._version, out.graph_ptr)
        return out
