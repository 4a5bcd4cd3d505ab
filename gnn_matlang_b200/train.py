"""Training step of the reference's scripts (Zinc12k.py:354-371, counting.py:400-417, exp_classify.py:318-337):
forward, SUM-reduced loss, backward, Adam(lr=1e-3) -- with data parallelism over the graph-minibatch axis.

Graphs never interact (block-diagonal supports, per-graph readout), so a global minibatch is sharded over the
ranks as whole graphs and the only exchange is ONE SUM all-reduce of the flat gradient buffer per step (SUM,
not mean: every loss of the reference uses reduction='sum', so the single-process result for the same global
batch is reproduced).  Parameters and Adam state are replicated.
"""
import torch
import torch.distributed as dist
import torch.nn.functional as F


def loss_fn(kind, out, y):
    if kind == "l1":                                   # Zinc12k.py:365
        return F.l1_loss(out, y.to(out.dtype).reshape(out.shape), reduction="sum")
    if kind == "mse":                                  # counting.py:411
        return torch.square(out - y.to(out.dtype).reshape(out.shape)).sum()
    if kind == "bce":                                  # exp_classify.py:327-329
        return F.binary_cross_entropy(torch.sigmoid(out), y.to(out.dtype).reshape(out.shape), reduction="sum")
    raise ValueError(kind)


def shard_graphs(sizes, world, rank=None):
    """Contiguous split of a global minibatch over ``world`` ranks balanced by the graphs' sizes (nodes or support entries) and
    not by their count (SURVEY.md 8e: 30-100-node mixes): the cut points are the positions where the running sum of ``sizes``
    crosses k / world of the total.  Returns the list of (begin, end) graph ranges, or rank's range.  Pure host arithmetic."""
    import numpy as np
    s = np.asarray(sizes, dtype=np.float64)
    c = np.concatenate([[0.0], np.cumsum(s)])
    cuts = [0]
    for k in range(1, world):
        target = c[-1] * k / world
        j = int(np.searchsorted(c, target, side="left"))
        if j > 0 and abs(c[j - 1] - target) <= abs(c[min(j, len(c) - 1)] - target):
            j -= 1
        cuts.append(min(max(j, cuts[-1]), len(s)))
    cuts.append(len(s))
    ranges = [(cuts[k], cuts[k + 1]) for k in range(world)]
    return ranges if rank is None else ranges[rank]


class Trainer(object):
    def __init__(self, model, loss="l1", lr=1e-3, distributed=False):
        self.model = model
        self.loss_kind = loss
        self.distributed = distributed and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        self.params = [p for p in model.parameters()]
        fused = self.params[0].is_cuda
        self.opt = torch.optim.Adam(self.params, lr=lr, fused=fused) if fused else torch.optim.Adam(self.params, lr=lr)

    def step(self, batch):
        """One optimisation step on a device-resident batch; returns the (device) loss tensor.

        Gradients start as None, so autograd hands every parameter its freshly computed gradient tensor instead of
        accumulating into a zeroed buffer (44 tiny add kernels per step for the ZINC model).  With more than one rank the
        gradients are flattened into ONE bucket, SUM-all-reduced (all losses use reduction='sum', Zinc12k.py:365) and the
        parameters' .grad become views of the reduced bucket."""
        for p in self.params:
            p.grad = None
        out = self.model(batch)
        loss = loss_fn(self.loss_kind, out, batch.y)
        loss.backward()
        if self.distributed:
            grads = [p.grad if p.grad is not None else torch.zeros_like(p) for p in self.params]
            flat = torch.cat([g.reshape(-1) for g in grads])
            dist.all_reduce(flat, op=dist.ReduceOp.SUM)
            off = 0
            for p in self.params:
                p.grad = flat[off:off + p.numel()].view_as(p)
                off += p.numel()
        self.opt.step()
        return loss.detach()


class HostFeeder(object):
    """Streams pinned host batches to the device one step ahead of the compute stream (H2D overlaps compute).

    Host ``Batch`` objects are converted ONCE (first time they are seen) to the compact wire format (``batch.CompactBatch``:
    int32 per-graph sizes instead of the int64 batch vector, graph-local uint8 edge ids instead of int64 global ids, one-hot
    ``x`` as uint8 class codes); every step copies the compact tensors host -> device on the copy stream and the reference's
    attributes are rebuilt on the device (``expand``) on the compute stream."""

    format_note = ("compact wire format: n/e int32 per graph, graph-local uint8 edge ids, one-hot x as uint8 class codes, FP32 "
                   "supports; edge_index2 (int64, global), batch and x are rebuilt on the device")

    def __init__(self, device, onehot_widths=None):
        self.device = device
        self.copy_stream = torch.cuda.Stream(device=device)
        self.onehot_widths = onehot_widths
        self._next = None
        self._compact = {}

    def compact(self, host_batch):
        from .batch import CompactBatch
        key = id(host_batch)
        cb = self._compact.get(key)
        if cb is None:
            if isinstance(host_batch, CompactBatch):
                cb = host_batch
            else:
                cb = CompactBatch.from_batch(host_batch, self.onehot_widths).pin_memory()
            self._compact[key] = cb
        return cb

    def bytes_per_batch(self, host_batch):
        return self.compact(host_batch).nbytes()

    def prefetch(self, host_batch):
        cb = self.compact(host_batch)
        with torch.cuda.stream(self.copy_stream):
            b = cb.to(self.device, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(self.copy_stream)
        self._next = (b, ev)

    def get_compact(self):
        """The prefetched batch, still in the wire format, on the device (ordered behind its copy on the current stream)."""
        b, ev = self._next
        torch.cuda.current_stream().wait_event(ev)
        for v in b._tensors().values():
            v.record_stream(torch.cuda.current_stream())
        self._next = None
        return b

    def get(self):
        return self.get_compact().expand()


class DesignFeeder(object):
    """BASELINE.json configs[2] (exp_classify.py with the supports rebuilt on the GPU for every batch): designs the NEXT raw
    batches (``synthetic.design_and_collate``: SpectralDesign of all graphs of a batch in one launch + collation) on side streams
    while the current batch trains on the main stream.  At the reference's batch size (50 graphs) the one-block-per-graph Jacobi
    is latency-bound (1.8 ms for 50 blocks on 148 SMs) and independent of the training step: ``depth`` designs in flight on
    ``depth`` streams overlap with each other and with the step.  The raw tensors handed to ``prefetch`` must already be valid
    on the device (the side streams do not wait for the main stream)."""

    def __init__(self, sd, device, depth=2):
        self.sd, self.device = sd, device
        self.streams = [torch.cuda.Stream(device=device) for _ in range(depth)]
        self._queue = []
        self._k = 0

    def prefetch(self, raw, records=False):
        """``records=False``: a collated device ``Batch`` (``design_and_collate``); ``records=True``: the per-graph records of
        ``synthetic.design_raw`` for ``GraphedTrainer.load_designed`` (collation + padding straight into the captured buffers)."""
        from .synthetic import design_and_collate, design_raw
        st = self.streams[self._k % len(self.streams)]
        self._k += 1
        with torch.cuda.stream(st):
            b = design_raw(raw, self.sd, self.device) if records else design_and_collate(raw, self.sd, self.device)
        ev = torch.cuda.Event()
        ev.record(st)
        self._queue.append((b, ev))

    def pending(self):
        return len(self._queue)

    def get(self):
        b, ev = self._queue.pop(0)
        cur = torch.cuda.current_stream(self.device)
        cur.wait_event(ev)
        vals = list(b.values()) + list(b["design"].values()) if isinstance(b, dict) else list(b.__dict__.values())
        for v in vals:
            if isinstance(v, torch.Tensor) and v.is_cuda:
                v.record_stream(cur)
        return b


def _pad_loops(N, n_nodes, first, total):
    """[2, total - first] self-loops spread round-robin over the dummy nodes N .. n_nodes - 1."""
    return (N + torch.arange(total - first) % (n_nodes - N)).unsqueeze(0).expand(2, -1)


def pad_batch(hb, n_nodes, n_entries=None, n_edges=None):
    """Host ``Batch`` -> the same batch padded to ``n_nodes`` nodes and ``n_entries`` support entries (static shapes for CUDA
    graph replay).  The padding is exactly neutral: the extra nodes are isolated, carry zero features and form ONE extra
    (dummy) graph at the end whose read-out row the loss never sees (``GraphedTrainer`` slices it off); the extra entries are
    self-loops spread round-robin over the dummy nodes with all-zero supports (a bias-free edge MLP maps them to zero, they
    add 0 to those nodes and receive zero gradients).  ``n_nodes`` must exceed the batch's node count (the dummy graph is
    never empty); ``padded_shapes`` picks shapes that keep the dummy nodes' degree small (a hub row would serialise the
    row-parallel kernels).

    ``n_edges``: the batch's plain ``edge_index`` (``collate(..., adjacency=True)``, what GNNML1 reads) is padded to
    ``n_edges`` columns with the same round-robin self-loops on the dummy nodes; a batch without supports passes
    ``n_entries=None``.  Without ``n_edges`` the result has no ``edge_index``.  GNNML1 has no edge weights, so these self-loops
    DO add a dummy node's features to itself -- still neutral for the real graphs and for training:

    * no edge joins a dummy node to a real one, so the dummy nodes form one extra graph whose activations never reach a real
      node's;
    * that graph's read-out row is sliced off before the loss (``out[:real]``), so the gradient of every dummy row is exactly
      zero at every layer, and so is the dummy rows' contribution to the weight and bias gradients;
    * this holds while the dummy activations stay finite (0 * inf is NaN): the round-robin spread keeps each dummy node's
      self-loop count at most ``max_pad_degree`` of ``padded_shapes``, i.e. in the range of a real node's degree."""
    import numpy as np
    from .batch import Batch
    sup = getattr(hb, "edge_index2", None) is not None
    N = hb.x.size(0)
    E = hb.edge_index2.size(1) if sup else 0
    if sup and n_entries is None:
        raise ValueError("pad_batch: the batch has supports: give n_entries")
    if n_edges is not None and getattr(hb, "edge_index", None) is None:
        raise ValueError("pad_batch: n_edges given but the batch has no edge_index")
    M = hb.edge_index.size(1) if n_edges is not None else 0
    if n_nodes <= N or (sup and n_entries < E) or (n_edges is not None and n_edges < M):
        raise ValueError("pad_batch: need n_nodes > %d, n_entries >= %d and n_edges >= %d" % (N, E, M))
    B = hb.num_graphs
    x = torch.zeros(n_nodes, hb.x.size(1), dtype=hb.x.dtype)
    x[:N] = hb.x
    kw = dict(x=x)
    if sup:
        ei = torch.empty((2, n_entries), dtype=torch.int64)
        ei[:, :E] = hb.edge_index2
        ei[:, E:] = _pad_loops(N, n_nodes, E, n_entries)
        ea = torch.zeros(n_entries, hb.edge_attr2.size(1), dtype=hb.edge_attr2.dtype)
        ea[:E] = hb.edge_attr2
        kw.update(edge_index2=ei, edge_attr2=ea)
    batch = torch.full((n_nodes,), B, dtype=torch.int64)
    batch[:N] = hb.batch
    gp = torch.cat([hb.graph_ptr.to(torch.int32), torch.tensor([n_nodes], dtype=torch.int32)])
    out = Batch(**kw, batch=batch, num_graphs=B + 1, graph_ptr=gp, y=hb.y, real_graphs=B)
    if n_edges is not None:
        adj = torch.empty((2, n_edges), dtype=torch.int64)
        adj[:, :M] = hb.edge_index
        adj[:, M:] = _pad_loops(N, n_nodes, M, n_edges)
        out.edge_index = adj
    return out


def padded_shapes(batches, max_pad_degree=8, adjacency=False):
    """(n_nodes, n_entries) for ``pad_batch`` / ``GraphedTrainer`` covering every batch of the list: the largest entry count,
    and enough dummy nodes that the padding self-loops of the SMALLEST batch give no dummy node more than ``max_pad_degree``.

    ``adjacency=True``: (n_nodes, n_entries, n_edges), sizing the plain ``edge_index`` as well (``n_entries`` is None for batches
    without supports); the dummy nodes then bound the self-loops a dummy node receives from BOTH lists together."""
    nodes = [int(b.x.shape[0]) for b in batches]
    if not adjacency:
        return padded_shapes_from_sizes(nodes, [int(b.edge_index2.shape[1]) for b in batches], max_pad_degree=max_pad_degree)
    sup = getattr(batches[0], "edge_index2", None) is not None
    return padded_shapes_from_sizes(nodes, [int(b.edge_index2.shape[1]) for b in batches] if sup else None,
                                    [int(b.edge_index.shape[1]) for b in batches], max_pad_degree=max_pad_degree)


def padded_shapes_from_sizes(nodes, entries=None, edges=None, max_pad_degree=8):
    """The rule of ``padded_shapes`` on per-batch totals (nodes, support entries, plain edges of every batch) instead of
    collated batches, so that shapes can be fixed from a dataset's size arrays alone.  ``edges=None``: (n_nodes, n_entries);
    otherwise (n_nodes, n_entries or None when ``entries`` is None, n_edges)."""
    nmax = max(int(n) for n in nodes)
    if edges is None:
        emax, emin = max(int(e) for e in entries), min(int(e) for e in entries)
        return nmax + 1 + (emax - emin + max_pad_degree - 1) // max_pad_degree, emax
    sup = entries is not None
    es = [int(e) for e in entries] if sup else [0]
    ms = [int(m) for m in edges]
    pe, pm = max(es) - min(es), max(ms) - min(ms)             # most padding either list can need (smallest batch)
    if pe and pm and max_pad_degree < 2:
        raise ValueError("padded_shapes: padding both lists needs max_pad_degree >= 2")
    # a dummy node gets ceil(pe / nd) + ceil(pm / nd) self-loops at most (both lists start the round-robin at node N)
    nd = max(1, -(-(pe + pm) // max_pad_degree))
    while -(-pe // nd) + -(-pm // nd) > max_pad_degree:
        nd += 1
    return nmax + nd, (max(es) if sup else None), max(ms)


class GraphedTrainer(object):
    """The whole optimisation step -- CSR build of the new batch, forward, SUM loss, backward, (all-reduce,) Adam -- captured
    ONCE into a CUDA graph and replayed per step (SURVEY.md 8f rank 2: the step's ~120 launches cost ~2 ms of host time to
    enqueue, more than the GPU needs at the reference's batch sizes).  Batches must have static shapes (``pad_batch``); a
    step copies the new batch into the captured input buffers (device -> device, or host -> device when given a pinned host
    batch) and replays.  Everything inside is capture-safe: the library never synchronises, workspaces are allocated during
    the warm-up steps, tensor-map descriptors are kernel parameters."""

    def __init__(self, model, example, loss="l1", lr=1e-3, distributed=False, warmup=3):
        from .graph import set_range_check
        set_range_check(False)                         # the range check reads a flag back from the device
        self.model, self.loss_kind = model, loss
        self.distributed = distributed and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        self.params = [p for p in model.parameters()]
        self.opt = torch.optim.Adam(self.params, lr=lr, fused=True, capturable=True)
        dev = self.params[0].device
        self.static = example.to(dev, non_blocking=False) if not example.x.is_cuda else example
        self.real = int(getattr(example, "real_graphs", example.num_graphs))
        # the inputs the example carries: a GNNML3 batch brings the supports, a GNNML1 batch the plain edge list
        self.fields = tuple(k for k in ("x", "edge_index2", "edge_attr2", "edge_index", "batch", "graph_ptr", "y")
                            if getattr(example, k, None) is not None)
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s):
            for _ in range(warmup):
                self._eager_step()
        torch.cuda.current_stream(dev).wait_stream(s)
        torch.cuda.synchronize(dev)
        # Single process: ONE graph holds the whole step.  Data parallel: the NCCL all-reduce stays outside the capture (a
        # captured collective ties the graph to the communicator's stream ordering and watchdog); the step is two graphs --
        # CSR build + forward + loss + backward + gradient flattening | Adam on views of the reduced bucket -- with the one
        # all-reduce launch between them.
        self.graph = torch.cuda.CUDAGraph()
        self.graph2 = None
        if not self.distributed:
            with torch.cuda.graph(self.graph):
                self.static_loss = self._eager_step()
        else:
            with torch.cuda.graph(self.graph):
                self.static_loss, self.flat = self._fwd_bwd_flat()
            self._grads_from(self.flat)
            self.graph2 = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph2, pool=self.graph.pool()):
                self.opt.step()

    def _grads_from(self, flat):
        off = 0
        for p in self.params:
            p.grad = flat[off:off + p.numel()].view_as(p)
            off += p.numel()

    def _fwd_bwd_flat(self):
        b = self.static.fresh()
        for p in self.params:
            p.grad = None
        out = self.model(b)
        loss = loss_fn(self.loss_kind, out[:self.real], b.y)
        loss.backward()
        grads = [p.grad if p.grad is not None else torch.zeros_like(p) for p in self.params]
        return loss.detach(), torch.cat([g.reshape(-1) for g in grads])

    def _eager_step(self):
        if self.distributed:
            loss, flat = self._fwd_bwd_flat()
            dist.all_reduce(flat, op=dist.ReduceOp.SUM)
            self._grads_from(flat)
            self.opt.step()
            return loss
        b = self.static.fresh()
        for p in self.params:
            p.grad = None
        out = self.model(b)
        loss = loss_fn(self.loss_kind, out[:self.real], b.y)
        loss.backward()
        self.opt.step()
        return loss.detach()

    def load(self, batch):
        """Copy a padded batch (device or pinned host, same shapes as the example) into the captured input buffers."""
        for k in self.fields:
            getattr(self.static, k).copy_(getattr(batch, k), non_blocking=True)

    def load_unpadded(self, b):
        """Write a DEVICE batch of any size that fits (N < captured nodes, E <= captured entries, M <= captured plain edges, same
        number of graphs) into the captured input buffers and fill the rest with the neutral padding of ``pad_batch``
        (device-side, no host sync)."""
        st = self.static
        sup, adj = "edge_index2" in self.fields, "edge_index" in self.fields
        N = b.x.size(0)
        E, M = (b.edge_index2.size(1) if sup else 0), (b.edge_index.size(1) if adj else 0)
        Np, Ep, Mp = st.x.size(0), (st.edge_index2.size(1) if sup else 0), (st.edge_index.size(1) if adj else 0)
        if N >= Np or E > Ep or M > Mp or b.num_graphs != self.real:
            raise ValueError("batch (%d nodes, %d entries, %d edges, %d graphs) does not fit the captured shapes (%d, %d, %d, %d)"
                             % (N, E, M, b.num_graphs, Np, Ep, Mp, self.real))
        st.x[:N].copy_(b.x, non_blocking=True)
        st.x[N:].zero_()
        if sup:
            st.edge_index2[:, :E].copy_(b.edge_index2, non_blocking=True)
            if Ep > E:
                st.edge_index2[:, E:].copy_((N + torch.arange(Ep - E, device=st.x.device) % (Np - N)).unsqueeze(0))
            st.edge_attr2[:E].copy_(b.edge_attr2, non_blocking=True)
            st.edge_attr2[E:].zero_()
        if adj:
            st.edge_index[:, :M].copy_(b.edge_index, non_blocking=True)
            if Mp > M:
                st.edge_index[:, M:].copy_((N + torch.arange(Mp - M, device=st.x.device) % (Np - N)).unsqueeze(0))
        st.batch[:N].copy_(b.batch, non_blocking=True)
        st.batch[N:].fill_(self.real)
        st.graph_ptr[:self.real + 1].copy_(b.graph_ptr, non_blocking=True)
        st.graph_ptr[self.real + 1:].fill_(Np)
        st.y.copy_(b.y, non_blocking=True)

    def load_compact(self, cb):
        """Device ``CompactBatch`` (wire format) -> the captured input buffers, padding included: two library launches
        (``gnnml3_collate``, or ``gnnml3_collate_graphs`` with the plain edge list) + the label copy, instead of ~20 index kernels
        of ``expand`` and ~12 copies of ``load_unpadded``."""
        st = self.static
        N, E, M = cb.sizes()
        sup, adj = "edge_index2" in self.fields, "edge_index" in self.fields
        if N >= st.x.size(0) or cb.num_graphs != self.real or (E is None) == sup or (M is None and adj) \
                or (sup and E > st.edge_index2.size(1)) or (adj and M > st.edge_index.size(1)):
            raise ValueError("batch does not fit the captured shapes")
        cb.expand_into(st)

    def load_designed(self, rec):
        """Per-graph records of a batch whose supports were just designed on the GPU (``synthetic.design_raw``) -> the captured
        input buffers: collation, global ids and the neutral padding in two library launches."""
        from . import ops
        d = rec["design"]
        if rec["num_graphs"] != self.real:
            raise ValueError("batch does not fit the captured shapes")
        ops.collate_device(rec["n32"], d["counts"], d["edge_index2"], d["edge_attr2"], rec["num_graphs"], self.static, x=rec["x"])
        self.static.y.copy_(rec["y"].reshape(self.static.y.shape), non_blocking=True)

    def load_from_dataset(self, dataset, idx_host):
        """Graph ids -> the captured input buffers, collated on the device from an HBM-resident ``DeviceDataset``."""
        dataset.collate_into(idx_host, self.static)

    def step(self, batch=None):
        """One optimisation step; returns the (device, captured) loss tensor -- valid until the next step."""
        if batch is not None:
            self.load(batch)
        self.graph.replay()
        if self.graph2 is not None:
            dist.all_reduce(self.flat, op=dist.ReduceOp.SUM)
            self.graph2.replay()
        return self.static_loss


EVAL_METRICS = ("l1", "mse", "bce", None)


def eval_terms(metric, out, y):
    """Per-graph terms of ``loss_fn(metric, out, y)`` (its SUM over graphs is the loss): out [B, d], labels y (any shape with
    B * d elements) -> (term [B], correct [B] or None).  ``correct`` = [(o > 0) == (y > 0.5)] for a single-output "bce" head (the
    accuracy of exp_classify.py's test loop); None for the other metrics and for wider heads."""
    y = y.to(out.dtype).reshape(out.shape)
    if metric == "l1":
        return (out - y).abs().sum(1), None
    if metric == "mse":
        return torch.square(out - y).sum(1), None
    if metric == "bce":
        term = F.binary_cross_entropy(torch.sigmoid(out), y, reduction="none").sum(1)
        correct = ((out[:, 0] > 0) == (y[:, 0] > 0.5)).to(out.dtype) if out.size(1) == 1 else None
        return term, correct
    raise ValueError(metric)


def eval_chunks(ids, batch_size, n_nodes):
    """The batches of an evaluation pass over the split ``ids``: consecutive chunks of ``batch_size`` ids (clipped to len(ids)),
    in order, as the reference's ``DataLoader(shuffle=False)``; a short last chunk is filled up to ``batch_size`` with copies of
    the split's smallest graph (fewest nodes, first such id).  ``n_nodes``: the dataset's node count per graph.
    -> (chunks [n_chunks, B] int64, weights [n_chunks, B] float32: 1 for the split's graphs, 0 for the fillers)."""
    import numpy as np
    ids = np.asarray(ids, dtype=np.int64).reshape(-1)
    B = min(int(batch_size), len(ids))
    nc = -(-len(ids) // B)
    filler = ids[int(np.argmin(np.asarray(n_nodes)[ids]))]
    chunks = np.full(nc * B, filler, dtype=np.int64)
    chunks[:len(ids)] = ids
    w = np.zeros(nc * B, dtype=np.float32)
    w[:len(ids)] = 1.0
    return chunks.reshape(nc, B), w.reshape(nc, B)


def eval_shapes(dataset, chunks, max_pad_degree=8):
    """Padded shapes of the captured evaluation batch from the dataset's host size arrays (``n_h``, ``e_h``, ``m_h``) and the
    chunks of ``eval_chunks``, with the rule of ``padded_shapes``: (n_nodes, n_entries or None, n_edges or None).  The batch
    carries the lists the dataset keeps: supports (``e_h``) and / or plain edges (``m_h``)."""
    nodes = dataset.n_h[chunks].sum(1)
    entries = dataset.e_h[chunks].sum(1) if dataset.e_h is not None else None
    if dataset.m_h is None:
        Np, Ep = padded_shapes_from_sizes(nodes, entries, max_pad_degree=max_pad_degree)
        return Np, Ep, None
    return padded_shapes_from_sizes(nodes, entries, dataset.m_h[chunks].sum(1), max_pad_degree=max_pad_degree)


class GraphedEvaluator(object):
    """The test loop of the reference's scripts (``test()``: MAE on ZINC, MSE on counting, accuracy on EXP, the embeddings of the
    isomorphism scripts) over a split of a resident ``synthetic.DeviceDataset``, captured ONCE into a CUDA graph and replayed per
    batch: device collation into static buffers, the model's forward under ``no_grad`` (the forward-only kernels: nothing is saved
    for a backward) and the metric accumulated on the device in float64.

        ev = GraphedEvaluator(model, dataset, ids, batch_size, metric="l1")
        res = ev.run()                  # {"graphs": n, "sum": s, "mean": s / n} (+ "correct", "accuracy" for "bce")
        res = ev.run(outputs=True)      # also res["outputs"]: [len(ids), out] device tensor in id order

    Batches are consecutive chunks of ``ids`` (``eval_chunks``); a short last chunk is filled with copies of the split's smallest
    graph, which a per-graph weight (0 for fillers) keeps out of the metric and the outputs.  Shapes come from the dataset's host
    size arrays (``eval_shapes``), so nothing is collated on the host.  The model runs in eval mode (BatchNorm running statistics,
    no dropout) during warm-up and capture; its previous mode is restored afterwards.  The graph reads parameters and buffers in
    place: a trainer stepping the same model between two ``run()`` calls is seen by the second.  ``run()`` reads the device once,
    at the end.  ``distributed=True``: every rank passes its own ids and ``run()`` SUM-all-reduces the metric once (outputs stay per
    rank).  ``metric``: "l1", "mse", "bce" (the per-graph terms of ``loss_fn``) or None (outputs only)."""

    def __init__(self, model, dataset, ids, batch_size, metric="l1", max_pad_degree=8, distributed=False, warmup=2):
        import numpy as np
        from .batch import Batch
        from .graph import set_range_check
        if metric not in EVAL_METRICS:
            raise ValueError("GraphedEvaluator: metric must be one of %s, got %r" % (EVAL_METRICS, metric))
        ids = np.asarray(ids, dtype=np.int64).reshape(-1)
        if len(ids) == 0:
            raise ValueError("GraphedEvaluator: ids is empty")
        if ids.min() < 0 or ids.max() >= len(dataset.n_h):
            raise ValueError("GraphedEvaluator: ids outside the dataset's %d graphs" % len(dataset.n_h))
        if int(batch_size) < 1:
            raise ValueError("GraphedEvaluator: batch_size must be positive")
        self.model, self.dataset, self.metric = model, dataset, metric
        self.n = len(ids)
        self.chunks, weights = eval_chunks(ids, batch_size, dataset.n_h)
        self.B = B = self.chunks.shape[1]
        Np, Ep, Mp = eval_shapes(dataset, self.chunks, max_pad_degree)
        self.shapes = (Np, Ep, Mp)
        self.distributed = distributed and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        set_range_check(False)                         # the range check reads a flag back from the device
        dev = dataset.x.device
        self._ids = [torch.from_numpy(c).pin_memory() for c in self.chunks]
        self._w_all = torch.from_numpy(weights).to(dev)
        f32 = dict(dtype=torch.float32, device=dev)
        st = Batch(x=torch.zeros(Np, dataset.x.size(1), **f32), batch=torch.zeros(Np, dtype=torch.int64, device=dev),
                   graph_ptr=torch.zeros(B + 2, dtype=torch.int32, device=dev), num_graphs=B + 1, real_graphs=B,
                   y=torch.zeros(B, dataset.y[:1].numel(), dtype=dataset.y.dtype, device=dev))
        if dataset.e_h is not None:
            st.edge_index2 = torch.zeros(2, Ep, dtype=torch.int64, device=dev)
            st.edge_attr2 = torch.zeros(Ep, dataset.ea.size(1), **f32)
        if dataset.m_h is not None:
            st.edge_index = torch.zeros(2, Mp, dtype=torch.int64, device=dev)
        self.static = st
        self.w = torch.zeros(B, **f32)
        self.acc = torch.zeros(3, dtype=torch.float64, device=dev)        # metric sum | correct | graphs
        dataset.collate_into(self._ids[0], st)
        self.w.copy_(self._w_all[0])
        was_training = model.training
        model.eval()
        try:
            s = torch.cuda.Stream(device=dev)
            s.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(s), torch.no_grad():
                for _ in range(warmup):
                    self._step()
            torch.cuda.current_stream(dev).wait_stream(s)
            torch.cuda.synchronize(dev)
            self.graph = torch.cuda.CUDAGraph()
            with torch.no_grad(), torch.cuda.graph(self.graph):
                self.static_out = self._step()
        finally:
            model.train(was_training)

    def _step(self):
        """Forward of the static batch and the metric of its real graphs, added to the accumulator."""
        out = self.model(self.static.fresh())[:self.B]
        if out.dim() == 1:
            out = out.unsqueeze(1)
        if self.metric is not None:
            real = self.w > 0
            term, correct = eval_terms(self.metric, out, self.static.y)
            self.acc[0] += torch.where(real, term, torch.zeros_like(term)).double().sum()
            if correct is not None:
                self.acc[1] += torch.where(real, correct, torch.zeros_like(correct)).double().sum()
        self.acc[2] += self.w.double().sum()
        return out

    def run(self, outputs=False):
        """One pass over the split: per batch, device collation into the captured buffers, the weights and one replay."""
        self.acc.zero_()
        out_all = torch.empty(len(self._ids) * self.B, self.static_out.size(1), dtype=self.static_out.dtype,
                              device=self.static_out.device) if outputs else None
        for c, ix in enumerate(self._ids):
            self.dataset.collate_into(ix, self.static)
            self.w.copy_(self._w_all[c])
            self.graph.replay()
            if outputs:
                out_all[c * self.B:(c + 1) * self.B].copy_(self.static_out)
        if self.distributed:
            dist.all_reduce(self.acc, op=dist.ReduceOp.SUM)
        vals = self.acc.tolist()                       # the pass's one read from the device
        res = {"graphs": int(round(vals[2]))}
        if self.metric is not None:
            res["sum"] = vals[0]
            res["mean"] = vals[0] / max(res["graphs"], 1)
            if self.metric == "bce" and self.static_out.size(1) == 1:
                res["correct"] = int(round(vals[1]))
                res["accuracy"] = vals[1] / max(res["graphs"], 1)
        if outputs:
            res["outputs"] = out_all[:self.n]
        return res
