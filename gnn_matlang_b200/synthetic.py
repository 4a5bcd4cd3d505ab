"""Synthetic graph generators shaped like the reference's datasets (SURVEY.md section 8d) -- the real ZINC /
subgraph-counting .mat files are not shipped with the reference (``.MISSING_LARGE_BLOBS``), so bench.py and
the tests train on graphs of the same shape:

* ``zinc``      -- molecule-like: random tree with max degree 4 plus 1-3 ring closures, n ~ clipped
                   N(23.2, 4.3) in [9, 37]; x = 21-way atom one-hot + 4-way degree one-hot
                   (libs/utils.py:253-259); supports over the 2-hop mask (Zinc12k.py:12: recfield=2, nfreq=7 -> K=8)
* ``counting``  -- random regular graphs (n, d) in {(10,6), (15,6), (20,5), (30,5)}; x = [1, deg/max];
                   1-hop mask, K = 12 (counting.py:16: nfreq=10, addadj)
* ``sweep``     -- G(n, 4/(n-1)), n ~ U{30..100}; 1-hop or 2-hop mask; K = 10

A pool of distinct graphs is generated once; batches are drawn from the pool and collated with vectorised
numpy (same result as ``batch.collate`` on the drawn records).
"""
import numpy as np
import torch

from .batch import Batch


def _sym_sorted(u, v):
    ei = np.concatenate([np.vstack((u, v)), np.vstack((v, u))], 1)
    order = np.lexsort((ei[1], ei[0]))
    return ei[:, order].astype(np.int64)


def zinc_graph(rng):
    n = int(np.clip(round(rng.normal(23.2, 4.3)), 9, 37))
    deg = np.zeros(n, dtype=np.int64)
    us, vs = [], []
    for v in range(1, n):
        lo = max(0, v - 6)
        cand = np.arange(lo, v)
        cand = cand[deg[cand] < 3]
        if len(cand) == 0:
            cand = np.arange(0, v)
            cand = cand[deg[cand] < 4]
        u = int(cand[rng.integers(len(cand))])
        us.append(u)
        vs.append(v)
        deg[u] += 1
        deg[v] += 1
    have = set(zip(us, vs))
    for _ in range(int(rng.integers(1, 4))):
        for _try in range(10):
            u, v = sorted(int(t) for t in rng.integers(0, n, 2))
            if 2 <= v - u <= 6 and (u, v) not in have and deg[u] < 4 and deg[v] < 4:
                have.add((u, v))
                us.append(u)
                vs.append(v)
                deg[u] += 1
                deg[v] += 1
                break
    ei = _sym_sorted(np.array(us), np.array(vs))
    x = np.zeros((n, 25), np.float32)
    x[np.arange(n), rng.integers(0, 21, n)] = 1
    x[np.arange(n), 25 - np.clip(deg, 1, 4)] = 1
    return n, ei, x


def regular_graph(rng, n, d):
    while True:
        stubs = np.repeat(np.arange(n), d)
        rng.shuffle(stubs)
        a, b = stubs[0::2], stubs[1::2]
        if np.any(a == b):
            continue
        key = np.minimum(a, b) * n + np.maximum(a, b)
        if len(np.unique(key)) != len(key):
            continue
        return _sym_sorted(a, b)


def counting_graph(rng):
    n, d = [(10, 6), (15, 6), (20, 5), (30, 5)][int(rng.integers(4))]
    ei = regular_graph(rng, n, d)
    x = np.ones((n, 2), np.float32)
    x[:, 1] = np.bincount(ei[0], minlength=n) / 6.0
    return n, ei, x


def sweep_graph(rng, nfeat):
    n = int(rng.integers(30, 101))
    up = np.triu(rng.random((n, n)) < 4.0 / (n - 1), 1)
    u, v = np.where(up)
    ei = _sym_sorted(u, v)
    return n, ei, rng.standard_normal((n, nfeat)).astype(np.float32)


def _local_graph(rng, n, extra, window):
    """Connected graph of n nodes: a random tree whose edges join nodes at most ``window`` apart, plus ``extra`` distinct chords
    of the same reach (molecule / protein-contact like, no hubs)."""
    have = set()
    for v in range(1, n):
        have.add((int(rng.integers(max(0, v - window), v)), v))
    for _ in range(extra):
        u = int(rng.integers(0, n))
        v = int(min(n - 1, u + rng.integers(2, window + 1)))
        if u < v:
            have.add((u, v))
    if not have:
        return np.zeros((2, 0), np.int64)
    u, v = (np.array(a, dtype=np.int64) for a in zip(*sorted(have)))
    return _sym_sorted(u, v)


def tu_records(kind, count, seed=0):
    """Reader-shaped records (``datasets.read_mat``: ``dict(x, edge_index, y)``) of synthetic graphs shaped like two TU datasets
    the ``enzymes`` / ``mutag`` presets train on (their ``.mat`` files are not part of this repository):

    * ``enzymes`` -- n ~ Gamma(4.5, 7.3) clipped to [2, 126] (ENZYMES: 2-126 nodes, mean ~33), every 50th graph 120-126 nodes
                     (beyond the one-block eigensolver's envelope), ~1.9 edges per node; x = one-hot of 3 node labels (the three
                     feature columns ``read_mat`` keeps); y = int64 [1] class in 0..5, a function of the dominant node label and
                     the size (learnable, so that a short training run shows a falling loss)
    * ``mutag``   -- n ~ N(18, 4.6) clipped to [10, 28], tree plus 1-3 ring chords; x = one-hot of 7 atom types; y = float32 [1]
                     in {0, 1} (whether the graph holds at least two atoms of type 1)"""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(count):
        if kind == "enzymes":
            n = int(rng.integers(120, 127)) if i % 50 == 49 else int(np.clip(round(rng.gamma(4.5, 7.3)), 2, 126))
            ei = _local_graph(rng, n, int(round(0.9 * n)), 6)
            lab = rng.choice(3, size=n, p=rng.dirichlet([1.0, 1.0, 1.0]))
            x = np.eye(3, dtype=np.float32)[lab]
            y = np.array([(int(np.bincount(lab, minlength=3).argmax()) * 2 + int(n > 30)) % 6], np.int64)
        elif kind == "mutag":
            n = int(np.clip(round(rng.normal(18.0, 4.6)), 10, 28))
            ei = _local_graph(rng, n, int(rng.integers(1, 4)), 4)
            lab = rng.choice(7, size=n, p=[0.7, 0.1, 0.1, 0.04, 0.03, 0.02, 0.01])
            x = np.eye(7, dtype=np.float32)[lab]
            y = np.array([float((lab == 1).sum() >= 2)], np.float32)
        else:
            raise ValueError("tu_records: kind must be 'enzymes' or 'mutag', got %r" % (kind,))
        out.append(dict(x=x, edge_index=ei, y=y))
    return out


def mask_edges(n, ei, recfield):
    """Row-major coordinates of the receptive-field mask (libs/utils.py:566-573, :608): recfield 0 -> A,
    r >= 1 -> (A + I)^(2^(r-1)) > 0."""
    A = np.zeros((n, n), dtype=bool)
    A[ei[0], ei[1]] = True
    if recfield == 0:
        M = A
    else:
        M = A | np.eye(n, dtype=bool)
        for _ in range(1, recfield):
            M = (M.astype(np.float32) @ M.astype(np.float32)) > 0
    r, c = np.where(M)
    return np.vstack((r, c)).astype(np.int64)


class GraphPool(object):
    """``count`` distinct graphs stored as flat arrays; ``draw(rng, B)`` collates a host Batch of B graphs."""

    def __init__(self, kind, count, seed=0, K=None, nfeat=None, recfield=None, supports="normal"):
        rng = np.random.default_rng(seed)
        self.kind = kind
        defaults = dict(zinc=(8, 25, 2), counting=(12, 2, 1), sweep=(10, 64, 1))[kind]
        self.K = K or defaults[0]
        self.F = nfeat or defaults[1]
        self.recfield = defaults[2] if recfield is None else recfield
        ns, xs, eis, eis1, ys = [], [], [], [], []
        for _ in range(count):
            if kind == "zinc":
                n, ei, x = zinc_graph(rng)
            elif kind == "counting":
                n, ei, x = counting_graph(rng)
            else:
                n, ei, x = sweep_graph(rng, self.F)
            ei2 = mask_edges(n, ei, self.recfield)
            ns.append(n)
            xs.append(x)
            eis.append(ei2)
            eis1.append(ei)
            ys.append(rng.standard_normal())
        self.n = np.array(ns, dtype=np.int64)
        self.e = np.array([e.shape[1] for e in eis], dtype=np.int64)
        self.node_off = np.concatenate([[0], np.cumsum(self.n)])
        self.edge_off = np.concatenate([[0], np.cumsum(self.e)])
        self.x = np.concatenate(xs, 0)
        self.ei2 = np.concatenate(eis, 1)
        self.ei1 = np.concatenate(eis1, 1)                  # the graphs' own edge lists (local ids): SpectralDesign's input
        self.e1 = np.array([e.shape[1] for e in eis1], dtype=np.int64)
        self.edge_off1 = np.concatenate([[0], np.cumsum(self.e1)])
        self.y = np.array(ys, dtype=np.float32)
        # edge features: N(0,1) placeholders unless real supports are attached with set_supports()
        self.ea2 = rng.standard_normal((self.ei2.shape[1], self.K)).astype(np.float32)
        self.supports = supports

    def set_supports(self, ea2):
        assert ea2.shape == self.ea2.shape
        self.ea2 = np.ascontiguousarray(ea2, dtype=np.float32)
        self.supports = "spectral_design"

    # SpectralDesign configuration of the reference script each pool kind mimics
    SPECTRAL_CONFIGS = {
        "zinc": dict(recfield=2, dv=2, nfreq=7),                                       # Zinc12k.py:12  -> K = 8
        "counting": dict(recfield=1, dv=1, nfreq=10, laplacien=False, addadj=True),    # counting.py:16 -> K = 12
        "sweep": dict(recfield=1, dv=2, nfreq=9),                                      # K = 10
    }

    def attach_spectral_supports(self, device):
        """Replace the N(0,1) placeholder edge features by the real supports: gnn_matlang_b200's SpectralDesign (one launch
        over the whole pool) with the reference script's settings.  The designed ``edge_index2`` must equal the pool's mask
        coordinates bit for bit (same row-major order) -- checked."""
        import torch
        from .libs.utils import SpectralDesign
        cfg = dict(self.SPECTRAL_CONFIGS[self.kind])
        cfg["recfield"] = self.recfield
        sd = SpectralDesign(**cfg)
        if sd.num_supports != self.K:
            raise RuntimeError("pool has K=%d, SpectralDesign config gives %d supports" % (self.K, sd.num_supports))
        out = sd.design_batch(torch.from_numpy(self.ei1), torch.from_numpy(self.edge_off1), torch.from_numpy(self.node_off),
                              device=device)
        ei2 = out["edge_index2"].cpu().numpy()
        if ei2.shape != self.ei2.shape or not np.array_equal(ei2, self.ei2):
            raise RuntimeError("SpectralDesign mask coordinates differ from the pool's")
        self.set_supports(out["edge_attr2"].cpu().numpy())
        return self

    def draw(self, rng, B):
        idx = rng.integers(0, len(self.n), B)
        return self.collate(idx)

    def collate(self, idx, adjacency=False):
        """Host ``Batch`` of the pool's graphs ``idx`` (same result as ``batch.collate`` on the records).  ``adjacency=True``:
        the batch also carries the graphs' plain ``edge_index`` (what GNNML1 reads), as ``batch.collate(..., adjacency=True)``."""
        idx = np.asarray(idx)
        n, e = self.n[idx], self.e[idx]
        goff = np.concatenate([[0], np.cumsum(n)])
        eoff = np.concatenate([[0], np.cumsum(e)])
        # vectorised range gather: node rows
        nsel = np.repeat(self.node_off[idx] - goff[:-1], n) + np.arange(goff[-1])
        esel = np.repeat(self.edge_off[idx] - eoff[:-1], e) + np.arange(eoff[-1])
        x = torch.from_numpy(self.x[nsel])
        ei = torch.from_numpy(self.ei2[:, esel] + np.repeat(goff[:-1], e)[None, :])
        ea = torch.from_numpy(self.ea2[esel])
        batch = torch.from_numpy(np.repeat(np.arange(len(idx), dtype=np.int64), n))
        out = Batch(x=x, edge_index2=ei, edge_attr2=ea, batch=batch, num_graphs=len(idx),
                    graph_ptr=torch.from_numpy(goff.astype(np.int32)), y=torch.from_numpy(self.y[idx]).reshape(-1, 1))
        if adjacency:
            m = self.e1[idx]
            moff = np.concatenate([[0], np.cumsum(m)])
            msel = np.repeat(self.edge_off1[idx] - moff[:-1], m) + np.arange(moff[-1])
            out.edge_index = torch.from_numpy(self.ei1[:, msel] + np.repeat(goff[:-1], m)[None, :])
        return out


class ExpPool(object):
    """Pool of REAL EXP graphs (the first 200 records of the reference's ``dataset/EXP/raw/GRAPHSAT.pkl``, committed as
    ``tests/golden/exp_first200.npz`` by the golden-fixture script): BASELINE.json configs[2].  Unlike ``GraphPool`` the records
    carry no supports: a batch is the raw graphs (node type ``x [n,1]``, local ``edge_index``) and the supports are rebuilt on
    the GPU for every batch (``design_and_collate``), as the config asks."""

    kind = "exp"
    K = 6                      # exp_classify.py:16: SpectralDesign(recfield=1, dv=2, nfreq=5, adddegree=True) -> nfreq + 1 supports
    F = 2                      # node type + degree column (adddegree)
    supports = "spectral_design (rebuilt on the GPU every step)"

    def __init__(self, path=None):
        import os
        if path is None:
            path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "exp_first200.npz")
        z = np.load(path)
        self.n = z["n"].astype(np.int64)
        self.e1 = z["ne"].astype(np.int64)
        self.node_off = np.concatenate([[0], np.cumsum(self.n)])
        self.edge_off1 = np.concatenate([[0], np.cumsum(self.e1)])
        self.x = z["x"].astype(np.float32).reshape(-1, 1)
        self.ei1 = z["edge_index"].astype(np.int64)
        self.y = z["y"].astype(np.float32)

    def draw_raw(self, rng, B):
        """Host batch of B raw graphs: dict of torch tensors (x [N,1], edge_index [2,Etot] LOCAL ids, edge_ptr, node_ptr, y)."""
        idx = rng.integers(0, len(self.n), B)
        n, e = self.n[idx], self.e1[idx]
        goff = np.concatenate([[0], np.cumsum(n)])
        eoff = np.concatenate([[0], np.cumsum(e)])
        nsel = np.repeat(self.node_off[idx] - goff[:-1], n) + np.arange(goff[-1])
        esel = np.repeat(self.edge_off1[idx] - eoff[:-1], e) + np.arange(eoff[-1])
        return dict(x=torch.from_numpy(self.x[nsel]), edge_index=torch.from_numpy(self.ei1[:, esel]),
                    edge_ptr=torch.from_numpy(eoff.astype(np.int32)), node_ptr=torch.from_numpy(goff.astype(np.int32)),
                    node_ptr_dev=torch.from_numpy(goff.astype(np.int32)), nmax=int(n.max()) if B > 0 else 1,
                    y=torch.from_numpy(self.y[idx]).reshape(-1, 1), num_graphs=int(B))


def design_and_collate(raw, sd, device):
    """Raw graphs (``ExpPool.draw_raw``, host or device tensors) -> device ``Batch`` with the supports designed on the GPU:
    one ``SpectralDesign.design_batch(global_ids=True)`` launch emits the batched ``edge_index2`` / ``edge_attr2`` directly
    (PyG's collation of ``edge_index2`` is the per-graph node offset the kernel adds), ``x`` gets the degree column
    (``adddegree``) and ``batch`` / ``graph_ptr`` come from ``node_ptr``."""
    node_ptr = raw["node_ptr"]
    npd = raw.get("node_ptr_dev")                  # device copy made when the batch was drawn: nothing is uploaded per step
    if npd is not None and npd.is_cuda:
        out = sd.design_batch(raw["edge_index"], raw["edge_ptr"], npd, device=device, global_ids=True, nmax=raw["nmax"],
                              num_nodes=int(node_ptr[-1]))
        gp = npd.to(torch.int32)
    else:
        out = sd.design_batch(raw["edge_index"], raw["edge_ptr"], node_ptr, device=device, global_ids=True)
        gp = node_ptr.to(device=device, dtype=torch.int32)
    x = raw["x"].to(device, non_blocking=True)
    if sd.adddegree:
        x = torch.cat([x, out["degree"].unsqueeze(-1)], 1)
    B = node_ptr.numel() - 1
    batch = torch.repeat_interleave(torch.arange(B, device=device), (gp[1:] - gp[:-1]).long(), output_size=int(x.size(0)))
    b = Batch(x=x, edge_index2=out["edge_index2"], edge_attr2=out["edge_attr2"], batch=batch, num_graphs=B, graph_ptr=gp,
              y=raw["y"].to(device, non_blocking=True))
    b.batch._gnnml3_ptr = (b.batch._version, gp)
    return b


def design_raw(raw, sd, device):
    """Raw graphs with device-resident fields (``ExpPool.draw_raw`` moved to the device, incl. ``node_ptr_dev`` / ``nmax``) -> the
    per-graph records ``gnnml3_collate`` batches: supports with graph-LOCAL ids, entry counts, features with the degree column.
    No upload, one read-back (the entry total that sizes the outputs)."""
    npd = raw["node_ptr_dev"]
    out = sd.design_batch(raw["edge_index"], raw["edge_ptr"], npd, device=device, global_ids=False, nmax=raw["nmax"],
                          num_nodes=int(raw["node_ptr"][-1]))
    x = raw["x"]
    if sd.adddegree:
        x = torch.cat([x, out["degree"].unsqueeze(-1)], 1)
    return dict(design=out, x=x.contiguous(), n32=(npd[1:] - npd[:-1]).to(torch.int32), num_graphs=int(npd.numel() - 1), y=raw["y"])


def _id_dtype(nmax):
    """Smallest integer dtype of graph-local node ids (the kernel reads uint8 / int16 / int32 / int64)."""
    return np.uint8 if nmax <= 256 else np.int16 if nmax <= 32768 else np.int32


class DeviceDataset(object):
    """A ``GraphPool`` resident in HBM + collation ON THE DEVICE (SURVEY.md 8f rank 1): the reference keeps its
    ``InMemoryDataset`` in host memory, collates every batch on the host and copies all attributes host -> device each step
    (Zinc12k.py:20-22, :360).  Here the per-graph records (features, graph-local support coordinates, supports, labels) are
    uploaded once; a step's only host -> device traffic is the list of graph ids, and ``collate`` builds the reference's batch
    attributes with a handful of index kernels -- bit-exact with ``GraphPool.collate`` / ``batch.collate`` (tested).

    ``adjacency=True`` also keeps the graphs' plain edge lists (graph-local ids, smallest integer dtype) and batches fill
    ``edge_index`` (what GNNML1 reads); ``supports=False`` leaves the support lists out (GNNML1 needs no SpectralDesign), and
    batches then carry no ``edge_index2`` / ``edge_attr2``."""

    def __init__(self, pool, device, adjacency=False, supports=True):
        if not adjacency and not supports:
            raise ValueError("DeviceDataset: keep the supports, the plain edge lists or both")
        self.device = device
        self.n_h = pool.n                                        # host copies: batch sizes are known without a device round trip
        t = lambda a, dt=None: torch.as_tensor(a if dt is None else a.astype(dt)).to(device)
        self.n = t(pool.n)
        self.n32 = self.n.to(torch.int32)
        self.node_off = t(pool.node_off)
        self.x = t(pool.x)
        self.y = t(pool.y)
        self.e_h = self.e = self.e32 = self.edge_off = self.el = self.ea = None
        if supports:
            self.e_h = pool.e
            self.e = t(pool.e)
            self.e32 = self.e.to(torch.int32)
            self.edge_off = t(pool.edge_off)
            self.el = t(pool.ei2)                                # support coordinates, node ids local to their graph
            self.ea = t(pool.ea2)
        self.m_h = self.m32 = self.adj_off = self.al = None
        if adjacency:
            self.m_h = pool.e1
            self.m32 = t(pool.e1, np.int32)
            self.adj_off = t(pool.edge_off1)
            self.al = t(np.ascontiguousarray(pool.ei1), _id_dtype(int(pool.n.max()) if len(pool.n) else 0))

    @classmethod
    def from_graphs(cls, records, device):
        """Resident dataset straight from per-graph records ``dict(x [n, F], edge_index [2, m] graph-local, y)`` -- what
        ``datasets.read_graph6``, ``read_exp_pickle`` and ``read_mat`` return: the plain edge lists only (GNNML1), batches
        carry ``x`` (float32), ``edge_index``, ``batch``, ``graph_ptr`` and ``y`` as ``batch.collate(records, adjacency=True)``."""
        self = cls.__new__(cls)
        self.device = device
        def get(g, k):
            return g.get(k) if isinstance(g, dict) else getattr(g, k, None)
        xs = [np.asarray(get(g, "x"), dtype=np.float32).reshape(np.shape(get(g, "x"))[0], -1) for g in records]
        eis = [np.asarray(get(g, "edge_index"), dtype=np.int64).reshape(2, -1) for g in records]
        self.n_h = np.array([x.shape[0] for x in xs], dtype=np.int64)
        self.m_h = np.array([ei.shape[1] for ei in eis], dtype=np.int64)
        for ei, n in zip(eis, self.n_h):
            if ei.size and (ei.min() < 0 or ei.max() >= n):
                raise ValueError("DeviceDataset.from_graphs: edge_index holds ids outside its graph")
        t = lambda a: torch.as_tensor(a).to(device)
        self.n = t(self.n_h)
        self.n32 = self.n.to(torch.int32)
        self.node_off = t(np.concatenate([[0], np.cumsum(self.n_h)]).astype(np.int64))
        self.x = t(np.concatenate(xs, 0))
        self.m32 = t(self.m_h.astype(np.int32))
        self.adj_off = t(np.concatenate([[0], np.cumsum(self.m_h)]).astype(np.int64))
        dt = _id_dtype(int(self.n_h.max()) if len(self.n_h) else 0)
        self.al = t(np.ascontiguousarray(np.concatenate(eis, 1).astype(dt)))
        ys = [torch.as_tensor(get(g, "y")) for g in records]         # batch.collate's label layout: one row per graph
        self.y = t(torch.cat([y.reshape(1, -1) if y.dim() < 2 else y for y in ys], 0))
        self.e_h = self.e = self.e32 = self.edge_off = self.el = self.ea = None
        return self

    @classmethod
    def from_records(cls, records, sd, device):
        """Resident GNNML3 dataset straight from reader records ``dict(x [n, F], edge_index [2, m] graph-local, y)`` (what
        ``datasets.read_mat``, ``read_graph6`` and ``read_exp_pickle`` return): the supports of ``sd`` (a ``SpectralDesign``) are
        designed on the device -- every graph within ``sd.max_kernel_nodes()`` in ONE ``design_batch`` launch, larger ones one by
        one on the dense path, as ``design_list`` routes them -- ``x`` gets the degree column when ``sd.adddegree`` is set, and
        features, supports and labels stay resident.  Batches carry ``x``, ``edge_index2``, ``edge_attr2``, ``batch``,
        ``graph_ptr`` and ``y`` as per-record ``sd(data)`` + ``batch.collate`` give them."""
        def get(g, k):
            return g.get(k) if isinstance(g, dict) else getattr(g, k, None)
        if len(records) == 0:
            raise ValueError("DeviceDataset.from_records: no records")
        xs = [np.asarray(get(g, "x"), dtype=np.float32).reshape(np.shape(get(g, "x"))[0], -1) for g in records]
        if len({x.shape[1] for x in xs}) != 1:
            raise ValueError("DeviceDataset.from_records: the records' x differ in width")
        eis = [np.asarray(get(g, "edge_index"), dtype=np.int64).reshape(2, -1) for g in records]
        n_h = np.array([x.shape[0] for x in xs], dtype=np.int64)
        for ei, n in zip(eis, n_h):
            if ei.size and (ei.min() < 0 or ei.max() >= n):
                raise ValueError("DeviceDataset.from_records: edge_index holds ids outside its graph")
        if any(get(g, "y") is None for g in records):
            raise ValueError("DeviceDataset.from_records: every record needs a label y")
        limit = sd.max_kernel_nodes()
        small = np.flatnonzero(n_h <= limit)
        large = np.flatnonzero(n_h > limit)
        # per-record blocks laid out as [all kernel-designed graphs | the large graphs one by one]; the collation reads every
        # record through its own node / entry offset, so the layout need not follow record order
        order = np.concatenate([small, large])
        els, eas, degs, counts = [], [], [], np.zeros(len(records), dtype=np.int64)
        if len(small):
            ns, ms = n_h[small], np.array([eis[i].shape[1] for i in small], dtype=np.int64)
            ei = np.concatenate([eis[i] for i in small], 1)
            out = sd.design_batch(torch.from_numpy(ei).to(device), torch.from_numpy(np.concatenate([[0], np.cumsum(ms)])).to(device),
                                  torch.from_numpy(np.concatenate([[0], np.cumsum(ns)])), device=device)
            els.append(out["edge_index2"])
            eas.append(out["edge_attr2"])
            degs.append(out["degree"])
            counts[small] = out["counts"].cpu().numpy()
        for i in large:
            o = sd._design_large(eis[i], int(n_h[i]), device=device)
            els.append(o["edge_index2"])
            eas.append(o["edge_attr2"])
            degs.append(o["degree"])
            counts[i] = o["edge_index2"].size(1)
        self = cls.__new__(cls)
        self.device = device
        self.n_h, self.e_h = n_h, counts
        node_off, edge_off = np.zeros(len(records) + 1, dtype=np.int64), np.zeros(len(records) + 1, dtype=np.int64)
        node_off[order] = np.concatenate([[0], np.cumsum(n_h[order])])[:-1]
        edge_off[order] = np.concatenate([[0], np.cumsum(counts[order])])[:-1]
        node_off[-1], edge_off[-1] = n_h.sum(), counts.sum()
        t = lambda a: torch.as_tensor(a).to(device)
        self.n, self.e = t(n_h), t(counts)
        self.n32, self.e32 = self.n.to(torch.int32), self.e.to(torch.int32)
        self.node_off, self.edge_off = t(node_off), t(edge_off)
        x = t(np.concatenate([xs[i] for i in order], 0))
        if sd.adddegree:
            x = torch.cat([x, torch.cat(degs).unsqueeze(-1)], 1)
        self.x = x.contiguous()
        self.el = torch.cat(els, 1).contiguous()
        self.ea = torch.cat(eas, 0).contiguous()
        ys = [torch.as_tensor(get(g, "y")) for g in records]         # batch.collate's label layout: one row per graph
        self.y = t(torch.cat([y.reshape(1, -1) if y.dim() < 2 else y for y in ys], 0))
        self.m_h = self.m32 = self.adj_off = self.al = None
        return self

    @classmethod
    def from_design(cls, design, node_ptr, x, y=None):
        """Resident dataset straight from ``SpectralDesign.design_batch(global_ids=False)`` (everything stays on the device):
        ``design['edge_index2']`` holds graph-local ids, ``design['e2_ptr']`` / ``node_ptr`` are the record offsets, ``x [Ntot, F]``
        the node features (degree column already appended when the design asks for it)."""
        self = cls.__new__(cls)
        dev = design["edge_attr2"].device
        self.device = dev
        npd = torch.as_tensor(node_ptr).to(dev, torch.int64)
        e2 = design["e2_ptr"].to(dev, torch.int64)
        self.n, self.e = npd[1:] - npd[:-1], e2[1:] - e2[:-1]
        self.n32, self.e32 = self.n.to(torch.int32), self.e.to(torch.int32)
        self.n_h, self.e_h = self.n.cpu().numpy(), self.e.cpu().numpy()
        self.node_off, self.edge_off = npd.contiguous(), e2.contiguous()
        self.x = x.to(dev, torch.float32).contiguous()
        self.el = design["edge_index2"].contiguous()
        self.ea = design["edge_attr2"].contiguous()
        B = self.n.numel()
        self.y = (torch.zeros(B, device=dev) if y is None else torch.as_tensor(y).to(dev)).reshape(B, -1)
        self.m_h = self.m32 = self.adj_off = self.al = None
        return self

    def _idx(self, idx_host):
        idx_np = idx_host.numpy() if isinstance(idx_host, torch.Tensor) else np.asarray(idx_host)
        idx = (idx_host if isinstance(idx_host, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(idx_np))).to(
            self.device, non_blocking=True).long()
        return idx_np, idx

    def _collate(self, idx, idx_np, out):
        from . import ops
        B = idx.numel()
        adj = self.al is not None and getattr(out, "edge_index", None) is not None
        if self.ea is None and not adj:
            raise ValueError("DeviceDataset: the output batch has no edge_index and the dataset keeps no supports")
        N = int(self.n_h[idx_np].sum())
        E = int(self.e_h[idx_np].sum()) if self.ea is not None else 0
        M = int(self.m_h[idx_np].sum()) if adj else 0
        Np, Ep, Mp = out.x.size(0), (out.edge_index2.size(1) if self.ea is not None else 0), (out.edge_index.size(1) if adj else 0)
        if N > Np or E > Ep or M > Mp or (Np == N and (Ep > E or Mp > M)):
            raise ValueError("DeviceDataset: the batch (%d nodes, %d entries, %d edges) does not fit the output (%d, %d, %d; padding "
                             "needs at least one dummy node)" % (N, E, M, Np, Ep, Mp))
        kw = dict(m=self.m32, al=self.al, adj_off=self.adj_off) if adj else {}
        ops.collate_device(self.n32, self.e32, self.el, self.ea, B, out, idx=idx, node_off=self.node_off, edge_off=self.edge_off,
                           x=self.x, **kw)
        return out

    def collate_into(self, idx_host, out):
        """Graph ids (int64 numpy array or pinned CPU tensor) -> the preallocated device ``Batch`` ``out`` (larger tensors get the
        neutral padding of ``train.pad_batch``; ``out.edge_index`` is filled when the dataset keeps the plain lists): ONE host ->
        device copy of the id list and two library launches."""
        idx_np, idx = self._idx(idx_host)
        self._collate(idx, idx_np, out)
        if getattr(out, "y", None) is not None:
            out.y.copy_(self.y[idx].reshape(out.y.shape))
        return out

    def collate(self, idx_host):
        """``idx_host``: int64/int32 numpy array or pinned CPU tensor of graph ids -> device ``Batch`` (exact sizes)."""
        idx_np, idx = self._idx(idx_host)
        N = int(self.n_h[idx_np].sum())
        dev = self.device
        B = idx.numel()
        out = Batch(x=torch.empty(N, self.x.size(1), dtype=torch.float32, device=dev))
        if self.ea is not None:
            E = int(self.e_h[idx_np].sum())
            out.edge_index2 = torch.empty(2, E, dtype=torch.int64, device=dev)
            out.edge_attr2 = torch.empty(E, self.ea.size(1), dtype=torch.float32, device=dev)
        out.batch = torch.empty(N, dtype=torch.int64, device=dev)
        out.graph_ptr = torch.empty(B + 1, dtype=torch.int32, device=dev)
        out.num_graphs = B
        if self.al is not None:
            out.edge_index = torch.empty(2, int(self.m_h[idx_np].sum()), dtype=torch.int64, device=dev)
        self._collate(idx, idx_np, out)
        out.y = self.y[idx].reshape(B, -1)
        out.batch._gnnml3_ptr = (out.batch._version, out.graph_ptr)
        return out
