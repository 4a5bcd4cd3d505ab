"""GNNML1's data path on the host: the pool's vectorised adjacency collation, the wire format of plain edge lists, the padding
of ``edge_index`` and its shapes, and the library's new collation entry points.  No GPU needed."""
import ctypes
import os

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _records(pool, idx, supports=True):
    out = []
    for i in idx:
        a, b = pool.node_off[i], pool.node_off[i + 1]
        r = dict(x=pool.x[a:b], edge_index=pool.ei1[:, pool.edge_off1[i]:pool.edge_off1[i + 1]], y=pool.y[i])
        if supports:
            e0, e1 = pool.edge_off[i], pool.edge_off[i + 1]
            r.update(edge_index2=pool.ei2[:, e0:e1], edge_attr2=pool.ea2[e0:e1])
        out.append(r)
    return out


@pytest.mark.parametrize("kind", ["zinc", "counting", "sweep"])
def test_pool_adjacency_collation_equals_batch_collate(kind):
    from gnn_matlang_b200.batch import collate
    from gnn_matlang_b200.synthetic import GraphPool
    pool = GraphPool(kind, 40, seed=2)
    idx = np.random.default_rng(1).integers(0, 40, 90)
    got, ref = pool.collate(idx, adjacency=True), collate(_records(pool, idx), adjacency=True)
    assert set(got.__dict__) == set(ref.__dict__)
    for k, v in ref.__dict__.items():
        w = getattr(got, k)
        if isinstance(v, torch.Tensor):
            assert v.dtype == w.dtype and torch.equal(v, w), k
        else:
            assert v == w, k
    plain = pool.collate(idx)
    assert not hasattr(plain, "edge_index")
    for k, v in plain.__dict__.items():
        assert (torch.equal(v, getattr(got, k)) if isinstance(v, torch.Tensor) else v == getattr(got, k)), k


def _bare_batch(sizes, seed):
    """Adjacency batch without supports; graph i has sizes[i] = (nodes, edges)."""
    from gnn_matlang_b200.batch import collate
    rng = np.random.default_rng(seed)
    gs = [dict(x=rng.standard_normal((n, 3)).astype(np.float32), edge_index=rng.integers(0, max(n, 1), (2, m)).astype(np.int64),
               y=np.float32(i)) for i, (n, m) in enumerate(sizes)]
    return collate(gs, adjacency=True)


@pytest.mark.parametrize("nmax,dtype", [(200, torch.uint8), (256, torch.uint8), (257, torch.int16), (40000, torch.int32)])
def test_compact_batch_of_plain_edges_picks_the_smallest_id_dtype(nmax, dtype):
    from gnn_matlang_b200.batch import CompactBatch
    hb = _bare_batch([(5, 7), (nmax, 30), (1, 0), (3, 4)], seed=nmax)
    cb = CompactBatch.from_batch(hb)
    assert cb.el is None and cb.e is None and cb.ea is None
    assert cb.al.dtype == dtype and cb.al.is_contiguous() and cb.m.dtype == torch.int32
    assert cb.m.tolist() == [7, 30, 0, 4]
    gp = np.concatenate([[0], np.cumsum(cb.n.numpy().astype(np.int64))])
    assert np.array_equal(cb.al.numpy().astype(np.int64) + np.repeat(gp[:-1], cb.m.numpy())[None, :], hb.edge_index.numpy())
    assert cb.sizes() == (hb.x.shape[0], None, hb.edge_index.shape[1])


def test_compact_batch_with_both_lists_and_its_size():
    from gnn_matlang_b200.batch import CompactBatch
    from gnn_matlang_b200.synthetic import GraphPool
    pool = GraphPool("zinc", 64, seed=3)
    idx = np.random.default_rng(2).integers(0, 64, 300)
    hb = pool.collate(idx, adjacency=True)
    cb = CompactBatch.from_batch(hb, (21, 4))
    ref = CompactBatch.from_batch(pool.collate(idx), (21, 4))
    for k in ("n", "e", "el", "ea", "xc", "y"):
        assert torch.equal(getattr(cb, k), getattr(ref, k)), k
    assert cb.al.dtype == torch.uint8 and cb.m.tolist() == pool.e1[idx].tolist()
    # GNNML1 wire format (no supports): 2 bytes per node, 2 per plain edge, 8 per graph, the labels
    bare = CompactBatch.from_batch(hb.__class__(**{k: v for k, v in hb.__dict__.items() if k not in ("edge_index2", "edge_attr2")}),
                                   (21, 4))
    N, M, B = hb.x.shape[0], hb.edge_index.shape[1], len(idx)
    assert bare.nbytes() == 2 * N + 2 * M + 8 * B + 4 * B


def test_compact_batch_rejects_cross_graph_and_ungrouped_plain_edges():
    from gnn_matlang_b200.batch import CompactBatch
    hb = _bare_batch([(4, 5), (6, 8), (3, 2)], seed=4)
    bad = hb.__class__(**hb.__dict__)
    ei = hb.edge_index.clone()
    ei[1, 0] = 5                                              # graph 0's first edge ends in graph 1
    bad.edge_index = ei
    with pytest.raises(ValueError, match="edge_index crosses graph boundaries"):
        CompactBatch.from_batch(bad)
    ei = torch.cat([hb.edge_index[:, 5:13], hb.edge_index[:, :5], hb.edge_index[:, 13:]], 1)
    bad.edge_index = ei
    with pytest.raises(ValueError, match="edge_index is not grouped by graph"):
        CompactBatch.from_batch(bad)
    with pytest.raises(ValueError):
        CompactBatch.from_batch(hb.__class__(**{k: v for k, v in hb.__dict__.items() if k != "edge_index"}))


def test_pad_batch_pads_the_plain_list_on_dummy_nodes_only():
    from gnn_matlang_b200.synthetic import GraphPool
    from gnn_matlang_b200.train import pad_batch, padded_shapes
    pool = GraphPool("zinc", 64, seed=5)
    rng = np.random.default_rng(3)
    host = [pool.collate(rng.integers(0, 64, b), adjacency=True) for b in (40, 48, 33)]
    for deg in (2, 3, 8):
        Np, Ep, Mp = padded_shapes(host, max_pad_degree=deg, adjacency=True)
        assert Ep == max(h.edge_index2.shape[1] for h in host) and Mp == max(h.edge_index.shape[1] for h in host)
        for hb in host:
            N, E, M, B = hb.x.shape[0], hb.edge_index2.shape[1], hb.edge_index.shape[1], hb.num_graphs
            p = pad_batch(hb, Np, Ep, Mp)
            assert p.num_graphs == B + 1 and p.real_graphs == B
            assert p.graph_ptr.tolist() == hb.graph_ptr.tolist() + [Np]      # one dummy graph
            assert torch.equal(p.edge_index[:, :M], hb.edge_index) and torch.equal(p.edge_index2[:, :E], hb.edge_index2)
            tail = p.edge_index[:, M:]
            assert torch.equal(tail[0], tail[1]) and bool((tail[0] >= N).all()) and bool((tail[0] < Np).all())
            assert bool((p.batch[N:] == B).all()) and bool((p.x[N:] == 0).all())
            # self-loops per dummy node, both lists together
            loops = torch.cat([p.edge_index2[0, E:], tail[0]])
            assert int(torch.bincount(loops - N, minlength=Np - N).max()) <= deg
    # a batch without supports
    bare = [h.__class__(**{k: v for k, v in h.__dict__.items() if k not in ("edge_index2", "edge_attr2")}) for h in host]
    Np, Ep, Mp = padded_shapes(bare, adjacency=True)
    assert Ep is None
    p = pad_batch(bare[0], Np, None, Mp)
    assert not hasattr(p, "edge_index2") and p.edge_index.shape == (2, Mp)
    with pytest.raises(ValueError):
        pad_batch(host[0], Np, None, Mp)                      # supports need n_entries
    with pytest.raises(ValueError):
        pad_batch(host[0], host[0].x.shape[0], host[0].edge_index2.shape[1], Mp)      # no dummy node


def test_existing_pad_batch_and_padded_shapes_calls_are_unchanged():
    """Two-size calls: the result has exactly the fields and values of the support-only padding (no edge_index), and
    padded_shapes keeps its (n_nodes, n_entries) formula."""
    from gnn_matlang_b200.synthetic import GraphPool
    from gnn_matlang_b200.train import pad_batch, padded_shapes
    pool = GraphPool("zinc", 64, seed=6)
    rng = np.random.default_rng(4)
    host = [pool.collate(rng.integers(0, 64, 48), adjacency=a) for a in (False, True)]
    n = [h.x.shape[0] for h in host]
    e = [h.edge_index2.shape[1] for h in host]
    assert padded_shapes(host) == (max(n) + 1 + (max(e) - min(e) + 7) // 8, max(e))
    assert padded_shapes(host, max_pad_degree=3) == (max(n) + 1 + (max(e) - min(e) + 2) // 3, max(e))
    Np, Ep = padded_shapes(host)
    for hb in host:
        p = pad_batch(hb, Np, Ep)
        assert list(p.__dict__) == ["x", "edge_index2", "edge_attr2", "batch", "num_graphs", "graph_ptr", "y", "real_graphs"]
        N, E = hb.x.shape[0], hb.edge_index2.shape[1]
        want = (N + torch.arange(Ep - E) % (Np - N)).unsqueeze(0).expand(2, -1)
        assert torch.equal(p.edge_index2[:, E:], want) and bool((p.edge_attr2[E:] == 0).all())


def test_from_graphs_reads_reader_records_and_refuses_bad_ids():
    from gnn_matlang_b200.datasets import read_graph6
    from gnn_matlang_b200.synthetic import DeviceDataset
    recs = read_graph6(os.path.join(ROOT, "tests", "golden", "sr251256.g6"))
    with pytest.raises(RuntimeError):
        DeviceDataset.from_graphs(recs, torch.device("cpu")).collate(np.arange(4))      # CPU tensors: no CPU fallback
    dds = DeviceDataset.from_graphs(recs, torch.device("cpu"))
    assert dds.al.dtype == torch.uint8 and dds.ea is None and dds.y.shape == (len(recs), 1)
    assert dds.m_h.tolist() == [r["edge_index"].shape[1] for r in recs]
    with pytest.raises(ValueError):
        DeviceDataset.from_graphs([dict(x=np.ones((3, 1)), edge_index=np.array([[0], [3]]), y=0)], torch.device("cpu"))


def test_library_exports_the_collate_graphs_entry_points():
    from gnn_matlang_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in ("gnnml3_collate_graphs", "gnnml3_collate_graphs_workspace_bytes", "gnnml3_collate", "gnnml3_collate_workspace_bytes"):
        assert hasattr(lib, name), name
        assert name in _lib.SIGNATURES, name
    L = _lib.load()
    assert L.gnnml3_collate_graphs_workspace_bytes(8191) == 3 * 8192 * 8
    assert L.gnnml3_collate_workspace_bytes(8191) == 2 * 8192 * 8
    hdr = open(os.path.join(ROOT, "include", "gnnml3_b200.h")).read()
    assert "gnnml3_collate_graphs(" in hdr and "gnnml3_collate_graphs_workspace_bytes(" in hdr
