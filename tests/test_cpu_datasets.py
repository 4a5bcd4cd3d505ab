"""CPU tests of the PyG-free raw-file readers (gnn_matlang_b200/datasets.py; reference: libs/utils.py:440-442, 473-478)."""
import os
import pickle
import sys
import types

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import gnnml3_oracle as O


def test_read_graph6_matches_the_oracle_on_graph8c():
    from gnn_matlang_b200.datasets import read_graph6
    g = read_graph6(os.path.join(GOLDEN, "graph8c.g6"))
    ref = O.parse_graph6(os.path.join(GOLDEN, "graph8c.g6"))
    assert len(g) == len(ref) == 11117
    for a, (n, ei) in zip(g, ref):
        assert a["x"].shape == (n, 1) and a["x"].dtype == np.float32 and float(a["x"].min()) == 1.0 and a["y"] == 0
        assert a["edge_index"].dtype == np.int64 and np.array_equal(a["edge_index"], ei)      # bit-exact, same order
    # undirected, both directions present, sorted by (source, target) like to_undirected's coalesce
    ei = g[5000]["edge_index"]
    key = ei[0] * 8 + ei[1]
    assert bool((key[1:] > key[:-1]).all()) and set(map(tuple, ei.T)) == set(map(tuple, ei[::-1].T))


def test_read_graph6_known_encodings_and_edge_cases():
    from gnn_matlang_b200.datasets import read_graph6
    for n, s in [(2, b"A_"), (3, b"Bw"), (4, b"C~"), (5, b"D~{")]:                 # complete graphs K_n (McKay's formats.txt)
        (g,) = read_graph6(s)
        assert g["x"].shape == (n, 1) and g["edge_index"].shape == (2, n * (n - 1))
        assert all(int(a) != int(b) for a, b in g["edge_index"].T)
    (g,) = read_graph6(b">>graph6<<B?\n")                                            # optional header, empty graph on 3 nodes
    assert g["x"].shape == (3, 1) and g["edge_index"].shape == (2, 0) and g["edge_index"].dtype == np.int64
    (g,) = read_graph6(b"@")                                                         # single node, no bit payload
    assert g["x"].shape == (1, 1) and g["edge_index"].shape == (2, 0)
    big = b"~??~" + b"?" * 326                                                       # n = 63 uses the 4-byte size field
    (g,) = read_graph6(big)
    assert g["x"].shape == (63, 1) and g["edge_index"].shape == (2, 0)
    path = b"DQc"                                                                    # 5 nodes: edges 0-2, 0-4, 1-3, 3-4
    (g,) = read_graph6(path)
    assert sorted(map(tuple, g["edge_index"].T)) == sorted([(0, 2), (2, 0), (0, 4), (4, 0), (1, 3), (3, 1), (3, 4), (4, 3)])
    assert len(read_graph6(b"A_\n\nBw\n")) == 2
    with pytest.raises(ValueError):
        read_graph6(b"D~")                                                           # truncated: 6 bits for n = 5
    with pytest.raises(ValueError):
        read_graph6(b"A\x1f")                                                        # byte below the 63 offset


def _pyg_pickle(graphs):
    """Pickle of a list of PyG 1.x ``Data`` objects (the layout of the EXP dataset's GRAPHSAT.pkl) holding the tensors of
    ``graphs`` = [(x, edge_index, y), ...], made without torch_geometric: a class is registered under the module path PyG
    pickles ``Data`` with, and unregistered again."""
    assert not any(m.startswith("torch_geometric") for m in sys.modules)
    names = ["torch_geometric", "torch_geometric.data", "torch_geometric.data.data"]
    mods = {n: types.ModuleType(n) for n in names}

    class Data(object):
        pass

    Data.__module__, Data.__qualname__ = "torch_geometric.data.data", "Data"
    mods["torch_geometric.data.data"].Data = Data
    sys.modules.update(mods)
    try:
        objs = []
        for x, ei, y in graphs:
            d = Data()
            d.x, d.edge_index, d.edge_attr, d.y, d.pos, d.normal, d.face = x, ei, None, y, None, None, None
            objs.append(d)
        return pickle.dumps(objs)
    finally:
        for n in names:
            sys.modules.pop(n, None)


def test_read_exp_pickle_without_torch_geometric():
    """A pickle of objects whose class lives in `torch_geometric.data.data` is read with the class mapped to a plain record:
    torch_geometric is never imported (the product does not depend on it)."""
    from gnn_matlang_b200.datasets import read_exp_pickle
    graphs = []
    for i, (n, e) in enumerate([(4, 6), (1, 0), (7, 10)]):
        graphs.append((torch.arange(n).reshape(n, 1) % 2, torch.randint(0, n, (2, e), generator=torch.Generator().manual_seed(i)),
                       torch.tensor([i % 2])))
    out = read_exp_pickle(_pyg_pickle(graphs))
    assert not any(m.startswith("torch_geometric") for m in sys.modules)
    assert len(out) == 3
    for (x, ei, y), o in zip(graphs, out):
        assert o["x"].dtype == np.int64 and np.array_equal(o["x"], x.numpy())
        assert o["edge_index"].dtype == np.int64 and np.array_equal(o["edge_index"], ei.numpy())
        assert o["y"] == int(y)


def test_read_exp_pickle_matches_the_committed_fixture():
    """The first 200 graphs of the EXP dataset (tests/golden/exp_first200.npz, taken from the reference's GRAPHSAT.pkl by
    oracle/make_golden.py), pickled as the dataset file stores them (int64 tensors: x [n, 1] node types, edge_index [2, e],
    y [1]), are read back exactly and in file order."""
    from gnn_matlang_b200.datasets import read_exp_pickle
    z = np.load(os.path.join(GOLDEN, "exp_first200.npz"))
    xo, eo = np.cumsum(np.r_[0, z["n"]]), np.cumsum(np.r_[0, z["ne"]])
    t = lambda a: torch.from_numpy(a.astype(np.int64))
    e = read_exp_pickle(_pyg_pickle([(t(z["x"][xo[i]:xo[i + 1]]).reshape(-1, 1), t(z["edge_index"][:, eo[i]:eo[i + 1]]), t(z["y"][i:i + 1]))
                                     for i in range(200)]))
    assert len(e) == 200
    for i in range(200):
        assert e[i]["x"].shape == (z["n"][i], 1)
        assert np.array_equal(e[i]["x"].reshape(-1), z["x"][xo[i]:xo[i + 1]])
        assert np.array_equal(e[i]["edge_index"], z["edge_index"][:, eo[i]:eo[i + 1]])
        assert e[i]["y"] == int(z["y"][i])


def test_read_mat_zinc_and_counting_schemas(tmp_path):
    """Synthetic files in the schemas of libs/utils.py:240-261 (Zinc.mat) and :386-413 (randomgraph.mat); expected values from a
    direct restatement of those lines."""
    import scipy.io as sio
    from scipy.special import comb
    from gnn_matlang_b200.datasets import read_mat
    rng = np.random.default_rng(0)
    graphs = []
    for n in (5, 9, 23):
        A = np.triu((rng.random((n, n)) < 0.3).astype(np.uint8), 1)
        A = A + A.T
        graphs.append(A)
    E = np.empty((1, len(graphs)), dtype=object)
    F = np.empty((1, len(graphs)), dtype=object)
    for i, A in enumerate(graphs):
        A4 = np.minimum(A, 1) * (A.sum(1, keepdims=True) <= 4)          # keep degrees <= 4 like molecules
        A4 = np.minimum(A4, A4.T)
        graphs[i] = A4
        E[0, i] = A4
        F[0, i] = np.array([rng.integers(0, 21, A4.shape[0])])
    Y = rng.normal(size=(len(graphs), 1))
    sio.savemat(str(tmp_path / "Zinc.mat"), {"E": E, "F": F, "Y": Y})
    recs = read_mat(str(tmp_path / "Zinc.mat"), "zinc")
    assert len(recs) == 3
    for i, r in enumerate(recs):
        A = graphs[i]
        ref_ei = np.vstack(np.where(A > 0))
        assert np.array_equal(r["edge_index"], ref_ei) and r["edge_index"].dtype == np.int64
        x = np.zeros((A.shape[0], 25), np.float32)
        deg = (A > 0).sum(1)
        for j in range(A.shape[0]):
            x[j, F[0, i][0][j]] = 1
            x[j, -int(deg[j])] = 1
        assert np.array_equal(r["x"], x) and np.allclose(r["y"], Y[i, :])
    Ac = np.empty((1, len(graphs)), dtype=object)
    for i, A in enumerate(graphs):
        Ac[0, i] = A.astype(np.float64)
    sio.savemat(str(tmp_path / "randomgraph.mat"), {"A": Ac, "F": np.zeros((3, 5))})
    recs = read_mat(str(tmp_path / "randomgraph.mat"), "counting")
    for i, r in enumerate(recs):
        a = graphs[i].astype(np.float64)
        A2 = a.dot(a); A3 = A2.dot(a)
        tri = np.trace(A3) / 6
        tailed = ((np.diag(A3) / 2) * (a.sum(0) - 2)).sum()
        cyc4 = 1 / 8 * (np.trace(A3.dot(a)) + np.trace(A2) - 2 * A2.sum())
        cus = a.dot(np.diag(np.exp(-a.dot(a).sum(1)))).dot(a).sum()
        star = sum(comb(int(d), 3) for d in a.sum(0))
        assert np.allclose(r["y"], [[tri, tailed, star, cyc4, cus]], rtol=0, atol=1e-12)
        assert r["x"].shape == (a.shape[0], 1) and float(r["x"].min()) == 1.0
        assert np.array_equal(r["edge_index"], np.vstack(np.where(a > 0)))


def _write_tu_mat(path, kind, count):
    """A file in the schema of the reference's TU file ``kind``, with ``count`` seeded random graphs: ``A`` and ``F`` are
    1 x count cells of sparse adjacencies and node feature matrices; the labels are ``Y`` (1 x count, ENZYMES' classes 1..6),
    ``Y`` (count x 1, PROTEINS / PTC) or ``y`` (count x 1 in {-1, 1}, MUTAG)."""
    import scipy.io as sio
    import scipy.sparse as sp
    rng = np.random.default_rng(count)
    width = dict(enzymes=21, proteins=4, ptc=18, mutag=7)[kind]
    A = np.empty((1, count), dtype=object)
    F = np.empty((1, count), dtype=object)
    for i in range(count):
        n = int(rng.integers(1, 30))
        up = np.triu(rng.random((n, n)) < 3.0 / n, 1)
        A[0, i] = sp.csc_matrix((up | up.T).astype(np.float64))
        F[0, i] = rng.integers(0, 2, (n, width)).astype(np.float64)
    if kind == "enzymes":
        labels = {"Y": rng.integers(1, 7, (1, count))}
    elif kind == "mutag":
        labels = {"y": rng.choice([-1, 1], (count, 1))}
    else:
        labels = {"Y": rng.integers(0, 2, (count, 1))}
    os.makedirs(os.path.dirname(path), exist_ok=True)
    sio.savemat(path, dict(A=A, F=F, **labels))


@pytest.mark.parametrize("kind,rel,count,nfeat", [("enzymes", "enzymes/raw/enzymes.mat", 600, 3), ("proteins", "proteins/raw/proteins.mat", 1113, 3),
                                                  ("ptc", "PTC/raw/ptc.mat", 344, None), ("mutag", "mutag/raw/mutag.mat", 188, None)])
def test_read_mat_tu_files_shipped_with_the_reference(kind, rel, count, nfeat, tmp_path):
    """Files in the schema of the TU files that ship with the reference (as many graphs as each of them holds), against a
    restatement of the dataset classes' process() lines (libs/utils.py:46-61, 93-112, 146-165, 195-211)."""
    import scipy.io as sio
    from gnn_matlang_b200.datasets import read_mat
    path = str(tmp_path / rel)
    _write_tu_mat(path, kind, count)
    recs = read_mat(path, kind)
    a = sio.loadmat(path)
    assert len(recs) == count
    A, F = a["A"][0], a["F"][0]
    for i in (0, 1, count // 2, count - 1):
        Ai = A[i].toarray() if hasattr(A[i], "toarray") else A[i]
        assert np.array_equal(recs[i]["edge_index"], np.vstack(np.where(Ai > 0)))
        f = np.asarray(F[i])
        assert np.array_equal(recs[i]["x"], (f[:, 0:3] if nfeat else f).astype(np.float32))
    if kind == "mutag":
        assert set(float(r["y"][0]) for r in recs) == {0.0, 1.0}
    elif kind == "enzymes":
        assert sorted(set(int(r["y"][0]) for r in recs)) == sorted(set(int(v) for v in a["Y"][0]))
