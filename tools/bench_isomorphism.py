#!/usr/bin/env python
"""bench_isomorphism.py -- the paper's isomorphism test on one B200.  Prints ONE JSON line with

* ``graph8c``: the protocol of graph8c.py:281-302 on all 11,117 graphs, 100 seeds, for GNNML3 (``"graph8c"``, ne=6, ninp=2,
  supports from ``design_batch(recfield=1, dv=2, nfreq=5, adddegree=True)``) and GNNML1 (``"graph8c"``, ninp=1).  Two arms:
  - ``reference``: what the reference does -- a fresh model per seed, ``dds.collate`` + a ``no_grad`` forward per 100-graph
    batch, and ``cdist > 1e-3`` chunks of 2048 rows OR-ed into an ``n x n`` bool;
  - ``library``: ``isomorphism.isomorphism_test`` (one captured evaluator, models reloaded in place, the pair bitmap).
  Wall time per seed and in total; the per-seed counts of both arms, which must be identical (any difference is listed);
* ``pair_step``: the pair step alone at n = 11,117, 65,536 and 131,072 with d = 10 (random normal embeddings, which separate
  every pair): ``PairTracker.update`` + ``count`` on a fresh bitmap and on a full one (the skip rule), against one cdist-chunk
  step into an ``n x n`` bool (fresh), in CUDA-event milliseconds;
* the card's name and power limit, read in the same run.

    python tools/bench_isomorphism.py [--seeds 100] [--out FILE]

Nothing is written unless --out is given.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

THR = 1e-3


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                   # pragma: no cover
        q = "unavailable (%s)" % e
    return dict(name=name, power_limit_and_max_sm_clock=q)


def graph8c_datasets(dev):
    """graph8c as resident datasets: GNNML3's (designed supports, x = [1 | degree]) and GNNML1's (plain edge lists)."""
    from gnn_matlang_b200.datasets import read_graph6
    from gnn_matlang_b200.libs.utils import SpectralDesign
    from gnn_matlang_b200.synthetic import DeviceDataset
    recs = read_graph6(os.path.join(ROOT, "tests", "golden", "graph8c.g6"))
    ns = np.array([r["x"].shape[0] for r in recs], np.int64)
    es = np.array([r["edge_index"].shape[1] for r in recs], np.int64)
    node_ptr, edge_ptr = np.concatenate([[0], np.cumsum(ns)]), np.concatenate([[0], np.cumsum(es)])
    ei = torch.from_numpy(np.concatenate([r["edge_index"] for r in recs], 1)).to(dev)
    sd = SpectralDesign(recfield=1, dv=2, nfreq=5, adddegree=True)
    design = sd.design_batch(ei, torch.from_numpy(edge_ptr).to(dev), torch.from_numpy(node_ptr), device=dev)
    x = torch.cat([torch.ones(int(node_ptr[-1]), 1, device=dev), design["degree"].unsqueeze(-1)], 1)
    return DeviceDataset.from_design(design, node_ptr, x), DeviceDataset.from_graphs(recs, dev)


def cdist_step(emb, seen):
    """The reference's pair step: OR ``cdist > thr`` in 2048-row chunks into the n x n bool."""
    for r in range(0, emb.size(0), 2048):
        seen[r:r + 2048] |= torch.cdist(emb[r:r + 2048], emb, p=1) > THR


def reference_arm(make_model, dds, seeds, dev):
    G = len(dds.n_h)
    idx = [torch.arange(s, min(s + 100, G)).pin_memory() for s in range(0, G, 100)]
    seen = torch.zeros(G, G, dtype=torch.bool, device=dev)
    upper = torch.ones(G, G, dtype=torch.bool, device=dev).triu_(1)
    counts, per_seed = [], []
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for seed in seeds:
        ts = time.perf_counter()
        torch.manual_seed(seed)
        model = make_model().to(dev).eval()
        with torch.no_grad():
            emb = torch.cat([model(dds.collate(ix)) for ix in idx])
        cdist_step(emb, seen)
        counts.append(int((~seen & upper).sum()))
        per_seed.append((time.perf_counter() - ts) * 1e3)
    total = (time.perf_counter() - t0) * 1e3
    return counts, total, per_seed


def library_arm(make_model, dds, seeds):
    from gnn_matlang_b200.isomorphism import isomorphism_test
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = isomorphism_test(make_model, dds, seeds=seeds, batch_size=100)
    total = (time.perf_counter() - t0) * 1e3
    return res["counts"], total


def protocol(dev, seeds):
    from gnn_matlang_b200.models import GNNML1, GNNML3
    dds3, dds1 = graph8c_datasets(dev)
    out = {}
    for name, make, dds in (("GNNML3", lambda: GNNML3("graph8c", ne=6, ninp=2), dds3),
                            ("GNNML1", lambda: GNNML1("graph8c", ninp=1), dds1)):
        library_arm(make, dds, seeds[:2])                     # warm-up: module loads, allocator, capture
        ref_counts, ref_ms, ref_per_seed = reference_arm(make, dds, seeds, dev)
        lib_counts, lib_ms = library_arm(make, dds, seeds)
        diff = [dict(seed=s, reference=a, library=b) for s, a, b in zip(seeds, ref_counts, lib_counts) if a != b]
        out[name] = {"graphs": len(dds.n_h), "seeds": len(seeds), "counts_identical": ref_counts == lib_counts,
                     "count_differences": diff, "counts_library": lib_counts,
                     "reference_total_ms": ref_ms, "library_total_ms": lib_ms,
                     "reference_ms_per_seed": ref_ms / len(seeds), "library_ms_per_seed": lib_ms / len(seeds),
                     "reference_first_seed_ms": ref_per_seed[0], "speedup": ref_ms / lib_ms}
        if diff:
            print("%s: per-seed counts differ: %s" % (name, diff), file=sys.stderr)
    return out


def _events(fn, reps, before=None):
    ts = []
    for _ in range(reps):
        if before is not None:
            before()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def pair_step(dev, sizes, reps):
    from gnn_matlang_b200.isomorphism import PairTracker
    out = []
    for n in sizes:
        g = torch.Generator(device=dev).manual_seed(n)
        emb = torch.randn(n, 10, generator=g, device=dev)
        tr = PairTracker(n, dev)
        cnt = torch.zeros((), dtype=torch.int64, device=dev)

        def step():
            tr.update(emb)
            tr.count(out=cnt)
        step()
        fresh = _events(step, reps, before=tr.reset)
        full = _events(step, reps)                            # the bitmap is full after the first update
        undist = int(cnt)
        seen = torch.zeros(n, n, dtype=torch.bool, device=dev)

        def ref():
            cdist_step(emb, seen)
            return (~seen).sum()
        ref()
        ref_ms = _events(ref, 2 if n > 20000 else reps, before=seen.zero_)
        ref_undist = (int((~seen).sum()) - n) // 2
        del seen
        torch.cuda.empty_cache()
        out.append({"n": n, "d": 10, "bitmap_MB": tr.bits.numel() * 4 / 1e6, "update_count_fresh_ms": fresh,
                    "update_count_full_ms": full, "cdist_step_ms": ref_ms, "cdist_bool_MB": n * n / 1e6,
                    "undistinguished": undist, "undistinguished_cdist": ref_undist})
        del tr
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seeds", type=int, default=100)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--sizes", default="11117,65536,131072")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_isomorphism.py measures on a CUDA device; none is visible")
    from gnn_matlang_b200 import _lib
    from gnn_matlang_b200.graph import set_range_check
    _lib.load()
    set_range_check(False)
    dev = torch.device("cuda:0")
    res = {"bench": "bench_isomorphism", "card": card()}
    res["graph8c"] = protocol(dev, list(range(args.seeds)))
    res["pair_step"] = pair_step(dev, [int(s) for s in args.sizes.split(",")], args.reps)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
