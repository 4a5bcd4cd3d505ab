#!/usr/bin/env python
"""bench_gnnml1.py -- GNNML1 (the paper's 1-WL model) on one B200.  Prints ONE JSON line with

* the training step (forward, L1-sum loss, backward, Adam) of the GNNML1 ``zinc`` preset on a batch of ZINC-shaped graphs
  (``synthetic.zinc_graph``; 8192 by default), with the fused GNNML1 layers of this library;
* in the same process, alternating with it, the same model as a user would compose it today: this package's
  ``SpectConv(K=1, selfconn=False)`` on a ``ones[E, 1]`` edge weight plus three ``torch.nn.Linear`` and torch elementwise ops;
* the largest deviation between the two paths' losses and gradients on that batch (same weights);
* CUDA-event times of one ``gnnml3_ml1layer_forward`` / ``_backward`` call at the layer-2 shape (64 -> 64) and, from a separate
  ``torch.profiler`` pass, the device time of the fused kernel in the forward and in the dx pass, with the algorithmic bytes of
  each launch (every operand once) and their share of the 7.7 TB/s HBM3e bandwidth of one B200 (NVIDIA HGX B200 data sheet);
* the time to embed all 11,117 graph8c graphs (one batch, eval mode);
* the training data path (key ``train``): the same step captured in one CUDA graph (``GraphedTrainer``), each step collating a
  new id list on the device from an HBM-resident ``DeviceDataset(supports=False)`` of ``--pool`` graphs (larger than the
  126 MB L2); the captured step fed end to end by ``HostFeeder`` from pinned wire-format batches with the loss read back; the
  eager step on fresh batches (so that both arms build the CSR); captured against eager at batch 64; the host's
  ``collate(adjacency=True)`` (the feed without this data path) at both batch sizes; one ``gnnml3_collate_graphs`` call at the
  bench batch with its algorithmic bytes;
* the precision modes (key ``precision``): for each of ``fp32`` (3xTF32), ``tf32`` and ``bf16`` the captured ``zinc`` training
  step at the bench batch from the resident ``DeviceDataset``, the ``no_grad`` forward of the bench batch, one layer call and
  the fused kernel at 64 -> 64 (forward and dx), and the largest deviation of loss, outputs and gradients from the fp32 run on
  the same batch and weights; the arms alternate within every round;
* the card's name and power limit, read in the same run.

    python tools/bench_gnnml1.py [--batch 8192] [--steps 20] [--warmup 5] [--rounds 3] [--pool 65536] [--out FILE]

Nothing is written unless --out is given.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_PEAK = 7.7e12        # bytes/s, one B200 (HGX B200 data sheet)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                   # pragma: no cover
        q = "unavailable (%s)" % e
    return dict(name=name, power_limit_and_max_sm_clock=q)


def zinc_batch(B, seed):
    from gnn_matlang_b200.batch import collate
    from gnn_matlang_b200.synthetic import zinc_graph
    rng = np.random.default_rng(seed)
    gs = []
    for _ in range(B):
        n, ei, x = zinc_graph(rng)
        gs.append(dict(x=x, edge_index=ei, y=np.float32(rng.standard_normal())))
    return collate(gs, adjacency=True)


class ComposedGNNML1(nn.Module):
    """GNNML1 as a user writes it without the fused layer: SpectConv on ones[E, 1], three nn.Linear (cuBLAS), torch glue.
    Same parameter names as models.GNNML1, so one state_dict serves both."""

    def __init__(self, ref):
        super().__init__()
        from gnn_matlang_b200.libs.spect_conv import SpectConv
        self.cfg, self.nlayer = ref.cfg, ref.nlayer
        for l in range(1, ref.nlayer + 1):
            c = getattr(ref, "conv%d1" % l)
            setattr(self, "conv%d1" % l, SpectConv(c.in_channels, c.out_channels, 1, selfconn=False))
            for j in (1, 2, 3):
                fc = getattr(ref, "fc%d%d" % (l, j))
                setattr(self, "fc%d%d" % (l, j), nn.Linear(fc.in_features, fc.out_features))
        self.fc1 = nn.Linear(ref.fc1.in_features, ref.fc1.out_features)
        self.fc2 = nn.Linear(ref.fc2.in_features, ref.fc2.out_features)
        self.load_state_dict(ref.state_dict())

    def forward(self, data):
        from gnn_matlang_b200.pool import global_add_pool
        x, ei = data.x, data.edge_index
        ones = torch.ones(ei.size(1), 1, device=x.device)
        for l in range(1, self.nlayer + 1):
            x = F.relu(getattr(self, "fc%d1" % l)(x) + getattr(self, "conv%d1" % l)(x, ei, ones)
                       + getattr(self, "fc%d2" % l)(x) * getattr(self, "fc%d3" % l)(x))
        x = global_add_pool(x, data.batch, data.num_graphs)
        return self.fc2(F.relu(self.fc1(x)))


def timed_steps(model, opt, b, steps):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(steps):
        opt.zero_grad(set_to_none=True)
        loss = (model(b).view(-1) - b.y.view(-1)).abs().sum()
        loss.backward()
        opt.step()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / steps


def _events(fn, steps):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for i in range(steps):
        fn(i)
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / steps


def _strip(hb):
    return hb.__class__(**{k: v for k, v in hb.__dict__.items() if k not in ("edge_index2", "edge_attr2")})


def kernel_us(fn, reps=20):
    """Device time per call of each ml1 kernel that ``fn`` launches (torch.profiler), microseconds."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for evt in prof.key_averages():
        if evt.device_type.name == "CUDA" and "ml1" in evt.key:
            t = getattr(evt, "device_time_total", None) or getattr(evt, "cuda_time_total", 0)
            out[evt.key.split("(")[0].split("<")[0]] = t / max(evt.count, 1)
    return out


def precision_path(a, d, b):
    """GNNML1 in its three precisions on the same batch ``b``, weights and id lists; arms alternate within every round."""
    from gnn_matlang_b200 import ops
    from gnn_matlang_b200.graph import get_plan
    from gnn_matlang_b200.libs.spect_conv import _PRECISIONS
    from gnn_matlang_b200.models import GNNML1
    from gnn_matlang_b200.synthetic import DeviceDataset, GraphPool
    from gnn_matlang_b200.train import GraphedTrainer, pad_batch, padded_shapes
    precs = ("fp32", "tf32", "bf16")
    out = {"modes": {p: {} for p in precs}}
    # deviation from fp32: one forward + L1-sum loss + backward per mode, identical weights, before any update
    ref = {}
    for p in precs:
        torch.manual_seed(0)
        m = GNNML1("zinc", ninp=25, precision=p).to(d)
        o = m(b)
        loss = (o.view(-1) - b.y.view(-1)).abs().sum()
        loss.backward()
        r = dict(loss=loss.detach().double(), out=o.detach().double(), grads={k: v.grad.double() for k, v in m.named_parameters()})
        if p == "fp32":
            ref = r
        dev_g = {k: float((g - ref["grads"][k]).abs().max() / ref["grads"][k].abs().max().clamp_min(1e-30)) for k, g in r["grads"].items()}
        out["modes"][p].update(
            loss=float(r["loss"]), loss_rel_dev_vs_fp32=float((r["loss"] - ref["loss"]).abs() / ref["loss"].abs()),
            out_max_rel_dev_vs_fp32=float((r["out"] - ref["out"]).abs().max() / ref["out"].abs().max()),
            grad_max_rel_dev_vs_fp32=max(dev_g.values()), grad_max_rel_dev_param=max(dev_g, key=dev_g.get))
    pool = GraphPool("zinc", a.pool, seed=11)
    dds = DeviceDataset(pool, d, adjacency=True, supports=False)
    rng = np.random.default_rng(2)
    ids = [rng.integers(0, a.pool, a.batch) for _ in range(8)]
    host = [_strip(pool.collate(i, adjacency=True)) for i in ids[:2]]
    Np, _, Mp = padded_shapes([_strip(pool.collate(i, adjacency=True)) for i in ids], adjacency=True)
    pinned = [torch.from_numpy(i).pin_memory() for i in ids]
    N = int(b.x.shape[0])
    plan = get_plan(b.edge_index, N)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(N, 64, generator=g).to(d)
    gy = torch.randn(N, 64, generator=g).to(d)
    arms, calls = {}, {}
    for p in precs:
        torch.manual_seed(0)
        gt = GraphedTrainer(GNNML1("zinc", ninp=25, precision=p).to(d), pad_batch(host[0], Np, None, Mp), loss="l1")
        arms["captured_step_" + p] = lambda i, gt=gt: (gt.load_from_dataset(dds, pinned[i % len(pinned)]), gt.step())
        torch.manual_seed(0)
        m = GNNML1("zinc", ninp=25, precision=p).to(d)

        def fwd_nograd(i, m=m):
            with torch.no_grad():
                m(b)
        arms["no_grad_forward_" + p] = fwd_nograd
        L = m.conv21, m.fc21, m.fc22, m.fc23
        w = [l.weight.detach() for l in L]
        bs = [l.bias.detach() for l in L]
        pr = _PRECISIONS[p]
        y, aux, _ = ops.ml1layer_forward(plan, x, w[0], bs[0], w[1], bs[1], w[2], bs[2], w[3], bs[3], precision=pr)
        calls["fwd_" + p] = lambda w=w, bs=bs, pr=pr: ops.ml1layer_forward(plan, x, w[0], bs[0], w[1], bs[1], w[2], bs[2], w[3], bs[3],
                                                                           precision=pr)
        calls["bwd_" + p] = lambda w=w, y=y, aux=aux, pr=pr: ops.ml1layer_backward(plan, x, w[0], w[1], w[2], w[3], y, aux, gy, True,
                                                                                   precision=pr)
        arms["layer_forward_call_" + p] = lambda i, f=calls["fwd_" + p]: f()
        arms["layer_backward_call_" + p] = lambda i, f=calls["bwd_" + p]: f()
    for name, fn in arms.items():
        for i in range(a.warmup):
            fn(i)
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(a.rounds):
        for name, fn in arms.items():
            times[name].append(_events(fn, a.steps))
    for p in precs:
        r = out["modes"][p]
        r["ms_per_step"] = {k[:-len(p) - 1]: v for k, v in times.items() if k.endswith("_" + p)}
        best = {k: min(v) for k, v in r["ms_per_step"].items()}
        r["graphs_per_s_captured"] = a.batch / (best["captured_step"] * 1e-3)
        r["graphs_per_s_no_grad_forward"] = a.batch / (best["no_grad_forward"] * 1e-3)
        r["layer_forward_call_ms"], r["layer_backward_call_ms"] = best["layer_forward_call"], best["layer_backward_call"]
        kf, kb = kernel_us(calls["fwd_" + p]), kernel_us(calls["bwd_" + p])
        r["forward_kernel_us"] = next(v for k, v in kf.items() if "agg_proj" in k)
        r["dx_kernel_us"] = next(v for k, v in kb.items() if "agg_proj" in k)
        r["forward_call_kernels_us"], r["backward_call_kernels_us"] = kf, kb
    f32 = out["modes"]["fp32"]
    for p in ("tf32", "bf16"):
        r = out["modes"][p]
        r["captured_step_speedup_vs_fp32"] = min(f32["ms_per_step"]["captured_step"]) / min(r["ms_per_step"]["captured_step"])
        r["no_grad_forward_speedup_vs_fp32"] = min(f32["ms_per_step"]["no_grad_forward"]) / min(r["ms_per_step"]["no_grad_forward"])
        r["forward_kernel_speedup_vs_fp32"] = f32["forward_kernel_us"] / r["forward_kernel_us"]
        r["dx_kernel_speedup_vs_fp32"] = f32["dx_kernel_us"] / r["dx_kernel_us"]
    out.update(batch_graphs=a.batch, nodes=N, edges=int(b.edge_index.shape[1]), pool_graphs=a.pool, layer_shape="64 -> 64, sum mode",
               note=("captured_step: load_from_dataset + graph replay of the zinc preset (L1 loss, Adam); no_grad_forward: the bench "
                     "batch; ms_per_step and layer_*_call: CUDA events around the timed calls; *_kernel_us and *_call_kernels_us: "
                     "k_ml1_agg_proj (and the call's other ml1 kernels) device time per launch from a separate torch.profiler pass, "
                     "not CUDA events; deviations: one forward + backward per mode on the bench batch, same weights"))
    return out


def train_path(a, d):
    """GNNML1 training through the device data path; every arm alternates with the others in each of ``a.rounds`` rounds."""
    import time
    from gnn_matlang_b200 import ops
    from gnn_matlang_b200.batch import collate
    from gnn_matlang_b200.models import GNNML1
    from gnn_matlang_b200.synthetic import DeviceDataset, GraphPool
    from gnn_matlang_b200.train import GraphedTrainer, HostFeeder, Trainer, pad_batch, padded_shapes
    out = {}
    pool = GraphPool("zinc", a.pool, seed=11)
    dds = DeviceDataset(pool, d, adjacency=True, supports=False)
    out["pool_graphs"] = a.pool
    out["pool_resident_bytes"] = int(sum(t.numel() * t.element_size() for t in (dds.x, dds.al, dds.n, dds.m32, dds.node_off,
                                                                                 dds.adj_off, dds.y)))
    rng = np.random.default_rng(2)
    arms = {}
    for B in (a.batch, 64):
        nring = 8
        ids = [rng.integers(0, a.pool, B) for _ in range(nring)]
        host = [_strip(pool.collate(i, adjacency=True)) for i in ids]
        Np, _, Mp = padded_shapes(host, adjacency=True)
        torch.manual_seed(0)
        gt = GraphedTrainer(GNNML1("zinc", ninp=25).to(d), pad_batch(host[0], Np, None, Mp), loss="l1")
        pinned = [torch.from_numpy(i).pin_memory() for i in ids]
        torch.manual_seed(0)
        eager_model = GNNML1("zinc", ninp=25).to(d)
        eager = Trainer(eager_model, loss="l1")
        dev_batches = [hb.to(d) for hb in host]
        arms["captured_b%d" % B] = lambda i, gt=gt, pinned=pinned: (gt.load_from_dataset(dds, pinned[i % len(pinned)]), gt.step())
        arms["eager_b%d" % B] = lambda i, eager=eager, dev_batches=dev_batches: eager.step(dev_batches[i % len(dev_batches)].fresh())
        if B == a.batch:
            feeder = HostFeeder(d, onehot_widths=(21, 4))
            out["wire_bytes_per_step"] = int(np.mean([feeder.bytes_per_batch(hb) for hb in host]))
            out["host_batch_bytes_per_step"] = int(np.mean([hb.nbytes() for hb in host]))
            state = {"k": 0}
            feeder.prefetch(host[0])

            def e2e(i, gt=gt, feeder=feeder, host=host, state=state):
                cb = feeder.get_compact()
                state["k"] += 1
                feeder.prefetch(host[state["k"] % len(host)])
                gt.load_compact(cb)
                state["loss"] = float(gt.step())             # the loss read back every step
            arms["end_to_end_b%d" % B] = e2e
            # one collation call into the captured buffers
            st = gt.static
            ix = torch.from_numpy(ids[0]).to(d)
            Nb, Mb = int(pool.n[ids[0]].sum()), int(pool.e1[ids[0]].sum())
            call = lambda i, ix=ix, st=st: ops.collate_device(dds.n32, None, None, None, B, st, idx=ix, node_off=dds.node_off, x=dds.x,  # noqa: E731
                                                              m=dds.m32, al=dds.al, adj_off=dds.adj_off)
            F = dds.x.size(1)
            coll_bytes = (B * (8 + 4 + 4 + 8 + 8)                          # ids; n, m; node and edge offsets
                          + 2 * Nb * F * 4 + Nb * 8                         # features in and out; batch vector
                          + Mb * 2 * dds.al.element_size() + Mb * 16        # local ids in, int64 global ids out
                          + (Np - Nb) * (F * 4 + 8) + (Mp - Mb) * 16        # padding
                          + (B + 2) * 4 + 2 * 3 * (B + 1) * 8)              # graph_ptr; the three scans written and read
            out["collate_kernel"] = dict(graphs=B, nodes=Nb, edges=Mb, padded_nodes=Np, padded_edges=Mp, bytes=coll_bytes)
            arms["collate_call_b%d" % B] = call
    for name, fn in arms.items():                                          # warm-up of every arm and shape
        for i in range(a.warmup):
            fn(i)
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(a.rounds):
        for name, fn in arms.items():
            times[name].append(_events(fn, a.steps if not name.startswith("collate") else 50))
    out["ms_per_step"] = times
    best = {k: min(v) for k, v in times.items()}
    Bb = a.batch
    out["graphs_per_s_captured"] = Bb / (best["captured_b%d" % Bb] * 1e-3)
    out["graphs_per_s_end_to_end"] = Bb / (best["end_to_end_b%d" % Bb] * 1e-3)
    out["graphs_per_s_eager_fresh"] = Bb / (best["eager_b%d" % Bb] * 1e-3)
    out["end_to_end_over_captured"] = best["end_to_end_b%d" % Bb] / best["captured_b%d" % Bb]
    out["captured_speedup_vs_eager_fresh"] = best["eager_b%d" % Bb] / best["captured_b%d" % Bb]
    out["captured_speedup_vs_eager_b64"] = best["eager_b64"] / best["captured_b64"]
    ck = out["collate_kernel"]
    ck["call_ms"] = best["collate_call_b%d" % Bb]
    ck["hbm_share"] = ck["bytes"] / (ck["call_ms"] * 1e-3) / HBM_PEAK
    ck["bytes_rule"] = "every operand once: ids, sizes, offsets, features in and out, local ids in, global ids out, padding, scans"
    # the feed without this data path: host collation of the records (one process, this host)
    rec_rng = np.random.default_rng(0)
    recs = []
    for _ in range(Bb):
        from gnn_matlang_b200.synthetic import zinc_graph
        n, ei, x = zinc_graph(rec_rng)
        recs.append(dict(x=x, edge_index=ei, y=np.float32(rec_rng.standard_normal())))
    hc = {}
    for B, reps in ((Bb, 3), (64, 100)):
        sub = recs[:B]
        collate(sub, adjacency=True)
        t0 = time.perf_counter()
        for _ in range(reps):
            collate(sub, adjacency=True)
        hc["b%d_ms" % B] = (time.perf_counter() - t0) / reps * 1e3
    hc["host_cpus"] = os.cpu_count()
    out["host_collate_adjacency"] = hc
    out["note"] = ("captured: load_from_dataset (id list H2D + gnnml3_collate_graphs) + graph replay; end_to_end: HostFeeder H2D of "
                   "the wire format + load_compact + replay + loss read back; eager: Trainer.step on a fresh device batch (CSR build "
                   "included); ms_per_step lists one value per round, arms alternate within every round")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8192)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--pool", type=int, default=65536)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_gnnml1.py measures the GPU: no CUDA device")
    from gnn_matlang_b200 import ops
    from gnn_matlang_b200.batch import collate
    from gnn_matlang_b200.datasets import read_graph6
    from gnn_matlang_b200.graph import get_plan
    from gnn_matlang_b200.models import GNNML1
    d = torch.device("cuda:0")
    res = dict(metric="gnnml1_zinc_train_step", card=card(), batch_graphs=a.batch)

    hb = zinc_batch(a.batch, 0)
    b = hb.to(d)
    N, E = int(b.x.shape[0]), int(b.edge_index.shape[1])
    res.update(nodes=N, edges=E)
    torch.manual_seed(0)
    fused = GNNML1("zinc", ninp=25).to(d)
    comp = ComposedGNNML1(fused).to(d)
    res["model"] = "GNNML1 zinc preset: %d layers, width %d, sum mode, add-pool, fc2(relu(fc1 -> 32)) -> 1" % (fused.nlayer, 64)

    # deviation of the two paths at this size, identical weights, before any update
    for m in (fused, comp):
        m.zero_grad(set_to_none=True)
    losses = []
    for m in (fused, comp):
        loss = (m(b).view(-1) - b.y.view(-1)).abs().sum()
        loss.backward()
        losses.append(loss.detach().double())
    gf, gc = dict(fused.named_parameters()), dict(comp.named_parameters())
    dev_rel = {k: float((gf[k].grad.double() - gc[k].grad.double()).abs().max() / gc[k].grad.double().abs().max().clamp_min(1e-30))
               for k in gf}
    res["loss_fused"], res["loss_composed"] = float(losses[0]), float(losses[1])
    res["loss_rel_dev"] = float((losses[0] - losses[1]).abs() / losses[1].abs())
    res["grad_max_rel_dev"] = max(dev_rel.values())
    res["grad_max_rel_dev_param"] = max(dev_rel, key=dev_rel.get)

    of = torch.optim.Adam(fused.parameters(), lr=1e-3)
    oc = torch.optim.Adam(comp.parameters(), lr=1e-3)
    timed_steps(fused, of, b, a.warmup)
    timed_steps(comp, oc, b, a.warmup)
    tf, tc = [], []
    for _ in range(a.rounds):
        tf.append(timed_steps(fused, of, b, a.steps))
        tc.append(timed_steps(comp, oc, b, a.steps))
    res["ms_per_step_fused"] = tf
    res["ms_per_step_composed"] = tc
    res["graphs_per_s_fused"] = a.batch / (min(tf) * 1e-3)
    res["graphs_per_s_composed"] = a.batch / (min(tc) * 1e-3)
    res["speedup_vs_composed"] = min(tc) / min(tf)

    # the layer entry points at the layer-2 shape (64 -> 64, sum mode)
    plan = get_plan(b.edge_index, N)
    g = torch.Generator().manual_seed(1)
    Fi = Fo = 64
    x = torch.randn(N, Fi, generator=g).to(d)
    L = fused.conv21, fused.fc21, fused.fc22, fused.fc23
    w = [L[0].weight.detach(), L[1].weight.detach(), L[2].weight.detach(), L[3].weight.detach()]
    bs = [L[0].bias.detach(), L[1].bias.detach(), L[2].bias.detach(), L[3].bias.detach()]
    fwd = lambda: ops.ml1layer_forward(plan, x, w[0], bs[0], w[1], bs[1], w[2], bs[2], w[3], bs[3])   # noqa: E731
    y, aux, _ = fwd()
    gy = torch.randn(N, Fo, generator=g).to(d)
    bwd = lambda: ops.ml1layer_backward(plan, x, w[0], w[1], w[2], w[3], y, aux, gy, True)            # noqa: E731

    def ev(fn, reps=50):
        for _ in range(5):
            fn()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(reps):
            fn()
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e) / reps

    res["layer_forward_call_ms"] = ev(fwd)
    res["layer_backward_call_ms"] = ev(bwd)

    kf, kb = kernel_us(fwd), kernel_us(bwd)
    fk = next(v for k, v in kf.items() if "agg_proj" in k)
    bk = next(v for k, v in kb.items() if "agg_proj" in k)
    bytes_f = 4.0 * (N * Fi + E + (N + 1) + 4 * Fi * Fo + 4 * Fo + N * Fo + N * 2 * Fo)
    bytes_b = 4.0 * (N * 3 * Fo + N * Fo + E + (N + 1) + 4 * Fi * Fo + N * Fi + N * Fo)
    res["kernels_layer2"] = dict(
        forward_kernel_us=fk, forward_bytes=bytes_f, forward_hbm_share=bytes_f / (fk * 1e-6) / HBM_PEAK,
        dx_kernel_us=bk, dx_bytes=bytes_b, dx_hbm_share=bytes_b / (bk * 1e-6) / HBM_PEAK,
        forward_call_kernels_us=kf, backward_call_kernels_us=kb,
        hbm_peak="7.7 TB/s HBM3e, one B200 (HGX B200 data sheet)",
        bytes_rule="every operand once: x, CSR, weights, outputs (forward: y and aux; dx: G, gc, dx and the A^T gc side output)")

    # embedding all of graph8c
    gs = read_graph6(os.path.join(ROOT, "tests", "golden", "graph8c.g6"))
    g8 = collate(gs, adjacency=True).to(d)
    torch.manual_seed(0)
    m8 = GNNML1("graph8c", ninp=1).to(d).eval()
    with torch.no_grad():
        res["graph8c_graphs"] = len(gs)
        res["graph8c_embed_ms"] = ev(lambda: m8(g8), reps=20)
    res["train"] = train_path(a, d)
    res["precision"] = precision_path(a, d, b)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
