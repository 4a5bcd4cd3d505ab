#!/usr/bin/env python
"""bench.py -- GNNML3 training throughput (graphs/s) on dataset-shaped graphs, one process per GPU.

    python bench.py --gpus 1 --steps K --warmup W                      (this framework, default)
    python bench.py --impl reference --gpus N --steps K --warmup W     (the reference's CPU path: oracle port)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one optimisation step (CSR build for the new batch, forward, SUM loss, backward, gradient all-reduce when
N > 1, Adam) of the reference's GNNML3 model for the workload on one batch of `--batch` graphs per GPU.  Default workload:
the Zinc12k.py model on ZINC-shaped graphs with REAL SpectralDesign supports (BASELINE.json configs[1]).  Prints ONE JSON
line; at N = 1 it also carries bounded runs of the other BASELINE.json configurations (`other_configs`): the model at the
reference's own batch size, counting at batch 128, EXP with the supports rebuilt on the GPU every step, and the SpectConv
scale sweep (second headline metric).
"""
import argparse
import csv
import json
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (pool kind, model config, loss, default per-GPU batch, reference script, reference batch size)
    "zinc": ("zinc", "zinc", "l1", 8192, "Zinc12k.py GNNML3 (4 x ML3Layer 30||2, K=8, add-pool, L1-sum, Adam 1e-3)", 64),
    "counting": ("counting", "counting", "mse", 8192, "counting.py GNNML3 (5 x ML3Layer 16||16, K=12, add-pool, MSE-sum, Adam 1e-3)", 10),
    "exp": ("exp", "exp", "bce", 4096, "exp_classify.py GNNML3 (3 x ML3Layer 32||16, K=6, mean-pool, BCE-sum, Adam 1e-3), "
            "SpectralDesign(recfield=1, dv=2, nfreq=5, adddegree) rebuilt on the GPU every step", 50),
}
LAUNCH_PROFILE = os.path.join(ROOT, "profiles", "r02_ncu_launches_zinc_one_step_final.csv")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="zinc", choices=sorted(WORKLOADS) + ["spectconv_sweep"],
                    help="zinc (default, BASELINE.json configs[1]) / counting / exp: GNNML3 training; spectconv_sweep: one SpectConv "
                         "layer fwd+bwd on a 1M-node batch (BASELINE.json configs[4]), reported as HBM GB/s")
    ap.add_argument("--sweep-nodes", type=int, default=1000000)
    ap.add_argument("--sweep-f", type=int, default=64)
    ap.add_argument("--sweep-hops", type=int, default=1, choices=[1, 2])
    ap.add_argument("--batch", type=int, default=0, help="graphs per GPU per step (0 = workload default)")
    ap.add_argument("--pool", type=int, default=2048, help="distinct synthetic graphs in the pool")
    ap.add_argument("--ring", type=int, default=6, help="distinct resident batches cycled through (> L2 in total)")
    ap.add_argument("--precision", default="fp32", choices=["fp32", "tf32", "bf16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--placeholder-supports", action="store_true", help="N(0,1) edge features instead of SpectralDesign supports")
    ap.add_argument("--no-cuda-graph", action="store_true", help="enqueue every step's ~120 launches from the host instead of replaying "
                                                                  "the captured step")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the loss of the last timed step, the gradients "
                                                          "it computed and the parameters it left as DIR/<name>.npy (float32), to "
                                                          "compare two builds on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload == "spectconv_sweep"):
        ap.error("--dump-outputs applies to the training workloads of --impl b200")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, model, loss):
    """What a caller of the timed training step holds after its last step: the loss (loss.npy), every parameter's gradient
    (grad.<name>.npy) and every parameter after the Adam update (param.<name>.npy)."""
    arrays = {"loss": loss}
    for name, p in model.named_parameters():
        if p.grad is not None:
            arrays["grad." + name] = p.grad
        arrays["param." + name] = p
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML during the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def common_config(workload, B, desc, edge_attr):
    """The part of `config` both arms (this framework and --impl reference) share verbatim."""
    return {"workload": workload, "reference_script": desc, "graphs_per_step_per_process": int(B), "edge_attr": edge_attr,
            "timed_step": "fwd + SUM loss + bwd + Adam on one batch (b200: + CSR build of the new batch, + all-reduce when N > 1)"}


def oracle_supports(pool):
    """The reference's own SpectralDesign (oracle restatement, numpy, one graph at a time) over a GraphPool: the CPU arm's
    edge features."""
    from oracle import gnnml3_oracle as O
    cfg = dict(pool.SPECTRAL_CONFIGS[pool.kind])
    cfg["recfield"] = pool.recfield
    eas = []
    for g in range(len(pool.n)):
        ei = pool.ei1[:, pool.edge_off1[g]:pool.edge_off1[g + 1]]
        with np.errstate(all="ignore"):
            d = O.spectral_design(ei, np.zeros((int(pool.n[g]), 1), np.float32), **cfg)
        assert np.array_equal(d["edge_index2"], pool.ei2[:, pool.edge_off[g]:pool.edge_off[g + 1]])
        eas.append(d["edge_attr2"])
    pool.set_supports(np.concatenate(eas, 0))


def run_reference(args, rank, world):
    """The reference's CPU implementation of the path (oracle port of libs/spect_conv.py + the script's model and training
    step; for `exp` also its numpy SpectralDesign loop per batch), all host threads, same graphs per step as the b200 arm."""
    if rank != 0:
        return
    from oracle import gnnml3_oracle as O
    from gnn_matlang_b200.synthetic import ExpPool, GraphPool
    from gnn_matlang_b200.train import loss_fn
    kind, cfg, loss, defB, desc, _ = WORKLOADS[args.workload]
    torch.set_num_threads(os.cpu_count() or 1)
    B = args.batch or defB
    rng = np.random.default_rng(0)
    torch.manual_seed(0)
    if kind == "exp":
        pool = ExpPool()
        raws = [pool.draw_raw(rng, B) for _ in range(2)]

        def make(raw):
            graphs = []
            npt, ept = raw["node_ptr"].numpy(), raw["edge_ptr"].numpy()
            for b in range(B):
                with np.errstate(all="ignore"):
                    d = O.spectral_design(raw["edge_index"][:, ept[b]:ept[b + 1]].numpy(), raw["x"][npt[b]:npt[b + 1]].numpy(),
                                          recfield=1, dv=2, nfreq=5, adddegree=True)
                graphs.append(d)
            ob = O.collate(graphs)
            ob["y"] = raw["y"]
            return ob
        edge_attr = "spectral_design (reference numpy loop, rebuilt every step)"
    else:
        pool = GraphPool(kind, min(args.pool, 512), seed=0)
        if not args.placeholder_supports:
            oracle_supports(pool)
        hbs = [pool.draw(rng, B) for _ in range(2)]
        raws = [dict(x=hb.x, edge_index2=hb.edge_index2, edge_attr2=hb.edge_attr2, batch=hb.batch, num_graphs=hb.num_graphs, y=hb.y)
                for hb in hbs]

        def make(ob):
            return ob
        edge_attr = "spectral_design" if not args.placeholder_supports else "normal"
    model = O.OracleGNNML3(cfg, pool.K, pool.F)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)

    def step(raw):
        ob = make(raw)
        opt.zero_grad()
        l = loss_fn(loss, model(ob), ob["y"])
        l.backward()
        opt.step()
        return float(l)

    for i in range(args.warmup):
        step(raws[i % 2])
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(raws[i % 2])
    dt = time.perf_counter() - t0
    v = B * args.steps / dt
    print(json.dumps({
        "impl": "reference", "metric": "GNNML3 train graphs/s", "value": v, "unit": "graphs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": common_config(args.workload, B, desc, edge_attr),
        "cpu_baseline": {"value": v, "unit": "graphs/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": "%d steps of %d %s-shaped graphs, oracle port of the reference's PyG path on host CPU" % (args.steps, B, args.workload)},
        "e2e": {"value": v, "unit": "graphs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def sweep_one(dev, F, K, nodes, hops, steps, warmup):
    """SpectConv F -> F forward + backward on a `nodes`-node batch of 30-100-node graphs (BASELINE.json configs[4]).
    achieved = SURVEY.md 8d algorithmic bytes (fwd + bwd, every operand once, the [N, K*F] aggregate never credited) / time."""
    from gnn_matlang_b200 import ops
    from gnn_matlang_b200.graph import get_plan
    from gnn_matlang_b200.libs.spect_conv import SpectConv
    from gnn_matlang_b200.synthetic import GraphPool
    pool = GraphPool("sweep", 1024, seed=1, K=K, nfeat=4, recfield=hops)
    rng = np.random.default_rng(3)
    B = int(nodes / float(pool.n.mean()))
    hb = pool.draw(rng, B)
    N, E = hb.x.shape[0], hb.edge_index2.shape[1]
    torch.manual_seed(0)
    layer = SpectConv(F, F, K, selfconn=False).to(dev)
    ei = hb.edge_index2.to(dev)
    ea = hb.edge_attr2.to(dev).requires_grad_(True)
    nx = max(2, int(np.ceil(300e6 / (N * F * 4.0))))                   # distinct inputs: > 126 MB L2 in total
    xs = [torch.randn(N, F, device=dev).requires_grad_(True) for _ in range(nx)]
    gout = torch.randn(N, F, device=dev)
    get_plan(ei, N)

    def step(i):
        x = xs[i % len(xs)]
        out = layer(x, ei, ea)
        out.backward(gout)
        x.grad = None
        ea.grad = None
        layer.zero_grad(set_to_none=True)

    for i in range(warmup):
        step(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ops.fused_path_counts(reset=True)
    e0.record()
    for i in range(steps):
        step(i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    paths = ops.fused_path_counts()
    fwd = 4.0 * (N * F + E * K + E + (N + 1) + K * F * F + F + N * F)
    bwd = 4.0 * (N * F + N * F + E * K + 2 * E + (N + 1) + N * F + E * K + 2 * K * F * F + F)
    flops = 2.0 * (3 * E * K * F + 3 * N * K * F * F)                 # aggregate x3 on CUDA cores + three GEMMs on tensor cores
    pk = peaks()
    hbm = float(pk.get("hbm_gbs", 6650.0))
    tf32_peak = 0.5 * float(pk.get("bf16_tflops", 1590.0))            # TF32 dense = half the measured bf16 rate (not measured itself)
    t_hbm = (fwd + bwd) / (hbm * 1e9)
    t_tc = 3.0 * 2.0 * 3 * N * K * F * F / (tf32_peak * 1e12)         # 3xTF32: three tensor-core products per FP32-grade product
    ach = (fwd + bwd) / (ms * 1e-3) / 1e9
    del xs, gout, layer
    torch.cuda.empty_cache()
    return {"F": F, "K": K, "mask": "%d-hop" % hops, "nodes": int(N), "support_entries": int(E), "graphs": int(B), "ms_fwd_bwd": ms,
            "hbm_gbs_achieved": ach, "frac_of_hbm_peak": ach / hbm, "roof_ms": {"hbm": 1e3 * t_hbm, "tensor_3xtf32": 1e3 * t_tc},
            "frac_of_binding_roof": max(t_hbm, t_tc) / (ms * 1e-3), "graphs_per_s": B / (ms * 1e-3), "useful_tflops": flops / (ms * 1e-3) / 1e12,
            "fused_launches": {"tensor_memory_kernel": paths[0], "smem_plane_kernel": paths[1]}}


def run_sweep(args, local):
    from gnn_matlang_b200 import _lib
    from gnn_matlang_b200.graph import set_range_check
    _lib.load()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    set_range_check(False)
    r = sweep_one(dev, args.sweep_f, 10, args.sweep_nodes, args.sweep_hops, args.steps, max(args.warmup, 3))
    pk = peaks()
    peak = float(pk.get("hbm_gbs", 6650.0))
    print(json.dumps({
        "metric": "SpectConv fwd+bwd HBM GB/s", "value": r["hbm_gbs_achieved"], "unit": "GB/s", "n_gpus": 1, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": r["ms_fwd_bwd"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "spectconv_sweep", "nodes": r["nodes"], "support_entries": r["support_entries"], "graphs": r["graphs"], "K": 10,
                   "F_in": r["F"], "F_out": r["F"], "mask": r["mask"], "l2_policy": "distinct inputs cycled, > 126 MB in total"},
        "roofline": {"kernel": "SpectConv layer fwd+bwd (all launches)", "bound": "hbm", "achieved": r["hbm_gbs_achieved"], "peak": peak,
                     "unit": "GB/s", "frac": r["frac_of_hbm_peak"], "traffic": None},
        "sweep": r}), flush=True)


def time_steps(trainer, batches, steps, warmup, barrier):
    """-> (device ms for `steps` steps, host enqueue ms per step, last loss tensor)."""
    for i in range(warmup):
        trainer.step(batches(i))
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    th0 = time.perf_counter()
    loss_t = None
    for i in range(steps):
        loss_t = trainer.step(batches(i))
    host_ms = (time.perf_counter() - th0) * 1e3 / steps
    e1.record()
    barrier()
    return e0.elapsed_time(e1), host_ms, loss_t


def small_config(dev, workload, B, steps, warmup, supports=True):
    """One of the other BASELINE.json configurations at its own batch size, bounded: -> dict for `other_configs`.  At these
    sizes the step is launch-bound: reported both enqueued launch by launch and as ONE captured CUDA graph replayed per step."""
    from gnn_matlang_b200.models import GNNML3
    from gnn_matlang_b200.synthetic import GraphPool
    from gnn_matlang_b200.train import GraphedTrainer, Trainer, pad_batch, padded_shapes
    kind, cfg, loss, _, desc, _ = WORKLOADS[workload]
    pool = GraphPool(kind, 512, seed=5)
    if supports:
        pool.attach_spectral_supports(dev)
    rng = np.random.default_rng(11)
    host = [pool.draw(rng, B) for _ in range(8)]
    ring = [hb.to(dev, non_blocking=False) for hb in host]
    torch.manual_seed(0)
    model = GNNML3(cfg, pool.K, pool.F).to(dev)
    trainer = Trainer(model, loss=loss, lr=1e-3)
    ms, host_ms, loss_t = time_steps(trainer, lambda i: ring[i % len(ring)].fresh(), steps, warmup, torch.cuda.synchronize)
    Np, Ep = padded_shapes(host)
    pads = [pad_batch(hb, Np, Ep).to(dev, non_blocking=False) for hb in host]
    torch.manual_seed(0)
    model2 = GNNML3(cfg, pool.K, pool.F).to(dev)
    gt = GraphedTrainer(model2, pads[0], loss=loss, lr=1e-3)
    ms_g, host_g, loss_g = time_steps(gt, lambda i: pads[i % len(pads)], steps, warmup, torch.cuda.synchronize)
    return {"reference_script": desc, "graphs_per_step": B, "steps": steps, "edge_attr": pool.supports,
            "cuda_graph": {"ms_per_step": ms_g / steps, "graphs_per_s": B * steps / (ms_g * 1e-3), "host_enqueue_ms_per_step": host_g,
                           "final_loss": float(loss_g.item())},
            "launch_by_launch": {"ms_per_step": ms / steps, "graphs_per_s": B * steps / (ms * 1e-3), "host_enqueue_ms_per_step": host_ms,
                                 "final_loss": float(loss_t.item())},
            "ms_per_step": ms_g / steps, "graphs_per_s": B * steps / (ms_g * 1e-3)}


def exp_config(dev, B, steps, warmup, cpu_sample=True, pipelined=False):
    """BASELINE.json configs[2]: EXP graphs (real, first 200 records of GRAPHSAT.pkl), supports REBUILT ON THE GPU every step
    (SpectralDesign.design_batch), then the exp_classify.py GNNML3 training step.  Also times SpectralDesign alone beside the
    reference's numpy loop on one host core (libs/utils.py:546-610; single-threaded by construction)."""
    from gnn_matlang_b200.libs.utils import SpectralDesign
    from gnn_matlang_b200.models import GNNML3
    from gnn_matlang_b200.synthetic import ExpPool, design_and_collate
    from gnn_matlang_b200.train import Trainer
    pool = ExpPool()
    sd = SpectralDesign(recfield=1, dv=2, nfreq=5, adddegree=True)
    rng = np.random.default_rng(13)
    raws = []
    for _ in range(4):
        r = pool.draw_raw(rng, B)
        raws.append({k: (v.to(dev) if (isinstance(v, torch.Tensor) and k not in ("node_ptr",)) else v) for k, v in r.items()})
    torch.manual_seed(0)
    model = GNNML3("exp", pool.K, pool.F).to(dev)
    trainer = Trainer(model, loss="bce", lr=1e-3)
    ms, host_ms, loss_t = time_steps(trainer, lambda i: design_and_collate(raws[i % len(raws)], sd, dev), steps, warmup, torch.cuda.synchronize)
    # SpectralDesign alone
    for i in range(2):
        sd.design_batch(raws[i]["edge_index"], raws[i]["edge_ptr"], raws[i]["node_ptr"], device=dev, global_ids=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        sd.design_batch(raws[i % len(raws)]["edge_index"], raws[i % len(raws)]["edge_ptr"], raws[i % len(raws)]["node_ptr"], device=dev,
                        global_ids=True)
    e1.record()
    torch.cuda.synchronize()
    sd_ms = e0.elapsed_time(e1) / steps
    # the same configuration with the design of batch i + 1 on a side stream and the training step captured in a CUDA graph
    # (static shapes: the entries of the recfield-1 mask are n + e per graph, known on the host without running the design)
    piped = None
    if pipelined:
        from gnn_matlang_b200.train import DesignFeeder, GraphedTrainer, pad_batch
        raws_p = [pool.draw_raw(rng, B) for _ in range(8)]
        n_tot = [int(r["node_ptr"][-1]) for r in raws_p]
        e_tot = [int(r["node_ptr"][-1]) + int(r["edge_ptr"][-1]) for r in raws_p]
        Np, Ep = int(max(n_tot) * 1.15) + 64, int(max(e_tot) * 1.15) + 64
        raws_p = [{k: (v.to(dev) if (isinstance(v, torch.Tensor) and k not in ("node_ptr",)) else v) for k, v in r.items()} for r in raws_p]
        example = design_and_collate(raws_p[0], sd, dev)
        ex_host = type(example)(**{k: (v.cpu() if isinstance(v, torch.Tensor) else v) for k, v in example.__dict__.items()})
        torch.manual_seed(0)
        model_p = GNNML3("exp", pool.K, pool.F).to(dev)
        gt = GraphedTrainer(model_p, pad_batch(ex_host, Np, Ep), loss="bce", lr=1e-3)
        depth = 3
        feeder = DesignFeeder(sd, dev, depth=depth)

        def run(nsteps):
            for j in range(depth):
                feeder.prefetch(raws_p[j % len(raws_p)], records=True)
            lt = None
            for i in range(nsteps):
                rec = feeder.get()
                feeder.prefetch(raws_p[(i + depth) % len(raws_p)], records=True)
                gt.load_designed(rec)
                lt = gt.step()
            while feeder.pending():
                feeder.get()
            return lt

        run(warmup)
        torch.cuda.synchronize()
        e0p, e1p = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tp0 = time.perf_counter()
        e0p.record()
        ltp = run(steps)
        e1p.record()
        hostp = (time.perf_counter() - tp0) * 1e3 / steps
        torch.cuda.synchronize()
        msp = e0p.elapsed_time(e1p)
        piped = {"ms_per_step": msp / steps, "graphs_per_s": B * steps / (msp * 1e-3), "host_ms_per_step": hostp,
                 "final_loss": float(ltp.item()),
                 "note": "SpectralDesign of batches i + 1 .. i + 3 on side streams (train.DesignFeeder) while batch i trains; the training step is "
                         "ONE captured CUDA graph on shapes padded to %d nodes / %d entries" % (Np, Ep)}
    out = {"reference_script": WORKLOADS["exp"][4], "graphs_per_step": B, "steps": steps, "ms_per_step": ms / steps,
           "graphs_per_s": B * steps / (ms * 1e-3), "host_enqueue_ms_per_step": host_ms, "final_loss": float(loss_t.item()),
           "design_overlapped_and_step_captured": piped,
           "data": "real EXP graphs (tests/golden/exp_first200.npz), drawn with replacement",
           "spectral_design": {"gpu_graphs_per_s": B / (sd_ms * 1e-3), "gpu_ms_per_batch": sd_ms,
                               "kernel": "k_sd_count + k_sd_design: one thread block per graph, FP64 Jacobi in shared memory"}}
    if cpu_sample:
        from oracle import gnnml3_oracle as O
        torch.set_num_threads(1)
        nrep, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < 3.0:
            g = nrep % len(pool.n)
            with np.errstate(all="ignore"):
                O.spectral_design(pool.ei1[:, pool.edge_off1[g]:pool.edge_off1[g + 1]], pool.x[pool.node_off[g]:pool.node_off[g + 1]],
                                  recfield=1, dv=2, nfreq=5, adddegree=True)
            nrep += 1
        dt = time.perf_counter() - t0
        torch.set_num_threads(os.cpu_count() or 1)
        out["spectral_design"]["cpu_graphs_per_s"] = nrep / dt
        out["spectral_design"]["cpu_baseline"] = {"kind": "port", "cores": 1, "sample": "%d EXP graphs through the oracle restatement of "
                                                  "libs/utils.py:546-610 (numpy eigh per graph, single-threaded by construction)" % nrep}
    return out


def graph8c_config(dev, cpu_seconds=3.0):
    """BASELINE.json configs[0]: graph8c.py:281-302 -- embed all 11,117 8-node graphs with a fresh seed-0 GNNML3 in batches of 100
    and count the pairs whose embeddings differ by less than 1e-3 in L1 (known answer after seed 0: 1 pair).  Everything on the
    GPU through the product path: graph6 reader -> SpectralDesign (one launch for the whole dataset) -> HBM-resident dataset ->
    on-device collation -> forward.  The CPU figure beside it is the oracle port on a bounded sample of the same batches."""
    from gnn_matlang_b200.datasets import read_graph6
    from gnn_matlang_b200.libs.utils import SpectralDesign
    from gnn_matlang_b200.models import GNNML3
    from gnn_matlang_b200.synthetic import DeviceDataset
    path = os.path.join(ROOT, "tests", "golden", "graph8c.g6")
    recs = read_graph6(path)
    ns = np.array([r["x"].shape[0] for r in recs], np.int64)
    es = np.array([r["edge_index"].shape[1] for r in recs], np.int64)
    node_ptr, edge_ptr = np.concatenate([[0], np.cumsum(ns)]), np.concatenate([[0], np.cumsum(es)])
    ei = torch.from_numpy(np.concatenate([r["edge_index"] for r in recs], 1))
    sd = SpectralDesign(recfield=1, dv=2, nfreq=5, adddegree=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ei_d, ep_d, np_d = ei.to(dev), torch.from_numpy(edge_ptr).to(dev), torch.from_numpy(node_ptr)
    design = sd.design_batch(ei_d, ep_d, np_d, device=dev)              # warm-up (also sizes the outputs)
    torch.cuda.synchronize()
    e0.record()
    design = sd.design_batch(ei_d, ep_d, np_d, device=dev)
    e1.record()
    torch.cuda.synchronize()
    sd_ms = e0.elapsed_time(e1)
    x = torch.cat([torch.ones(int(node_ptr[-1]), 1, device=dev), design["degree"].unsqueeze(-1)], 1)
    dds = DeviceDataset.from_design(design, node_ptr, x)
    torch.manual_seed(0)
    model = GNNML3("graph8c", ne=6, ninp=2).to(dev).eval()
    G = len(recs)
    idx = [torch.arange(s, min(s + 100, G)).pin_memory() for s in range(0, G, 100)]

    def embed_all():
        out = []
        with torch.no_grad():
            for ix in idx:
                out.append(model(dds.collate(ix)))
        return torch.cat(out)

    embed_all()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e0.record()
    emb = embed_all()
    e1.record()
    torch.cuda.synchronize()
    ms, wall = e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3
    similar = 0
    for r in range(0, G, 2048):
        similar += int((torch.cdist(emb[r:r + 2048], emb, p=1) <= 0.001).sum())
    similar = (similar - G) // 2
    out = {"reference_script": "graph8c.py:281-302 GNNML3 (3 x ML3Layer 32||16, K=6, add-pool, tanh head) isomorphism test, 11,117 graphs, batches of 100, seed 0",
           "graphs": G, "batches": len(idx), "ms_embed_all": ms, "wall_ms_embed_all": wall, "graphs_per_s": G / (ms * 1e-3),
           "undistinguished_pairs_after_seed_0": similar, "known_answer": 1,
           "spectral_design": {"gpu_ms_all_graphs": sd_ms, "gpu_graphs_per_s": G / (sd_ms * 1e-3)},
           "note": "forward only, launch by launch (112 small batches: host-enqueue bound, wall = device time)"}
    if cpu_seconds > 0:
        from oracle import gnnml3_oracle as O
        g8 = O.parse_graph6(path)
        torch.manual_seed(0)
        ref = O.OracleGNNML3("graph8c", 6, 2)
        kw = dict(recfield=1, dv=2, nfreq=5, adddegree=True)
        done, t0 = 0, time.perf_counter()
        with torch.no_grad():
            while time.perf_counter() - t0 < cpu_seconds and done < G:
                graphs = [O.spectral_design(e, np.ones((n, 1), np.float32), **kw) for n, e in g8[done:done + 100]]
                ref(O.collate(graphs))
                done += len(graphs)
        out["cpu_baseline"] = {"kind": "port", "cores": os.cpu_count(), "value": done / (time.perf_counter() - t0), "unit": "graphs/s",
                               "sample": "%d graphs: oracle SpectralDesign (numpy eigh per graph) + oracle forward in batches of 100" % done}
    return out


def ncu_shares():
    """Per-kernel shares of ONE step of the timed code path, from the committed `ncu --metrics gpu__time_duration.sum` launch
    list of the same command (cold-cache, serialised: shares, not absolutes)."""
    try:
        rows = list(csv.reader(open(LAUNCH_PROFILE)))
    except Exception:
        return None
    out = {}
    for r in rows[1:]:
        if len(r) >= 4 and r[0] != "TOTAL":
            out[r[0]] = {"launches": int(r[1]), "us": float(r[2]), "share": float(r[3])}
    return {"source": os.path.relpath(LAUNCH_PROFILE, ROOT), "kernels": dict(list(out.items())[:14])}


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.workload == "spectconv_sweep":
        if rank == 0:
            run_sweep(args, local)
        return

    import torch.distributed as dist
    from gnn_matlang_b200 import _lib, ops
    from gnn_matlang_b200.graph import set_range_check
    from gnn_matlang_b200.libs.utils import SpectralDesign
    from gnn_matlang_b200.models import GNNML3
    from gnn_matlang_b200.synthetic import ExpPool, GraphPool, design_and_collate
    from gnn_matlang_b200.train import HostFeeder, Trainer

    lib = _lib.load()                # fails loudly if the CUDA library is missing
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"      # the NCCL version banner goes to stdout; stdout carries ONE JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    kind, cfg, loss, defB, desc, refB = WORKLOADS[args.workload]
    B = args.batch or defB
    set_range_check(False)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- data: pool of graphs -> ring of distinct batches (pinned host + HBM-resident copies)
    rng = np.random.default_rng(7 + rank)
    is_exp = kind == "exp"
    if is_exp:
        pool = ExpPool()
        sd = SpectralDesign(recfield=1, dv=2, nfreq=5, adddegree=True)
        host_ring = [pool.draw_raw(rng, B) for _ in range(args.ring)]
        host_ring = [{k: (v.pin_memory() if isinstance(v, torch.Tensor) else v) for k, v in r.items()} for r in host_ring]
        dev_ring = [{k: (v.to(dev) if (isinstance(v, torch.Tensor) and k != "node_ptr") else v) for k, v in r.items()} for r in host_ring]
        batch_bytes = sum(v.numel() * v.element_size() for v in host_ring[0].values() if isinstance(v, torch.Tensor))
        N0, E0 = int(host_ring[0]["x"].shape[0]), None
        get_batch = lambda i: design_and_collate(dev_ring[i % args.ring], sd, dev)
    else:
        pool = GraphPool(kind, args.pool, seed=1000 + rank)
        if not args.placeholder_supports:
            pool.attach_spectral_supports(dev)     # real supports, designed by this library's SpectralDesign (one launch)
        host_ring = [pool.draw(rng, B).pin_memory() for _ in range(args.ring)]
        dev_ring = [hb.to(dev, non_blocking=False) for hb in host_ring]
        batch_bytes = host_ring[0].nbytes()
        N0, E0 = int(host_ring[0].x.shape[0]), int(host_ring[0].edge_index2.shape[1])
        get_batch = lambda i: dev_ring[i % args.ring].fresh()

    torch.manual_seed(0)             # identical replicas
    model = GNNML3(cfg, pool.K, pool.F, precision=args.precision).to(dev)
    use_graph = not args.no_cuda_graph and not is_exp
    from gnn_matlang_b200.train import GraphedTrainer, pad_batch, padded_shapes
    if use_graph:
        # static shapes for the captured step: every ring batch padded (neutral padding, train.pad_batch) to the ring's largest
        Np, Ep = padded_shapes(host_ring)
        pad_ring = [pad_batch(hb, Np, Ep).to(dev, non_blocking=False) for hb in host_ring]
        trainer = GraphedTrainer(model, pad_ring[0], loss=loss, lr=1e-3, distributed=world > 1)
        run_step = lambda i: trainer.step(pad_ring[i % args.ring])
        pad_note = ("step captured in ONE CUDA graph and replayed; batches padded to %d nodes / %d entries (%.1f %% / %.1f %% neutral "
                    "padding), the new batch is copied device->device into the captured buffers inside the timed region"
                    % (Np, Ep, 100.0 * (Np - N0) / Np, 100.0 * (Ep - E0) / Ep))
    else:
        trainer = Trainer(model, loss=loss, lr=1e-3, distributed=world > 1)
        run_step = lambda i: trainer.step(get_batch(i))
        pad_note = "every launch enqueued from the host (no CUDA graph)"

    # ---- warm-up
    for i in range(max(args.warmup, 3)):
        run_step(i)
    barrier()

    # ---- timed region: inputs resident in HBM; successive steps use different batches (ring > L2)
    sampler = ClockSampler(local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    th0 = time.perf_counter()
    for i in range(args.steps):
        loss_t = run_step(i)
    host_ms = (time.perf_counter() - th0) * 1e3 / args.steps      # CPU time to ENQUEUE a step (no sync inside the loop)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model, loss_t)       # before the steps below train the same model further
    final_loss = float(loss_t.item())
    sampler.stop_flag = True
    sampler.join()
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = world * B * args.steps / (ms * 1e-3)

    # ---- the same step enqueued launch by launch (identical kernels and batches; a captured graph cannot carry timing events):
    #      per-launch CUDA events around the dominant kernel for the roofline, launch count, fused-path counters
    eager = Trainer(model, loss=loss, lr=1e-3, distributed=world > 1) if use_graph else trainer
    nprof = min(args.steps, 10)
    for i in range(2):
        eager.step(get_batch(i))
    barrier()
    lib.gnnml3_fused_profile(1)          # CUDA events around every fused layer-kernel launch, on the launching stream
    ops.fused_path_counts(reset=True)
    n0 = _lib.launch_count()
    e0.record()
    th0 = time.perf_counter()
    for i in range(nprof):
        eager.step(get_batch(i))
    eager_host_ms = (time.perf_counter() - th0) * 1e3 / nprof
    e1.record()
    barrier()
    eager_ms = e0.elapsed_time(e1) / nprof
    launches = (_lib.launch_count() - n0) // nprof
    paths = ops.fused_path_counts()
    import ctypes
    pbuf = (ctypes.c_double * (10 * 4096))()
    nrec = lib.gnnml3_fused_profile_fetch(pbuf, 4096)
    lib.gnnml3_fused_profile(0)
    per_step = nrec // max(nprof, 1)
    recs = []
    for j in range(nrec):
        msj, Nn, Kk, Ff, Ncc, Fss, smode, Nss, Gg, hp = [pbuf[j * 10 + t] for t in range(10)]
        Ee = float(E0 if E0 is not None else 0)
        if not is_exp:
            Ee = float(host_ring[(j // max(per_step, 1)) % args.ring].edge_index2.shape[1])
        # algorithmic HBM bytes (SURVEY.md 8d): every operand and result once, the [N, K*F] aggregate never credited
        nbytes = 4.0 * (Nn * Ff + (Nn * Fss if smode == 2 else 0) + Ee * Kk + Ee * (2 if hp else 1) + (Nn + 1) + Kk * Ff * Ncc
                        + Fss * (Nss if smode == 1 else (Ncc if smode == 2 else 0)) + Ncc + Nn * (Ncc + (Gg if smode == 1 else 0))
                        + (Nn * 2 * Gg if smode == 1 else 0))
        recs.append((msj, nbytes, "dx" if hp else "forward"))

    # ---- roofline of the dominant kernel (the fused aggregate+project layer kernel: forward launches and the transposed
    #      dx launches of the backward)
    pk = peaks()
    peak = float(pk.get("hbm_gbs", 6650.0))
    sp_ms = sum(r[0] for r in recs)
    sp_bytes = sum(r[1] for r in recs)
    roofline = None
    if recs and sp_ms > 0 and not is_exp:
        ach = sp_bytes / (sp_ms * 1e-3) / 1e9
        traffic = None
        try:      # dram bytes per launch from the committed ncu --set full capture of the same kernel (profiles/)
            traffic = json.load(open(os.path.join(ROOT, "profiles", "r02_fused_ts_ncu_summary.json")))["dram_bytes_per_launch"]
        except Exception:
            pass
        roofline = {"kernel": "k_fused_ts (gnnml3_fused_agg_proj, tensor-memory generation: SpectConv aggregate + projection + gates, "
                              "fwd and dx launches)" if paths[0] >= paths[1] else "k_fused_agg_proj (shared-memory plane generation)",
                    "bound": "hbm", "achieved": ach, "peak": peak,
                    "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                    "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in pk else "fallback 6650",
                    "launches": len(recs), "avg_launch_ms": sp_ms / len(recs), "share_of_step": sp_ms / nprof / eager_ms,
                    "algorithmic_bytes_per_launch": sp_bytes / len(recs),
                    "by_kind": {k: {"launches": len(v), "avg_launch_ms": sum(r[0] for r in v) / len(v),
                                    "frac": sum(r[1] for r in v) / (sum(r[0] for r in v) * 1e-3) / 1e9 / peak}
                                for k, v in (("forward", [r for r in recs if r[2] == "forward"]), ("dx", [r for r in recs if r[2] == "dx"])) if v},
                    "measured_in": "%d steps of the same training step enqueued launch by launch right after the timed region (CUDA "
                                   "events on the launching stream inside gnnml3_fused_agg_proj)" % nprof,
                    "traffic_note": "mean of 4 forward launches (66 MB each: x / y stay in L2 between kernels; the first layer's also writes its "
                                    "aggregate, 218 MB, for the weight gradient) and 3 dx launches (264 MB each: they also "
                                    "write the 190 MB aggregate side output the weight-gradient contraction reads); the side outputs are not "
                                    "credited as algorithmic bytes; no re-reads",
                    "note": "latency / hand-off bound, not bandwidth bound: FP32 FMA issue of the aggregation (61 % of the lanes active over ragged "
                            "rows) + per-pass fixed cost (set-up, residuals, tcgen05.st hand-off), see DESIGN.md section 4.1"}

    # ---- end to end: pinned host batches in the compact wire format -> H2D on a copy stream (one step ahead) -> rebuilt on the
    #      device -> written into the captured buffers -> graph replay; D2H of every step's loss inside the timed region
    e2e = None
    if not args.no_e2e and not is_exp:
        feeder = HostFeeder(dev, onehot_widths=(21, 4) if kind == "zinc" else None)
        for hb in host_ring:
            feeder.compact(hb)                  # wire-format conversion = data preparation, like collation: outside the timed region
        if use_graph:
            def e2e_step(cb):                   # wire format -> captured buffers (two library launches), graph replay
                trainer.load_compact(cb)
                return trainer.step()
            fetch = feeder.get_compact
        else:
            e2e_step = trainer.step
            fetch = feeder.get
        feeder.prefetch(host_ring[0])
        for i in range(3):
            b = fetch()
            feeder.prefetch(host_ring[(i + 1) % args.ring])
            float(e2e_step(b).item())
        barrier()
        e0.record()
        # every step's loss is read back to the host: the device -> host copy is enqueued right behind the step (pinned
        # buffer, non-blocking) and harvested while the next step is being enqueued, so the read never stalls the pipeline
        loss_host = [torch.empty(1, dtype=torch.float32).pin_memory() for _ in range(2)]
        loss_ev = [torch.cuda.Event(), torch.cuda.Event()]
        lv = float("nan")
        for i in range(args.steps):
            b = fetch()
            feeder.prefetch(host_ring[(i + 4) % args.ring])
            lt = e2e_step(b)
            loss_host[i & 1].copy_(lt.reshape(1), non_blocking=True)      # device -> host read of the step's loss
            loss_ev[i & 1].record()
            if i > 0:
                loss_ev[(i - 1) & 1].synchronize()
                lv = float(loss_host[(i - 1) & 1][0])
        loss_ev[(args.steps - 1) & 1].synchronize()
        lv = float(loss_host[(args.steps - 1) & 1][0])
        e1.record()
        barrier()
        ms2 = e0.elapsed_time(e1)
        t2 = torch.tensor([ms2], device=dev)
        if world > 1:
            dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        ms2 = float(t2.item())
        h2d = feeder.bytes_per_batch(host_ring[0])
        e2e = {"value": world * B * args.steps / (ms2 * 1e-3), "unit": "graphs/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": 4, "ms_per_step": ms2 / args.steps, "last_loss": lv,
               "h2d_format": feeder.format_note, "h2d_bytes_per_step_reference_format": int(batch_bytes)}
        # variant: the dataset (pool) resident in HBM, collation on the device; the step's host input is the graph-id list
        from gnn_matlang_b200.synthetic import DeviceDataset
        dds = DeviceDataset(pool, dev)
        idx_host = []
        for _ in range(args.ring):
            while True:                          # (draws that fit the captured shapes)
                idx = rng.integers(0, len(pool.n), B)
                if not use_graph or (pool.n[idx].sum() < Np and Ep - 8 * (Np - pool.n[idx].sum()) <= pool.e[idx].sum() <= Ep):
                    break
            idx_host.append(torch.from_numpy(idx.astype(np.int64)).pin_memory())
        if use_graph:
            def ds_step(ix):                    # id list -> captured buffers, collated on the device (two library launches)
                trainer.load_from_dataset(dds, ix)
                return trainer.step()
        else:
            def ds_step(ix):
                return trainer.step(dds.collate(ix))
        for i in range(3):
            float(ds_step(idx_host[i % args.ring]).item())
        barrier()
        e0.record()
        for i in range(args.steps):
            lt = ds_step(idx_host[i % args.ring])
            loss_host[i & 1].copy_(lt.reshape(1), non_blocking=True)
            loss_ev[i & 1].record()
            if i > 0:
                loss_ev[(i - 1) & 1].synchronize()
        loss_ev[(args.steps - 1) & 1].synchronize()
        e1.record()
        barrier()
        ms3 = e0.elapsed_time(e1)
        t3 = torch.tensor([ms3], device=dev)
        if world > 1:
            dist.all_reduce(t3, op=dist.ReduceOp.MAX)
        ms3 = float(t3.item())
        e2e["resident_dataset"] = {"value": world * B * args.steps / (ms3 * 1e-3), "unit": "graphs/s", "ms_per_step": ms3 / args.steps,
                                   "h2d_bytes_per_step": int(idx_host[0].numel() * 8), "d2h_bytes_per_step": 4,
                                   "note": "graph pool resident in HBM, batches collated on the device from the graph-id list"}

    # ---- CPU baseline on this box's host cores (rank 0, N = 1 only): oracle port, SAME graphs per step, bounded sample
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not is_exp:
        from oracle import gnnml3_oracle as O
        from gnn_matlang_b200.train import loss_fn
        torch.set_num_threads(os.cpu_count() or 1)
        hb = host_ring[0]
        ob = dict(x=hb.x, edge_index2=hb.edge_index2, edge_attr2=hb.edge_attr2, batch=hb.batch, num_graphs=hb.num_graphs)
        cm = O.OracleGNNML3(cfg, pool.K, pool.F)
        copt = torch.optim.Adam(cm.parameters(), lr=1e-3)

        def cstep():
            copt.zero_grad()
            l = loss_fn(loss, cm(ob), hb.y)
            l.backward()
            copt.step()

        cstep()
        t0 = time.perf_counter()
        nrep = 0
        while nrep < 3 or time.perf_counter() - t0 < 10.0:
            cstep()
            nrep += 1
        dt = time.perf_counter() - t0
        cpu = {"value": B * nrep / dt, "unit": "graphs/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": "%d training steps of %d %s-shaped graphs, the same batch size as the GPU arm (oracle port of the reference's "
                         "PyG path, torch CPU, all host threads)" % (nrep, B, args.workload)}

    # ---- the other BASELINE.json configurations, bounded (rank 0, N = 1 only)
    other = None
    if rank == 0 and world == 1 and not args.no_other_configs and args.workload == "zinc":
        other = {}

        def attempt(name, fn):           # a failure here must not take the headline line (or the other entries) down; it is reported
            try:
                other[name] = fn()
            except Exception as ex:
                other[name] = {"error": "%s: %s" % (type(ex).__name__, ex)}

        attempt("graph8c_isomorphism_eval", lambda: graph8c_config(dev, 0.0 if args.no_cpu_baseline else 3.0))
        attempt("zinc_reference_batch_64", lambda: small_config(dev, "zinc", 64, 100, 20))
        attempt("counting_batch_128", lambda: small_config(dev, "counting", 128, 100, 20))
        attempt("exp_spectral_design_on_gpu", lambda: exp_config(dev, 4096, 10, 3))
        attempt("exp_reference_batch_50", lambda: exp_config(dev, 50, 50, 10, cpu_sample=False, pipelined=True))
        attempt("spectconv_sweep_1M_nodes", lambda: [sweep_one(dev, F, 10, 1000000, hops, st, 2)
                                                     for F, hops, st in ((64, 1, 5), (64, 2, 3), (128, 1, 3), (256, 1, 2))])

    if rank == 0:
        edge_attr = pool.supports if not is_exp else ExpPool.supports
        config = common_config(args.workload, B, desc, edge_attr)
        config.update({"graphs_per_step_all_gpus": B * world, "nodes_per_step_per_gpu": N0, "support_entries_per_step_per_gpu": E0, "K": pool.K,
                       "gemm_arithmetic": {"fp32": "3xTF32 (FP32-grade)", "tf32": "single-pass TF32 (flagged)", "bf16": "BF16 projection in the fused layer kernel, TF32 elsewhere (flagged)"}[args.precision],
                       "sharding": "whole graphs over %d rank(s), one gradient SUM all-reduce per step" % world,
                       "l2_policy": "ring of %d distinct resident batches, %.0f MB in total (> 126 MB L2)" % (args.ring, args.ring * batch_bytes / 1e6)})
        print(json.dumps({
            "metric": "GNNML3 train graphs/s", "value": value, "unit": "graphs/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": {"fp32": "f32", "tf32": "tf32", "bf16": "bf16"}[args.precision], "data": "synthetic",
            "config": config, "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches) * args.steps, "gpu_launches_per_step": int(launches),
            "clocks": sampler.summary(), "host_enqueue_ms_per_step": host_ms, "step_mode": pad_note,
            "eager_step": {"ms_per_step": eager_ms, "host_enqueue_ms_per_step": eager_host_ms,
                           "note": "the same step enqueued launch by launch (no CUDA graph)"} if use_graph else None,
            "path_taken": {"fused_layer_launches_tensor_memory_kernel": paths[0] // nprof, "fused_layer_launches_smem_plane_kernel": paths[1] // nprof,
                           "unit": "launches per step"},
            "kernel_shares_one_step": ncu_shares(), "other_configs": other, "final_loss": final_loss}), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
