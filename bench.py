#!/usr/bin/env python
"""bench.py -- queries/sec of one training step of the hot path (BASELINE.json configs).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference|reference-cuda] [--config a|b|c|d|e]
                    [--dump-outputs DIR]

A "step" = scorer forward + fused loss/gradient + scorer backward + gradient all-reduce (N>1) + optimizer step over one
batch of synthetic MSLR-shaped queries per GPU (weak scaling).  Default --config b = BASELINE.json configs[1], the
configuration the headline metric is quoted on (LambdaRank + pointwise MLP, 256 docs x 136 features).  The other
configs: a ListNet 50x46 (the reference's CPU-runnable case), c ApproxNDCG + MHSA list scorer 512x136, d LambdaLoss
NDCG_Loss2++ 1024x136, e ListMLE with bf16-rounded GEMM operands (--docs 32..1024).

Prints ONE JSON line on rank 0:
  value        whole-job queries/s, inputs resident in HBM (CUDA events, max over ranks)
  e2e          the same metric through the reference-facing call ranker.train(host batches): pinned-host -> device copy
               of every batch and a device -> host read of every step's loss inside the timed region
  roofline     dominant kernel of the step, timed per launch with CUDA events in an instrumented pass of the same steps
               (ptrb200_timing_*), plus the STEP-level view: step_frac = SURVEY 8(d) algorithmic bytes per step / step
               time / HBM peak, pairs/s of the loss kernel against the MUFU peak, tensor-pipe fraction for config c
  cpu_baseline the oracle restatement of the reference's CPU PyTorch path on this box's cores (bounded sample), and
               reference_default_batch: both arms at the reference's own batching (B = 1 for lists of 100+ documents)
  reference_cuda  the same restatement as PyTorch eager on cuda:0 (the reference's `-cuda 0` path), N=1 only
  strong_scaling  (N>1) the same global batch as N=1 split over the ranks
--impl reference times the CPU restatement alone (rank 0 only); --impl reference-cuda the eager-GPU one.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

MSLR_P = np.array([1940952, 1225770, 504958, 69010, 30435], dtype=np.float64)
MSLR_P /= MSLR_P.sum()
MQ_P = np.array([12279, 2001, 931], dtype=np.float64)
MQ_P /= MQ_P.sum()
SEED = 137                                   # ptranking/ltr_global.py:5


def point_sf(F, dropout=0.1, **over):
    """The reference's default pointwise scorer (ptranking/ltr_adhoc/eval/parameter.py:142-146)."""
    d = dict(num_features=F, num_layers=5, AF="GE", TL_AF="S", apply_tl_af=True, BN=True, bn_type="BN", bn_affine=True,
             dropout=dropout)
    d.update(over)
    return dict(sf_id="pointsf", opt="Adam", lr=1e-4, pointsf=d)


def list_sf(F, L, dropout=0.1):
    """The reference's default list scorer (parameter.py:157-162): DASALC, 2 heads, no norm, Adagrad."""
    return dict(sf_id="listsf", opt="Adagrad", lr=1e-3,
                listsf=dict(num_features=F, ff_dims=[128, 256, 512], AF="R", TL_AF="GE", apply_tl_af=False, BN=False,
                            bn_type="BN2", bn_affine=False, n_heads=2, encoder_layers=L, encoder_type="DASALC", dropout=dropout))


def make_config(args):
    c = args.config
    if c == "a":
        return dict(key="a", model="ListNet", paras=None, sf=point_sf(46), n=50, F=46, B=args.batch or 1000, cpu_B=100,
                    labels=MQ_P, loss_kw={}, math=None,
                    workload="ListNet + pointwise-MLP (default scorer), 46 feat x 50 docs, MQ2008-shaped (BASELINE.json configs[0])",
                    metric="queries/sec (ListNet train step, 50-doc lists)")
    if c == "b":
        return dict(key="b", model="LambdaRank", paras=dict(model_id="LambdaRank", sigma=1.0), sf=point_sf(136), n=256, F=136,
                    B=args.batch or 1024, cpu_B=args.cpu_batch or 64, labels=MSLR_P, loss_kw=dict(sigma=1.0), math=None,
                    workload=("LambdaRank + pointwise-MLP (5x100 GELU, BN affine, sigmoid tail, dropout 0.1, Adam), "
                              "136 feat x 256 docs (BASELINE.json configs[1])"),
                    metric="queries/sec (LambdaRank train step, 256-doc lists)")
    if c == "c":
        L = args.enc_layers
        return dict(key="c", model="ApproxNDCG", paras=dict(model_id="ApproxNDCG", alpha=10.0), sf=list_sf(136, L), n=512, F=136,
                    B=args.batch or 64, cpu_B=2, labels=MSLR_P, loss_kw=dict(alpha=10.0), math=None, L=L,
                    workload=(f"ApproxNDCG + MHSA list scorer (DASALC, {L} encoder layers, 2 heads, 128/256/512 head and tail nets, "
                              "Adagrad), 136 feat x 512 docs (BASELINE.json configs[2])"),
                    metric="queries/sec (ApproxNDCG + list-scorer train step, 512-doc lists)")
    if c == "d":
        return dict(key="d", model="LambdaLoss", paras=dict(model_id="LambdaLoss", k=5, sigma=1.0, loss_type="NDCG_Loss2++", mu=5.0),
                    sf=point_sf(136), n=1024, F=136, B=args.batch or 256, cpu_B=4, labels=MSLR_P,
                    loss_kw=dict(k=5, sigma=1.0, loss_type="NDCG_Loss2++", mu=5.0), math=None,
                    workload="LambdaLoss NDCG_Loss2++ (k=5) + pointwise-MLP (default scorer), 136 feat x 1024 docs (BASELINE.json configs[3])",
                    metric="queries/sec (LambdaLoss train step, 1024-doc lists)")
    if c == "e":
        n = args.docs
        return dict(key="e", model="ListMLE", paras=None, sf=point_sf(136), n=n, F=136, B=args.batch or max(1, (1 << 18) // n),
                    cpu_B=max(1, 16384 // n), labels=MSLR_P, loss_kw={}, math="bf16",
                    workload=(f"ListMLE + pointwise-MLP (default scorer, GEMM operands rounded to bf16, fp32 accumulate / loss), "
                              f"136 feat x {n} docs (BASELINE.json configs[4])"),
                    metric=f"queries/sec (ListMLE bf16 train step, {n}-doc lists)")
    raise SystemExit(f"unknown config {c}")


def synth_batch(rng, B, n, F, probs):
    """MSLR-WEB30K-shaped synthetic batch: N(0,1) features, graded labels with the dataset's marginals, >=1 relevant doc
    per query, labels presorted descending (SURVEY.md 8d)."""
    X = rng.standard_normal((B, n, F), dtype=np.float32)
    y = rng.choice(len(probs), size=(B, n), p=probs).astype(np.float32)
    y[:, 0] = np.maximum(y[:, 0], 1.0)
    y = -np.sort(-y, axis=1)
    return torch.from_numpy(X), torch.from_numpy(y)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu_index, self.rows, self.proc = gpu_index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu_index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = max(mx, float(r[2]))
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"],
                    bf16_tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    sm_max_mhz=d.get("sm_max_mhz", 1965.0), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, sm_max_mhz=1965.0, source="fallback")


# --------------------------------------------------------------------------- #
# reference arms: the oracle restatement of the reference's PyTorch path, on the CPU or as eager PyTorch on the GPU
# --------------------------------------------------------------------------- #
def reference_run(cfg, steps, warmup, B, budget_s, device="cpu"):
    from oracle import ref_port as rp
    torch.manual_seed(SEED)
    rng = np.random.default_rng(SEED)
    sf = cfg["sf"]
    point = sf["sf_id"] == "pointsf"
    net = rp.point_scorer(**sf["pointsf"]) if point else rp.RefListScorer(**sf["listsf"])
    net = net.to(device)
    net.train()
    opt, _ = rp.make_optimizer(net.parameters(), sf["opt"], sf["lr"])
    batches = [tuple(t.to(device) for t in synth_batch(rng, B, cfg["n"], cfg["F"], cfg["labels"])) for _ in range(2)]
    sync = torch.cuda.synchronize if device != "cpu" else (lambda: None)
    for i in range(warmup):
        rp.train_op(net, opt, cfg["model"], *batches[i % 2], point=point, **cfg["loss_kw"])
    sync()
    t0 = time.perf_counter()
    done = 0
    for i in range(steps):
        rp.train_op(net, opt, cfg["model"], *batches[i % 2], point=point, **cfg["loss_kw"])
        done += 1
        if device == "cpu" and time.perf_counter() - t0 > budget_s and done >= 3:
            break
    sync()
    dt = time.perf_counter() - t0
    return dict(qps=done * B / dt, ms_per_step=1e3 * dt / done, steps=done, B=B, cores=torch.get_num_threads())


def host_threads():
    """Threads for the CPU arm: every PHYSICAL core this process may run on (torchrun exports OMP_NUM_THREADS=1, and
    oversubscribing the SMT siblings makes ATen's elementwise kernels several times slower)."""
    try:
        import psutil
        phys = psutil.cpu_count(logical=False) or 0
    except Exception:
        phys = 0
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    n = phys if phys > 0 else max(1, avail // 2)
    return max(1, min(n, avail))


def run_reference(args, cfg, device="cpu"):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    torch.set_num_threads(host_threads())
    cuda = device != "cpu"
    B = (cfg["B"] if cuda else cfg["cpu_B"])
    r = reference_run(cfg, args.steps, args.warmup, B, budget_s=240.0, device=device)
    sample = (f"{r['steps']} steps x {B} queries x {cfg['n']} docs x {cfg['F']} feat, oracle/ref_port.py train_op"
              + (" as PyTorch eager on cuda:0" if cuda else ""))
    line = {
        "impl": "reference-cuda" if cuda else "reference", "metric": cfg["metric"], "value": r["qps"],
        "unit": "queries/s", "n_gpus": args.gpus, "steps": r["steps"], "warmup": args.warmup,
        "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg["workload"], "queries_per_step": B, "n_docs": cfg["n"], "n_features": cfg["F"],
                   "device": device,
                   "sample": "each step is a bounded sample of the workload: one batch of %d queries (the B200 arm steps %d per GPU)" % (B, cfg["B"]),
                   "math": "fp32 ATen kernels"},
        "cpu_baseline": {"value": r["qps"], "unit": "queries/s", "cores": r["cores"], "kind": "port", "sample": sample},
        "e2e": {"value": r["qps"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- #
# B200 arm
# --------------------------------------------------------------------------- #
class HostBatches:
    """Iterable of (ids, X, y) pinned-host batches -- what ranker.train() consumes (the reference's DataLoader contract:
    data_utils.py:683-742, uniform n per batch)."""

    def __init__(self, batches, count):
        self.batches, self.count = batches, count

    def __iter__(self):
        for i in range(self.count):
            X, y = self.batches[i % len(self.batches)]
            yield [str(q) for q in range(X.size(0))], X, y


def build_ranker(cfg, dev):
    import ptranking_b200
    if cfg["math"]:
        os.environ["PTRANKING_B200_MATH"] = cfg["math"]
    cls = getattr(ptranking_b200, cfg["model"])
    r = cls(sf_para_dict=cfg["sf"], gpu=True, device=dev) if cfg["paras"] is None else \
        cls(sf_para_dict=cfg["sf"], model_para_dict=cfg["paras"], gpu=True, device=dev)
    r.init()
    r.train_mode()
    return r


def algorithmic(cfg, B):
    """SURVEY 8(d) per-step figures: HBM bytes n(F*4+8) per query (features + labels in, scores out), FLOPs of
    forward+backward (3x forward), loss pairs."""
    n, F = cfg["n"], cfg["F"]
    out = {"bytes_per_query": n * (F * 4 + 8)}
    if cfg["sf"]["sf_id"] == "pointsf":
        dims = [F] + [100] * cfg["sf"]["pointsf"]["num_layers"] + [1]
        out["flops_per_query"] = 3 * 2 * n * sum(a * b for a, b in zip(dims[:-1], dims[1:]))
        out["dims"] = dims
    else:
        L = cfg["L"]
        out["flops_per_query"] = 3 * n * (865280 + L * (147968 + 4 * n * F))
        out["attention_flops_per_query"] = 3 * 4 * n * n * F * L
    pairs = {"LambdaRank": n * (n - 1) // 2, "RankNet": n * (n - 1) // 2, "ApproxNDCG": 2 * n * n,
             "LambdaLoss": min(5, n) * (min(5, n) - 1) // 2}.get(cfg["model"])
    out["pairs_per_query"] = pairs
    return out


DUMP_LIMIT_BYTES = 64 << 20


def scorer_state(ranker):
    """name -> tensor of the scorer's checkpoint (what ranker.save writes): the weights the step updated."""
    if hasattr(ranker, "point_sf"):
        return dict(ranker.point_sf.state_dict())
    return {f"{part}.{k}": v for part, m in ranker.list_sf.items() for k, v in m.state_dict().items()}


def dump_outputs(out_dir, loss, state):
    """DIR/loss.npy and DIR/state.<name>.npy (float32) of one train step, so that two builds can be compared output for
    output.  Past DUMP_LIMIT_BYTES in all, each tensor is cut to a fixed, seeded sample of its flattened elements."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss.detach().float().reshape(1).cpu().numpy()}
    arrays.update((f"state.{k}", v.detach().float().cpu().numpy()) for k, v in state.items())
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_LIMIT_BYTES:
            keep = max(1, a.size * DUMP_LIMIT_BYTES // total)
            idx = np.sort(np.random.default_rng(SEED).choice(a.size, size=keep, replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_b200(args, cfg):
    import torch.distributed as dist
    from ptranking_b200 import _lib, LABEL_TYPE
    from ptranking_b200 import dist as b200dist

    rank, local, world = b200dist.init_from_env("nccl")
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    B, n, F = cfg["B"], cfg["n"], cfg["F"]
    torch.manual_seed(SEED)
    rng = np.random.default_rng(SEED + rank)
    ranker = build_ranker(cfg, dev)            # config_optimizer broadcasts rank 0's weights to every replica
    host = [tuple(t.pin_memory() for t in synth_batch(rng, B, n, F, cfg["labels"])) for _ in range(2)]
    devb = [(X.to(dev), y.to(dev)) for X, y in host]
    kw = dict(presort=True, label_type=LABEL_TYPE.MultiLabel, epoch_k=1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t)
        return ms

    def timed(batches, steps, warm):
        for i in range(warm):
            ranker.train_op(*batches[i % 2], **kw)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        loss = None
        for i in range(steps):
            loss, _ = ranker.train_op(*batches[i % 2], **kw)
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)), loss

    # ---- value: device-resident inputs -----------------------------------------
    for i in range(args.warmup):
        ranker.train_op(*devb[i % 2], **kw)
    barrier()
    l0 = _lib.launch_count()
    with ClockSampler(local) as clk:
        ms, loss = timed(devb, args.steps, 0)
    launches = _lib.launch_count() - l0
    value = world * B * args.steps / (ms / 1e3)
    last_loss = float(loss)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss, scorer_state(ranker))

    # ---- strong scaling: the N=1 global batch split over the ranks ----------------
    strong = None
    if world > 1 and B % world == 0:
        Bs = B // world
        sb = [(X[:Bs].contiguous(), y[:Bs].contiguous()) for X, y in devb]
        ms_s, _ = timed(sb, args.steps, 3)
        strong = {"value": B * args.steps / (ms_s / 1e3), "unit": "queries/s", "ms_per_step": ms_s / args.steps,
                  "global_queries_per_step": B, "queries_per_gpu_per_step": Bs,
                  "note": "same global batch as the N=1 run; efficiency vs N=1 is value / (N x value at N=1)"}

    # ---- e2e: host batches through ranker.train ---------------------------------
    ranker.train(HostBatches(host, args.warmup), epoch_k=1, presort=True, label_type=LABEL_TYPE.MultiLabel)
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0.record()
    ep_loss, _ = ranker.train(HostBatches(host, args.steps), epoch_k=1, presort=True, label_type=LABEL_TYPE.MultiLabel)
    ep_loss_host = float(ep_loss.cpu())
    t1.record()
    barrier()
    ms_e2e = max_over_ranks(t0.elapsed_time(t1))
    e2e = world * B * args.steps / (ms_e2e / 1e3)
    h2d = int(host[0][0].numel() * 4 + host[0][1].numel() * 4)

    # ---- roofline pass: per-launch CUDA events around every kernel of the same steps ----
    roof = None
    steps_timed = min(args.steps, 5)
    if rank == 0:       # every rank runs the same steps (they contain the gradient all-reduce); only rank 0 records events
        _lib.kernel_timings(enable=True)
    for i in range(steps_timed):
        ranker.train_op(*devb[i % 2], **kw)
    torch.cuda.synchronize()
    if rank == 0:
        tm = _lib.kernel_timings()
        _lib.kernel_timings(enable=False)
        roof = build_roofline(cfg, B, tm, steps_timed, ms / args.steps)
    barrier()

    # ---- baselines (rank 0, N=1 only) -----------------------------------------
    cpu = ref_b1 = ref_cuda = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # GPU-side comparators first: both are (partly) launch-bound, and the worker threads of the CPU runs below keep
        # spinning for a while after a parallel region -- measured 0.62 ms vs 2.0 ms per B = 1 step depending on the order
        B1 = max(1, 100 // n)       # the reference's own batching: B = max(1, 100 // n) queries per step (data_utils.py:683-718)
        one = [(X[:B1].contiguous(), y[:B1].contiguous()) for X, y in devb]
        ms1, _ = timed(one, 50, 5)
        try:
            rc = reference_run(cfg, steps=10, warmup=3, B=B, budget_s=60.0, device=dev)
            ref_cuda = {"value": rc["qps"], "unit": "queries/s", "ms_per_step": rc["ms_per_step"], "queries_per_step": B,
                        "kind": "port", "what": "oracle/ref_port.py train_op as PyTorch eager on cuda:0 (the reference's `-cuda 0` path)"}
        except Exception as e:      # e.g. the [B,n,n] temporaries do not fit
            ref_cuda = {"unavailable": repr(e)[:200]}
        torch.set_num_threads(host_threads())
        r = reference_run(cfg, steps=40, warmup=2, B=cfg["cpu_B"], budget_s=15.0)
        cpu = {"value": r["qps"], "unit": "queries/s", "cores": r["cores"], "kind": "port",
               "sample": f"{r['steps']} steps x {r['B']} queries x {n} docs (oracle/ref_port.py train_op, fp32 CPU PyTorch ops)"}
        r1 = reference_run(cfg, steps=200, warmup=3, B=B1, budget_s=5.0)
        ref_b1 = {"queries_per_step": B1, "cpu_port_qps": r1["qps"], "b200_qps": B1 * 50 / (ms1 / 1e3),
                  "b200_ms_per_step": ms1 / 50, "note": "launch-latency bound on the GPU: ~50 kernel launches per step"}

    if rank == 0:
        line = {
            "metric": cfg["metric"], "value": value, "unit": "queries/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["workload"], "config_key": cfg["key"],
                       "queries_per_gpu_per_step": B, "n_docs": n, "n_features": F,
                       "parallelism": f"dp{world}",
                       "gradient_exchange": ("none (one GPU)" if world == 1 else
                                             "summed inside the optimizer kernel over NVLink peer memory (CUDA IPC), one launch" if getattr(ranker.grad_bucket, "peer", None) is not None
                                             else "ncclAllReduce(SUM) of the flat gradient buffer, then the optimizer kernel"),
                       "l2": f"inputs (2 x {h2d / 1e6:.0f} MB rotating batches) " + ("larger than" if 2 * h2d > 126e6 else "NOT larger than") + " the 126 MB L2",
                       "normalisation": "BN (reference default, batch statistics" + (", synchronised over ranks)" if b200dist.sync_bn_active() else " per rank)") if cfg["sf"]["sf_id"] == "pointsf" else "none (listsf default)",
                       "math": ("GEMM operands rounded to bf16, fp32 accumulate" if cfg["math"] == "bf16" else
                                "fp32 in/out; Linear contractions on tcgen05 as 3xTF32 (error-compensated, fp32-equivalent) with fp32 TMEM accumulation")},
            "e2e": {"value": e2e, "unit": "queries/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / args.steps, "epoch_loss": ep_loss_host},
            "gpu_launches": int(launches), "clocks": clk.summary(), "roofline": roof, "cpu_baseline": cpu,
            "reference_default_batch": ref_b1, "reference_cuda": ref_cuda, "strong_scaling": strong,
            "last_loss": last_loss,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def build_roofline(cfg, B, tm, steps_timed, ms_per_step):
    """roofline object of the bench line from the per-kernel CUDA-event record ``tm`` {name: (launches, total_ms)}."""
    peaks = measured_peaks()
    alg = algorithmic(cfg, B)
    n, F = cfg["n"], cfg["F"]
    rows = B * n
    total_ms = sum(v[1] for v in tm.values())
    per_step = {k: round(v[1] / steps_timed, 4) for k, v in sorted(tm.items(), key=lambda kv: -kv[1][1])}
    step_bytes = alg["bytes_per_query"] * B
    roof = {}
    traffic_tab = {}
    tpath = os.path.join(ROOT, "profiles", "traffic.json")       # dram bytes per launch from the committed ncu --set full captures
    if os.path.exists(tpath):
        traffic_tab = json.load(open(tpath))
    if cfg["sf"]["sf_id"] == "pointsf":
        dims = alg["dims"]
        pairs = list(zip(dims[:-1], dims[1:]))
        # ALGORITHMIC HBM bytes one step must move through each kernel family (DESIGN.md section 4):
        # fwd layer: read its input, write its output; dgrad: read dZ, write dIn (layers 1..L-2; the 100->1 layer is an outer product);
        # wgrad: read dZ and the layer input; dY / dZ passes: two reads + one write of the layer width; loss: 12 n per query
        algo = {
            "rows_gemm_ws_fwd": sum(rows * (a + b) * 4 for a, b in pairs),
            "rows_gemm_tc_fwd": sum(rows * (a + b) * 4 for a, b in pairs),
            "rows_gemm_ws_dgrad": sum(rows * (a + b) * 4 for a, b in pairs[1:-1]),
            "rows_gemm_tc_dgrad": sum(rows * (a + b) * 4 for a, b in pairs[1:-1]),
            "wgrad_tc": sum(rows * (a + b) * 4 for a, b in pairs),
            "colstat_dy": sum(rows * b * 12 for a, b in pairs),
            "norm_bwd_apply4_kernel": sum(rows * b * 12 for a, b in pairs[:-1]),
            "gemm_simt_fwd": sum(rows * (a + b) * 4 for a, b in pairs),
            "gemm_simt_bwd_data": sum(rows * (a + b) * 4 for a, b in pairs[1:]),
            "gemm_simt_bwd_weight": sum(rows * (a + b) * 4 for a, b in pairs),
        }
        cand = [(k, v) for k, v in tm.items() if k in algo]
        name, (cnt, kms) = max(cand, key=lambda kv: kv[1][1])
        per_launch_bytes = algo[name] * steps_timed / cnt
        achieved = per_launch_bytes / (kms / cnt * 1e-3) / 1e9
        roof = {"bound": "hbm", "kernel": name, "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": achieved / peaks["hbm_gbs"], "traffic": traffic_tab.get(name),
                "peak_source": peaks["source"] + " (copy bandwidth)",
                "launches_per_step": cnt / steps_timed, "algorithmic_bytes_per_launch": per_launch_bytes,
                "share_of_step": kms / total_ms,
                "note": "fused Linear layer: 25 flop per HBM byte at d=100, far left of the tensor ridge (~210 flop/B), so HBM binds"}
    else:
        # list scorer: the contractions bind.  FLOP view of the whole step against the dense tensor peak for TF32
        # operands (half the measured bf16 peak); the 3xTF32 split issues 3 MMAs per algorithmic one.
        tf32_peak = peaks["bf16_tflops_sustained"] / 2.0
        flops = alg["flops_per_query"] * B
        tens = {k: v for k, v in tm.items() if k.startswith(("attn_tc", "rows_gemm", "wgrad_tc"))}
        name, (cnt, kms) = max(tens.items(), key=lambda kv: kv[1][1])
        tens_ms = sum(v[1] for v in tens.values()) / steps_timed
        achieved = flops / (tens_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "kernel": name, "achieved": achieved, "peak": tf32_peak, "unit": "TFLOP/s",
                "frac": achieved / tf32_peak,
                # per-launch DRAM bytes from the committed captures of THIS configuration only (wgrad_tc's entry is config b's)
                "traffic": traffic_tab.get(name) if (name.startswith("attn_tc") or name == "rows_gemm_tc_fwd") else None,
                "peak_source": peaks["source"] + " (bf16 sustained / 2 = dense TF32)",
                "share_of_step": kms / total_ms, "tensor_kernels_ms_per_step": tens_ms,
                "issued_frac_3xtf32": 3 * achieved / tf32_peak,
                "attention_gemms_ms_per_step": sum(v[1] for k, v in tm.items() if k.startswith("attn_tc")) / steps_timed,
                "note": "algorithmic FLOPs of the step (3x forward) over the time spent in tensor-core kernels; "
                        "issued_frac counts the three TF32 MMAs per product the fp32-grade split issues"}
    # ---- the step as a whole (SURVEY 8d) -----------------------------------------------------------
    roof["step_bytes_algorithmic"] = step_bytes
    roof["step_frac"] = step_bytes / (ms_per_step * 1e-3) / 1e9 / peaks["hbm_gbs"]
    dram = 0.0
    known = True
    for k, (cnt, _) in tm.items():
        if k in traffic_tab and traffic_tab[k]:
            dram += traffic_tab[k] * cnt / steps_timed
        elif _ > 0.02 * total_ms:
            known = False
    roof["dram_bytes_per_step"] = dram if (dram > 0 and known) else None
    roof["step_tflops_algorithmic"] = alg["flops_per_query"] * B / (ms_per_step * 1e-3) / 1e12
    if alg["pairs_per_query"]:
        loss_k = [k for k in tm if k.startswith(("pairwise_bce", "approxndcg_kernel", "lambdaloss_kernel"))]
        if loss_k:
            lms = sum(tm[k][1] for k in loss_k) / steps_timed
            mufu_peak = 16 * 148 * peaks["sm_max_mhz"] * 1e6          # MUFU results per second (16 / clk / SM)
            pps = alg["pairs_per_query"] * B / (lms * 1e-3)
            roof["loss"] = {"kernel": loss_k[0], "ms_per_step": lms, "pairs_per_s": pps,
                            "mufu_ops_per_pair": 4, "mufu_frac": 4 * pps / mufu_peak,
                            "hbm_frac": 12.0 * n * B / (lms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                            "note": "O(n^2) pair work on 12n bytes: SFU (ex2/rcp/lg2) and FP32 issue bind, not HBM"}
    roof["kernels_ms_per_step"] = per_step
    return roof


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default: 100 for configs a, b, e; 20 for c; 50 for d)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "reference-cuda"])
    ap.add_argument("--config", default="b", choices=["a", "b", "c", "d", "e"], help="BASELINE.json configs[0..4]")
    ap.add_argument("--batch", type=int, default=0, help="queries per GPU per step (0 = the config's default)")
    ap.add_argument("--cpu-batch", type=int, default=0, help="queries per step on the CPU arm (0 = the config's default)")
    ap.add_argument("--docs", type=int, default=256, help="config e: documents per query (32..1024)")
    ap.add_argument("--enc-layers", type=int, default=6, help="config c: encoder layers (6 = code default, 3 = test JSON)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (loss, updated scorer state) as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    cfg = make_config(args)
    if args.steps is None:
        args.steps = {"a": 100, "b": 100, "c": 20, "d": 50, "e": 100}[args.config]
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args, cfg, "cpu")
    elif args.impl == "reference-cuda":
        run_reference(args, cfg, "cuda:0")
    else:
        run_b200(args, cfg)


if __name__ == "__main__":
    main()
