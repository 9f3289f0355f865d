"""Time WassRank's loss forward + backward on the GPU: the fused kernel (ops.rank_loss_and_grad) against the reference's
algorithm restated with ATen ops (oracle/ref_port_wassrank.py, run eagerly on the same device, one query at a time as the
reference runs).  Default parameters (eg cost, ST histograms, lambda 0.1, 20 Sinkhorn rounds), B = 1024 queries,
n in {32, 128, 256, 1024}.  CUDA events around warmed-up calls; the card's name and power limit are read in the same run.

    python tools/wassrank_bench.py [--json out.json] [--ns 32,128,256,1024] [--B 1024] [--ref-queries 64]

Prints one JSON line.  exp terms per query: (2 * sh_itr + 1) * n^2 (both Sinkhorn half-steps, then the loss pass).
The inputs (B * n floats) stay in L2: the kernel is compute-bound, so no cache flushing between calls.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

PARA = dict(mode="SinkhornOT", sh_itr=20, lam=0.1, smooth_type="ST", norm_type="BothST", cost_type="eg",
            non_rele_gap=100, var_penalty=float(np.e), gain_base=4)
MSLR_P = np.array([1940952, 1225770, 504958, 69010, 30435], dtype=np.float64)
MSLR_P /= MSLR_P.sum()


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return name, q


def timed(fn, min_seconds=0.5, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); fn(); e1.record(); torch.cuda.synchronize()
    reps = max(3, int(min_seconds * 1e3 / max(e0.elapsed_time(e1), 1e-3)))
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--json", default=None)
    ap.add_argument("--ns", default="32,128,256,1024")
    ap.add_argument("--B", type=int, default=1024)
    ap.add_argument("--ref-queries", type=int, default=64,
                    help="queries of the batch the eager reference arm runs (it loops over queries; time scales linearly)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("wassrank_bench needs a CUDA device")
    from ptranking_b200 import ops, build
    from oracle import ref_port_wassrank as rp
    build.build()
    dev = torch.device("cuda", 0)
    name, smi = card()
    rows = []
    for n in [int(v) for v in args.ns.split(",")]:
        B = args.B
        rng = np.random.default_rng(n)
        y = -np.sort(-rng.choice(5, size=(B, n), p=MSLR_P).astype(np.float32), axis=1)
        s = (2.5 * rng.standard_normal((B, n))).astype(np.float32)
        st, yt = torch.from_numpy(s).to(dev), torch.from_numpy(y).to(dev)
        ms, reps = timed(lambda: ops.rank_loss_and_grad("WassRank", st, yt, **PARA), min_seconds=1.0)
        _, lq, g = ops.rank_loss_and_grad("WassRank", st, yt, **PARA)
        terms = B * (2 * PARA["sh_itr"] + 1) * n * n
        Br = min(args.ref_queries, B)

        def ref_step():
            leaf = st[:Br].clone().requires_grad_(True)
            loss = rp.wassrank_loss(leaf, yt[:Br], **PARA)
            loss.backward()
            return loss, leaf.grad

        ref_ms, ref_reps = timed(ref_step, min_seconds=1.0, warmup=1)
        rl, rg = ref_step()
        rows.append(dict(n=n, B=B, kernel_ms=round(ms, 4), kernel_reps=reps, kernel_queries_per_s=round(B / ms * 1e3, 1),
                         kernel_exp_terms_per_s=float(f"{terms / ms * 1e3:.4g}"),
                         kernel_finite=bool(torch.isfinite(lq).all() and torch.isfinite(g).all()),
                         ref_queries=Br, ref_ms=round(ref_ms, 3), ref_reps=ref_reps,
                         ref_queries_per_s=round(Br / ref_ms * 1e3, 1),
                         ref_exp_terms_per_s=float(f"{Br * (2 * PARA['sh_itr'] + 1) * n * n / ref_ms * 1e3:.4g}"),
                         ref_loss_finite=bool(torch.isfinite(rl).all()), ref_grad_finite=bool(torch.isfinite(rg).all()),
                         speedup_queries_per_s=round((B / ms) / (Br / ref_ms), 1)))
    out = dict(bench="wassrank_fwd_bwd", device=name, nvidia_smi_name_power_limit_max_sm_clock=smi, params=PARA,
               torch=torch.__version__, rows=rows)
    line = json.dumps(out)
    print(line)
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
