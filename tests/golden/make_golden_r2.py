"""Round-2 fixtures from the UNMODIFIED reference (VERDICT r1, next-round item 1):

  * pointwise scorer with the activations T / E / LR / SE (forward + every parameter gradient),
  * the list scorer at BASELINE config (c)'s REAL shape -- F=136, n=512, ff_dims [128,256,512], 2 heads, DASALC --
    with L=6 / no norm (the code default, ltr_adhoc/eval/parameter.py:157-162) and L=3 / BN2 (the test JSON,
    testing/ltr_adhoc/json/Data_Eval_ScoringFunction.json:50-60): forward scores, every parameter gradient and three
    ApproxNDCG train_op steps (Adagrad, the listsf default).

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden_r2.py      ->  scorers_r2.npz

To keep the file small, outputs above 1024 elements are stored as a strided sample (every k-th element of the flattened
tensor) plus their L2 norm and sum -- tests/helpers.py::sampled() reproduces the sampling.  Features and initial
weights are not stored: tests/helpers.py::load regenerates them from the same seeds and checks them against the stored
``<key>@probe`` elements (make_clones gives every encoder layer the same initial weights, list_ranker.py:48-50, so one
layer is probed).
"""
import os
import sys
import warnings

import numpy as np
import torch

warnings.filterwarnings("ignore")
REF = os.environ.get("PTRANKING_REFERENCE", "/root/reference")
sys.path.insert(0, REF)
sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

from make_golden import synth_labels, point_sf_dict, MSLR_P, ML, put_probe, put_sampled  # noqa: E402
from ptranking.ltr_adhoc.listwise.listnet import ListNet  # noqa: E402
from ptranking.ltr_adhoc.listwise.approxNDCG import ApproxNDCG  # noqa: E402


def main():
    out = {}
    rng = np.random.default_rng(2137)
    # ---- activations the round-1 fixtures did not cover -------------------------------------------
    for code in ("T", "E", "LR", "SE"):
        for (B, n, F) in [(3, 50, 46), (2, 64, 136)]:
            torch.manual_seed(137)
            sf = point_sf_dict(F, AF=code, TL_AF=code, num_layers=3)
            r = ListNet(sf_para_dict=sf, gpu=False, device="cpu")
            r.init()
            with torch.no_grad():
                for k, p in r.point_sf.named_parameters():
                    if "bn" in k:
                        p.add_(0.1 * torch.randn_like(p))
            X = torch.from_numpy(rng.standard_normal((B, n, F)).astype(np.float32))
            rvec = torch.from_numpy(rng.standard_normal((B, n)).astype(np.float32))
            s = r.forward(X)
            (s * rvec).sum().backward()
            key = f"point_af{code}_B{B}_n{n}_F{F}"
            put_probe(out, key + "__X", X.numpy())
            out[key + "__dscores"], out[key + "__scores"] = rvec.numpy(), s.detach().numpy()
            for k, v in r.point_sf.state_dict().items():
                put_probe(out, f"{key}__param::{k}", v.numpy())
            for k, p in r.point_sf.named_parameters():
                put_sampled(out, f"{key}__grad::{k}", p.grad.numpy())

    # ---- list scorer at config (c)'s real shape ----------------------------------------------------
    B, n, F = 2, 512, 136
    for tag, L, bn in (("L6_nonorm", 6, False), ("L3_bn2", 3, True)):
        d = dict(num_features=F, ff_dims=[128, 256, 512], AF="R", TL_AF="GE", apply_tl_af=False, BN=bn, bn_type="BN2",
                 bn_affine=False, n_heads=2, encoder_layers=L, encoder_type="DASALC", dropout=0.0)
        sf = dict(sf_id="listsf", opt="Adagrad", lr=1e-3, listsf=d)
        torch.manual_seed(137)
        r = ApproxNDCG(sf_para_dict=sf, model_para_dict=dict(model_id="ApproxNDCG", alpha=10.0), gpu=False, device="cpu")
        r.init()
        r.eval_mode()           # the tail FFN ignores the configured dropout (SURVEY B10): eval mode switches it off
        key = f"listc_{tag}"
        out[key + "__L"] = np.int64(L)
        for part in ("head_ffnns", "tail_ffnns"):
            for k, v in r.list_sf[part].state_dict().items():
                put_probe(out, f"{key}__init::{part}::{k}", v.numpy())
        enc_sd = r.list_sf["encoder"].state_dict()
        layer0 = {k[len("layers.0."):]: v for k, v in enc_sd.items() if k.startswith("layers.0.")}
        for l in range(1, L):   # make_clones: identical initial weights in every layer
            for k, v in layer0.items():
                assert torch.equal(enc_sd[f"layers.{l}.{k}"], v)
        for k, v in layer0.items():
            put_probe(out, f"{key}__init::encoder_layer::{k}", v.numpy())
        X = rng.standard_normal((3, B, n, F)).astype(np.float32)
        y = np.stack([synth_labels(rng, B, n, MSLR_P) for _ in range(3)])
        put_probe(out, key + "__X", X)
        out[key + "__labels"] = y
        # forward + every parameter gradient for a random upstream gradient
        rvec = torch.from_numpy(rng.standard_normal((B, n)).astype(np.float32))
        s = r.forward(torch.from_numpy(X[0]))
        (s * rvec).sum().backward()
        out[key + "__dscores"], out[key + "__scores"] = rvec.numpy(), s.detach().numpy()
        for part in ("head_ffnns", "encoder", "tail_ffnns"):
            for k, p in r.list_sf[part].named_parameters():
                put_sampled(out, f"{key}__grad::{part}::{k}", p.grad.numpy())
        # three ApproxNDCG train_op steps
        losses = []
        for t in range(3):
            loss, _ = r.train_op(torch.from_numpy(X[t]), torch.from_numpy(y[t]), presort=True, label_type=ML)
            losses.append(float(loss.detach()))
        out[key + "__losses"] = np.array(losses, dtype=np.float64)
        for part in ("head_ffnns", "encoder", "tail_ffnns"):
            for k, v in r.list_sf[part].state_dict().items():
                put_sampled(out, f"{key}__final::{part}::{k}", v.detach().numpy())
        out[key + "__final_scores"] = r.predict(torch.from_numpy(X[0])).detach().numpy()
    np.savez_compressed(os.path.join(HERE, "scorers_r2.npz"), **out)
    print("scorers_r2.npz:", len(out), "arrays", os.path.getsize(os.path.join(HERE, "scorers_r2.npz")) // 1024, "KiB")


if __name__ == "__main__":
    main()
