"""Golden fixtures for WassRank, produced by the UNMODIFIED reference.

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden_wassrank.py

fp32: the reference class's own WassRank.custom_loss_function (wassRank.py:43-86) at B=1 on a leaf score tensor, with a
throw-away SGD(lr=0) standing in for the optimizer it steps and its per-call print of the scores sent to /dev/null.
float64: the same reference functions (get_explicit_cost_mat, get_normalized_histograms, OldSinkhornOT) on float64
tensors.  Inputs: every cost type with the 'ST' histograms, 'NG' for 'eg' and 'p1', lambda in {0.1, 1, 10},
n in {1, 8, 50, 256, 1024}; plus 'NG' on a list whose minimum score is <= 0 and tied.  Which fp32 outputs are not
finite is stored beside them.  Output: wassrank.npz.
"""
import contextlib
import io
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

from make_golden import synth_labels, point_sf_dict, MSLR_P  # noqa: E402
from ptranking.ltr_adhoc.listwise.wassrank.wassRank import WassRank, WassRankParameter, wasserstein_distance  # noqa: E402
from ptranking.ltr_adhoc.listwise.wassrank.wasserstein_cost_mat import get_explicit_cost_mat, get_normalized_histograms  # noqa: E402

COMBOS = [("eg", "ST"), ("p1", "ST"), ("p2", "ST"), ("dg", "ST"), ("ddg", "ST"), ("eg", "NG"), ("p1", "NG")]
LAMS = [0.1, 1.0, 10.0]
NS = [1, 8, 50, 256, 1024]


def run_fp32(para, s, y):
    r = WassRank(sf_para_dict=point_sf_dict(4), wass_para_dict=para, gpu=False, device="cpu")
    r.dict_std_dists = None         # the constructor sets it only when given one (wassRank.py:35-36)
    leaf = torch.from_numpy(s).clone().requires_grad_(True)
    r.optimizer = torch.optim.SGD([leaf], lr=0.0)
    with contextlib.redirect_stdout(io.StringIO()):     # wassRank.py:46 prints the whole score tensor
        loss = r.custom_loss_function(leaf, torch.from_numpy(y), batch_ids=["q"])
    return float(loss.detach().reshape(())), leaf.grad.detach().numpy().copy()


def run_fp64(para, s, y):
    y64 = torch.from_numpy(y).double()
    leaf = torch.from_numpy(s).double().requires_grad_(True)
    C = get_explicit_cost_mat(y64, wass_para_dict=para).double()
    std_h, pred_h = get_normalized_histograms(batch_std_labels=y64, batch_preds=leaf, wass_dict_std_dists=None, qid="q",
                                              wass_para_dict=para, TL_AF=None)
    loss = wasserstein_distance(pred_h, std_h.double(), torch.squeeze(C, dim=0), para["lam"], para["sh_itr"])
    loss.backward()
    return float(loss.detach().reshape(())), leaf.grad.detach().numpy().copy()


def main():
    rng = np.random.default_rng(5150)
    torch.manual_seed(5150)
    base = WassRankParameter().default_para_dict()
    out = {}
    inputs = {}
    for n in NS:
        y = synth_labels(rng, 1, n, MSLR_P)
        wide = (2.5 * rng.standard_normal((1, n))).astype(np.float32)                       # 'ST': raw scores
        sig = (1.0 / (1.0 + np.exp(-rng.standard_normal((1, n))))).astype(np.float32)       # 'NG': positive scores
        inputs[n] = (y, wide, sig)
    tied = np.array([[0.7, -0.4, 1.3, 0.2, -0.4, 0.9, 0.0, 2.1]], dtype=np.float32)          # minimum <= 0, tied
    cases = []
    for cost, smooth in COMBOS:
        for lam in LAMS:
            for n in NS:
                y, wide, sig = inputs[n]
                cases.append((f"{cost}_{smooth}_lam{lam:g}_n{n}", cost, smooth, lam, wide if smooth == "ST" else sig, y))
    for cost in ("eg", "p1"):
        cases.append((f"{cost}_NG_lam1_n8_tiedmin", cost, "NG", 1.0, tied, inputs[8][0]))
    for key, cost, smooth, lam, s, y in cases:
        para = dict(base, cost_type=cost, smooth_type=smooth, lam=lam)
        l32, g32 = run_fp32(para, s, y)
        l64, g64 = run_fp64(para, s, y)
        out[key + "__scores"], out[key + "__labels"] = s, y
        out[key + "__loss32"], out[key + "__grad32"] = np.float32(l32), g32.astype(np.float32)
        out[key + "__loss64"], out[key + "__grad64"] = np.float64(l64), g64
        out[key + "__finite32"] = np.array([np.isfinite(l32), np.isfinite(g32).all()])
        out[key + "__finite64"] = np.array([np.isfinite(l64), np.isfinite(g64).all()])
        print(f"{key:28s} fp32 {l32:.6g} {'' if np.isfinite(g32).all() else '(grad not finite)'}  float64 {l64:.6g}")
    np.savez_compressed(os.path.join(HERE, "wassrank.npz"), **out)
    print(f"wassrank.npz: {len(cases)} cases, {len(out)} arrays")


if __name__ == "__main__":
    main()
