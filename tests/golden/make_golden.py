"""Generate the golden fixtures in this directory by running the UNMODIFIED reference.

Run where the reference checkout is importable (the tests themselves never need it):

    PTRANKING_REFERENCE=<reference checkout> PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py

Imports wildltr/ptranking from $PTRANKING_REFERENCE, feeds it seeded synthetic inputs
(seed 137 = ptranking/ltr_global.py:5) and stores inputs + outputs as .npz.
Nothing from the reference is copied: only tensors it computed are saved.

scorers.npz / train_steps.npz keep each file small: features and the pointwise scorers' initial weights are not
stored -- tests/helpers.py::load regenerates them from the same seeds and checks them against the stored
``<key>@probe`` elements -- and the pointwise scorers' gradients above 1024 elements are stored as a strided sample
plus their L2 norm and sum (put_sampled; tests/helpers.py::sampled reproduces the sampling).
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
sys.path.insert(0, os.path.dirname(HERE))

from helpers import probe, sampled, synth_labels  # noqa: E402
from ptranking.data.data_utils import LABEL_TYPE  # noqa: E402
from ptranking.ltr_adhoc.pairwise.ranknet import RankNet  # noqa: E402
from ptranking.ltr_adhoc.listwise.lambdarank import LambdaRank  # noqa: E402
from ptranking.ltr_adhoc.listwise.lambdaloss import LambdaLoss  # noqa: E402
from ptranking.ltr_adhoc.listwise.listnet import ListNet  # noqa: E402
from ptranking.ltr_adhoc.listwise.listmle import ListMLE  # noqa: E402
from ptranking.ltr_adhoc.listwise.approxNDCG import ApproxNDCG  # noqa: E402
import ptranking.ltr_adhoc.listwise.listmle as ref_listmle_mod  # noqa: E402
from ptranking.metric.adhoc.adhoc_metric import torch_ndcg_at_ks, torch_ndcg_at_k  # noqa: E402

ML = LABEL_TYPE.MultiLabel
MSLR_P = np.array([1940952, 1225770, 504958, 69010, 30435], dtype=np.float64)
MSLR_P /= MSLR_P.sum()
MQ_P = np.array([12279, 2001, 931], dtype=np.float64)
MQ_P /= MQ_P.sum()


def put_sampled(out, key, arr):
    """``arr`` in full when small, else its strided sample plus the whole tensor's L2 norm and sum."""
    arr = np.asarray(arr)
    s = sampled(arr)
    out[key] = arr.copy() if s.size == arr.size else s
    if s.size < arr.size:
        out[key + "@norm"] = np.float64(np.sqrt((arr.astype(np.float64) ** 2).sum()))
        out[key + "@sum"] = np.float64(arr.astype(np.float64).sum())


def put_probe(out, key, arr):
    out[key + "@probe"] = probe(arr)


def point_sf_dict(F, **over):
    d = dict(num_features=F, num_layers=5, AF="GE", TL_AF="S", apply_tl_af=True,
             BN=True, bn_type="BN", bn_affine=True, dropout=0.0)
    d.update(over)
    return dict(sf_id="pointsf", opt="Adam", lr=1e-4, pointsf=d)


def list_sf_dict(F, **over):
    d = dict(num_features=F, ff_dims=[16, 32, 24], AF="R", TL_AF="GE", apply_tl_af=False,
             BN=False, bn_type="BN2", bn_affine=False, n_heads=2, encoder_layers=2,
             encoder_type="DASALC", dropout=0.0)
    d.update(over)
    return dict(sf_id="listsf", opt="Adagrad", lr=1e-3, listsf=d)


class _LeafHarness:
    """Calls the reference loss classes' own custom_loss_function on a leaf score tensor.
    The optimizer they step is a throw-away SGD(lr=0) over the leaf, so the reference
    code path (including zero_grad/backward/step) runs unmodified."""

    def __init__(self, cls, model_para):
        sf = point_sf_dict(4)
        if model_para is None:
            self.r = cls(sf_para_dict=sf, gpu=False, device="cpu")
        else:
            self.r = cls(sf_para_dict=sf, model_para_dict=model_para, gpu=False, device="cpu")

    def __call__(self, scores, labels, presort=True):
        s = torch.from_numpy(scores).clone().requires_grad_(True)
        self.r.optimizer = torch.optim.SGD([s], lr=0.0)
        loss = self.r.custom_loss_function(s, torch.from_numpy(labels), presort=presort, label_type=ML)
        return float(loss.detach()), s.grad.detach().numpy().copy()


def loss_fixtures():
    rng = np.random.default_rng(137)
    torch.manual_seed(137)
    out = {}
    shapes = [(1, 8), (3, 50), (2, 256), (1, 1024), (4, 37)]
    cases = []
    for (B, n) in shapes:
        probs = MQ_P if n == 50 else MSLR_P
        y = synth_labels(rng, B, n, probs)
        for tag, s in (("sig", 1.0 / (1.0 + np.exp(-rng.standard_normal((B, n))))),
                       ("wide", 2.5 * rng.standard_normal((B, n)))):
            cases.append((f"B{B}_n{n}_{tag}", s.astype(np.float32), y))
    # an unsorted-label case for the losses that accept presort=False
    y_uns = synth_labels(rng, 3, 40, MSLR_P, presort=False)
    s_uns = rng.standard_normal((3, 40)).astype(np.float32)

    def put(name, case, s, y, loss, grad, **extra):
        key = f"{name}__{case}"
        out[key + "__scores"] = s
        out[key + "__labels"] = y
        out[key + "__loss"] = np.float64(loss)
        out[key + "__grad"] = grad
        for k, v in extra.items():
            out[key + "__" + k] = v

    for case, s, y in cases:
        for sigma in (1.0, 2.0):
            l, g = _LeafHarness(RankNet, dict(model_id="RankNet", sigma=sigma))(s, y)
            put(f"RankNet_sigma{sigma}", case, s, y, l, g)
            l, g = _LeafHarness(LambdaRank, dict(model_id="LambdaRank", sigma=sigma))(s, y)
            put(f"LambdaRank_sigma{sigma}", case, s, y, l, g)
        for lt, k in (("NDCG_Loss2++", 5), ("NDCG_Loss2", 5), ("NDCG_Loss2++", 10 ** 6), ("NDCG_Loss2", 20)):
            kk = min(k, s.shape[1])
            mp = dict(model_id="LambdaLoss", k=kk, sigma=1.0, loss_type=lt, mu=5.0)
            l, g = _LeafHarness(LambdaLoss, mp)(s, y)
            put(f"LambdaLoss_{lt}_k{kk}", case, s, y, l, g)
        if s.shape[0] == 1:  # NDCG_Loss1 only broadcasts for B == 1 (SURVEY B7)
            mp = dict(model_id="LambdaLoss", k=5, sigma=1.0, loss_type="NDCG_Loss1", mu=5.0)
            l, g = _LeafHarness(LambdaLoss, mp)(s, y)
            put("LambdaLoss_NDCG_Loss1_k5", case, s, y, l, g)
        l, g = _LeafHarness(ListNet, None)(s, y)
        put("ListNet", case, s, y, l, g)
        for alpha in (10.0, 1.0):
            l, g = _LeafHarness(ApproxNDCG, dict(model_id="ApproxNDCG", alpha=alpha))(s, y)
            put(f"ApproxNDCG_alpha{alpha}", case, s, y, l, g)
        # ListMLE: capture the permutation the reference drew, by wrapping its own sampler
        captured = {}
        orig = ref_listmle_mod.arg_shuffle_ties

        def spy(batch_rankings, descending=True, device=None):
            p = orig(batch_rankings=batch_rankings, descending=descending, device=device)
            captured["perm"] = p.numpy().astype(np.int32).copy()
            return p

        ref_listmle_mod.arg_shuffle_ties = spy
        try:
            l, g = _LeafHarness(ListMLE, None)(s, y)
        finally:
            ref_listmle_mod.arg_shuffle_ties = orig
        put("ListMLE", case, s, y, l, g, perm=captured["perm"])

    # presort=False branches
    mp = dict(model_id="LambdaLoss", k=7, sigma=1.0, loss_type="NDCG_Loss2++", mu=5.0)
    l, g = _LeafHarness(LambdaLoss, mp)(s_uns, y_uns, presort=False)
    put("LambdaLoss_NDCG_Loss2++_k7_unsorted", "B3_n40_uns", s_uns, y_uns, l, g)
    l, g = _LeafHarness(ApproxNDCG, dict(model_id="ApproxNDCG", alpha=10.0))(s_uns, y_uns, presort=False)
    put("ApproxNDCG_alpha10.0_unsorted", "B3_n40_uns", s_uns, y_uns, l, g)
    l, g = _LeafHarness(RankNet, dict(model_id="RankNet", sigma=1.0))(s_uns, y_uns, presort=False)
    put("RankNet_sigma1.0_unsorted", "B3_n40_uns", s_uns, y_uns, l, g)

    # BCE saturation regime (SURVEY B2): huge score gaps
    s_sat = np.array([[40.0, -35.0, 0.0, 18.0, -17.5, 100.0, -120.0, 3.0]], dtype=np.float32)
    y_sat = np.array([[4, 3, 2, 2, 1, 0, 0, 0]], dtype=np.float32)
    l, g = _LeafHarness(RankNet, dict(model_id="RankNet", sigma=1.0))(s_sat, y_sat)
    put("RankNet_sigma1.0_saturated", "B1_n8_sat", s_sat, y_sat, l, g)
    l, g = _LeafHarness(LambdaRank, dict(model_id="LambdaRank", sigma=1.0))(s_sat, y_sat)
    put("LambdaRank_sigma1.0_saturated", "B1_n8_sat", s_sat, y_sat, l, g)
    np.savez_compressed(os.path.join(HERE, "losses.npz"), **out)
    print("losses.npz:", len(out), "arrays")


def metric_fixtures():
    out = {}
    # the reference's own known-answer vectors (testing/metric/testing_metric.py:43-48)
    sys_l = torch.tensor([[1.0, 1.0, 0.0, 1.0, 0.0, 0.0, 1.0]])
    std_l = torch.tensor([[1.0, 1.0, 1.0, 1.0, 0.0, 0.0, 0.0]])
    out["kat_sys"] = sys_l.numpy(); out["kat_std"] = std_l.numpy()
    out["kat_ks"] = np.arange(1, 8)
    out["kat_ndcg_at_ks"] = torch_ndcg_at_ks(sys_l, std_l, ks=[1, 2, 3, 4, 5, 6, 7]).numpy()
    out["kat_expected_4dp"] = np.array([1.0, 1.0, 0.7654, 0.8048, 0.8048, 0.8048, 0.9349])
    out["kat_ndcg_at_4"] = torch_ndcg_at_k(sys_l, std_l, k=4).numpy()
    rng = np.random.default_rng(137)
    for (B, n) in [(5, 50), (3, 256), (2, 7), (2, 1024)]:
        y = synth_labels(rng, B, n, MSLR_P)
        s = rng.standard_normal((B, n)).astype(np.float32)
        ks = [1, 3, 5, 10, 20, 50]
        ts, ty = torch.from_numpy(s), torch.from_numpy(y)
        _, idx = torch.sort(ts, dim=1, descending=True)
        sys_r = torch.gather(ty, 1, idx)
        key = f"B{B}_n{n}"
        out[key + "__scores"] = s; out[key + "__labels"] = y; out[key + "__ks"] = np.array(ks)
        out[key + "__order"] = idx.numpy().astype(np.int32)
        out[key + "__ndcg_at_ks"] = torch_ndcg_at_ks(sys_r, ty, ks=ks).numpy()
        if n >= 10:
            out[key + "__ndcg_at_10"] = torch_ndcg_at_k(sys_r, ty, k=10).numpy()
    np.savez_compressed(os.path.join(HERE, "metrics.npz"), **out)
    print("metrics.npz:", len(out), "arrays")


def _flatten_sd(prefix, sd, out):
    for k, v in sd.items():
        out[f"{prefix}::{k}"] = v.detach().numpy().copy()


def scorer_fixtures():
    out = {}
    rng = np.random.default_rng(137)
    point_cfgs = {
        "default": dict(),                                                   # GE, S tail, BN affine
        "bn2_relu": dict(AF="R", TL_AF="R", bn_type="BN2", bn_affine=False, num_layers=3),
        "bn2_aff_celu": dict(AF="CE", TL_AF="S", bn_type="BN2", bn_affine=True, num_layers=2),
        "nobn_sig_notl": dict(AF="S", TL_AF="S", BN=False, apply_tl_af=False, num_layers=4),
        "bn_noaff_ge": dict(AF="GE", TL_AF="GE", bn_affine=False, num_layers=2),
    }
    for name, over in point_cfgs.items():
        for (B, n, F) in [(3, 50, 46), (2, 64, 136)]:
            torch.manual_seed(137)
            sf = point_sf_dict(F, **over)
            r = ListNet(sf_para_dict=sf, gpu=False, device="cpu")
            r.init()
            # perturb norm affine params so their gradients are exercised off the init point
            with torch.no_grad():
                for k, p in r.point_sf.named_parameters():
                    if "bn" in k:
                        p.add_(0.1 * torch.randn_like(p))
            X = torch.from_numpy(rng.standard_normal((B, n, F)).astype(np.float32))
            rvec = torch.from_numpy(rng.standard_normal((B, n)).astype(np.float32))
            s = r.forward(X)
            (s * rvec).sum().backward()
            key = f"point_{name}_B{B}_n{n}_F{F}"
            put_probe(out, key + "__X", X.numpy()); out[key + "__dscores"] = rvec.numpy()
            out[key + "__scores"] = s.detach().numpy()
            for k, v in r.point_sf.state_dict().items():
                put_probe(out, f"{key}__param::{k}", v.numpy())
            for k, p in r.point_sf.named_parameters():
                put_sampled(out, f"{key}__grad::{k}", p.grad.numpy())
    for enc in ("DASALC", "AllRank", "AttnDIN"):
        for bn in (False, True):
            torch.manual_seed(137)
            B, n, F = 2, 24, 20
            sf = list_sf_dict(F, encoder_type=enc, BN=bn)
            r = ListNet(sf_para_dict=sf, gpu=False, device="cpu")
            r.init()
            r.eval_mode()   # the tail FFN ignores the configured dropout (SURVEY B10)
            X = torch.from_numpy(rng.standard_normal((B, n, F)).astype(np.float32))
            rvec = torch.from_numpy(rng.standard_normal((B, n)).astype(np.float32))
            s = r.forward(X)
            (s * rvec).sum().backward()
            key = f"list_{enc}_bn{int(bn)}"
            out[key + "__X"] = X.numpy(); out[key + "__dscores"] = rvec.numpy()
            out[key + "__scores"] = s.detach().numpy()
            for part in ("head_ffnns", "encoder", "tail_ffnns"):
                _flatten_sd(f"{key}__param::{part}", r.list_sf[part].state_dict(), out)
                for k, p in r.list_sf[part].named_parameters():
                    out[f"{key}__grad::{part}::{k}"] = p.grad.numpy().copy()
    np.savez_compressed(os.path.join(HERE, "scorers.npz"), **out)
    print("scorers.npz:", len(out), "arrays")


def train_fixtures():
    """Three full train_op steps of the reference (forward, loss, backward, optimizer step)."""
    out = {}
    rng = np.random.default_rng(137)
    runs = [
        ("LambdaRank", LambdaRank, dict(model_id="LambdaRank", sigma=1.0), point_sf_dict(136), (4, 64, 136)),
        ("ListNet", ListNet, None, point_sf_dict(46), (2, 50, 46)),
        ("ApproxNDCG_list", ApproxNDCG, dict(model_id="ApproxNDCG", alpha=10.0),
         list_sf_dict(20), (2, 24, 20)),
        ("LambdaLoss_bn2", LambdaLoss, dict(model_id="LambdaLoss", k=5, sigma=1.0, loss_type="NDCG_Loss2++", mu=5.0),
         point_sf_dict(46, bn_type="BN2", bn_affine=False, AF="R", TL_AF="S", num_layers=3), (3, 50, 46)),
    ]
    for name, cls, mp, sf, (B, n, F) in runs:
        torch.manual_seed(137)
        r = cls(sf_para_dict=sf, gpu=False, device="cpu") if mp is None else \
            cls(sf_para_dict=sf, model_para_dict=mp, gpu=False, device="cpu")
        r.init()
        r.eval_mode()
        is_list = sf["sf_id"] == "listsf"
        if is_list:
            for part in ("head_ffnns", "encoder", "tail_ffnns"):
                _flatten_sd(f"{name}__init::{part}", r.list_sf[part].state_dict(), out)
        else:
            for k, v in r.point_sf.state_dict().items():
                put_probe(out, f"{name}__init::{k}", v.numpy())
        X = rng.standard_normal((3, B, n, F)).astype(np.float32)
        y = np.stack([synth_labels(rng, B, n, MSLR_P) for _ in range(3)])
        losses = []
        for t in range(3):
            loss, _ = r.train_op(torch.from_numpy(X[t]), torch.from_numpy(y[t]), presort=True, label_type=ML)
            losses.append(float(loss.detach()))
        put_probe(out, name + "__X", X); out[name + "__labels"] = y
        out[name + "__losses"] = np.array(losses, dtype=np.float64)
        if is_list:
            for part in ("head_ffnns", "encoder", "tail_ffnns"):
                _flatten_sd(f"{name}__final::{part}", r.list_sf[part].state_dict(), out)
        else:
            _flatten_sd(f"{name}__final", r.point_sf.state_dict(), out)
        Xe = torch.from_numpy(X[0])
        out[name + "__final_scores"] = r.predict(Xe).detach().numpy()
    np.savez_compressed(os.path.join(HERE, "train_steps.npz"), **out)
    print("train_steps.npz:", len(out), "arrays")


if __name__ == "__main__":
    loss_fixtures()
    metric_fixtures()
    scorer_fixtures()
    train_fixtures()
