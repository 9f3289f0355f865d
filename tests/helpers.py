"""Shared helpers for the parity tests (fixture parsing, tolerances)."""
import os
import re

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

MSLR_P = np.array([1940952, 1225770, 504958, 69010, 30435], dtype=np.float64)
MSLR_P /= MSLR_P.sum()

POINT_CFGS = {
    "default": dict(),
    "bn2_relu": dict(AF="R", TL_AF="R", bn_type="BN2", bn_affine=False, num_layers=3),
    "bn2_aff_celu": dict(AF="CE", TL_AF="S", bn_type="BN2", bn_affine=True, num_layers=2),
    "nobn_sig_notl": dict(AF="S", TL_AF="S", BN=False, apply_tl_af=False, num_layers=4),
    "bn_noaff_ge": dict(AF="GE", TL_AF="GE", bn_affine=False, num_layers=2),
}


def point_cfg(F, **over):
    d = dict(num_features=F, num_layers=5, AF="GE", TL_AF="S", apply_tl_af=True,
             BN=True, bn_type="BN", bn_affine=True, dropout=0.0)
    d.update(over)
    return d


class Fixture(dict):
    """name -> array, with the ``files`` attribute of an ``np.load`` archive."""

    @property
    def files(self):
        return list(self)


def load(name):
    """Arrays of tests/golden/<name>.  For the scorer fixtures the large INPUTS (features, initial weights) are not
    stored: they come from the seeds the fixtures were made with (see _REGEN) and are checked against the stored
    ``<key>@probe`` elements before any test sees them."""
    z = np.load(os.path.join(GOLDEN, name))
    if name not in _REGEN:
        return z
    out = Fixture((k, z[k]) for k in z.files if not k.endswith("@probe"))
    for k, v in _REGEN[name](out).items():
        if not np.array_equal(probe(v), z[k + "@probe"]):
            raise AssertionError(f"{name}: regenerated input {k} differs from the one the fixture was made with")
        out[k] = v
    return out


def probe(arr, count=64):
    """A few evenly spaced elements of ``arr``: stored beside each regenerated input to prove it is the same tensor."""
    flat = np.asarray(arr).reshape(-1)
    return flat[:: max(1, flat.size // count)][:count].copy()


def synth_labels(rng, B, n, probs, presort=True):
    """Graded labels with the given marginals, >= 1 relevant document per query (tests/golden/make_golden.py)."""
    y = rng.choice(len(probs), size=(B, n), p=probs).astype(np.float32)
    for b in range(B):
        if y[b].max() < 1:
            y[b, rng.integers(n)] = float(rng.integers(1, len(probs)))
    if presort:
        y = -np.sort(-y, axis=1)
    return y


def _point_init(F, over, perturb_norm):
    """Initial weights of the reference's pointwise scorer under seed 137: the oracle draws them in the same order."""
    import torch
    from oracle import ref_port as rp
    torch.manual_seed(137)
    net = rp.point_scorer(**point_cfg(F, **over))
    if perturb_norm:        # the fixtures move the norm parameters off their init point
        with torch.no_grad():
            for k, p in net.named_parameters():
                if "bn" in k:
                    p.add_(0.1 * torch.randn_like(p))
    return {k: v.numpy().copy() for k, v in net.state_dict().items()}


def _listc_init(L, bn):
    """Initial weights of the reference's list scorer at config (c)'s shape under seed 137, under the reference's
    names.  The reference builds ONE encoder layer and clones it, so the oracle is built with one layer."""
    import torch
    from oracle import ref_port as rp
    torch.manual_seed(137)
    net = rp.RefListScorer(136, ff_dims=[128, 256, 512], AF="R", TL_AF="GE", apply_tl_af=False, BN=bn, bn_type="BN2",
                           bn_affine=False, n_heads=2, encoder_layers=1, dropout=0.0, encoder_type="DASALC")
    out = {}
    for k, v in net.state_dict().items():
        if k.startswith("head."):
            k = "head_ffnns::" + k[len("head."):]
        elif k.startswith("tail."):
            k = "tail_ffnns::" + k[len("tail."):]
        else:
            k = "encoder_layer::" + k[len("layers.0."):].replace("norm.", "sublayer_cont.norm.")
        out[k] = v.numpy().copy()
    return out


def _regen_scorers(z):
    out = {}
    rng = np.random.default_rng(137)
    for name, over in POINT_CFGS.items():
        for (B, n, F) in [(3, 50, 46), (2, 64, 136)]:
            key = f"point_{name}_B{B}_n{n}_F{F}"
            out.update((f"{key}__param::{k}", v) for k, v in _point_init(F, over, True).items())
            out[key + "__X"] = rng.standard_normal((B, n, F)).astype(np.float32)
            assert np.array_equal(rng.standard_normal((B, n)).astype(np.float32), z[key + "__dscores"])
    return out


def _regen_scorers_r2(z):
    out = {}
    rng = np.random.default_rng(2137)
    for code in ("T", "E", "LR", "SE"):
        for (B, n, F) in [(3, 50, 46), (2, 64, 136)]:
            key = f"point_af{code}_B{B}_n{n}_F{F}"
            out.update((f"{key}__param::{k}", v) for k, v in _point_init(F, dict(AF=code, TL_AF=code, num_layers=3), True).items())
            out[key + "__X"] = rng.standard_normal((B, n, F)).astype(np.float32)
            assert np.array_equal(rng.standard_normal((B, n)).astype(np.float32), z[key + "__dscores"])
    B, n, F = 2, 512, 136
    for tag, L, bn in (("L6_nonorm", 6, False), ("L3_bn2", 3, True)):
        key = f"listc_{tag}"
        out.update((f"{key}__init::{k}", v) for k, v in _listc_init(L, bn).items())
        out[key + "__X"] = rng.standard_normal((3, B, n, F)).astype(np.float32)
        assert np.array_equal(np.stack([synth_labels(rng, B, n, MSLR_P) for _ in range(3)]), z[key + "__labels"])
        assert np.array_equal(rng.standard_normal((B, n)).astype(np.float32), z[key + "__dscores"])
    return out


TRAIN_RUNS = [      # name, pointwise scorer overrides (None = the list scorer, whose small init is stored), (B, n, F)
    ("LambdaRank", dict(), (4, 64, 136)),
    ("ListNet", dict(), (2, 50, 46)),
    ("ApproxNDCG_list", None, (2, 24, 20)),
    ("LambdaLoss_bn2", dict(bn_type="BN2", bn_affine=False, AF="R", TL_AF="S", num_layers=3), (3, 50, 46)),
]


def _regen_train_steps(z):
    out = {}
    rng = np.random.default_rng(137)
    for name, over, (B, n, F) in TRAIN_RUNS:
        if over is not None:
            out.update((f"{name}__init::{k}", v) for k, v in _point_init(F, over, False).items())
        out[name + "__X"] = rng.standard_normal((3, B, n, F)).astype(np.float32)
        assert np.array_equal(np.stack([synth_labels(rng, B, n, MSLR_P) for _ in range(3)]), z[name + "__labels"])
    return out


_REGEN = {"scorers.npz": _regen_scorers, "scorers_r2.npz": _regen_scorers_r2, "train_steps.npz": _regen_train_steps}


def check_fixture(z, key, full, tol, norm_rtol):
    """A tensor the test computed against the fixture's copy of the reference's ``key`` -- all of it, or for large
    tensors its strided sample (sampled()) plus the whole tensor's L2 norm: every stored element within ``tol``, the
    norm within ``norm_rtol``."""
    full = np.asarray(full)
    ref = z[key]
    err = float(np.abs(sampled(full).reshape(ref.shape) - ref).max())
    assert err <= tol, (key, err, tol)
    if key + "@norm" in z.files:
        norm, norm_ref = float(np.sqrt((full.astype(np.float64) ** 2).sum())), float(z[key + "@norm"])
        assert abs(norm - norm_ref) <= norm_rtol * norm_ref, (key, norm, norm_ref)


def reference_point_outputs(z, key, F, **over):
    """Scores and full-size parameter gradients of the reference's pointwise scorer on fixture ``key``'s inputs:
    the oracle's (the same ATen ops; bit-identical where the fixtures were made), each gradient checked against
    what the fixture stores of the reference's own."""
    import torch
    from oracle import ref_port as rp
    net = rp.point_scorer(**point_cfg(F, **over))
    prefix = key + "__param::"
    net.load_state_dict({k[len(prefix):]: torch.from_numpy(z[k]) for k in z.files if k.startswith(prefix)})
    s = rp.point_forward(net, torch.from_numpy(z[key + "__X"]))
    (s * torch.from_numpy(z[key + "__dscores"])).sum().backward()
    names = {n + "." for n, _ in net.named_modules()}
    gscale = max(np.abs(z[f"{key}__grad::{k}"]).max() for k, _ in net.named_parameters())
    grads = {}
    for k, p in net.named_parameters():
        ref = z[f"{key}__grad::{k}"]
        tol = 2e-5 * max(np.abs(ref).max(), 1e-3)
        layer = k.split(".")[0]
        if k.endswith(".bias") and any(n.startswith(f"bn_{layer[len('ff_'):]}.") for n in names):
            # a Linear bias feeding a norm has an exactly-zero true gradient: both sides hold fp32 rounding noise, which
            # follows the CPU's vector width (AVX2 vs AVX-512 kernels), hence a floor relative to the net's gradient scale
            tol += 1e-6 * gscale
        check_fixture(z, f"{key}__grad::{k}", p.grad.numpy(), tol, 2e-5)
        grads[k] = p.grad.numpy().copy()
    return s.detach().numpy(), grads


def loss_cases():
    """-> list of (loss_key, case, dict(scores, labels, loss, grad[, perm]))."""
    z = load("losses.npz")
    groups = {}
    for k in z.files:
        head, case, field = k.split("__")
        groups.setdefault((head, case), {})[field] = z[k]
    return [(h, c, v) for (h, c), v in sorted(groups.items())]


def parse_loss_key(head):
    """'LambdaLoss_NDCG_Loss2++_k5_unsorted' -> (name, params, presort)."""
    presort = True
    if head.endswith("_unsorted"):
        presort, head = False, head[: -len("_unsorted")]
    if head.endswith("_saturated"):
        head = head[: -len("_saturated")]
    name = head.split("_")[0]
    params = {}
    m = re.search(r"sigma([0-9.]+)", head)
    if m:
        params["sigma"] = float(m.group(1))
    m = re.search(r"alpha([0-9.]+)", head)
    if m:
        params["alpha"] = float(m.group(1))
    if name == "LambdaLoss":
        m = re.match(r"LambdaLoss_(NDCG_Loss(?:1|2\+\+|2))_k(\d+)", head)
        params.update(loss_type=m.group(1), k=int(m.group(2)), sigma=1.0, mu=5.0)
    return name, params, presort


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    denom = max(np.abs(b).max(), 1e-30)
    return float(np.abs(a - b).max() / denom)


def sibling_cases():
    """tests/golden/siblings.npz -> list of (loss_key, case, dict) for RankMSE / RankCosine / STListNet / SoftRank."""
    z = load("siblings.npz")
    groups = {}
    for k in z.files:
        head, case, field = k.split("__")
        if head in ("sinkstep", "sinkhorn"):
            continue
        groups.setdefault((head, case), {})[field] = z[k]
    return [(h, c, v) for (h, c), v in sorted(groups.items())]


def sinkhorn_cases(kind):
    z = load("siblings.npz")
    groups = {}
    for k in z.files:
        head, case, field = k.split("__")
        if head == kind:
            groups.setdefault(case, {})[field] = z[k]
    return sorted(groups.items())


def parse_sibling_key(head):
    """'SoftRank_delta2.0_kNone' -> ('SoftRank', dict(delta=2.0, top_k=None))."""
    name = head.split("_")[0]
    params = {}
    m = re.search(r"_T([0-9.]+)", head)
    if m:
        params["temperature"] = float(m.group(1))
    m = re.search(r"delta([0-9.]+)_k(\w+)", head)
    if m:
        params["delta"] = float(m.group(1))
        params["top_k"] = None if m.group(2) == "None" else int(m.group(2))
    return name, params


def sampled(arr, limit=1024, target=512):
    """Flattened tensor, or every k-th element of it when it has more than ``limit`` elements (k = size // target) --
    the storage rule of tests/golden/make_golden*.py for large gradients / weights (put_sampled)."""
    flat = np.asarray(arr).reshape(-1)
    if flat.size <= limit:
        return flat.copy()
    return flat[:: flat.size // target].copy()
