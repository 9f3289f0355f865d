"""Pin the oracle against the round-2 reference fixtures (tests/golden/scorers_r2.npz, made by make_golden_r2.py):
activations T / E / LR / SE, and the list scorer at BASELINE config (c)'s real shape (F=136, n=512, 128/256/512, 2 heads,
DASALC, L=6 no-norm and L=3 BN2) -- forward, parameter gradients (strided samples + norms), three ApproxNDCG steps."""
import numpy as np
import pytest
import torch

from oracle import ref_port as rp
from tests.helpers import load, reference_point_outputs, rel_err, sampled

AF_CODES = ["T", "E", "LR", "SE"]
LISTC = {"L6_nonorm": (6, False), "L3_bn2": (3, True)}


@pytest.mark.parametrize("code", AF_CODES)
@pytest.mark.parametrize("shape", [(3, 50, 46), (2, 64, 136)])
def test_point_scorer_activations_port(code, shape):
    z = load("scorers_r2.npz")
    B, n, F = shape
    key = f"point_af{code}_B{B}_n{n}_F{F}"
    s, _ = reference_point_outputs(z, key, F, AF=code, TL_AF=code, num_layers=3)     # checks every parameter gradient
    assert rel_err(s, z[key + "__scores"]) <= 2e-6


def listc_port_state(z, key, L):
    """The fixture stores head / tail and ONE encoder layer (make_clones: all layers start identical) -> RefListScorer names."""
    sd = {}
    for k in z.files:
        if k.startswith(f"{key}__init::head_ffnns::"):
            sd["head." + k.split("::")[2]] = torch.from_numpy(z[k])
        elif k.startswith(f"{key}__init::tail_ffnns::"):
            sd["tail." + k.split("::")[2]] = torch.from_numpy(z[k])
        elif k.startswith(f"{key}__init::encoder_layer::"):
            name = k.split("::")[2].replace("sublayer_cont.norm.", "norm.")
            for l in range(L):
                sd[f"layers.{l}.{name}"] = torch.from_numpy(z[k]).clone()
    return sd


def port_param_name(part, name):
    """reference parameter name (part, key) -> RefListScorer parameter name"""
    if part == "head_ffnns":
        return "head." + name
    if part == "tail_ffnns":
        return "tail." + name
    return name.replace("sublayer_cont.norm.", "norm.")


@pytest.mark.parametrize("tag", list(LISTC))
def test_list_scorer_real_shape_port(tag):
    z = load("scorers_r2.npz")
    L, bn = LISTC[tag]
    key = f"listc_{tag}"
    net = rp.RefListScorer(136, ff_dims=[128, 256, 512], AF="R", TL_AF="GE", apply_tl_af=False, BN=bn, bn_type="BN2",
                           bn_affine=False, n_heads=2, encoder_layers=L, dropout=0.0, encoder_type="DASALC")
    net.load_state_dict(listc_port_state(z, key, L), strict=True)
    net.eval()
    X, y = z[key + "__X"], z[key + "__labels"]
    s = net(torch.from_numpy(X[0]))
    assert rel_err(s.detach().numpy(), z[key + "__scores"]) <= 5e-6
    (s * torch.from_numpy(z[key + "__dscores"])).sum().backward()
    params = dict(net.named_parameters())
    refs = [k for k in z.files if k.startswith(key + "__grad::") and "@" not in k]
    gscale = max(np.abs(z[k]).max() for k in refs)
    for k in refs:
        _, part, name = k.split("::")
        g = params[port_param_name(part, name)].grad.numpy()
        assert np.abs(sampled(g) - z[k].reshape(-1)).max() <= 3e-5 * np.abs(z[k]).max() + 2e-6 * gscale, k
        if k + "@norm" in z.files:      # stored as a sample: the whole tensor's norm too
            assert abs(np.sqrt((g.astype(np.float64) ** 2).sum()) - float(z[k + "@norm"])) <= 3e-5 * float(z[k + "@norm"]) + 2e-6 * gscale, k
    # three ApproxNDCG steps with Adagrad (the listsf default optimizer)
    net.zero_grad()
    opt, _ = rp.make_optimizer(net.parameters(), "Adagrad", 1e-3)
    for t in range(3):
        loss = rp.train_op(net, opt, "ApproxNDCG", torch.from_numpy(X[t]), torch.from_numpy(y[t]), point=False, alpha=10.0)
        ref = float(z[key + "__losses"][t])
        assert abs(float(loss) - ref) <= 3e-5 * max(abs(ref), 1.0), (t, float(loss), ref)
    with torch.no_grad():
        s = net(torch.from_numpy(X[0]))
    assert rel_err(s.numpy(), z[key + "__final_scores"]) <= 5e-5
