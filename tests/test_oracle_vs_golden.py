"""Pin the oracle (oracle/ref_port.py, oracle/closed_form.py) against outputs of the
unmodified reference (tests/golden/*.npz, made by tests/golden/make_golden.py) and the
reference's own metric known-answer vectors (testing/metric/testing_metric.py:43-48)."""
import numpy as np
import pytest
import torch

from oracle import closed_form as cf
from oracle import ref_port as rp
from tests.helpers import POINT_CFGS, load, loss_cases, parse_loss_key, point_cfg, reference_point_outputs, rel_err  # noqa: F401

CASES = loss_cases()


@pytest.mark.parametrize("head,case,d", CASES, ids=[f"{h}-{c}" for h, c, _ in CASES])
def test_port_matches_reference_loss_and_grad(head, case, d):
    name, params, presort = parse_loss_key(head)
    s, y = torch.from_numpy(d["scores"]), torch.from_numpy(d["labels"])
    kw = dict(params)
    if name in ("LambdaLoss", "ApproxNDCG"):
        kw["presort"] = presort
    if name == "ListMLE":
        kw["perm"] = torch.from_numpy(d["perm"].astype(np.int64))
    loss, grad = rp.loss_and_grad(name, s, y, **kw)
    assert abs(float(loss) - float(d["loss"])) <= 2e-6 * max(1.0, abs(float(d["loss"])))
    assert rel_err(grad.numpy(), d["grad"]) <= 2e-6


@pytest.mark.parametrize("head,case,d", CASES, ids=[f"{h}-{c}" for h, c, _ in CASES])
def test_closed_form_matches_reference(head, case, d):
    name, params, presort = parse_loss_key(head)
    s, y = d["scores"], d["labels"]
    if "saturated" in head:
        pytest.skip("float64 closed form and fp32 ATen legitimately differ in BCE saturation")
    if name == "RankNet":
        loss, grad = cf.ranknet(s, y, **params)
    elif name == "LambdaRank":
        loss, grad = cf.lambdarank(s, y, **params)
    elif name == "LambdaLoss":
        loss, grad = cf.lambdaloss(s, y, presort=presort, **params)
    elif name == "ListNet":
        loss, grad = cf.listnet(s, y)
    elif name == "ListMLE":
        loss, grad = cf.listmle(s, d["perm"])
    elif name == "ApproxNDCG":
        loss, grad = cf.approxndcg(s, y, presort=presort, **params)
    # the reference is fp32 with O(n^2)-term sums: 2e-5 covers its own rounding
    assert abs(loss - float(d["loss"])) <= 2e-5 * max(1.0, abs(float(d["loss"])))
    assert rel_err(grad, d["grad"]) <= 5e-5


def test_metric_known_answers():
    z = load("metrics.npz")
    got = rp.ndcg_at_ks(torch.from_numpy(z["kat_sys"]), torch.from_numpy(z["kat_std"]), list(z["kat_ks"]))
    assert np.array_equal(got.numpy(), z["kat_ndcg_at_ks"])
    assert np.allclose(got.numpy()[0], z["kat_expected_4dp"], atol=5e-5)   # the comment vector in the reference test
    assert np.array_equal(rp.ndcg_at_k(torch.from_numpy(z["kat_sys"]), torch.from_numpy(z["kat_std"]), 4).numpy(),
                          z["kat_ndcg_at_4"])


@pytest.mark.parametrize("key", ["B5_n50", "B3_n256", "B2_n7", "B2_n1024"])
def test_metric_ndcg_fixtures(key):
    z = load("metrics.npz")
    s, y, ks = z[key + "__scores"], z[key + "__labels"], [int(k) for k in z[key + "__ks"]]
    got = rp.evaluator_ndcg_at_ks(torch.from_numpy(s), torch.from_numpy(y), ks, presort=True)
    assert np.array_equal(got.numpy(), z[key + "__ndcg_at_ks"])            # same ATen ops -> bit equal
    cf_vals, order = cf.ndcg_at_ks(s, y, ks)
    assert np.array_equal(order.astype(np.int32), z[key + "__order"])      # integer ranks exact
    assert np.allclose(cf_vals, z[key + "__ndcg_at_ks"], rtol=0, atol=2e-6)


def _load_sd(z, prefix):
    return {k[len(prefix) + 2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith(prefix + "::")}


@pytest.mark.parametrize("name", list(POINT_CFGS))
@pytest.mark.parametrize("shape", [(3, 50, 46), (2, 64, 136)])
def test_point_scorer_port(name, shape):
    z = load("scorers.npz")
    B, n, F = shape
    key = f"point_{name}_B{B}_n{n}_F{F}"
    s, _ = reference_point_outputs(z, key, F, **POINT_CFGS[name])      # checks every parameter gradient
    assert rel_err(s, z[key + "__scores"]) <= 2e-6


def list_sd_to_port(z, key):
    """Map the reference's three state_dicts onto oracle.ref_port.RefListScorer names."""
    sd = {}
    for k in z.files:
        if not k.startswith(key + "__param::"):
            continue
        _, part, name = k.split("::")
        v = torch.from_numpy(z[k])
        if part == "head_ffnns":
            sd["head." + name] = v
        elif part == "tail_ffnns":
            sd["tail." + name] = v
        else:
            name = name.replace("sublayer_cont.norm.", "norm.")
            name = name.replace("sublayer_cont.0.norm.", "norm0.").replace("sublayer_cont.1.norm.", "norm1.")
            name = name.replace("fc.w1.", "w1.").replace("fc.w2.", "w2.")
            if name.startswith("norm."):
                name = "final_norm." + name[len("norm."):]
            sd[name] = v
    return sd


@pytest.mark.parametrize("enc", ["DASALC", "AllRank", "AttnDIN"])
@pytest.mark.parametrize("bn", [0, 1])
def test_list_scorer_port(enc, bn):
    z = load("scorers.npz")
    key = f"list_{enc}_bn{bn}"
    net = rp.RefListScorer(20, ff_dims=[16, 32, 24], AF="R", TL_AF="GE", apply_tl_af=False, BN=bool(bn),
                           bn_type="BN2", bn_affine=False, n_heads=2, encoder_layers=2, dropout=0.0,
                           encoder_type=enc)
    missing = net.load_state_dict(list_sd_to_port(z, key), strict=True)
    net.eval()
    s = net(torch.from_numpy(z[key + "__X"]))
    assert rel_err(s.detach().numpy(), z[key + "__scores"]) <= 5e-6


def test_p_ap_nerr_known_answers_and_fixtures():
    """P / AP / nERR restatements against the reference's own known answers (testing_metric.py:20-60)
    and against reference outputs on seeded rankings."""
    z = load("metrics2.npz")
    for name in ("ap1", "ap2", "ap3"):
        got = rp.ap_at_ks(torch.from_numpy(z[name + "__sys"]), torch.from_numpy(z[name + "__std"]), list(z[name + "__ks"]))
        assert np.array_equal(got.numpy(), z[name + "__ap"])
        assert np.allclose(got.numpy()[0], z[name + "__expect4dp"], atol=5e-5)
    got = rp.nerr_at_ks(torch.from_numpy(z["nerr__sys"]), torch.from_numpy(z["nerr__std"]), [1, 2, 3])
    assert np.array_equal(got.numpy(), z["nerr__val"]) and np.allclose(got.numpy()[0], z["nerr__expect4dp"], atol=5e-5)
    for key in ("B5_n50", "B3_n256", "B2_n7", "B2_n1024"):
        s, y = torch.from_numpy(z[key + "__scores"]), torch.from_numpy(z[key + "__labels"])
        ks = [int(k) for k in z[key + "__ks"]]
        nd, ne, ap, p = rp.evaluator_metrics_at_ks(s, y, ks, presort=True, max_label=4.0)
        assert np.array_equal(nd.numpy(), z[key + "__ndcg"]) and np.array_equal(ne.numpy(), z[key + "__nerr4"])
        assert np.array_equal(ap.numpy(), z[key + "__ap"]) and np.array_equal(p.numpy(), z[key + "__p"])
        ne2 = rp.evaluator_metrics_at_ks(s, y, ks, presort=True, max_label=None)[1]
        assert np.array_equal(ne2.numpy(), z[key + "__nerrNone"])
