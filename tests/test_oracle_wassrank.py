"""Pin the oracle's WassRank statements against outputs of the unmodified reference (tests/golden/wassrank.npz, made by
tests/golden/make_golden_wassrank.py): the ATen restatement against the reference's fp32 run, NaN pattern included, and
the float64 log-domain closed form against the reference's float64 run.  Plus the registry entry the drop-in adds."""
import os
import types

import numpy as np
import pytest
import torch

from oracle import closed_form_wassrank as cf
from oracle import ref_port_wassrank as rp
from tests.helpers import GOLDEN, rel_err


def wassrank_cases():
    """[(case, wass_para_dict, arrays)] of tests/golden/wassrank.npz; the case name carries cost type, histogram type,
    lambda and list length (``eg_ST_lam0.1_n256``); the other settings are WassRankParameter's defaults."""
    z = np.load(os.path.join(GOLDEN, "wassrank.npz"))
    heads = sorted({k.split("__")[0] for k in z.files})
    out = []
    for h in heads:
        cost, smooth, lam = h.split("_")[:3]
        para = dict(mode="SinkhornOT", sh_itr=20, lam=float(lam[3:]), smooth_type=smooth, norm_type="BothST",
                    cost_type=cost, non_rele_gap=100, var_penalty=np.e, gain_base=4)
        out.append((h, para, {k.split("__")[1]: z[k] for k in z.files if k.split("__")[0] == h}))
    return out


CASES = wassrank_cases()
IDS = [c for c, _, _ in CASES]


@pytest.mark.parametrize("case,para,d", CASES, ids=IDS)
def test_port_matches_reference_fp32(case, para, d):
    loss, grad = rp.loss_and_grad(torch.from_numpy(d["scores"]), torch.from_numpy(d["labels"]), **para)
    loss, grad = float(loss), grad.numpy()
    want_l, want_g = float(d["loss32"]), d["grad32"]
    assert np.isnan(loss) == np.isnan(want_l)
    assert np.array_equal(np.isfinite(grad), np.isfinite(want_g)) and np.array_equal(np.isnan(grad), np.isnan(want_g))
    if np.isfinite(want_l):
        assert abs(loss - want_l) <= 2e-6 * max(1.0, abs(want_l)), (loss, want_l)
    fin = np.isfinite(want_g)
    if fin.any():
        assert rel_err(grad[fin], want_g[fin]) <= 2e-6


@pytest.mark.parametrize("case,para,d", CASES, ids=IDS)
def test_closed_form_matches_reference_float64(case, para, d):
    loss, grad = cf.wassrank(d["scores"], d["labels"], **para)
    want_l, want_g = float(d["loss64"]), d["grad64"]
    if not np.isfinite(want_l):
        # the reference's per-vector stabilisation underflows even in float64 here (exp(-C/lam) < 1e-308); the
        # log-domain form stays finite
        assert np.isfinite(loss)
        return
    assert abs(loss - want_l) <= 1e-10 * max(1.0, abs(want_l)), (loss, want_l)
    if np.isfinite(want_g).all():
        assert np.abs(grad - want_g).max() <= 1e-10 * max(np.abs(want_g).max(), 1e-300)
    else:       # 'NG' with a minimum score <= 0: that document's mass is 0, log 0 enters the centring, every entry is NaN
        assert np.isnan(want_g).all() and np.isnan(grad).all()


def test_fixture_covers_the_issue_grid():
    heads = {(p["cost_type"], p["smooth_type"], p["lam"], d["scores"].shape[1]) for _, p, d in CASES}
    for cost in ("eg", "p1", "p2", "dg", "ddg"):
        for lam in (0.1, 1.0, 10.0):
            for n in (1, 8, 50, 256, 1024):
                assert (cost, "ST", lam, n) in heads
                if cost in ("eg", "p1"):
                    assert (cost, "NG", lam, n) in heads
    # the reference's default setting is not finite in fp32 on realistic lists: that is what the kernel fixes
    assert not np.isfinite(float(dict((c, d) for c, _, d in CASES)["eg_ST_lam0.1_n1024"]["loss32"]))


def test_install_registers_wassrank():
    import ptranking_b200
    mod = types.SimpleNamespace()
    prev = ptranking_b200.install(module=mod)
    assert mod.WassRank is ptranking_b200.WassRank and prev["WassRank"] is None
    assert len(ptranking_b200.MODELS) == 11


def test_entropic_mode_and_unknown_settings_raise():
    import ptranking_b200
    sf = dict(sf_id="pointsf", opt="Adam", lr=1e-4, pointsf=dict(num_features=4))
    wpd = dict(model_id="WassRank", mode="EntropicOT", sh_itr=20, lam=0.1, smooth_type="ST", norm_type="BothST",
               cost_type="eg", non_rele_gap=100, var_penalty=np.e, gain_base=4)
    with pytest.raises(NotImplementedError, match="EntropicOT"):
        ptranking_b200.WassRank(sf_para_dict=sf, wass_para_dict=wpd, gpu=True, device="cuda:0")
    for bad in (dict(smooth_type="XX"), dict(norm_type="XX"), dict(cost_type="XX")):
        with pytest.raises(NotImplementedError):
            ptranking_b200.WassRank(sf_para_dict=sf, wass_para_dict=dict(wpd, mode="SinkhornOT", **bad), gpu=True,
                                    device="cuda:0")
