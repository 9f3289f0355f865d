"""Round-2 parity gaps (VERDICT r1): activations T / E / LR / SE, the list scorer at BASELINE config (c)'s real shape
against fixtures from the unmodified reference (tests/golden/scorers_r2.npz), one full-width pointwise batch
(64 x 256 x 136, default BN scorer) against the oracle run on this box's CPU."""
import numpy as np
import pytest
import torch

from oracle import ref_port as rp
from tests.helpers import load, point_cfg, reference_point_outputs, rel_err, sampled
from tests.test_oracle_r2 import AF_CODES, LISTC
from tests.test_gpu_scorer import _point_ranker, _sd

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GRAD_TOL = 3e-5


@pytest.mark.parametrize("code", AF_CODES)
@pytest.mark.parametrize("shape", [(3, 50, 46), (2, 64, 136)])
def test_point_scorer_activations(code, shape):
    z = load("scorers_r2.npz")
    B, n, F = shape
    key = f"point_af{code}_B{B}_n{n}_F{F}"
    r = _point_ranker("ListNet", F, AF=code, TL_AF=code, num_layers=3)
    r.point_sf.load_state_dict(_sd(z, key + "__param"))
    r.eval_mode()
    s = r.forward(torch.from_numpy(z[key + "__X"]).to(DEV))
    assert rel_err(s.detach().cpu().numpy(), z[key + "__scores"]) <= 1e-5
    (s * torch.from_numpy(z[key + "__dscores"]).to(DEV)).sum().backward()
    _, ref_grads = reference_point_outputs(z, key, F, AF=code, TL_AF=code, num_layers=3)
    gscale = max(np.abs(g).max() for g in ref_grads.values())
    for k, p in r.point_sf.named_parameters():
        ref = ref_grads[k]
        err = np.abs(p.grad.cpu().numpy() - ref).max()
        assert err <= 2e-5 * np.abs(ref).max() + 1e-6 * gscale + 1e-9, (k, err, np.abs(ref).max(), gscale)


def _listc_ranker(L, bn):
    import ptranking_b200
    d = dict(num_features=136, ff_dims=[128, 256, 512], AF="R", TL_AF="GE", apply_tl_af=False, BN=bn, bn_type="BN2",
             bn_affine=False, n_heads=2, encoder_layers=L, encoder_type="DASALC", dropout=0.0)
    sf = dict(sf_id="listsf", opt="Adagrad", lr=1e-3, listsf=d)
    r = ptranking_b200.ApproxNDCG(sf_para_dict=sf, model_para_dict=dict(model_id="ApproxNDCG", alpha=10.0), gpu=True, device=DEV)
    r.init()
    return r


def _load_listc(r, z, key, L):
    for part in ("head_ffnns", "tail_ffnns"):
        sd = {k.split("::")[2]: torch.from_numpy(z[k]) for k in z.files if k.startswith(f"{key}__init::{part}::")}
        r.list_sf[part].load_state_dict(sd)
    layer = {k.split("::")[2]: torch.from_numpy(z[k]) for k in z.files if k.startswith(f"{key}__init::encoder_layer::")}
    r.list_sf["encoder"].load_state_dict({f"layers.{l}.{k}": v for l in range(L) for k, v in layer.items()})


@pytest.mark.parametrize("tag", list(LISTC))
def test_list_scorer_real_shape(tag):
    """F=136, n=512, ff_dims 128/256/512, 2 heads (d=68), DASALC: column-tiled rows_gemm_tc, column-blocked wgrad_tc,
    split accumulators, MN-major operands -- against the reference's own outputs."""
    from ptranking_b200 import LABEL_TYPE
    z = load("scorers_r2.npz")
    L, bn = LISTC[tag]
    key = f"listc_{tag}"
    r = _listc_ranker(L, bn)
    _load_listc(r, z, key, L)
    r.eval_mode()
    X, y = z[key + "__X"], z[key + "__labels"]
    # float64 truth and the fp32 reference's own distance from it, from the oracle (pinned to these fixtures by
    # tests/test_oracle_r2.py) in double precision on this box's CPU
    import copy
    from tests.test_oracle_r2 import listc_port_state, port_param_name
    net = rp.RefListScorer(136, ff_dims=[128, 256, 512], AF="R", TL_AF="GE", apply_tl_af=False, BN=bn, bn_type="BN2",
                           bn_affine=False, n_heads=2, encoder_layers=L, dropout=0.0, encoder_type="DASALC")
    net.load_state_dict(listc_port_state(z, key, L), strict=True)
    net.eval()
    net64 = copy.deepcopy(net).double()
    w = torch.from_numpy(z[key + "__dscores"])
    s32 = net(torch.from_numpy(X[0])); (s32 * w).sum().backward()
    s64 = net64(torch.from_numpy(X[0]).double()); (s64 * w.double()).sum().backward()
    s64n = s64.detach().numpy()
    g64_base = {k: p.grad.clone() for k, p in net64.named_parameters()}
    # How discontinuous is the gradient at this point?  ReLU kinks: in EXACT arithmetic (float64) a relative perturbation of
    # 1e-6 of the input -- below the fp32 resolution of the forward pass -- flips pre-activations that sit within rounding of
    # zero and moves some gradients by a fixed jump (4.5 % of head.ff_3.weight for the BN2 fixture).  No fp32 implementation can
    # be asked to land on the reference's side of such a kink; the jump size is the floor of the comparison.
    kink = {k: torch.zeros_like(v) for k, v in g64_base.items()}
    if bn:
        for seed in range(3):
            gen = torch.Generator().manual_seed(seed)
            Xp = torch.from_numpy(X[0]).double()
            Xp = Xp * (1.0 + 1e-6 * torch.randn(Xp.shape, generator=gen, dtype=torch.float64))
            net64.zero_grad()
            (net64(Xp) * w.double()).sum().backward()
            for k, p_ in net64.named_parameters():
                kink[k] = torch.maximum(kink[k], (p_.grad - g64_base[k]).abs())
        for k, p_ in net64.named_parameters():
            p_.grad = g64_base[k]
    ref_fwd = rel_err(z[key + "__scores"], s64n)
    s = r.forward(torch.from_numpy(X[0]).to(DEV))
    e_fwd, e_fwd64 = rel_err(s.detach().cpu().numpy(), z[key + "__scores"]), rel_err(s.detach().cpu().numpy(), s64n)
    # 3xTF32 carries a per-product error of 2^-21 against 2^-24 for an fp32 FMA chain: through 14 Linear layers and 2 L attention
    # contractions in sequence the scores stay within 2e-5 of the reference (1e-5 for the 3-layer encoder) and within 5x the
    # reference's own distance from float64
    assert e_fwd <= (2e-5 if L > 3 else 1e-5), (e_fwd, e_fwd64, ref_fwd)
    assert e_fwd64 <= max(1e-5, 5.0 * ref_fwd), (e_fwd64, ref_fwd)
    (s * w.to(DEV)).sum().backward()
    refs = [k for k in z.files if k.startswith(key + "__grad::") and "@" not in k]
    gscale = max(np.abs(z[k]).max() for k in refs)
    p32, p64 = dict(net.named_parameters()), dict(net64.named_parameters())
    checked, bad, worst = 0, [], (0.0, 0.0)
    for part in ("head_ffnns", "encoder", "tail_ffnns"):
        for name, p in r.list_sf[part].named_parameters():
            k = f"{key}__grad::{part}::{name}"
            g = p.grad.cpu().numpy().astype(np.float64) if p.grad is not None else np.zeros(p.shape)
            pn = port_param_name(part, name)
            g32, g64 = p32[pn].grad.numpy().astype(np.float64), p64[pn].grad.numpy()
            assert np.abs(sampled(g32) - z[k]).max() <= 1e-4 * np.abs(z[k]).max() + 2e-6 * gscale      # oracle == fixture (sanity)
            # Per-query BN2 over nearly constant channels (dead ReLU units) divides by sqrt(var + 1e-5) ~ 3e-3: rounding noise in
            # the forward pass is amplified ~300x in these gradients.  The fp32 reference itself sits 1e-3 from float64 here, so
            # the bar is float64 truth: within GRAD_TOL, or within 8x the reference's own distance from it.
            e_ours, e_ref = np.abs(g - g64).max(), np.abs(g32 - g64).max()
            e_kink = float(kink[pn].max())
            if e_ours > max(GRAD_TOL * np.abs(g64).max() + 2e-6 * gscale + 1e-9, 8.0 * e_ref, 1.5 * e_kink):
                bad.append((part, name, float(e_ours / max(np.abs(g64).max(), 1e-30)), float(e_ref / max(np.abs(g64).max(), 1e-30))))
            worst = max(worst, (float(e_ours / gscale), float(e_ref / gscale)))
            checked += 1
    assert not bad, bad
    assert checked == len(refs)
    print(f"[{tag}] scores: vs reference {e_fwd:.2e}, vs float64 {e_fwd64:.2e} (reference vs float64 {ref_fwd:.2e}); "
          f"worst parameter gradient / gradient scale: ours {worst[0]:.2e}, reference {worst[1]:.2e}")
    # three ApproxNDCG train steps (fused Adagrad over the flat bucket) from the reference's initial weights
    r.grad_bucket.zero()
    # The first step sees the fixture's weights: its loss must match.  Adagrad's first update is lr * g / |g| -- a sign step --
    # so elements whose gradient is rounding noise move by +-lr on a coin flip, and with 0.9 M parameters the trajectories
    # separate: later losses and the final scores agree to 2e-3 / 2e-2, the weights to a few lr.
    for t in range(3):
        loss, stop = r.train_op(torch.from_numpy(X[t]).to(DEV), torch.from_numpy(y[t]).to(DEV), presort=True, label_type=LABEL_TYPE.MultiLabel)
        ref = float(z[key + "__losses"][t])
        tol = 3e-5 if t == 0 else 2e-3
        assert not stop and abs(float(loss.detach()) - ref) <= tol * max(abs(ref), 1.0), (t, float(loss.detach()), ref)
    s = r.predict(torch.from_numpy(X[0]).to(DEV)).detach().cpu().numpy()
    assert rel_err(s, z[key + "__final_scores"]) <= 2e-2
    for part in ("head_ffnns", "encoder", "tail_ffnns"):
        for name, v in r.list_sf[part].state_dict().items():
            k = f"{key}__final::{part}::{name}"
            assert np.abs(sampled(v.cpu().numpy()) - z[k]).max() <= 4 * 3 * 1e-3 + 2e-4 * max(np.abs(z[k]).max(), 1e-3), (part, name)
    # nDCG@10 on the final scores: integer ranks exact
    from ptranking_b200 import ops
    _, order = ops.ndcg_at_ks(torch.from_numpy(s).to(DEV), torch.from_numpy(y[0]).to(DEV), [10], presort=True, return_order=True)
    own_order = np.argsort(-s, axis=1, kind="stable")
    assert (order.cpu().numpy() == own_order).all()          # the device ranking is the stable descending sort of the device scores


def test_full_width_point_batch_matches_oracle():
    """One full-width batch of the headline configuration -- 64 queries x 256 docs x 136 features, default scorer
    (5 x 100 GELU, batch-level BN affine, sigmoid tail), LambdaRank -- forward, every parameter gradient and three Adam
    steps against the oracle (the reference's ATen ops) on this box's CPU."""
    from ptranking_b200 import LABEL_TYPE
    B, n, F = 64, 256, 136
    torch.manual_seed(137)
    r = _point_ranker("LambdaRank", F, dict(model_id="LambdaRank", sigma=1.0))
    net = rp.point_scorer(**point_cfg(F))
    net.load_state_dict({k: v.cpu() for k, v in r.point_sf.state_dict().items()})
    net.eval(); r.eval_mode()
    rng = np.random.default_rng(137)
    p = np.array([1940952, 1225770, 504958, 69010, 30435], dtype=np.float64); p /= p.sum()
    Xs = [torch.from_numpy(rng.standard_normal((B, n, F), dtype=np.float32)) for _ in range(3)]
    ys = []
    for _ in range(3):
        y = rng.choice(5, size=(B, n), p=p).astype(np.float32)
        y[:, 0] = np.maximum(y[:, 0], 1.0)
        ys.append(torch.from_numpy(-np.sort(-y, axis=1)))
    # forward + parameter gradients under the LambdaRank loss
    s_ref = rp.point_forward(net, Xs[0])
    loss_ref = rp.lambdarank_loss(s_ref, ys[0], sigma=1.0)
    loss_ref.backward()
    s = r.forward(Xs[0].to(DEV))
    assert rel_err(s.detach().cpu().numpy(), s_ref.detach().numpy()) <= 1e-5
    from ptranking_b200 import ops
    loss = ops.rank_loss("LambdaRank", s, ys[0].to(DEV), sigma=1.0)
    r.grad_bucket.zero()
    loss.backward()
    assert abs(float(loss) - float(loss_ref)) <= 2e-5 * abs(float(loss_ref))
    ref_grads = {k: p_.grad.numpy() for k, p_ in net.named_parameters()}
    gscale = max(np.abs(g).max() for g in ref_grads.values())
    for k, p_ in r.point_sf.named_parameters():
        err = np.abs(p_.grad.cpu().numpy() - ref_grads[k]).max()
        assert err <= 3e-5 * np.abs(ref_grads[k]).max() + 2e-6 * gscale + 1e-9, (k, err, np.abs(ref_grads[k]).max(), gscale)
    # three full train steps
    net.zero_grad()
    opt, _ = rp.make_optimizer(net.parameters(), "Adam", 1e-4)
    init = {k: v.clone() for k, v in net.state_dict().items()}
    for t in range(3):
        l_ref = rp.train_op(net, opt, "LambdaRank", Xs[t], ys[t], sigma=1.0)
        l, stop = r.train_op(Xs[t].to(DEV), ys[t].to(DEV), presort=True, label_type=LABEL_TYPE.MultiLabel)
        assert not stop and abs(float(l) - float(l_ref)) <= 2e-5 * abs(float(l_ref)), (t, float(l), float(l_ref))
    for k, v in r.point_sf.state_dict().items():
        upd_ref = (net.state_dict()[k] - init[k]).numpy()
        upd = v.cpu().numpy() - init[k].numpy()
        # Adam normalises the step.  A Linear bias that feeds a BatchNorm has an exactly-zero true gradient: the reference holds
        # rounding noise there (comparable to its weight-decay term over 16384 rows), this path an exact zero, so Adam moves
        # those elements by +-lr on a coin flip in the reference; everything else agrees to 5 % of the step.
        if k.startswith("ff_") and k.endswith(".bias"):
            continue        # (the scores do not depend on these biases at all: BatchNorm removes every per-channel shift)
        assert np.abs(upd - upd_ref).max() <= 0.05 * max(np.abs(upd_ref).max(), 1e-7) + 1e-7, k
    with torch.no_grad():
        s_ref = rp.point_forward(net, Xs[0]).numpy()
    s = r.predict(Xs[0].to(DEV)).detach().cpu().numpy()
    assert rel_err(s, s_ref) <= 2e-5
    _, order = ops.ndcg_at_ks(torch.from_numpy(s).to(DEV), ys[0].to(DEV), [10], presort=True, return_order=True)
    nd = ops.ndcg_at_ks(torch.from_numpy(s_ref).to(DEV), ys[0].to(DEV), [10], presort=True).cpu().numpy()
    nd_ref = rp.evaluator_ndcg_at_ks(torch.from_numpy(s_ref), ys[0], [10], presort=True).numpy()
    assert np.abs(nd - nd_ref).max() <= 1e-6               # same scores -> identical nDCG@10
