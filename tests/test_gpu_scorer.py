"""GPU parity of the pointwise stacked-FF scorer (forward, parameter gradients, full train steps)
against tensors the unmodified reference produced (tests/golden/scorers.npz, train_steps.npz)."""
import numpy as np
import pytest
import torch

from tests.helpers import POINT_CFGS, load, point_cfg, reference_point_outputs, rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _sd(z, prefix):
    return {k[len(prefix) + 2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith(prefix + "::")}


def _point_ranker(cls, F, model_para=None, **over):
    import ptranking_b200
    sf = dict(sf_id="pointsf", opt="Adam", lr=1e-4, pointsf=point_cfg(F, **over))
    C = getattr(ptranking_b200, cls)
    r = C(sf_para_dict=sf, gpu=True, device=DEV) if model_para is None else \
        C(sf_para_dict=sf, model_para_dict=model_para, gpu=True, device=DEV)
    r.init()
    return r


@pytest.mark.parametrize("name", list(POINT_CFGS))
@pytest.mark.parametrize("shape", [(3, 50, 46), (2, 64, 136)])
def test_point_scorer_forward_backward(name, shape):
    z = load("scorers.npz")
    B, n, F = shape
    key = f"point_{name}_B{B}_n{n}_F{F}"
    r = _point_ranker("ListNet", F, **POINT_CFGS[name])
    r.point_sf.load_state_dict(_sd(z, key + "__param"))       # the reference's own checkpoint keys
    r.eval_mode()
    X = torch.from_numpy(z[key + "__X"]).to(DEV)
    s = r.forward(X)
    assert s.shape == (B, n)
    assert rel_err(s.detach().cpu().numpy(), z[key + "__scores"]) <= 1e-5
    (s * torch.from_numpy(z[key + "__dscores"]).to(DEV)).sum().backward()
    _, ref_grads = reference_point_outputs(z, key, F, **POINT_CFGS[name])
    gscale = max(np.abs(g).max() for g in ref_grads.values())
    for k, p in r.point_sf.named_parameters():
        ref = ref_grads[k]
        err = np.abs(p.grad.cpu().numpy() - ref).max()
        # Linear biases feeding a norm have an exactly-zero true gradient: both sides hold pure rounding
        # noise there, hence the floor relative to the net's gradient scale
        assert err <= 2e-5 * np.abs(ref).max() + 1e-6 * gscale + 1e-9, (k, err, np.abs(ref).max(), gscale)


def test_state_dict_keys_match_reference_checkpoint_format():
    z = load("scorers.npz")
    for name, over in POINT_CFGS.items():
        key = f"point_{name}_B3_n50_F46"
        r = _point_ranker("ListNet", 46, **over)
        assert sorted(r.point_sf.state_dict().keys()) == sorted(_sd(z, key + "__param").keys())


RUNS = {
    "LambdaRank": ("LambdaRank", dict(model_id="LambdaRank", sigma=1.0), dict(), 136),
    "ListNet": ("ListNet", None, dict(), 46),
    "LambdaLoss_bn2": ("LambdaLoss", dict(model_id="LambdaLoss", k=5, sigma=1.0, loss_type="NDCG_Loss2++", mu=5.0),
                       dict(bn_type="BN2", bn_affine=False, AF="R", TL_AF="S", num_layers=3), 46),
}


@pytest.mark.parametrize("run", list(RUNS))
def test_three_train_steps_match_reference(run):
    """forward + loss + backward + Adam step, three times, from the reference's initial weights."""
    from ptranking_b200 import LABEL_TYPE
    z = load("train_steps.npz")
    cls, mp, over, F = RUNS[run]
    r = _point_ranker(cls, F, mp, **over)
    r.point_sf.load_state_dict(_sd(z, run + "__init"))
    r.eval_mode()                                   # fixtures were made with dropout off
    X, y = z[run + "__X"], z[run + "__labels"]
    for t in range(3):
        loss, stop = r.train_op(torch.from_numpy(X[t]).to(DEV), torch.from_numpy(y[t]).to(DEV),
                                presort=True, label_type=LABEL_TYPE.MultiLabel)
        ref = z[run + "__losses"][t]
        assert not stop and abs(float(loss) - ref) <= 2e-5 * max(abs(ref), 1.0), (t, float(loss), ref)
    final = _sd(z, run + "__final")
    for k, v in r.point_sf.state_dict().items():
        # Adam normalises the step, so weights move by ~lr regardless of gradient scale:
        # compare the update itself, not just the weight
        init = z[f"{run}__init::{k}"]
        upd_ref = final[k].numpy() - init
        upd = v.cpu().numpy() - init
        # (an element whose gradient is dominated by fp32 rounding noise moves by a different fraction of lr: 5 %)
        assert np.abs(upd - upd_ref).max() <= 0.05 * max(np.abs(upd_ref).max(), 1e-7) + 1e-7, k
    s = r.predict(torch.from_numpy(X[0]).to(DEV)).detach().cpu().numpy()
    assert rel_err(s, z[run + "__final_scores"]) <= 2e-5
    # nDCG@10 on the final scores, integer ranks exact
    from ptranking_b200 import ops
    _, order = ops.ndcg_at_ks(torch.from_numpy(s).cuda(), torch.from_numpy(y[0]).cuda(), [10], presort=True, return_order=True)
    ref_order = np.argsort(-z[run + "__final_scores"], axis=1, kind="stable")
    assert (order.cpu().numpy() == ref_order).mean() >= 0.999


def test_dropout_mask_statistics_and_consistency():
    """Training-mode dropout: unbiased in expectation, same mask in forward and backward."""
    from ptranking_b200.base.utils import StackedFFNet
    torch.manual_seed(0)
    F = 32
    net = StackedFFNet([F, 1], AF="R", TL_AF="S", apply_tl_af=False, dropout=0.0, BN=False).to(DEV)
    net2 = StackedFFNet([F, 8, 1], AF="R", TL_AF="S", apply_tl_af=False, dropout=0.25, BN=False).to(DEV)
    X = torch.randn(8, 512, F, device=DEV, requires_grad=True)
    net2.train()
    out = net2(X)
    out.sum().backward()
    # dX is zero exactly where the first-layer dropout zeroed the input, and scaled by 1/(1-p) elsewhere
    frac_zero = float((X.grad == 0).float().mean())
    assert abs(frac_zero - 0.25) < 0.01
    net2.eval()
    out_eval = net2(X.detach())
    assert torch.isfinite(out_eval).all()
    # a bare Linear equals the torch op (sanity of the tall-skinny GEMM path)
    ref = torch.nn.functional.linear(X.detach(), net.ff_2.weight, net.ff_2.bias)
    assert rel_err(net(X.detach()).detach().cpu().numpy(), ref.detach().cpu().numpy()) <= 1e-5


TC_CASES = [
    # B, n, dims, AF, TL_AF(None = no tail AF), norm, affine, dropout
    (4, 256, [136, 100, 100, 1], "GE", "S", "BN", True, 0.1),
    (3, 200, [136, 100, 100, 1], "R", "S", "BN2", False, 0.1),       # n > 128: groups span several row tiles
    (5, 50, [136, 100, 1], "GE", "S", "BN2", True, 0.0),             # n < 128: several groups per row tile
    (7, 33, [64, 48, 32, 1], "CE", None, None, False, 0.2),          # no norm, bare last Linear, ragged rows
    (2, 300, [136, 100, 8], "S", "R", "BN", False, 0.0),             # wider output, rows % 128 != 0
    (1, 1, [136, 100, 1], "GE", "S", None, False, 0.0),              # a single document
]


@pytest.mark.parametrize("case", TC_CASES, ids=[f"tc{i}" for i in range(len(TC_CASES))])
def test_tensor_core_path_matches_simt_path(case):
    """The tcgen05 (3xTF32) layer kernels against the fp32 SIMT kernels on identical inputs,
    dropout streams included: forward scores, parameter gradients and dX."""
    from ptranking_b200 import ops
    B, n, dims, AF, TL, norm, affine, p = case
    torch.manual_seed(B * 100 + n)
    specs = {m: ops.FFNetSpec(dims, AF if len(dims) > 2 else None, TL, norm, affine, p, math_mode=m) for m in ("simt", "3xtf32")}
    params = []
    for names, l in zip(specs["simt"].slots, range(len(dims) - 1)):
        for nm in names:
            if nm == "weight":
                t = torch.randn(dims[l + 1], dims[l], device=DEV) / np.sqrt(dims[l])
            elif nm in ("gamma", "aff_w"):
                t = 1.0 + 0.1 * torch.randn(dims[l + 1], device=DEV)
            else:
                t = 0.1 * torch.randn(dims[l + 1], device=DEV)
            params.append(t.requires_grad_(True))
    X = torch.randn(B, n, dims[0], device=DEV)
    dO = torch.randn(B, n, dims[-1], device=DEV)
    res = {}
    for m, spec in specs.items():
        Xm = X.clone().requires_grad_(True)
        pm = [q.detach().clone().requires_grad_(True) for q in params]
        out = ops.ffnet_apply(Xm, spec, pm, training=True, seed=1234, offset=7)
        (out * dO).sum().backward()
        res[m] = (out.detach().cpu().numpy(), [q.grad.cpu().numpy() for q in pm], Xm.grad.cpu().numpy())
    o_s, g_s, dx_s = res["simt"]
    o_t, g_t, dx_t = res["3xtf32"]
    assert rel_err(o_t, o_s) <= 1e-5, rel_err(o_t, o_s)
    gscale = max(np.abs(g).max() for g in g_s)
    for i, (a, b) in enumerate(zip(g_t, g_s)):
        assert np.abs(a - b).max() <= 2e-5 * np.abs(b).max() + 2e-6 * gscale + 1e-9, (i, np.abs(a - b).max(), np.abs(b).max())
    assert rel_err(dx_t, dx_s) <= 2e-5, rel_err(dx_t, dx_s)


def test_tf32_single_pass_is_looser_than_3xtf32():
    from ptranking_b200 import ops
    dims = [136, 100, 100, 1]
    torch.manual_seed(0)
    X = torch.randn(4, 128, 136, device=DEV)
    params = []
    spec0 = ops.FFNetSpec(dims, "GE", "S", None, False, 0.0, math_mode="simt")
    for names, l in zip(spec0.slots, range(3)):
        params += [torch.randn(dims[l + 1], dims[l], device=DEV) / np.sqrt(dims[l]), torch.zeros(dims[l + 1], device=DEV)]
    outs = {m: ops.ffnet_apply(X, ops.FFNetSpec(dims, "GE", "S", None, False, 0.0, math_mode=m), params, training=False).cpu().numpy()
            for m in ("simt", "3xtf32", "tf32")}
    e3, e1 = rel_err(outs["3xtf32"], outs["simt"]), rel_err(outs["tf32"], outs["simt"])
    assert e3 <= 1e-5 and 1e-5 < e1 <= 5e-3, (e3, e1)


WIDE_CASES = [
    # the list scorer's head / tail nets (list_ranker.py:309-341): widths beyond one MMA tile
    (2, 96, [136, 128, 256, 512, 136], "R", "R", None, False, 0.1),
    (2, 64, [136, 128, 256, 512, 1], "R", None, "BN2", False, 0.0),
    (3, 40, [64, 320, 8], "GE", "S", "BN", True, 0.0),
    # per-query BN2 with lists longer than one row tile (statistics groups span several tiles) AND wide layers:
    # BASELINE config (c)'s head net at its real shape, and its layers one at a time
    (2, 512, [136, 128, 256, 512, 136], "R", "R", "BN2", False, 0.0),
    (2, 512, [136, 128, 8], "R", "R", "BN2", False, 0.0),
    (2, 512, [136, 256, 8], "R", "R", "BN2", False, 0.0),
    (2, 512, [128, 512, 8], "R", "R", "BN2", False, 0.0),
    (2, 200, [136, 128, 8], "R", "R", "BN2", False, 0.0),
    (2, 512, [136, 128, 8], "R", "R", "BN", False, 0.0),
    (2, 512, [136, 100, 8], "R", "R", "BN2", False, 0.0),
]


@pytest.mark.parametrize("case", WIDE_CASES, ids=[f"wide{i}" for i in range(len(WIDE_CASES))])
def test_wide_layers_on_tensor_cores_match_simt(case):
    """Column-tiled rows_gemm and column-blocked wgrad (layers wider than 256 / 128) vs the fp32 SIMT kernels."""
    test_tensor_core_path_matches_simt_path(case)


FULL_CASES = [
    # BASELINE.json configs[1]: 1024 queries x 256 documents x 136 features through the default 5x100 GELU+BN scorer
    (1024, 256, [136, 100, 100, 100, 100, 100, 1], "GE", "S", "BN", True, 0.1),
    (256, 1024, [136, 100, 100, 100, 100, 100, 1], "GE", "S", "BN2", False, 0.1),
]


@pytest.mark.parametrize("case", FULL_CASES, ids=[f"full{i}" for i in range(len(FULL_CASES))])
def test_full_size_tensor_core_path_matches_simt(case):
    """Same comparison at the benchmark's full size: the weight-gradient contraction runs over 262144 rows."""
    test_tensor_core_path_matches_simt_path(case)


@pytest.mark.parametrize("wd", [0.0, 1e-3])
def test_flat_adam_matches_torch_adam(wd):
    """ops.adam_step (one kernel over flat buffers) against torch.optim.Adam over several steps, lr schedule included."""
    from ptranking_b200 import ops
    torch.manual_seed(5)
    n = 55204
    p0 = torch.randn(n, device=DEV)
    ref = torch.nn.Parameter(p0.clone())
    opt = torch.optim.Adam([ref], lr=1e-2, weight_decay=wd)
    sched = torch.optim.lr_scheduler.StepLR(opt, step_size=3, gamma=0.5)
    p, m, v = p0.clone(), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    for step in range(1, 8):
        g = torch.randn(n, device=DEV) * (10.0 ** float(torch.randint(-3, 2, (1,))))
        ref.grad = g.clone()
        opt.step()
        ops.adam_step(p, g, m, v, step, lr=opt.param_groups[0]["lr"], weight_decay=wd)
        sched.step()
        assert rel_err(p.cpu().numpy(), ref.detach().cpu().numpy()) <= 1e-6, step
    st = opt.state[ref]
    assert rel_err(m.cpu().numpy(), st["exp_avg"].cpu().numpy()) <= 1e-6
    assert rel_err(v.cpu().numpy(), st["exp_avg_sq"].cpu().numpy()) <= 1e-6


@pytest.mark.parametrize("wd", [0.0, 1e-3])
@pytest.mark.parametrize("which", ["Adagrad", "RMS"])
def test_flat_adagrad_rmsprop_match_torch(which, wd):
    """SURVEY 8f-3: ops.adagrad_step / ops.rmsprop_step (one kernel over the flat buffers) against torch.optim.Adagrad /
    torch.optim.RMSprop as ranker.py:517-520 configures them, over several steps with the StepLR schedule."""
    from ptranking_b200 import ops
    torch.manual_seed(6)
    n = 883370                                           # the default list scorer's parameter count (+1: tail loop)
    p0 = torch.randn(n, device=DEV)
    ref = torch.nn.Parameter(p0.clone())
    opt = (torch.optim.Adagrad if which == "Adagrad" else torch.optim.RMSprop)([ref], lr=1e-2, weight_decay=wd)
    sched = torch.optim.lr_scheduler.StepLR(opt, step_size=3, gamma=0.5)
    p, st = p0.clone(), torch.zeros(n, device=DEV)
    for step in range(1, 8):
        g = torch.randn(n, device=DEV) * (10.0 ** float(torch.randint(-3, 2, (1,))))
        ref.grad = g.clone()
        opt.step()
        if which == "Adagrad":
            ops.adagrad_step(p, g, st, step, lr=opt.param_groups[0]["lr"], weight_decay=wd)
        else:
            ops.rmsprop_step(p, g, st, lr=opt.param_groups[0]["lr"], weight_decay=wd)
        sched.step()
        assert rel_err(p.cpu().numpy(), ref.detach().cpu().numpy()) <= 1e-6, step
    key = "sum" if which == "Adagrad" else "square_avg"
    assert rel_err(st.cpu().numpy(), opt.state[ref][key].cpu().numpy()) <= 1e-6


@pytest.mark.parametrize("opt_id", ["Adagrad", "RMS"])
def test_ranker_steps_with_fused_adagrad_rmsprop(opt_id):
    """Three LambdaRank train steps with the fused optimizer against the same steps with torch.optim over the same flat
    gradient bucket (identical kernels upstream of the optimizer, dropout off): parameters agree to fp32 rounding."""
    import ptranking_b200
    from ptranking_b200 import LABEL_TYPE
    from ptranking_b200.base import ranker as rk
    F = 136
    sf = dict(sf_id="pointsf", opt=opt_id, lr=1e-3, pointsf=point_cfg(F))
    sf["pointsf"]["dropout"] = 0.0
    torch.manual_seed(11)
    a = ptranking_b200.LambdaRank(sf_para_dict=sf, model_para_dict=dict(model_id="LambdaRank", sigma=1.0), gpu=True, device=DEV)
    a.init()
    assert isinstance(a.optimizer, rk.FlatAdagrad if opt_id == "Adagrad" else rk.FlatRMSprop)
    b = ptranking_b200.LambdaRank(sf_para_dict=sf, model_para_dict=dict(model_id="LambdaRank", sigma=1.0), gpu=True, device=DEV)
    b.init()
    b.point_sf.load_state_dict({k: v.clone() for k, v in a.point_sf.state_dict().items()})
    cls = torch.optim.Adagrad if opt_id == "Adagrad" else torch.optim.RMSprop
    b.optimizer = cls(list(b.get_parameters()), lr=1e-3, weight_decay=b.weight_decay)
    g = torch.Generator().manual_seed(3)
    X = torch.randn(8, 64, F, generator=g).to(DEV)
    y = torch.sort(torch.randint(0, 5, (8, 64), generator=g).float(), dim=1, descending=True)[0].to(DEV)
    for _ in range(3):
        la, _ = a.train_op(X, y, presort=True, label_type=LABEL_TYPE.MultiLabel)
        lb, _ = b.train_op(X, y, presort=True, label_type=LABEL_TYPE.MultiLabel)
        assert abs(float(la) - float(lb)) <= 1e-5 * abs(float(lb))
    for (k, va), (_, vb) in zip(a.point_sf.state_dict().items(), b.point_sf.state_dict().items()):
        assert rel_err(va.cpu().numpy(), vb.cpu().numpy()) <= 1e-5, k


def test_ranker_parameters_live_in_one_flat_buffer():
    r = _point_ranker("ListNet", 136)
    b = r.grad_bucket
    assert b.params_are_flat() and b.flat_param.numel() == b.flat.numel() and b.flat.numel() % 4 == 0
    assert all(p.data_ptr() % 16 == 0 and p.grad.data_ptr() % 16 == 0 for p in b.params)
    sd = {k: v.clone() for k, v in r.point_sf.state_dict().items()}
    r.point_sf.load_state_dict(sd)                      # in-place copies keep the parameters inside the flat buffer
    assert b.params_are_flat()


def _bf16r(t):
    return t.to(torch.bfloat16).to(t.dtype)


class _Bf16Linear(torch.autograd.Function):
    """nn.Linear whose three GEMMs take bf16-rounded operands and accumulate in float64 (the semantics of math_mode='bf16')."""

    @staticmethod
    def forward(ctx, x, w, b):
        ctx.save_for_backward(x, w)
        return (_bf16r(x).double() @ _bf16r(w).double().t() + b.double()).float()

    @staticmethod
    def backward(ctx, g):
        x, w = ctx.saved_tensors
        gr = _bf16r(g).double()
        return (gr @ _bf16r(w).double()).float(), (gr.t() @ _bf16r(x).double()).float(), g.sum(0)


def test_bf16_math_mode_is_a_bf16_gemm_with_fp32_accumulation():
    """SURVEY 8d config (e): bf16 feature / GEMM inputs.  Every operand of every contraction is rounded to bf16, products are
    exact, accumulation fp32 -- checked against a float64-accumulating emulation with the same roundings; it must also
    differ measurably from (and stay near) the fp32-grade default."""
    from ptranking_b200 import ops
    dims = [136, 100, 100, 1]
    torch.manual_seed(11)
    B, n = 4, 96
    X = torch.randn(B, n, dims[0], device=DEV)
    dO = torch.randn(B, n, 1, device=DEV)
    params = []
    for l in range(3):
        params += [torch.randn(dims[l + 1], dims[l], device=DEV) / np.sqrt(dims[l]), 0.1 * torch.randn(dims[l + 1], device=DEV)]
    res = {}
    for mode in ("bf16", "3xtf32"):
        pm = [q.clone().requires_grad_(True) for q in params]
        Xm = X.clone().requires_grad_(True)
        out = ops.ffnet_apply(Xm, ops.FFNetSpec(dims, "R", None, None, False, 0.0, math_mode=mode), pm, training=False)
        (out * dO).sum().backward()
        res[mode] = [out.detach()] + [q.grad for q in pm] + [Xm.grad]
    pe = [q.clone().requires_grad_(True) for q in params]
    Xe = X.clone().requires_grad_(True)
    h = Xe.reshape(-1, dims[0])
    for l in range(3):
        h = _Bf16Linear.apply(h, pe[2 * l], pe[2 * l + 1])
        if l < 2:
            h = torch.relu(h)
    (h.reshape(B, n, 1) * dO).sum().backward()
    emu = [h.reshape(B, n, 1).detach()] + [q.grad for q in pe] + [Xe.grad]
    for i, (a, e, f) in enumerate(zip(res["bf16"], emu, res["3xtf32"])):
        a, e, f = (t.cpu().numpy() for t in (a, e, f))
        # an fp32-vs-fp64 accumulation difference occasionally flips one downstream bf16 rounding (2^-8 of one operand)
        assert rel_err(a, e) <= (2e-3 if i == 0 else 5e-3), (i, rel_err(a, e))
        # ... and bf16 really is coarser than the default: scores move by ~1e-2, gradients (ReLU gates flip) by more
        # (the last bias gradient is sum(dO) in every mode, hence no lower bound on the gradients)
        assert rel_err(a, f) <= (3e-2 if i == 0 else 0.5), (i, rel_err(a, f))
        if i == 0:
            assert rel_err(a, f) > 1e-4, rel_err(a, f)


@pytest.mark.parametrize("n", [32, 256, 1024])
def test_listmle_with_bf16_scorer_tracks_the_fp32_scorer(n, monkeypatch):
    """Config (e) end to end: ListMLE over a bf16-input scorer vs the fp32-grade scorer on the same weights and batch --
    loss within bf16 tolerance, ranks compared (top-10 overlap reported through the assertion)."""
    import ptranking_b200
    from ptranking_b200 import LABEL_TYPE
    rng = np.random.default_rng(n)
    B = 8
    X = torch.from_numpy(rng.standard_normal((B, n, 136)).astype(np.float32)).to(DEV)
    y = torch.from_numpy(np.sort(rng.integers(0, 5, size=(B, n)).astype(np.float32), axis=1)[:, ::-1].copy()).to(DEV)
    out = {}
    for mode in ("3xtf32", "bf16"):
        monkeypatch.setenv("PTRANKING_B200_MATH", mode)
        torch.manual_seed(3)
        r = _point_ranker("ListMLE", 136, dropout=0.0)
        r.eval_mode()
        with torch.no_grad():
            s = r.forward(X)
        r.train_mode()
        loss = float(r.train_op(X, y, presort=True, label_type=LABEL_TYPE.MultiLabel, epoch_k=1)[0])
        out[mode] = (s.cpu().numpy(), loss)
    s32, l32 = out["3xtf32"]
    s16, l16 = out["bf16"]
    assert np.isfinite(l16) and abs(l16 - l32) <= 2e-2 * abs(l32), (l16, l32)
    assert rel_err(s16, s32) <= 5e-2
    top = lambda s: np.argsort(-s, axis=1, kind="stable")[:, :10]
    overlap = np.mean([len(set(a) & set(b)) / 10.0 for a, b in zip(top(s16), top(s32))])
    assert overlap >= 0.6, overlap


def test_gelu_matches_exact_erf_gelu_to_fp32_rounding():
    """The scorer's GELU evaluates the normal CDF directly (csrc/ffnet_act.cuh::normal_cdf) instead of calling erff; it must
    be as close to the exact-erf GELU of nn.GELU() (get_AF 'GE', base/utils.py:125) as a correctly rounded erff would be:
    dense grid over [-8, 8] plus normal samples, value and derivative, against float64."""
    from ptranking_b200 import ops
    x = torch.cat([torch.linspace(-8.0, 8.0, 2_000_001), torch.randn(1_000_000) * 1.5,
                   torch.tensor([0.0, -0.0, 5.75, -5.75, 6.0, -6.0, 30.0, -30.0, 1e-30, -1e-30, 1e30, -1e30])]).to(DEV)
    y = ops.activation(x, "GE").double().cpu()
    dy = ops.activation(x, "GE", grad=True).double().cpu()
    x64 = x.double().cpu()
    cdf = 0.5 * torch.erfc(-x64 / 2 ** 0.5)
    want = x64 * cdf
    dwant = cdf + x64 * torch.exp(-0.5 * x64 * x64) / (2 * torch.pi) ** 0.5
    fin = x64.abs() <= 8.0
    # torch's own fp32 GELU (erff based) as the yardstick
    base = torch.nn.functional.gelu(x.cpu()).double()
    err, err_base = (y - want).abs()[fin].max().item(), (base - want).abs()[fin].max().item()
    assert err <= max(1.25 * err_base, 6e-7), (err, err_base)
    rms, rms_base = ((y - want)[fin] ** 2).mean().sqrt().item(), ((base - want)[fin] ** 2).mean().sqrt().item()
    assert rms <= 1.25 * rms_base, (rms, rms_base)
    assert (dy - dwant).abs()[fin].max().item() <= 6e-7
    # far tails: exact limits, no NaN from the flushed half
    assert y[-1].item() == 0.0 and y[-2].item() == float(np.float32(1e30)) and torch.isfinite(y).all()
    assert ops.activation(torch.tensor([float("nan")], device=DEV), "GE").isnan().all()
