"""oracle/closed_form_wassrank.py -- float64 numpy closed form of WassRank's SinkhornOT loss and its gradient.

TEST INFRASTRUCTURE, NOT PRODUCT (same import rule as oracle/ref_port.py).

An independent statement written from the math rather than from the reference's code path: the Sinkhorn updates run as
row-wise log-sum-exps in float64, so it stays finite where the reference's per-vector stabilisation underflows (even in
float64 at lambda = 0.1).  Pinned by tests/test_oracle_wassrank.py against the reference's own float64 run
(tests/golden/wassrank.npz) wherever that run is finite.
"""
from __future__ import annotations

import numpy as np


def _lse(a, axis):
    """log-sum-exp that keeps an all -inf slice at -inf (and NaN as NaN)."""
    m = np.max(a, axis=axis, keepdims=True)
    mf = np.where(np.isfinite(m), m, 0.0)
    with np.errstate(divide="ignore", invalid="ignore"):
        out = np.log(np.exp(a - mf).sum(axis=axis, keepdims=True)) + mf
    out = np.where(np.isneginf(m), -np.inf, out)
    return np.squeeze(out, axis=axis)


def wass_cost(y, cost_type, gain_base=4.0, non_rele_gap=100.0, var_penalty=np.e):
    """get_explicit_cost_mat, wasserstein_cost_mat.py:47-139, for one query's labels y[n] -> C[n,n].  Two values stay in
    fp32 as the reference holds them: var_penalty (a FloatTensor, :103) and the rank discounts of 'ddg' (:73-76)."""
    y = y.astype(np.float64)
    n = y.shape[0]
    pos = np.arange(n, dtype=np.float64) + 1.0
    if cost_type == "p1":
        return np.abs(pos[:, None] - pos[None, :])
    if cost_type == "p2":
        return (pos[:, None] - pos[None, :]) ** 2
    if cost_type == "eg":
        g = np.power(float(gain_base), y) - 1.0
        a = np.where(g < 1.0, -float(non_rele_gap), g)
        d = np.abs(a[:, None] - a[None, :])
        C = np.where(d < 1.0, float(np.float32(var_penalty)), d)
        np.fill_diagonal(C, 0.0)
        return C
    if cost_type in ("dg", "ddg"):
        g = np.power(2.0, y) - 1.0
        C = np.abs(g[:, None] - g[None, :])
        if cost_type == "ddg":
            r = np.arange(n, dtype=np.float32) + np.float32(2.0)
            disc = (1.0 / np.log2(r.astype(np.float64)).astype(np.float32)).astype(np.float32)
            C = C * np.abs(disc[:, None] - disc[None, :]).astype(np.float64)
        return C
    raise NotImplementedError(cost_type)


def wassrank(s, y, cost_type="eg", smooth_type="ST", norm_type="BothST", lam=0.1, sh_itr=20, gain_base=4.0,
             non_rele_gap=100.0, var_penalty=np.e, mode="SinkhornOT", **_):
    """WassRank's SinkhornOT loss per query (wassRank.py:63-73 with OldSinkhornOT, pytorch_wasserstein.py:323-394),
    summed over the queries of s[B,n] with the reference's 1/B, and the gradient its backward hands the scores.

    The Sinkhorn updates are the reference's, written as row-wise log-sum-exps:
        log_v_j = log nu_j - LSE_i(-C_ij/lam + log_u_i),   log_u_i = log mu_i - LSE_j(-C_ij/lam + log_v_j),
    loss = (1/B) sum_i exp(log_u_i + LSE_{j: C_ij > 0}(log C_ij - C_ij/lam + log_v_j)).
    d loss / d mu is the reference's envelope term lam * log_u centred twice, over B (:371-380); it is chained through
    the histogram map: softmax for 'ST', s/sum(s) or (s - min)/sum(s - min) for 'NG' (wasserstein_cost_mat.py:181-246),
    the min's gradient split evenly over tied minima as ATen's full min reduction does."""
    if mode != "SinkhornOT":
        raise NotImplementedError(mode)
    s = np.asarray(s, dtype=np.float64)
    yy = np.asarray(y, dtype=np.float64)
    B, n = s.shape
    loss, grad = 0.0, np.zeros_like(s)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        for b in range(B):
            sb, yb = s[b], yy[b]
            C = wass_cost(yb, cost_type, gain_base, non_rele_gap, var_penalty)
            if smooth_type == "ST":
                if norm_type != "BothST":
                    raise NotImplementedError(norm_type)
                log_nu = yb - _lse(yb, 0)
                log_mu = sb - _lse(sb, 0)
            elif smooth_type == "NG":
                gy = np.power(2.0, yb) - 1.0
                log_nu = np.log(gy / gy.sum())
                m = sb.min()
                t = sb if m > 0.0 else sb - m
                T = t.sum()
                log_mu = np.log(t / T)
            else:
                raise NotImplementedError(smooth_type)
            KL = -C / lam
            log_u = np.full(n, -np.log(n))
            log_v = np.full(n, -np.log(n))
            for _ in range(sh_itr):
                log_v = log_nu - _lse(KL + log_u[:, None], 0)
                log_u = log_mu - _lse(KL + log_v[None, :], 1)
            Lc = np.where(C > 0, np.log(np.where(C > 0, C, 1.0)) + KL + log_v[None, :], -np.inf)
            loss += np.exp(log_u + _lse(Lc, 1)).sum() / B
            g = lam * log_u
            g = g - g.mean()
            g = g - g.mean()
            g = g / B
            if smooth_type == "ST":
                mu = np.exp(log_mu)
                grad[b] = mu * (g - (mu * g).sum())
            else:
                mu = t / T
                gt = (g - (mu * g).sum()) / T
                if m > 0.0:
                    grad[b] = gt
                else:
                    tied = sb == m
                    grad[b] = gt - tied * gt.sum() / tied.sum()
    return loss, grad
