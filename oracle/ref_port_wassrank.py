"""oracle/ref_port_wassrank.py -- CPU restatement of WassRank's SinkhornOT loss with the reference's ATen operators.

TEST INFRASTRUCTURE, NOT PRODUCT (same import rule as oracle/ref_port.py).

Follows ltr_adhoc/listwise/wassrank/wassRank.py:43-86, pytorch_wasserstein.py:323-394 (OldSinkhornOT) and
wasserstein_cost_mat.py:47-244 operator by operator, in the tensors' dtype and on their device, so the fp32 run
reproduces the reference's values, including where its per-vector stabilisation underflows into NaN.  Pinned by
tests/test_oracle_wassrank.py against outputs of the unmodified reference (tests/golden/wassrank.npz).
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F


def wass_cost_mat(labels, cost_type="eg", gain_base=4.0, non_rele_gap=100.0, var_penalty=math.e):
    """get_explicit_cost_mat, ltr_adhoc/listwise/wassrank/wasserstein_cost_mat.py:47-139 -> [B,n,n]."""
    B, n = labels.shape
    dev = labels.device                                             # the reference's gpu=True branch: cuda tensors
    if cost_type in ("p1", "p2"):                                   # torch_cost_mat_dist, :47-60
        pos = torch.arange(n, device=dev).float() + 1.0
        C = torch.abs(pos.view(-1, 1) - pos.view(1, -1)).expand(B, -1, -1)
        return torch.pow(C, 2.0) if cost_type == "p2" else C
    if cost_type == "eg":                                           # torch_cost_mat_group, :84-111
        g = torch.pow(gain_base, labels) - 1.0
        a = torch.where(g < 1.0, -torch.tensor([non_rele_gap], dtype=torch.float32, device=dev), g)
        C = torch.abs(a.view(B, n, 1) - a.view(B, 1, n))
        C = torch.where(C < 1.0, torch.tensor([var_penalty], dtype=torch.float32, device=dev), C)
        return C - (torch.eye(n, device=dev).float() * var_penalty).expand(B, -1, -1)
    if cost_type in ("dg", "ddg"):                                  # get_delta_gains, :63-81
        g = torch.pow(2.0, labels) - 1.0
        dg = torch.unsqueeze(g, 2) - torch.unsqueeze(g, 1)
        if cost_type == "dg":
            return torch.abs(dg)
        disc = torch.unsqueeze(1.0 / torch.log2(torch.arange(n, device=dev).float() + 2.0), 0)
        return torch.abs(dg) * torch.abs(torch.unsqueeze(disc, 2) - torch.unsqueeze(disc, 1))
    raise NotImplementedError(cost_type)


def wass_histograms(labels, preds, smooth_type="ST", norm_type="BothST"):
    """get_normalized_histograms, wasserstein_cost_mat.py:181-246, as it runs: the 'S' tail rescaling (:196-199) is
    skipped because WassRank's TL_AF is None (its get_tl_af returns nothing, SURVEY B11)."""
    if smooth_type == "ST":
        if norm_type != "BothST":
            raise NotImplementedError(norm_type)
        return F.softmax(labels, dim=1), F.softmax(preds, dim=1)
    if smooth_type == "NG":
        gy = torch.pow(2.0, labels) - 1.0
        std = gy / torch.sum(gy, dim=1).view(-1, 1)
        mini = torch.min(preds)
        if not mini > 0.0:
            preds = preds - mini
        return std, preds / torch.sum(preds, dim=1).view(-1, 1)
    raise NotImplementedError(smooth_type)


class _OldSinkhornOT(torch.autograd.Function):
    """OldSinkhornOT, pytorch_wasserstein.py:323-394: per-vector-max stabilised Sinkhorn on K = exp(-C/lam), returns the
    1-element loss; backward hands pred the envelope term lam * log_u centred twice, over the batch size."""

    @staticmethod
    def forward(ctx, pred, target, cost, lam, sh_itr):
        na, nb = cost.size(0), cost.size(1)
        K = torch.exp(-cost / lam)
        KM = cost * K
        B = pred.size(0)
        log_a, log_b = torch.log(pred), torch.log(target)
        log_u = cost.new(B, na).fill_(-math.log(na))
        log_v = cost.new(B, nb).fill_(-math.log(nb))
        for _ in range(sh_itr):
            mu_ = torch.max(log_u, dim=1, keepdim=True)[0]
            log_v = log_b - torch.log(torch.mm(K.t(), torch.exp(log_u - mu_).t()).t()) - mu_
            mv_ = torch.max(log_v, dim=1, keepdim=True)[0]
            log_u = log_a - torch.log(torch.mm(K, torch.exp(log_v - mv_).t()).t()) - mv_
        mv_ = torch.max(log_v, dim=1, keepdim=True)[0]
        part1 = torch.log(torch.mm(KM, torch.exp(log_v - mv_).t()).t()) + mv_
        wnorm = torch.exp(log_u + part1).mean(0).sum()
        g = log_u * lam
        g = g - torch.mean(g, dim=1, keepdim=True)
        g = g - torch.mean(g, dim=1, keepdim=True)
        ctx.save_for_backward(g / B)
        return cost.new((wnorm,))

    @staticmethod
    def backward(ctx, grad_output):
        g = ctx.saved_tensors[0].clone()
        if grad_output[0] != 1:
            g.mul_(grad_output[0])
        return g, None, None, None, None


def wassrank_loss(preds, labels, mode="SinkhornOT", sh_itr=20, lam=0.1, smooth_type="ST", norm_type="BothST",
                  cost_type="eg", non_rele_gap=100.0, var_penalty=math.e, gain_base=4.0, **_):
    """WassRank.custom_loss_function, ltr_adhoc/listwise/wassrank/wassRank.py:43-86.  The reference runs at B=1 only
    (torch.squeeze(cost, 0), :73); a batch here is its queries run one at a time, each loss scaled by 1/B."""
    if mode != "SinkhornOT":
        raise NotImplementedError(mode)
    B = preds.size(0)
    C = wass_cost_mat(labels, cost_type, gain_base, non_rele_gap, var_penalty)
    total = 0.0
    for b in range(B):
        std, pred = wass_histograms(labels[b:b + 1], preds[b:b + 1], smooth_type, norm_type)
        loss = _OldSinkhornOT.apply(pred, std, C[b], lam, sh_itr)
        total = total + (loss if B == 1 else loss / B)
    return total.reshape(())


def loss_and_grad(scores: torch.Tensor, labels: torch.Tensor, **params):
    """(loss, d loss / d scores) on a leaf copy of ``scores`` (fp32), as oracle/ref_port.py's loss_and_grad does."""
    s = scores.detach().clone().float().requires_grad_(True)
    loss = wassrank_loss(s, labels, **params)
    loss.backward()
    g = s.grad if s.grad is not None else torch.zeros_like(s)
    return loss.detach(), g.detach()
