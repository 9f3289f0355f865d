"""Torch-side glue over the C ABI: device memory, streams and autograd plumbing only.

Every function takes CUDA fp32 tensors, passes raw device pointers + the current
CUDA stream to libptranking_b200.so and returns tensors allocated by torch.  No
arithmetic of the hot path happens in Python/ATen here.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import functools
import os
from typing import Optional, Sequence

import torch

from . import _lib


def _stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def _on_tensor_device(fn):
    """Run ``fn`` with the CUDA device of its first CUDA tensor argument current.

    The C library launches on the *current* device and ``_stream_ptr`` returns the current device's current stream, so a
    tensor on ``cuda:1`` while ``cuda:0`` is current would be dereferenced by a kernel on the wrong GPU (the reference
    driver avoids this only because it calls ``torch.cuda.set_device``, ltr.py:48).  Every entry point that reaches the
    C ABI is wrapped with this guard."""
    @functools.wraps(fn)
    def guarded(*args, **kw):
        for a in args:
            if isinstance(a, torch.Tensor) and a.is_cuda:
                if a.device.index != torch.cuda.current_device():
                    with torch.cuda.device(a.device):
                        return fn(*args, **kw)
                break
        return fn(*args, **kw)
    return guarded


def _dev_f32(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise _lib.B200LibraryError(f"{name} must be a CUDA tensor: ptranking_b200 has no CPU path")
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def _list_layout(s: torch.Tensor, offsets, max_len):
    """-> (B, n, offsets tensor or None, offsets pointer or None).  Dense batches: ``s`` is [B,n] and offsets is None.
    Ragged batches (SURVEY 8f-2): ``s`` is the flat [total_docs] array, ``offsets`` the int32 [B+1] prefix offsets on the
    same device, ``max_len`` the longest list (host int: it sizes the CTAs, so no device read-back is needed)."""
    if offsets is None:
        if s.dim() != 2:
            raise ValueError(f"expected [B,n] scores, got {tuple(s.shape)} (pass offsets= and max_len= for a ragged batch)")
        return s.shape[0], s.shape[1], None, None
    if s.dim() != 1:
        raise ValueError(f"ragged batches are flat [total_docs] arrays, got {tuple(s.shape)}")
    if max_len is None:
        raise ValueError("ragged batches need max_len= (longest list of the batch)")
    if not (offsets.is_cuda and offsets.device == s.device):
        raise _lib.B200LibraryError("offsets must live on the device of the scores")
    offsets = offsets.to(torch.int32).contiguous()
    return offsets.numel() - 1, max(int(max_len), 1), offsets, offsets.data_ptr()


# --------------------------------------------------------------------------- #
# ranking losses
# --------------------------------------------------------------------------- #
def _launch_ranges(B, n, offsets, buckets, coupled):
    """(first query, query count, longest list) per launch.  ``buckets`` (ragged batches only): host-side
    [(q_begin, q_end, max_len), ...] covering the queries in order -- data.RaggedBatches sorts a batch by length and cuts
    it at power-of-two lengths, so each launch gets CTAs (and the pair schedule) sized for ITS lists instead of for the
    longest list of the whole batch.  Losses coupled across the batch (ApproxNDCG's [B]/[B,1] broadcast, RankMSE's mean)
    take one launch."""
    if offsets is None or not buckets or coupled:
        return [(0, B, n)]
    out = [(int(b0), int(b1) - int(b0), max(int(ml), 1)) for b0, b1, ml in buckets if int(b1) > int(b0)]
    if sum(c for _, c, _ in out) != B or out[0][0] != 0:
        raise ValueError("buckets must cover the queries of the batch in order")
    return out


@_on_tensor_device
def _loss_call(name: str, scores: torch.Tensor, labels: torch.Tensor, params: dict):
    """-> (loss_per_query[B], grad[B,n]) from one fused kernel launch (one per length bucket of a ragged batch)."""
    lib = _lib.load()
    s = _dev_f32(scores, "scores")
    B, n, offsets, op = _list_layout(s, params.get("offsets"), params.get("max_len"))
    grad = torch.empty_like(s)
    loss_q = torch.empty(B, dtype=torch.float32, device=s.device)
    st = _stream_ptr()
    sp, gp, lq = s.data_ptr(), grad.data_ptr(), loss_q.data_ptr()
    # Length buckets pay for the O(n^2) losses only (the O(n) ones are launch-bound: one launch is best), and not for losses
    # coupled across the batch (ApproxNDCG's [B]/[B,1] broadcast, RankMSE's mean over queries)
    quadratic = name in ("RankNet", "LambdaRank", "LambdaLoss", "SoftRank", "ApproxNDCG", "WassRank")
    coupled = name == "RankMSE" or (name == "ApproxNDCG" and bool(params.get("batch_coupled", True)))
    ranges = _launch_ranges(B, n, offsets, params.get("buckets"), coupled or not quadratic)
    if name == "ListMLE":
        perm = params.get("perm")
        if perm is None:
            perm = shuffle_ties_perm(labels, offsets=offsets, max_len=n if offsets is not None else None, buckets=params.get("buckets"))
        perm = perm.to(device=s.device, dtype=torch.int32).contiguous()
        if perm.shape != s.shape:
            raise ValueError(f"perm {tuple(perm.shape)} does not match scores {tuple(s.shape)}")
        aux = perm
    else:
        y = _dev_f32(labels, "labels")
        if y.shape != s.shape:
            raise ValueError(f"expected scores/labels of identical shape, got {tuple(s.shape)} / {tuple(y.shape)}")
        aux = y
    yp = aux.data_ptr()
    unif = None
    if name == "STListNet":
        unif = params.get("unif")
        if unif is not None:
            unif = _dev_f32(unif, "unif")
            if unif.shape != s.shape:
                raise ValueError("unif must have the shape of scores")
        seed, offset = params.get("seed"), params.get("offset")
        if seed is None:
            seed = torch.initial_seed()
        if offset is None:
            offset = next_noise_offset()
    if name == "WassRank":
        wass = wassrank_settings(params)
    # ApproxNDCG scratch: Bq + 1 floats per launch; concurrent buckets get disjoint pieces
    scratch = torch.empty(B + len(ranges), dtype=torch.float32, device=s.device) if name == "ApproxNDCG" else None
    # The first bucket holds the longest lists: few CTAs that run long.  It goes onto a side stream so that the short-list
    # buckets (many CTAs, done quickly) fill the rest of the GPU meanwhile; the buckets write disjoint slices.
    side = None
    if len(ranges) > 1:
        cur = torch.cuda.current_stream(s.device)
        side = _side_stream(s.device)
        side.wait_stream(cur)
    for bi, (q0, Bq, nq) in enumerate(ranges):
        # a bucket is addressed through its slice of the (absolute) prefix offsets and of the per-query loss vector; the flat
        # score / label / gradient arrays are shared
        opq = None if op is None else op + 4 * q0
        lqq = lq + 4 * q0
        st = side.cuda_stream if (side is not None and bi == 0) else _stream_ptr()
        if name == "ListMLE":
            rc = lib.ptrb200_listmle_fwd_bwd(sp, yp, opq, gp, lqq, Bq, nq, st)
        elif name == "RankNet":
            rc = lib.ptrb200_ranknet_fwd_bwd(sp, yp, opq, gp, lqq, Bq, nq, float(params.get("sigma", 1.0)), st)
        elif name == "LambdaRank":
            rc = lib.ptrb200_lambdarank_fwd_bwd(sp, yp, opq, gp, lqq, Bq, nq, float(params.get("sigma", 1.0)), st)
        elif name == "LambdaLoss":
            lt = _lib.LAMBDALOSS_TYPES[params.get("loss_type", "NDCG_Loss2++")]
            rc = lib.ptrb200_lambdaloss_fwd_bwd(sp, yp, opq, gp, lqq, Bq, nq, int(params.get("k", 5)), float(params.get("sigma", 1.0)),
                                                float(params.get("mu", 5.0)), lt, int(bool(params.get("presort", True))), st)
        elif name == "ListNet":
            rc = lib.ptrb200_listnet_fwd_bwd(sp, yp, opq, gp, lqq, Bq, nq, st)
        elif name == "ApproxNDCG":
            rc = lib.ptrb200_approxndcg_fwd_bwd(sp, yp, opq, gp, lqq, scratch.data_ptr() + 4 * (q0 + bi), Bq, nq, float(params.get("alpha", 10.0)),
                                                int(bool(params.get("presort", True))), int(bool(params.get("batch_coupled", True))), st)
        elif name == "RankMSE":
            rc = lib.ptrb200_rankmse_fwd_bwd(sp, yp, opq, gp, lqq, Bq, nq, st)
        elif name == "RankCosine":
            rc = lib.ptrb200_rankcosine_fwd_bwd(sp, yp, opq, gp, lqq, Bq, nq, st)
        elif name == "STListNet":
            rc = lib.ptrb200_stlistnet_fwd_bwd(sp, yp, opq, unif.data_ptr() if unif is not None else None, gp, lqq, Bq, nq,
                                               float(params.get("temperature", 1.0)), seed & (2 ** 64 - 1), offset & (2 ** 64 - 1), st)
        elif name == "SoftRank":
            top_k = params.get("top_k")
            rc = lib.ptrb200_softrank_fwd_bwd(sp, yp, opq, gp, lqq, Bq, nq, float(params.get("delta", 2.0)), int(top_k) if top_k else 0, st)
        elif name == "WassRank":
            rc = lib.ptrb200_wassrank_fwd_bwd(sp, yp, opq, gp, lqq, Bq, nq, B, *wass, st)
        else:
            raise NotImplementedError(name)
        _lib.check(rc, f"{name} loss kernel")
    if side is not None:
        torch.cuda.current_stream(s.device).wait_stream(side)
    return loss_q, grad


def wassrank_settings(params: dict):
    """WassRank's parameters (the keys of the reference's wass_para_dict, defaults of WassRankParameter,
    wassRank.py:102-103) -> the kernel's (cost_type, smooth_type, lam, sh_itr, gain_base, non_rele_gap, var_penalty).
    Raises NotImplementedError for what the reference does not run: mode 'EntropicOT' (not built here), any other mode,
    smooth_type or norm_type, and unknown cost types (wassRank.py:79-80, wasserstein_cost_mat.py:136-137, :202-203, :243-244)."""
    mode = params.get("mode", "SinkhornOT")
    if mode == "EntropicOT":
        raise NotImplementedError("WassRank mode 'EntropicOT' is not built in ptranking_b200; use mode='SinkhornOT'")
    if mode != "SinkhornOT":
        raise NotImplementedError(f"WassRank mode {mode!r}")
    cost, smooth = params.get("cost_type", "eg"), params.get("smooth_type", "ST")
    if cost not in _lib.WASS_COST_TYPES:
        raise NotImplementedError(f"WassRank cost_type {cost!r}")
    if smooth not in _lib.WASS_SMOOTH_TYPES:
        raise NotImplementedError(f"WassRank smooth_type {smooth!r}")
    if smooth == "ST" and params.get("norm_type", "BothST") != "BothST":
        raise NotImplementedError(f"WassRank norm_type {params.get('norm_type')!r}")
    return (_lib.WASS_COST_TYPES[cost], _lib.WASS_SMOOTH_TYPES[smooth], float(params.get("lam", 0.1)),
            int(params.get("sh_itr", 20)), float(params.get("gain_base", 4)), float(params.get("non_rele_gap", 100)),
            float(params.get("var_penalty", 2.718281828459045)))


_side_streams = {}


def _side_stream(device) -> "torch.cuda.Stream":
    key = torch.device(device).index
    if key not in _side_streams:
        _side_streams[key] = torch.cuda.Stream(device=device)
    return _side_streams[key]


_noise_offset = 0


def next_noise_offset() -> int:
    """Counter that keys the Gumbel draw of successive STListNet calls (same role as the tie-shuffle counter)."""
    global _noise_offset
    _noise_offset += 1
    return _noise_offset


@_on_tensor_device
def sinkstep(dist: torch.Tensor, log_nu: torch.Tensor, log_u: torch.Tensor, lam: float) -> torch.Tensor:
    """log_v[b,j] = log_nu[b,j] - logsumexp_i(-dist[i,j]/lam + log_u[b,i]) (pytorch_wasserstein.py:277-291)."""
    lib = _lib.load()
    dist, log_nu, log_u = _dev_f32(dist, "dist"), _dev_f32(log_nu, "log_nu"), _dev_f32(log_u, "log_u")
    if dist.dim() != 2 or log_nu.dim() != 2 or log_u.dim() != 2 or dist.size(0) != log_u.size(1) or \
            dist.size(1) != log_nu.size(1) or log_u.size(0) != log_nu.size(0):
        raise ValueError("sinkstep: expected dist[d1,d2], log_nu[B,d2], log_u[B,d1]")
    log_v = torch.empty_like(log_nu)
    _lib.check(lib.ptrb200_sinkstep(dist.data_ptr(), log_nu.data_ptr(), log_u.data_ptr(), log_v.data_ptr(),
                                    log_u.size(0), dist.size(0), dist.size(1), float(lam), _stream_ptr()), "sinkstep")
    return log_v


class SinkhornOT(torch.autograd.Function):
    """SinkhornOT of pytorch_wasserstein.py:294-324 with every half-step on the sinkstep kernel: entropic OT distances
    between batches of histograms mu[B,d1], nu[B,d2] under the cost matrix dist[d1,d2]; backward returns
    lam * log_u / lam * log_v like the reference."""

    @staticmethod
    def forward(ctx, mu, nu, dist, lam=1e-3, N=100):
        import math
        d1, d2 = dist.shape
        log_mu, log_nu = mu.log(), nu.log()
        log_u = torch.full_like(mu, -math.log(d1))
        log_v = torch.full_like(nu, -math.log(d2))
        dist_t = dist.t().contiguous()
        for _ in range(N):
            log_v = sinkstep(dist, log_nu, log_u, lam)
            log_u = sinkstep(dist_t, log_mu, log_v, lam)
        distances = (-sinkstep(-dist.log() + dist / lam, -log_v, log_u, 1.0)).logsumexp(1).exp()
        ctx.save_for_backward(log_u, log_v)
        ctx.lam = lam
        return distances

    @staticmethod
    def backward(ctx, grad_out):
        log_u, log_v = ctx.saved_tensors
        return grad_out[:, None] * log_u * ctx.lam, grad_out[:, None] * log_v * ctx.lam, None, None, None


@_on_tensor_device
def sum_f32(x: torch.Tensor) -> torch.Tensor:
    """Fixed-order device sum -> 0-dim tensor."""
    lib = _lib.load()
    x = _dev_f32(x, "x").reshape(-1)
    out = torch.empty(1, dtype=torch.float32, device=x.device)
    _lib.check(lib.ptrb200_sum_f32(x.data_ptr(), out.data_ptr(), x.numel(), _stream_ptr()), "sum_f32")
    return out.reshape(())


@_on_tensor_device
def adam_step(param: torch.Tensor, grad: torch.Tensor, exp_avg: torch.Tensor, exp_avg_sq: torch.Tensor, step: int,
              lr: float, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.0, peer=None) -> None:
    """In-place torch.optim.Adam update of flat fp32 device buffers with identical layouts (one kernel).
    ``peer`` (a :class:`_lib.PeerGroup` from ``dist.PeerExchange.group()``): the gradient is the SUM of every rank's
    buffer, read over NVLink peer memory inside the same kernel -- ``grad`` is then only this rank's share."""
    lib = _lib.load()
    for name, t in (("param", param), ("grad", grad), ("exp_avg", exp_avg), ("exp_avg_sq", exp_avg_sq)):
        if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and t.numel() == param.numel()):
            raise ValueError(f"adam_step: {name} must be a contiguous fp32 CUDA tensor of {param.numel()} elements")
    if peer is not None:
        _lib.check(lib.ptrb200_adam_step_peer(C.byref(peer), param.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(), param.numel(),
                                              float(lr), float(betas[0]), float(betas[1]), float(eps), float(weight_decay), int(step),
                                              _stream_ptr()), "adam_step_peer")
        return
    _lib.check(lib.ptrb200_adam_step(param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(), param.numel(),
                                     float(lr), float(betas[0]), float(betas[1]), float(eps), float(weight_decay), int(step),
                                     _stream_ptr()), "adam_step")


@_on_tensor_device
def peer_allreduce_sum(out: torch.Tensor, peer) -> torch.Tensor:
    """out[i] = sum over ranks of their exchange buffers (rank order, identical on every rank) -- the bare exchange."""
    if not (out.is_cuda and out.dtype == torch.float32 and out.is_contiguous()):
        raise ValueError("peer_allreduce_sum: out must be a contiguous fp32 CUDA tensor")
    _lib.check(_lib.load().ptrb200_peer_allreduce_sum(C.byref(peer), out.data_ptr(), out.numel(), _stream_ptr()), "peer_allreduce_sum")
    return out


def _check_flat(who, param, *others):
    for t in (param, *others):
        if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and t.numel() == param.numel()):
            raise ValueError(f"{who}: every buffer must be a contiguous fp32 CUDA tensor of {param.numel()} elements")


@_on_tensor_device
def adagrad_step(param: torch.Tensor, grad: torch.Tensor, state_sum: torch.Tensor, step: int, lr: float,
                 lr_decay: float = 0.0, eps: float = 1e-10, weight_decay: float = 0.0, peer=None) -> None:
    """In-place torch.optim.Adagrad update of flat fp32 device buffers (one kernel; ``peer`` as in :func:`adam_step`)."""
    _check_flat("adagrad_step", param, grad, state_sum)
    if peer is not None:
        _lib.check(_lib.load().ptrb200_adagrad_step_peer(C.byref(peer), param.data_ptr(), state_sum.data_ptr(), param.numel(),
                                                         float(lr), float(lr_decay), float(eps), float(weight_decay), int(step),
                                                         _stream_ptr()), "adagrad_step_peer")
        return
    _lib.check(_lib.load().ptrb200_adagrad_step(param.data_ptr(), grad.data_ptr(), state_sum.data_ptr(), param.numel(),
                                                float(lr), float(lr_decay), float(eps), float(weight_decay), int(step),
                                                _stream_ptr()), "adagrad_step")


@_on_tensor_device
def rmsprop_step(param: torch.Tensor, grad: torch.Tensor, square_avg: torch.Tensor, lr: float, alpha: float = 0.99,
                 eps: float = 1e-8, weight_decay: float = 0.0, peer=None) -> None:
    """In-place torch.optim.RMSprop (momentum=0, centered=False) update of flat fp32 device buffers (one kernel;
    ``peer`` as in :func:`adam_step`)."""
    _check_flat("rmsprop_step", param, grad, square_avg)
    if peer is not None:
        _lib.check(_lib.load().ptrb200_rmsprop_step_peer(C.byref(peer), param.data_ptr(), square_avg.data_ptr(), param.numel(),
                                                         float(lr), float(alpha), float(eps), float(weight_decay),
                                                         _stream_ptr()), "rmsprop_step_peer")
        return
    _lib.check(_lib.load().ptrb200_rmsprop_step(param.data_ptr(), grad.data_ptr(), square_avg.data_ptr(), param.numel(),
                                                float(lr), float(alpha), float(eps), float(weight_decay),
                                                _stream_ptr()), "rmsprop_step")


class _RankLoss(torch.autograd.Function):
    """batch loss = sum of per-query losses; backward hands the fused gradient to the scorer."""

    @staticmethod
    @_on_tensor_device
    def forward(ctx, scores, labels, name, params):
        loss_q, grad = _loss_call(name, scores.detach(), labels, params)
        ctx.save_for_backward(grad)
        ctx.mark_non_differentiable(loss_q)
        ctx.set_materialize_grads(False)        # no zero-filled gradient for the per-query by-product
        return sum_f32(loss_q), loss_q

    @staticmethod
    @_on_tensor_device
    def backward(ctx, g_loss, _g_lq):
        (grad,) = ctx.saved_tensors
        if g_loss is None:
            return None, None, None, None
        # d(sum_q loss_q)/d scores scaled by the incoming scalar gradient -- our elementwise kernel, not an ATen launch
        return _ew(EW_MUL_SCALAR, grad, g_loss.reshape(1)), None, None, None


def rank_loss(name: str, scores: torch.Tensor, labels: torch.Tensor, **params) -> torch.Tensor:
    """0-dim batch loss of the named ranking loss, differentiable w.r.t. ``scores``."""
    loss, _ = _RankLoss.apply(scores, labels, name, params)
    return loss


def rank_loss_and_grad(name: str, scores: torch.Tensor, labels: torch.Tensor, **params):
    """(batch loss, per-query losses, d loss / d scores) without autograd."""
    loss_q, grad = _loss_call(name, scores.detach(), labels, params)
    return sum_f32(loss_q), loss_q, grad


_tie_offset = 0


@_on_tensor_device
def shuffle_ties_perm(labels: torch.Tensor, seed: Optional[int] = None, offset: Optional[int] = None,
                      offsets: Optional[torch.Tensor] = None, max_len: Optional[int] = None, buckets=None) -> torch.Tensor:
    """int32 ordering (positions within each query's list) of each query's labels, descending, ties in random order;
    same layout as ``labels`` ([B,n], or flat with ``offsets``/``max_len`` for a ragged batch)."""
    global _tie_offset
    lib = _lib.load()
    y = _dev_f32(labels, "labels")
    B, n, offsets, op = _list_layout(y, offsets, max_len)
    perm = torch.empty(y.shape, dtype=torch.int32, device=y.device)
    if seed is None:
        seed = torch.initial_seed()
    if offset is None:
        _tie_offset += 1
        offset = _tie_offset
    for q0, Bq, nq in _launch_ranges(B, n, offsets, buckets, False):
        _lib.check(lib.ptrb200_shuffle_ties_perm(y.data_ptr(), None if op is None else op + 4 * q0, perm.data_ptr(), Bq, nq,
                                                 seed & (2 ** 64 - 1), offset & (2 ** 64 - 1), _stream_ptr()), "shuffle_ties_perm")
    return perm


# --------------------------------------------------------------------------- #
# input side
# --------------------------------------------------------------------------- #
@_on_tensor_device
def standard_scale(X: torch.Tensor, offsets: Optional[torch.Tensor] = None, max_len: Optional[int] = None,
                   clip_max: Optional[float] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Per-query StandardScaler (data_utils.py:482-487) on the device.  X: [B,n,F], or flat [total_docs,F] with
    ``offsets``/``max_len``.  ``clip_max``: clamp features first (the loader's ISTELLA_MAX clip)."""
    lib = _lib.load()
    X = _dev_f32(X, "X")
    if offsets is None:
        if X.dim() != 3:
            raise ValueError(f"expected [B,n,F] features, got {tuple(X.shape)}")
        B, n, F, op = X.shape[0], X.shape[1], X.shape[2], None
    else:
        if X.dim() != 2 or max_len is None:
            raise ValueError("ragged features are [total_docs, F] with offsets= and max_len=")
        offsets = offsets.to(device=X.device, dtype=torch.int32).contiguous()
        B, n, F, op = offsets.numel() - 1, max(int(max_len), 1), X.shape[1], offsets.data_ptr()
    if out is None:
        out = torch.empty_like(X)
    _lib.check(lib.ptrb200_standard_scale(X.data_ptr(), op, out.data_ptr(), B, n, F, int(clip_max is not None),
                                          float(clip_max if clip_max is not None else 0.0), _stream_ptr()), "standard_scale")
    return out


# --------------------------------------------------------------------------- #
# metric
# --------------------------------------------------------------------------- #
@_on_tensor_device
def ndcg_at_ks(scores: torch.Tensor, labels: torch.Tensor, ks: Sequence[int], presort: bool = False,
               return_order: bool = False, offsets: Optional[torch.Tensor] = None, max_len: Optional[int] = None, buckets=None):
    """Per-query nDCG at the cutoffs ``ks`` -> [B, len(ks)] (zero where k > n).  ``offsets``/``max_len``: ragged batch."""
    lib = _lib.load()
    s, y = _dev_f32(scores, "scores"), _dev_f32(labels, "labels")
    if s.shape != y.shape:
        raise ValueError(f"expected scores/labels of identical shape, got {tuple(s.shape)} / {tuple(y.shape)}")
    B, n, offsets, op = _list_layout(s, offsets, max_len)
    ks = [int(k) for k in ks]
    order_ix = sorted(range(len(ks)), key=lambda i: ks[i])
    ks_sorted = [ks[i] for i in order_ix]
    arr = (C.c_int32 * len(ks))(*ks_sorted)
    out = torch.empty((B, len(ks)), dtype=torch.float32, device=s.device)
    order = torch.empty(s.shape, dtype=torch.int32, device=s.device) if return_order else None
    for q0, Bq, nq in _launch_ranges(B, n, offsets, buckets, False):
        _lib.check(lib.ptrb200_ndcg_at_ks(s.data_ptr(), y.data_ptr(), None if op is None else op + 4 * q0, arr, len(ks),
                                          out.data_ptr() + 4 * q0 * len(ks), order.data_ptr() if return_order else None, Bq, nq,
                                          int(bool(presort)), _stream_ptr()), "ndcg_at_ks")
    if order_ix != list(range(len(ks))):
        inv = torch.empty(len(ks), dtype=torch.long)
        inv[torch.tensor(order_ix)] = torch.arange(len(ks))
        out = out[:, inv.to(out.device)]
    return (out, order) if return_order else out


@_on_tensor_device
def adhoc_metrics_at_ks(scores: torch.Tensor, labels: torch.Tensor, ks: Sequence[int], presort: bool = False,
                        max_label: Optional[float] = None, offsets: Optional[torch.Tensor] = None,
                        max_len: Optional[int] = None, buckets=None):
    """(nDCG, nERR, AP, P) per query at the cutoffs ``ks`` -> four [B, len(ks)] tensors from one kernel."""
    lib = _lib.load()
    s, y = _dev_f32(scores, "scores"), _dev_f32(labels, "labels")
    if s.shape != y.shape:
        raise ValueError(f"expected scores/labels of identical shape, got {tuple(s.shape)} / {tuple(y.shape)}")
    B, n, offsets, op = _list_layout(s, offsets, max_len)
    ks = [int(k) for k in ks]
    order_ix = sorted(range(len(ks)), key=lambda i: ks[i])
    arr = (C.c_int32 * len(ks))(*[ks[i] for i in order_ix])
    if max_label is None:                       # the reference falls back to the maximum over the batch
        max_label = float(y.max())
    out = torch.empty((B, 4, len(ks)), dtype=torch.float32, device=s.device)
    for q0, Bq, nq in _launch_ranges(B, n, offsets, buckets, False):
        _lib.check(lib.ptrb200_adhoc_metrics_at_ks(s.data_ptr(), y.data_ptr(), None if op is None else op + 4 * q0, arr, len(ks),
                                                   out.data_ptr() + 16 * q0 * len(ks), Bq, nq, int(bool(presort)), float(max_label),
                                                   _stream_ptr()), "adhoc_metrics_at_ks")
    if order_ix != list(range(len(ks))):
        inv = torch.empty(len(ks), dtype=torch.long)
        inv[torch.tensor(order_ix)] = torch.arange(len(ks))
        out = out[:, :, inv.to(out.device)]
    return out[:, 0], out[:, 1], out[:, 2], out[:, 3]


# --------------------------------------------------------------------------- #
# stacked feed-forward scorer
# --------------------------------------------------------------------------- #
_dropout_offset = 0


def next_dropout_offset() -> int:
    global _dropout_offset
    _dropout_offset += 1
    return _dropout_offset


def _b200dist():
    from . import dist as b200dist          # late import: dist imports nothing from ops, ops only needs it at call time
    return b200dist


class FFNetSpec:
    """Static description of one stacked FF net + the order its parameters are passed in."""

    def __init__(self, dims, act_hidden, act_tail, norm, norm_affine, dropout_p, math_mode="3xtf32"):
        if len(dims) - 1 > _lib.MAX_FF_LAYERS:
            raise ValueError("too many layers")
        self.dims = [int(d) for d in dims]
        self.act_hidden, self.act_tail = act_hidden, act_tail
        self.norm, self.norm_affine, self.dropout_p = norm, bool(norm_affine), float(dropout_p)
        if math_mode not in _lib.MATH_MODES:
            raise ValueError(f"math_mode must be one of {sorted(_lib.MATH_MODES)}")
        self.math_mode = math_mode
        self.L = len(dims) - 1
        # slots[l] = names of the parameter tensors layer l owns, in flattening order
        self.slots = []
        for l in range(self.L):
            names = ["weight", "bias"]
            has_act = l < self.L - 1 or act_tail is not None
            if has_act and norm == "BN" and self.norm_affine:
                names += ["gamma", "beta"]
            if has_act and norm == "BN2":
                names += ["gamma", "beta"] + (["aff_w", "aff_b"] if self.norm_affine else [])
            self.slots.append(names)

    def describe(self, params: Sequence[torch.Tensor]) -> "_lib.FFNetDesc":
        d = _lib.FFNetDesc()
        d.num_linear = self.L
        for i, v in enumerate(self.dims):
            d.dims[i] = v
        d.act_hidden = _lib.AF_CODES[self.act_hidden]
        d.act_tail = _lib.AF_CODES[self.act_tail]
        d.norm = _lib.NORM_CODES[self.norm]
        d.norm_affine = int(self.norm_affine)
        d.dropout_p = self.dropout_p
        d.math_mode = _lib.MATH_MODES[self.math_mode]
        d.sync_bn = int(self.norm == "BN" and _b200dist().sync_bn_active())
        it = iter(params)
        for l, names in enumerate(self.slots):
            for nm in names:
                getattr(d, nm)[l] = next(it).data_ptr()
        return d

    def grads(self, params: Sequence[torch.Tensor], targets=None):
        """Gradient descriptor.  ``targets`` (optional, one tensor per parameter) are written in place --
        the flat data-parallel gradient bucket -- instead of fresh tensors autograd would have to add."""
        g = _lib.FFNetGrads()
        outs = []
        it = iter(params)
        i = 0
        for l, names in enumerate(self.slots):
            for nm in names:
                p = next(it)
                t = targets[i] if targets is not None else torch.empty_like(p)
                i += 1
                outs.append(t)
                getattr(g, nm)[l] = t.data_ptr()
        return g, outs


class _FFNetFn(torch.autograd.Function):
    @staticmethod
    @_on_tensor_device
    def forward(ctx, X, spec: FFNetSpec, training: bool, seed: int, offset: int, grad_targets, need_backward, ragged, *params):
        lib = _lib.load()
        X = _dev_f32(X, "X")
        if ragged is None:          # dense [B,n,F]
            B, n, F = X.shape
            offsets, op, total = None, None, 0
            out_shape = (B, n, spec.dims[-1])
        else:                       # ragged: [total_docs, F] rows cut into queries by int32 prefix offsets
            offsets, n = ragged
            offsets = offsets.to(device=X.device, dtype=torch.int32).contiguous()
            total, F = X.shape
            B, op = offsets.numel() - 1, offsets.data_ptr()
            out_shape = (total, spec.dims[-1])
        if F != spec.dims[0]:
            raise ValueError(f"feature width {F} != net input width {spec.dims[0]}")
        params = [p.detach().contiguous() for p in params]
        desc = spec.describe(params)
        nbytes = lib.ptrb200_ffnet_workspace_bytes(C.byref(desc), B, n, total)
        if nbytes < 0:
            _lib.check(int(nbytes), "ffnet_workspace_bytes")
        ws = torch.empty(int(nbytes), dtype=torch.uint8, device=X.device)
        out = torch.empty(out_shape, dtype=torch.float32, device=X.device)
        # bit 1 = forward only (PTRB200_FFNET_FORWARD_ONLY): no backward will follow (nothing requires grad, or the
        # caller runs under torch.no_grad()), so the by-products the backward pass reads are not written
        flags = int(training) | (0 if need_backward else 2)
        with _b200dist().call_context(ws, None):
            _lib.check(lib.ptrb200_ffnet_forward(C.byref(desc), X.data_ptr(), out.data_ptr(), ws.data_ptr(), int(nbytes),
                                                 B, n, op, total, flags, seed, offset, _stream_ptr()), "ffnet_forward")
        ctx.spec, ctx.training, ctx.seed, ctx.offset = spec, training, seed, offset
        ctx.shape = (B, n, offsets, total)
        ctx.grad_targets = grad_targets
        ctx.ws, ctx.nbytes = (ws if need_backward else None), int(nbytes)
        ctx.need_dx = X.requires_grad
        ctx.save_for_backward(X, *params)
        return out

    @staticmethod
    @_on_tensor_device
    def backward(ctx, d_out):
        lib = _lib.load()
        X, *params = ctx.saved_tensors
        spec = ctx.spec
        B, n, offsets, total = ctx.shape
        desc = spec.describe(params)
        gdesc, gouts = spec.grads(params, ctx.grad_targets)
        d_out = _dev_f32(d_out, "d_out")
        dX = torch.empty_like(X) if ctx.need_dx else None
        # per-layer gradient tensors (write-through targets only): lets a data-parallel bucket start reducing a layer's
        # slice as soon as the library reports it complete
        layer_targets = None
        if ctx.grad_targets is not None:
            layer_targets, i = [], 0
            for names in spec.slots:
                layer_targets.append(gouts[i: i + len(names)])
                i += len(names)
        with _b200dist().call_context(ctx.ws, layer_targets):
            _lib.check(lib.ptrb200_ffnet_backward(C.byref(desc), C.byref(gdesc), X.data_ptr(), d_out.data_ptr(),
                                                  dX.data_ptr() if dX is not None else None, ctx.ws.data_ptr(), ctx.nbytes,
                                                  B, n, offsets.data_ptr() if offsets is not None else None, total,
                                                  int(ctx.training), ctx.seed, ctx.offset, _stream_ptr()),
                       "ffnet_backward")
        ctx.ws = None
        if ctx.grad_targets is not None:            # written straight into the parameters' .grad storage
            return (dX, None, None, None, None, None, None, None, *([None] * len(gouts)))
        return (dX, None, None, None, None, None, None, None, *gouts)


def ffnet_apply(X: torch.Tensor, spec: FFNetSpec, params: Sequence[torch.Tensor], training: bool,
                seed: Optional[int] = None, offset: Optional[int] = None, grad_targets=None,
                offsets: Optional[torch.Tensor] = None, max_len: Optional[int] = None) -> torch.Tensor:
    """[B,n,F] -> [B,n,out] through the fused stacked-FF kernels (differentiable).  ``grad_targets``: tensors the
    parameter gradients are written into directly (each parameter must be used by exactly one call per step).
    ``offsets``/``max_len``: X is a ragged batch [total_docs, F] -> [total_docs, out] (per-query BN2 uses the boundaries)."""
    if seed is None:
        seed = torch.initial_seed() & (2 ** 64 - 1)
    if offset is None:
        offset = next_dropout_offset()
    need_backward = torch.is_grad_enabled() and (X.requires_grad or any(p.requires_grad for p in params))
    ragged = None
    if offsets is not None:
        if X.dim() != 2 or max_len is None:
            raise ValueError("a ragged batch is [total_docs, F] with offsets= and max_len=")
        ragged = (offsets, max(int(max_len), 1))
    return _FFNetFn.apply(X, spec, bool(training), int(seed), int(offset), grad_targets, bool(need_backward), ragged, *params)


# --------------------------------------------------------------------------- #
# list scorer pieces: linear, attention core, reference LayerNorm, elementwise glue
# --------------------------------------------------------------------------- #
_linear_specs = {}


def linear(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, math_mode: str = "3xtf32") -> torch.Tensor:
    """nn.Linear over [B,n,in] through the stacked-FF kernels (a one-layer net without activation)."""
    key = (weight.shape[1], weight.shape[0], math_mode)
    if key not in _linear_specs:
        _linear_specs[key] = FFNetSpec([key[0], key[1]], None, None, None, False, 0.0, math_mode=math_mode)
    return ffnet_apply(x, _linear_specs[key], [weight, bias], training=False, seed=0, offset=0)


# ---- ragged batches through the list scorer: pad in, mask the padded keys, gather out ----------------------------------
_key_lens: Optional[torch.Tensor] = None      # int32[B] on the device while a padded ragged batch is inside the list scorer


@contextlib.contextmanager
def key_lens_context(lens: Optional[torch.Tensor]):
    """Inside the context every tensor-core attention call masks, for query b, the keys at positions >= lens[b]."""
    global _key_lens
    prev, _key_lens = _key_lens, lens
    try:
        yield
    finally:
        _key_lens = prev


class _PadLists(torch.autograd.Function):
    """flat [total, F] + offsets[B+1] -> padded [B, n_max, F] (zeros behind each list); backward gathers the rows back."""

    @staticmethod
    @_on_tensor_device
    def forward(ctx, flat, offsets, n_max):
        lib = _lib.load()
        flat = _dev_f32(flat, "flat")
        F = flat.shape[1] if flat.dim() == 2 else 1
        B = offsets.numel() - 1
        out = torch.empty((B, n_max, F) if flat.dim() == 2 else (B, n_max), dtype=torch.float32, device=flat.device)
        _lib.check(lib.ptrb200_pad_lists(flat.data_ptr(), offsets.data_ptr(), out.data_ptr(), B, n_max, F, _stream_ptr()), "pad_lists")
        ctx.save_for_backward(offsets)
        ctx.shape = tuple(flat.shape)
        return out

    @staticmethod
    @_on_tensor_device
    def backward(ctx, g):
        (offsets,) = ctx.saved_tensors
        lib = _lib.load()
        g = _dev_f32(g, "g")
        F = ctx.shape[1] if len(ctx.shape) == 2 else 1
        out = torch.zeros(ctx.shape, dtype=torch.float32, device=g.device)     # offsets may address a sub-range of the rows
        _lib.check(lib.ptrb200_unpad_lists(g.data_ptr(), offsets.data_ptr(), out.data_ptr(), offsets.numel() - 1, g.shape[1], F,
                                           _stream_ptr()), "unpad_lists")
        return out, None, None


class _UnpadLists(torch.autograd.Function):
    """padded [B, n_max(, F)] -> flat [total(, F)]; backward pads the gradient (zeros at the padding)."""

    @staticmethod
    @_on_tensor_device
    def forward(ctx, padded, offsets, total):
        lib = _lib.load()
        padded = _dev_f32(padded, "padded")
        F = padded.shape[2] if padded.dim() == 3 else 1
        B, n_max = padded.shape[0], padded.shape[1]
        out = torch.empty((total, F) if padded.dim() == 3 else (total,), dtype=torch.float32, device=padded.device)
        _lib.check(lib.ptrb200_unpad_lists(padded.data_ptr(), offsets.data_ptr(), out.data_ptr(), B, n_max, F, _stream_ptr()), "unpad_lists")
        ctx.save_for_backward(offsets)
        ctx.shape = tuple(padded.shape)
        return out

    @staticmethod
    @_on_tensor_device
    def backward(ctx, g):
        (offsets,) = ctx.saved_tensors
        lib = _lib.load()
        g = _dev_f32(g, "g")
        F = ctx.shape[2] if len(ctx.shape) == 3 else 1
        out = torch.empty(ctx.shape, dtype=torch.float32, device=g.device)
        _lib.check(lib.ptrb200_pad_lists(g.data_ptr(), offsets.data_ptr(), out.data_ptr(), ctx.shape[0], ctx.shape[1], F,
                                         _stream_ptr()), "pad_lists")
        return out, None, None


class _UnpadBuckets(torch.autograd.Function):
    """Padded score blocks of consecutive query ranges -> one flat [total] vector (every block gathers into ITS rows through
    the absolute prefix offsets); backward pads the gradient block by block."""

    @staticmethod
    @_on_tensor_device
    def forward(ctx, offsets, total, q0s, *blocks):
        lib = _lib.load()
        blocks = [_dev_f32(b, "block") for b in blocks]
        out = torch.empty((total,), dtype=torch.float32, device=blocks[0].device)
        for q0, b in zip(q0s, blocks):
            _lib.check(lib.ptrb200_unpad_lists(b.data_ptr(), offsets.data_ptr() + 4 * q0, out.data_ptr(), b.shape[0], b.shape[1], 1,
                                               _stream_ptr()), "unpad_lists")
        ctx.save_for_backward(offsets)
        ctx.q0s, ctx.shapes = list(q0s), [tuple(b.shape) for b in blocks]
        return out

    @staticmethod
    @_on_tensor_device
    def backward(ctx, g):
        (offsets,) = ctx.saved_tensors
        lib = _lib.load()
        g = _dev_f32(g, "g")
        outs = []
        for q0, shp in zip(ctx.q0s, ctx.shapes):
            o = torch.empty(shp, dtype=torch.float32, device=g.device)
            _lib.check(lib.ptrb200_pad_lists(g.data_ptr(), offsets.data_ptr() + 4 * q0, o.data_ptr(), shp[0], shp[1], 1, _stream_ptr()), "pad_lists")
            outs.append(o)
        return (None, None, None, *outs)


def unpad_buckets(blocks: Sequence[torch.Tensor], offsets: torch.Tensor, total: int, q0s: Sequence[int]) -> torch.Tensor:
    """Flat [total] scores from padded blocks [B_k, n_k] of consecutive query ranges starting at queries ``q0s``."""
    if sum(b.shape[0] for b in blocks) != offsets.numel() - 1:
        raise ValueError("the blocks must cover every query once")
    return _UnpadBuckets.apply(_offsets_i32(offsets, blocks[0].device), int(total), [int(q) for q in q0s], *blocks)


def _offsets_i32(offsets: torch.Tensor, device) -> torch.Tensor:
    return offsets.to(device=device, dtype=torch.int32).contiguous()


def pad_lists(flat: torch.Tensor, offsets: torch.Tensor, n_max: int) -> torch.Tensor:
    """Ragged rows [total, F] (or [total]) -> dense [B, n_max, F] ([B, n_max]), zero behind each list (differentiable)."""
    return _PadLists.apply(flat, _offsets_i32(offsets, flat.device), int(n_max))


def unpad_lists(padded: torch.Tensor, offsets: torch.Tensor, total: int) -> torch.Tensor:
    """Inverse of :func:`pad_lists`: the first len_b rows of every list, concatenated (differentiable)."""
    return _UnpadLists.apply(padded, _offsets_i32(offsets, padded.device), int(total))


class _Attention(torch.autograd.Function):
    @staticmethod
    @_on_tensor_device
    def forward(ctx, Q, K, V, n_heads, dropout_p, seed, offset):
        lib = _lib.load()
        Q, K, V = _dev_f32(Q, "Q"), _dev_f32(K, "K"), _dev_f32(V, "V")
        B, n, F = Q.shape
        D = F // n_heads
        O = torch.empty_like(Q)
        lse = torch.empty((B, n_heads, n), dtype=torch.float32, device=Q.device)
        _lib.check(lib.ptrb200_attention_fwd(Q.data_ptr(), K.data_ptr(), V.data_ptr(), O.data_ptr(), lse.data_ptr(),
                                             B, n, n_heads, D, float(dropout_p), seed, offset, _stream_ptr()), "attention_fwd")
        ctx.save_for_backward(Q, K, V, O, lse)
        ctx.cfg = (n_heads, float(dropout_p), seed, offset)
        return O

    @staticmethod
    @_on_tensor_device
    def backward(ctx, dO):
        lib = _lib.load()
        Q, K, V, O, lse = ctx.saved_tensors
        H, p, seed, offset = ctx.cfg
        B, n, F = Q.shape
        dO = _dev_f32(dO, "dO")
        dQ, dK, dV = torch.empty_like(Q), torch.empty_like(K), torch.empty_like(V)
        scratch = torch.empty(B * H * n, dtype=torch.float32, device=Q.device)
        _lib.check(lib.ptrb200_attention_bwd(Q.data_ptr(), K.data_ptr(), V.data_ptr(), O.data_ptr(), dO.data_ptr(),
                                             lse.data_ptr(), dQ.data_ptr(), dK.data_ptr(), dV.data_ptr(), scratch.data_ptr(),
                                             B, n, H, F // H, p, seed, offset, _stream_ptr()), "attention_bwd")
        return dQ, dK, dV, None, None, None, None


def _key_lens_ptr(B: int, device):
    """Device pointer of the active key-length vector (None outside :func:`key_lens_context`)."""
    if _key_lens is None:
        return None
    if _key_lens.numel() != B or _key_lens.device != device or _key_lens.dtype != torch.int32:
        raise ValueError("key_lens_context: expected an int32 vector with one entry per query on the tensors' device")
    return _key_lens.data_ptr()


class _AttentionTC(torch.autograd.Function):
    """Tensor-core attention: batched tcgen05 GEMMs around a materialised [B*H,n,n] probability tensor."""

    @staticmethod
    @_on_tensor_device
    def forward(ctx, Q, K, V, n_heads, dropout_p, seed, offset, passes):
        lib = _lib.load()
        Q, K, V = _dev_f32(Q, "Q"), _dev_f32(K, "K"), _dev_f32(V, "V")
        B, n, F = Q.shape
        D = F // n_heads
        O = torch.empty_like(Q)
        P = torch.empty((B * n_heads, n, n), dtype=torch.float32, device=Q.device)
        scratch = torch.empty(lib.ptrb200_attention_tc_workspace_floats(B, n, n_heads, D, 0), dtype=torch.float32, device=Q.device)
        _lib.check(lib.ptrb200_attention_tc_fwd_ld(Q.data_ptr(), K.data_ptr(), V.data_ptr(), O.data_ptr(), P.data_ptr(),
                                                   scratch.data_ptr(), B, n, n_heads, D, 0, 0, _key_lens_ptr(B, Q.device),
                                                   float(dropout_p), seed, offset, passes, _stream_ptr()), "attention_tc_fwd")
        ctx.save_for_backward(Q, K, V, P)
        ctx.cfg = (n_heads, float(dropout_p), seed, offset, passes)
        return O

    @staticmethod
    @_on_tensor_device
    def backward(ctx, dO):
        lib = _lib.load()
        Q, K, V, P = ctx.saved_tensors
        H, p, seed, offset, passes = ctx.cfg
        B, n, F = Q.shape
        dO = _dev_f32(dO, "dO")
        dQ, dK, dV = torch.empty_like(Q), torch.empty_like(K), torch.empty_like(V)
        scratch = torch.empty(lib.ptrb200_attention_tc_workspace_floats(B, n, H, F // H, 1), dtype=torch.float32, device=Q.device)
        _lib.check(lib.ptrb200_attention_tc_bwd(Q.data_ptr(), K.data_ptr(), V.data_ptr(), P.data_ptr(), dO.data_ptr(),
                                                dQ.data_ptr(), dK.data_ptr(), dV.data_ptr(), scratch.data_ptr(),
                                                B, n, H, F // H, p, seed, offset, passes, _stream_ptr()), "attention_tc_bwd")
        return dQ, dK, dV, None, None, None, None, None


def attention(Q, K, V, n_heads: int, dropout_p: float = 0.0, seed: Optional[int] = None, offset: Optional[int] = None,
              impl: Optional[str] = None):
    """softmax(Q K^T / sqrt(d)) [dropout] V per head; Q,K,V: [B,n,H*d].

    impl: "tc" (tcgen05 3xTF32 GEMMs, default), "tc_tf32" (single-pass TF32), "simt" (flash-style fp32 FMA kernels);
    None reads PTRANKING_B200_ATTN.  All three draw the same dropout stream."""
    if seed is None:
        seed = torch.initial_seed() & (2 ** 64 - 1)
    if offset is None:
        offset = next_dropout_offset()
    if impl is None:
        impl = os.environ.get("PTRANKING_B200_ATTN", "tc")
    if impl == "simt":
        if _key_lens is not None:
            raise NotImplementedError("padded ragged batches need a tensor-core attention impl (PTRANKING_B200_ATTN=tc)")
        return _Attention.apply(Q, K, V, int(n_heads), float(dropout_p), int(seed), int(offset))
    if impl not in ("tc", "tc_tf32"):
        raise ValueError(f"unknown attention impl {impl!r}")
    return _AttentionTC.apply(Q, K, V, int(n_heads), float(dropout_p), int(seed), int(offset), 3 if impl == "tc" else 1)


class _AdjacentRows(torch.autograd.Function):
    """Stack parameter tensors along dim 0.  When they already sit side by side in one storage (the ranker's flat
    parameter buffer orders an attention block's three projection weights that way) the stack is a strided view of that
    storage -- no copy, no kernel; otherwise a plain copy.  Backward hands every tensor its rows of the gradient."""

    @staticmethod
    def forward(ctx, *ts):
        ctx.sizes = [t.shape[0] for t in ts]
        first = ts[0]
        off, adjacent = first.storage_offset(), True
        for t in ts:
            adjacent = adjacent and t.is_contiguous() and t.shape[1:] == first.shape[1:] and t.dtype == first.dtype \
                and t.untyped_storage().data_ptr() == first.untyped_storage().data_ptr() and t.storage_offset() == off
            off += t.numel()
        if adjacent:
            return torch.as_strided(first.detach(), (sum(ctx.sizes), *first.shape[1:]), first.stride(), first.storage_offset())
        return torch.cat([t.detach() for t in ts], 0)

    @staticmethod
    def backward(ctx, g):
        return tuple(torch.split(g, ctx.sizes, 0))


def adjacent_rows(*ts: torch.Tensor) -> torch.Tensor:
    return _AdjacentRows.apply(*ts)


class _AttentionTCPacked(torch.autograd.Function):
    """_AttentionTC over Q|K|V side by side in one [B,n,3*F] tensor (the output of one F -> 3F projection): the kernels
    read the three column blocks in place through their row pitch and the backward pass fills one [B,n,3*F] gradient."""

    @staticmethod
    @_on_tensor_device
    def forward(ctx, qkv, n_heads, dropout_p, seed, offset, passes):
        lib = _lib.load()
        qkv = _dev_f32(qkv, "qkv")
        B, n, F3 = qkv.shape
        F = F3 // 3
        D = F // n_heads
        O = torch.empty((B, n, F), dtype=torch.float32, device=qkv.device)
        P = torch.empty((B * n_heads, n, n), dtype=torch.float32, device=qkv.device)
        scratch = torch.empty(lib.ptrb200_attention_tc_workspace_floats(B, n, n_heads, D, 0), dtype=torch.float32, device=qkv.device)
        q = qkv.data_ptr()
        _lib.check(lib.ptrb200_attention_tc_fwd_ld(q, q + 4 * F, q + 8 * F, O.data_ptr(), P.data_ptr(), scratch.data_ptr(),
                                                   B, n, n_heads, D, F3, 0, _key_lens_ptr(B, qkv.device), float(dropout_p), seed, offset,
                                                   passes, _stream_ptr()), "attention_tc_fwd")
        ctx.save_for_backward(qkv, P)
        ctx.cfg = (n_heads, float(dropout_p), seed, offset, passes)
        return O

    @staticmethod
    @_on_tensor_device
    def backward(ctx, dO):
        lib = _lib.load()
        qkv, P = ctx.saved_tensors
        H, p, seed, offset, passes = ctx.cfg
        B, n, F3 = qkv.shape
        F = F3 // 3
        dO = _dev_f32(dO, "dO")
        dqkv = torch.empty_like(qkv)
        scratch = torch.empty(lib.ptrb200_attention_tc_workspace_floats(B, n, H, F // H, 1), dtype=torch.float32, device=qkv.device)
        q, g = qkv.data_ptr(), dqkv.data_ptr()
        _lib.check(lib.ptrb200_attention_tc_bwd_ld(q, q + 4 * F, q + 8 * F, P.data_ptr(), dO.data_ptr(),
                                                   g, g + 4 * F, g + 8 * F, scratch.data_ptr(),
                                                   B, n, H, F // H, F3, 0, p, seed, offset, passes, _stream_ptr()), "attention_tc_bwd")
        return dqkv, None, None, None, None, None


def attention_impl() -> str:
    return os.environ.get("PTRANKING_B200_ATTN", "tc")


def attention_packed(qkv, n_heads: int, dropout_p: float = 0.0, seed: Optional[int] = None, offset: Optional[int] = None,
                     impl: Optional[str] = None):
    """:func:`attention` for Q|K|V stored side by side in the last dimension of one tensor (tensor-core paths only)."""
    if seed is None:
        seed = torch.initial_seed() & (2 ** 64 - 1)
    if offset is None:
        offset = next_dropout_offset()
    if impl is None:
        impl = attention_impl()
    if impl not in ("tc", "tc_tf32"):
        raise ValueError(f"attention_packed needs a tensor-core impl, got {impl!r}")
    if qkv.shape[-1] % (3 * n_heads) != 0:
        raise ValueError("last dimension must be 3 * n_heads * head_dim")
    return _AttentionTCPacked.apply(qkv, int(n_heads), float(dropout_p), int(seed), int(offset), 3 if impl == "tc" else 1)


class _LayerNormRef(torch.autograd.Function):
    @staticmethod
    @_on_tensor_device
    def forward(ctx, x, a2, b2, eps):
        lib = _lib.load()
        x = _dev_f32(x, "x")
        F = x.shape[-1]
        rows = x.numel() // F
        y = torch.empty_like(x)
        mean = torch.empty(rows, dtype=torch.float32, device=x.device)
        std = torch.empty(rows, dtype=torch.float32, device=x.device)
        a2c, b2c = a2.detach().contiguous(), b2.detach().contiguous()
        _lib.check(lib.ptrb200_layernorm_fwd(x.data_ptr(), a2c.data_ptr(), b2c.data_ptr(), y.data_ptr(), mean.data_ptr(),
                                             std.data_ptr(), rows, F, float(eps), _stream_ptr()), "layernorm_fwd")
        ctx.save_for_backward(x, a2c, mean, std)
        ctx.eps = float(eps)
        return y

    @staticmethod
    @_on_tensor_device
    def backward(ctx, dy):
        lib = _lib.load()
        x, a2, mean, std = ctx.saved_tensors
        F = x.shape[-1]
        rows = x.numel() // F
        dy = _dev_f32(dy, "dy")
        dx = torch.empty_like(x)
        da2, db2 = torch.empty_like(a2), torch.empty_like(a2)
        scratch = torch.empty(297 * 2 * F, dtype=torch.float32, device=x.device)
        _lib.check(lib.ptrb200_layernorm_bwd(x.data_ptr(), a2.data_ptr(), dy.data_ptr(), mean.data_ptr(), std.data_ptr(),
                                             dx.data_ptr(), da2.data_ptr(), db2.data_ptr(), scratch.data_ptr(), rows, F,
                                             ctx.eps, _stream_ptr()), "layernorm_bwd")
        return dx, da2, db2, None


def layernorm_ref(x, a2, b2, eps: float = 1e-6):
    """The reference's hand-written LayerNorm (unbiased std, eps added to the std)."""
    return _LayerNormRef.apply(x, a2, b2, eps)


EW_ADD, EW_LATENT_CROSS, EW_MUL, EW_RELU, EW_RELU_BWD, EW_DROPOUT, EW_SCALE_ADD1, EW_MUL_SCALAR, EW_ACT, EW_ACT_GRAD = range(10)


@_on_tensor_device
def _ew(op, a, b=None, p=0.0, seed=0, offset=0):
    lib = _lib.load()
    a = _dev_f32(a, "a")
    bb = _dev_f32(b, "b") if b is not None else None
    out = torch.empty_like(a)
    _lib.check(lib.ptrb200_elementwise(op, a.data_ptr(), bb.data_ptr() if bb is not None else None, out.data_ptr(),
                                       a.numel(), float(p), seed, offset, _stream_ptr()), "elementwise")
    return out


def activation(x: torch.Tensor, code: str, grad: bool = False) -> torch.Tensor:
    """act(x) (or act'(x)) exactly as the scorer kernels evaluate get_AF's activation ``code`` -- for accuracy tests."""
    return _ew(EW_ACT_GRAD if grad else EW_ACT, x, None, 0.0, _lib.AF_CODES[code], 0)


class _Add(torch.autograd.Function):
    @staticmethod
    @_on_tensor_device
    def forward(ctx, a, b):
        return _ew(EW_ADD, a, b)

    @staticmethod
    @_on_tensor_device
    def backward(ctx, g):
        return g, g


class _LatentCross(torch.autograd.Function):
    """(enc + 1) * head -- DASALC's latent cross (list_ranker.py:366)."""

    @staticmethod
    @_on_tensor_device
    def forward(ctx, enc, head):
        ctx.save_for_backward(enc, head)
        return _ew(EW_LATENT_CROSS, enc, head)

    @staticmethod
    @_on_tensor_device
    def backward(ctx, g):
        enc, head = ctx.saved_tensors
        return _ew(EW_MUL, g, head), _ew(EW_SCALE_ADD1, g, enc)


class _Relu(torch.autograd.Function):
    @staticmethod
    @_on_tensor_device
    def forward(ctx, x):
        ctx.save_for_backward(x)
        return _ew(EW_RELU, x)

    @staticmethod
    @_on_tensor_device
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        return _ew(EW_RELU_BWD, g, x)


class _Dropout(torch.autograd.Function):
    @staticmethod
    @_on_tensor_device
    def forward(ctx, x, p, seed, offset):
        ctx.cfg = (p, seed, offset)
        return _ew(EW_DROPOUT, x, None, p, seed, offset)

    @staticmethod
    @_on_tensor_device
    def backward(ctx, g):
        p, seed, offset = ctx.cfg
        return _ew(EW_DROPOUT, g, None, p, seed, offset), None, None, None


def add(a, b):
    return _Add.apply(a, b)


def latent_cross(enc, head):
    return _LatentCross.apply(enc, head)


def relu(x):
    return _Relu.apply(x)


def dropout(x, p: float, training: bool):
    if not training or p <= 0.0:
        return x
    return _Dropout.apply(x, float(p), torch.initial_seed() & (2 ** 64 - 1), next_dropout_offset())
