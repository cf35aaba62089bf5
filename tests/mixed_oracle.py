"""The float64 training-step oracle (oracle/x3d_train_oracle.py) with the GEMM rounding of the
'mixed_bfloat16' policy -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Under that policy every 1x1x1 conv and Dense layer multiplies operands rounded to bf16 (round-to-
nearest-even of the fp32 value, as torch's `.to(torch.bfloat16)`) and accumulates exactly (here: in
float64):
    forward          y  = bf16(x) @ bf16(W)
    backward-data    dx = bf16(dy) @ bf16(W)^T
    backward-filter  dW = bf16(x)^T @ bf16(dy)
Everything else is the unchanged oracle.  `train_step(..., gemm_round=False)` is the oracle itself.

Rounding to bf16 is a kink at every tie, like ReLU at zero: the fp32 run and this float64 run hold
values ~1e-6 apart, so a few operands close to a tie round to different neighbours, and each such
element differs by a whole bf16 step (2^-8 relative).  Those differences feed the next rounded GEMM,
and within a few layers the two runs differ at the bf16 level (measured: 0.10 of the logits' scale at
X3D-XS).  So, as the ReLU branch masks do, the oracle can be told where the CUDA run rounded:
`operands` maps a layer name to the fp32 operands the device rounded ('fwd': the activation, 'bwd':
the output gradient).  An element then takes the device's bf16 value only if that value is one of its
own two bf16 neighbours; anything else keeps the oracle's rounding.  `FORCED` counts the elements whose
neighbour that changed.
"""
from __future__ import annotations

from unittest import mock

import numpy as np
import torch
import torch.nn.functional as F

from oracle import x3d_oracle as O
from oracle import x3d_train_oracle as TO


def bf16_rne(a: np.ndarray) -> np.ndarray:
    """Values of bf16(fp32(a)), round-to-nearest-even on the fp32 bit pattern (NaN not handled);
    returned as float64."""
    u = np.ascontiguousarray(np.asarray(a, np.float64).astype(np.float32)).view(np.uint32).astype(np.uint64)
    r = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return r.astype(np.uint32).view(np.float32).astype(np.float64)


FORCED = {"elements": 0, "forced": 0}


def _r(t: torch.Tensor, dev: np.ndarray = None) -> torch.Tensor:
    a = t.detach().cpu().numpy()
    own = bf16_rne(a)
    if dev is not None:
        d = bf16_rne(np.asarray(dev)[:a.shape[0], :a.shape[1]])
        lo = np.asarray(a, np.float32).view(np.uint32) & np.uint32(0xFFFF0000)
        hi = lo + np.uint32(0x10000)
        db = d.astype(np.float32).view(np.uint32)
        take = (db == lo) | (db == hi)
        FORCED["elements"] += a.size
        FORCED["forced"] += int((take & (d != own)).sum())
        own = np.where(take, d, own)
    return torch.from_numpy(own).to(t.dtype)


class RoundedMatmul(torch.autograd.Function):
    """x [M, K] @ w [K, N] with the policy's operand rounding in forward, backward-data and
    backward-filter; `xdev` / `dydev`: the device's fp32 operands (see the module docstring)."""

    @staticmethod
    def forward(ctx, x, w, xdev=None, dydev=None):
        ctx.save_for_backward(x, w)
        ctx.dev = (xdev, dydev)
        return _r(x, xdev) @ _r(w)

    @staticmethod
    def backward(ctx, dy):
        x, w = ctx.saved_tensors
        xdev, dydev = ctx.dev
        rdy = _r(dy, dydev)
        return rdy @ _r(w).t(), _r(x, xdev).t() @ rdy, None, None


def _mm(x, w, name, operands):
    fwd, bwd = (operands or {}).get(name, (None, None))
    return RoundedMatmul.apply(x, w, fwd, bwd)


def pw(x: torch.Tensor, k: torch.Tensor, name: str = None, operands: dict = None) -> torch.Tensor:
    """1x1x1 conv of NCDHW `x` with the DHWIO kernel `k` through RoundedMatmul."""
    n, c, d, h, w = x.shape
    y = _mm(x.permute(0, 2, 3, 4, 1).reshape(-1, c), k.reshape(c, -1), name, operands)
    return y.reshape(n, d, h, w, -1).permute(0, 4, 1, 2, 3)


def forward_train(P, spec, x, dropout_mask, stats, taps=None, relu_masks=None, operands=None):
    """`x3d_train_oracle.forward_train` with every 1x1x1 conv / Dense layer through `pw`."""
    def tap(name, t):
        if taps is not None:
            t.retain_grad()
            taps[name] = t
        return t
    masks = None if relu_masks is None else list(relu_masks)

    def relu(t):
        if masks is None:
            return F.relu(t)
        m = torch.from_numpy(np.asarray(masks.pop(0))).to(t.dtype)
        c = t.shape[1]
        m = m.reshape(t.shape[0], *t.shape[2:], -1)[..., :c].permute(0, 4, 1, 2, 3) if t.dim() == 5 \
            else m.reshape(t.shape[0], -1)[:, :c]
        return t * m
    eps = spec.bn_eps
    out = F.pad(x, (1, 1, 1, 1, 0, 0))
    out = F.conv3d(out, TO._k(P["conv1/conv_s/kernel"]), None, stride=(1, 2, 2))
    tp = spec.temp_filter // 2
    out = F.pad(out, (0, 0, 0, 0, tp, tp))
    out = F.conv3d(out, TO._k(P["conv1/conv_t/kernel"]), None, groups=spec.conv1_dim)
    out = relu(TO._bn_train(out, P, "conv1/bn", eps, stats))
    for (s, j, cin, inner, cout, stride, se, shortcut) in spec.blocks:
        p = f"stages/{s}/stage/layer_with_weights-{j}"
        q = p + "/bottleneck"
        xin = out
        out = pw(xin, P[q + "/a/kernel"], q + "/a/kernel", operands)
        out = relu(TO._bn_train(out, P, q + "/bn_a", eps, stats))
        out = O.conv3d_same(out, TO._k(P[q + "/b/kernel"]), (1, stride, stride), inner)
        out = TO._bn_train(out, P, q + "/bn_b", eps, stats)
        if se:
            m = out.mean(dim=(2, 3, 4), keepdim=True)
            z = F.relu(pw(m, P[q + "/se_fc1/kernel"], q + "/se_fc1/kernel", operands) + P[q + "/se_fc1/bias"].view(1, -1, 1, 1, 1))
            sc = torch.sigmoid(pw(z, P[q + "/se_fc2/kernel"], q + "/se_fc2/kernel", operands) + P[q + "/se_fc2/bias"].view(1, -1, 1, 1, 1))
            out = out * sc
        out = out * torch.sigmoid(out)
        out = pw(out, P[q + "/c/kernel"], q + "/c/kernel", operands)
        out = TO._bn_train(out, P, q + "/bn_c", eps, stats)
        if shortcut:
            res = pw(xin[:, :, :, ::stride, ::stride], P[p + "/residual/kernel"], p + "/residual/kernel", operands)
            res = TO._bn_train(res, P, p + "/bn_r", eps, stats)
        else:
            res = xin
        out = tap(p, relu(res + out))
    out = tap("conv5_pre", pw(out, P["conv5/layer_with_weights-0/kernel"], "conv5/layer_with_weights-0/kernel", operands))
    out = tap("conv5", relu(TO._bn_train(out, P, "conv5/layer_with_weights-1", eps, stats)))
    out = tap("pool5", out.mean(dim=(2, 3, 4), keepdim=True))
    out = pw(out, P["fc1/kernel"], "fc1/kernel", operands).reshape(out.shape[0], -1)
    out = tap("fc1", relu(out))
    if dropout_mask is not None:
        out = out * dropout_mask
    return _mm(out, P["fc2/kernel"], "fc2/kernel", operands) + P["fc2/bias"]


def train_step(*args, gemm_round: bool = True, operands: dict = None, **kw):
    """`x3d_train_oracle.train_step` (same arguments and result); `gemm_round` selects the policy's
    rounded GEMMs, False runs the oracle unchanged; `operands`: {layer name: (fwd, bwd)} as above."""
    if not gemm_round:
        return TO.train_step(*args, **kw)

    def fwd(*a, **k):
        return forward_train(*a, operands=operands, **k)
    with mock.patch.object(TO, "forward_train", fwd):
        return TO.train_step(*args, **kw)
