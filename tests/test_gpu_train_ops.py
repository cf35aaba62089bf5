"""Per-kernel parity of the training-step kernels (C ABI section "Training step") against
torch-CPU float64 autograd of the same op."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.gpu_util import dev, to_dev, to_np

pytestmark = pytest.mark.gpu


def _L():
    from x3d_tf_b200._lib import check, lib
    return lib(), check


def _st():
    return torch.cuda.current_stream().cuda_stream


def _close(got, want, tol=2e-5):
    want = np.asarray(want, np.float64)
    err = np.abs(np.asarray(got, np.float64) - want).max() / max(np.abs(want).max(), 1e-12)
    assert err < tol, err


@pytest.mark.parametrize("M,C,relu", [(32, 432, True), (1000, 56, False), (4099, 24, True), (8, 8, False)])
def test_batchnorm_train_fwd_bwd(M, C, relu):
    L, check = _L()
    rng = np.random.default_rng(M + C)
    x = (rng.normal(size=(M, C)) * rng.uniform(0.2, 3, size=C) + rng.normal(size=C)).astype(np.float32)
    gamma = rng.uniform(0.5, 1.5, size=C).astype(np.float32)
    beta = rng.normal(size=C).astype(np.float32) * 0.3
    dy = rng.normal(size=(M, C)).astype(np.float32)
    xt = torch.from_numpy(x).double().requires_grad_(True)
    gt = torch.from_numpy(gamma).double().requires_grad_(True)
    bt = torch.from_numpy(beta).double().requires_grad_(True)
    mean, var = xt.mean(0), xt.var(0, unbiased=False)
    yt = (xt - mean) * torch.rsqrt(var + 1e-5) * gt + bt
    if relu:
        yt = F.relu(yt)
    yt.backward(torch.from_numpy(dy).double())
    xd, dyd = to_dev(x), to_dev(dy)
    sums = torch.zeros((2, C), dtype=torch.float64, device=dev())
    check(L.x3d_colreduce(xd.data_ptr(), None, None, None, None, M, C, M, sums.data_ptr(), 0, _st()))
    m_, v_, r_ = (torch.empty(C, device=dev()) for _ in range(3))
    mm, mv = torch.zeros(C, device=dev()), torch.ones(C, device=dev())
    check(L.x3d_bn_finalize(sums.data_ptr(), M, C, 1e-5, 0.9, m_.data_ptr(), v_.data_ptr(), r_.data_ptr(),
                            mm.data_ptr(), mv.data_ptr(), _st()))
    y = torch.empty_like(xd)
    gd, bd = to_dev(gamma), to_dev(beta)
    check(L.x3d_bn_apply_fwd(xd.data_ptr(), m_.data_ptr(), r_.data_ptr(), gd.data_ptr(), bd.data_ptr(),
                             y.data_ptr(), M, C, int(relu), _st()))
    _close(to_np(y), yt.detach().numpy())
    _close(to_np(m_), mean.detach().numpy()); _close(to_np(v_), var.detach().numpy())
    _close(to_np(mm), 0.1 * mean.detach().numpy()); _close(to_np(mv), 0.9 + 0.1 * var.detach().numpy())
    s2 = torch.zeros((2, C), dtype=torch.float64, device=dev())
    check(L.x3d_colreduce(dyd.data_ptr(), xd.data_ptr(), m_.data_ptr(), r_.data_ptr(),
                          y.data_ptr() if relu else None, M, C, M, s2.data_ptr(), 1, _st()))
    dx = torch.empty_like(xd)
    check(L.x3d_bn_bwd_apply(dyd.data_ptr(), xd.data_ptr(), y.data_ptr() if relu else None, m_.data_ptr(),
                             r_.data_ptr(), gd.data_ptr(), s2.data_ptr(), dx.data_ptr(), M, C, _st()))
    torch.cuda.synchronize()
    _close(s2[0].cpu().numpy(), bt.grad.numpy(), 1e-5)
    _close(s2[1].cpu().numpy(), gt.grad.numpy(), 1e-4)
    _close(to_np(dx), xt.grad.numpy(), 1e-4)


@pytest.mark.parametrize("M,K,N,gather", [(1000, 24, 56, False), (77, 432, 192, False), (2, 2048, 400, False),
                                           (5000, 48, 112, False), (0, 24, 48, True)])
def test_pointwise_backward(M, K, N, gather):
    from x3d_tf_b200 import ops
    L, check = _L()
    rng = np.random.default_rng(K + N)
    if gather:
        NT, H, W, s = 6, 9, 11, 2
        Ho, Wo = (H - 1) // s + 1, (W - 1) // s + 1
        x = rng.normal(size=(NT, H, W, K)).astype(np.float32)
        A = x[:, ::s, ::s, :].reshape(-1, K)
        M = A.shape[0]
        geom = (1, Ho, Wo, H, W, s)
    else:
        A = rng.normal(size=(M, K)).astype(np.float32)
        x, geom = A, (0, 0, 0, 0, 0, 1)
    w = rng.normal(size=(K, N)).astype(np.float32) / np.sqrt(K)
    dD = rng.normal(size=(M, N)).astype(np.float32)
    xd, dd, wd = to_dev(x), to_dev(dD), to_dev(w)
    dW = torch.zeros((K, N), dtype=torch.float64, device=dev())
    check(L.x3d_pw_wgrad(xd.data_ptr(), dd.data_ptr(), dW.data_ptr(), M, K, N, K, N, int(gather), geom[1], geom[2],
                         geom[3], geom[4], geom[5], _st()))
    dx = ops.pw_fwd(dd, wd.t().contiguous(), None, M=M, K=N, Nc=K, out_dtype=torch.float32)
    torch.cuda.synchronize()
    _close(dW.cpu().numpy(), A.astype(np.float64).T @ dD.astype(np.float64), 1e-5)
    _close(to_np(dx), dD.astype(np.float64) @ w.astype(np.float64).T, 1e-5)


@pytest.mark.parametrize("N,T,H,W,C,stride", [(2, 4, 8, 8, 56, 1), (1, 3, 9, 13, 24, 2), (1, 4, 16, 16, 56, 2),
                                              (1, 5, 7, 10, 112, 1), (1, 2, 23, 23, 8, 2),
                                              (1, 2, 6, 6, 632, 1)])
def test_channelwise_backward(N, T, H, W, C, stride):
    from oracle import x3d_oracle as O
    L, check = _L()
    rng = np.random.default_rng(H * W + C)
    x = rng.normal(size=(N, T, H, W, C)).astype(np.float32)
    k = rng.normal(size=(3, 3, 3, 1, C)).astype(np.float32) * 0.3
    xt = torch.from_numpy(x).double().permute(0, 4, 1, 2, 3).contiguous().requires_grad_(True)
    kt = torch.from_numpy(k).double().requires_grad_(True)
    yt = O.conv3d_same(xt, kt.permute(4, 3, 0, 1, 2), (1, stride, stride), C)
    Ho, Wo = yt.shape[3], yt.shape[4]
    dy = rng.normal(size=(N, T, Ho, Wo, C)).astype(np.float32)
    yt.backward(torch.from_numpy(dy).double().permute(0, 4, 1, 2, 3))
    ph, pw = O.tf_same_pads(H, 3, stride)[0], O.tf_same_pads(W, 3, stride)[0]
    xd, dyd, kd = to_dev(x), to_dev(dy), to_dev(k.reshape(27, C))
    dx = torch.empty_like(xd)
    check(L.x3d_dw_dgrad(dyd.data_ptr(), kd.data_ptr(), dx.data_ptr(), N, T, H, W, C, stride, ph, pw, _st()))
    dw = torch.zeros((27, C), dtype=torch.float64, device=dev())
    check(L.x3d_dw_wgrad(xd.data_ptr(), dyd.data_ptr(), dw.data_ptr(), N, T, H, W, C, stride, ph, pw, _st()))
    torch.cuda.synchronize()
    _close(to_np(dx), xt.grad.permute(0, 2, 3, 4, 1).numpy(), 1e-5)
    _close(dw.cpu().numpy(), kt.grad.numpy().reshape(27, C), 1e-5)


def test_stem_training_pieces():
    L, check = _L()
    rng = np.random.default_rng(5)
    N, T, H, W, C, kt = 2, 5, 13, 18, 24, 5
    x = rng.normal(size=(N, T, H, W, 3)).astype(np.float32)
    ws = rng.normal(size=(1, 3, 3, 3, C)).astype(np.float32) * 0.3
    wt = rng.normal(size=(kt, 1, 1, 1, C)).astype(np.float32) * 0.5
    xt = torch.from_numpy(x).double().permute(0, 4, 1, 2, 3).contiguous()
    wst = torch.from_numpy(ws).double().requires_grad_(True)
    wtt = torch.from_numpy(wt).double().requires_grad_(True)
    s = F.conv3d(F.pad(xt, (1, 1, 1, 1, 0, 0)), wst.permute(4, 3, 0, 1, 2), None, stride=(1, 2, 2))
    y = F.conv3d(F.pad(s, (0, 0, 0, 0, 2, 2)), wtt.permute(4, 3, 0, 1, 2), None, groups=C)
    Ho, Wo = y.shape[3], y.shape[4]
    dy = rng.normal(size=(N, T, Ho, Wo, C)).astype(np.float32)
    y.backward(torch.from_numpy(dy).double().permute(0, 4, 1, 2, 3))
    xd, wsd, wtd, dyd = to_dev(x), to_dev(ws.reshape(27, C)), to_dev(wt.reshape(kt, C)), to_dev(dy)
    sd = torch.empty((N, T, Ho, Wo, C), device=dev())
    check(L.x3d_stem_convs_fwd(xd.data_ptr(), wsd.data_ptr(), sd.data_ptr(), N, T, H, W, C, _st()))
    yd = torch.empty_like(sd)
    check(L.x3d_tconv_fwd(sd.data_ptr(), wtd.data_ptr(), yd.data_ptr(), N, T, Ho * Wo, C, kt, 0, _st()))
    dwt = torch.zeros((kt, C), dtype=torch.float64, device=dev())
    check(L.x3d_tconv_wgrad(sd.data_ptr(), dyd.data_ptr(), dwt.data_ptr(), N, T, Ho * Wo, C, kt, _st()))
    ds = torch.empty_like(sd)
    check(L.x3d_tconv_fwd(dyd.data_ptr(), wtd.data_ptr(), ds.data_ptr(), N, T, Ho * Wo, C, kt, 1, _st()))
    dws = torch.zeros((27, C), dtype=torch.float64, device=dev())
    check(L.x3d_stem_convs_wgrad(xd.data_ptr(), ds.data_ptr(), dws.data_ptr(), N, T, H, W, C, _st()))
    torch.cuda.synchronize()
    _close(to_np(yd), y.detach().permute(0, 2, 3, 4, 1).numpy(), 1e-5)
    _close(dwt.cpu().numpy(), wtt.grad.numpy().reshape(kt, C), 1e-5)
    _close(dws.cpu().numpy(), wst.grad.numpy().reshape(27, C), 1e-5)


@pytest.mark.parametrize("with_se", [True, False])
def test_scale_swish_fwd_bwd(with_se):
    L, check = _L()
    rng = np.random.default_rng(9)
    N, P, C = 3, 700, 56
    y = rng.normal(size=(N * P, C)).astype(np.float32) * 2
    s = rng.uniform(0.1, 0.9, size=(N, C)).astype(np.float32)
    dout = rng.normal(size=(N * P, C)).astype(np.float32)
    yt = torch.from_numpy(y).double().requires_grad_(True)
    st_ = torch.from_numpy(s).double().requires_grad_(True)
    v = yt.view(N, P, C) * st_[:, None, :] if with_se else yt.view(N, P, C)
    out = (v * torch.sigmoid(v)).reshape(N * P, C)
    out.backward(torch.from_numpy(dout).double())
    yd, sd, dd = to_dev(y), to_dev(s), to_dev(dout)
    o = torch.empty_like(yd)
    check(L.x3d_scale_swish_fwd(yd.data_ptr(), sd.data_ptr() if with_se else None, o.data_ptr(), N * P, C, P, _st()))
    dy = torch.empty_like(yd)
    ds = torch.zeros((N, C), dtype=torch.float64, device=dev()) if with_se else None
    check(L.x3d_scale_swish_bwd(dd.data_ptr(), yd.data_ptr(), sd.data_ptr() if with_se else None, dy.data_ptr(),
                                ds.data_ptr() if with_se else None, N * P, C, P, _st()))
    torch.cuda.synchronize()
    _close(to_np(o), out.detach().numpy(), 1e-5)
    _close(to_np(dy), yt.grad.numpy(), 1e-5)
    if with_se:
        _close(ds.cpu().numpy(), st_.grad.numpy(), 1e-5)


def test_softmax_xent_and_sgd():
    L, check = _L()
    rng = np.random.default_rng(11)
    N, ncls = 5, 400
    logits = rng.normal(size=(N, ncls)).astype(np.float32) * 3
    labels = rng.integers(0, ncls, size=N).astype(np.int32)
    lt = torch.from_numpy(logits).double().requires_grad_(True)
    p = torch.softmax(lt, -1).gather(1, torch.from_numpy(labels).long()[:, None])[:, 0].clamp(1e-7, 1 - 1e-7)
    loss_t = -torch.log(p)
    (loss_t.sum() / (N * 2)).backward()
    ld, yd = to_dev(logits), torch.from_numpy(labels).to(dev())
    loss, dl = torch.empty(N, device=dev()), torch.empty((N, ncls), device=dev())
    check(L.x3d_softmax_xent(ld.data_ptr(), yd.data_ptr(), loss.data_ptr(), dl.data_ptr(), N, ncls, 1.0 / (N * 2), _st()))
    torch.cuda.synchronize()
    _close(to_np(loss), loss_t.detach().numpy(), 1e-5)
    _close(to_np(dl), lt.grad.numpy(), 1e-5)
    n = 1003
    w, g, v = (rng.normal(size=n).astype(np.float32) for _ in range(3))
    wd = np.where(rng.random(n) < 0.5, 1e-4, 0.0).astype(np.float32)
    wd_, gd, vd, wdd = to_dev(w), to_dev(g), to_dev(v), to_dev(wd)
    check(L.x3d_sgd_nesterov_step(wd_.data_ptr(), gd.data_ptr(), vd.data_ptr(), wdd.data_ptr(), n, 0.05, 0.9, _st()))
    torch.cuda.synchronize()
    gg = g.astype(np.float64) + wd * w
    v1 = 0.9 * v - 0.05 * gg
    _close(to_np(vd), v1, 1e-6)
    _close(to_np(wd_), w + 0.9 * v1 - 0.05 * gg, 1e-6)


@pytest.mark.parametrize("M,K,N,relu,use_bias", [(1000, 24, 56, True, True), (4096, 56, 24, False, True),
                                                 (300, 432, 192, False, False), (129, 192, 432, True, True),
                                                 (64, 432, 2048, True, False), (32, 2048, 400, False, True),
                                                 (5000, 48, 216, True, True), (12345, 216, 96, False, True),
                                                 (3000, 280, 632, True, True), (2000, 632, 280, False, True),
                                                 (4000, 136, 312, False, False)])
def test_pointwise_tf32x3_tcgen05(M, K, N, relu, use_bias):
    """x3d_pw_tf32_fwd (tcgen05.mma kind::tf32, 3xTF32 split) against float64: fp32-level accuracy
    (2e-5 of the output's scale, the bound of the fp32 kernels) in both orientations -- forward
    a . w and backward-data dy . w^T with the kernel read as stored."""
    from x3d_tf_b200 import ops
    rng = np.random.default_rng(M + K + N)
    a = rng.normal(size=(M, K)).astype(np.float32)
    w = (rng.normal(size=(K, N)) / np.sqrt(K)).astype(np.float32)
    b = rng.normal(size=N).astype(np.float32) if use_bias else None
    want = a.astype(np.float64) @ w.astype(np.float64) + (b if use_bias else 0.0)
    if relu:
        want = np.maximum(want, 0.0)
    got = ops.pw_tf32(torch.from_numpy(a).cuda(), torch.from_numpy(w).cuda(),
                      torch.from_numpy(b).cuda() if use_bias else None, relu=relu, transpose_w=True)
    torch.cuda.synchronize()
    scale = np.abs(want).max()
    err = np.abs(got.cpu().numpy() - want).max() / scale
    assert got.shape == (M, N) and err < 2e-5, err
    # a single-pass TF32 product would be ~1e-3: make sure the split is really in effect (the tensor
    # core's fp32 accumulation truncates, so the error grows with the reduction length)
    assert err < (5e-6 if K <= 512 else 2e-5), err
    dy = rng.normal(size=(M, N)).astype(np.float32)
    want_dx = dy.astype(np.float64) @ w.astype(np.float64).T
    dx = ops.pw_tf32(torch.from_numpy(dy).cuda(), torch.from_numpy(w).cuda(), None, transpose_w=False)
    torch.cuda.synchronize()
    assert dx.shape == (M, K)
    assert np.abs(dx.cpu().numpy() - want_dx).max() / np.abs(want_dx).max() < (5e-6 if N <= 512 else 2e-5)
