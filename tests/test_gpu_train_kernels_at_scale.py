"""Each training-step kernel against float64 at the sizes the training step runs: X3D-M at batch 32,
16x224^2 (the benchmarked step) and X3D-XL at batch 16, 16x312^2.

The per-kernel tests in test_gpu_train_ops.py / test_gpu_mixed_training.py use small shapes, where
every persistent CTA of the tcgen05 GEMMs does one tile, every backward-filter block keeps 256 rows
and no grid-stride loop wraps.  The kernels choose their launch geometry (and often the kernel) from
the sizes they are given, so here:
- every case asserts, through the profiler, the kernel it meant to run (`_run`), so that a change to
  the dispatch cannot move a case onto another path unnoticed;
- every reference is float64 on the device (the CPU oracle is far too slow at these sizes);
- every tolerance is the bound the small-size tests already hold the kernel to, and each case also
  asserts that the tolerance is smaller than what the reference changes by when the last tile / row
  block of the input is dropped (`_sharp`): a tail that is lost or counted twice cannot pass;
- `test_training_step_launches_only_pinned_kernels` profiles whole steps and requires every kernel
  they launch to be pinned by a case of this file (`PINNED`).
"""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

EPS = 1e-5


# ---------------------------------------------------------------- helpers
def _L():
    from x3d_tf_b200._lib import check, lib
    return lib(), check


def _st():
    return torch.cuda.current_stream().cuda_stream


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _randn(shape, g, dtype=torch.float32):
    return torch.randn(shape, device="cuda", generator=g, dtype=dtype)


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _launched(fn):
    """Names (demangled) of the kernels `fn` launched."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type == DeviceType.CUDA
            and not e.name.startswith(("Memcpy", "Memset"))}


def _run(fn, *kernels):
    """Runs `fn` once, asserts that it launched every kernel named (by substring) and returns its result."""
    out = []
    names = _launched(lambda: out.append(fn()))
    for k in kernels:
        assert any(k in n for n in names), (k, sorted(names))
    return out[0]


def _rel(got, want):
    got, want = torch.as_tensor(got).detach().double(), torch.as_tensor(want).detach().double()
    return float((got - want).abs().max() / max(float(want.abs().max()), 1e-30))


def _sharp(tol, delta, what=""):
    """The tolerance must resolve the change a dropped tail makes (delta, in the same relative units)."""
    assert delta > tol, f"{what}: tolerance {tol:.2e} does not see a dropped tail ({delta:.2e})"


def _bound(K):
    # test_gpu_mixed_training._bound: the tf32 kernels' bound against float64 (DESIGN section 9) for
    # K <= 512, scaled by K / 512 above
    return 5e-6 * max(1.0, K / 512)


def _r64(t):
    return t.to(torch.bfloat16).double()



# Training shapes: X3D-M at batch 32 (the benchmark), X3D-XL at batch 16, both 16 frames.
BENCH_M = 32 * 16 * 112 * 112          # rows of the first block's expand conv (input of stage 1 at 112^2)
M_STAGE4 = 32 * 16 * 7 * 7             # X3D-M last stage: (192, 432)
XL_M10 = 16 * 16 * 10 * 10             # X3D-XL last stage: (280, 632), (632, 280)
XL_M20 = 16 * 16 * 20 * 20             # X3D-XL stage 3: (136, 312)


def _odd_m():
    """M mod 128 != 0 with every persistent CTA walking at least four tiles."""
    return 4 * _sms() * 128 + 77


# ---------------------------------------------------------------- tcgen05 GEMMs
GEMM_SHAPES = [("bench", 24, 56, BENCH_M), ("bench", 56, 24, BENCH_M), ("stage4", 192, 432, M_STAGE4),
               ("xl", 280, 632, XL_M10), ("xl", 632, 280, XL_M10), ("xl", 136, 312, XL_M20), ("odd", 56, 24, None)]


def _gemm_inputs(K, N, M, seed):
    g = _gen(seed)
    a = _randn((M, K), g)
    # the last tile's rows are 4x larger: a lost (or doubled) tail tile moves the statistics by
    # 16 * rows / M of their size, above the bound even at 6.4 M rows
    tail = M % 128 or 128
    a[-tail:] *= 4
    w = _randn((K, N), g) / K ** 0.5
    return a, w, tail


def _check_rows(got, want, tail, tol, what):
    # bulk and tail rows separately: each against its own scale
    assert _rel(got[:-tail], want[:-tail]) < tol, (what, "bulk", _rel(got[:-tail], want[:-tail]))
    assert _rel(got[-tail:], want[-tail:]) < tol, (what, "tail", _rel(got[-tail:], want[-tail:]))
    _sharp(tol, float(want[-tail:].abs().max() / want.abs().max()), what)


def _check_stats(st, ref, tail, tol):
    s1, s2 = ref.sum(0), (ref * ref).sum(0)
    assert _rel(st[0], s1) < tol and _rel(st[1], s2) < tol, (_rel(st[0], s1), _rel(st[1], s2))
    t = ref[-tail:]
    _sharp(tol, _rel(s1 - t.sum(0), s1), "column sums")
    _sharp(tol, _rel(s2 - (t * t).sum(0), s2), "column sums of squares")


def _persist(M, persistent):
    if persistent:
        assert math.ceil(M / 128) >= 4 * _sms(), M


@pytest.mark.parametrize("where,K,N,M", GEMM_SHAPES)
def test_pw_tf32_at_training_sizes(where, K, N, M):
    """ops.pw_tf32 (3xTF32 on tcgen05): forward with the BN statistics epilogue, forward with bias + ReLU,
    backward-data; 5e-6 of the output's scale for K <= 512, 2e-5 above (test_pointwise_tf32x3_tcgen05),
    the statistics to _bound(K) * 4 (the bf16 test's bound for the same epilogue)."""
    from x3d_tf_b200 import ops
    M = M or _odd_m()
    _persist(M, where in ("bench", "odd"))
    a, w, tail = _gemm_inputs(K, N, M, K * 7 + N)
    ref = a.double() @ w.double()
    tol, tol_dx = (5e-6 if K <= 512 else 2e-5), (5e-6 if N <= 512 else 2e-5)
    st = torch.zeros(2, N, dtype=torch.float64, device="cuda")
    y = _run(lambda: ops.pw_tf32(a, w, stats=st), "pw_tf32_tc_kernel", "tf32_split_kernel")
    _check_rows(y, ref, tail, tol, "forward")
    del y
    _check_stats(st, ref, tail, _bound(K) * 4)
    bias = _randn((N,), _gen(N))
    yb = _run(lambda: ops.pw_tf32(a, w, bias, relu=True), "pw_tf32_tc_kernel")
    _check_rows(yb, torch.relu(ref + bias.double()), tail, tol, "bias + relu")
    del yb, ref
    dy = _randn((M, N), _gen(M + 1))
    dy[-tail:] *= 4
    dx = _run(lambda: ops.pw_tf32(dy, w, None, transpose_w=False), "pw_tf32_tc_kernel")
    _check_rows(dx, dy.double() @ w.double().t(), tail, tol_dx, "backward-data")


@pytest.mark.parametrize("where,K,N,M", GEMM_SHAPES)
def test_pw_bf16_train_at_training_sizes(where, K, N, M):
    """ops.pw_bf16_train / ops.pw_wgrad_bf16 against float64 products of the same bf16-rounded operands,
    with the bounds of test_gpu_mixed_training (_bound; the statistics _bound(K) * 4).  The backward-filter
    is held to 1e-5, the 3xTF32 backward-filter's bound (test_pointwise_backward): bf16 x bf16 products
    are exact in fp32, so, as there, only the fp32 accumulation over a block's rows remains."""
    from x3d_tf_b200 import ops
    M = M or _odd_m()
    _persist(M, where in ("bench", "odd"))
    a, w, tail = _gemm_inputs(K, N, M, K * 11 + N)
    ref = _r64(a) @ _r64(w)
    st = torch.zeros(2, N, dtype=torch.float64, device="cuda")
    wf = ops.bf16_round(w, transpose_w=True)
    y = _run(lambda: ops.pw_bf16_train(a, wf, K, stats=st), "pw_bf16_train_tc_kernel")
    _check_rows(y, ref, tail, _bound(K), "forward")
    del y
    _check_stats(st, ref, tail, _bound(K) * 4)
    bias = _randn((N,), _gen(N))
    yb = _run(lambda: ops.pw_bf16_train(a, wf, K, bias, relu=True), "pw_bf16_train_tc_kernel")
    _check_rows(yb, torch.relu(ref + bias.double()), tail, _bound(K), "bias + relu")
    del yb, ref
    dy = _randn((M, N), _gen(M + 1))
    dy[-tail:] *= 4
    wb = _run(lambda: ops.bf16_round(w, transpose_w=False), "bf16_round_kernel")
    dx = _run(lambda: ops.pw_bf16_train(dy, wb, N), "pw_bf16_train_tc_kernel")
    _check_rows(dx, _r64(dy) @ _r64(w).t(), tail, _bound(N), "backward-data")
    del dx
    dw = torch.zeros(K, N, dtype=torch.float64, device="cuda")
    _run(lambda: ops.pw_wgrad_bf16(a, dy, dw), "pw_wgrad_bf16_kernel")
    want = _r64(a).t() @ _r64(dy)
    assert _rel(dw, want) < 1e-5, _rel(dw, want)
    lo = M - (M % _wgrad_rpb(M, K, N) or _wgrad_rpb(M, K, N))
    _sharp(1e-5, _rel(_r64(a[lo:]).t() @ _r64(dy[lo:]), want), "last row block")


# ---------------------------------------------------------------- pointwise backward-filter
def _wgrad_rpb(M, K, N):
    """Rows per block of x3d_pw_wgrad / x3d_pw_wgrad_bf16 (pw_wgrad_grid in csrc/x3d_train.cu)."""
    TK, TN = (64 if K > 32 else 32), (64 if N > 32 else 32)
    tiles = -(-K // TK) * -(-N // TN)
    zb = -(-148 * 8 // tiles)
    rpb = max(-(-M // zb), 256)
    rpb = -(-rpb // 32) * 32
    if -(-M // rpb) > 65535:
        rpb = -(-(-(-M // 65535)) // 32) * 32
    return rpb


def _pw_wgrad(a, dy, M, K, N, gather=None):
    L, check = _L()
    dw = torch.zeros(K, N, dtype=torch.float64, device="cuda")
    g = gather or (0, 0, 0, 0, 0, 1)
    check(L.x3d_pw_wgrad(a.data_ptr(), dy.data_ptr(), dw.data_ptr(), M, K, N, a.shape[-1], N, int(gather is not None),
                         g[1], g[2], g[3], g[4], g[5], _st()), "x3d_pw_wgrad")
    return dw


@pytest.mark.parametrize("K,N,tile", [(24, 24, "32, 32"), (24, 56, "32, 64"), (56, 24, "64, 32"), (56, 112, "64, 64")])
def test_pw_wgrad_tf32x3_every_tile_at_bench_m(K, N, tile):
    """x3d_pw_wgrad (3xTF32 mma.sync path) for every tile template at the bench M, where each block sums
    thousands of rows in fp32 (not the 256-row floor of the small tests); 1e-5 as test_pointwise_backward."""
    M = BENCH_M
    rpb = _wgrad_rpb(M, K, N)
    assert rpb > 256, rpb
    g = _gen(K * N)
    a, dy = _randn((M, K), g), _randn((M, N), g)
    dw = _run(lambda: _pw_wgrad(a, dy, M, K, N), f"pw_wgrad_tf32x3_kernel<{tile}>")
    want = a.double().t() @ dy.double()
    assert _rel(dw, want) < 1e-5, _rel(dw, want)
    lo = (M - 1) // rpb * rpb
    _sharp(1e-5, _rel(a[lo:].double().t() @ dy[lo:].double(), want), "last row block")


def test_strided_shortcut_gemms_at_stage2_geometry():
    """The gathered stride-2 shortcut from stage 1 (56^2, 24 channels) into stage 2 (28^2, 48 channels) at
    batch 32: forward (x3d_pw_fwd's 3xTF32 SIMT kernel in fp32; x3d_gather_rows_fwd + the bf16 GEMM when
    mixed) and backward-filter (x3d_pw_wgrad / x3d_pw_wgrad_bf16 with the gather)."""
    from x3d_tf_b200 import ops
    N, T, H, W, C, Co, s = 32, 16, 56, 56, 24, 48, 2
    Ho, Wo = (H - 1) // s + 1, (W - 1) // s + 1
    g = _gen(5)
    x5 = _randn((N, T, H, W, C), g)
    w = _randn((C, Co), g) / C ** 0.5
    rows = x5[:, :, ::s, ::s].reshape(-1, C)
    M = rows.shape[0]
    dy = _randn((M, Co), g)
    gth = (T, Ho, Wo, H, W, s)
    y = _run(lambda: ops.pw_fwd(x5.view(-1, C), w, None, M=M, K=C, Nc=Co, out_dtype=torch.float32, gather=gth),
             "pw_gemm_tf32x3_kernel")
    want = rows.double() @ w.double()
    assert _rel(y, want) < 2e-5, _rel(y, want)
    _sharp(2e-5, float(want[-1].abs().max() / want.abs().max()), "last row")
    gr = _run(lambda: ops.gather_rows_fwd(x5, s), "gather_rows_kernel")
    assert torch.equal(gr, rows)
    yb = ops.pw_bf16_train(gr, ops.bf16_round(w), C)
    assert _rel(yb, _r64(rows) @ _r64(w)) < _bound(C)
    rpb = _wgrad_rpb(M, C, Co)
    lo = (M - 1) // rpb * rpb
    dw = _run(lambda: _pw_wgrad(x5.view(-1, C), dy, M, C, Co, gather=gth), "pw_wgrad_tf32x3_kernel<32, 64>")
    want = rows.double().t() @ dy.double()
    assert _rel(dw, want) < 1e-5, _rel(dw, want)
    _sharp(1e-5, _rel(rows[lo:].double().t() @ dy[lo:].double(), want), "last row block")
    dwb = torch.zeros(C, Co, dtype=torch.float64, device="cuda")
    _run(lambda: ops.pw_wgrad_bf16(x5.view(-1, C), dy, dwb, M=M, gather=gth), "pw_wgrad_bf16_kernel<32, 64>")
    want = _r64(rows).t() @ _r64(dy)
    assert _rel(dwb, want) < 1e-5, _rel(dwb, want)
    _sharp(1e-5, _rel(_r64(rows[lo:]).t() @ _r64(dy[lo:]), want), "last row block")


# ---------------------------------------------------------------- channelwise 3x3x3 (SAME) backward
def _dw_ref(x, w, s, ph, pw):
    """Channelwise 3x3x3 SAME conv, stride (1, s, s): the sum of 27 shifted zero-padded slices (float64)."""
    N, T, H, W, C = x.shape
    Ho, Wo = -(-H // s), -(-W // s)
    xp = F.pad(x, (0, 0, pw, max(0, s * (Wo - 1) + 3 - W - pw), ph, max(0, s * (Ho - 1) + 3 - H - ph), 1, 1))
    y = 0
    for dt in range(3):
        for dh in range(3):
            for dw in range(3):
                y = y + xp[:, dt:dt + T, dh:dh + s * (Ho - 1) + 1:s, dw:dw + s * (Wo - 1) + 1:s, :] * w[(dt * 3 + dh) * 3 + dw]
    return y


def _dw_grads(x, w, dy, s, ph, pw):
    """(dx, dw) of _dw_ref by float64 autograd on the device."""
    x64 = x.double().requires_grad_(True)
    w64 = w.double().requires_grad_(True)
    _dw_ref(x64, w64, s, ph, pw).backward(dy.double())
    return x64.grad, w64.grad


def _last_row(dy):
    """dy restricted to its last output row (the grads of a lost last row block contain this one's)."""
    t = torch.zeros_like(dy)
    t[-1, -1, -1] = dy[-1, -1, -1]
    return t


def _pads(H, W, s):
    from x3d_tf_b200.arch import same_pad
    return same_pad(H, 3, s)[1], same_pad(W, 3, s)[1]


@pytest.mark.parametrize("N,T,H,W,C,s,kernel", [
    (32, 16, 56, 56, 56, 1, "dw_wgrad_pair_kernel"),        # X3D-M stage 1, batch 32
    (16, 16, 10, 10, 632, 1, "dw_wgrad_kernel<1, 4>"),      # X3D-XL last stage, batch 16
    (32, 16, 56, 56, 112, 2, "dw_wgrad_slide_kernel"),      # X3D-M first block of stage 2 (even)
    (16, 16, 39, 39, 312, 2, "dw_wgrad_slide_kernel"),      # X3D-XL first block of stage 3 (odd)
])
def test_dw_wgrad_paths(N, T, H, W, C, s, kernel):
    """x3d_dw_wgrad on each of its three paths against float64 autograd; 1e-5 as test_channelwise_backward."""
    L, check = _L()
    ph, pw = _pads(H, W, s)
    g = _gen(H * C + s)
    x = _randn((N, T, H, W, C), g)
    w = _randn((27, C), g) * 0.3
    Ho, Wo = -(-H // s), -(-W // s)
    dy = _randn((N, T, Ho, Wo, C), g)
    dw = torch.zeros(27, C, dtype=torch.float64, device="cuda")
    _run(lambda: check(L.x3d_dw_wgrad(x.data_ptr(), dy.data_ptr(), dw.data_ptr(), N, T, H, W, C, s, ph, pw, _st()),
                       "x3d_dw_wgrad"), kernel)
    _, want = _dw_grads(x, w, dy, s, ph, pw)
    assert _rel(dw, want) < 1e-5, _rel(dw, want)
    _, tail = _dw_grads(x, w, _last_row(dy), s, ph, pw)
    _sharp(1e-5, _rel(tail, want), "last output row")


@pytest.mark.parametrize("N,T,H,W,C,s", [
    (32, 16, 56, 56, 56, 1), (32, 16, 112, 112, 56, 2),     # X3D-M stage 1 at batch 32
    (16, 16, 10, 10, 632, 1), (16, 16, 20, 20, 632, 2),     # X3D-XL last stage at batch 16
    (8, 16, 39, 39, 56, 1), (8, 16, 39, 39, 56, 2),         # odd H / W
    (2, 16, 39, 39, 632, 1), (2, 16, 39, 39, 632, 2),
])
def test_channelwise_dgrad_of_the_training_step(N, T, H, W, C, s):
    """The backward-data the training step runs (training.channelwise_dgrad: the forward kernel with the
    taps reversed, after the x3d_strided_add zero-dilation for stride 2) against float64 autograd; 1e-5
    as x3d_dw_dgrad in test_channelwise_backward."""
    from x3d_tf_b200.training import channelwise_dgrad
    ph, pw = _pads(H, W, s)
    g = _gen(H * C + s + 1)
    x = _randn((N, T, H, W, C), g)
    w = _randn((27, C), g) * 0.3
    Ho, Wo = -(-H // s), -(-W // s)
    dy = _randn((N, T, Ho, Wo, C), g)
    zero = torch.zeros(C, device="cuda")
    kernels = ("dw_tma_kernel",) + (("strided_add_kernel",) if s == 2 else ())
    dx = _run(lambda: channelwise_dgrad(dy, w, zero, H, W, s, ph, pw), *kernels)
    want, _ = _dw_grads(x, w, dy, s, ph, pw)
    assert dx.shape == want.shape
    assert _rel(dx, want) < 1e-5, _rel(dx, want)
    tail, _ = _dw_grads(x, w, _last_row(dy), s, ph, pw)
    _sharp(1e-5, _rel(tail, want), "last output row")


# ---------------------------------------------------------------- column reductions and BatchNorm
def _vec_rows_per_pass(M, C):
    """Rows one grid-stride pass of colreduce_vec_kernel covers (bn_grid(M, C, 4) in csrc/x3d_train.cu)."""
    C4 = C // 4
    threads = min(148 * 4 * 256, M * C4)
    threads = -(-threads // C4) * C4
    blocks = -(-threads // 256)
    return blocks * 256 // C4 * C4 // C4


def _colreduce(a, M, C, seg, out, mode, x=None, mean=None, rstd=None, relu_out=None):
    L, check = _L()
    p = lambda t: None if t is None else t.data_ptr()
    check(L.x3d_colreduce(a.data_ptr(), p(x), p(mean), p(rstd), p(relu_out), M, C, seg, out.data_ptr(), mode, _st()),
          "x3d_colreduce")


def _bn_data(M, C, seed):
    """Per-channel scale 0.2..3 and offset; every fourth channel has a mean of 20x its standard deviation."""
    g = _gen(seed)
    sd = torch.rand(C, device="cuda", generator=g) * 2.8 + 0.2
    mu = torch.randn(C, device="cuda", generator=g)
    mu[::4] = 20 * sd[::4]
    return _randn((M, C), g) * sd + mu


@pytest.mark.parametrize("M,C,relu", [(BENCH_M, 56, False), (BENCH_M, 56, True), (400_003, 632, True)])
def test_batchnorm_chain_at_scale(M, C, relu):
    """x3d_colreduce modes 0 and 1 (vec path), x3d_bn_finalize, x3d_bn_apply_fwd and x3d_bn_bwd_apply at
    the bench M (C = 56) and at 632 channels (400 k rows: the bench M at 632 channels is 16 GB a tensor),
    with the bounds of test_batchnorm_train_fwd_bwd.  The ReLU branch is the device's (as in the whole-step
    tests): at 360 M elements hundreds sit within rounding of zero."""
    L, check = _L()
    x = _bn_data(M, C, M + C)
    g = _gen(C)
    gamma = torch.rand(C, device="cuda", generator=g) + 0.5
    beta = torch.randn(C, device="cuda", generator=g) * 0.3
    dy = _randn((M, C), g)
    sums = torch.zeros(2, C, dtype=torch.float64, device="cuda")
    _run(lambda: _colreduce(x, M, C, M, sums, 0), "colreduce_vec_kernel")
    m_, v_, r_ = (torch.empty(C, device="cuda") for _ in range(3))
    mm, mv = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda")
    _run(lambda: check(L.x3d_bn_finalize(sums.data_ptr(), M, C, EPS, 0.9, m_.data_ptr(), v_.data_ptr(), r_.data_ptr(),
                                         mm.data_ptr(), mv.data_ptr(), _st())), "bn_finalize_kernel")
    y = torch.empty_like(x)
    _run(lambda: check(L.x3d_bn_apply_fwd(x.data_ptr(), m_.data_ptr(), r_.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                                          y.data_ptr(), M, C, int(relu), _st())), "bn_apply_kernel")
    x64 = x.double()
    mean, var = x64.mean(0), x64.var(0, unbiased=False)
    # statistics the kernel would report if it lost the rows of its last grid-stride pass
    rows = _vec_rows_per_pass(M, C)
    xt = x64[:-rows]
    mean_d = xt.sum(0) / M
    var_d = (xt * xt).sum(0) / M - mean_d * mean_d
    assert _rel(m_, mean) < 2e-5 and _rel(v_, var) < 2e-5, (_rel(m_, mean), _rel(v_, var))
    _sharp(2e-5, min(_rel(mean_d, mean), _rel(var_d, var)), "last grid-stride pass")
    # The variance is E[x^2] - mean^2 in fp64 from fp32 partial sums (a thread's run of M / rows rows).
    # Where the mean is 20 standard deviations, E[x^2] is 401 variances, so E[x^2]'s relative error is
    # amplified 401x.  A run's sum carries ~sqrt(run) * 2^-24 of relative rounding (~1e-6 at 600 rows);
    # averaged over the ~10^4 runs of a channel it is ~1e-8, i.e. 4e-6 of the variance.  1e-4 leaves
    # 25x for correlated rounding; it is still 100x below the change of dropping the last pass.
    off = torch.arange(0, C, 4, device="cuda")
    e_var = float(((v_.double() - var).abs() / var)[off].max())
    assert e_var < 1e-4, e_var
    _sharp(1e-4, float(((var_d - var).abs() / var)[off].min()), "variance, last pass")
    assert _rel(mm, 0.1 * mean) < 2e-5 and _rel(mv, 0.9 + 0.1 * var) < 2e-5
    rstd = torch.rsqrt(var + EPS)
    xhat = (x64 - mean) * rstd
    del x64, xt
    y_ref = xhat * gamma.double() + beta.double()
    if relu:
        y_ref = torch.relu(y_ref)
    assert _rel(y, y_ref) < 2e-5, _rel(y, y_ref)
    del y_ref
    s2 = torch.zeros(2, C, dtype=torch.float64, device="cuda")
    _run(lambda: _colreduce(dy, M, C, M, s2, 1, x, m_, r_, y if relu else None), "colreduce_vec_kernel")
    dx = torch.empty_like(x)
    _run(lambda: check(L.x3d_bn_bwd_apply(dy.data_ptr(), x.data_ptr(), y.data_ptr() if relu else None, m_.data_ptr(),
                                          r_.data_ptr(), gamma.data_ptr(), s2.data_ptr(), dx.data_ptr(), M, C, _st())),
         "bn_bwd_apply_kernel")
    gd = dy.double() * (y > 0) if relu else dy.double()
    sg, sgx = gd.sum(0), (gd * xhat).sum(0)
    assert _rel(s2[0], sg) < 1e-5 and _rel(s2[1], sgx) < 1e-4, (_rel(s2[0], sg), _rel(s2[1], sgx))
    _sharp(1e-5, _rel(gd[-rows:].sum(0), sg), "BN backward sums, last pass")
    _sharp(1e-4, _rel((gd[-rows:] * xhat[-rows:]).sum(0), sgx), "BN backward sums, last pass")
    dx_ref = gamma.double() * rstd * (gd - sg / M - xhat * (sgx / M))
    assert _rel(dx, dx_ref) < 1e-4, _rel(dx, dx_ref)


@pytest.mark.parametrize("M,C,seg,kernel", [(BENCH_M, 56, BENCH_M, "colreduce_vec_kernel"),
                                            (400_003, 632, 400_003, "colreduce_vec_kernel"),
                                            (32 * 50176, 56, 50176, "colreduce_kernel")])
def test_colreduce_sums(M, C, seg, kernel):
    """Mode 2 (bias gradients) on the vec path, and the segmented generic path exactly as the SE squeeze
    calls it (32 clips x 50,176 rows of X3D-M's stage 1): 1e-5 of the scale."""
    a = _bn_data(M, C, C + 3)
    out = torch.zeros(M // seg, 2, C, dtype=torch.float64, device="cuda")
    _run(lambda: _colreduce(a, M, C, seg, out, 2), kernel)
    a64 = a.double().view(M // seg, seg, C)
    want = a64.sum(1)
    assert _rel(out[:, 0], want) < 1e-5, _rel(out[:, 0], want)
    assert not out[:, 1].any()
    drop = 256 if kernel == "colreduce_kernel" else _vec_rows_per_pass(M, C)   # the last row block of a segment
    _sharp(1e-5, _rel(a64[:, -drop:].sum(1), want), "last row block")


@pytest.mark.parametrize("C,clips", [(56, 32), (632, 4)])
@pytest.mark.parametrize("with_se", [True, False])
def test_scale_swish_at_scale(C, clips, with_se):
    """x3d_scale_swish_fwd / _bwd (vec path, blocks of 256 / (C/4) * (C/4) threads) at 50,176 rows per clip;
    1e-5 as test_scale_swish_fwd_bwd."""
    L, check = _L()
    P = 50176
    M = clips * P
    g = _gen(C + with_se)
    y = _randn((M, C), g) * 2
    s = torch.rand(clips, C, device="cuda", generator=g) * 0.8 + 0.1
    dout = _randn((M, C), g)
    sp = s.data_ptr() if with_se else None
    o = torch.empty_like(y)
    _run(lambda: check(L.x3d_scale_swish_fwd(y.data_ptr(), sp, o.data_ptr(), M, C, P, _st())), "scale_swish_fwd_kernel")
    dy = torch.empty_like(y)
    ds = torch.zeros(clips, C, dtype=torch.float64, device="cuda") if with_se else None
    _run(lambda: check(L.x3d_scale_swish_bwd(dout.data_ptr(), y.data_ptr(), sp, dy.data_ptr(),
                                             ds.data_ptr() if with_se else None, M, C, P, _st())),
         "scale_swish_bwd_vec_kernel")
    y64 = y.double().view(clips, P, C).requires_grad_(True)
    s64 = s.double().requires_grad_(True)
    v = y64 * s64[:, None, :] if with_se else y64
    out = v * torch.sigmoid(v)
    out.backward(dout.double().view(clips, P, C))
    assert _rel(o, out.detach().view(M, C)) < 1e-5
    assert _rel(dy, y64.grad.view(M, C)) < 1e-5
    _sharp(1e-5, float(out.detach()[-1, -1].abs().max() / out.detach().abs().max()), "last row")
    if with_se:
        assert _rel(ds, s64.grad) < 1e-5, _rel(ds, s64.grad)
        dv = (y64.grad / s64.detach()[:, None, :])[:, -256:]          # the last row block of each clip
        _sharp(1e-5, _rel((dv * y64.detach()[:, -256:]).sum(1), s64.grad), "last row block")


# ---------------------------------------------------------------- stem
@pytest.mark.parametrize("N,T,H,W,C", [(32, 16, 224, 224, 24), (16, 16, 312, 312, 32)])
def test_stem_pieces_at_scale(N, T, H, W, C):
    """x3d_stem_convs_fwd / _wgrad and x3d_tconv_fwd (flip 0 and 1) / _wgrad at X3D-M's batch-32 and
    X3D-XL's batch-16 stem, where the capped grids of the backward-filters grid-stride several times;
    1e-5 as test_stem_training_pieces."""
    L, check = _L()
    kt = 5
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    P = Ho * Wo
    opix = N * T * P
    assert opix > 148 * 16 * (256 // (C // 4)) and N * P * (C // 4) > 148 * 8 * (256 // (C // 4)) * (C // 4)
    g = _gen(C)
    x = _randn((N, T, H, W, 3), g)
    ws = _randn((27, C), g) * 0.3
    wt = _randn((kt, C), g) * 0.5
    dy = _randn((N, T, Ho, Wo, C), g)
    sd = torch.empty((N, T, Ho, Wo, C), device="cuda")
    _run(lambda: check(L.x3d_stem_convs_fwd(x.data_ptr(), ws.data_ptr(), sd.data_ptr(), N, T, H, W, C, _st())),
         "stem_convs_fwd_kernel")
    yd = torch.empty_like(sd)
    _run(lambda: check(L.x3d_tconv_fwd(sd.data_ptr(), wt.data_ptr(), yd.data_ptr(), N, T, P, C, kt, 0, _st())),
         "tconv_fwd_kernel")
    dwt = torch.zeros(kt, C, dtype=torch.float64, device="cuda")
    _run(lambda: check(L.x3d_tconv_wgrad(sd.data_ptr(), dy.data_ptr(), dwt.data_ptr(), N, T, P, C, kt, _st())),
         "tconv_wgrad_vec_kernel")
    ds = torch.empty_like(sd)
    _run(lambda: check(L.x3d_tconv_fwd(dy.data_ptr(), wt.data_ptr(), ds.data_ptr(), N, T, P, C, kt, 1, _st())),
         "tconv_fwd_kernel")
    dws = torch.zeros(27, C, dtype=torch.float64, device="cuda")
    _run(lambda: check(L.x3d_stem_convs_wgrad(x.data_ptr(), ds.data_ptr(), dws.data_ptr(), N, T, H, W, C, _st())),
         "stem_convs_wgrad_vec_kernel")
    # float64 reference: 3x3 taps at stride 2 (pad 1 before) as nine [rows, 3] x [3, C] products, then the
    # temporal conv as five shifted products; gradients by autograd
    xp = F.pad(x.double(), (0, 0, 1, max(0, 2 * (Wo - 1) + 2 - W), 1, max(0, 2 * (Ho - 1) + 2 - H)))
    ws64, wt64 = ws.double().requires_grad_(True), wt.double().requires_grad_(True)
    s64 = 0
    for dh in range(3):
        for dw in range(3):
            k = (dh * 3 + dw) * 3
            s64 = s64 + xp[:, :, dh:dh + 2 * (Ho - 1) + 1:2, dw:dw + 2 * (Wo - 1) + 1:2, :] @ ws64[k:k + 3]
    s64.retain_grad()
    sp = F.pad(s64, (0, 0, 0, 0, 0, 0, 2, 2))
    y64 = sum(sp[:, j:j + T] * wt64[j] for j in range(kt))
    y64.backward(dy.double())
    assert _rel(sd, s64) < 1e-5 and _rel(yd, y64) < 1e-5, (_rel(sd, s64), _rel(yd, y64))
    assert _rel(ds, s64.grad) < 1e-5, _rel(ds, s64.grad)
    assert _rel(dwt, wt64.grad) < 1e-5 and _rel(dws, ws64.grad) < 1e-5, (_rel(dwt, wt64.grad), _rel(dws, ws64.grad))
    # what the last clip's last output frame adds to the filter gradients (a lost tail of the grid-stride walk)
    s_last, ds_last = s64.detach()[-1:], s64.grad[-1:, -1:]
    xl = xp[-1:, -1:]
    dws_tail = torch.stack([xl[:, :, dh:dh + 2 * (Ho - 1) + 1:2, dw:dw + 2 * (Wo - 1) + 1:2, ci].reshape(-1)
                            for dh in range(3) for dw in range(3) for ci in range(3)]) @ ds_last.reshape(-1, C)
    _sharp(1e-5, _rel(dws_tail, ws64.grad), "stem filter gradient, last frame")
    dwt_tail = torch.stack([(F.pad(s_last, (0, 0, 0, 0, 0, 0, 2, 2))[:, T - 1 + j] * dy.double()[-1:, -1]).sum((0, 1, 2))
                            for j in range(kt)])
    _sharp(1e-5, _rel(dwt_tail, wt64.grad), "temporal filter gradient, last frame")


# ---------------------------------------------------------------- small kernels, element-wise
def test_optimizers_elementwise():
    """x3d_adam_step (Keras Adam with the bias-corrected lr_t training.py passes) and x3d_sgd_nesterov_step
    at an odd n with a mixed weight-decay mask, element-wise against float64."""
    L, check = _L()
    n = 1_000_003
    g = _gen(17)
    w, grad, m = _randn((n,), g) * 0.1, _randn((n,), g) * 0.1, _randn((n,), g) * 0.01
    v = torch.rand(n, device="cuda", generator=g) * 1e-3
    wd = torch.where(torch.rand(n, device="cuda", generator=g) < 0.5, 1e-4, 0.0)
    # the kernel takes its hyper-parameters as fp32 and forms 1 - b1, 1 - b2 in fp32 (exact), as Keras does
    # with its fp32 beta tensors; 1 - fp32(0.999) is 1.3e-5 away from 0.001, so the reference uses them too
    f32 = lambda v: float(np.float32(v))
    b1, b2, eps, lr, t = f32(0.9), f32(0.999), f32(1e-7), f32(0.05), 3
    lr_t = f32(lr * (1.0 - 0.999 ** t) ** 0.5 / (1.0 - 0.9 ** t))
    w64, g64, m64, v64 = w.double(), grad.double() + wd.double() * w.double(), m.double(), v.double()
    wn, mn, vn = w.clone(), m.clone(), v.clone()
    _run(lambda: check(L.x3d_adam_step(wn.data_ptr(), grad.data_ptr(), mn.data_ptr(), vn.data_ptr(), wd.data_ptr(), n,
                                       lr_t, b1, b2, eps, _st())), "adam_kernel")
    m1 = b1 * m64 + (1 - b1) * g64
    v1 = b2 * v64 + (1 - b2) * g64 * g64
    step = lr_t * m1 / (v1.sqrt() + eps)
    assert _rel(mn, m1) < 1e-6 and _rel(vn, v1) < 1e-6, (_rel(mn, m1), _rel(vn, v1))
    assert _rel(w64 - wn.double(), step) < 1e-5, _rel(w64 - wn.double(), step)
    _sharp(1e-5, float(step[-256:].abs().max() / step.abs().max()), "Adam tail")
    wn, vs = w.clone(), m.clone()
    _run(lambda: check(L.x3d_sgd_nesterov_step(wn.data_ptr(), grad.data_ptr(), vs.data_ptr(), wd.data_ptr(), n, lr, f32(0.9),
                                               _st())), "sgd_nesterov_kernel")
    mu = f32(0.9)
    v1 = mu * m64 - lr * g64
    assert _rel(vs, v1) < 1e-6 and _rel(wn.double() - w64, mu * v1 - lr * g64) < 1e-5


@pytest.mark.parametrize("op", range(6))
def test_ew_ops(op):
    """x3d_ew ops 0-5 (add + ReLU, ReLU', sigmoid, sigmoid', add, mask) at an odd n."""
    L, check = _L()
    n = 1_000_003
    g = _gen(op)
    a, b = _randn((n,), g) * 3, _randn((n,), g)
    if op == 3:
        b = torch.sigmoid(b)
    out = torch.empty_like(a)
    _run(lambda: check(L.x3d_ew(a.data_ptr(), None if op == 2 else b.data_ptr(), out.data_ptr(), n, op, _st())),
         "ew_kernel")
    a64, b64 = a.double(), b.double()
    want = [torch.relu(a64 + b64), a64 * (b64 > 0), torch.sigmoid(a64), a64 * b64 * (1 - b64), a64 + b64,
            a64 * b64][op]
    assert _rel(out, want) < 1e-6, _rel(out, want)
    _sharp(1e-6, float(want[-256:].abs().max() / want.abs().max()), "tail")


@pytest.mark.parametrize("accumulate", [0, 1])
def test_pool_bwd(accumulate):
    """x3d_pool_bwd at the SE pool of X3D-M stage 1 (32 clips x 50,176 rows, 56 channels)."""
    L, check = _L()
    clips, P, C = 32, 50176, 56
    g = _gen(accumulate)
    dm = _randn((clips, C), g)
    dy = _randn((clips * P, C), g)
    want = dy.double().view(clips, P, C) * accumulate + dm.double()[:, None, :] / P
    _run(lambda: check(L.x3d_pool_bwd(dm.data_ptr(), dy.data_ptr(), clips * P, C, P, 1.0 / P, accumulate, _st())),
         "pool_bwd_kernel")
    assert _rel(dy.view(clips, P, C), want) < 1e-6


def test_d2f_dropout_softmax_avgpool():
    """x3d_d2f (one rounding), x3d_dropout_mask (the splitmix64 stream, bit-exact), x3d_softmax_xent at
    N = 32 with a label below the 1e-7 clamp, and the head's avgpool against float64."""
    from x3d_tf_b200 import ops
    L, check = _L()
    g = _gen(23)
    n = 1_000_003
    d = _randn((n,), g, torch.float64) * 1e3
    f = torch.empty(n, device="cuda")
    _run(lambda: check(L.x3d_d2f(d.data_ptr(), f.data_ptr(), n, 0.25, _st())), "d2f_kernel")
    want = d * 0.25
    assert bool(((f.double() - want).abs() <= 2.0 ** -24 * want.abs()).all())
    # dropout: 32 x 2048 at rate 0.5
    n_m, rate, seed = 32 * 2048, 0.5, 0x1234_5678_9ABC_DEF0
    mask = torch.empty(n_m, device="cuda")
    _run(lambda: check(L.x3d_dropout_mask(mask.data_ptr(), n_m, rate, seed, _st())), "dropout_mask_kernel")
    with np.errstate(over="ignore"):
        z = np.uint64(seed) + np.uint64(0x9E3779B97F4A7C15) * np.arange(1, n_m + 1, dtype=np.uint64)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z ^= z >> np.uint64(31)
    u = (z >> np.uint64(40)).astype(np.float64) / 16777216.0
    keep = np.float32(1.0) / (np.float32(1.0) - np.float32(rate))
    assert np.array_equal(mask.cpu().numpy(), np.where(u >= rate, keep, np.float32(0)).astype(np.float32))
    # softmax cross-entropy, row 0's label far below the clamp
    N, ncls = 32, 400
    logits = _randn((N, ncls), g) * 3
    labels = torch.randint(0, ncls, (N,), device="cuda", generator=g, dtype=torch.int32)
    logits[0, labels[0]] = -40.0
    loss, dl = torch.empty(N, device="cuda"), torch.empty(N, ncls, device="cuda")
    _run(lambda: check(L.x3d_softmax_xent(logits.data_ptr(), labels.data_ptr(), loss.data_ptr(), dl.data_ptr(), N, ncls,
                                          1.0 / N, _st())), "softmax_xent_kernel")
    lt = logits.double().requires_grad_(True)
    p = torch.softmax(lt, -1).gather(1, labels.long()[:, None])[:, 0]
    assert float(p[0].detach()) < 1e-7
    lref = -torch.log(p.clamp(1e-7, 1 - 1e-7))
    (lref.sum() / N).backward()
    assert _rel(loss, lref) < 1e-5 and _rel(dl, lt.grad) < 1e-5
    assert not dl[0].any()
    _sharp(1e-5, float(lt.grad[-1].abs().max() / lt.grad.abs().max()), "last row")
    # head average pool: 32 clips x 16x7x7 positions x 432 channels
    a5 = _randn((32, 16 * 49, 432), g)
    pool = _run(lambda: ops.avgpool_fwd(a5), "avgpool_kernel")
    assert _rel(pool, a5.double().mean(1)) < 1e-5


# ---------------------------------------------------------------- coverage closure
# Kernel-name substring -> the case of this file that pins it at training sizes.
PINNED = {
    "pw_tf32_tc_kernel": "test_pw_tf32_at_training_sizes",
    "tf32_split_kernel": "test_pw_tf32_at_training_sizes",
    "pw_bf16_train_tc_kernel": "test_pw_bf16_train_at_training_sizes",
    "bf16_round_kernel": "test_pw_bf16_train_at_training_sizes",
    "pw_wgrad_bf16_kernel": "test_pw_bf16_train_at_training_sizes",
    "pw_wgrad_tf32x3_kernel": "test_pw_wgrad_tf32x3_every_tile_at_bench_m",
    "pw_gemm_tf32x3_kernel": "test_strided_shortcut_gemms_at_stage2_geometry",
    "gather_rows_kernel": "test_strided_shortcut_gemms_at_stage2_geometry",
    "dw_wgrad_pair_kernel": "test_dw_wgrad_paths",
    "dw_wgrad_kernel<1, 4>": "test_dw_wgrad_paths",
    "dw_wgrad_slide_kernel": "test_dw_wgrad_paths",
    "dw_tma_kernel": "test_channelwise_dgrad_of_the_training_step",
    "strided_add_kernel": "test_channelwise_dgrad_of_the_training_step",
    "colreduce_vec_kernel": "test_batchnorm_chain_at_scale",
    "colreduce_kernel": "test_colreduce_sums",
    "bn_finalize_kernel": "test_batchnorm_chain_at_scale",
    "bn_apply_kernel": "test_batchnorm_chain_at_scale",
    "bn_bwd_apply_kernel": "test_batchnorm_chain_at_scale",
    "scale_swish_fwd_kernel": "test_scale_swish_at_scale",
    "scale_swish_bwd_vec_kernel": "test_scale_swish_at_scale",
    "stem_convs_fwd_kernel": "test_stem_pieces_at_scale",
    "stem_convs_wgrad_vec_kernel": "test_stem_pieces_at_scale",
    "tconv_fwd_kernel": "test_stem_pieces_at_scale",
    "tconv_wgrad_vec_kernel": "test_stem_pieces_at_scale",
    "adam_kernel": "test_optimizers_elementwise",
    "sgd_nesterov_kernel": "test_optimizers_elementwise",
    "ew_kernel": "test_ew_ops",
    "pool_bwd_kernel": "test_pool_bwd",
    "d2f_kernel": "test_d2f_dropout_softmax_avgpool",
    "dropout_mask_kernel": "test_d2f_dropout_softmax_avgpool",
    "softmax_xent_kernel": "test_d2f_dropout_softmax_avgpool",
    "avgpool_kernel": "test_d2f_dropout_softmax_avgpool",
}
# torch's own kernels the step launches: zero fills, the contiguous copies and the tap flip
TORCH_KERNELS = ("FillFunctor", "copy_kernel", "flip")


def test_pinned_table_names_cases_of_this_file():
    assert all(callable(globals().get(case)) for case in PINNED.values())


@pytest.mark.parametrize("variant,crop,precision", [("X3D_M", 224, "float32"), ("X3D_M", 224, "mixed_bfloat16"),
                                                    ("X3D_XL", 312, "float32")])
def test_training_step_launches_only_pinned_kernels(variant, crop, precision):
    """One X3DTrainer.step (1 x 16 x crop^2) under the profiler: every kernel it launches is pinned by a
    case above or is one of torch's fill / copy / flip kernels, so a new launch path in the training
    step fails here until it has a parity case."""
    from x3d_tf_b200.arch import build_arch
    from x3d_tf_b200.config import get_config
    from x3d_tf_b200.synth import synthetic_clips, synthetic_weights
    from x3d_tf_b200.training import X3DTrainer
    cfg = get_config(variant)
    tr = X3DTrainer(cfg, precision=precision).load(synthetic_weights(build_arch(cfg), seed=1))
    x = torch.from_numpy(synthetic_clips(1, 16, crop, crop, cfg.DATA.MEAN, cfg.DATA.STD, seed=2)).cuda()
    labels = torch.zeros(1, dtype=torch.int32, device="cuda")
    names = _launched(lambda: tr.step(x, labels, 0.01))
    loose = sorted(n for n in names if not any(k in n for k in PINNED) and not any(k in n for k in TORCH_KERNELS))
    assert not loose, loose
    if variant == "X3D_XL":
        assert any("dw_wgrad_kernel<1, 4>" in n for n in names)
