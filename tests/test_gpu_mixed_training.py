"""The 'mixed_bfloat16' training policy on the GPU: the bf16 GEMM kernels against float64 products of
the same bf16-rounded operands, the whole step against the rounding oracle (tests/mixed_oracle.py),
and the policy through the trainer, the driver, `fit` and two replicas."""
import numpy as np
import pytest
import torch

from oracle import x3d_oracle as O
from oracle import x3d_train_oracle as TO
from tests import mixed_oracle as MO

pytestmark = pytest.mark.gpu
MIXED = "mixed_bfloat16"


def _p8(c):
    return (c + 7) // 8 * 8


def _layer_shapes():
    """(K, N, dense) of every 1x1x1 conv / Dense layer of X3D-XS, -M, -L and -XL training (device layouts).
    X3D-XL adds a 160-column N tile (N = 312) and three N tiles (N = 632)."""
    from x3d_tf_b200.arch import build_arch
    from x3d_tf_b200.config import get_config
    out = set()
    for v in ("X3D_XS", "X3D_M", "X3D_L", "X3D_XL"):
        ar = build_arch(get_config(v))
        for b in ar.blocks:
            cin, ci, co = _p8(b.cin), _p8(b.cinner), _p8(b.cout)
            out |= {(cin, ci, False), (ci, co, False)}
            if b.has_shortcut:
                out.add((cin, co, False))
            if b.se_width:
                out |= {(ci, b.se_width, True), (b.se_width, ci, True)}
        c5 = _p8(ar.conv5_channels)
        out |= {(_p8(ar.blocks[-1].cout), c5, False), (c5, ar.fc1_channels, True),
                (ar.fc1_channels, ar.num_classes, True)}
    return sorted(out)


def _r64(t):
    return t.to(torch.bfloat16).double()


def _rel(got, want):
    got, want = torch.as_tensor(got).double(), torch.as_tensor(want).double()
    return float((got - want).abs().max() / max(float(want.abs().max()), 1e-30))


def _bound(K):
    # the tf32 kernels' bound against float64 (DESIGN section 9) for K <= 512; fp32 accumulation error
    # grows with the number of terms, so fc2 (K = 2048) gets it scaled by K / 512
    return 5e-6 * max(1.0, K / 512)


@pytest.mark.parametrize("K,N,dense", _layer_shapes())
def test_bf16_gemms_match_float64_of_rounded_operands(K, N, dense):
    from x3d_tf_b200 import ops
    torch.cuda.set_device(0)
    g = torch.Generator(device="cuda").manual_seed(K * 1000 + N)
    M = 2 if dense else 1000                                 # dense layers see the batch; 1000 % 128 != 0
    a = torch.randn(M, K, device="cuda", generator=g)
    w = torch.randn(K, N, device="cuda", generator=g) / K ** 0.5
    dy = torch.randn(M, N, device="cuda", generator=g)
    ref = _r64(a) @ _r64(w)
    # forward: plain with the BatchNorm statistics epilogue, and with bias + ReLU
    st = torch.zeros(2, N, dtype=torch.float64, device="cuda")
    y = ops.pw_bf16_train(a, ops.bf16_round(w, transpose_w=True), K, stats=st)
    assert _rel(y, ref) < _bound(K)
    assert _rel(st[0], ref.sum(0)) < _bound(K) * 4 and _rel(st[1], (ref * ref).sum(0)) < _bound(K) * 4
    bias = torch.randn(N, device="cuda", generator=g)
    yb = ops.pw_bf16_train(a, ops.bf16_round(w, transpose_w=True), K, bias, relu=True)
    assert _rel(yb, torch.relu(ref + bias.double())) < _bound(K)
    # backward-data: dx = bf16(dy) . bf16(w)^T
    dx = ops.pw_bf16_train(dy, ops.bf16_round(w, transpose_w=False), N)
    assert _rel(dx, _r64(dy) @ _r64(w).t()) < _bound(N)
    # backward-filter: dw = bf16(a)^T . bf16(dy), accumulated into fp64
    dw = torch.zeros(K, N, dtype=torch.float64, device="cuda")
    ops.pw_wgrad_bf16(a, dy, dw)
    assert _rel(dw, _r64(a).t() @ _r64(dy)) < _bound(M)
    # the kernel is the rounded product, not the fp32 one
    if not dense:
        assert _rel(y, a.double() @ w.double()) > 10 * _bound(K)


@pytest.mark.parametrize("C,Co,H,W,s", [(24, 24, 32, 32, 2), (48, 48, 9, 7, 2), (96, 192, 14, 14, 2)])
def test_bf16_gemms_on_gathered_shortcut_rows(C, Co, H, W, s):
    from x3d_tf_b200 import ops
    torch.cuda.set_device(0)
    g = torch.Generator(device="cuda").manual_seed(C + H)
    N, T = 2, 3
    x5 = torch.randn(N, T, H, W, C, device="cuda", generator=g)
    w = torch.randn(C, Co, device="cuda", generator=g) / C ** 0.5
    Ho, Wo = (H - 1) // s + 1, (W - 1) // s + 1
    rows = x5[:, :, ::s, ::s].reshape(-1, C)
    dy = torch.randn(rows.shape[0], Co, device="cuda", generator=g)
    y = ops.pw_bf16_train(ops.gather_rows_fwd(x5, s), ops.bf16_round(w), C)
    assert _rel(y, _r64(rows) @ _r64(w)) < _bound(C)
    dw = torch.zeros(C, Co, dtype=torch.float64, device="cuda")
    ops.pw_wgrad_bf16(x5.view(-1, C), dy, dw, M=rows.shape[0], gather=(T, Ho, Wo, H, W, s))
    assert _rel(dw, _r64(rows).t() @ _r64(dy)) < _bound(rows.shape[0])


def _setup(variant="X3D_XS", n=2, t=4, s=64, dropout=0.5, seed=3, optimizer=None):
    from x3d_tf_b200.arch import build_arch
    from x3d_tf_b200.config import get_config
    from x3d_tf_b200.synth import synthetic_clips, synthetic_weights
    from x3d_tf_b200.training import X3DTrainer
    cfg = get_config(variant, freeze=False)
    cfg.NETWORK.DROPOUT_RATE = dropout
    if optimizer:
        cfg.TRAIN.OPTIMIZER = optimizer
    cfg.freeze()
    W = synthetic_weights(build_arch(cfg), seed=seed)
    x = synthetic_clips(n, t, s, s, cfg.DATA.MEAN, cfg.DATA.STD, seed=seed + 1)
    rng = np.random.default_rng(seed + 2)
    labels = rng.integers(0, cfg.NETWORK.NUM_CLASSES, size=n).astype(np.int32)
    mask = None
    if dropout > 0:
        mask = ((rng.random((n, 2048)) >= dropout) / (1.0 - dropout)).astype(np.float32)
    torch.cuda.set_device(0)
    tr = X3DTrainer(cfg, precision=MIXED).load(W)
    if mask is not None:
        tr.fixed_dropout_mask = torch.from_numpy(mask).cuda()
    return cfg, W, x, labels, mask, tr


@pytest.mark.parametrize("variant,n,t,s,optimizer", [("X3D_XS", 2, 4, 64, "sgd"), ("X3D_S", 2, 4, 91, "sgd"),
                                                     ("X3D_XS", 2, 4, 64, "adam"), ("X3D_M", 2, 16, 224, "sgd")])
def test_mixed_step_matches_rounding_oracle(variant, n, t, s, optimizer):
    """Loss, logits, every gradient, the update and the moving statistics of one mixed step against
    the rounding oracle, with the fp32 test's tolerances and its ReLU branch masks (see
    test_gpu_training.py).  The oracle is also told which bf16 neighbour the device rounded each GEMM
    operand to (tests/mixed_oracle.py: without that, elements near a tie round apart and the two runs
    drift to the bf16 level within a few layers: 0.10 of the logits' scale measured at X3D-XS); at most
    2 % of the operands may take the device's neighbour.  The same step is also compared with the
    plain float64 oracle: that gap is the precision the policy gives up, and it must be at least 10x
    the gap to the rounding oracle."""
    cfg, W, x, labels, mask, tr = _setup(variant, n=n, t=t, s=s, optimizer=optimizer)
    tr.relu_masks = []
    tr.gemm_operands = {}
    lr, wd = (0.05 if optimizer == "sgd" else 1e-3), float(cfg.NETWORK.WEIGHT_DECAY)
    loss = tr.step(torch.from_numpy(x).cuda(), torch.from_numpy(labels).cuda(), lr)
    torch.cuda.synchronize()
    spec = O.OracleSpec.from_cfg(cfg)
    kw = dict(lr=lr, momentum=0.9, weight_decay=wd, dropout_mask=mask, relu_masks=tr.relu_masks,
              optimizer=optimizer)
    operands = {name: (tr.gemm_operands[("fwd", tr.P(name).data_ptr())],
                       tr.gemm_operands[("bwd", tr.P(name).data_ptr())])
                for name in tr.layout.slots if ("fwd", tr.P(name).data_ptr()) in tr.gemm_operands}
    assert len(operands) == sum(1 for k in W if k.endswith("/kernel") and not k.endswith("/b/kernel")
                                and not k.startswith("conv1/"))
    MO.FORCED.update(elements=0, forced=0)
    ref = MO.train_step(W, spec, x, labels, operands=operands, **kw)
    forced = MO.FORCED["forced"] / MO.FORCED["elements"]
    plain = MO.train_step(W, spec, x, labels, gemm_round=False, **kw)
    logits = tr.last_logits.cpu().numpy()
    gap_round, gap_plain = _rel(logits, ref["logits"]), _rel(logits, plain["logits"])
    print(f"{variant} {optimizer}: logits vs rounding oracle {gap_round:.3e}, vs float64 oracle {gap_plain:.3e}; "
          f"device's bf16 neighbour taken for {forced:.2e} of the GEMM operands")
    assert forced < 2e-2
    assert gap_round < 1e-4
    assert abs(float(loss.mean().item()) - ref["loss"]) < 1e-4 * max(1.0, abs(ref["loss"]))
    assert gap_plain >= 10 * gap_round
    G = tr.grads()
    bad = []
    for k, g_ref in ref["grads"].items():
        got = G[k].astype(np.float64)
        if TO.is_regularised(k):
            got = got + 2.0 * wd * W[k]
        if _rel(got, g_ref) > 1e-3:
            bad.append((k, _rel(got, g_ref)))
    assert not bad, bad[:10]
    Wn = tr.weights()
    if optimizer == "sgd":
        bad = [(k, _rel(Wn[k], v)) for k, v in ref["weights"].items()
               if _rel(Wn[k], v) > (2e-4 if k.startswith("conv1/") else 1e-4)]
    else:
        # Adam's first step is lr * sign(g) where g is far from zero: the displacement's L2 distance
        # (as test_gpu_training.test_adam_step_matches_oracle), moving statistics element-wise
        bad = []
        for k, v in ref["weights"].items():
            if k.endswith("moving_mean") or k.endswith("moving_variance"):
                e = _rel(Wn[k], v)
                lim = 1e-4
            else:
                d = Wn[k].astype(np.float64) - W[k]
                e = float(np.linalg.norm(d - (v - W[k])) / max(np.linalg.norm(v - W[k]), 1e-30))
                lim = 5e-2
            if e > lim:
                bad.append((k, e))
    assert not bad, bad[:10]


def test_mixed_training_lowers_the_loss_as_fp32_does():
    """Twenty SGD steps on one fixed batch (which the model can memorise): both policies lower the
    loss, and the mixed run ends within 0.1 of the initial loss of where fp32 ends.  (At lr 0.05 this
    batch is chaotic: the float64 oracle, with and without the GEMM rounding, jumps to a loss of 7 at
    step 6 and settles at 4.03, where the fp32 kernels reach 0.0014 -- so the check runs at 0.01.)"""
    from x3d_tf_b200.training import X3DTrainer
    cfg, W, x, labels, _, _ = _setup("X3D_XS", n=4, dropout=0.0, seed=11)
    xd, ld = torch.from_numpy(x).cuda(), torch.from_numpy(labels).cuda()
    curves = {}
    for prec in ("float32", MIXED):
        tr = X3DTrainer(cfg, precision=prec).load(W)
        curves[prec] = [float(tr.step(xd, ld, 0.01).mean().item()) for _ in range(20)]
    print({k: [round(v, 4) for v in c] for k, c in curves.items()})
    f, m = curves["float32"], curves[MIXED]
    assert abs(m[0] - f[0]) < 1e-2 * f[0]
    assert f[-1] < 0.5 * f[0] and m[-1] < 0.5 * m[0]
    assert abs(m[-1] - f[-1]) < 0.1 * f[0]


def test_mixed_checkpoint_has_fp32_keys_and_evaluates(tmp_path, capsys):
    from x3d_tf_b200 import eval as E
    from x3d_tf_b200 import model as M
    from x3d_tf_b200 import tf_bundle as B
    from x3d_tf_b200 import train as T
    from x3d_tf_b200.config import get_config
    args = ["--config", "X3D_XS", "--synthetic", "4", "--batch_size", "2", "--crop_size", "64",
            "--steps_per_epoch", "2", "--epochs", "1"]
    r = T.run(args + ["--model_dir", str(tmp_path / "mixed"), "--mixed_precision"])
    assert r["iteration"] == 2 and np.isfinite(r["history"][0]["loss"])
    assert r["history"][0]["policy"] == MIXED and "policy: mixed_bfloat16" in capsys.readouterr().out
    T.run(args + ["--model_dir", str(tmp_path / "fp32")])
    pm, pf = str(tmp_path / "mixed" / "ckpt-1"), str(tmp_path / "fp32" / "ckpt-1")
    assert sorted(B.load_model_variables(pm)) == sorted(B.load_model_variables(pf))
    sm, sf = B.load_optimizer_state(pm), B.load_optimizer_state(pf)
    assert sorted(sm["slots"]) == sorted(sf["slots"])
    cfg = get_config("X3D_XS")
    M.reset_block_counters()
    m = M.X3D(cfg, dtype="bfloat16")
    m.set_weights_dict(B.load_model_variables(pm))
    num_preds = cfg.TEST.NUM_TEMPORAL_VIEWS * cfg.TEST.NUM_SPATIAL_CROPS
    vpb = max(cfg.TEST.BATCH_SIZE // num_preds, 1)
    want = m.compile().evaluate(E.synthetic_batches(0, 3, vpb, num_preds, cfg.DATA.TEMP_DURATION,
                                                    cfg.DATA.TEST_CROP_SIZE, cfg.NETWORK.NUM_CLASSES))
    M.reset_block_counters()
    got = E.run(["--cfg", "X3D_XS", "--model_folder", str(tmp_path / "mixed"), "--synthetic", "3"])
    assert got == want and got["videos"] == 3


def test_fit_mixed_precision_equals_trainer():
    from x3d_tf_b200 import model as M
    from x3d_tf_b200.training import X3DTrainer
    cfg, W, x, labels, _, _ = _setup("X3D_XS", dropout=0.5, seed=5)
    data = [(x, labels), (x[::-1].copy(), labels[::-1].copy())]
    M.reset_block_counters()
    m = M.X3D(cfg)
    m.set_weights_dict(W)
    hist = m.fit(data, epochs=2, lr_schedule=lambda e: 0.02 * (e + 1), mixed_precision=True)
    assert m._tr.precision == MIXED
    tr = X3DTrainer(cfg, precision=MIXED).load(W)
    losses = []
    for e in range(2):
        tot = 0.0
        for cx, cl in data:
            tot += float(tr.step(torch.from_numpy(np.ascontiguousarray(cx)).cuda(),
                                 torch.from_numpy(np.ascontiguousarray(cl)).cuda(), 0.02 * (e + 1)).double().mean())
        losses.append(tot / len(data))
    np.testing.assert_allclose(hist["loss"], losses, rtol=1e-12)
    got, want = m.named_variables(), tr.weights()
    for k, v in want.items():
        assert np.array_equal(got[k], v), k


def _mixed_train_worker(rank, world, port, q):
    from tests.test_gpu_multi import _init
    dist = _init(rank, world, port)
    from x3d_tf_b200.arch import build_arch
    from x3d_tf_b200.config import get_config
    from x3d_tf_b200.synth import synthetic_clips, synthetic_weights
    from x3d_tf_b200.training import X3DTrainer
    cfg = get_config("X3D_XS")
    W = synthetic_weights(build_arch(cfg), seed=9)
    x = synthetic_clips(2, 4, 64, 64, cfg.DATA.MEAN, cfg.DATA.STD, seed=30 + rank)
    lab = np.random.default_rng(40 + rank).integers(0, 400, size=2).astype(np.int32)
    dev = torch.device("cuda", rank)
    tr = X3DTrainer(cfg, device=dev, world=world, rank=rank, precision=MIXED).load(W)
    for lr in (0.05, 0.02):
        tr.step(torch.from_numpy(x).to(dev), torch.from_numpy(lab).to(dev), lr)
    torch.cuda.synchronize()
    out = (tr.g.cpu().numpy(), tr.w.cpu().numpy())
    dist.barrier()
    dist.destroy_process_group()
    q.put((rank, out))


def test_mixed_replicas_stay_identical_on_two_gpus():
    from tests.test_gpu_multi import _need_two, _spawn
    _need_two()
    out = _spawn(_mixed_train_worker)
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])
