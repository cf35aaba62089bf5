"""One data-parallel training step of X3D on B200 (BASELINE.json configs[4]).

Mirrors what Keras `fit` does per replica for the reference (train.py:85-152; model.py with
training=True; SURVEY.md Appendix A.7) with hand-written CUDA kernels behind the C ABI
(`include/x3d_b200.h`, section "Training step"):

    forward   batch-statistics BatchNorm, dropout, softmax + sparse CE on the probabilities
    backward  backward-data / backward-filter of every convolution, BN / SE / swish / ReLU / pool
    exchange  ONE sum all-reduce of the flat fp32 gradient arena over NCCL (MirroredStrategy's
              cross-replica sum, utils.py:160-167); loss scaled by 1/world first
    update    SGD(nesterov=True) + L2 on conv/dense kernels except se_fc1 (train.py:88-92, model.py:47)

PyTorch owns device memory, the stream and the NCCL communicator; all arithmetic is in the kernels.
fp32 activations (the reference's default precision).  First correct version: kernels are simple
and unfused (DESIGN.md section 9).

precision="mixed_bfloat16" (train.py --mixed_precision): every 1x1x1 conv and Dense layer multiplies
bf16 operands (round-to-nearest-even) with fp32 accumulation -- forward, backward-data and
backward-filter; activations, BatchNorm, the channelwise and stem convs, SE, softmax, the fp32 master
weights, the fp64 gradient accumulators, the optimizers and the all-reduce stay as in float32.  bf16
has fp32's exponent range, so no loss scaling.
"""
from __future__ import annotations

from collections import OrderedDict
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch

from . import arch as A
from . import ops
from ._lib import check, lib


def _pad8(c: int) -> int:
    return (c + 7) // 8 * 8


def _s() -> int:
    return torch.cuda.current_stream().cuda_stream


class _Arena:
    """Flat fp32 parameter arena with named views; gradient (fp32 + fp64 accumulation), velocity
    and weight-decay arenas share the layout."""

    def __init__(self):
        self.slots: "OrderedDict[str, Tuple[int, Tuple[int, ...]]]" = OrderedDict()
        self.size = 0

    def add(self, name: str, shape: Tuple[int, ...]):
        n = int(np.prod(shape))
        self.slots[name] = (self.size, tuple(shape))
        self.size += (n + 3) // 4 * 4           # keep every slot 16-byte aligned

    def view(self, flat: torch.Tensor, name: str) -> torch.Tensor:
        off, shape = self.slots[name]
        return flat[off:off + int(np.prod(shape))].view(shape)


def channelwise_dgrad(dy5: torch.Tensor, wb: torch.Tensor, zero_b: torch.Tensor, H: int, W: int, s: int, ph: int,
                      pw_: int) -> torch.Tensor:
    """Backward-data of the channelwise 3x3x3 SAME conv (taps `wb` [27, C], stride (1, s, s), pads before
    `ph`, `pw_`): dy5 [N, T, Ho, Wo, C] -> dx [N, T, H, W, C], through the forward kernel.  For stride 1 it
    is the SAME convolution of dy with the taps reversed; for stride 2 dy is first zero-dilated onto the
    input grid (at offset 1 - pad_before per axis), which makes it the same stride-1 convolution.
    tests/test_gpu_train_kernels_at_scale.py checks this function against float64 autograd; x3d_dw_dgrad,
    the direct gather form, stays in the ABI.  `zero_b`: a zero [C] bias."""
    N, T, Ho, Wo, ci = dy5.shape
    wflip = wb.flip(0).contiguous()
    if s == 1:
        g = dy5
    else:
        g = torch.zeros((N, T, H, W, ci), dtype=torch.float32, device=dy5.device)
        off = ((1 - ph) * W + (1 - pw_)) * ci
        check(lib().x3d_strided_add(dy5.data_ptr(), g.data_ptr() + 4 * off, N * T, Ho, Wo, H, W, s, ci, _s()),
              "x3d_strided_add")
    dx, _ = ops.dw_fwd(g, wflip, zero_b, 1, 1, 1, False)
    return dx


def _mix64(z: int) -> int:
    """splitmix64 finaliser (the same hash the dropout kernel applies per element)."""
    z &= (1 << 64) - 1
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & ((1 << 64) - 1)
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & ((1 << 64) - 1)
    return z ^ (z >> 31)


class X3DTrainer:
    """`X3DTrainer(cfg).load(weights)`; `loss = trainer.step(clips, labels, lr)`."""

    PRECISIONS = ("float32", "mixed_bfloat16")

    def __init__(self, cfg, device=None, world: int = 1, process_group=None, seed: int = 1111, rank: int = 0,
                 precision: str = "float32"):
        if precision not in self.PRECISIONS:
            raise ValueError(f"precision {precision!r}: expected one of {self.PRECISIONS}")
        self.precision = precision
        self.mixed = precision == "mixed_bfloat16"
        self._wb: Dict[Tuple[int, bool], torch.Tensor] = {}     # bf16 kernels of this step (mixed)
        self.cfg = cfg
        self.rank = rank                    # mixed into the dropout stream: replicas draw independent masks
        self.arch = A.build_arch(cfg)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else device
        self.world, self.pg = world, process_group
        net = cfg.NETWORK
        self.eps, self.bn_momentum = float(net.BN.EPS), float(net.BN.MOMENTUM)
        self.wd2 = 2.0 * float(net.WEIGHT_DECAY)
        self.dropout = float(net.DROPOUT_RATE)
        self.momentum = float(cfg.TRAIN.MOMENTUM) if hasattr(cfg, "TRAIN") and hasattr(cfg.TRAIN, "MOMENTUM") else 0.9
        # train.py:85-97: 'sgd' (Nesterov momentum) or 'adam' (Keras defaults)
        self.optimizer = str(cfg.TRAIN.OPTIMIZER).lower() if hasattr(cfg, "TRAIN") and hasattr(cfg.TRAIN, "OPTIMIZER") else "sgd"
        if self.optimizer not in ("sgd", "adam"):
            raise NotImplementedError(f"{self.optimizer} not supported")
        self.adam = (0.9, 0.999, 1e-7)
        self.seed, self.iteration = seed, 0
        # fp32 pointwise GEMMs (forward / backward-data): "tcgen05" = kind::tf32 MMA with the 3xTF32 split
        # (x3d_pw_tf32_fwd); "mma_sync" = the legacy-path kernel of round 1 (x3d_pw_fwd).  X3D_TRAIN_GEMM overrides.
        import os as _os
        self.gemm = _os.environ.get("X3D_TRAIN_GEMM", "tcgen05")
        self.fixed_dropout_mask: Optional[torch.Tensor] = None      # tests inject a mask
        self.relu_masks: Optional[list] = None                      # tests: record every ReLU's sign pattern
        self.gemm_operands: Optional[dict] = None                   # tests (mixed): record every GEMM's fp32
        #                                                             activation operand, by (pass, kernel ptr)
        ar = self.arch
        self.layout = _Arena()
        self.tf_shape: Dict[str, Tuple[int, ...]] = {}
        self.decay: Dict[str, bool] = {}
        self.stats: List[str] = []                                     # BN prefixes (moving stats)

        def conv(name, tf_shape, dev_shape, decay=True):
            self.layout.add(name, dev_shape); self.tf_shape[name] = tf_shape; self.decay[name] = decay

        def bn(prefix, c):
            cs = _pad8(c)
            conv(prefix + "/beta", (c,), (cs,), False)                 # beta, gamma adjacent: the BN
            conv(prefix + "/gamma", (c,), (cs,), False)                # backward sums land on both
            self.stats.append(prefix)

        c1 = ar.stem_channels
        conv("conv1/conv_s/kernel", (1, 3, 3, 3, c1), (27, _pad8(c1)))
        conv("conv1/conv_t/kernel", (ar.temp_filter, 1, 1, 1, c1), (ar.temp_filter, _pad8(c1)))
        bn("conv1/bn", c1)
        for b in ar.blocks:
            p = f"stages/{b.stage}/stage/layer_with_weights-{b.index}"
            q = p + "/bottleneck"
            cin, ci, co = _pad8(b.cin), _pad8(b.cinner), _pad8(b.cout)
            if b.has_shortcut:
                conv(p + "/residual/kernel", (1, 1, 1, b.cin, b.cout), (cin, co))
                bn(p + "/bn_r", b.cout)
            conv(q + "/a/kernel", (1, 1, 1, b.cin, b.cinner), (cin, ci))
            bn(q + "/bn_a", b.cinner)
            conv(q + "/b/kernel", (3, 3, 3, 1, b.cinner), (27, ci))
            bn(q + "/bn_b", b.cinner)
            if b.se_width:
                conv(q + "/se_fc1/kernel", (1, 1, 1, b.cinner, b.se_width), (ci, b.se_width), False)
                conv(q + "/se_fc1/bias", (b.se_width,), (b.se_width,), False)
                conv(q + "/se_fc2/kernel", (1, 1, 1, b.se_width, b.cinner), (b.se_width, ci))
                conv(q + "/se_fc2/bias", (b.cinner,), (ci,), False)
            conv(q + "/c/kernel", (1, 1, 1, b.cinner, b.cout), (ci, co))
            bn(q + "/bn_c", b.cout)
        cl, c5 = ar.blocks[-1].cout, ar.conv5_channels
        conv("conv5/layer_with_weights-0/kernel", (1, 1, 1, cl, c5), (_pad8(cl), _pad8(c5)))
        bn("conv5/layer_with_weights-1", c5)
        conv("fc1/kernel", (1, 1, 1, c5, ar.fc1_channels), (_pad8(c5), ar.fc1_channels))
        conv("fc2/kernel", (ar.fc1_channels, ar.num_classes), (ar.fc1_channels, ar.num_classes))
        conv("fc2/bias", (ar.num_classes,), (ar.num_classes,), False)

        n, dev = self.layout.size, self.device
        self.w = torch.zeros(n, dtype=torch.float32, device=dev)
        self.g = torch.zeros(n, dtype=torch.float32, device=dev)
        self.g64 = torch.zeros(n, dtype=torch.float64, device=dev)
        self.v = torch.zeros(n, dtype=torch.float32, device=dev)          # SGD momentum / Adam m
        self.v2 = torch.zeros(n, dtype=torch.float32, device=dev) if self.optimizer == "adam" else None   # Adam v
        self.wd = torch.zeros(n, dtype=torch.float32, device=dev)
        # gradient exchange (exchange.py): buckets cut where stages 4 and 5 (s = 2, 3) start, in backward
        # order: [stage 5 + conv5 + fc1 + fc2] (83 % of the bytes), [stage 4] (15 %), [stem + stages 2, 3]
        from .exchange import GradientExchange, make_buckets
        edges, self._bucket_of_stage = [], {}
        for st in (2, 3):
            first = next((k for k in self.layout.slots if k.startswith(f"stages/{st}/")), None)
            if first is not None:
                edges.append(self.layout.slots[first][0])
        buckets = make_buckets(n, edges)
        for st in (2, 3):
            first = next((k for k in self.layout.slots if k.startswith(f"stages/{st}/")), None)
            if first is not None:
                self._bucket_of_stage[st] = next(i for i, (lo, hi) in enumerate(buckets)
                                                 if lo == self.layout.slots[first][0])
        self.exchange = GradientExchange(self.g, buckets, world, process_group)
        self._exchange_in_backward = False
        # BatchNorm batch statistics of one step: fp64 [2, C] per BN layer, zeroed once per step
        self._stat_arena = torch.zeros(2 * sum(_pad8(c) for c in self._bn_channels()), dtype=torch.float64, device=dev)
        self._stat_used = 0
        self._converted: list = []
        for name in self.layout.slots:
            if self.decay[name]:
                self.layout.view(self.wd, name).fill_(self.wd2)
        self.moving: Dict[str, torch.Tensor] = {}
        for pfx in self.stats:
            cs = self.layout.slots[pfx + "/gamma"][1][0]
            self.moving[pfx + "/moving_mean"] = torch.zeros(cs, dtype=torch.float32, device=dev)
            self.moving[pfx + "/moving_variance"] = torch.ones(cs, dtype=torch.float32, device=dev)

    # ------------------------------------------------------------------ weights in / out
    def _bn_channels(self):
        ar = self.arch
        yield ar.stem_channels
        for b in ar.blocks:
            if b.has_shortcut:
                yield b.cout
            yield b.cinner
            yield b.cinner
            yield b.cout
        yield ar.conv5_channels

    def P(self, name: str) -> torch.Tensor:
        return self.layout.view(self.w, name)

    def G64(self, name: str) -> torch.Tensor:
        return self.layout.view(self.g64, name)

    def _to_dev_layout(self, name: str, a: np.ndarray) -> np.ndarray:
        shape = self.layout.slots[name][1]
        a = np.asarray(a, np.float32)
        if name.endswith("conv_s/kernel"):
            a = a.reshape(27, -1)
        elif name.endswith("conv_t/kernel") or name.endswith("/b/kernel"):
            a = a.reshape(a.shape[0] * a.shape[1] * a.shape[2], -1)
        elif a.ndim == 5:
            a = a.reshape(a.shape[3], a.shape[4])
        out = np.zeros(shape, np.float32)
        out[tuple(slice(0, s) for s in a.shape)] = a
        return out

    def load(self, weights: Dict[str, np.ndarray]) -> "X3DTrainer":
        for name in self.layout.slots:
            self.P(name).copy_(torch.from_numpy(self._to_dev_layout(name, weights[name])))
        for name, t in self.moving.items():
            a = np.asarray(weights[name], np.float32)
            t.zero_() if name.endswith("mean") else t.fill_(1.0)
            t[:a.shape[0]].copy_(torch.from_numpy(a))
        return self

    def _from_dev_layout(self, name: str, t: torch.Tensor) -> np.ndarray:
        tf = self.tf_shape[name]
        a = t.detach().float().cpu().numpy()
        if len(tf) == 5 and tf[0] * tf[1] * tf[2] > 1:          # conv_s / conv_t / b
            taps = tf[0] * tf[1] * tf[2] * tf[3]
            return a[:taps, :tf[4]].reshape(tf)
        if len(tf) == 5:
            return a[:tf[3], :tf[4]].reshape(tf)
        return a[tuple(slice(0, s) for s in tf)].reshape(tf)

    def weights(self) -> Dict[str, np.ndarray]:
        out = {n: self._from_dev_layout(n, self.P(n)) for n in self.layout.slots}
        for name, t in self.moving.items():
            c = self.tf_shape[name.rsplit("/", 1)[0] + "/gamma"][0]
            out[name] = t[:c].cpu().numpy()
        return out

    def grads(self) -> Dict[str, np.ndarray]:
        """Data-loss gradients of the last step (after the all-reduce; without the L2 term)."""
        return {n: self._from_dev_layout(n, self.layout.view(self.g, n)) for n in self.layout.slots}

    def velocity(self) -> Dict[str, np.ndarray]:
        """Momentum slots (the `.OPTIMIZER_SLOT/optimizer/momentum` variables of a Keras checkpoint;
        Adam: the first-moment slots `.../optimizer/m`)."""
        return {n: self._from_dev_layout(n, self.layout.view(self.v, n)) for n in self.layout.slots}

    def second_moment(self) -> Dict[str, np.ndarray]:
        """Adam's `.OPTIMIZER_SLOT/optimizer/v` slots."""
        return {n: self._from_dev_layout(n, self.layout.view(self.v2, n)) for n in self.layout.slots}

    # ------------------------------------------------------------------ checkpoints (utils.py:128-132)
    def save_checkpoint(self, prefix: str, lr: float = 0.0) -> None:
        """What Keras `ModelCheckpoint(.../ckpt-{epoch})` writes for this model and optimizer: the
        model variables, `optimizer/{iter,learning_rate,momentum,decay}` and one momentum slot per
        trainable variable (key map: SURVEY.md Appendix C.4), as a TF tensor bundle plus the
        `checkpoint` state file.  (No object graph: readable by name, see tf_bundle.write_bundle.)"""
        from . import tf_bundle
        tensors = dict(self.weights())
        if self.optimizer == "adam":
            tensors.update(tf_bundle.adam_tensors(self.iteration, lr, self.adam[0], self.adam[1],
                                                  self.velocity(), self.second_moment()))
        else:
            tensors.update(tf_bundle.optimizer_tensors(self.iteration, lr, self.momentum, self.velocity()))
        tf_bundle.write_bundle(prefix, tensors)

    def load_checkpoint(self, prefix: str, strict_slots: bool = False) -> dict:
        """Restore weights, moving statistics, momentum slots and the iteration counter from a
        checkpoint written by `save_checkpoint` or by the reference's `train.py`.  A checkpoint
        without optimizer state (`model.save_weights`) restarts the momentum at zero unless
        `strict_slots`."""
        from . import tf_bundle
        self.load(tf_bundle.load_model_variables(prefix))
        st = tf_bundle.load_optimizer_state(prefix)
        adam = self.optimizer == "adam"
        slots = st["slots_m"] if adam else st["slots"]
        self.v.zero_()
        if adam:
            self.v2.zero_()
        for name in self.layout.slots:
            if name in slots:
                self.layout.view(self.v, name).copy_(torch.from_numpy(self._to_dev_layout(name, slots[name])))
                if adam and name in st["slots_v"]:
                    self.layout.view(self.v2, name).copy_(
                        torch.from_numpy(self._to_dev_layout(name, st["slots_v"][name])))
            elif strict_slots:
                raise KeyError(f"{prefix}: no optimizer slot for {name}")
        if st["iter"] is not None:
            self.iteration = int(st["iter"])
        return st

    # ------------------------------------------------------------------ primitive ops
    def _bf16_kernel(self, w, transpose_w):
        """`w` rounded to bf16 in the orientation the GEMM reads, once per step: the cache is emptied when
        a step starts, i.e. after the previous update."""
        key = (w.data_ptr(), transpose_w)
        if key not in self._wb:
            self._wb[key] = ops.bf16_round(w, transpose_w=transpose_w)
        return self._wb[key]

    def _pw(self, x2d, w, bias=None, relu=False, gather=None, M=None, stats=None):
        """`stats`: None, or a zeroed fp64 [2, N] slice that the GEMM epilogue fills with the column sums /
        sums of squares of the result (the following BatchNorm's batch statistics); returns (y, filled)."""
        K, N = w.shape
        if self.mixed:
            if gather is not None:
                T, _, _, H, W, s = gather
                x2d = ops.gather_rows_fwd(x2d.view(-1, T, H, W, x2d.shape[-1]), s)
            if self.gemm_operands is not None:
                self.gemm_operands[("fwd", w.data_ptr())] = x2d.cpu().numpy()
            y = ops.pw_bf16_train(x2d, self._bf16_kernel(w, True), K, bias, relu=relu, stats=stats)
            return y if stats is None else (y, True)
        if gather is None and self.gemm == "tcgen05":
            # tcgen05.mma kind::tf32, 3xTF32 split (csrc/x3d_pw_tf32_tc.cu)
            y = ops.pw_tf32(x2d, w, bias, relu=relu, transpose_w=True, M=M, stats=stats)
            return y if stats is None else (y, True)
        if stats is not None:
            return ops.pw_fwd(x2d, w, bias, M=M if M is not None else x2d.shape[0], K=K, Nc=N,
                              out_dtype=torch.float32, relu=relu, gather=gather), False
        return ops.pw_fwd(x2d, w, bias, M=M if M is not None else x2d.shape[0], K=K, Nc=N,
                          out_dtype=torch.float32, relu=relu, gather=gather)

    def _pw_bwd(self, x2d, dy2d, name, need_dx=True, gather=None):
        w = self.P(name)
        K, N = w.shape
        M = dy2d.shape[0]
        if self.mixed:
            if self.gemm_operands is not None:
                self.gemm_operands[("bwd", w.data_ptr())] = dy2d.cpu().numpy()
            ops.pw_wgrad_bf16(x2d, dy2d, self.G64(name), M=M, gather=gather)
            if not need_dx:
                return None
            return ops.pw_bf16_train(dy2d, self._bf16_kernel(w, False), N)
        g = gather or (0, 0, 0, 0, 0, 1)
        check(lib().x3d_pw_wgrad(x2d.data_ptr(), dy2d.data_ptr(), self.G64(name).data_ptr(), M, K, N,
                                 x2d.shape[-1], N, int(gather is not None), g[1], g[2], g[3], g[4], g[5],
                                 _s()), "x3d_pw_wgrad")
        if not need_dx:
            return None
        if self.gemm == "tcgen05":
            return ops.pw_tf32(dy2d, w, None, transpose_w=False, M=M)       # dx = dy . w^T, w read as stored
        return ops.pw_fwd(dy2d, w.t().contiguous(), None, M=M, K=N, Nc=K, out_dtype=torch.float32)

    def _bias_grad(self, dy2d, name):
        M, C = dy2d.shape
        check(lib().x3d_colreduce(dy2d.data_ptr(), None, None, None, None, M, C, M,
                                  self.G64(name).data_ptr(), 2, _s()), "x3d_colreduce")

    def _stat_slot(self, C: int) -> torch.Tensor:
        """A zeroed fp64 [2, C] slice of the per-step statistics arena (one memset per step instead of
        one fill kernel per BatchNorm)."""
        n = 2 * C
        if self._stat_used + n > self._stat_arena.numel():
            return torch.zeros((2, C), dtype=torch.float64, device=self.device)
        t = self._stat_arena[self._stat_used:self._stat_used + n].view(2, C)
        self._stat_used += n
        return t

    def _bn_fwd(self, x2d, prefix, relu, tape, sums=None):
        """`sums`: the batch statistics if the producing GEMM's epilogue already accumulated them."""
        M, C = x2d.shape
        if sums is None:
            sums = self._stat_slot(C)
            check(lib().x3d_colreduce(x2d.data_ptr(), None, None, None, None, M, C, M, sums.data_ptr(), 0, _s()),
                  "x3d_colreduce")
        mean, var, rstd = (torch.empty(C, dtype=torch.float32, device=x2d.device) for _ in range(3))
        check(lib().x3d_bn_finalize(sums.data_ptr(), M, C, self.eps, self.bn_momentum, mean.data_ptr(),
                                    var.data_ptr(), rstd.data_ptr(),
                                    self.moving[prefix + "/moving_mean"].data_ptr(),
                                    self.moving[prefix + "/moving_variance"].data_ptr(), _s()), "x3d_bn_finalize")
        y = torch.empty_like(x2d)
        check(lib().x3d_bn_apply_fwd(x2d.data_ptr(), mean.data_ptr(), rstd.data_ptr(),
                                     self.P(prefix + "/gamma").data_ptr(), self.P(prefix + "/beta").data_ptr(),
                                     y.data_ptr(), M, C, int(relu), _s()), "x3d_bn_apply_fwd")

        def bwd(dy):
            off = self.layout.slots[prefix + "/beta"][0]            # [dbeta | dgamma] adjacent
            sums_g = self.g64[off:off + 2 * C]
            check(lib().x3d_colreduce(dy.data_ptr(), x2d.data_ptr(), mean.data_ptr(), rstd.data_ptr(),
                                      y.data_ptr() if relu else None, M, C, M, sums_g.data_ptr(), 1, _s()),
                  "x3d_colreduce")
            dx = torch.empty_like(x2d)
            check(lib().x3d_bn_bwd_apply(dy.data_ptr(), x2d.data_ptr(), y.data_ptr() if relu else None,
                                         mean.data_ptr(), rstd.data_ptr(), self.P(prefix + "/gamma").data_ptr(),
                                         sums_g.data_ptr(), dx.data_ptr(), M, C, _s()), "x3d_bn_bwd_apply")
            return dx
        tape.append(bwd)
        if relu and self.relu_masks is not None:
            self.relu_masks.append((y > 0).cpu().numpy())
        return y

    def _ew(self, a, b, op):
        out = torch.empty_like(a)
        check(lib().x3d_ew(a.data_ptr(), None if b is None else b.data_ptr(), out.data_ptr(), a.numel(), op, _s()),
              "x3d_ew")
        return out

    # ------------------------------------------------------------------ the step
    def forward_training(self, clips: torch.Tensor) -> torch.Tensor:
        """`model(clips, training=True)` of the reference (model.py:113-127 in training mode): batch-
        statistics BatchNorm (moving statistics are updated, as Keras does), dropout, no view
        averaging.  Returns the fc2 logits [N, classes]; no gradients are computed."""
        return self.forward_backward(clips, None, backward=False)

    def forward_backward(self, clips: torch.Tensor, labels: Optional[torch.Tensor], backward: bool = True):
        """clips [N,T,H,W,3] fp32 on the device, labels [N] int32.  Leaves data-loss gradients
        (scaled by 1/world) in self.g64 and returns the per-clip losses."""
        ar, L = self.arch, lib()
        x = clips.contiguous()
        N, T, H, W, _ = x.shape
        self.g64.zero_()
        self._wb.clear()
        self._stat_arena.zero_()
        self._stat_used = 0
        tape: List = []                       # backward closures, each maps dy -> dx of its op

        # ---- stem (model.py:202-208)
        cs = _pad8(ar.stem_channels)
        Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
        s_out = torch.empty((N, T, Ho, Wo, cs), dtype=torch.float32, device=x.device)
        check(L.x3d_stem_convs_fwd(x.data_ptr(), self.P("conv1/conv_s/kernel").data_ptr(), s_out.data_ptr(),
                                   N, T, H, W, cs, _s()), "x3d_stem_convs_fwd")
        t_out = torch.empty_like(s_out)
        kt = ar.temp_filter
        check(L.x3d_tconv_fwd(s_out.data_ptr(), self.P("conv1/conv_t/kernel").data_ptr(), t_out.data_ptr(),
                              N, T, Ho * Wo, cs, kt, 0, _s()), "x3d_tconv_fwd")

        def stem_bwd(dy):
            check(L.x3d_tconv_wgrad(s_out.data_ptr(), dy.data_ptr(), self.G64("conv1/conv_t/kernel").data_ptr(),
                                    N, T, Ho * Wo, cs, kt, _s()), "x3d_tconv_wgrad")
            ds = torch.empty_like(s_out)
            check(L.x3d_tconv_fwd(dy.data_ptr(), self.P("conv1/conv_t/kernel").data_ptr(), ds.data_ptr(),
                                  N, T, Ho * Wo, cs, kt, 1, _s()), "x3d_tconv_fwd")
            check(L.x3d_stem_convs_wgrad(x.data_ptr(), ds.data_ptr(), self.G64("conv1/conv_s/kernel").data_ptr(),
                                         N, T, H, W, cs, _s()), "x3d_stem_convs_wgrad")
            return None
        tape.append(stem_bwd)
        act = self._bn_fwd(t_out.view(-1, cs), "conv1/bn", True, tape).view(N, T, Ho, Wo, cs)

        # ---- residual stages (model.py:384-394, 305-320)
        for b in ar.blocks:
            if self.world > 1 and self._exchange_in_backward and b.index == 0 and b.stage in self._bucket_of_stage:
                # replayed AFTER every backward closure of this stage and of everything behind it: the
                # gradients of the bucket that starts at this stage are complete -> start its all-reduce
                tape.append(lambda d, k=self._bucket_of_stage[b.stage]: self._bucket_ready(k, d))
            act = self._block(act, b, tape)

        # ---- head (model.py:117-122)
        Nn, Tt, Hh, Ww, cl = act.shape
        P5 = Tt * Hh * Ww
        x5 = act.view(-1, cl)
        st5 = self._stat_slot(_pad8(ar.conv5_channels))
        y5, ok5 = self._pw(x5, self.P("conv5/layer_with_weights-0/kernel"), stats=st5)
        tape.append(lambda dy, x5=x5: self._pw_bwd(x5, dy, "conv5/layer_with_weights-0/kernel"))
        a5 = self._bn_fwd(y5, "conv5/layer_with_weights-1", True, tape, sums=st5 if ok5 else None)
        c5 = a5.shape[1]
        pool = ops.avgpool_fwd(a5.view(Nn, P5, c5))

        def pool_bwd(dm):
            dy = torch.empty_like(a5)
            check(L.x3d_pool_bwd(dm.data_ptr(), dy.data_ptr(), a5.shape[0], c5, P5, 1.0 / P5, 0, _s()), "x3d_pool_bwd")
            return dy
        tape.append(pool_bwd)
        h1 = self._pw(pool, self.P("fc1/kernel"), relu=True)
        if self.relu_masks is not None:
            self.relu_masks.append((h1 > 0).cpu().numpy())

        def fc1_bwd(dh):
            d = self._ew(dh, h1, 1)
            return self._pw_bwd(pool, d, "fc1/kernel")
        tape.append(fc1_bwd)
        if self.dropout > 0.0:
            if self.fixed_dropout_mask is not None:
                mask = self.fixed_dropout_mask
            else:
                mask = torch.empty_like(h1)
                check(L.x3d_dropout_mask(mask.data_ptr(), mask.numel(), self.dropout,
                                         self._dropout_seed(), _s()), "x3d_dropout_mask")
            hd = self._ew(h1, mask, 5)
            tape.append(lambda d, mask=mask: self._ew(d, mask, 5))
        else:
            hd = h1
        logits = self._pw(hd, self.P("fc2/kernel"), bias=self.P("fc2/bias"))

        def fc2_bwd(dl):
            self._bias_grad(dl, "fc2/bias")
            return self._pw_bwd(hd, dl, "fc2/kernel")
        tape.append(fc2_bwd)
        self.last_logits = logits
        if not backward:
            return logits
        loss = torch.empty(Nn, dtype=torch.float32, device=x.device)
        dlogits = torch.empty_like(logits)
        check(L.x3d_softmax_xent(logits.data_ptr(), labels.data_ptr(), loss.data_ptr(), dlogits.data_ptr(), Nn,
                                 logits.shape[1], 1.0 / (Nn * self.world), _s()), "x3d_softmax_xent")
        # ---- backward: replay the tape
        d = dlogits
        for fn in reversed(tape):
            d = fn(d)
        return loss

    def _block(self, x, b, tape):
        L = lib()
        N, T, H, W, cin = x.shape
        p = f"stages/{b.stage}/stage/layer_with_weights-{b.index}"
        q = p + "/bottleneck"
        s = b.stride
        ci, co = _pad8(b.cinner), _pad8(b.cout)
        Ho, Wo = -(-H // s), -(-W // s)
        _, ph, _ = A.same_pad(H, 3, s)
        _, pw_, _ = A.same_pad(W, 3, s)
        x2 = x.view(-1, cin)
        Pout = T * Ho * Wo
        st: dict = {}                                   # gradient w.r.t. the block input accumulates here

        # The tape is replayed in reverse, so the closures are appended in forward order:
        # [split] -> shortcut branch ... -> main branch ... -> [join]
        def split_bwd(dx_main):                         # runs LAST for this block: sum of both paths
            if b.has_shortcut:
                dxs = st["d_short"]                     # [N*T*Ho*Wo, cin] at the sampled pixels
                if s == 1:
                    return self._ew(dx_main, dxs, 4).view(N, T, H, W, cin)
                dx = dx_main.contiguous()
                check(L.x3d_strided_add(dxs.data_ptr(), dx.data_ptr(), N * T, Ho, Wo, H, W, s, cin, _s()),
                      "x3d_strided_add")
                return dx.view(N, T, H, W, cin)
            return self._ew(dx_main, st["d_short"], 4).view(N, T, H, W, cin)
        tape.append(split_bwd)

        # ---- main branch: a -> bn_a -> relu
        st_a = self._stat_slot(ci)                       # bn_a's batch statistics come out of the GEMM epilogue
        a_pre, ok_a = self._pw(x2, self.P(q + "/a/kernel"), stats=st_a)
        tape.append(lambda dy: self._pw_bwd(x2, dy, q + "/a/kernel"))
        a_out = self._bn_fwd(a_pre, q + "/bn_a", True, tape, sums=st_a if ok_a else None).view(N, T, H, W, ci)
        # ---- b (channelwise 3x3x3, SAME) -> bn_b
        wb = self.P(q + "/b/kernel")
        zero_b = torch.zeros(ci, dtype=torch.float32, device=x.device)
        b_pre, _ = ops.dw_fwd(a_out, wb, zero_b, s, ph, pw_, False)

        def dw_bwd(dy):
            dy5 = dy.view(N, T, Ho, Wo, ci)
            check(L.x3d_dw_wgrad(a_out.data_ptr(), dy5.data_ptr(), self.G64(q + "/b/kernel").data_ptr(), N, T, H, W,
                                 ci, s, ph, pw_, _s()), "x3d_dw_wgrad")
            return channelwise_dgrad(dy5, wb, zero_b, H, W, s, ph, pw_).view(-1, ci)
        tape.append(dw_bwd)
        b_out = self._bn_fwd(b_pre.view(-1, ci), q + "/bn_b", False, tape)
        # ---- SE (model.py:311-315) + swish (:316)
        scale = None
        if b.se_width:
            # se_pool: per-clip column sums over the whole [T*Ho*Wo, ci] activation (fp64 atomics,
            # thousands of CTAs; the head's avgpool kernel has one CTA per clip and 64 channels)
            m64 = torch.zeros((N, 2, ci), dtype=torch.float64, device=x.device)
            check(L.x3d_colreduce(b_out.data_ptr(), None, None, None, None, b_out.shape[0], ci, Pout,
                                  m64.data_ptr(), 2, _s()), "x3d_colreduce")
            m2 = torch.empty((N, 2, ci), dtype=torch.float32, device=x.device)
            check(L.x3d_d2f(m64.data_ptr(), m2.data_ptr(), m2.numel(), 1.0 / Pout, _s()), "x3d_d2f")
            m = m2[:, 0, :].contiguous()
            z = self._pw(m, self.P(q + "/se_fc1/kernel"), bias=self.P(q + "/se_fc1/bias"), relu=True)
            s_pre = self._pw(z, self.P(q + "/se_fc2/kernel"), bias=self.P(q + "/se_fc2/bias"))
            scale = self._ew(s_pre, None, 2)
        sw = torch.empty_like(b_out)
        check(L.x3d_scale_swish_fwd(b_out.data_ptr(), None if scale is None else scale.data_ptr(), sw.data_ptr(),
                                    b_out.shape[0], ci, Pout, _s()), "x3d_scale_swish_fwd")

        def se_swish_bwd(dout):
            dy = torch.empty_like(b_out)
            ds64 = None
            if scale is not None:
                ds64 = torch.zeros((N, ci), dtype=torch.float64, device=x.device)
            check(L.x3d_scale_swish_bwd(dout.data_ptr(), b_out.data_ptr(),
                                        None if scale is None else scale.data_ptr(), dy.data_ptr(),
                                        None if ds64 is None else ds64.data_ptr(), b_out.shape[0], ci, Pout, _s()),
                  "x3d_scale_swish_bwd")
            if scale is not None:
                ds = torch.empty((N, ci), dtype=torch.float32, device=x.device)
                check(L.x3d_d2f(ds64.data_ptr(), ds.data_ptr(), ds.numel(), 1.0, _s()), "x3d_d2f")
                dpre2 = self._ew(ds, scale, 3)                              # sigmoid'
                self._bias_grad(dpre2, q + "/se_fc2/bias")
                dz = self._pw_bwd(z, dpre2, q + "/se_fc2/kernel")
                dpre1 = self._ew(dz, z, 1)                                  # relu'
                self._bias_grad(dpre1, q + "/se_fc1/bias")
                dm = self._pw_bwd(m, dpre1, q + "/se_fc1/kernel")
                check(L.x3d_pool_bwd(dm.data_ptr(), dy.data_ptr(), b_out.shape[0], ci, Pout, 1.0 / Pout, 1, _s()),
                      "x3d_pool_bwd")
            return dy
        tape.append(se_swish_bwd)
        # ---- c -> bn_c
        st_c = self._stat_slot(co)
        c_pre, ok_c = self._pw(sw, self.P(q + "/c/kernel"), stats=st_c)
        tape.append(lambda dy: self._pw_bwd(sw, dy, q + "/c/kernel"))
        c_out = self._bn_fwd(c_pre, q + "/bn_c", False, tape, sums=st_c if ok_c else None)
        # ---- shortcut (model.py:386-389) and add + relu (:389-392)
        if b.has_shortcut:
            gather = (T, Ho, Wo, H, W, s)
            r_pre = self._pw(x2, self.P(p + "/residual/kernel"), gather=gather, M=N * Pout)
            short_tape: List = []
            res = self._bn_fwd(r_pre, p + "/bn_r", False, short_tape)
        else:
            res = x2
        out = self._ew(c_out, res, 0)
        if self.relu_masks is not None:
            self.relu_masks.append((out > 0).cpu().numpy())

        def join_bwd(dout):                              # runs FIRST for this block
            d = self._ew(dout.reshape(-1, co), out, 1)   # relu'
            if b.has_shortcut:
                dr = short_tape[0](d)
                st["d_short"] = self._pw_bwd(x2, dr, p + "/residual/kernel", gather=(T, Ho, Wo, H, W, s))
            else:
                st["d_short"] = d
            return d                                     # continues into bn_c
        tape.append(join_bwd)
        return out.view(N, T, Ho, Wo, co)

    def _bucket_ready(self, k: int, d):
        """Backward has finished bucket k of the gradient arena: fp64 accumulators -> fp32 arena for that
        range, then its all-reduce starts while the backward pass continues (exchange.py)."""
        lo, hi = self.exchange.buckets[k]
        check(lib().x3d_d2f(self.g64[lo:hi].data_ptr(), self.g[lo:hi].data_ptr(), hi - lo, 1.0, _s()), "x3d_d2f")
        self.exchange.start(k)
        self._converted.append((lo, hi))
        return d

    def _dropout_seed(self) -> int:
        """64-bit seed of this step's dropout stream: a hash of (seed, rank, iteration), so every
        data-parallel replica draws its own mask (per-replica RNG under MirroredStrategy) and the
        iteration counter never runs into the seed bits."""
        return _mix64(_mix64(_mix64(self.seed) + self.rank) + self.iteration)

    def step(self, clips: torch.Tensor, labels: torch.Tensor, lr: float) -> torch.Tensor:
        """forward + backward + gradient all-reduce + SGD-Nesterov update.  Returns per-clip losses."""
        self._converted = []
        self._exchange_in_backward = True       # only step() communicates; forward_backward alone never does
        try:
            loss = self.forward_backward(clips, labels)
        finally:
            self._exchange_in_backward = False
        n = self.layout.size
        if self.world > 1:
            # buckets whose all-reduce already runs behind the backward pass are done; the rest (the
            # stem and the first stages, < 3 % of the bytes) is converted and exchanged now
            for k, (lo, hi) in enumerate(self.exchange.buckets):
                if (lo, hi) not in self._converted:
                    self._bucket_ready(k, None)
            self.exchange.finish()
        else:
            check(lib().x3d_d2f(self.g64.data_ptr(), self.g.data_ptr(), n, 1.0, _s()), "x3d_d2f")
        if self.optimizer == "adam":
            b1, b2, eps = self.adam
            t = self.iteration + 1
            lr_t = float(lr) * (1.0 - b2 ** t) ** 0.5 / (1.0 - b1 ** t)
            check(lib().x3d_adam_step(self.w.data_ptr(), self.g.data_ptr(), self.v.data_ptr(), self.v2.data_ptr(),
                                      self.wd.data_ptr(), n, lr_t, b1, b2, eps, _s()), "x3d_adam_step")
        else:
            check(lib().x3d_sgd_nesterov_step(self.w.data_ptr(), self.g.data_ptr(), self.v.data_ptr(),
                                              self.wd.data_ptr(), n, float(lr), self.momentum, _s()),
                  "x3d_sgd_nesterov_step")
        self.iteration += 1
        return loss


def lr_schedule(cfg, epoch: int) -> float:
    """train.py:114-125: linear warm-up WARMUP_LR -> BASE_LR, then half-cosine per epoch."""
    import math
    t = cfg.TRAIN
    if epoch > t.WARMUP_EPOCHS:
        return float(t.BASE_LR) * 0.5 * (math.cos(math.pi * epoch / t.EPOCHS) + 1.0)
    return float(t.WARMUP_LR) + epoch * (float(t.BASE_LR) - float(t.WARMUP_LR)) / max(int(t.WARMUP_EPOCHS), 1)
