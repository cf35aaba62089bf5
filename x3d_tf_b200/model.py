"""X3D model and blocks with the reference's Keras class API, executed by sm_100a CUDA kernels.

Drop-in surface (reference `model.py`): `X3D(cfg)`, `X3D_Stem`, `Bottleneck`, `ResBlock`,
`ResStage`, `AdaptiveAvgPool3D` -- same constructor arguments, `call(input, training=False)`,
`model.stages[i]._inner_channels`, `load_weights(prefix).expect_partial()`, `summary()`, and the
TF-checkpoint variable names (`conv1/conv_s/kernel`, `stages/0/stage/layer_with_weights-0/
bottleneck/a/kernel`, ...).  Inputs are channels-last NDHWC clips.

Everything numeric runs in the C-ABI library (`include/x3d_b200.h`); this file only holds the
weights (numpy, TF layouts), folds the inference BatchNorm into them, and sequences launches.
There is no CPU / PyTorch fallback: without the CUDA library or a GPU, `call` raises.
"""
from __future__ import annotations

import os

import math
from collections import OrderedDict
from typing import Dict, Iterable, List, Optional, Tuple

import numpy as np
import torch

from . import arch as A
from . import ops
from . import tf_bundle
from .video import VideoBatch

_BN_LEAVES = ("gamma", "beta", "moving_mean", "moving_variance")


def _pad8(c: int) -> int:
    return (c + 7) // 8 * 8


def _glorot(rng, shape, fan_in, fan_out):
    lim = math.sqrt(6.0 / (fan_in + fan_out))
    return rng.uniform(-lim, lim, size=shape).astype(np.float32)


class _LoadStatus:
    """What `tf.keras.Model.load_weights` returns for TF-format checkpoints (eval.py:81)."""

    def __init__(self, missing, unused):
        self.missing, self.unused = list(missing), list(unused)

    def expect_partial(self):
        return self

    def assert_consumed(self):
        if self.missing or self.unused:
            raise AssertionError(f"unresolved: missing={self.missing[:3]} unused={self.unused[:3]}")
        return self

    def assert_existing_objects_matched(self):
        if self.missing:
            raise AssertionError(f"variables without a checkpoint value: {self.missing[:3]}")
        return self


class Layer:
    """Minimal stand-in for `tf.keras.layers.Layer`: named variables (numpy, TF layout), child
    layers, `__call__(x, training=False)`.  Variables are created at construction with the
    Keras default initialisers (Glorot-uniform kernels, zeros biases, BN gamma=1/beta=0/mean=0/
    var=1), so a freshly built layer is usable like in the reference."""

    _init_seed = 0

    def __init__(self, name: Optional[str] = None):
        self.name = name or type(self).__name__.lower()
        self._vars: "OrderedDict[str, np.ndarray]" = OrderedDict()
        self._children: "OrderedDict[str, Layer]" = OrderedDict()
        self._dev: Dict[tuple, dict] = {}

    # ---- variables
    def _rng(self):
        Layer._init_seed += 1
        return np.random.default_rng(Layer._init_seed)

    def _add_conv(self, key: str, shape: Tuple[int, ...], groups: int = 1):
        # Keras `_compute_fans`: receptive field x shape[-2] / x shape[-1] of the KERNEL tensor, so a
        # channelwise (3,3,3,1,C) kernel has fan_in = 27 and fan_out = 27*C (groups play no part)
        rf = int(np.prod(shape[:-2]))
        fan_in, fan_out = rf * shape[-2], rf * shape[-1]
        self._vars[key] = _glorot(self._rng(), shape, fan_in, fan_out)

    def _add_bn(self, key: str, c: int):
        self._vars[f"{key}/gamma"] = np.ones(c, np.float32)
        self._vars[f"{key}/beta"] = np.zeros(c, np.float32)
        self._vars[f"{key}/moving_mean"] = np.zeros(c, np.float32)
        self._vars[f"{key}/moving_variance"] = np.ones(c, np.float32)

    def _child(self, key: str, layer: "Layer") -> "Layer":
        self._children[key] = layer
        return layer

    def named_variables(self, prefix: str = "") -> "OrderedDict[str, np.ndarray]":
        out: "OrderedDict[str, np.ndarray]" = OrderedDict()
        for k, v in self._vars.items():
            out[prefix + k] = v
        for ck, ch in self._children.items():
            out.update(ch.named_variables(f"{prefix}{ck}/"))
        return out

    def set_weights_dict(self, weights: Dict[str, np.ndarray], prefix: str = "",
                         strict: bool = True) -> List[str]:
        """Assign variables by (prefixed) checkpoint name.  Returns names that had no value."""
        missing = []
        for k in list(self._vars):
            full = prefix + k
            if full in weights:
                w = np.asarray(weights[full], dtype=np.float32)
                if w.shape != self._vars[k].shape:
                    raise ValueError(f"{full}: shape {w.shape} != expected {self._vars[k].shape}")
                self._vars[k] = np.ascontiguousarray(w)
            else:
                missing.append(full)
        for ck, ch in self._children.items():
            missing += ch.set_weights_dict(weights, f"{prefix}{ck}/", strict=False)
        self._invalidate()
        if strict and missing:
            raise KeyError(f"no value for {len(missing)} variables, e.g. {missing[:3]}")
        return missing

    def count_params(self) -> int:
        return sum(int(v.size) for v in self.named_variables().values())

    def _invalidate(self):
        self._dev.clear()
        for ch in self._children.values():
            ch._invalidate()

    # ---- execution
    def __call__(self, x, training: bool = False):
        return self.call(x, training=training)

    def call(self, x, training: bool = False):
        raise NotImplementedError

    @staticmethod
    def _no_training(training: bool):
        if training:
            raise NotImplementedError(
                "training=True on a stand-alone block: the training kernels (batch-statistics BatchNorm, "
                "dropout, backward) run on the whole model's flat parameter arena -- use "
                "X3D.call(x, training=True) / X3D.fit(...) (training.X3DTrainer), see INTEGRATION.md")

    def _fold_bn(self, key: str, eps: float) -> Tuple[np.ndarray, np.ndarray]:
        g = self._vars[f"{key}/gamma"].astype(np.float64)
        b = self._vars[f"{key}/beta"].astype(np.float64)
        m = self._vars[f"{key}/moving_mean"].astype(np.float64)
        v = self._vars[f"{key}/moving_variance"].astype(np.float64)
        s = g / np.sqrt(v + eps)
        return s, b - m * s


def _dev_f32(a: np.ndarray, device) -> torch.Tensor:
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(device)


def _pad_to(a: np.ndarray, axis: int, size: int) -> np.ndarray:
    if a.shape[axis] == size:
        return a
    pad = [(0, 0)] * a.ndim
    pad[axis] = (0, size - a.shape[axis])
    return np.pad(a, pad)


def _as_device_clip(x, device) -> torch.Tensor:
    if isinstance(x, np.ndarray):
        x = torch.from_numpy(np.ascontiguousarray(x))
    if not isinstance(x, torch.Tensor):
        raise TypeError("input must be a torch.Tensor or numpy array in NDHWC layout")
    if x.dim() != 5:
        raise ValueError(f"expected a 5-D NDHWC tensor, got shape {tuple(x.shape)}")
    if x.dtype == torch.float16:
        # the reference's mixed_float16 input cast (dataloader.py:118-120): this build's 16-bit policy is
        # bfloat16 (runtime.py); fp16 clips enter as bf16 (normalised pixels are within +-4: no range issue)
        x = x.to(torch.bfloat16)
    elif x.dtype == torch.float64:
        x = x.to(torch.float32)
    if x.dtype not in (torch.float32, torch.bfloat16, torch.uint8):
        raise TypeError(f"unsupported input dtype {x.dtype}")
    if not x.is_cuda:
        if device is None:
            if not torch.cuda.is_available():
                raise RuntimeError("no CUDA device: the X3D path has no CPU implementation")
            device = torch.device("cuda", torch.cuda.current_device())
        x = x.to(device, non_blocking=True)
    return x.contiguous()


def _pad_channels(x: torch.Tensor, cs: int) -> torch.Tensor:
    c = x.shape[-1]
    if c == cs:
        return x
    out = torch.zeros(x.shape[:-1] + (cs,), dtype=x.dtype, device=x.device)
    out[..., :c] = x
    return out


class PointwiseConv:
    """Device-side state of one 1x1x1 conv (+ folded BN): fp32 [K,N] weights for the SIMT kernel
    and packed bf16 [Npad,Kpad] weights for the tcgen05 kernel."""

    def __init__(self, kernel: np.ndarray, scale, shift, device, bias=None):
        k2 = kernel.reshape(kernel.shape[-2], kernel.shape[-1]).astype(np.float64)
        K, N = k2.shape
        self.K, self.N, self.Ks, self.Ns = K, N, _pad8(K), _pad8(N)
        if scale is not None:
            k2 = k2 * scale[None, :]
        b = np.zeros(N, np.float64) if shift is None else np.asarray(shift, np.float64)
        if bias is not None:
            b = b + np.asarray(bias, np.float64)
        wt = _pad_to(_pad_to(k2, 0, self.Ks), 1, self.Ns)
        self.wt = _dev_f32(wt, device)
        self.bias = _dev_f32(_pad_to(b, 0, self.Ns), device)
        npad, kpad = (self.Ns + 15) // 16 * 16, (self.Ks + 63) // 64 * 64
        wp = _pad_to(_pad_to(k2.T, 0, npad), 1, kpad)
        self.wp = torch.from_numpy(np.ascontiguousarray(wp, dtype=np.float32)).to(device).to(
            torch.bfloat16).contiguous()
        self._k2t = _pad_to(_pad_to(k2.T, 0, self.Ns), 1, self.Ks)               # [Ns, Ks], fp64
        self._paired: Dict[int, Tuple[torch.Tensor, torch.Tensor]] = {}
        self._stacked: Dict[int, tuple] = {}

    # Pixel pairing (Options.pair_pixels): rows of 24 or 56 bf16 channels are 48 / 112 bytes and straddle
    # 32-byte sectors, so TMA moves 1.33x / 1.14x the useful bytes between L2 and shared memory, and a
    # 128-row tile of them is small against the per-tile cost of the GEMM pipeline.  P consecutive
    # pixels form one row (the activation is contiguous, so this is only a different view) and the
    # weight becomes blockdiag(W, ..., W): [M/P, P*K] x [P*K, P*N].  The extra MMA work is on exact
    # zeros and the tensor pipe is far from busy.  The products of a pixel are grouped into K=16 MMA
    # steps differently than in the unpaired GEMM, so results agree to fp32-accumulation rounding
    # (at most one bf16 ulp after the output rounding), not bit for bit; pairs never straddle clips
    # (rows_per_clip % P == 0), which keeps a clip's result independent of its position in the batch.
    def _pair_factor(self, M: int, rows_per_clip: int = 0) -> int:
        for P in (4, 2):
            if P > Options.pair_pixels or M % P or (rows_per_clip and rows_per_clip % P):
                continue
            if P * self.Ks > Options.pair_max_k or P * self.Ns > Options.pair_max_n:
                continue
            if not Options.pair_aligned and self.Ks % 16 == 0 and self.Ns % 16 == 0:
                continue
            return P
        return 1

    def _paired_weights(self, P: int, device) -> Tuple[torch.Tensor, torch.Tensor]:
        if P not in self._paired:
            w = np.zeros((P * self.Ns, P * self.Ks), np.float64)
            for i in range(P):
                w[i * self.Ns:(i + 1) * self.Ns, i * self.Ks:(i + 1) * self.Ks] = self._k2t
            npad, kpad = (P * self.Ns + 15) // 16 * 16, (P * self.Ks + 63) // 64 * 64
            w = _pad_to(_pad_to(w, 0, npad), 1, kpad)
            wp = torch.from_numpy(np.ascontiguousarray(w, dtype=np.float32)).to(device).to(
                torch.bfloat16).contiguous()
            self._paired[P] = (wp, self.bias.repeat(P).contiguous())
        return self._paired[P]

    def _stacked_weights(self, other: "PointwiseConv", device) -> Tuple[torch.Tensor, torch.Tensor]:
        """Packed weight of  self(a) + other(a2)  as ONE GEMM over [a | a2]: other's K rows start at the
        packed column 64*ceil(Ks/64) (x3d_pw_tc_fwd's second source); the two BN shifts add up."""
        key = id(other)
        if key not in self._stacked:
            if other.Ns != self.Ns:
                raise ValueError("stacked pointwise convs need the same output width")
            k1, k2 = (self.Ks + 63) // 64 * 64, (other.Ks + 63) // 64 * 64
            w = np.zeros(((self.Ns + 15) // 16 * 16, k1 + k2), np.float64)
            w[:self.Ns, :self.Ks] = self._k2t
            w[:self.Ns, k1:k1 + other.Ks] = other._k2t
            wp = torch.from_numpy(np.ascontiguousarray(w, dtype=np.float32)).to(device).to(
                torch.bfloat16).contiguous()
            self._stacked[key] = (wp, (self.bias + other.bias).contiguous(), other)
        return self._stacked[key][:2]

    def run_with_shortcut(self, a: torch.Tensor, M: int, shortcut: "PointwiseConv", x: torch.Tensor,
                          stride: int, *, se=None, rows_per_clip=0, swish=False, relu=False) -> torch.Tensor:
        """act(self(pro(a)) + shortcut(x sampled with `stride`)): ResBlock's add with the shortcut conv as
        extra K columns of the projection GEMM (reference model.py:386-392)."""
        wp, bias = self._stacked_weights(shortcut, a.device)
        return ops.pw_tc_fwd(a, wp, bias, M=M, K=self.Ks, Nc=self.Ns, se=se, rows_per_clip=rows_per_clip,
                             swish=swish, relu=relu, a2=x, a2_stride=stride)

    def run(self, a: torch.Tensor, M: int, *, use_tc: bool, out_dtype=None, residual=None,
            se=None, rows_per_clip=0, swish=False, relu=False, gather=None, pair_rows=0) -> torch.Tensor:
        if use_tc and a.dtype == torch.bfloat16 and gather is None and \
                (out_dtype is None or out_dtype == torch.bfloat16):
            # (not with an SE scale: that prologue indexes the scale by column, and pairing measured no
            # gain on the projection GEMMs anyway)
            P = self._pair_factor(M, pair_rows or rows_per_clip) if se is None else 1
            if P > 1 and a.is_contiguous() and (residual is None or residual.is_contiguous()):
                wp, bias = self._paired_weights(P, a.device)
                return ops.pw_tc_fwd(a, wp, bias, M=M // P, K=P * self.Ks, Nc=P * self.Ns, residual=residual,
                                     swish=swish, relu=relu).view(M, self.Ns)
            return ops.pw_tc_fwd(a, self.wp, self.bias, M=M, K=self.Ks, Nc=self.Ns,
                                 residual=residual, se=se, rows_per_clip=rows_per_clip,
                                 swish=swish, relu=relu)
        return ops.pw_fwd(a, self.wt, self.bias, M=M, K=self.Ks, Nc=self.Ns, out_dtype=out_dtype,
                          residual=residual, se=se, rows_per_clip=rows_per_clip, swish=swish,
                          relu=relu, gather=gather)


# Execution options shared by all layers of a process (the reference has no such switch; these
# only choose between equivalent CUDA kernels).
class Options:
    pointwise = "tc"          # "tc": tcgen05 kernel for bf16 activations; "simt": CUDA-core GEMM
    stem = "tc"               # "tc": tcgen05 implicit-GEMM stem for bf16 activations; "simt"
    # bf16 + "tc": run a/bn_a/relu/b/bn_b (+ swish) as ONE kernel, the persistent warp-specialised
    # x3d_expand_dw2_fwd (csrc/x3d_ab_persist.cu).  Parity-green on every layer shape, but NOT faster
    # than the two-kernel path on B200: at 80 clips of 16x256^2 the three stage-2 blocks take 2.56 ms
    # fused against 2.46 ms for the pair (with pixel pairing and the swish epilogue), all 26 blocks
    # 8.37 against 7.61 ms; step 10.95 ms off / 11.09 ms stage 2 only / 11.88 ms everywhere.  The
    # stencil half is bound by register-file bandwidth of the packed FFMA2 stream, not by the HBM
    # traffic fusion removes (profiles/r02_fused_expand_dw.md), so it stays opt-in:
    #   "off" (default); "auto": layers whose inner width fits one channel chunk (<= 72: stage 2);
    #   "all": every layer with a tile plan; "v1": the round-1 one-CTA-per-tile kernel.
    fuse_expand = os.environ.get("X3D_FUSE_EXPAND", "off")
    # uint8 clips in bf16 mode: "normalize" = x3d_normalize_u8 then the ordinary stem;
    # "fused" = x3d_stem_tc_u8_fwd (the stem's loader reads bytes through a lookup table)
    stem_u8 = os.environ.get("X3D_STEM_U8", "normalize")
    # blocks without SE: apply swish in the channelwise kernel's epilogue (x3d_dw3x3x3_act_fwd)
    # instead of the projection GEMM's prologue, which then runs without its transform warps.
    # Measured back to back at 80 clips of 16x256^2: c 2.83 -> 2.50 ms, b 4.97 -> 5.18 ms (the stencil
    # is the FMA/issue-bound kernel), step 11.91 -> 11.75 ms (+1.4 % clips/s); X3D_SWISH_IN_DW=0 turns
    # it off.
    swish_in_dw = os.environ.get("X3D_SWISH_IN_DW", "1") == "1"
    # bf16 + "tc": ResBlock's strided shortcut conv + bn_r as extra K columns of the projection GEMM
    # (x3d_pw_tc_fwd's second source: no gather kernel, no shortcut GEMM, no residual tensor) wherever
    # 128-pixel tiles align with the output frames (64/32/16/8-wide: every stage at 256^2).
    fold_shortcut = os.environ.get("X3D_FOLD_SHORTCUT", "1") == "1"
    # bf16 + "tc": conv_5's epilogue also produces the pooled means (no conv_5 output tensor, pool_5 reads
    # 1/64 of the rows) whenever a clip has a multiple of 64 positions at that point
    pool_in_conv5 = os.environ.get("X3D_POOL_IN_CONV5", "1") == "1"
    # channelwise 3x3x3 kernel for bf16 activations: "tma" = x3d_dw3x3x3_act_fwd (thread = channel pair,
    # csrc/x3d_dw_tma.cu) everywhere; "auto" = the planar kernel (lanes = pixels, taps in uniform
    # registers, csrc/x3d_dw_planar.cu) for the stride-1 layers that fill >= 85 % of its lane grid (all of
    # them at 256^2 -- 8x8 frames four clips at a time --, the 28/14-wide ones at 224^2), where it measures 5-13 % faster
    # (profiles/r02_dw_planar.md); "planar" = wherever it has a plan.
    channelwise = os.environ.get("X3D_CHANNELWISE", "auto")
    # pointwise convs whose rows are not a multiple of 32 bytes (24 / 56 channels): two pixels per GEMM
    # row with a block-diagonal weight (PointwiseConv).  Measured at 80 clips of 16x256^2 (step, a,
    # shortcut in ms): off 11.66 / 2.95 / 0.52; factor 2 10.97 / 2.47 / 0.37; factor 4 11.07; factor 2
    # also on sector-aligned rows (X3D_PAIR_ALIGNED=1) 11.23; pairing the 432-byte rows of stage 4 as
    # well (X3D_PAIR_MAX_N=512, two N tiles) 11.03 against 10.94.  X3D_PAIR_PIXELS=1 turns it off.
    pair_pixels = int(os.environ.get("X3D_PAIR_PIXELS", "2"))       # largest pairing factor (1 = off, 2, 4)
    pair_max_k = int(os.environ.get("X3D_PAIR_MAX_K", "256"))
    pair_max_n = int(os.environ.get("X3D_PAIR_MAX_N", "256"))
    pair_aligned = os.environ.get("X3D_PAIR_ALIGNED", "0") == "1"   # also pair rows that are sector-aligned


def _use_tc() -> bool:
    return Options.pointwise == "tc"


# ======================================================================================
class X3D_Stem(Layer):
    """Reference `model.py:134-210`."""

    def __init__(self, bn_cfg, regularizer=None, out_channels: int = 24,
                 temp_filter_size: int = 5, in_channels: int = 3):
        super().__init__(name="conv_1")
        self.bn_momentum, self.bn_eps = bn_cfg.MOMENTUM, bn_cfg.EPS
        self.out_channels, self.temp_filter_size = out_channels, temp_filter_size
        self._add_conv("conv_s/kernel", (1, 3, 3, in_channels, out_channels))
        self._add_conv("conv_t/kernel", (temp_filter_size, 1, 1, 1, out_channels),
                       groups=out_channels)
        self._add_bn("bn", out_channels)
        # uint8 clips are normalised on the device the way dataloader.py does on the host
        # (utils.normalize, utils.py:42-72); X3D sets this from cfg.DATA.MEAN / STD
        self.input_norm: Optional[Tuple[tuple, tuple]] = None

    def _prep(self, device):
        key = (str(device),)
        if key not in self._dev:
            C, cs = self.out_channels, _pad8(self.out_channels)
            s, t = self._fold_bn("bn", self.bn_eps)
            ws = self._vars["conv_s/kernel"].reshape(27, C).astype(np.float64)
            wt = self._vars["conv_t/kernel"].reshape(self.temp_filter_size, C).astype(np.float64) * s
            d = {"ws": _dev_f32(_pad_to(ws, 1, cs), device),
                 "wt": _dev_f32(_pad_to(wt, 1, cs), device),
                 "bias": _dev_f32(_pad_to(t, 0, cs), device)}
            if cs <= 32 and self.temp_filter_size == 5:
                # merged kt x3x3 kernel for the tensor-core stem: [dt][k/8][c][k%8], K and C padded to 32
                wc = np.zeros((self.temp_filter_size, 4, 32, 8), np.float64)
                full = ws[None, :, :] * wt[:, None, :]                    # [dt, 27, C]
                for k in range(27):
                    wc[:, k // 8, :C, k % 8] = full[:, k, :]
                d["wc"] = torch.from_numpy(wc.astype(np.float32)).to(device).to(
                    torch.bfloat16).contiguous()
            self._dev[key] = d
        return self._dev[key]

    def _forward(self, x: torch.Tensor, out_dtype) -> torch.Tensor:
        d = self._prep(x.device)
        ops.Profiler.tag = "stem"
        tc = out_dtype == torch.bfloat16 and "wc" in d and Options.stem == "tc"
        if x.dtype == torch.uint8:
            if self.input_norm is None:
                raise ValueError("uint8 clips need input_norm = (mean, std) (cfg.DATA.MEAN / cfg.DATA.STD)")
            mean, std = self.input_norm
            if tc and Options.stem_u8 == "fused":
                return ops.stem_tc_u8_fwd(x, mean, std, d["wc"], d["bias"])
            # default: one streaming pass (table lookup, ~0.15 ms for 80 clips of 16x256x256) and the
            # ordinary stem; measured faster than byte gathers inside the stem's im2col loader
            x = ops.normalize_u8(x, mean, std, out_dtype)
        if tc:
            return ops.stem_tc_fwd(x, d["wc"], d["bias"])
        return ops.stem_fwd(x, d["ws"], d["wt"], d["bias"], out_dtype)

    def call(self, input, training: bool = False):
        self._no_training(training)
        x = _as_device_clip(input, None)
        out_dtype = torch.float32 if x.dtype == torch.uint8 else x.dtype
        return self._forward(x, out_dtype)[..., :self.out_channels]


class AdaptiveAvgPool3D(Layer):
    """Reference `model.py:457-492` (only the global (1,1,1) case does anything there too)."""

    def __init__(self, spatial_out_shape=(1, 1, 1), data_format="channels_last", **kwargs):
        super().__init__(name=kwargs.get("name"))
        assert len(spatial_out_shape) == 3, "Please specify 3D shape"
        assert data_format in ("channels_last", "channels_first")
        self.data_format, self.out_shape = data_format, tuple(spatial_out_shape)

    def call(self, input, training: bool = False):
        x = _as_device_clip(input, None)
        if self.data_format == "channels_first":
            x = x.permute(0, 2, 3, 4, 1).contiguous()
        m = ops.avgpool_fwd(x)                                   # [N, C] fp32
        n, c = m.shape
        o = self.out_shape
        if self.data_format == "channels_last":
            return m.reshape(-1, o[0], o[1], o[2], c)
        return m.reshape(-1, c, o[0], o[1], o[2])


class Bottleneck(Layer):
    """Reference `model.py:212-320`."""

    def __init__(self, channels: tuple, bn_cfg, regularizer=None, stride: int = 1,
                 block_index: int = 0, se_ratio: float = 0.0625, temp_kernel_size: int = 3,
                 in_channels: Optional[int] = None):
        super().__init__()
        if temp_kernel_size != 3:
            raise NotImplementedError("only the 3x3x3 channelwise kernel is built")
        self.block_index, self._bn_cfg = block_index, bn_cfg
        self.inner, self.out_channels, self.stride = channels[0], channels[1], stride
        self.in_channels = in_channels        # Keras infers it at first call; see _ensure_built
        self.has_se = A.se_enabled(block_index)
        self.se_width = A.round_width(self.inner, se_ratio) if self.has_se else 0
        if in_channels is not None:
            self._build(in_channels)

    def _build(self, cin: int):
        self.in_channels = cin
        inner, cout = self.inner, self.out_channels
        v = OrderedDict()
        old, self._vars = self._vars, v
        self._add_conv("a/kernel", (1, 1, 1, cin, inner))
        self._add_bn("bn_a", inner)
        self._add_conv("b/kernel", (3, 3, 3, 1, inner), groups=inner)
        self._add_bn("bn_b", inner)
        if self.has_se:
            self._add_conv("se_fc1/kernel", (1, 1, 1, inner, self.se_width))
            self._vars["se_fc1/bias"] = np.zeros(self.se_width, np.float32)
            self._add_conv("se_fc2/kernel", (1, 1, 1, self.se_width, inner))
            self._vars["se_fc2/bias"] = np.zeros(inner, np.float32)
        self._add_conv("c/kernel", (1, 1, 1, inner, cout))
        self._add_bn("bn_c", cout)
        self._vars.update(old)

    def _prep(self, device):
        key = (str(device),)
        if key not in self._dev:
            eps = self._bn_cfg.EPS
            ci = _pad8(self.inner)
            sa, ta = self._fold_bn("bn_a", eps)
            sb, tb = self._fold_bn("bn_b", eps)
            sc, tc = self._fold_bn("bn_c", eps)
            d = {"a": PointwiseConv(self._vars["a/kernel"], sa, ta, device),
                 "c": PointwiseConv(self._vars["c/kernel"], sc, tc, device)}
            wb = self._vars["b/kernel"].reshape(27, self.inner).astype(np.float64) * sb
            d["wb"] = _dev_f32(_pad_to(wb, 1, ci), device)
            d["bb"] = _dev_f32(_pad_to(tb, 0, ci), device)
            d["wbp"] = ops.dw_planar_taps(d["wb"], d["bb"])
            if self.has_se:
                w1 = self._vars["se_fc1/kernel"].reshape(self.inner, self.se_width)
                w2 = self._vars["se_fc2/kernel"].reshape(self.se_width, self.inner)
                d["w1"] = _dev_f32(_pad_to(w1, 0, ci), device)
                d["b1"] = _dev_f32(self._vars["se_fc1/bias"], device)
                d["w2"] = _dev_f32(_pad_to(w2, 1, ci), device)
                d["b2"] = _dev_f32(_pad_to(self._vars["se_fc2/bias"], 0, ci), device)
            self._dev[key] = d
        return self._dev[key]

    def _forward(self, x: torch.Tensor, residual: Optional[torch.Tensor] = None,
                 relu: bool = False, shortcut: Optional[PointwiseConv] = None,
                 shortcut_rows: Optional[torch.Tensor] = None) -> torch.Tensor:
        """x: [N,T,H,W,pad8(cin)].  `residual`/`relu`: the ResBlock add + ReLU fused into c's epilogue;
        `shortcut`: ResBlock's strided conv + bn_r, run on x as extra K columns of c (then no `residual`)."""
        if self.in_channels is None:
            raise RuntimeError("Bottleneck used before its input width is known")
        d = self._prep(x.device)
        N, T, H, W, _ = x.shape
        ci = _pad8(self.inner)
        tc = _use_tc()
        _, ph, _ = A.same_pad(H, 3, self.stride)
        _, pw, _ = A.same_pad(W, 3, self.stride)
        mode = Options.fuse_expand
        fuse2 = tc and x.dtype == torch.bfloat16 and (mode == "all" or (mode == "auto" and ci <= 72)) and \
            ops.expand_dw2_supported(T, H, W, x.shape[-1], ci, self.stride) > 0
        if fuse2:
            ops.Profiler.tag = "ab"
            swish_in_b = Options.swish_in_dw and not self.has_se
            b, partial = ops.expand_dw2_fwd(x, d["a"].wp, d["a"].bias, d["wb"], d["bb"],
                                            self.stride, ph, pw, self.has_se, swish=swish_in_b)
        elif tc and mode == "v1" and x.dtype == torch.bfloat16 and \
                ops.expand_dw_supported(T, H, W, x.shape[-1], ci, self.stride) > 0:
            ops.Profiler.tag = "ab"
            b, partial = ops.expand_dw_fwd(x, d["a"].wp, d["a"].bias, d["wb"], d["bb"],
                                           self.stride, ph, pw, self.has_se)
            swish_in_b = False
        else:
            ops.Profiler.tag = "a"
            a = d["a"].run(x, N * T * H * W, use_tc=tc, relu=True, pair_rows=T * H * W).view(N, T, H, W, ci)
            ops.Profiler.tag = "b"
            # blocks without SE: the swish that follows bn_b goes into the stencil's epilogue, so the
            # projection GEMM runs without its transform warps (its fastest form)
            swish_in_b = Options.swish_in_dw and not self.has_se
            cw = Options.channelwise
            planar = a.dtype == torch.bfloat16 and cw != "tma" and \
                ops.dw_planar_supported(T, H, W, ci, self.stride) > 0 and \
                (cw == "planar" or (self.stride == 1 and
                                    ops.dw_planar_lane_use(T, H, W, ci, self.stride) >= 0.85))
            if planar:
                b, partial = ops.dw_planar_fwd(a, d["wbp"], self.stride, ph, pw, self.has_se, swish=swish_in_b)
            else:
                b, partial = ops.dw_fwd(a, d["wb"], d["bb"], self.stride, ph, pw, self.has_se, swish=swish_in_b)
            del a
        _, _, Ho, Wo, _ = b.shape
        se = None
        if self.has_se:
            ops.Profiler.tag = "se"
            se = ops.se_mlp_fwd(partial, T * Ho * Wo, d["w1"], d["b1"], d["w2"], d["b2"])
        ops.Profiler.tag = "c"
        if shortcut is not None:
            out = d["c"].run_with_shortcut(b, N * T * Ho * Wo, shortcut, x if shortcut_rows is None else shortcut_rows,
                                           self.stride, se=se,
                                           rows_per_clip=T * Ho * Wo, swish=not swish_in_b, relu=relu)
        else:
            out = d["c"].run(b, N * T * Ho * Wo, use_tc=tc, se=se, rows_per_clip=T * Ho * Wo,
                             swish=not swish_in_b, residual=residual, relu=relu)
        return out.view(N, T, Ho, Wo, _pad8(self.out_channels))

    def call(self, input, training: bool = False):
        self._no_training(training)
        x = _as_device_clip(input, None)
        if self.in_channels is None:
            self._build(x.shape[-1])
        if x.shape[-1] != self.in_channels:
            raise ValueError(f"expected {self.in_channels} input channels, got {x.shape[-1]}")
        y = self._forward(_pad_channels(x, _pad8(self.in_channels)))
        return y[..., :self.out_channels]


class ResBlock(Layer):
    """Reference `model.py:322-394`.  `_block_index` is the same process-global class counter."""

    _block_index = 0

    def __init__(self, channels: tuple, bn_cfg, regularizer=None, stride: int = 1,
                 se_ratio: float = 0.0625, temp_kernel_size: int = 3):
        super().__init__(name="ResBlock_%u" % ResBlock._block_index)
        ResBlock._block_index += 1
        self.in_channels, self.inner_channels, self.out_channels = channels
        self._bn_cfg, self.stride = bn_cfg, stride
        self.has_shortcut = self.in_channels != self.out_channels or stride != 1
        if self.has_shortcut:
            self._add_conv("residual/kernel", (1, 1, 1, self.in_channels, self.out_channels))
            self._add_bn("bn_r", self.out_channels)
        self.bottleneck = self._child("bottleneck", Bottleneck(
            channels=channels[1:], stride=stride, bn_cfg=bn_cfg, regularizer=regularizer,
            block_index=ResBlock._block_index, se_ratio=se_ratio,
            temp_kernel_size=temp_kernel_size, in_channels=self.in_channels))

    def _prep(self, device):
        key = (str(device),)
        if key not in self._dev:
            d = {}
            if self.has_shortcut:
                s, t = self._fold_bn("bn_r", self._bn_cfg.EPS)
                d["r"] = PointwiseConv(self._vars["residual/kernel"], s, t, device)
            self._dev[key] = d
        return self._dev[key]

    def _forward(self, x: torch.Tensor) -> torch.Tensor:
        d = self._prep(x.device)
        N, T, H, W, _ = x.shape
        if self.has_shortcut:
            s = self.stride
            Ho, Wo = (H - 1) // s + 1, (W - 1) // s + 1
            ops.Profiler.tag = "shortcut"
            if _use_tc() and x.dtype == torch.bfloat16 and Options.fold_shortcut:
                # the shortcut conv as extra K columns of the projection GEMM: sampled by TMA straight from
                # x where 128-pixel tiles align with the output frames, else from the gathered rows
                rows = None if ops.pw_tc_sampler_supported(H, W, s) else \
                    (x.view(-1, x.shape[-1]) if s == 1 else ops.gather_rows_fwd(x, s))
                return self.bottleneck._forward(x, relu=True, shortcut=d["r"], shortcut_rows=rows)
            if _use_tc() and x.dtype == torch.bfloat16:
                # sampled pixels -> dense matrix -> tensor-core GEMM (bn_r folded)
                rows = x.view(-1, x.shape[-1]) if s == 1 else ops.gather_rows_fwd(x, s)
                res = d["r"].run(rows, N * T * Ho * Wo, use_tc=True, pair_rows=T * Ho * Wo)
            else:
                res = d["r"].run(x, N * T * Ho * Wo, use_tc=False, gather=(T, Ho, Wo, H, W, s))
        else:
            res = x
        return self.bottleneck._forward(x, residual=res, relu=True)

    def call(self, input, training: bool = False):
        self._no_training(training)
        x = _as_device_clip(input, None)
        if x.shape[-1] != self.in_channels:
            raise ValueError(f"expected {self.in_channels} input channels, got {x.shape[-1]}")
        y = self._forward(_pad_channels(x, _pad8(self.in_channels)))
        return y[..., :self.out_channels]


class ResStage(Layer):
    """Reference `model.py:396-455`."""

    _stage_index = 2

    def __init__(self, in_channels: int, inner_channels: int, out_channels: int, depth: int,
                 bn_cfg, regularizer=None, se_ratio: float = 0.0625, temp_kernel_size: int = 3):
        super().__init__(name="res_stage_%u" % ResStage._stage_index)
        ResStage._stage_index += 1
        self._bn_cfg, self._inner_channels = bn_cfg, inner_channels
        self.in_channels, self.out_channels = in_channels, out_channels
        self.blocks: List[ResBlock] = []
        for i in range(depth):
            blk = ResBlock(bn_cfg=bn_cfg, se_ratio=se_ratio, regularizer=regularizer,
                           temp_kernel_size=temp_kernel_size, stride=2 if i == 0 else 1,
                           channels=(in_channels if i == 0 else out_channels, inner_channels,
                                     out_channels))
            # checkpoint path of the i-th layer of the inner K.Sequential `self.stage`
            self.blocks.append(self._child(f"stage/layer_with_weights-{i}", blk))

    def _forward(self, x):
        for b in self.blocks:
            x = b._forward(x)
        return x

    def call(self, input, training: bool = False):
        self._no_training(training)
        x = _as_device_clip(input, None)
        y = self._forward(_pad_channels(x, _pad8(self.in_channels)))
        return y[..., :self.out_channels]


def finalize_metrics(acc: torch.Tensor, group=None, k: int = 5, return_dict: bool = True):
    """[sum loss, top-1 hits, top-k hits, videos] (per rank) -> Keras-style results.  Sums over the
    ranks of `group` first when torch.distributed is initialised (sum all-reduce of 32 bytes)."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        backend = dist.get_backend(group)
        buf = acc if (backend == "nccl") == acc.is_cuda else (acc.cuda() if backend == "nccl" else acc.cpu())
        dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
        acc = buf
    a = [float(v) for v in acc.detach().cpu().tolist()]
    count = max(a[3], 1.0)
    res = {"loss": a[0] / count, "acc": a[1] / count, f"top_{k}_acc": a[2] / count, "videos": int(a[3])}
    return res if return_dict else [res["loss"], res["acc"], res[f"top_{k}_acc"]]


def keras_default_weights(cfg, seed: int = 0) -> "OrderedDict[str, np.ndarray]":
    """The variables of a freshly constructed `X3D(cfg)` (train.py:128): Keras default initialisers,
    seeded.  What a from-scratch training run starts from; `synth.synthetic_weights` (randomised BN
    statistics and biases) is a parity/benchmark fixture only."""
    saved = (ResBlock._block_index, ResStage._stage_index, Layer._init_seed)
    reset_block_counters()
    Layer._init_seed = int(seed) * 100003
    try:
        return X3D(cfg).named_variables()
    finally:
        ResBlock._block_index, ResStage._stage_index, Layer._init_seed = saved


def reset_block_counters() -> None:
    """Back to the fresh-process state of the reference's class counters (model.py:326,401)."""
    ResBlock._block_index = 0
    ResStage._stage_index = 2


class _Conv5(Layer):
    """`K.Sequential(name='conv_5')` of Conv3D + BN + ReLU (model.py:78-93)."""

    def __init__(self, cin: int, cout: int, bn_cfg):
        super().__init__(name="conv_5")
        self.cin, self.cout, self._bn_cfg = cin, cout, bn_cfg
        self._add_conv("layer_with_weights-0/kernel", (1, 1, 1, cin, cout))
        self._add_bn("layer_with_weights-1", cout)

    def _prep(self, device):
        key = (str(device),)
        if key not in self._dev:
            s, t = self._fold_bn("layer_with_weights-1", self._bn_cfg.EPS)
            self._dev[key] = PointwiseConv(self._vars["layer_with_weights-0/kernel"], s, t, device)
        return self._dev[key]

    def _forward(self, x):
        N, T, H, W, _ = x.shape
        ops.Profiler.tag = "conv5"
        y = self._prep(x.device).run(x, N * T * H * W, use_tc=_use_tc(), relu=True)
        return y.view(N, T, H, W, _pad8(self.cout))

    def _forward_pooled(self, x) -> Optional[torch.Tensor]:
        """conv_5 + pool_5 (model.py:117-118) in one kernel: the GEMM's epilogue reduces its tiles over
        rows and the conv output is never written.  [N, pad8(cout)] fp32, or None when this path does
        not apply (not bf16 / tcgen05, or a clip is not a multiple of 64 positions)."""
        N, T, H, W, _ = x.shape
        P = T * H * W
        if not (_use_tc() and x.dtype == torch.bfloat16 and Options.pool_in_conv5 and P % 64 == 0):
            return None
        ops.Profiler.tag = "conv5"
        pc = self._prep(x.device)
        means = ops.pw_tc_fwd(x, pc.wp, pc.bias, M=N * P, K=pc.Ks, Nc=pc.Ns, relu=True, colmean=True, store=False)
        ops.Profiler.tag = "head_pool"
        return ops.avgpool_fwd(means[:N * P // 64].view(N, P // 64, pc.Ns))


class _Dense(Layer):
    def __init__(self, name, key_shape, bias: bool):
        super().__init__(name=name)
        if len(key_shape) == 5:
            self._add_conv("kernel", key_shape)
        else:
            self._vars["kernel"] = _glorot(self._rng(), key_shape, key_shape[0], key_shape[1])
        if bias:
            self._vars["bias"] = np.zeros(key_shape[-1], np.float32)

    def _prep(self, device):
        key = (str(device),)
        if key not in self._dev:
            self._dev[key] = PointwiseConv(self._vars["kernel"], None, None, device,
                                           bias=self._vars.get("bias"))
        return self._dev[key]


class X3D(Layer):
    """Reference `model.py:8-132`.

    `dtype`: None (default) = compute in the dtype of the clips passed to `call` (float32 ->
    fp32 kernels, bfloat16 -> bf16 storage / fp32 accumulate); "bfloat16" = store activations in
    bf16 whatever the input dtype (float32 clips are read directly by the stem)."""

    def __init__(self, cfg, dtype: Optional[str] = None, device=None, use_cuda_graph: bool = True):
        super().__init__(name="X3D")
        self.cfg = cfg
        self.num_classes = cfg.NETWORK.NUM_CLASSES
        self._bn_cfg = cfg.NETWORK.BN
        self._num_preds = cfg.TEST.NUM_TEMPORAL_VIEWS * cfg.TEST.NUM_SPATIAL_CROPS
        self._arch = A.build_arch(cfg, first_block_index=ResBlock._block_index + 1)
        self._conv1_dim = self._arch.stem_channels
        self._dtype = {None: None, "float32": torch.float32, "bfloat16": torch.bfloat16,
                       "bf16": torch.bfloat16, "fp32": torch.float32}[dtype]
        self._device = torch.device(device) if device is not None else None
        self._use_graph = use_cuda_graph
        self._graphs: Dict[tuple, tuple] = {}
        self.last_logits: Optional[torch.Tensor] = None

        self.conv1 = self._child("conv1", X3D_Stem(
            regularizer=None, bn_cfg=cfg.NETWORK.BN, out_channels=self._conv1_dim,
            temp_filter_size=cfg.NETWORK.C1_TEMP_FILTER,
            in_channels=cfg.DATA.NUM_INPUT_CHANNELS))
        if cfg.DATA.NUM_INPUT_CHANNELS == 3:
            self.conv1.input_norm = (tuple(cfg.DATA.MEAN), tuple(cfg.DATA.STD))
        self.stages: List[ResStage] = []
        for s, (depth, cin, inner, cout) in enumerate(self._arch.stage_dims):
            st = ResStage(in_channels=cin, inner_channels=inner, out_channels=cout, depth=depth,
                          bn_cfg=self._bn_cfg, regularizer=None)
            self.stages.append(self._child(f"stages/{s}", st))
        last_out = self._arch.stage_dims[-1][3]
        c5 = self.stages[-1]._inner_channels
        self.conv5 = self._child("conv5", _Conv5(last_out, c5, self._bn_cfg))
        self.pool5 = AdaptiveAvgPool3D(name="pool_5")
        self.fc1 = self._child("fc1", _Dense("fc_1", (1, 1, 1, c5, 2048), bias=False))
        self.dropout_rate = cfg.NETWORK.DROPOUT_RATE
        self.fc2 = self._child("fc2", _Dense("fc_2", (2048, self.num_classes), bias=True))

    # ---- weights
    def load_weights(self, filepath: str, verify: bool = True) -> _LoadStatus:
        """Restore from a TF-format checkpoint prefix (`train.py:137-143`, `eval.py:78-81`)."""
        names = set(self.named_variables())
        got = tf_bundle.load_model_variables(filepath, verify=verify)
        missing = self.set_weights_dict(got, strict=False)
        return _LoadStatus(missing, sorted(set(got) - names))

    def save_weights(self, filepath: str) -> None:
        tf_bundle.write_bundle(filepath, dict(self.named_variables()))

    # ---- forward
    def _forward(self, x: torch.Tensor, training: bool) -> Tuple[torch.Tensor, torch.Tensor]:
        act_dtype = self._dtype or (torch.float32 if x.dtype == torch.uint8 else x.dtype)
        out = self.conv1._forward(x, act_dtype)
        for st in self.stages:
            out = st._forward(out)
        pooled = self.conv5._forward_pooled(out)                        # [N, C5s] fp32
        if pooled is None:
            out = self.conv5._forward(out)
            ops.Profiler.tag = "head_pool"
            pooled = ops.avgpool_fwd(out)
        N = pooled.shape[0]
        ops.Profiler.tag = "head_fc"
        f1 = self.fc1._prep(x.device)
        h = ops.head_fc_fwd(pooled, f1.wt, None, K=f1.Ks, Nc=f1.Ns, relu=True)
        f2 = self.fc2._prep(x.device)
        logits_p = ops.head_fc_fwd(h, f2.wt, f2.bias, K=f2.Ks, Nc=f2.Ns)
        logits = logits_p if f2.Ns == self.num_classes else \
            logits_p[:, :self.num_classes].contiguous()
        ops.Profiler.tag = "head_softmax"
        probs = ops.softmax_viewmean_fwd(logits, 1 if training else self._num_preds)
        return probs, logits

    def _check_input(self, shape):
        if len(shape) != 5 or shape[-1] != self.cfg.DATA.NUM_INPUT_CHANNELS:
            raise ValueError(f"expected NDHWC clips with {self.cfg.DATA.NUM_INPUT_CHANNELS} channels, "
                             f"got shape {tuple(shape)}")
        if shape[0] % self._num_preds != 0:
            raise ValueError(f"batch {shape[0]} must be a multiple of "
                             f"NUM_TEMPORAL_VIEWS*NUM_SPATIAL_CROPS = {self._num_preds}")

    def _graph(self, shape, dtype, device, slot: int = 0, training: bool = False):
        """(graph, static input, static probs, static logits) for one input shape.  Captured on
        first use (after one eager run that warms lazy CUDA state).  Slots > 0 are extra captures
        over their own input/output buffers that share slot 0's memory pool (replays are
        stream-ordered), used by `predict` to overlap the H2D copy of the next batch."""
        key = (tuple(shape), dtype, str(device), Options.pointwise, Options.stem, Options.stem_u8, Options.swish_in_dw,
               Options.fuse_expand, Options.channelwise, Options.fold_shortcut, Options.pool_in_conv5, slot)
        if key not in self._graphs:
            static_in = torch.zeros(tuple(shape), dtype=dtype, device=device)
            self._forward(static_in, training)
            torch.cuda.current_stream().synchronize()
            g = torch.cuda.CUDAGraph()
            pool = None
            if slot:
                pool = self._graph(shape, dtype, device, 0, training)[0].pool()
            with torch.cuda.graph(g, pool=pool):
                s_probs, s_logits = self._forward(static_in, training)
            self._graphs[key] = (g, static_in, s_probs, s_logits)
        return self._graphs[key]

    def __call__(self, x, training: bool = False, copy: bool = True):
        return self.call(x, training=training, copy=copy)

    # ---- training mode behind the class API (train.py:128-152)
    def _trainer(self):
        """The training engine for this model's variables (training.X3DTrainer: batch-statistics BN,
        dropout, backward kernels, gradient exchange, optimizer), created on first use from the
        current variables; `_sync_from_trainer` copies trained values back into them."""
        if getattr(self, "_tr", None) is None:
            import torch.distributed as dist
            from .training import X3DTrainer
            world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
            rank = dist.get_rank() if world > 1 else 0
            dev = self._device or torch.device("cuda", torch.cuda.current_device())
            self._tr = X3DTrainer(self.cfg, device=dev, world=world, rank=rank).load(dict(self.named_variables()))
        return self._tr

    def _sync_from_trainer(self):
        if getattr(self, "_tr", None) is not None:
            self.set_weights_dict(self._tr.weights(), strict=False)

    def set_weights_dict(self, weights, prefix: str = "", strict: bool = True):
        self._graphs.clear()
        missing = super().set_weights_dict(weights, prefix, strict)
        if getattr(self, "_tr", None) is not None and not getattr(self, "_syncing", False):
            self._tr = None                              # rebuilt from the new values on next use
        return missing

    def fit(self, dataset, epochs: int = 1, initial_epoch: int = 0, steps_per_epoch: Optional[int] = None,
            lr_schedule=None, verbose: int = 0, **_):
        """Keras `model.fit` as train.py:145-152 uses it: for every epoch the learning rate comes from
        `lr_schedule(epoch)` (train.py:114-125, default training.lr_schedule of this model's cfg),
        `steps_per_epoch` batches `(clips, labels)` are taken from `dataset` (re-iterated per epoch; clips
        as for `call`, or a video.VideoBatch whose clips are built on the device),
        each one forward + backward + gradient all-reduce over the initialised torch.distributed
        group + optimizer step (cfg.TRAIN.OPTIMIZER).  Returns {"loss": [per-epoch mean]}.  The model's
        variables hold the trained values afterwards (call / evaluate / save_weights see them)."""
        from . import ops
        from .training import lr_schedule as default_schedule
        tr = self._trainer()
        sched = lr_schedule or (lambda e: default_schedule(self.cfg, e))
        dev = tr.device
        mean, std = tuple(self.cfg.DATA.MEAN), tuple(self.cfg.DATA.STD)
        hist = {"loss": [], "lr": []}
        for epoch in range(initial_epoch, epochs):
            lr = float(sched(epoch))
            tot, n = torch.zeros((), dtype=torch.float64, device=dev), 0
            for i, (clips, labels) in enumerate(dataset):
                if steps_per_epoch is not None and i >= steps_per_epoch:
                    break
                x = clips.clips(dev) if isinstance(clips, VideoBatch) else _as_device_clip(clips, dev)
                if x.dtype == torch.uint8:
                    x = ops.normalize_u8(x, mean, std, torch.float32)
                lab = torch.as_tensor(np.asarray(labels.cpu() if isinstance(labels, torch.Tensor) else labels)
                                      .reshape(-1), dtype=torch.int32).to(dev)
                loss = tr.step(x.float(), lab, lr)
                tot += loss.double().mean()
                n += 1
            hist["loss"].append(float(tot / max(n, 1)))
            hist["lr"].append(lr)
            if verbose:
                print(f"Epoch {epoch + 1}/{epochs} - loss: {hist['loss'][-1]:.4f} - lr: {lr:.5f}")
        self._syncing = True
        try:
            self._sync_from_trainer()
        finally:
            self._syncing = False
        return hist

    def call(self, input, training: bool = False, copy: bool = True):
        """`copy=False` returns the CUDA graph's static output buffers (valid until the next call
        with the same input shape) instead of fresh tensors: the zero-allocation path bench.py times.
        `training=True`: batch-statistics BatchNorm + dropout through the training kernels (fp32;
        moving statistics are updated as Keras does), per-clip softmax without view averaging
        (model.py:122-127)."""
        if training:
            x = _as_device_clip(input, self._device)
            if x.dtype == torch.uint8:
                x = ops.normalize_u8(x, tuple(self.cfg.DATA.MEAN), tuple(self.cfg.DATA.STD), torch.float32)
            tr = self._trainer()
            logits = tr.forward_training(x.float())
            tr.iteration += 1                            # a fresh dropout mask per training-mode call
            self.last_logits = logits
            self._syncing = True
            try:
                self._sync_from_trainer()                # the moving statistics moved
            finally:
                self._syncing = False
            return ops.softmax_viewmean_fwd(logits.contiguous(), 1)
        x = _as_device_clip(input, self._device)
        self._check_input(x.shape)
        if not self._use_graph:
            probs, self.last_logits = self._forward(x, training)
            return probs
        g, static_in, s_probs, s_logits = self._graph(x.shape, x.dtype, x.device, 0, training)
        if x.data_ptr() != static_in.data_ptr():
            static_in.copy_(x, non_blocking=True)
        g.replay()
        if not copy:
            # the captured graph's own output buffers: overwritten by the next call of this shape
            self.last_logits = s_logits
            return s_probs
        # like a Keras call, every result is a tensor of its own (1.6 kB per video)
        self.last_logits = s_logits.clone()
        return s_probs.clone()

    def static_input(self, shape, dtype=torch.bfloat16):
        """The captured graph's input buffer for `shape` (fill it in place and pass it to
        `call` to skip the staging copy).  None until the first call with that shape."""
        for key, (_, static_in, _, _) in self._graphs.items():
            if tuple(key[0]) == tuple(shape) and key[1] == dtype and key[-1] == 0:
                return static_in
        return None

    def predict(self, batches, training: bool = False, on_device=None):
        """Generator over host batches -> host probabilities: what `model.predict(dataset)` /
        `model.evaluate(dataset)` do in the reference (eval.py:83-89, Keras prefetches the next
        batch while the current one runs).  Each batch is an NDHWC numpy array or CPU tensor
        (pinned memory makes the copy asynchronous); its host->device copy is issued on a copy
        stream while the previous batch computes, the forward is one CUDA-graph replay, and the
        probabilities come back through a pinned buffer.  Yields float32 CPU tensors
        [videos, classes] in order.  uint8 batches are normalised on the device (fused into the
        stem's loader in bf16 mode).  `on_device(probs, i)`, if given, is called right after the
        replay of batch i with the device-resident probabilities (stream-ordered: enqueue work on
        the current stream, do not keep the tensor).  A batch can also be a video.VideoBatch: its
        packed decoded frames are copied on the copy stream and x3d_video_clips_u8 builds the uint8
        clips on that stream directly in the graph's input buffer.  A VideoBatch of JPEG frames
        (video.pack_jpeg) is decoded on the copy stream first; its status words come back with the
        probabilities, and a corrupt frame raises ValueError naming its record and frame when that
        batch's results are synchronised."""
        self._no_training(training)
        if not torch.cuda.is_available():
            raise RuntimeError("no CUDA device: the X3D path has no CPU implementation")
        device = self._device or torch.device("cuda", torch.cuda.current_device())
        main = torch.cuda.current_stream(device)
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(device)
        cs = self._copy_stream
        slots: Dict[tuple, dict] = {}

        def stage(hb, slot):
            if isinstance(hb, VideoBatch):
                return stage_video(hb, slot)
            if isinstance(hb, np.ndarray):
                hb = torch.from_numpy(np.ascontiguousarray(hb))
            if hb.dtype in (torch.float16, torch.float64):
                hb = hb.to(torch.float32)
            self._check_input(hb.shape)
            g, static_in, s_probs, s_logits = self._graph(hb.shape, hb.dtype, device, slot, training)
            st = slots.setdefault((tuple(hb.shape), hb.dtype, slot), {
                "host_out": torch.empty(tuple(s_probs.shape), dtype=torch.float32).pin_memory(),
                "done": torch.cuda.Event(), "copied": torch.cuda.Event()})
            st.update(g=g, s_probs=s_probs, s_logits=s_logits)
            cs.wait_event(st["done"])               # the replay that last read this buffer is over
            cs.wait_stream(main) if not st.get("used") else None
            st["used"] = True
            with torch.cuda.stream(cs):
                static_in.copy_(hb, non_blocking=True)
                st["copied"].record(cs)
            return st

        def stage_video(vb, slot):
            # the packed frames go to this slot's own staging buffer on the copy stream, and the clip
            # kernel runs on that stream straight into the graph's uint8 input: `done` (the replay that
            # last read the slot) orders both buffers, `copied` orders the replay behind the kernel
            self._check_input(vb.shape)
            g, static_in, s_probs, s_logits = self._graph(vb.shape, torch.uint8, device, slot, training)
            st = slots.setdefault((tuple(vb.shape), torch.uint8, slot), {
                "host_out": torch.empty(tuple(s_probs.shape), dtype=torch.float32).pin_memory(),
                "done": torch.cuda.Event(), "copied": torch.cuda.Event()})
            st.update(g=g, s_probs=s_probs, s_logits=s_logits)
            cs.wait_event(st["done"])
            cs.wait_stream(main) if not st.get("used") else None
            st["used"] = True
            nbytes = vb.frames.numel()
            with torch.cuda.stream(cs):
                if vb.encoded is not None:
                    # JPEG frames: decoded on this stream into the slot's scratch (coefficients, planes,
                    # frames); the status words come back with the probabilities and are checked when
                    # this batch's results are synchronised
                    frames, status = vb.encoded.decode(device, st)
                    if st.get("host_status") is None or st["host_status"].numel() < status.numel():
                        st["host_status"] = torch.empty(status.numel(), dtype=torch.int32).pin_memory()
                    st["status"] = status
                    decode_checks[batch_no[0]] = vb.encoded
                else:
                    if st.get("frames") is None or st["frames"].numel() < nbytes:
                        st["frames"] = torch.empty(nbytes, dtype=torch.uint8, device=device)
                    frames = st["frames"][:nbytes]
                    frames.copy_(vb.frames, non_blocking=True)
                    st["status"] = None
                if st.get("frame_off") is None or st["frame_off"].shape != vb.frame_off.shape:
                    st["frame_off"] = torch.empty(vb.frame_off.shape, dtype=torch.int64, device=device)
                    st["desc"] = torch.empty(vb.desc.shape, dtype=torch.int32, device=device)
                st["frame_off"].copy_(vb.frame_off, non_blocking=True)
                st["desc"].copy_(vb.desc, non_blocking=True)
                ops.video_clips_u8(frames, st["frame_off"], st["desc"], vb.shape[1], vb.shape[2], out=static_in)
                st["copied"].record(cs)
            return st

        # batch index -> EncodedFrames of a JPEG batch, then (EncodedFrames, the pinned buffer its status
        # words were copied to): the next staging of the slot may replace the slot's buffer before the check
        decode_checks: Dict[int, object] = {}
        batch_no = [0]                                # index of the batch being staged

        def finish(st, j):
            st["done"].synchronize()
            chk = decode_checks.pop(j, None)
            if chk is not None:
                chk[0].check(chk[1].numpy())
            return st["host_out"].clone()

        it = iter(batches)
        first = next(it, None)
        if first is None:
            return
        nxt, pending, i = stage(first, 0), None, 0
        while nxt is not None:
            cur = nxt
            hb = next(it, None)
            batch_no[0] = i + 1
            nxt = stage(hb, (i + 1) & 1) if hb is not None else None
            main.wait_event(cur["copied"])
            cur["g"].replay()
            if on_device is not None:
                on_device(cur["s_probs"], i)
            cur["host_out"].copy_(cur["s_probs"], non_blocking=True)
            if i in decode_checks:
                hs = cur["host_status"][:cur["status"].numel()]
                hs.copy_(cur["status"], non_blocking=True)
                decode_checks[i] = (decode_checks[i], hs)
            cur["done"].record(main)
            self.last_logits = cur["s_logits"]
            if pending is not None:
                yield finish(pending, i - 1)
            pending, i = cur, i + 1
        yield finish(pending, i - 1)

    def compile(self, optimizer=None, loss=None, metrics=None, top_k: int = 5, **_):
        """Keras `model.compile` as eval.py:62-70 uses it: the loss and the two metrics are fixed
        (SparseCategoricalCrossentropy on probabilities, SparseCategoricalAccuracy 'acc',
        SparseTopKCategoricalAccuracy(k) 'top_5_acc'); the arguments are accepted for source
        compatibility, `top_k` sets k."""
        self._top_k = int(top_k)
        return self

    def evaluate(self, dataset, group=None, return_dict: bool = True, verbose: int = 0):
        """`model.evaluate(dataset)` of eval.py:83-89.  `dataset` yields (clips, labels): clips as
        for `predict`, labels one int per video.  Loss and metrics are accumulated on the device
        (x3d_eval_metrics) from the same replay that produced the probabilities; with a
        torch.distributed `group` (or an initialised default group) the four sums are
        all-reduced, so every rank returns the metrics of the whole sharded set."""
        device = self._device or torch.device("cuda", torch.cuda.current_device())
        acc = torch.zeros(4, dtype=torch.float64, device=device)
        labels_dev: List[torch.Tensor] = []
        k = getattr(self, "_top_k", 5)

        def clips_only():
            for clips, labels in dataset:
                lab = torch.as_tensor(np.asarray(labels).reshape(-1), dtype=torch.int32)
                if lab.numel() * self._num_preds != clips.shape[0]:
                    raise ValueError(f"{clips.shape[0]} clips need {clips.shape[0] // self._num_preds} "
                                     f"labels, got {lab.numel()}")
                labels_dev.append(lab.to(device))
                yield clips

        def on_device(probs, i):
            ops.eval_metrics(probs, labels_dev[i], acc, k)
            labels_dev[i] = None

        n = 0
        for _ in self.predict(clips_only(), on_device=on_device):
            n += 1
            if verbose:
                print(f"\r{n} batches", end="", flush=True)
        return finalize_metrics(acc, group, k, return_dict)

    def summary(self, input_shape) -> str:
        """Keras-style table (`model.py:129-132`, dumps in `models/*/X3D_*.txt`)."""
        T, H, W, _ = input_shape
        plan = A.plan_shapes(self._arch, T, H, W)
        rows = [("input_1 (InputLayer)", f"[(None, {T}, {H}, {W}, {input_shape[3]})]", 0),
                ("conv_1 (X3D_Stem)", f"(None, {T}, {plan.stem.H}, {plan.stem.W}, {self._conv1_dim})",
                 self.conv1.count_params())]
        for s, st in enumerate(self.stages):
            lv = plan.stages[s]
            rows.append((f"res_stage_{s + 2} (ResStage)",
                         f"(None, {T}, {lv.H}, {lv.W}, {st.out_channels})", st.count_params()))
        lv = plan.stages[-1]
        rows += [("conv_5 (Sequential)", f"(None, {T}, {lv.H}, {lv.W}, {self.conv5.cout})",
                  self.conv5.count_params()),
                 ("pool_5 (AdaptiveAvgPool3D)", f"(None, 1, 1, 1, {self.conv5.cout})", 0),
                 ("fc_1 (Conv3D)", "(None, 1, 1, 1, 2048)", self.fc1.count_params()),
                 ("dropout (Dropout)", "(None, 1, 1, 1, 2048)", 0),
                 ("fc_2 (Dense)", f"(None, 1, 1, 1, {self.num_classes})", self.fc2.count_params())]
        total = self.count_params()
        nontrain = sum(int(v.size) for k, v in self.named_variables().items()
                       if not A.is_trainable(k))
        lines = ['Model: "X3D"', "_" * 65, f"{'Layer (type)':<29}{'Output Shape':<26}Param #",
                 "=" * 65]
        for name, shape, n in rows:
            lines += [f"{name:<29}{shape:<26}{n}", "_" * 65]
        lines[-1] = "=" * 65
        lines += [f"Total params: {total:,}", f"Trainable params: {total - nontrain:,}",
                  f"Non-trainable params: {nontrain:,}", "_" * 65]
        text = "\n".join(lines)
        print(text)
        return text
