"""Thin tensor-level wrappers over the C ABI (`include/x3d_b200.h`).

PyTorch is used only to own device memory and the CUDA stream; every function below launches
one hand-written kernel through ctypes and returns the output tensor.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import X3D_BF16, X3D_F32, PwArgs, PwTcArgs, check, lib


class Profiler:
    """Optional per-launch timing (CUDA events on the launching stream) used by bench.py to
    attribute time to kernel classes.  Off by default; never changes what is launched."""
    enabled = False
    tag = ""
    records: list = []
    launches = 0

    @classmethod
    def start(cls):
        cls.enabled, cls.records, cls.launches = True, [], 0

    @classmethod
    def stop(cls):
        cls.enabled = False
        torch.cuda.synchronize()
        out = [(tag, name, e0.elapsed_time(e1)) for tag, name, e0, e1 in cls.records]
        cls.records = []
        return out


def _launch(name: str, fn) -> None:
    Profiler.launches += 1
    if Profiler.enabled:
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        status = fn()
        e1.record()
        Profiler.records.append((Profiler.tag, name, e0, e1))
    else:
        status = fn()
    check(status, name)


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return X3D_F32
    if t.dtype == torch.bfloat16:
        return X3D_BF16
    raise TypeError(f"unsupported activation dtype {t.dtype} (float32 or bfloat16)")


def _torch_dt(code: int):
    return torch.float32 if code == X3D_F32 else torch.bfloat16


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _req(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor (there is no CPU path)")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    return t


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def stem_fwd(x: torch.Tensor, ws: torch.Tensor, wt: torch.Tensor, bias: torch.Tensor,
             out_dtype: torch.dtype) -> torch.Tensor:
    _req(x, "x")
    N, T, H, W, ci = x.shape
    if ci != 3:
        raise ValueError("stem input must have 3 channels")
    C = bias.numel()
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    out = torch.empty((N, T, Ho, Wo, C), dtype=out_dtype, device=x.device)
    _launch("x3d_stem_fwd", lambda: lib().x3d_stem_fwd(x.data_ptr(), _dt(x), ws.data_ptr(), wt.data_ptr(), bias.data_ptr(),
                             out.data_ptr(), _dt(out), N, T, H, W, C, wt.shape[0], _stream()))
    return out


def stem_tc_fwd(x: torch.Tensor, wc: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """Tensor-core stem: fp32 or bf16 clips in, bf16 activations out."""
    _req(x, "x")
    N, T, H, W, ci = x.shape
    if ci != 3:
        raise ValueError("stem input must have 3 channels")
    C = bias.numel()
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    out = torch.empty((N, T, Ho, Wo, C), dtype=torch.bfloat16, device=x.device)
    _launch("x3d_stem_tc_fwd", lambda: lib().x3d_stem_tc_fwd(
        x.data_ptr(), _dt(x), wc.data_ptr(), bias.data_ptr(), out.data_ptr(), N, T, H, W, C,
        wc.shape[0], _stream()))
    return out


def _f3(vals) -> "_lib.C.Array":
    v = [float(x) for x in vals]
    if len(v) != 3:
        raise ValueError("mean / std must have 3 entries (RGB)")
    return (_lib.C.c_float * 3)(*v)


def normalize_u8(x: torch.Tensor, mean, std, out_dtype: torch.dtype, norm_value: float = 255.0) -> torch.Tensor:
    """utils.normalize (reference utils.py:42-72) on uint8 NDHWC clips -> fp32 / bf16."""
    _req(x, "x")
    if x.dtype != torch.uint8 or x.shape[-1] != 3:
        raise TypeError("normalize_u8 needs uint8 clips with 3 channels")
    out = torch.empty(x.shape, dtype=out_dtype, device=x.device)
    _launch("x3d_normalize_u8", lambda: lib().x3d_normalize_u8(
        x.data_ptr(), out.data_ptr(), x.numel() // 3, _f3(mean), _f3(std), float(norm_value), _dt(out), _stream()))
    return out


def eval_views_u8(video: torch.Tensor, T: int, views: int, crops: int, size: int) -> torch.Tensor:
    """Evaluation clips of one decoded, resized video [F,H,W,3] uint8 (device): temporal views
    (transforms.py:48-65) x uniform crops (transforms.py:149-222) -> [crops*views, T, size, size, 3]."""
    _req(video, "video")
    if video.dtype != torch.uint8 or video.dim() != 4 or video.shape[-1] != 3:
        raise TypeError("eval_views_u8 needs a [F,H,W,3] uint8 video")
    F, H, W, _ = video.shape
    out = torch.empty((crops * views, T, size, size, 3), dtype=torch.uint8, device=video.device)
    _launch("x3d_eval_views_u8", lambda: lib().x3d_eval_views_u8(video.data_ptr(), out.data_ptr(), F, H, W, T, views,
                                                               crops, size, _stream()))
    return out


def video_clips_u8(frames: torch.Tensor, frame_off: torch.Tensor, desc: torch.Tensor, T: int, S: int,
                   out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Clips of a ragged batch of decoded videos (device): per clip a bilinear short-side resize, an
    S x S crop and a flip, as x3d_video_clips_u8 describes.  `frames` packed uint8 frames, `frame_off`
    int64 [N*T] byte offsets of each output frame's source, `desc` int32 [N, 7] x3d_clip_desc rows
    (validated on the host: video.validate) -> [N, T, S, S, 3] uint8 (written into `out` if given)."""
    for t, name in ((frames, "frames"), (frame_off, "frame_off"), (desc, "desc")):
        _req(t, name)
    if frames.dtype != torch.uint8 or frame_off.dtype != torch.int64 or desc.dtype != torch.int32:
        raise TypeError("video_clips_u8: frames uint8, frame_off int64, desc int32")
    N = desc.shape[0]
    if desc.dim() != 2 or desc.shape[1] != 7 or frame_off.numel() != N * T:
        raise ValueError(f"video_clips_u8: desc {tuple(desc.shape)} / frame_off {frame_off.numel()} for T={T}")
    shape = (N, T, S, S, 3)
    if out is None:
        out = torch.empty(shape, dtype=torch.uint8, device=frames.device)
    elif tuple(out.shape) != shape or out.dtype != torch.uint8 or not out.is_contiguous():
        raise ValueError(f"video_clips_u8: out must be contiguous uint8 {shape}")
    _launch("x3d_video_clips_u8", lambda: lib().x3d_video_clips_u8(
        frames.data_ptr(), frame_off.data_ptr(), desc.data_ptr(), N, T, S, out.data_ptr(), _stream()))
    return out


def jpeg_entropy(data: torch.Tensor, frames: torch.Tensor, tables: torch.Tensor, nframes: int,
                 coef: torch.Tensor, status: torch.Tensor) -> None:
    """x3d_jpeg_entropy: Huffman-decode `nframes` frames (`frames` / `tables`: the x3d_jpeg_frame /
    x3d_jpeg_tables records as raw uint8 device buffers, validated on the host by video.pack_jpeg)
    into `coef` (int16 blocks x 64) and their status words (int32)."""
    for t, name in ((data, "data"), (frames, "frames"), (tables, "tables"), (coef, "coef"), (status, "status")):
        _req(t, name)
    if coef.dtype != torch.int16 or status.dtype != torch.int32:
        raise TypeError("jpeg_entropy: coef int16, status int32")
    _launch("x3d_jpeg_entropy", lambda: lib().x3d_jpeg_entropy(
        data.data_ptr(), frames.data_ptr(), tables.data_ptr(), nframes, coef.data_ptr(), status.data_ptr(), _stream()))


def jpeg_entropy_rst(data: torch.Tensor, frames: torch.Tensor, tables: torch.Tensor, intervals: torch.Tensor,
                     nintervals: int, coef: torch.Tensor, status: torch.Tensor, status_lo: int, status_hi: int) -> None:
    """x3d_jpeg_entropy_rst: Huffman-decode `nintervals` restart intervals (`intervals`: the
    x3d_jpeg_interval records as a raw uint8 device buffer, validated on the host by video.pack_jpeg)
    into `coef`.  The kernel only raises status words (atomicMax), so the words status[status_lo:
    status_hi] of the frames the intervals belong to are cleared on the stream first."""
    for t, name in ((data, "data"), (frames, "frames"), (tables, "tables"), (intervals, "intervals"),
                    (coef, "coef"), (status, "status")):
        _req(t, name)
    if coef.dtype != torch.int16 or status.dtype != torch.int32:
        raise TypeError("jpeg_entropy_rst: coef int16, status int32")
    if not 0 <= status_lo <= status_hi <= status.numel():
        raise ValueError(f"jpeg_entropy_rst: status words {status_lo}..{status_hi} of {status.numel()}")
    status[status_lo:status_hi].zero_()
    _launch("x3d_jpeg_entropy_rst", lambda: lib().x3d_jpeg_entropy_rst(
        data.data_ptr(), frames.data_ptr(), tables.data_ptr(), intervals.data_ptr(), nintervals, coef.data_ptr(),
        status.data_ptr(), _stream()))


def jpeg_idct(coef: torch.Tensor, frames: torch.Tensor, tables: torch.Tensor, nframes: int, max_blocks: int,
              method: int, planes: torch.Tensor) -> None:
    """x3d_jpeg_idct: dequantise + 8x8 IDCT (method _lib.X3D_JPEG_ISLOW / X3D_JPEG_IFAST) into `planes`."""
    for t, name in ((coef, "coef"), (frames, "frames"), (tables, "tables"), (planes, "planes")):
        _req(t, name)
    _launch("x3d_jpeg_idct", lambda: lib().x3d_jpeg_idct(
        coef.data_ptr(), frames.data_ptr(), tables.data_ptr(), nframes, max_blocks, method, planes.data_ptr(), _stream()))


def jpeg_color(planes: torch.Tensor, frames: torch.Tensor, nframes: int, max_pixels: int, out: torch.Tensor) -> None:
    """x3d_jpeg_color: chroma upsampling + YCbCr -> RGB into the packed frames `out` (uint8)."""
    for t, name in ((planes, "planes"), (frames, "frames"), (out, "out")):
        _req(t, name)
    _launch("x3d_jpeg_color", lambda: lib().x3d_jpeg_color(
        planes.data_ptr(), frames.data_ptr(), nframes, max_pixels, out.data_ptr(), _stream()))


def _req_all(what: str, dtypes: dict) -> None:
    for name, (t, dtype) in dtypes.items():
        _req(t, name)
        if t.dtype != dtype:
            raise TypeError(f"{what}: {name} must be {dtype}, got {t.dtype}")


def jpeg_fdct(rgb: torch.Tensor, frames: torch.Tensor, tables: torch.Tensor, nframes: int, max_blocks: int,
              coef: torch.Tensor) -> None:
    """x3d_jpeg_fdct: colour conversion, downsampling, ISLOW FDCT and quantisation of `nframes` packed RGB
    frames (`frames` / `tables`: x3d_jpeg_enc_frame / x3d_jpeg_enc_tables records as raw uint8 device
    buffers, built by jpeg.encode_frames) into `coef` (int16 blocks x 64)."""
    _req_all("jpeg_fdct", {"rgb": (rgb, torch.uint8), "frames": (frames, torch.uint8),
                           "tables": (tables, torch.uint8), "coef": (coef, torch.int16)})
    _launch("x3d_jpeg_fdct", lambda: lib().x3d_jpeg_fdct(
        rgb.data_ptr(), frames.data_ptr(), tables.data_ptr(), nframes, max_blocks, coef.data_ptr(), _stream()))


def jpeg_enc_bits(coef: torch.Tensor, frames: torch.Tensor, tables: torch.Tensor, nframes: int, boff: torch.Tensor,
                  res: torch.Tensor, words: torch.Tensor) -> None:
    """x3d_jpeg_enc_bits: the bit offset of every block (int64 `boff`), each frame's bit count and status
    (x3d_jpeg_enc_result records in the uint8 `res`), and the frame's words zeroed."""
    _req_all("jpeg_enc_bits", {"coef": (coef, torch.int16), "frames": (frames, torch.uint8),
                               "tables": (tables, torch.uint8), "boff": (boff, torch.int64),
                               "res": (res, torch.uint8), "words": (words, torch.int32)})
    _launch("x3d_jpeg_enc_bits", lambda: lib().x3d_jpeg_enc_bits(
        coef.data_ptr(), frames.data_ptr(), tables.data_ptr(), nframes, boff.data_ptr(), res.data_ptr(),
        words.data_ptr(), _stream()))


def jpeg_enc_emit(coef: torch.Tensor, frames: torch.Tensor, tables: torch.Tensor, nframes: int, max_blocks: int,
                  boff: torch.Tensor, res: torch.Tensor, words: torch.Tensor) -> None:
    """x3d_jpeg_enc_emit: every block's Huffman codes into the frame's 32-bit words (int32 `words`)."""
    _req_all("jpeg_enc_emit", {"coef": (coef, torch.int16), "frames": (frames, torch.uint8),
                               "tables": (tables, torch.uint8), "boff": (boff, torch.int64),
                               "res": (res, torch.uint8), "words": (words, torch.int32)})
    _launch("x3d_jpeg_enc_emit", lambda: lib().x3d_jpeg_enc_emit(
        coef.data_ptr(), frames.data_ptr(), tables.data_ptr(), nframes, max_blocks, boff.data_ptr(), res.data_ptr(),
        words.data_ptr(), _stream()))


def jpeg_enc_stuff(words: torch.Tensor, frames: torch.Tensor, nframes: int, res: torch.Tensor,
                   out: torch.Tensor) -> None:
    """x3d_jpeg_enc_stuff: byte stuffing into `out` (uint8); each segment's offset and length in `res`."""
    _req_all("jpeg_enc_stuff", {"words": (words, torch.int32), "frames": (frames, torch.uint8),
                                "res": (res, torch.uint8), "out": (out, torch.uint8)})
    _launch("x3d_jpeg_enc_stuff", lambda: lib().x3d_jpeg_enc_stuff(
        words.data_ptr(), frames.data_ptr(), nframes, res.data_ptr(), out.data_ptr(), out.numel(), _stream()))


def stem_tc_u8_fwd(x: torch.Tensor, mean, std, wc: torch.Tensor, bias: torch.Tensor,
                   norm_value: float = 255.0) -> torch.Tensor:
    """Tensor-core stem with the uint8 input stage fused into its loader; bf16 activations out."""
    _req(x, "x")
    if x.dtype != torch.uint8 or x.shape[-1] != 3:
        raise TypeError("stem_tc_u8_fwd needs uint8 clips with 3 channels")
    N, T, H, W, _ = x.shape
    C = bias.numel()
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    out = torch.empty((N, T, Ho, Wo, C), dtype=torch.bfloat16, device=x.device)
    _launch("x3d_stem_tc_u8_fwd", lambda: lib().x3d_stem_tc_u8_fwd(
        x.data_ptr(), _f3(mean), _f3(std), float(norm_value), wc.data_ptr(), bias.data_ptr(), out.data_ptr(),
        N, T, H, W, C, wc.shape[0], _stream()))
    return out


def eval_metrics(probs: torch.Tensor, labels: torch.Tensor, acc: torch.Tensor, k: int = 5) -> None:
    """acc[0..3] += (sum loss, top-1 hits, top-k hits, videos); eval.py:62-70."""
    _req(probs, "probs"); _req(labels, "labels"); _req(acc, "acc")
    if probs.dtype != torch.float32 or labels.dtype != torch.int32 or acc.dtype != torch.float64:
        raise TypeError("eval_metrics: probs fp32, labels int32, acc fp64")
    V, ncls = probs.shape
    if labels.numel() != V or acc.numel() < 4:
        raise ValueError(f"eval_metrics: {V} videos but {labels.numel()} labels / acc of {acc.numel()}")
    _launch("x3d_eval_metrics", lambda: lib().x3d_eval_metrics(
        probs.data_ptr(), labels.data_ptr(), acc.data_ptr(), V, ncls, int(k), _stream()))


def pw_fwd(a: torch.Tensor, wt: torch.Tensor, bias: Optional[torch.Tensor], *, M: int, K: int,
           Nc: int, out: Optional[torch.Tensor] = None, out_dtype: Optional[torch.dtype] = None,
           residual: Optional[torch.Tensor] = None, se: Optional[torch.Tensor] = None,
           rows_per_clip: int = 0, swish: bool = False, relu: bool = False,
           gather: Optional[Tuple[int, int, int, int, int, int]] = None) -> torch.Tensor:
    """Generic SIMT pointwise GEMM.  `a` is viewed as [*, lda=K]; `gather`=(T,Ho,Wo,Hi,Wi,stride)
    selects strided input pixels (shortcut conv)."""
    _req(a, "a")
    if out is None:
        out = torch.empty((M, Nc), dtype=out_dtype or a.dtype, device=a.device)
    args = PwArgs()
    args.A, args.Wt, args.bias = a.data_ptr(), wt.data_ptr(), _ptr(bias)
    args.R, args.se, args.D = _ptr(residual), _ptr(se), out.data_ptr()
    args.M, args.K, args.Nc = M, K, Nc
    args.lda, args.ldw, args.ldr, args.ldd = K, wt.shape[1], Nc, Nc
    args.rows_per_clip = rows_per_clip
    args.a_dtype, args.d_dtype = _dt(a), _dt(out)
    args.swish, args.relu = int(swish), int(relu)
    if gather is not None:
        args.gather = 1
        args.T, args.Ho, args.Wo, args.Hi, args.Wi, args.stride = gather
    _launch("x3d_pw_fwd", lambda: lib().x3d_pw_fwd(args, _stream()))
    return out


def pw_tc_fwd(a: torch.Tensor, wp: torch.Tensor, bias: Optional[torch.Tensor], *, M: int, K: int,
              Nc: int, out: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None,
              se: Optional[torch.Tensor] = None, rows_per_clip: int = 0, swish: bool = False,
              relu: bool = False, a2: Optional[torch.Tensor] = None, a2_stride: int = 1,
              colmean: bool = False, store: bool = True):
    """tcgen05 pointwise GEMM (bf16).  `wp` is the packed [Npad, Kpad] bf16 weight.
    `a2` [N,T,Hi,Wi,K2]: second K source sampled at (t, s*ho, s*wo) -- the shortcut conv folded in;
    or an already gathered dense [M,K2] matrix.
    `colmean`: also return the fp32 means over 64-row groups [2*ceil(M/128), Nc] (conv_5 + pool_5);
    with `store=False` the GEMM output itself is not written and only the means are returned."""
    _req(a, "a")
    if a.dtype != torch.bfloat16:
        raise TypeError("pw_tc_fwd needs bf16 activations")
    if not store and not colmean:
        raise ValueError("pw_tc_fwd: store=False only together with colmean=True")
    if out is None:
        # (the kernel still wants a valid D for its tensor map; without a store one row is enough)
        out = torch.empty((M if store else 128, Nc), dtype=torch.bfloat16, device=a.device)
    means = torch.empty((2 * -(-M // 128), Nc), dtype=torch.float32, device=a.device) if colmean else None
    args = PwTcArgs()
    args.A, args.Wp, args.bias = a.data_ptr(), wp.data_ptr(), _ptr(bias)
    args.R, args.se, args.D = _ptr(residual), _ptr(se), out.data_ptr()
    args.colmean, args.store_d = _ptr(means), int(store)
    args.M, args.K, args.Nc = M, K, Nc
    args.lda, args.ldr, args.ldd = K, Nc, Nc
    args.Npad, args.Kpad = wp.shape
    args.rows_per_clip = rows_per_clip
    args.swish, args.relu = int(swish), int(relu)
    if a2 is not None:
        _req(a2, "a2")
        if a2.dtype != torch.bfloat16 or a2.dim() not in (2, 5):
            raise TypeError("pw_tc_fwd: a2 must be a bf16 [N,T,H,W,C] tensor or a dense [M,C] matrix")
        if a2.dim() == 5:
            args.A2, args.a2_nt, args.K2 = a2.data_ptr(), a2.shape[0] * a2.shape[1], a2.shape[4]
            args.a2_stride, args.a2_hi, args.a2_wi = a2_stride, a2.shape[2], a2.shape[3]
        else:
            if a2.shape[0] != M:
                raise ValueError("pw_tc_fwd: dense a2 needs M rows")
            args.A2, args.K2, args.a2_stride = a2.data_ptr(), a2.shape[1], 0
    _launch("x3d_pw_tc_fwd", lambda: lib().x3d_pw_tc_fwd(args, _stream()))
    if colmean:
        return (out, means) if store else means
    return out


def pw_tc_sampler_supported(Hi: int, Wi: int, stride: int) -> bool:
    """Can x3d_pw_tc_fwd read a stride-`stride` pixel sample of Hi x Wi frames as its second source?"""
    return bool(lib().x3d_pw_tc_sampler_supported(Hi, Wi, stride))


def gather_rows_fwd(x: torch.Tensor, stride: int) -> torch.Tensor:
    """[N,T,H,W,C] -> dense [N*T*Ho*Wo, C] of the pixels a stride-(1,s,s) 'valid' 1x1x1 conv reads."""
    _req(x, "x")
    N, T, H, W, C = x.shape
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    out = torch.empty((N * T * Ho * Wo, C), dtype=x.dtype, device=x.device)
    _launch("x3d_gather_rows_fwd", lambda: lib().x3d_gather_rows_fwd(
        x.data_ptr(), out.data_ptr(), N * T, H, W, stride, C, _dt(x), _stream()))
    return out


def head_fc_fwd(a: torch.Tensor, wt: torch.Tensor, bias: Optional[torch.Tensor], *, K: int, Nc: int,
                relu: bool = False) -> torch.Tensor:
    """Small-M fp32 GEMM of the head: act(a[M,K] @ wt[K,Nc] + bias)."""
    _req(a, "a")
    if a.dtype != torch.float32:
        raise TypeError("head_fc_fwd needs float32 input")
    M = a.shape[0]
    out = torch.empty((M, Nc), dtype=torch.float32, device=a.device)
    _launch("x3d_head_fc_fwd", lambda: lib().x3d_head_fc_fwd(
        a.data_ptr(), wt.data_ptr(), _ptr(bias), out.data_ptr(), M, K, Nc, a.shape[1], wt.shape[1],
        Nc, int(relu), _stream()))
    return out


def dw_fwd(x: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, stride: int, pad_h: int,
           pad_w: int, want_se: bool, swish: bool = False) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """`swish`: apply the activation that follows bn_b in the kernel's epilogue (blocks without SE)."""
    _req(x, "x")
    if swish and want_se:
        raise ValueError("swish can only be fused when no SE sums are requested")
    N, T, H, W, C = x.shape
    Ho, Wo = -(-H // stride), -(-W // stride)
    out = torch.empty((N, T, Ho, Wo, C), dtype=x.dtype, device=x.device)
    partial = None
    if want_se:
        nblk = lib().x3d_dw_partial_blocks(T, H, W, C, stride, _dt(x))
        if nblk <= 0:
            raise _lib.X3DLibError("x3d_dw_partial_blocks rejected the shape")
        partial = torch.empty((N, nblk, C), dtype=torch.float32, device=x.device)
    _launch("x3d_dw3x3x3_fwd", lambda: lib().x3d_dw3x3x3_act_fwd(x.data_ptr(), w.data_ptr(), bias.data_ptr(), out.data_ptr(),
                                _ptr(partial), N, T, H, W, C, stride, pad_h, pad_w, _dt(x), int(swish),
                                _stream()))
    return out, partial


def dw_planar_taps(w: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """[27, C] BN-folded taps + [C] shift -> the planar kernel's table [C/2, 28, 2] (fp32, device)."""
    C = w.shape[1]
    t = torch.cat([w, bias.view(1, C)], 0)                       # [28, C]
    return t.view(28, C // 2, 2).permute(1, 0, 2).contiguous()


def dw_planar_supported(T: int, H: int, W: int, c: int, stride: int) -> int:
    """SE partial blocks per clip of the planar channelwise kernel, 0 if it does not take the shape."""
    if c % 8 or c // 2 > 288:
        return 0
    return int(lib().x3d_dw_planar_partial_blocks(T, H, W, c, stride))


def dw_planar_lane_use(T: int, H: int, W: int, c: int, stride: int) -> float:
    """Fraction of the planar kernel's lane grid that a shape fills (1.0: no padding lanes); 0 without a plan."""
    if c % 8 or c // 2 > 288:
        return 0.0
    return int(lib().x3d_dw_planar_lane_permille(T, H, W, c, stride)) / 1000.0


def dw_planar_fwd(x: torch.Tensor, taps: torch.Tensor, stride: int, pad_h: int, pad_w: int, want_se: bool,
                  swish: bool = False) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """Channelwise 3x3x3 + BN (+ swish | SE sums), lanes = pixels / uniform-register taps (bf16)."""
    _req(x, "x")
    if x.dtype != torch.bfloat16:
        raise TypeError("dw_planar_fwd needs bf16 activations")
    if swish and want_se:
        raise ValueError("swish in the epilogue only without SE (the SE scale comes before the swish)")
    N, T, H, W, C = x.shape
    Ho, Wo = -(-H // stride), -(-W // stride)
    out = torch.empty((N, T, Ho, Wo, C), dtype=x.dtype, device=x.device)
    partial = None
    if want_se:
        nblk = dw_planar_supported(T, H, W, C, stride)
        if nblk <= 0:
            raise _lib.X3DLibError("x3d_dw_planar_partial_blocks rejected the shape")
        partial = torch.empty((N, nblk, C), dtype=torch.float32, device=x.device)
    _launch("x3d_dw3x3x3_planar_fwd", lambda: lib().x3d_dw3x3x3_planar_fwd(
        x.data_ptr(), taps.data_ptr(), out.data_ptr(), _ptr(partial), N, T, H, W, C, stride, pad_h, pad_w,
        1 if swish else 0, _stream()))
    return out, partial


def expand_dw_supported(T: int, H: int, W: int, cin: int, c: int, stride: int) -> int:
    """Number of SE partial blocks of the fused kernel's launch, 0 if no tile plan fits."""
    return int(lib().x3d_expand_dw_partial_blocks(T, H, W, cin, c, stride))


def expand_dw_fwd(x: torch.Tensor, wa: torch.Tensor, bias_a: torch.Tensor, wb: torch.Tensor,
                  bias_b: torch.Tensor, stride: int, pad_h: int, pad_w: int,
                  want_se: bool) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """Fused expand (1x1x1 + BN + ReLU) -> channelwise 3x3x3 (+ BN, SE sums); bf16 only.
    `wa` is the packed [Npad, Kpad] bf16 expand weight of `pw_tc_fwd`."""
    _req(x, "x")
    if x.dtype != torch.bfloat16:
        raise TypeError("expand_dw_fwd needs bf16 activations")
    N, T, H, W, cin = x.shape
    C = wb.shape[1]
    Ho, Wo = -(-H // stride), -(-W // stride)
    out = torch.empty((N, T, Ho, Wo, C), dtype=x.dtype, device=x.device)
    partial = None
    if want_se:
        nblk = expand_dw_supported(T, H, W, cin, C, stride)
        if nblk <= 0:
            raise _lib.X3DLibError("x3d_expand_dw_partial_blocks rejected the shape")
        partial = torch.empty((N, nblk, C), dtype=torch.float32, device=x.device)
    npad, kpad = wa.shape
    _launch("x3d_expand_dw_fwd", lambda: lib().x3d_expand_dw_fwd(
        x.data_ptr(), wa.data_ptr(), bias_a.data_ptr(), wb.data_ptr(), bias_b.data_ptr(),
        out.data_ptr(), _ptr(partial), N, T, H, W, cin, C, kpad, npad, stride, pad_h, pad_w,
        _stream()))
    return out, partial


def pw_tf32(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, *, relu: bool = False,
            transpose_w: bool = True, M: Optional[int] = None, stats: Optional[torch.Tensor] = None) -> torch.Tensor:
    """fp32 pointwise conv on the tcgen05 tensor cores (3xTF32 split, x3d_pw_tf32_fwd).
    `w` is the stored [K, N] fp32 kernel.  transpose_w=True: D[M, N] = a[M, K] . w (forward);
    transpose_w=False: D[M, K] = a[M, N] . w^T (backward-data) -- no transposed copy is made either way:
    x3d_tf32_split writes the hi / lo planes in the orientation the GEMM reads.  `stats`: zeroed fp64
    [2, N] that receives the column sums / sums of squares of the result (BatchNorm batch statistics)."""
    _req(a, "a")
    _req(w, "w")
    if a.dtype != torch.float32 or w.dtype != torch.float32:
        raise TypeError("pw_tf32 needs fp32 operands")
    K, N = w.shape
    red, nout = (K, N) if transpose_w else (N, K)
    M = a.shape[0] if M is None else M
    lda = a.shape[-1]
    if lda < red:
        raise ValueError(f"a has {lda} columns, the reduction needs {red}")
    bs = torch.empty((2, nout, red), dtype=torch.float32, device=a.device)
    _launch("x3d_tf32_split", lambda: lib().x3d_tf32_split(w.data_ptr(), bs.data_ptr(), nout, red, N,
                                                         1 if transpose_w else 0, _stream()))
    out = torch.empty((M, nout), dtype=torch.float32, device=a.device)
    _launch("x3d_pw_tf32_fwd", lambda: lib().x3d_pw_tf32_fwd(a.data_ptr(), bs.data_ptr(), _ptr(bias), out.data_ptr(),
                                                           M, red, nout, lda, nout, 1 if relu else 0, _ptr(stats),
                                                           _stream()))
    return out


def expand_dw2_supported(T: int, H: int, W: int, cin: int, c: int, stride: int) -> int:
    """SE partial blocks per clip of the persistent fused kernel's plan, 0 if no tile plan fits."""
    return int(lib().x3d_expand_dw2_partial_blocks(T, H, W, cin, c, stride))


def expand_dw2_fwd(x: torch.Tensor, wa: torch.Tensor, bias_a: torch.Tensor, wb: torch.Tensor,
                   bias_b: torch.Tensor, stride: int, pad_h: int, pad_w: int, want_se: bool,
                   swish: bool = False) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """Fused expand (1x1x1 + BN + ReLU) -> channelwise 3x3x3 (+ BN, SE sums or swish), persistent
    warp-specialised kernel (x3d_expand_dw2_fwd); bf16 in / out, fp32 in between."""
    _req(x, "x")
    if x.dtype != torch.bfloat16:
        raise TypeError("expand_dw2_fwd needs bf16 activations")
    if swish and want_se:
        raise ValueError("swish in the epilogue only without SE (the SE scale comes before the swish)")
    N, T, H, W, cin = x.shape
    C = wb.shape[1]
    Ho, Wo = -(-H // stride), -(-W // stride)
    out = torch.empty((N, T, Ho, Wo, C), dtype=x.dtype, device=x.device)
    partial = None
    if want_se:
        nblk = expand_dw2_supported(T, H, W, cin, C, stride)
        if nblk <= 0:
            raise _lib.X3DLibError("x3d_expand_dw2_partial_blocks rejected the shape")
        partial = torch.empty((N, nblk, C), dtype=torch.float32, device=x.device)
    npad, kpad = wa.shape
    _launch("x3d_expand_dw2_fwd", lambda: lib().x3d_expand_dw2_fwd(
        x.data_ptr(), wa.data_ptr(), bias_a.data_ptr(), wb.data_ptr(), bias_b.data_ptr(),
        out.data_ptr(), _ptr(partial), N, T, H, W, cin, C, kpad, npad, stride, pad_h, pad_w,
        1 if swish else 0, _stream()))
    return out, partial


def se_mlp_fwd(partial: torch.Tensor, count: int, w1: torch.Tensor, b1: torch.Tensor,
               w2: torch.Tensor, b2: torch.Tensor) -> torch.Tensor:
    N, nblk, C = partial.shape
    scale = torch.empty((N, C), dtype=torch.float32, device=partial.device)
    _launch("x3d_se_mlp_fwd", lambda: lib().x3d_se_mlp_fwd(partial.data_ptr(), nblk, 1.0 / float(count), w1.data_ptr(),
                               b1.data_ptr(), w2.data_ptr(), b2.data_ptr(), scale.data_ptr(),
                               N, C, w1.shape[1], _stream()))
    return scale


def avgpool_fwd(x: torch.Tensor) -> torch.Tensor:
    """[N, ..., C] -> [N, C] fp32 mean over all middle positions."""
    _req(x, "x")
    N, C = x.shape[0], x.shape[-1]
    P = x.numel() // (N * C)
    out = torch.empty((N, C), dtype=torch.float32, device=x.device)
    _launch("x3d_avgpool_fwd", lambda: lib().x3d_avgpool_fwd(x.data_ptr(), out.data_ptr(), N, P, C, _dt(x), _stream()))
    return out


def softmax_viewmean_fwd(logits: torch.Tensor, num_preds: int) -> torch.Tensor:
    _req(logits, "logits")
    N, ncls = logits.shape
    if N % num_preds:
        raise ValueError(f"batch {N} is not a multiple of num_preds {num_preds}")
    probs = torch.empty((N // num_preds, ncls), dtype=torch.float32, device=logits.device)
    _launch("x3d_softmax_viewmean_fwd", lambda: lib().x3d_softmax_viewmean_fwd(logits.data_ptr(), probs.data_ptr(), N, ncls, num_preds,
                                         _stream()))
    return probs
