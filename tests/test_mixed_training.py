"""The 'mixed_bfloat16' training policy without a GPU: the rounding oracle (tests/mixed_oracle.py),
the new C-ABI entry points, the driver's flag and what the compiler makes of the new kernels."""
import ctypes
import os
import re
import subprocess
from unittest import mock

import numpy as np
import pytest
import torch

from oracle import x3d_oracle as O
from oracle import x3d_train_oracle as TO
from tests import mixed_oracle as MO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "x3d_tf_b200", "csrc")
NEW_SYMBOLS = ("x3d_bf16_round", "x3d_pw_bf16_train_fwd", "x3d_pw_wgrad_bf16")


def _bits(u):
    return np.asarray(u, np.uint32).view(np.float32)


def test_rounding_equals_torch_bfloat16():
    rng = np.random.default_rng(0)
    vals = [rng.normal(size=4000) * 10.0 ** rng.integers(-30, 30, size=4000)]
    # exact ties (low half 0x8000) with even and odd kept halves, one ulp either side of them, values
    # near the largest bf16 (0x7F7F) and the fp32 maximum, subnormals, signed zeros
    hi = rng.integers(0, 0x7F7F, size=2000, dtype=np.uint32) << 16
    for low in (0x8000, 0x7FFF, 0x8001, 0x0000, 0xFFFF):
        vals.append(_bits(hi | low))
        vals.append(-_bits(hi | low))
    vals.append(_bits([0x7F7F0000, 0x7F7F7FFF, 0x7F7F8000, 0x7F7F8001, 0x7F7FFFFF, 0x7F7E8000,
                       0x00000001, 0x00008000, 0x00018000, 0x007FFFFF, 0x80000000, 0x00000000]))
    x = np.concatenate([np.asarray(v, np.float64) for v in vals])
    want = torch.from_numpy(x.astype(np.float32)).to(torch.bfloat16).double().numpy()
    got = MO.bf16_rne(x)
    assert np.array_equal(got, want, equal_nan=False)
    assert np.isinf(MO.bf16_rne(_bits([0x7F7F8000]))).all()              # the tie above the max rounds to inf
    assert MO.bf16_rne(_bits([0x7F7F7FFF]))[0] == float(_bits([0x7F7F0000])[0])


def test_rounded_matmul_hand_worked():
    """2x3 . 3x2 with operands off the bf16 grid: 1 + 2^-8 is a tie that rounds to the even 1, 1 + 3*2^-8
    a tie that rounds up to 1 + 2^-6, 1 + 3*2^-9 rounds up to 1 + 2^-7."""
    e8, e9 = 2.0 ** -8, 2.0 ** -9
    x = torch.tensor([[1 + e8, 2.0, -1.0], [0.5, 1 + 3 * e8, 3.0]], dtype=torch.float64, requires_grad=True)
    w = torch.tensor([[1.0, 0.0], [0.0, 1 + 3 * e9], [1.0, 2.0]], dtype=torch.float64, requires_grad=True)
    y = MO.RoundedMatmul.apply(x, w)
    np.testing.assert_array_equal(y.detach().numpy(), [[0.0, 0.015625], [3.5, 7.0235595703125]])
    dy = torch.tensor([[1 + e8, 0.0], [0.0, 1.0]], dtype=torch.float64)
    y.backward(dy)
    np.testing.assert_array_equal(x.grad.numpy(), [[1.0, 0.0, 1.0], [0.0, 1.0078125, 2.0]])
    np.testing.assert_array_equal(w.grad.numpy(), [[1.0, 0.5], [2.0, 1.015625], [-1.0, 3.0]])


def _small_step(**kw):
    from x3d_tf_b200.arch import build_arch
    from x3d_tf_b200.config import get_config
    from x3d_tf_b200.synth import synthetic_clips, synthetic_weights
    cfg = get_config("X3D_XS")
    W = synthetic_weights(build_arch(cfg), seed=3)
    x = synthetic_clips(2, 4, 32, 32, cfg.DATA.MEAN, cfg.DATA.STD, seed=4)
    labels = np.array([3, 17], np.int32)
    mask = ((np.random.default_rng(5).random((2, 2048)) >= 0.5) * 2.0).astype(np.float32)
    return W, O.OracleSpec.from_cfg(cfg), x, labels, dict(lr=0.05, weight_decay=5e-5, dropout_mask=mask, **kw)


def test_option_off_is_the_oracle_and_restatement_is_faithful():
    W, spec, x, labels, kw = _small_step()
    ref = TO.train_step(W, spec, x, labels, **kw)
    off = MO.train_step(W, spec, x, labels, gemm_round=False, **kw)
    assert off["loss"] == ref["loss"]
    for part in ("logits",):
        assert np.array_equal(off[part], ref[part])
    for d in ("grads", "weights", "velocity"):
        assert ref[d].keys() == off[d].keys()
        for k in ref[d]:
            assert np.array_equal(off[d][k], ref[d][k]), (d, k)
    # the restated forward with the rounding replaced by the identity is the oracle's forward, up to the
    # float64 reordering of the 1x1x1 convs as matrix products
    with mock.patch.object(MO, "_r", lambda t, dev=None: t):
        same = MO.train_step(W, spec, x, labels, **kw)
    assert abs(same["loss"] - ref["loss"]) < 1e-12
    for k, g in ref["grads"].items():
        assert np.abs(same["grads"][k] - g).max() <= 1e-9 * max(np.abs(g).max(), 1e-30), k
    # ... and with the rounding the step is measurably different
    mixed = MO.train_step(W, spec, x, labels, **kw)
    assert abs(mixed["loss"] - ref["loss"]) > 1e-7


def test_new_symbols_are_declared_bound_and_validate_arguments():
    from x3d_tf_b200 import _lib
    from x3d_tf_b200 import build as b
    b.build()
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "x3d_b200.h")).read(), flags=re.S)
    h = ctypes.CDLL(_lib.LIB_PATH)
    for n in NEW_SYMBOLS:
        assert re.search(r"\b%s\s*\(" % n, src), n
        assert hasattr(h, n) and n in _lib.SIGNATURES, n
    L = _lib.lib()
    assert L.x3d_bf16_round(None, None, 4, 4, 4, 0, None) == -1 and b"bad argument" in L.x3d_last_error()
    assert L.x3d_pw_bf16_train_fwd(None, None, None, None, 128, 32, 32, 32, 32, 0, None, None) == -1
    assert b"null" in L.x3d_last_error()
    assert L.x3d_pw_wgrad_bf16(None, None, None, 128, 32, 32, 32, 32, 0, 0, 0, 0, 0, 1, None) == -1
    buf = (ctypes.c_float * 64)()
    dw = (ctypes.c_double * 64)()
    p = ctypes.addressof(buf) // 16 * 16 + 16 if ctypes.addressof(buf) % 16 else ctypes.addressof(buf)
    assert L.x3d_pw_wgrad_bf16(p, p, ctypes.addressof(dw), 4, 6, 4, 6, 4, 0, 0, 0, 0, 0, 1, None) == -1
    assert b"multiples of 4" in L.x3d_last_error()


def test_train_driver_selects_the_mixed_policy(monkeypatch):
    from x3d_tf_b200 import runtime
    from x3d_tf_b200 import train as T
    from x3d_tf_b200.config import get_config
    from x3d_tf_b200.training import X3DTrainer
    a = T.build_parser().parse_args(["--config", "X3D_XS", "--model_dir", "m", "--synthetic", "4",
                                     "--mixed_precision"])
    assert a.mixed_precision
    assert not T.build_parser().parse_args(["--config", "X3D_XS", "--model_dir", "m"]).mixed_precision
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    assert runtime.get_precision(a.mixed_precision) == "mixed_bfloat16"
    assert runtime.policy_dtype("mixed_bfloat16") == "bfloat16"
    assert runtime.get_precision(False) == "float32"
    with pytest.raises(ValueError, match="precision"):
        X3DTrainer(get_config("X3D_XS"), precision="mixed_float16")


def _compile(src, out, tmp_path):
    cmd = ["/usr/local/cuda/bin/nvcc" if os.path.exists("/usr/local/cuda/bin/nvcc") else "nvcc",
           "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "--expt-relaxed-constexpr",
           "-Xptxas", "-v", "-cubin", "-o", str(tmp_path / out), os.path.join(CSRC, src)]
    return subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)


def _sass(cubin, func_pattern):
    txt = subprocess.run(["cuobjdump" if not os.path.exists("/usr/local/cuda/bin/cuobjdump")
                          else "/usr/local/cuda/bin/cuobjdump", "-sass", str(cubin)],
                         check=True, capture_output=True, text=True).stdout
    funcs = re.split(r"\n\s*Function : ", txt)
    return [f for f in funcs if re.match(func_pattern, f)]


def test_new_kernels_compile_to_tensor_core_code_without_spills(tmp_path):
    jobs = {"pw": _compile("x3d_pw_tf32_tc.cu", "pw.cubin", tmp_path),
            "train": _compile("x3d_train.cu", "train.cubin", tmp_path)}
    logs = {k: j.communicate()[0] for k, j in jobs.items()}
    for k, j in jobs.items():
        assert j.returncode == 0, logs[k]
    for k, kernel in (("pw", "pw_bf16_train_tc_kernel"), ("train", "pw_wgrad_bf16_kernel"),
                      ("pw", "bf16_round_kernel")):
        blocks = re.findall(r"Compiling entry function '(\S*%s\S*)'.*?\n(.*?\n.*?)\n" % kernel, logs[k])
        assert blocks, kernel
        for name, props in blocks:
            assert "0 bytes spill stores, 0 bytes spill loads" in props, (name, props)
    fwd = _sass(tmp_path / "pw.cubin", r"\S*pw_bf16_train_tc_kernel")
    assert len(fwd) == 1 and "UTCHMMA" in fwd[0]
    wg = _sass(tmp_path / "train.cubin", r"\S*pw_wgrad_bf16_kernel")
    assert len(wg) == 4 and all("HMMA.16816.F32.BF16" in f for f in wg)
