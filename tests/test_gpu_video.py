"""GPU: clips built from decoded videos by x3d_video_clips_u8 are byte-identical to the numpy
restatement (tests/video_oracle.py), and every consumer (X3D.evaluate / predict, X3D.fit, the eval
driver) gives exactly what it gives on the oracle's clips.  Every kernel case writes >= 100 k
output bytes: about 0.4 % of a random resize's values sit just below an integer, so a contracted
multiply-add would show."""
import numpy as np
import pytest
import torch

from tests import video_oracle as VO
from x3d_tf_b200 import video as V
from x3d_tf_b200.arch import build_arch
from x3d_tf_b200.config import get_config
from x3d_tf_b200.synth import synthetic_weights

pytestmark = pytest.mark.gpu


def _videos(shapes, seed):
    rng = np.random.default_rng(seed)
    return [rng.integers(0, 256, size=s, dtype=np.uint8) for s in shapes]


def _run(videos, plan):
    b = V.pack(videos, plan)
    got = b.clips("cuda").cpu().numpy()
    want = np.stack([VO.train_clip(videos[plan.video[n]], plan.frames[n], plan.desc[n], plan.S)
                     for n in range(plan.frames.shape[0])])
    assert got.shape == want.shape == plan.shape and got.nbytes >= 100_000
    return got, want


def _eval(shapes, T, views, crops, size, seed):
    videos = _videos(shapes, seed)
    return _run(videos, V.eval_plan([v.shape for v in videos], T, views, crops, size))


def _train(shapes, T, rate, jitter, S, seed, flip=None):
    videos = _videos(shapes, seed)
    plan = V.train_plan([v.shape for v in videos], T, rate, jitter, S, V.train_rng(seed, 0))
    if flip is not None:
        plan.desc[:, 6] = flip
    return _run(videos, plan)


@pytest.mark.parametrize("case", [
    "downscale_360x480", "upscale_100x140", "portrait_odd", "s16", "s356", "flip0", "flip1", "f_lt_t", "ragged3"])
def test_video_clips_byte_identical_to_oracle(case):
    got, want = {
        "downscale_360x480": lambda: _eval([(20, 360, 480, 3)], 4, 2, 3, 128, 1),          # 256 x 170 -> crops
        "upscale_100x140": lambda: _train([(30, 100, 140, 3)], 4, 5, (256, 320), 224, 2),
        "portrait_odd": lambda: _eval([(9, 481, 359, 3)], 4, 1, 3, 182, 3),                 # S % 4 == 2
        "s16": lambda: _eval([(40, 37, 53, 3)], 16, 10, 1, 16, 4),
        "s356": lambda: _eval([(5, 400, 601, 3)], 2, 1, 1, 356, 5),
        "flip0": lambda: _train([(12, 130, 97, 3)], 4, 3, (120, 150), 96, 6, flip=0),
        "flip1": lambda: _train([(12, 130, 97, 3)], 4, 3, (120, 150), 96, 6, flip=1),
        "f_lt_t": lambda: _train([(3, 90, 120, 3)], 16, 5, (80, 100), 64, 7),               # loops the video
        "ragged3": lambda: _train([(50, 360, 480, 3), (7, 100, 140, 3), (13, 241, 179, 3)], 8, 5,
                                  (160, 200), 144, 8),
    }[case]()
    assert np.array_equal(got, want), f"{(got != want).sum()} of {got.size} bytes differ"


def test_flip_mirrors_the_crop():
    got0, _ = _train([(12, 130, 97, 3)], 4, 3, (120, 150), 96, 6, flip=0)
    got1, _ = _train([(12, 130, 97, 3)], 4, 3, (120, 150), 96, 6, flip=1)
    assert np.array_equal(got1, got0[:, :, :, ::-1, :])


def _model(dtype, views=2):
    from x3d_tf_b200 import model as M
    M.reset_block_counters()
    cfg = get_config("X3D_XS", freeze=False)
    cfg.TEST.NUM_TEMPORAL_VIEWS, cfg.TEST.NUM_SPATIAL_CROPS = views, 1
    cfg.freeze()
    m = M.X3D(cfg, dtype=dtype)
    m.set_weights_dict(synthetic_weights(build_arch(cfg), seed=21))
    return m.compile(top_k=5), cfg


@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
def test_evaluate_video_batches_equals_oracle_clips(dtype):
    """Three VideoBatches (ragged last one, videos of different sizes and lengths) through
    X3D.evaluate == the same evaluate over the oracle's uint8 clips, to the bit."""
    m, cfg = _model(dtype)
    shapes = [[(20, 120, 160, 3), (9, 200, 170, 3), (31, 90, 100, 3)],
              [(6, 160, 160, 3), (40, 240, 320, 3), (12, 181, 163, 3)],
              [(17, 144, 256, 3), (5, 170, 120, 3)]]
    rng = np.random.default_rng(9)
    vb, oracle = [], []
    for i, group in enumerate(shapes):
        videos = _videos(group, 100 + i)
        labels = rng.integers(0, 400, size=len(group)).astype(np.int32)
        vb.append((V.eval_batch(videos, cfg), labels))
        clips = np.concatenate([VO.eval_clips(v, cfg.DATA.TEMP_DURATION, 2, 1, cfg.DATA.TEST_CROP_SIZE) for v in videos])
        oracle.append((clips, labels))
    want = m.evaluate(oracle)
    got = m.evaluate(vb)
    assert got == want and got["videos"] == 8
    # predict alternating both kinds of batch of the same shape shares one graph and its buffers
    seq = [vb[0][0], oracle[1][0], vb[1][0], oracle[0][0]]
    outs = list(m.predict(seq))
    ref = list(m.predict([oracle[0][0], oracle[1][0], oracle[1][0], oracle[0][0]]))
    assert all(torch.equal(a, b) for a, b in zip(outs, ref))


def test_eval_driver_decoded_videos(tmp_path):
    from x3d_tf_b200 import eval as E
    from x3d_tf_b200 import model as M
    cfg = get_config("X3D_XS")
    M.reset_block_counters()
    m = M.X3D(cfg, dtype="bfloat16")
    m.set_weights_dict(synthetic_weights(build_arch(cfg), seed=77))
    m.save_weights(str(tmp_path / "ckpt-1"))
    (tmp_path / "checkpoint").write_text('model_checkpoint_path: "ckpt-1"\nall_model_checkpoint_paths: "ckpt-1"\n')
    videos = _videos([(40, 180, 240, 3), (9, 240, 180, 3), (25, 161, 163, 3)], 12)
    labels = [3, 200, 17]
    lines = []
    for i, v in enumerate(videos):
        np.save(tmp_path / f"v{i}.npy", v)
        lines.append(f"v{i}.npy {labels[i]}")
    (tmp_path / "list.txt").write_text("\n".join(lines) + "\n")
    T, views, crops, S = (cfg.DATA.TEMP_DURATION, cfg.TEST.NUM_TEMPORAL_VIEWS, cfg.TEST.NUM_SPATIAL_CROPS,
                          cfg.DATA.TEST_CROP_SIZE)
    vpb = max(cfg.TEST.BATCH_SIZE // (views * crops), 1)
    oracle = [(np.concatenate([VO.eval_clips(v, T, views, crops, S) for v in videos[i:i + vpb]]),
               np.asarray(labels[i:i + vpb], np.int32)) for i in range(0, 3, vpb)]
    want = m.compile().evaluate(oracle)
    got = E.run(["--cfg", "X3D_XS", "--model_folder", str(tmp_path), "--test_file_pattern",
                 str(tmp_path / "list.txt"), "--decoded_videos"])
    assert got == want and got["videos"] == 3


def test_fit_on_video_batches_equals_trainer_on_oracle_clips():
    """Two training steps from VideoBatches (random start, scale jitter, crop, flip on the device)
    leave bit-identical losses and weights to the trainer fed the oracle's clips of the same plans."""
    from x3d_tf_b200 import model as M
    from x3d_tf_b200 import ops
    from x3d_tf_b200.training import X3DTrainer
    cfg = get_config("X3D_XS", freeze=False)
    cfg.NETWORK.DROPOUT_RATE = 0.0
    cfg.TEST.NUM_TEMPORAL_VIEWS, cfg.TEST.NUM_SPATIAL_CROPS = 1, 1
    cfg.freeze()
    W = synthetic_weights(build_arch(cfg), seed=5)
    rng = V.train_rng(31, 0)
    data, oracle = [], []
    for step in range(2):
        videos = _videos([(30, 240, 320, 3), (6, 200, 150, 3)], 40 + step)
        plan = V.train_plan([v.shape for v in videos], cfg.DATA.TEMP_DURATION, cfg.DATA.FRAME_RATE,
                            cfg.DATA.TRAIN_JITTER_SCALES, cfg.DATA.TRAIN_CROP_SIZE, rng)
        labels = np.array([7 + step, 311 - step], np.int32)
        data.append((V.pack(videos, plan), labels))
        oracle.append((np.stack([VO.train_clip(videos[n], plan.frames[n], plan.desc[n], plan.S) for n in range(2)]),
                       labels))
    M.reset_block_counters()
    m = M.X3D(cfg)
    m.set_weights_dict(W)
    hist = m.fit(data, epochs=1, lr_schedule=lambda e: 0.01)
    tr = X3DTrainer(cfg).load(W)
    tot = torch.zeros((), dtype=torch.float64, device="cuda")
    for c, l in oracle:
        x = ops.normalize_u8(torch.from_numpy(c).cuda(), tuple(cfg.DATA.MEAN), tuple(cfg.DATA.STD), torch.float32)
        tot += tr.step(x, torch.from_numpy(l).cuda(), 0.01).double().mean()
    torch.cuda.synchronize()
    assert hist["loss"][0] == float(tot / 2)
    Wt, Wm = tr.weights(), m.named_variables()
    assert all(np.array_equal(Wt[k], Wm[k]) for k in Wt)
    assert not np.array_equal(Wm["fc2/kernel"], W["fc2/kernel"])
