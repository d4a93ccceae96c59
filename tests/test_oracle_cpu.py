"""CPU tests: the oracle restatement against the golden vectors recorded from the reference's
own source (oracle/make_golden*.py)."""
import hashlib

import numpy as np
import torch

from oracle import fear_oracle as fo
from tests.helpers import assert_maps_close, golden, load_full_state

R, C = fo.TARGET_REGRESSION_LABEL_KEY, fo.TARGET_CLASSIFICATION_KEY


def test_state_fixture_complete(state_dict):
    full = load_full_state()
    assert len(full) == 520
    assert set(fo.hot_path_keys(full)) == set(state_dict)
    live = sum(v.numel() for k, v in state_dict.items() if "running_" not in k)
    assert live == 1370194  # SURVEY.md appendix A


def test_seed0_maps_fp32_bit_exact(state_dict):
    """C1: FEARNet.forward on the seed-0 randn pair reproduces the reference's fp32 output."""
    g = golden("maps_seed0.npz")
    torch.manual_seed(0)
    z = torch.randn(1, 3, 128, 128)
    x = torch.randn(1, 3, 256, 256)
    out = fo.forward(state_dict, z, x)
    # same torch build + same op sequence => bit-identical on the build container; allow fp32
    # noise elsewhere (different oneDNN kernels on another host CPU)
    assert_maps_close(out[R].numpy(), g["reg32"], "reg", tol=1e-4)
    assert_maps_close(out[C].numpy(), g["cls32"], "cls", tol=1e-4)
    bbox, coords = fo.decode(out[R], out[C])
    assert coords == [tuple(g["coords"][0])] == [(6, 8)]
    np.testing.assert_allclose(bbox.numpy(), g["bbox"], rtol=1e-5)
    assert bbox.dtype == torch.float64


def test_seed0_maps_fp64(state_dict):
    g = golden("maps_seed0.npz")
    torch.manual_seed(0)
    z = torch.randn(1, 3, 128, 128).double()
    x = torch.randn(1, 3, 256, 256).double()
    out = fo.forward(fo.to_dtype(state_dict, torch.float64), z, x)
    np.testing.assert_allclose(out[R].numpy(), g["reg64"], rtol=1e-10)
    np.testing.assert_allclose(out[C].numpy(), g["cls64"], rtol=1e-9, atol=1e-11)


def test_synthetic_and_template_broadcast(state_dict):
    g = golden("synthetic_b4.npz")
    sd64 = fo.to_dtype(state_dict, torch.float64)
    zt, xt, _, _ = fo.synthetic_crops(4)
    zf = fo.get_features(sd64, zt.double())
    np.testing.assert_allclose(zf.numpy(), g["zf64"], rtol=1e-9, atol=1e-11)
    out = fo.track(sd64, xt.double(), zf)
    np.testing.assert_allclose(out[R].numpy(), g["reg64"], rtol=1e-9)
    out1 = fo.track(sd64, xt.double(), zf[:1])  # Bz = 1 broadcasts over B (blocks.py:123)
    np.testing.assert_allclose(out1[R].numpy(), g["reg64_bz1"], rtol=1e-9)
    np.testing.assert_allclose(out1[R][0].numpy(), out[R][0].numpy(), rtol=1e-12)
    bbox, coords = fo.decode(out[R], out[C])
    assert [list(c) for c in coords] == g["coords"].tolist()
    np.testing.assert_allclose(bbox.numpy(), g["bbox"], rtol=1e-9)


def test_decode_tie_break_and_grid():
    gx, gy = fo.make_grid(16, 16, 256)
    assert gx.dtype == torch.float64 and gx.shape == (1, 16, 16)
    assert gx[0, 0, 0] == 0 and gx[0, 0, 15] == 240 and gy[0, 15, 0] == 240
    cls = torch.zeros(2, 1, 16, 16)
    cls[0, 0, 3, 5] = cls[0, 0, 9, 1] = 2.0  # tie -> first (row-major) wins
    cls[1, 0, 15, 15] = 1.0
    reg = torch.ones(2, 4, 16, 16)
    bbox, coords = fo.decode(reg, cls)
    assert coords == [(3, 5), (15, 15)]
    assert bbox[0].tolist() == [5 * 16 - 1.0, 3 * 16 - 1.0, 2.0, 2.0]


def test_teacher_forced_video_frames(state_dict):
    """C3 (teacher-forced): recorded search crops -> same maps, argmax and integer boxes."""
    g = golden("video_teacher.npz")
    sd64 = fo.to_dtype(state_dict, torch.float64)
    zf = torch.from_numpy(g["template_features"]).double()
    for i, crop in enumerate(g["search_crops"]):
        out = fo.track(sd64, fo.preprocess_image(crop).double(), zf)
        np.testing.assert_allclose(out[R].numpy(), g["reg64"][i:i + 1], rtol=1e-9)
        np.testing.assert_allclose(out[C].numpy(), g["cls64"][i:i + 1], rtol=1e-9, atol=1e-11)


def test_video_prefix_trajectory(state_dict, golden_dir):
    """C3 (free-running): first 30 frames of the demo clip reproduce the reference trajectory."""
    import os

    g = golden("video_teacher.npz")
    frames = fo.read_video_rgb(os.path.join(golden_dir, "test.mp4"))
    assert frames.shape == (661, 256, 480, 3)
    assert hashlib.sha1(g["trajectory"].tobytes()).hexdigest() == str(g["sha1"])
    trk = fo.OracleTracker(state_dict)
    trk.initialize(frames[0], g["init_bbox"])
    np.testing.assert_allclose(trk.template_features.numpy(), g["template_features"], rtol=1e-4, atol=1e-5)
    for i in range(1, 31):
        box = trk.update(frames[i])["bbox"]
        assert list(box) == g["trajectory"][i - 1].tolist(), i


def test_update_branch_golden(state_dict):
    """BoxTower.forward(search, kernel, update) (blocks.py:174-179) vs the reference's float64 output."""
    g = golden("update_branch.npz")
    sd64 = fo.to_dtype(state_dict, torch.float64)
    zf, xf, uf = (torch.from_numpy(g[k]) for k in ("zf", "xf", "uf"))
    bbox, cls, _, _ = fo.box_tower(sd64, xf, zf, uf)
    np.testing.assert_allclose(bbox.numpy(), g["bbox"], rtol=1e-9)
    np.testing.assert_allclose(cls.numpy(), g["cls"], rtol=1e-9, atol=1e-11)
    plain = fo.box_tower(sd64, xf, zf)
    assert torch.equal(plain[0], bbox) and not torch.equal(plain[1], cls)  # only the cls branch sees `update`


def test_smooth_tracker_prefix_trajectory(state_dict, golden_dir):
    """``smooth: true`` (base_tracker.py:126-205): first 25 frames reproduce the reference trajectory."""
    import os

    g = golden("smooth_tracker.npz")
    frames = fo.read_video_rgb(os.path.join(golden_dir, "test.mp4"))[:26]
    trk = fo.OracleTracker(state_dict, dict(fo.TRACKER_CONFIG, smooth=True))
    trk.initialize(frames[0], g["init_bbox"])
    for i in range(1, 26):
        assert list(trk.update(frames[i])["bbox"]) == g["trajectory"][i - 1].tolist(), i


def test_restatement_equals_reference_source(state_dict):
    """oracle == the reference's own FEARNet on the seed-7 crops, against its outputs recorded by
    oracle/make_golden_restatement.py (which also asserts bit-equality where it runs).  The weight fixture must be
    the checkpoint byte for byte.  fp64 maps to rounding level; fp32 maps within the noise of another host CPU's
    kernels (measured 2e-6 inf-norm, 1.2e-4 element-wise between AVX-512 and AVX2)."""
    g = golden("restatement_seed7.npz")
    assert sorted(state_dict) == g["keys"].tolist()
    for k, digest in zip(g["keys"], g["sha256"]):
        assert hashlib.sha256(state_dict[k].contiguous().numpy().tobytes()).hexdigest() == digest, k
    zt, xt, _, _ = fo.synthetic_crops(2, seed=7)
    mine = fo.forward(fo.to_dtype(state_dict, torch.float64), zt.double(), xt.double())
    np.testing.assert_allclose(mine[R].numpy(), g["reg64"], rtol=1e-10)
    np.testing.assert_allclose(mine[C].numpy(), g["cls64"], rtol=1e-9, atol=1e-11)
    mine = fo.forward(state_dict, zt, xt)
    assert_maps_close(mine[R].numpy(), g["reg32"], "reg fp32", inf_tol=1e-5)
    assert_maps_close(mine[C].numpy(), g["cls32"], "cls fp32", inf_tol=1e-5)
