"""CPU: host-side logic of the product (API surface, crops, sharding) against the oracle."""
import json
import os

import numpy as np
import pytest
import torch

import feartracker_b200 as fb
from feartracker_b200 import image_ops, sharding
from oracle import fear_oracle as fo
from tests.helpers import GOLDEN, load_full_state


def test_fearnet_state_dict_is_checkpoint_compatible():
    net = fb.FEARNet(**fb.FEAR_XS_MODEL_KWARGS)
    with open(os.path.join(GOLDEN, "state_dict_keys.json")) as f:
        keys = json.load(f)
    sd = net.state_dict()
    assert set(sd) == set(keys) and len(sd) == 520
    for k, (shape, dtype) in keys.items():
        assert list(sd[k].shape) == shape and str(sd[k].dtype) == "torch." + dtype, k
    net.load_state_dict(load_full_state(), strict=True)
    assert net.search_size == 256 and net.max_layer == 4 and net.grid_x.dtype == torch.float64
    assert net.encoder.encoder_channels["layer1"] == 112 and len(net.encoder.stages) == 5


def test_fearnet_constructor_contract():
    with pytest.raises(AssertionError):
        fb.FEARNet(backbone="x", img_size=256, max_layer=5)
    with pytest.raises(NotImplementedError):
        fb.FEARNet(backbone="x", img_size=256)  # reference defaults (towernum=4, max_layer=3) are not FEAR-XS
    fb.FEARNet(backbone="custom_fbnet", img_size=256, towernum=2, max_layer=4, growth_factor=1.2, num_filters=32)


def test_eval_has_no_cpu_path_and_containers_never_compute():
    net = fb.FEARNet(**fb.FEAR_XS_MODEL_KWARGS).eval()
    with pytest.raises(RuntimeError, match="no CPU path"):
        net((torch.zeros(1, 3, 128, 128), torch.zeros(1, 3, 256, 256)))
    with pytest.raises(RuntimeError, match="no CPU path"):
        net.get_features(torch.zeros(1, 3, 128, 128))
    with pytest.raises(RuntimeError, match="no CPU path"):
        net.connect_model(torch.zeros(1, 256, 16, 16), torch.zeros(1, 256, 8, 8), torch.zeros(1, 256, 8, 8))
    with pytest.raises(RuntimeError):
        net.encoder(torch.zeros(1, 3, 32, 32))  # parameter containers never compute


def test_train_mode_forward_matches_reference_training_step():
    """f3: in train() mode FEARNet.forward is a differentiable torch graph over the same parameters (BatchNorm batch
    statistics, autograd) -- what FEARLightningModel.forward calls (reference fear_lightning_model.py:60-62).
    Golden: the reference's own FEARNet in train() mode, one forward + backward (oracle/make_golden_r2.py)."""
    g = np.load(os.path.join(GOLDEN, "train_step.npz"))
    net = fb.FEARNet(**fb.FEAR_XS_MODEL_KWARGS)
    net.load_state_dict(load_full_state(), strict=True)
    net.train()
    gen = torch.Generator().manual_seed(5)
    z = torch.randn(2, 3, 128, 128, generator=gen)
    x = torch.randn(2, 3, 256, 256, generator=gen)
    out = net((z, x))
    R, C = fo.TARGET_REGRESSION_LABEL_KEY, fo.TARGET_CLASSIFICATION_KEY
    np.testing.assert_allclose(out[R].detach().numpy(), g["reg"], rtol=2e-4, atol=1e-6)
    np.testing.assert_allclose(out[C].detach().numpy(), g["cls"], rtol=2e-4, atol=1e-5)
    loss = out[R].log().mean() + out[C].mean()
    assert abs(float(loss) - float(g["loss"])) < 1e-4
    loss.backward()
    grads = {k: float(p.grad.norm()) for k, p in net.named_parameters() if p.grad is not None}
    assert sorted(grads) == g["grad_names"].tolist()
    # gradient norms in float64: in float32 the biases of convolutions that feed a train-mode BatchNorm (exact
    # gradient zero) hold rounding noise that differs between host CPUs
    g64 = np.load(os.path.join(GOLDEN, "train_step_fp64.npz"))
    net64 = fb.FEARNet(**fb.FEAR_XS_MODEL_KWARGS)
    net64.load_state_dict(load_full_state(), strict=True)
    net64 = net64.double().train()
    out64 = net64((z.double(), x.double()))
    (out64[R].log().mean() + out64[C].mean()).backward()
    grads64 = {k: float(p.grad.norm()) for k, p in net64.named_parameters() if p.grad is not None}
    assert sorted(grads64) == g64["grad_names"].tolist() == g["grad_names"].tolist()
    np.testing.assert_allclose([grads64[k] for k in sorted(grads64)], g64["grad_norms"], rtol=2e-3, atol=1e-7)
    sd = net.state_dict()
    for key in g.files:
        if key.startswith("bn__"):  # running statistics were updated with the batch statistics
            np.testing.assert_allclose(sd[key[4:]].numpy(), g[key], rtol=1e-4, atol=1e-6)
    # the 4-tuple of BoxTower.forward and track() also work in train mode; eval() switches back to the library
    zf, xf = net.get_features(z), net.get_features(x)
    assert len(net.connect_model(xf, zf)) == 4 and net.track(x, zf)[C].shape == (2, 1, 16, 16)
    net.eval()
    with pytest.raises(RuntimeError, match="no CPU path"):
        net((z, x))


def test_smooth_postprocess_matches_reference():
    """f4: the ``smooth: true`` post-processing (penalty, cosine window, size smoothing; reference
    base_tracker.py:126-205) on maps / prev_size recorded from the reference tracker itself."""
    g = np.load(os.path.join(GOLDEN, "smooth_tracker.npz"))
    trk = fb.FEARTracker(None, cuda_id="cpu", smooth=True, **fb.FEAR_XS_TRACKER_KWARGS)
    oracle = fo.OracleTracker({"neck.downsample.0.weight": torch.zeros(1)}, dict(fo.TRACKER_CONFIG, smooth=True))
    for i in range(len(g["frames"])):
        trk.tracking_state.prev_size = g["prev_size"][i]
        maps = {fo.TARGET_REGRESSION_LABEL_KEY: torch.from_numpy(g["reg"][i:i + 1]),
                fo.TARGET_CLASSIFICATION_KEY: torch.from_numpy(g["cls"][i:i + 1])}
        box, score = trk._postprocess(maps)
        np.testing.assert_allclose(box, g["box"][i], rtol=1e-12, atol=1e-12)
        assert np.float32(score) == g["score"][i]
        oracle.prev_size = g["prev_size"][i]
        obox, oscore, coords = oracle.postprocess(maps)
        assert list(coords) == g["coords"][i].tolist() and np.array_equal(obox, g["box"][i])


def test_device_crop_formula_matches_cv2_resize():
    """f1: the integer arithmetic crop_resize_u8_kernel runs (numpy model image_ops.crop_resize_reference + the
    host-computed coefficient tables) == copyMakeBorder + cv2.resize(INTER_LINEAR) of get_extended_crop, bit for bit,
    including windows that leave the frame, up- and down-scaling and the 1:1 case."""
    rng = np.random.default_rng(5)
    frame = rng.integers(0, 256, (256, 480, 3), dtype=np.uint8)
    mean = np.mean(frame, axis=(0, 1))
    boxes = [[163, 53, 45, 174], [0, 0, 30, 40], [450, 230, 30, 26], [200, 100, 3, 3], [-5, -7, 50, 60],
             [10, 200, 400, 56], [100, 100, 64, 64], [300, 20, 17, 201], [177, 64, 128, 128]]
    for box in boxes:
        box = image_ops.clamp_bbox(box, frame.shape)
        for size, off, pad in ((128, 0.2, None), (256, 2, mean), (256, 0.5, mean)):
            want = image_ops.extended_crop(frame, box, size, off, pad)
            params, inbox, ctx = image_ops.crop_params(box, size, off, mean if pad is None else pad)
            assert params.dtype == np.int32 and params.size == 8 + 6 * size
            got = image_ops.crop_resize_reference(frame, params, size)
            assert np.array_equal(got, want[0]), (box, size, off)
            np.testing.assert_allclose(inbox, want[1], rtol=0, atol=1e-12)
            assert list(ctx) == list(want[2])


def test_hydra_style_composer_and_reference_module_names(tmp_path):
    """f2: defaults list, ``# @package _global_``, ``${...}`` interpolation, overrides, ``_target_`` instantiate and
    the model_training.* / hydra / fire / imageio stand-ins (reference utils/hydra.py:33-39, demo_video.py:1-19)."""
    import sys

    from feartracker_b200 import compat

    (tmp_path / "model").mkdir()
    (tmp_path / "extra").mkdir()
    (tmp_path / "main.yaml").write_text(
        "hydra:\n  run:\n    dir: ${now:%Y}\ntop: 1\ndefaults:\n  - model: small\n  - extra: glob\n")
    (tmp_path / "model" / "small.yaml").write_text("_target_: collections.OrderedDict\nstride: 2\nname: m${top}\n")
    (tmp_path / "model" / "big.yaml").write_text("_target_: collections.OrderedDict\nstride: 4\n")
    (tmp_path / "extra" / "glob.yaml").write_text("# @package _global_\nbatch: {train: 8}\nuses: ${model.stride}\n")
    cfg = compat.load_hydra_config_from_path(str(tmp_path), "main")
    assert cfg == {"top": 1, "model": {"_target_": "collections.OrderedDict", "stride": 2, "name": "m1"},
                   "batch": {"train": 8}, "uses": 2}
    cfg = compat.load_hydra_config_from_path(str(tmp_path), "main", overrides=["model=big", "batch.train=3", "top=7"])
    assert cfg["model"]["stride"] == 4 and cfg["uses"] == 4 and cfg["batch"]["train"] == 3 and cfg["top"] == 7
    assert dict(compat.instantiate(cfg["model"], extra=5)) == {"stride": 4, "extra": 5}

    ours = os.path.join(os.path.dirname(os.path.dirname(GOLDEN)), "feartracker_b200", "config")
    cfg = compat.load_hydra_config_from_path(ours, "fear_tracker")
    assert cfg["tracker"]["stride"] == cfg["model"]["stride"] == 2
    assert {k: v for k, v in cfg["tracker"].items() if k != "_target_"} == fb.FEAR_XS_TRACKER_KWARGS
    saved = {k: sys.modules.get(k) for k in list(sys.modules)}
    try:
        names = compat.install()
        if "model_training.model.fear_net" in names:  # not shadowed by a real reference package on the path
            from hydra.utils import instantiate
            from model_training.model.fear_net import FEARNet
            from model_training.tracker.fear_tracker import FEARTracker

            assert FEARNet is fb.FEARNet and FEARTracker is fb.FEARTracker
            model = instantiate(dict(cfg["model"], _target_="model_training.model.fear_net.FEARNet"))
            tracker = instantiate(dict(cfg["tracker"], _target_="model_training.tracker.fear_tracker.FEARTracker"),
                                  model=model)
            assert isinstance(tracker, fb.FEARTracker) and tracker.tracking_config["instance_size"] == 256
    finally:
        for k in list(sys.modules):
            if k not in saved:
                del sys.modules[k]


def test_load_from_lighting_semantics(tmp_path):
    """utils/torch.py:11-24: ``model.`` prefix stripped, strict load, strict=False skips mismatching tensors."""
    net = fb.FEARNet(**fb.FEAR_XS_MODEL_KWARGS)
    sd = load_full_state()
    ck = {"state_dict": {"model." + k: v for k, v in sd.items()}}
    ck["state_dict"]["criterion.weight"] = torch.zeros(3)
    path = str(tmp_path / "ck.ckpt")
    torch.save(ck, path)
    fb.load_from_lighting(net, path)
    assert torch.equal(net.state_dict()["neck.downsample.0.weight"], sd["neck.downsample.0.weight"])
    ck["state_dict"]["model.neck.downsample.0.weight"] = torch.zeros(7, 7)
    torch.save(ck, path)
    with pytest.raises(RuntimeError):
        fb.load_from_lighting(net, path)
    with pytest.warns(UserWarning, match="skipped 1 tensors"):
        fb.load_from_lighting(net, path, strict=False)


def test_crop_helpers_match_oracle():
    rng = np.random.default_rng(0)
    frame = rng.integers(0, 256, (256, 480, 3), dtype=np.uint8)
    mean = np.mean(frame, axis=(0, 1))
    boxes = [[163, 53, 45, 174], [0, 0, 30, 40], [450, 230, 30, 26], [200, 100, 3, 3], [-5, -7, 50, 60],
             [10, 200, 400, 56]]
    for box in boxes:
        box = image_ops.clamp_bbox(box, frame.shape)
        assert list(box) == list(fo.clamp_bbox(box, frame.shape))
        for size, off, pad in ((128, 0.2, None), (256, 2, mean)):
            a = image_ops.extended_crop(frame, box, size, off, pad)
            b = fo.get_extended_crop(frame, box, size, off, pad)
            np.testing.assert_array_equal(a[0], b[0])
            np.testing.assert_allclose(a[1], b[1], rtol=0, atol=1e-12)
            np.testing.assert_array_equal(a[2], b[2])
    crop = rng.integers(0, 256, (256, 256, 3), dtype=np.uint8)
    np.testing.assert_array_equal(image_ops.normalize(crop), fo.normalize_image(crop))
    for pred in ([106.2, 88.3, 44.6, 49.1], [0.4999, 255.5, 1.0, 2.5]):
        ctx = [100, 20, 225, 225]
        assert image_ops.rescale_bbox(np.array(pred), ctx, 256) == fo.rescale_bbox(np.array(pred), ctx, 256)


def test_tracker_constructs_without_gpu_and_fails_loudly():
    net = fb.FEARNet(**fb.FEAR_XS_MODEL_KWARGS).eval()
    trk = fb.FEARTracker(net, cuda_id="cpu", **fb.FEAR_XS_TRACKER_KWARGS)
    assert trk.window.shape == (16, 16) and trk.box_coder.grid_x.shape == (1, 16, 16)
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):
            trk.initialize(np.zeros((64, 64, 3), np.uint8), np.array([10, 10, 20, 20]))


def test_shard_range_partitions():
    for total, world in ((2048, 8), (10, 4), (3, 8), (256, 1)):
        spans = [sharding.shard_range(total, r, world) for r in range(world)]
        assert spans[0][0] == 0 and spans[-1][1] == total
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        sizes = [e - b for b, e in spans]
        assert max(sizes) - min(sizes) <= 1
