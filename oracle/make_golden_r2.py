"""Round-2 golden fixtures (TEST INFRASTRUCTURE; run in the build container where /root/reference exists):

    python -m oracle.make_golden_r2

Imports the reference's UNMODIFIED source through ``oracle/ref_shims.py`` and records, after asserting that the
oracle restatement reproduces each of them bit-for-bit:

* ``tests/golden/smooth_tracker.npz``  -- FEARTracker with ``smooth: true`` (reference base_tracker.py:126-205):
  free-running trajectory over the first 120 frames of the demo clip + per-frame post-processing cases
  (maps, prev_size -> box, score) for a host-only test of the product's smoothing code;
* ``tests/golden/update_branch.npz``   -- BoxTower.forward(search, kernel, update) (blocks.py:174-179) in float64
  on the synthetic crops, template batch B and 1;
* ``tests/golden/train_step.npz``      -- FEARNet in train() mode (BatchNorm batch statistics): forward maps,
  gradient norms and the updated running statistics of one step (fear_lightning_model.py:60-62 calls
  ``model.forward`` in training);
* ``tests/golden/train_step_fp64.npz`` -- the gradient norms of the same step in float64.
"""
import os

import numpy as np
import torch

from oracle import fear_oracle as fo
from oracle import ref_shims

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
R, C = fo.TARGET_REGRESSION_LABEL_KEY, fo.TARGET_CLASSIFICATION_KEY
SMOOTH_FRAMES = 120
SMOOTH_CASES = (1, 2, 3, 11, 51, 90, 119)


def _eq(a, b, what):
    assert torch.equal(torch.as_tensor(a), torch.as_tensor(b)), what


def smooth(net, sd32):
    frames = fo.read_video_rgb(ref_shims.REF_VIDEO)[: SMOOTH_FRAMES + 1]
    ref_shims.install()
    from model_training.tracker.fear_tracker import FEARTracker  # reference source

    cfg = dict(ref_shims.REF_TRACKER_KWARGS, smooth=True)
    ref_trk = FEARTracker(model=net, cuda_id="cpu", **cfg)
    mine = fo.OracleTracker(sd32, dict(fo.TRACKER_CONFIG, smooth=True))
    init = np.array(ref_shims.REF_INIT_BBOX)
    ref_trk.initialize(frames[0], init)
    mine.initialize(frames[0], init)
    traj, cases = [], {}
    for i in range(1, len(frames)):
        rb = ref_trk.update(frames[i])["bbox"]
        mb = mine.update(frames[i])["bbox"]
        assert list(rb) == list(mb), (i, rb, mb)
        traj.append(list(map(int, rb)))
        if i in SMOOTH_CASES:
            # replay the post-processing of this frame through the reference's own _postprocess
            ref_trk.tracking_state.prev_size = mine.prev_size
            with torch.no_grad():
                rbox, rscore = ref_trk._postprocess(mine.last_maps)
            mbox, mscore, coords = mine.postprocess(mine.last_maps)
            assert np.array_equal(np.asarray(rbox), np.asarray(mbox)) and float(rscore) == float(mscore)
            cases[i] = (mine.last_maps[R].numpy().copy(), mine.last_maps[C].numpy().copy(),
                        np.asarray(mine.prev_size, dtype=np.float64), np.asarray(mbox, dtype=np.float64),
                        np.float32(mscore), np.array(coords))
    ks = sorted(cases)
    np.savez_compressed(
        os.path.join(OUT, "smooth_tracker.npz"), trajectory=np.array(traj, dtype=np.int64), init_bbox=init,
        frames=np.array(ks), reg=np.concatenate([cases[k][0] for k in ks]), cls=np.concatenate([cases[k][1] for k in ks]),
        prev_size=np.stack([cases[k][2] for k in ks]), box=np.stack([cases[k][3] for k in ks]),
        score=np.array([cases[k][4] for k in ks]), coords=np.stack([cases[k][5] for k in ks]))
    print("smooth: trajectory tail", traj[-1], "cases", ks)


def update_branch(sd64):
    net64 = ref_shims.build_reference_net().double()
    zt, xt, _, _ = fo.synthetic_crops(3)
    zu, _, _, _ = fo.synthetic_crops(3, seed=77)
    with torch.no_grad():
        zf, xf, uf = net64.get_features(zt.double()), net64.get_features(xt.double()), net64.get_features(zu.double())
        ref = net64.connect_model(xf, zf, uf)
        ref1 = net64.connect_model(xf, zf[:1], uf[:1])
    mine = fo.box_tower(sd64, xf, zf, uf)
    for a, b, n in zip(ref, mine, ("bbox", "cls", "cls_dw", "x_reg")):
        _eq(a, b, "update branch " + n)
    np.savez_compressed(os.path.join(OUT, "update_branch.npz"), zf=zf.numpy(), xf=xf.numpy(), uf=uf.numpy(),
                        bbox=ref[0].numpy(), cls=ref[1].numpy(), bbox_b1=ref1[0].numpy(), cls_b1=ref1[1].numpy())
    print("update: cls argmax", ref[1].flatten(1).argmax(1).tolist())


def train_step():
    net = ref_shims.build_reference_net().train()
    g = torch.Generator().manual_seed(5)
    z = torch.randn(2, 3, 128, 128, generator=g)
    x = torch.randn(2, 3, 256, 256, generator=g)
    out = net((z, x))
    loss = out[R].log().mean() + out[C].mean()
    loss.backward()
    grads = {k: float(p.grad.norm()) for k, p in net.named_parameters() if p.grad is not None}
    bn = {k: v.detach().numpy().copy() for k, v in net.state_dict().items()
          if k.endswith(("xif0_0.bn.running_mean", "xif4_7.pwl.bn.running_var", "neck.downsample.1.running_mean"))}
    np.savez_compressed(os.path.join(OUT, "train_step.npz"), reg=out[R].detach().numpy(), cls=out[C].detach().numpy(),
                        loss=np.float64(loss.item()), grad_names=np.array(sorted(grads)),
                        grad_norms=np.array([grads[k] for k in sorted(grads)]), **{"bn__" + k: v for k, v in bn.items()})
    print("train: loss", float(loss), "params with grad", len(grads))


def train_step_fp64():
    """The gradient norms of train_step() in float64.  In float32 the biases of convolutions that feed a train-mode
    BatchNorm (exact gradient zero: the batch mean cancels them) carry rounding noise that differs between host CPUs."""
    net = ref_shims.build_reference_net().double().train()
    g = torch.Generator().manual_seed(5)
    z = torch.randn(2, 3, 128, 128, generator=g).double()
    x = torch.randn(2, 3, 256, 256, generator=g).double()
    out = net((z, x))
    (out[R].log().mean() + out[C].mean()).backward()
    grads = {k: float(p.grad.norm()) for k, p in net.named_parameters() if p.grad is not None}
    np.savez_compressed(os.path.join(OUT, "train_step_fp64.npz"), grad_names=np.array(sorted(grads)),
                        grad_norms=np.array([grads[k] for k in sorted(grads)]))
    print("train fp64: params with grad", len(grads))


def main():
    torch.set_num_threads(os.cpu_count())
    net = ref_shims.build_reference_net()
    sd32 = fo.load_lightning_state(ref_shims.REF_CKPT)
    smooth(net, sd32)
    update_branch(fo.to_dtype(sd32, torch.float64))
    train_step()
    train_step_fp64()


if __name__ == "__main__":
    main()
