"""GPU: the batched tracking loop with device-resident state (fear_track_crops_u8, fear_track_advance,
FEARMultiTracker) against the host arithmetic of image_ops and against FEARTracker run alone, bit for bit."""
import os

import numpy as np
import pytest
import torch

import feartracker_b200 as fb
from feartracker_b200 import _lib, image_ops
from oracle import fear_oracle as fo
from tests.helpers import GOLDEN, golden, load_full_state

pytestmark = pytest.mark.gpu
CFG = fb.FEAR_XS_TRACKER_KWARGS


@pytest.fixture(scope="module")
def net():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    n = fb.FEARNet(**fb.FEAR_XS_MODEL_KWARGS)
    n.load_state_dict(load_full_state(), strict=True)
    return n.cuda().eval()


@pytest.fixture(scope="module")
def clips():
    """Three variants of the demo clip: original (256x480), horizontally flipped, transposed (480x256), each with the
    golden initial box mapped into it."""
    frames = fo.read_video_rgb(os.path.join(GOLDEN, "test.mp4"))
    x, y, w, h = (int(v) for v in golden("video_teacher.npz")["init_bbox"])
    width = frames.shape[2]
    return [(frames, [x, y, w, h]),
            (np.ascontiguousarray(frames[:, :, ::-1]), [width - x - w, y, w, h]),
            (np.ascontiguousarray(frames.transpose(0, 2, 1, 3)), [y, x, h, w])]


def _single(net, frames, rect, start=0, skip=()):
    """FEARTracker(gpu_crop=True) alone: initialised on frames[start], then updated on every later frame except the
    indices in ``skip``.  Returns {frame index: box}."""
    trk = fb.FEARTracker(net, cuda_id=0, gpu_crop=True, **CFG)
    trk.initialize(frames[start], np.asarray(rect))
    return {t: [int(v) for v in trk.update(frames[t])["bbox"]] for t in range(start + 1, len(frames)) if t not in skip}


@pytest.fixture(scope="module")
def single_traj(net, clips):
    return [np.array(list(_single(net, f, r).values())) for f, r in clips]


def _track_rows(boxes, pads, ctx=None):
    rows = np.zeros(len(boxes), dtype=_lib.TRACK_DTYPE)
    for i, b in enumerate(boxes):
        c = ctx[i] if ctx is not None else (0, 0, 0, 0)
        rows[i] = tuple(int(v) for v in b) + tuple(int(v) for v in c) + tuple(int(v) for v in pads[i]) + (0,)
    return rows


def _frame_table(frames_dev):
    table = np.zeros(len(frames_dev), dtype=_lib.FRAME_DTYPE)
    for i, f in enumerate(frames_dev):
        table[i] = (f.data_ptr(), f.shape[0], f.shape[1])
    return torch.from_numpy(table.view(np.uint8).copy()).cuda()


def _rows_dev(rows):
    return torch.from_numpy(rows.view(np.uint8).copy()).cuda()


def test_track_crops_match_host_crop_and_cv2(net):
    lib = _lib.init(0)
    rng = np.random.default_rng(11)
    frames = [rng.integers(0, 256, s, dtype=np.uint8) for s in ((20, 30, 3), (256, 480, 3), (1080, 1920, 3))]
    frames_dev = [torch.from_numpy(f).cuda() for f in frames]
    table = _frame_table(frames_dev)
    cases = [(0, [3, 4, 10, 8]), (0, [0, 0, 30, 20]), (0, [25, 15, 5, 5]), (1, [163, 53, 45, 174]),
             (1, [-5, -7, 50, 60]), (1, [450, 230, 30, 26]), (1, [10, 200, 400, 56]), (2, [900, 500, 120, 80]),
             (2, [0, 0, 7, 9]), (2, [1800, 1000, 200, 150]), (2, [37, 1040, 300, 200]), (1, [177, 64, 128, 128])]
    boxes = [image_ops.clamp_bbox(b, frames[f].shape) for f, b in cases]
    means = [np.mean(frames[f], axis=(0, 1)) for f, _ in cases]
    pads = [np.clip(np.rint(m), 0, 255).astype(np.int32) for m in means]
    fot = np.array([f for f, _ in cases], dtype=np.int32)
    skipped = [2, 7]
    fot[skipped] = -1
    st = torch.cuda.current_stream().cuda_stream
    for size, off in ((256, 2), (128, 0.2), (256, 0.5)):
        n = len(cases)
        rows = _track_rows(boxes, pads, ctx=[(-1, -2, -3, -4)] * n)
        tracks = _rows_dev(rows)
        crops = torch.full((n, size, size, 3), 77, dtype=torch.uint8, device="cuda")
        fot_dev = torch.from_numpy(fot).cuda()
        _lib.check(lib.fear_track_crops_u8(table.data_ptr(), len(frames), fot_dev.data_ptr(), tracks.data_ptr(), n,
                                           size, float(off), crops.data_ptr(), st), "fear_track_crops_u8")
        got_rows = tracks.cpu().numpy().view(_lib.TRACK_DTYPE)
        got = crops.cpu().numpy()
        for i, (f, _) in enumerate(cases):
            if i in skipped:
                assert (got[i] == 77).all() and got_rows[i] == rows[i], i
                continue
            want, _, ctx = image_ops.extended_crop(frames[f], boxes[i], size, off, means[i])
            assert np.array_equal(got[i], want), (i, size, off)
            params, _, _ = image_ops.crop_params(boxes[i], size, off, means[i])
            one = torch.empty((size, size, 3), dtype=torch.uint8, device="cuda")
            pd = torch.from_numpy(params).cuda()
            _lib.check(lib.fear_crop_resize_u8(frames_dev[f].data_ptr(), frames[f].shape[0], frames[f].shape[1],
                                               pd.data_ptr(), one.data_ptr(), size, st), "fear_crop_resize_u8")
            assert np.array_equal(got[i], one.cpu().numpy()), (i, size, off)
            r = got_rows[i]
            assert [r["cx"], r["cy"], r["cw"], r["ch"]] == ctx.tolist(), i
            assert [r["x"], r["y"], r["w"], r["h"]] == list(boxes[i]) and [r["pad_r"], r["pad_g"], r["pad_b"]] == \
                pads[i].tolist()


def test_track_advance_matches_host_rescale_and_clamp(net):
    lib = _lib.init(0)
    rng = np.random.default_rng(5)
    sizes = [(20, 30), (256, 480), (480, 256), (1080, 1920)]
    frames_dev = [torch.zeros((h, w, 3), dtype=torch.uint8, device="cuda") for h, w in sizes]
    table = _frame_table(frames_dev)
    recs, ctxs, fot = [], [], []
    # crafted: exact .5 ties (context width 512 -> scale 2), sides rounding below 3, boxes past every frame edge
    for bx, by, bw, bh, c, f in [
            (10.25, 10.75, 10.25, 10.75, (0, 0, 512, 512), 1), (10.75, 10.25, 0.75, 1.25, (0, 0, 512, 512), 1),
            (0.6, 0.7, 0.6, 0.7, (5, 6, 256, 256), 0), (0.2, 0.2, 1.2, 1.3, (3, 4, 256, 256), 1),
            (-300.0, -300.0, 50.0, 50.0, (0, 0, 256, 256), 1), (900.0, 900.0, 50.0, 50.0, (0, 0, 256, 256), 1),
            (250.0, 10.0, 40.0, 30.0, (1700, 900, 512, 512), 3), (-20.0, 250.0, 400.0, 400.0, (-50, -60, 256, 256), 2),
            (128.0, 128.0, 2000.0, 3000.0, (10, 10, 700, 700), 0), (255.5, 255.5, 0.5, 0.5, (0, 0, 256, 256), 0),
            (127.5, 126.5, 3.5, 2.5, (100, 100, 256, 256), 2), (-0.5, -1.5, 4.5, 5.5, (0, 0, 256, 256), 1)]:
        recs.append((bx, by, bw, bh))
        ctxs.append(c)
        fot.append(f)
    for _ in range(4000):  # random records, half of them on a quarter-pixel grid so ties are common
        q = rng.random() < 0.5
        xy = rng.uniform(-80, 340, 2)
        wh = rng.uniform(0, 300, 2)
        if q:
            xy, wh = np.round(xy * 4) / 4, np.round(wh * 4) / 4
        f = int(rng.integers(0, len(sizes)))
        h, w = sizes[f]
        cw, ch = (int(v) for v in rng.choice([128, 256, 320, 512, 640, 1024, int(rng.integers(10, 1500))], 2))
        recs.append((xy[0], xy[1], wh[0], wh[1]))
        ctxs.append((int(rng.integers(-cw, w)), int(rng.integers(-ch, h)), cw, ch))
        fot.append(f)
    n = len(recs)
    fot = np.array(fot, dtype=np.int32)
    frozen = np.arange(3, n, 97)
    fot[frozen] = -1
    boxes = np.zeros(n, dtype=_lib.BOX_DTYPE)
    for i, (x, y, w, h) in enumerate(recs):
        boxes[i]["x"], boxes[i]["y"], boxes[i]["w"], boxes[i]["h"] = x, y, w, h
    prev = [(7, 8, 9, 10)] * n
    rows = _track_rows(prev, [(1, 2, 3)] * n, ctx=ctxs)
    tracks = _rows_dev(rows)
    boxes_dev = torch.from_numpy(boxes.view(np.uint8).copy()).cuda()
    fot_dev = torch.from_numpy(fot).cuda()
    _lib.check(lib.fear_track_advance(boxes_dev.data_ptr(), table.data_ptr(), fot_dev.data_ptr(), tracks.data_ptr(), n,
                                      256, torch.cuda.current_stream().cuda_stream), "fear_track_advance")
    got = tracks.cpu().numpy().view(_lib.TRACK_DTYPE)
    for i in range(n):
        g = [int(got[i][k]) for k in ("x", "y", "w", "h")]
        if fot[i] < 0:
            assert g == list(prev[i]), i
            continue
        h, w = sizes[fot[i]]
        want = image_ops.clamp_bbox(image_ops.rescale_bbox(recs[i], np.array(ctxs[i], dtype=np.int32), 256), (h, w, 3))
        assert g == [int(v) for v in want], (i, recs[i], ctxs[i], sizes[fot[i]], g, want)
    assert [int(got[0][k]) for k in ("x", "y")] == [20, 22] and [int(got[1][k]) for k in ("x", "y")] == [22, 20]


@pytest.mark.parametrize("source", ["numpy", "cuda"])
def test_multi_stream_matches_single_trackers(net, clips, single_traj, source):
    """8 tracks on mixed-size clip variants over the whole clip: every trajectory is the one FEARTracker(gpu_crop=True)
    gives alone (Bz = N against Bz = 1), track 0 is the reference trajectory."""
    n = 8
    variant = [i % len(clips) for i in range(n)]
    if source == "cuda":
        dev_clips = [torch.from_numpy(f).cuda() for f, _ in clips]
        pick = lambda v, t: dev_clips[v][t]  # noqa: E731
    else:
        pick = lambda v, t: clips[v][0][t]  # noqa: E731
    mt = fb.FEARMultiTracker(net, cuda_id=0, max_tracks=n, **CFG)
    mt.initialize([pick(v, 0) for v in variant], [clips[v][1] for v in variant])
    steps = len(clips[0][0]) - 1
    traj = np.stack([mt.update([pick(v, t) for v in variant])["bbox"] for t in range(1, steps + 1)])
    assert mt._st["graph"] is not None
    for i, v in enumerate(variant):
        same = (traj[:, i] == single_traj[v]).all(1)
        assert same.all(), (i, v, int(np.argmin(same)))
    assert (traj[:, 0] == golden("video_teacher.npz")["trajectory"]).all()


def test_multi_object_on_one_frame_sequence(net, clips):
    frames = clips[0][0][:301]
    rects = [clips[0][1], [300, 120, 60, 80], [20, 150, 40, 40], [150, 60, 30, 30], [400, 10, 70, 90]]
    mt = fb.FEARMultiTracker(net, cuda_id=0, max_tracks=16, **CFG)
    mt.initialize(frames[0], rects)
    outs = [mt.update(f) for f in frames[1:]]
    traj = np.stack([o["bbox"] for o in outs])
    assert np.isfinite(np.stack([o["score"] for o in outs])).all()
    for i, r in enumerate(rects):
        want = np.array(list(_single(net, frames, r).values()))
        same = (traj[:, i] == want).all(1)
        assert same.all(), (i, int(np.argmin(same)))


def test_reinitialise_and_freeze(net, clips, single_traj):
    """Tracks 1 and 3 are re-initialised on frame 100 and follow a fresh single tracker from there; track 2 is frozen
    for frames 101..150 (its box stays put) and then continues like a single tracker that skipped those frames;
    track 0 is unaffected."""
    n, t_re, frozen = 4, 100, range(101, 151)
    variant = [0, 1, 2, 0]
    steps = 250
    mt = fb.FEARMultiTracker(net, cuda_id=0, max_tracks=n, **CFG)
    mt.initialize([clips[v][0][0] for v in variant], [clips[v][1] for v in variant])
    new_rects = {1: [200, 80, 50, 60], 3: [300, 100, 40, 70]}
    box = {}
    for t in range(1, steps + 1):
        fot = np.arange(n)
        if t == t_re:  # like FEARTracker: initialize on frame t, first update on frame t + 1
            mt.initialize([clips[variant[i]][0][t] for i in new_rects], list(new_rects.values()),
                          track_ids=list(new_rects))
            fot[list(new_rects)] = -1
        if t in frozen:
            fot[2] = -1
        out = mt.update([clips[v][0][t] for v in variant], frame_of_track=fot)
        assert np.isnan(out["score"][fot < 0]).all() and np.isfinite(out["score"][fot >= 0]).all()
        box[t] = out["bbox"]
    for t in box:
        assert box[t][0].tolist() == single_traj[0][t - 1].tolist(), t
    for i, r in new_rects.items():
        want = _single(net, clips[variant[i]][0][:steps + 1], r, start=t_re)
        assert all(box[t][i].tolist() == want[t] for t in want), i
    for t in frozen:
        assert box[t][2].tolist() == box[t_re][2].tolist(), t
    want2 = _single(net, clips[2][0][:steps + 1], clips[2][1], skip=set(frozen))
    assert all(box[t][2].tolist() == want2[t] for t in want2)


def test_cuda_graph_survives_workspace_growth(clips, single_traj):
    """A workspace-growing batched call on the same net between two steps invalidates the captured step graph
    (generation counter) instead of replaying into freed buffers."""
    n2 = fb.FEARNet(**fb.FEAR_XS_MODEL_KWARGS)
    n2.load_state_dict(load_full_state(), strict=True)
    n2 = n2.cuda().eval()
    variant = [0, 1, 2]
    mt = fb.FEARMultiTracker(n2, cuda_id=0, max_tracks=4, **CFG)
    mt.initialize([clips[v][0][0] for v in variant], [clips[v][1] for v in variant])
    out = [mt.update([clips[v][0][t] for v in variant])["bbox"] for t in range(1, 6)]
    assert mt._st["graph"] is not None
    gen = n2.generation()
    zt, xt, _, _ = fo.synthetic_crops(12)
    n2.track(xt.cuda(), n2.get_features(zt.cuda()))  # batch 12 > reserved 4: workspace is freed and re-allocated
    assert n2.generation() != gen
    out += [mt.update([clips[v][0][t] for v in variant])["bbox"] for t in range(6, 40)]
    traj = np.stack(out)
    for i, v in enumerate(variant):
        assert (traj[:, i] == single_traj[v][:len(out)]).all(), i
