"""Throughput of FEARMultiTracker (batched tracking loop, track state on the device) on one GPU.

    python tools/bench_multitrack.py [--steps 660] [--tracks 1,16,64,256] [--out FILE]

Multi-stream: N tracks, track n follows variant n % 3 of tests/golden/test.mp4 (original 256x480, horizontally
flipped, transposed 480x256: mixed frame sizes in one step), once with the frames handed over as numpy arrays (packed
into pinned memory and uploaded every step) and once with the clips preloaded as CUDA tensors (read in place).
Multi-object: N targets on one shared frame per step.  Per run: track-updates/s and ms/step (host clock around
update(), which ends in a device synchronise), device-only ms/step (CUDA events around replays of the captured step
graph) and, from a separate eager run with events between the kernels, the split crop / network / advance.
Parity: track 0 reproduces the reference trajectory (video_teacher.npz) and every track its own N = 1 run.
Prints one JSON line with the GPU's name, power limit and max SM clock (read-only nvidia-smi query) beside the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import feartracker_b200 as fb  # noqa: E402
from feartracker_b200 import _lib  # noqa: E402
from oracle import fear_oracle as fo  # noqa: E402
from tests.helpers import GOLDEN, golden, load_full_state  # noqa: E402

CFG = fb.FEAR_XS_TRACKER_KWARGS


def device_info(index: int) -> dict:
    try:
        out = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = (s.strip() for s in out.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as exc:  # the numbers stay valid; say what could not be read
        return {"name": torch.cuda.get_device_name(index), "nvidia_smi_error": str(exc)}


def clip_variants():
    frames = fo.read_video_rgb(os.path.join(GOLDEN, "test.mp4"))
    x, y, w, h = (int(v) for v in golden("video_teacher.npz")["init_bbox"])
    width = frames.shape[2]
    return [(frames, [x, y, w, h]),
            (np.ascontiguousarray(frames[:, :, ::-1]), [width - x - w, y, w, h]),
            (np.ascontiguousarray(frames.transpose(0, 2, 1, 3)), [y, x, h, w])]


def timed_run(net, n, steps, frames_at, rects, init_frames):
    """Track over ``steps`` steps; returns (trajectory (steps, n, 4), metrics, tracker)."""
    mt = fb.FEARMultiTracker(net, cuda_id=0, max_tracks=n, **CFG)
    mt.initialize(init_frames, rects)
    traj, warm = [], 3  # step 1 eager, step 2 captures the graph
    for t in range(1, warm + 1):
        traj.append(mt.update(frames_at(t))["bbox"])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for t in range(warm + 1, steps + 1):
        traj.append(mt.update(frames_at(t))["bbox"])
    wall = time.perf_counter() - t0
    timed = steps - warm
    graph = mt._st["graph"]
    reps = max(20, min(200, 20000 // n))
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(reps):
        graph.replay()
    ev[1].record()
    torch.cuda.synchronize()
    metrics = {"tracks": n, "timed_steps": timed, "updates_per_s": n * timed / wall, "ms_per_step": 1e3 * wall / timed,
               "device_ms_per_step": ev[0].elapsed_time(ev[1]) / reps}
    return np.stack(traj), metrics, mt


def split_run(net, mt, reps=20):
    """Eager steps with CUDA events between crop, network + decode and advance (a separate run: the events add
    launches)."""
    st, lib, n = mt._st, _lib.load(), mt.num_tracks
    stream = torch.cuda.current_stream().cuda_stream
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    acc = np.zeros(3)
    for _ in range(reps + 2):
        ev[0].record()
        _lib.check(lib.fear_track_crops_u8(st["table"].data_ptr(), mt.max_tracks, st["fot_ptr"], st["tracks"].data_ptr(),
                                           n, 256, float(CFG["search_context"]), st["search"].data_ptr(), stream), "crop")
        ev[1].record()
        boxes = net.track_boxes(st["search"][:n], st["zf"][:n])
        ev[2].record()
        _lib.check(lib.fear_track_advance(boxes.data_ptr(), st["table"].data_ptr(), st["fot_ptr"],
                                          st["tracks"].data_ptr(), n, 256, stream), "advance")
        ev[3].record()
        torch.cuda.synchronize()
        if _ >= 2:
            acc += [ev[i].elapsed_time(ev[i + 1]) for i in range(3)]
    acc /= reps
    return {"crop_ms": acc[0], "network_ms": acc[1], "advance_ms": acc[2]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=660)
    ap.add_argument("--tracks", default="1,16,64,256")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_multitrack.py needs a CUDA device")
    ns = [int(v) for v in args.tracks.split(",")]
    net = fb.FEARNet(**fb.FEAR_XS_MODEL_KWARGS)
    net.load_state_dict(load_full_state(), strict=True)
    net = net.cuda().eval()
    clips = clip_variants()
    steps = min(args.steps, len(clips[0][0]) - 1)
    ref = golden("video_teacher.npz")["trajectory"][:steps]
    result = {"metric": "FEARMultiTracker track-updates/s", "device": device_info(0), "steps": steps,
              "variants": ["original 256x480", "flipped 256x480", "transposed 480x256"]}

    # single FEARTracker(gpu_crop=True) for scale
    trk = fb.FEARTracker(net, cuda_id=0, gpu_crop=True, **CFG)
    trk.initialize(clips[0][0][0], np.asarray(clips[0][1]))
    for t in range(1, 4):
        trk.update(clips[0][0][t])
    t0 = time.perf_counter()
    for t in range(4, steps + 1):
        trk.update(clips[0][0][t])
    result["single_fear_tracker_gpu_crop_updates_per_s"] = (steps - 3) / (time.perf_counter() - t0)

    solo = []  # N = 1 run of every variant (numpy frames): the per-track parity reference
    for frames, rect in clips:
        traj, _, _ = timed_run(net, 1, steps, lambda t, f=frames: [f[t]], [rect], [frames[0]])
        solo.append(traj[:, 0])
    dev_clips = [torch.from_numpy(f[:steps + 1]).cuda() for f, _ in clips]
    streams, parity_ref, parity_solo = [], True, True
    for source in ("numpy", "cuda"):
        for n in ns:
            variant = [i % 3 for i in range(n)]
            if source == "numpy":
                frames_at = lambda t, v=variant: [clips[j][0][t] for j in v]  # noqa: E731
            else:
                frames_at = lambda t, v=variant: [dev_clips[j][t] for j in v]  # noqa: E731
            traj, m, mt = timed_run(net, n, steps, frames_at, [clips[j][1] for j in variant], frames_at(0))
            m["frames"] = source
            m["track0_equals_reference"] = bool((traj[:, 0] == ref).all())
            m["every_track_equals_its_n1_run"] = bool(all((traj[:, i] == solo[j]).all() for i, j in enumerate(variant)))
            parity_ref &= m["track0_equals_reference"]
            parity_solo &= m["every_track_equals_its_n1_run"]
            m.update(split_run(net, mt))
            streams.append(m)
            print(json.dumps(m), file=sys.stderr)
    result["multi_stream"] = streams

    objects = []
    frames = clips[0][0]
    for n in ns:  # N targets on one frame sequence: boxes on a grid over the 256x480 frame
        k = int(np.ceil(np.sqrt(n)))
        rects = [[int(20 + (i % k) * 420 / k), int(10 + (i // k) * 200 / k), 40, 50] for i in range(n)]
        rects[0] = clips[0][1]
        traj, m, mt = timed_run(net, n, steps, lambda t: frames[t], rects, frames[0])
        m["frames"] = "numpy, one shared frame"
        m["track0_equals_reference"] = bool((traj[:, 0] == ref).all())
        parity_ref &= m["track0_equals_reference"]
        objects.append(m)
        print(json.dumps(m), file=sys.stderr)
    result["multi_object"] = objects
    result["parity"] = {"track0_equals_reference": parity_ref, "every_track_equals_its_n1_run": parity_solo}
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
