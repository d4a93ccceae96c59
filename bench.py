#!/usr/bin/env python
"""bench.py -- FEAR-XS per-frame inference throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--dump-outputs DIR]

A "step" = one pass of the hot path (FEARNet.track + box decode) over one batch of synthetic
crops: 256 search crops (3x256x256 fp32, ImageNet-normalised uniform uint8, seed 20260924) with
their 256 template feature maps, per GPU (BASELINE config 2; at N GPUs each rank owns a contiguous
256-frame shard of the 256*N batch -- config 4 at N=8 -- and the step ends with ONE all-gather of
the 48-byte box records).  One JSON line on stdout (rank 0).  See DESIGN.md section "Measurement".

--dump-outputs DIR writes the gathered box records of the last timed step (rank 0) as DIR/box_xywh.npy
(float64, (N,4)), DIR/score.npy (float32, (N,)) and DIR/cell_row_col_flat.npy (float64, (N,3)); the inputs
depend only on the seed, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "FEAR-XS frames/sec (track + decode, batch 256 per GPU)"
CORR_BYTES_PER_FRAME = 2 * (65536 + 262144 + 65536)  # 2 branches x (z + x + s) fp32, SURVEY.md 8(d)
PATH_BYTES_PER_FRAME = 14_947_328  # block-fused budget of the whole track(), SURVEY.md 8(d)
SEED = 20260924


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_state():
    with np.load(os.path.join(ROOT, "tests", "golden", "fear_xs_hotpath_state.npz")) as f:
        hot = {k: torch.from_numpy(f[k]) for k in f.files}
    with open(os.path.join(ROOT, "tests", "golden", "state_dict_keys.json")) as f:
        keys = json.load(f)
    return {k: hot[k] if k in hot else torch.zeros(s, dtype=getattr(torch, d)) for k, (s, d) in keys.items()}


def synthetic_batch(batch, rank, with_u8=False):
    """uint8-derived, ImageNet-normalised crops; every rank regenerates its own shard from the seed."""
    g = torch.Generator().manual_seed(SEED + rank)
    mean = torch.tensor([0.485, 0.456, 0.406]).view(1, 3, 1, 1) * 255.0
    inv = 1.0 / (torch.tensor([0.229, 0.224, 0.225]).view(1, 3, 1, 1) * 255.0)
    zu = torch.randint(0, 256, (batch, 3, 128, 128), generator=g, dtype=torch.uint8)
    xu = torch.randint(0, 256, (batch, 3, 256, 256), generator=g, dtype=torch.uint8)
    if with_u8:
        return (zu.float() - mean) * inv, (xu.float() - mean) * inv, xu
    return (zu.float() - mean) * inv, (xu.float() - mean) * inv


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, str(gpu_index)
        self.mark_a = self.mark_b = None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", self.gpu], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def wait_first_sample(self, timeout=5.0):
        t0 = time.time()
        while not self.rows and time.time() - t0 < timeout and self.proc is not None:
            time.sleep(0.05)

    def begin(self):
        self.mark_a = len(self.rows)

    def end(self):
        time.sleep(0.25)  # let the sample(s) covering the end of the timed region arrive
        self.mark_b = len(self.rows)

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self):
        a = max(0, (self.mark_a or 0) - 1)
        rows = self.rows[a:self.mark_b] if self.mark_b is not None else self.rows[a:]
        rows = rows or self.rows[-3:]
        sm = [float(r[1]) for r in rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            if len(r) >= 9:
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def pick_cpu_threads():
    """Thread count for the CPU baseline: the host may expose far more logical CPUs than this container
    can actually run on (oversubscription makes torch's intra-op pool collapse), so probe a few counts
    on a 4-frame slice and keep the fastest."""
    from oracle import fear_oracle as fo

    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    sd = {k: v for k, v in load_state().items() if v.is_floating_point()}
    zt, xt = synthetic_batch(4, 0)
    zf = fo.get_features(sd, zt)
    best, best_t = 1, float("inf")
    for n in sorted({min(avail, c) for c in (8, 16, 32, 64, avail)}):
        torch.set_num_threads(n)
        fo.track(sd, xt[:1], zf[:1])
        t0 = time.perf_counter()
        fo.track(sd, xt, zf)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = n, dt
        if dt > 20:
            break
    return best, 4 / best_t


def time_cpu_oracle(batch, steps, warmup, threads):
    """The oracle port (reference source restated, torch CPU fp32) on the host cores: frames/s."""
    from oracle import fear_oracle as fo

    torch.set_num_threads(threads)
    sd = {k: v for k, v in load_state().items() if v.is_floating_point()}
    zt, xt = synthetic_batch(batch, 0)
    zf = fo.get_features(sd, zt)
    for _ in range(warmup):
        fo.decode(*[fo.track(sd, xt, zf)[k] for k in (fo.TARGET_REGRESSION_LABEL_KEY, fo.TARGET_CLASSIFICATION_KEY)])
    t0 = time.perf_counter()
    for _ in range(steps):
        out = fo.track(sd, xt, zf)
        fo.decode(out[fo.TARGET_REGRESSION_LABEL_KEY], out[fo.TARGET_CLASSIFICATION_KEY])
    dt = time.perf_counter() - t0
    return batch * steps / dt, dt / steps * 1e3


def parity_check(net, boxes_all, world, B, frames_per_rank=4):
    """Rank 0, after the timed region: the GATHERED (world*B, 48) box records of the benchmarked batch against the
    fp64 CPU oracle on ``frames_per_rank`` frames of every rank's shard (first, last and two interior frames):
    argmax (row, col) exact, box coordinates relative error, scores.  Every rank's inputs are regenerated from the
    shared seed, so this also proves the all-gather put each shard where it belongs."""
    from oracle import fear_oracle as fo

    sd64 = fo.to_dtype({k: v for k, v in load_state().items() if v.is_floating_point()}, torch.float64)
    rec = net.boxes_to_numpy(boxes_all)
    idx = sorted({0, B // 3, (2 * B) // 3, B - 1})[:frames_per_rank]
    exact, max_rel, max_score, n, min_margin, tie_sensitive = True, 0.0, 0.0, 0, float("inf"), 0
    for r in range(world):
        zt, xt = synthetic_batch(B, r)
        sel = torch.tensor(idx)
        with torch.no_grad():
            zf = fo.get_features(sd64, zt[sel].double())
            out = fo.track(sd64, xt[sel].double(), zf)
        bbox, coords = fo.decode(out[fo.TARGET_REGRESSION_LABEL_KEY], out[fo.TARGET_CLASSIFICATION_KEY])
        score = out[fo.TARGET_CLASSIFICATION_KEY].sigmoid().flatten(1).max(1).values.numpy()
        top2 = out[fo.TARGET_CLASSIFICATION_KEY].flatten(1).topk(2, dim=1).values
        margin = (top2[:, 0] - top2[:, 1]).numpy()  # top-1 / top-2 logit margin of the oracle (SURVEY.md 8(c))
        for j, i in enumerate(idx):
            m = rec[r * B + i]
            min_margin = min(min_margin, float(margin[j]))
            if margin[j] < 1e-4:  # a tie at fp32 resolution: reported, not counted as an argmax failure
                tie_sensitive += 1
                continue
            exact &= (int(m["row"]), int(m["col"])) == tuple(coords[j])
            mine = np.array([m["x"], m["y"], m["w"], m["h"]])
            ref = bbox[j].numpy()
            max_rel = max(max_rel, float(np.max(np.abs(mine - ref) / np.maximum(np.abs(ref), 1.0))))
            max_score = max(max_score, abs(float(m["score"]) - float(score[j])))
            n += 1
    return {"frames": n, "frames_per_rank": len(idx), "argmax_exact": bool(exact), "max_rel": max_rel,
            "max_score_abs": max_score, "min_logit_margin": min_margin, "tie_sensitive_frames": tie_sensitive, "against": "fp64 CPU oracle (reference source restated), inputs regenerated "
            "from the seed per rank; template features are this library's own (fp32) for the timed run and the "
            "oracle's (fp64) for the check"}


def dump_outputs(out_dir, rec):
    """The decoded FearBox records (``net.boxes_to_numpy``) as float64 / float32 .npy files."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"box_xywh": np.stack([rec[k] for k in ("x", "y", "w", "h")], 1),
              "score": np.ascontiguousarray(rec["score"]),
              "cell_row_col_flat": np.stack([rec[k] for k in ("row", "col", "flat")], 1).astype(np.float64)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def read_video(path):
    import cv2

    cap, frames = cv2.VideoCapture(path), []
    while True:
        ok, f = cap.read()
        if not ok:
            break
        frames.append(cv2.cvtColor(f, cv2.COLOR_BGR2RGB))
    cap.release()
    return frames


def run_stream(net, dev, repeat=2):
    """BASELINE config 3: FEARTracker.update over the demo clip (tests/golden/test.mp4, 661 frames 480x256, init box
    [163,53,45,174]); sequentially dependent frames, batch 1, one B200.  frames/s includes host crop/resize, H2D,
    kernels, D2H of the box record; also the device-only time of the per-frame step and the agreement with the
    reference's trajectory (golden fixture recorded from the reference's own source)."""
    import feartracker_b200 as fb

    g = np.load(os.path.join(ROOT, "tests", "golden", "video_teacher.npz"))
    frames = read_video(os.path.join(ROOT, "tests", "golden", "test.mp4"))
    modes = {}
    for name, cfg_extra in (("host_crop", {}), ("gpu_crop", {"gpu_crop": True})):
        cfg = dict(fb.FEAR_XS_TRACKER_KWARGS, **cfg_extra)
        best, traj = None, None
        try:
            for _ in range(repeat):
                trk = fb.FEARTracker(net, cuda_id=dev.index, **cfg)
                trk.initialize(frames[0], g["init_bbox"])
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                out = [trk.update(f)["bbox"] for f in frames[1:]]
                torch.cuda.synchronize(dev)
                dt = time.perf_counter() - t0
                if best is None or dt < best:
                    best, traj = dt, np.array([list(map(int, b)) for b in out])
        except NotImplementedError as exc:
            modes[name] = {"unavailable": str(exc)}
            continue
        same = (traj == g["trajectory"]).all(1)
        a, b = traj.astype(np.float64), g["trajectory"].astype(np.float64)
        x1, y1 = np.maximum(a[:, 0], b[:, 0]), np.maximum(a[:, 1], b[:, 1])
        x2 = np.minimum(a[:, 0] + a[:, 2], b[:, 0] + b[:, 2])
        y2 = np.minimum(a[:, 1] + a[:, 3], b[:, 1] + b[:, 3])
        inter = np.clip(x2 - x1, 0, None) * np.clip(y2 - y1, 0, None)
        iou = inter / (a[:, 2] * a[:, 3] + b[:, 2] * b[:, 3] - inter)
        n = len(frames) - 1
        modes[name] = {"value": n / best, "unit": "frames/s", "ms_per_frame": best / n * 1e3,
                       "trajectory_identical": bool(same.all()), "identical_boxes": int(same.sum()), "of": n,
                       "min_iou": float(iou.min()), "mean_iou": float(iou.mean())}
    # device-only time of the batch-1 step (CUDA events around eager launches and around graph replays)
    trk = fb.FEARTracker(net, cuda_id=dev.index, **fb.FEAR_XS_TRACKER_KWARGS)
    trk.initialize(frames[0], g["init_bbox"])
    crop = trk._preprocess_image(np.ascontiguousarray(frames[1][:256, :256]))
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(10):
        net.track_boxes(crop, trk._template_features)
    torch.cuda.synchronize(dev)
    a.record()
    for _ in range(100):
        net.track_boxes(crop, trk._template_features)
    b.record()
    torch.cuda.synchronize(dev)
    eager_ms = a.elapsed_time(b) / 100
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        net.track_boxes(crop, trk._template_features)
    torch.cuda.synchronize(dev)
    a.record()
    for _ in range(100):
        gr.replay()
    b.record()
    torch.cuda.synchronize(dev)
    graph_ms = a.elapsed_time(b) / 100
    head = modes.get("host_crop", {})
    out = {"workload": "FEAR-XS streaming video track loop (BASELINE config 3): tests/golden/test.mp4, 660 updates, "
                       "batch 1, sequentially dependent; replicas only (does not shard)",
           "value": head.get("value"), "unit": "frames/s", "modes": modes,
           "device_step_ms": {"eager_launches": eager_ms, "cuda_graph_replay": graph_ms}}
    if head.get("ms_per_frame"):
        out["host_share"] = 1.0 - graph_ms / head["ms_per_frame"]
    return out


def run_reference(args, rank):
    """--impl reference: the reference's own CPU implementation of the path (oracle port) on all host
    threads, same metric/config; rank 0 only."""
    if rank != 0:
        return
    threads, probe_fps = pick_cpu_threads()
    # bounded sample: size the per-step slice so warm-up + K steps stay around a minute
    sample = int(max(1, min(32, probe_fps * 60.0 / (args.steps + 2))))
    fps, ms = time_cpu_oracle(sample, args.steps, max(1, min(args.warmup, 2)), threads)
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "FEAR-XS batched inference, batch=256 synthetic crops (BASELINE config 2)",
                   "sample": f"{sample}-frame slice of the workload per step"},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                         "sample": f"oracle port (reference source restated, torch CPU fp32), track()+decode on "
                                   f"{sample} frames x {args.steps} steps"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=256, help="frames per GPU per step")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--corr", default=None, help="correlation kernel implementation: ffma | tcgen05")
    ap.add_argument("--pw", default=None, help="1x1-conv implementation: ffma | tcgen05")
    ap.add_argument("--dw", default=None, help="depthwise implementation: pixel | strip | roll | auto")
    ap.add_argument("--dw-wide", type=int, default=None)
    ap.add_argument("--fuse", type=int, default=None, help="1 = fused pw-expand+dw kernels for the stride-2 blocks")
    ap.add_argument("--fuse-stem", type=int, default=None, help="0 = separate stem / xif1_0 kernels")
    ap.add_argument("--early-sub", type=int, default=None, help="sub-batch (frames) of the high-resolution blocks")
    ap.add_argument("--opt", action="append", default=[], metavar="KEY=VALUE",
                    help="extra fear_set_option pairs (experiments), e.g. --opt small_const=0")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="batch", choices=["batch", "stream"],
                    help="batch = BASELINE config 2/4 (default, the contract line); stream = config 3 only")
    ap.add_argument("--no-stream", action="store_true", help="skip the config-3 streaming measurement")
    ap.add_argument("--no-parity", action="store_true", help="skip the post-run oracle parity check")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the box records of the last timed step as .npy files under DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "batch"):
        ap.error("--dump-outputs applies to the batch workload of --impl ours")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank)

    import feartracker_b200 as fb
    from feartracker_b200 import _lib, sharding

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the FEAR hot path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # stdout must carry exactly ONE JSON line.  NCCL prints its version banner on stdout when the communicator is
        # created (NCCL_DEBUG_FILE is read too early to help from here), so fd 1 points at stderr while the process
        # group and its communicator come up (the barrier forces the lazy creation), then it is restored.
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier(device_ids=[local_rank])
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    B, total = args.batch, args.batch * world

    net = fb.FEARNet(**fb.FEAR_XS_MODEL_KWARGS)
    net.load_state_dict(load_state(), strict=True)
    net = net.to(dev).eval()
    net.reserve(B)
    if args.corr:
        net.set_option("corr", args.corr)
        _lib.check(_lib.load().fear_set_option(None, b"corr", args.corr.encode()), "fear_set_option")
    if args.pw:
        net.set_option("pw", args.pw)
    if args.dw:
        net.set_option("dw", args.dw)
    if args.dw_wide is not None:
        net.set_option("dw_wide", str(args.dw_wide))
    if args.fuse is not None:
        net.set_option("fuse", str(args.fuse))
    if args.fuse_stem is not None:
        net.set_option("fuse_stem", str(args.fuse_stem))
    for kv in args.opt:
        k, v = kv.split("=", 1)
        net.set_option(k, v)
    if args.early_sub is not None:
        net.set_option("early_sub", str(args.early_sub))

    if args.workload == "stream":
        if rank == 0:
            line = run_stream(net, dev, repeat=3)
            line.update({"metric": "FEAR-XS streaming track loop frames/sec (BASELINE config 3)", "n_gpus": 1,
                         "higher_is_better": True, "dtype": "f32", "data": "tests/golden/test.mp4"})
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    zt, xt, xu = synthetic_batch(B, rank, with_u8=True)
    x_host, z_dev = xt.pin_memory(), net.get_features(zt.to(dev))
    xu_host = xu.permute(0, 2, 3, 1).contiguous().pin_memory()  # raw uint8 HWC crops, as the tracker holds them
    zf_host = z_dev.cpu().pin_memory()
    x_dev = x_host.to(dev)
    box_host = torch.empty((total, 48), dtype=torch.uint8).pin_memory()
    stream = torch.cuda.current_stream(dev)

    def step_device():
        boxes = net.track_boxes(x_dev, z_dev)
        return sharding.all_gather_boxes(boxes, total)

    def step_e2e(src=None):
        # public API on pinned HOST buffers: chunked H2D overlapped with compute, boxes copied back
        boxes = net.track_boxes_from_host(xu_host if src is None else src, zf_host)
        boxes = sharding.all_gather_boxes(boxes, total)
        box_host.copy_(boxes, non_blocking=True)
        return boxes

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps):
        """(ms for ``steps`` calls of fn, what the last call returned)"""
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        a.record(stream)
        for _ in range(steps):
            out = fn()
        b.record(stream)
        sync_all()
        ms = torch.tensor([a.elapsed_time(b)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    clocks = ClockSampler(local_rank).__enter__()
    for _ in range(args.warmup):
        step_device()
    clocks.wait_first_sample()
    l0 = net.launch_count()
    clocks.begin()
    ms_total, last_boxes = timed(step_device, args.steps)
    if ms_total < 400.0:  # keep the GPU under the same load until nvidia-smi (100 ms period) has sampled it
        extra = int(400.0 / (ms_total / args.steps)) + 1
        for _ in range(extra):
            step_device()
        torch.cuda.synchronize(dev)
    clocks.end()
    clocks.__exit__()
    launches = (net.launch_count() - l0) // (args.steps + (extra if ms_total < 400.0 else 0))
    fps = total * args.steps / (ms_total * 1e-3)

    for _ in range(args.warmup):
        step_e2e()
    ms_e2e, _ = timed(step_e2e, args.steps)
    fps_e2e = total * args.steps / (ms_e2e * 1e-3)
    for _ in range(args.warmup):
        step_e2e(x_host)
    ms_e2e32, _ = timed(lambda: step_e2e(x_host), args.steps)

    # ---- per-stage device time over another K steps (CUDA events around every launch, same stream) ----
    net.profile(True)
    sync_all()
    for _ in range(args.steps):
        step_device()
    sync_all()
    stages = net.stage_times()
    net.profile(False)
    corr_ms, corr_n = stages["corr"]
    peak, peak_src = load_peaks()
    roofline = None
    if corr_n:
        per_launch_s = corr_ms * 1e-3 / corr_n
        bytes_per_launch = CORR_BYTES_PER_FRAME * B / (corr_n / args.steps)  # one launch covers both branches
        achieved = bytes_per_launch / per_launch_s / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "corr_traffic.json")
        if os.path.isfile(tpath):
            with open(tpath) as f:
                traffic = json.load(f).get("dram_bytes_per_launch")
        roofline = {
            "kernel": "tc::corr_ts_kernel -- pixel-wise correlation, both head branches in one launch", "bound": "hbm",
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
            "peak_source": peak_src, "us_per_launch": per_launch_s * 1e6,
            "algorithmic_bytes_per_launch": int(bytes_per_launch),
            "how": "CUDA events around every correlation launch inside K extra steps (includes the launch latency the event "
                   "pair exposes); back_to_back = the same launch shape issued 40 times in a row on rotating > L2 buffers",
        }
        if rank == 0:
            # the same kernel and launch shape (2 B frames) in a tight loop: what the kernel sustains once launch latency and
            # the prologue are hidden behind the previous launch, as they are inside the step with programmatic dependent launch
            frames = 2 * B
            zt_b = torch.randn(frames, 64, 256, device=dev)
            cats = [torch.randn(frames, 256, 320, device=dev) for _ in range(2)]
            lib_c, st = _lib.load(), torch.cuda.current_stream(dev).cuda_stream
            for c_ in cats:
                _lib.check(lib_c.fear_corr_nhwc_f32(zt_b.data_ptr(), frames, c_.data_ptr(), frames, st), "fear_corr_nhwc_f32")
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i_ in range(40):
                _lib.check(lib_c.fear_corr_nhwc_f32(zt_b.data_ptr(), frames, cats[i_ & 1].data_ptr(), frames, st), "fear_corr_nhwc_f32")
            e1.record()
            torch.cuda.synchronize(dev)
            us_b2b = e0.elapsed_time(e1) * 1e3 / 40
            gbs = CORR_BYTES_PER_FRAME // 2 * frames / (us_b2b * 1e-6) / 1e9
            roofline["back_to_back"] = {"us_per_launch": us_b2b, "achieved": gbs, "frac": gbs / peak}
            del zt_b, cats
    step_ms_sum = sum(v[0] for v in stages.values()) / args.steps
    path_gbs = PATH_BYTES_PER_FRAME * B / (ms_total / args.steps * 1e-3) / 1e9
    stage_report = {k: {"ms_per_step": v[0] / args.steps, "launches_per_step": v[1] / args.steps,
                        "share": (v[0] / args.steps) / step_ms_sum if step_ms_sum else None}
                    for k, v in stages.items()}

    # ---- parity of exactly what was timed: the gathered records of the benchmarked batch vs the oracle (rank 0) ----
    final_boxes = step_device()
    final_boxes_e2e = step_e2e()
    sync_all()
    parity = None
    if rank == 0 and not args.no_parity:
        parity = parity_check(net, final_boxes, world, B)
        parity["e2e_records_identical"] = bool(torch.equal(final_boxes, final_boxes_e2e))
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, net.boxes_to_numpy(last_boxes))
    stream_line = None
    if rank == 0 and world == 1 and not args.no_stream:
        stream_line = run_stream(net, dev)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads, probe_fps = pick_cpu_threads()
        sample = int(max(1, min(32, probe_fps * 3.0)))
        cfps, cms = time_cpu_oracle(sample, 6, 1, threads)
        cpu = {"value": cfps, "unit": "frames/s", "cores": threads, "kind": "port",
               "sample": f"oracle port (reference source restated, torch CPU fp32): track()+decode on a {sample}-frame "
                         f"slice of the workload, 1 warm-up + 6 timed steps ({cms:.0f} ms/step), best of probed "
                         "thread counts"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": "FEAR-XS batched inference, batch=256 synthetic crops per GPU (BASELINE config 2; "
                            "config 4 at 8 GPUs), FEAR-XS checkpoint weights",
                "global_batch": total, "per_gpu_batch": B, "parallelism": f"frames sharded over {world} rank(s)",
                "l2": "inputs larger than L2 (201 MB search batch per step; >2 GB of workspace traffic per step)",
                "impl": {"corr": args.corr or "default", "pw": args.pw or "default", "dw": args.dw or "default",
                         "early_sub": args.early_sub},
            },
            "e2e": {"value": fps_e2e, "unit": "frames/s", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": int(xu_host.numel() + zf_host.numel() * 4),
                    "d2h_bytes_per_step": int(box_host.numel()),
                    "api": "FEARNet.track_boxes_from_host on pinned host buffers: raw uint8 HWC crops (what "
                           "FEARTracker holds; ImageNet normalisation fused into the stem kernel, bit-identical to "
                           "host normalisation) + fp32 template features; double-buffered staging, so the copy of step "
                           "i+1 overlaps the kernels of step i; box records copied back every step"},
            "e2e_fp32_inputs": {"value": total * args.steps / (ms_e2e32 * 1e-3), "unit": "frames/s",
                                "ms_per_step": ms_e2e32 / args.steps,
                                "h2d_bytes_per_step": int(x_host.numel() * 4 + zf_host.numel() * 4),
                                "d2h_bytes_per_step": int(box_host.numel()),
                                "api": "same call with host-normalised fp32 (B,3,256,256) crops (PCIe-bound)"},
            "gpu_launches": int(launches * args.steps),
            "gpu_launches_per_step": int(launches),
            "clocks": clocks.summary(),
            "roofline": roofline,
            "roofline_path": {"bound": "hbm", "achieved": path_gbs, "peak": peak, "unit": "GB/s",
                              "frac": path_gbs / peak, "what": "whole track() against the block-fused byte budget "
                                                               "(14,947,328 B/frame)"},
            "stages": stage_report,
            "parity_check": parity,
            "stream": stream_line,
            "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
