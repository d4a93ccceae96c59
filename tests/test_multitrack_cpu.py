"""CPU: FearFrame / FearTrack layouts against the C header, and FEARMultiTracker's argument checks (no GPU needed)."""
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

import feartracker_b200 as fb
from feartracker_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_LAYOUT_C = r"""
#include <stddef.h>
#include <stdio.h>
#include "fear_b200.h"
#define F(T, m) printf("%s.%s %zu\n", #T, #m, offsetof(T, m))
int main(void) {
  printf("FearFrame %zu\nFearTrack %zu\n", sizeof(FearFrame), sizeof(FearTrack));
  F(FearFrame, data); F(FearFrame, h); F(FearFrame, w);
  F(FearTrack, x); F(FearTrack, y); F(FearTrack, w); F(FearTrack, h);
  F(FearTrack, cx); F(FearTrack, cy); F(FearTrack, cw); F(FearTrack, ch);
  F(FearTrack, pad_r); F(FearTrack, pad_g); F(FearTrack, pad_b); F(FearTrack, reserved);
  return 0;
}
"""


def test_frame_and_track_layouts_match_the_header(tmp_path):
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no host C compiler")
    src, exe = tmp_path / "layout.c", tmp_path / "layout"
    src.write_text(_LAYOUT_C)
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(line.rsplit(" ", 1) for line in subprocess.run([str(exe)], capture_output=True, text=True,
                                                              check=True).stdout.split("\n") if line)
    assert int(got["FearFrame"]) == _lib.FRAME_DTYPE.itemsize
    assert int(got["FearTrack"]) == _lib.TRACK_DTYPE.itemsize
    for struct, dtype in (("FearFrame", _lib.FRAME_DTYPE), ("FearTrack", _lib.TRACK_DTYPE)):
        for name in dtype.names:
            assert int(got[f"{struct}.{name}"]) == dtype.fields[name][1], (struct, name)


@pytest.fixture()
def tracker():
    net = fb.FEARNet(**fb.FEAR_XS_MODEL_KWARGS)
    return fb.FEARMultiTracker(net, cuda_id=0, max_tracks=8, **fb.FEAR_XS_TRACKER_KWARGS)


def test_unsupported_configurations_raise():
    net = fb.FEARNet(**fb.FEAR_XS_MODEL_KWARGS)
    for extra in ({"smooth": True}, {"host_normalize": True}):
        with pytest.raises(NotImplementedError):
            fb.FEARMultiTracker(net, **extra, **fb.FEAR_XS_TRACKER_KWARGS)
    with pytest.raises(ValueError):
        fb.FEARMultiTracker(net, max_tracks=0, **fb.FEAR_XS_TRACKER_KWARGS)


def test_initialize_argument_validation(tracker):
    frame = np.zeros((48, 64, 3), np.uint8)
    with pytest.raises(ValueError, match="rects"):
        tracker.initialize(frame, np.zeros((2, 3)))
    with pytest.raises(ValueError, match="max_tracks"):
        tracker.initialize(frame, np.zeros((9, 4)))
    with pytest.raises(ValueError, match="one frame per rect"):
        tracker.initialize([frame, frame], np.zeros((3, 4)))
    with pytest.raises(ValueError, match="uint8"):
        tracker.initialize(frame.astype(np.float32), [[1, 1, 4, 4]])
    with pytest.raises(ValueError, match="uint8"):
        tracker.initialize(np.zeros((48, 64, 4), np.uint8), [[1, 1, 4, 4]])
    with pytest.raises(ValueError, match="uint8"):
        tracker.initialize([frame, np.zeros((48, 64), np.uint8)], np.zeros((2, 4)))
    with pytest.raises(TypeError):
        tracker.initialize(["not a frame"], [[1, 1, 4, 4]])
    with pytest.raises(ValueError, match="track_ids"):
        tracker.initialize(frame, [[1, 1, 4, 4]], track_ids=[0])  # no tracks yet


def test_update_argument_validation(tracker):
    frame = np.zeros((48, 64, 3), np.uint8)
    with pytest.raises(RuntimeError, match="before initialize"):
        tracker.update(frame)
    tracker.num_tracks = 3  # as after initialize(frame, three rects)
    frames = [frame, frame]
    with pytest.raises(ValueError, match="pass frame_of_track"):
        tracker.update(frames)
    for bad in ([0, 1], [0, 1, 2], [0, -2, 1], [0.0, 1.0, 1.0], [[0, 1, 1]]):
        with pytest.raises(ValueError, match="frame_of_track"):
            tracker.update(frames, frame_of_track=bad)
    with pytest.raises(ValueError, match="uint8"):
        tracker.update(np.zeros((3, 48, 64, 2), np.uint8))
    with pytest.raises(ValueError, match="max_tracks"):
        tracker.update([frame] * 9, frame_of_track=[0, 1, 2])


def test_fails_loudly_without_a_gpu(tracker):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    frame = np.zeros((48, 64, 3), np.uint8)
    with pytest.raises(RuntimeError, match="CUDA"):
        tracker.initialize(frame, [[1, 1, 4, 4]])
    tracker.num_tracks = 1
    with pytest.raises(RuntimeError, match="CUDA"):
        tracker.update(frame)
