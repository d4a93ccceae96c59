"""Golden fixture for the restatement test (TEST INFRASTRUCTURE; needs the reference source tree):

    python -m oracle.make_golden_restatement

Imports the reference's UNMODIFIED ``FEARNet`` through ``oracle/ref_shims.py``, strict-loads its shipped checkpoint,
asserts that ``oracle.fear_oracle`` reproduces it bit-for-bit here (fp32 and fp64), and records in
``tests/golden/restatement_seed7.npz`` what ``tests/test_oracle_cpu.py::test_restatement_equals_reference_source``
compares against, so that test runs wherever the repository does:

* ``keys`` / ``sha256`` -- digest of every hot-path checkpoint tensor (fp32 bytes), against which the committed
  weight fixture ``fear_xs_hotpath_state.npz`` is checked;
* ``reg32`` / ``cls32`` / ``reg64`` / ``cls64`` -- the reference network's maps on ``synthetic_crops(2, seed=7)``.
"""
import hashlib
import os

import numpy as np
import torch

from oracle import fear_oracle as fo
from oracle import ref_shims

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden",
                   "restatement_seed7.npz")
R, C = fo.TARGET_REGRESSION_LABEL_KEY, fo.TARGET_CLASSIFICATION_KEY


def tensor_sha256(t: torch.Tensor) -> str:
    return hashlib.sha256(t.detach().contiguous().numpy().tobytes()).hexdigest()


def main() -> None:
    net = ref_shims.build_reference_net()
    net64 = ref_shims.build_reference_net().double()
    sd32 = fo.load_lightning_state(ref_shims.REF_CKPT)
    keys = sorted(fo.hot_path_keys(sd32))
    zt, xt, _, _ = fo.synthetic_crops(2, seed=7)
    with torch.no_grad():
        ref32 = net((zt, xt))
        ref64 = net64((zt.double(), xt.double()))
    mine32 = fo.forward(sd32, zt, xt)
    mine64 = fo.forward(fo.to_dtype(sd32, torch.float64), zt.double(), xt.double())
    for key in (R, C):
        assert torch.equal(ref32[key], mine32[key]), f"restatement differs from reference (fp32 {key})"
        assert torch.equal(ref64[key], mine64[key]), f"restatement differs from reference (fp64 {key})"
    np.savez_compressed(
        OUT, keys=np.array(keys), sha256=np.array([tensor_sha256(sd32[k]) for k in keys]),
        reg32=ref32[R].numpy(), cls32=ref32[C].numpy(), reg64=ref64[R].numpy(), cls64=ref64[C].numpy())
    print("restatement golden written to", OUT, "--", len(keys), "checkpoint tensors")


if __name__ == "__main__":
    main()
