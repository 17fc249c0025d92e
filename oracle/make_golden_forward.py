"""Generate tests/golden/reference_forward.npz from the UNMODIFIED reference source tree:

    python oracle/make_golden_forward.py <reference source tree>

The fixture holds what tests/test_cpu_oracle.py::test_oracle_against_live_reference compares the oracle with: the
state-dict layout of the reference's `BeatThis` module (names and shapes; `load_model` loads strictly, so a synthetic
checkpoint of that layout is one the reference accepts), its forward on a seeded [2, 100, 128] batch through the small0
checkpoint, and the chunk starts of its `split_piece` for a few lengths around the chunk borders.
"""
from __future__ import annotations

import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

# the seeded inputs; the test regenerates them from the same values
FORWARD_SEED = 4
SPLIT_LENGTHS = (1, 1488, 1489, 3001)


def main(reference_dir: str):
    sys.path.insert(0, os.path.join(HERE, "shims"))
    sys.path.insert(0, os.path.abspath(reference_dir))
    sys.path.insert(0, ROOT)
    import tempfile

    import numpy as np
    import torch

    import beat_this.inference as ref_inf  # the reference

    from beat_this_b200 import synthetic
    from oracle import beat_this_oracle as O

    out = {}
    with tempfile.TemporaryDirectory() as td:
        path = synthetic.write_checkpoint(os.path.join(td, "small0_s0.ckpt"), "small0", 0)
        model = ref_inf.load_model(path, "cpu")
        sd = O.strip_prefix(torch.load(path, weights_only=True)["state_dict"])
    layout = model.state_dict()
    out["state_keys"] = np.asarray(list(layout))
    out["state_shapes"] = np.asarray([str(tuple(v.shape)) for v in layout.values()])
    out["small0_ckpt_sum"] = np.float64(synthetic.tensor_checksum(sd))
    torch.manual_seed(FORWARD_SEED)
    x = torch.rand(2, 100, 128) * 7
    with torch.inference_mode():
        ref = model(x)
    out["beat"] = ref["beat"].numpy()
    out["downbeat"] = ref["downbeat"].numpy()
    for T in SPLIT_LENGTHS:
        _, starts = ref_inf.split_piece(torch.zeros(T, 1), 1500, 6, True)
        out[f"starts_{T}"] = np.asarray(starts, dtype=np.int64)
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "reference_forward.npz"), **out)
    print(f"{len(layout)} state entries, beat logits {tuple(ref['beat'].shape)}")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
