"""Records what the PLY codec reads from the reference's content/sample.ply, so that tests/test_ply_codec.py can check the
committed column pack (sample_ply_full.npz) against the original file without having it:

    python tests/golden/make_sample_ply_check.py <reference checkout>/content/sample.ply

Stored in sample_ply_check.npz, for both load conventions ("training", "animation") and every parameter tensor of
params_from_ply(sample.ply, sh_degree=0): `<conv>_<key>_sha256` = SHA-256 of the tensor's contiguous float32 bytes
(a bit-exact check of all 531 327 rows), `<conv>_<key>_rows` = the rows at `row_index` (a seed-0 sample of 512 rows, so that a
mismatch shows where and by how much), and `<conv>_<key>_shape`.
"""
import hashlib
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from humangaussian_b200.scene import params_from_ply  # noqa: E402

KEYS = ("xyz", "features_dc", "features_rest", "opacity", "scaling", "rotation")
N_ROWS = 512


def sha256(t):
    return hashlib.sha256(np.ascontiguousarray(t.numpy(), dtype=np.float32).tobytes()).hexdigest()


def main(ply):
    out = {}
    for conv in ("training", "animation"):
        p = params_from_ply(ply, 0, conv)
        if "row_index" not in out:
            g = torch.Generator().manual_seed(0)
            out["row_index"] = torch.randperm(p.P, generator=g)[:N_ROWS].sort().values.numpy()
        for k in KEYS:
            t = getattr(p, k)
            out[f"{conv}_{k}_sha256"] = np.array(sha256(t))
            out[f"{conv}_{k}_shape"] = np.array(t.shape, np.int64)
            out[f"{conv}_{k}_rows"] = t[torch.from_numpy(out["row_index"])].numpy()
    path = os.path.join(HERE, "sample_ply_check.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path) / 1e3, "kB")


if __name__ == "__main__":
    main(sys.argv[1])
