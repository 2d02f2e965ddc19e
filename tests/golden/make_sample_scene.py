"""Packs the reference's only real scene, content/sample.ply (531 327 Gaussians, SH degree 0), into
tests/golden/sample_ply_full.npz so that the GPU box (no /root/reference there) can run BASELINE configs 2, 4 and 5 on
the real anisotropy / opacity distribution.  Run in the authoring container only:

    python tests/golden/make_sample_scene.py

Stored: `data` float32 [N,14] = the 14 non-constant PLY columns (x y z f_dc_0..2 opacity scale_0..2 rot_0..3) in file
order, `columns` = their names.  The three normal columns of the file are identically 0 (checked) and not stored.
humangaussian_b200.scene.sample_ply_scene() rebuilds the raw GaussianParams exactly as the reference's load_ply does
(gaussiansplatting/scene/gaussian_model.py:225-266); tests/test_ply_codec.py checks the rebuilt tensors against what the
PLY codec reads from the file itself (recorded by make_sample_ply_check.py).
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from humangaussian_b200.scene import SAMPLE_COLUMNS, read_ply  # noqa: E402

REF_PLY = "/root/reference/content/sample.ply"


def main():
    c = read_ply(REF_PLY)
    for k in ("nx", "ny", "nz"):
        assert not np.any(c[k]), "normals are expected to be all zero"
    data = np.stack([c[k] for k in SAMPLE_COLUMNS], axis=1).astype(np.float32)
    out = os.path.join(HERE, "sample_ply_full.npz")
    np.savez_compressed(out, data=data, columns=np.array(SAMPLE_COLUMNS))
    print(out, data.shape, os.path.getsize(out) / 1e6, "MB")


if __name__ == "__main__":
    main()
