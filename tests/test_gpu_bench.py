"""GPU: bench.py --dump-outputs writes what the timed path computed, and two runs with the same arguments agree."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from util import ROOT

FIELDS = ("xyz", "scales", "rotations", "opacities", "shs")


def _run(out_dir, steps):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1", "--gaussians", "2000",
                          "--res", "64", "--views", "4", "--no-cpu-baseline", "--no-extras", "--dump-outputs", str(out_dir)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    return json.loads(lines[0]), {f[:-4]: np.load(os.path.join(out_dir, f)) for f in os.listdir(out_dir)}


@pytest.mark.gpu
def test_dump_outputs_are_the_same_for_the_same_arguments(tmp_path):
    """The inputs are fixed by the workload arguments and no step changes them, so the last step of two runs (here with
    different step counts) returns bit-identical images and radii, and gradients that agree to rounding (float atomics in
    the blend backward).  --steps sets the timed step count of the headline and of the e2e arm."""
    line, a = _run(tmp_path / "a", 2)
    assert line["steps"] == 2 and line["e2e"]["steps"] == 2
    line, b = _run(tmp_path / "b", 3)
    assert line["steps"] == 3 and line["e2e"]["steps"] == 3
    assert set(a) == {"color", "depth", "alpha", "radii"} | {"grad_" + f for f in FIELDS} == set(b)
    assert all(v.dtype == np.float32 for v in a.values()) and sum(v.nbytes for v in a.values()) <= 64 << 20
    assert a["color"].shape == (4, 3, 64 * 64) and a["radii"].shape == (4, 2000) and a["grad_shs"].shape == (2000, 16, 3)
    assert (a["radii"] > 0).any() and float(np.abs(a["grad_xyz"]).max()) > 0
    for k in ("color", "depth", "alpha", "radii"):
        assert np.array_equal(a[k], b[k]), k
    for f in FIELDS:
        got, want = b["grad_" + f], a["grad_" + f]
        assert float(np.abs(got - want).max()) <= 1e-6 + 1e-5 * float(np.abs(want).max()), f
