"""CPU: the PLY codec (humangaussian_b200/scene.py) against fixtures produced by RUNNING the reference's own save_ply /
load_ply (tests/golden/make_golden_ply.py): gaussiansplatting/scene/gaussian_model.py:187-266 (training convention) and
gs_renderer.py:525-610 (animation convention: y/z swap, quaternion 2<->3 swap, component-0 negation, file-order columns)."""
import hashlib
import os

import numpy as np
import pytest
import torch

from util import ROOT

from humangaussian_b200.scene import GaussianParams, params_from_ply, params_to_ply, read_ply, sample_ply_scene, write_ply

G = np.load(os.path.join(ROOT, "tests", "golden", "ref_ply.npz"))
KEYS = ("xyz", "features_dc", "features_rest", "opacity", "scaling", "rotation")


def _file(tmp_path, key):
    p = tmp_path / (key + ".ply")
    p.write_bytes(G[key].tobytes())
    return str(p)


@pytest.mark.parametrize("deg", [0, 2])
def test_load_matches_reference_loaders(tmp_path, deg):
    path = _file(tmp_path, f"deg{deg}_file")
    for conv, tag in (("training", "train"), ("animation", "anim")):
        p = params_from_ply(path, sh_degree=deg, convention=conv)
        for k in KEYS:
            ref = G[f"deg{deg}_{tag}_{k}"]
            got = getattr(p, k).numpy()
            assert got.shape == ref.shape, (conv, k, got.shape, ref.shape)
            assert np.array_equal(got, ref), (conv, k)


@pytest.mark.parametrize("deg", [0, 2])
def test_save_writes_the_reference_file_byte_for_byte(tmp_path, deg):
    t = lambda k: torch.tensor(G[f"deg{deg}_saved_{k}"])
    p = GaussianParams(t("xyz"), t("features_dc"), t("features_rest"), t("scaling"), t("rotation"), t("opacity"), deg)
    out = tmp_path / "out.ply"
    params_to_ply(str(out), p)
    assert out.read_bytes() == G[f"deg{deg}_file"].tobytes()
    # and the round trip through our own loader returns the saved tensors exactly
    q = params_from_ply(str(out), sh_degree=deg)
    for k in KEYS:
        assert torch.equal(getattr(q, k), getattr(p, k)), k


def test_column_order_conventions_differ_as_in_the_reference(tmp_path):
    """scale_*/rot_* columns stored out of index order: the training loader sorts them, the animation loader takes file
    order (then applies its axis swaps) -- both reproduced."""
    path = _file(tmp_path, "shuf_file")
    for conv, tag in (("training", "train"), ("animation", "anim")):
        p = params_from_ply(path, sh_degree=0, convention=conv)
        for k in ("xyz", "scaling", "rotation", "opacity", "features_dc"):
            assert np.array_equal(getattr(p, k).numpy(), G[f"shuf_{tag}_{k}"]), (conv, k)
    assert not np.array_equal(G["shuf_train_scaling"], G["shuf_anim_scaling"][:, [0, 2, 1]])


def test_animation_convention_is_the_documented_permutation(tmp_path):
    path = _file(tmp_path, "deg0_file")
    a, b = params_from_ply(path, 0, "training"), params_from_ply(path, 0, "animation")
    assert torch.equal(b.xyz, a.xyz[:, [0, 2, 1]]) and torch.equal(b.scaling, a.scaling[:, [0, 2, 1]])
    assert torch.equal(b.rotation[:, 0], -a.rotation[:, 0]) and torch.equal(b.rotation[:, 1], a.rotation[:, 1])
    assert torch.equal(b.rotation[:, 2], a.rotation[:, 3]) and torch.equal(b.rotation[:, 3], a.rotation[:, 2])


def test_reader_rejects_what_it_cannot_parse(tmp_path):
    bad = tmp_path / "ascii.ply"
    bad.write_bytes(b"ply\nformat ascii 1.0\nelement vertex 1\nproperty float x\nend_header\n0.0\n")
    with pytest.raises(ValueError):
        read_ply(str(bad))
    bad.write_bytes(b"ply\nformat binary_little_endian 1.0\nelement vertex 1\nproperty double x\nend_header\n" + b"\0" * 8)
    with pytest.raises(ValueError):
        read_ply(str(bad))
    ok = tmp_path / "ok.ply"
    write_ply(str(ok), {"x": np.arange(3, dtype=np.float32), "y": np.ones(3, np.float32)})
    c = read_ply(str(ok))
    assert list(c) == ["x", "y"] and np.array_equal(c["x"], [0, 1, 2])
    with pytest.raises(ValueError):
        params_from_ply(_file(tmp_path, "deg2_file"), sh_degree=1)  # wrong number of f_rest columns for the degree


def test_sample_scene_pack_matches_the_ply():
    """tests/golden/sample_ply_full.npz is content/sample.ply repacked: same tensors as loading the PLY itself, as recorded
    from the reference's file by tests/golden/make_sample_ply_check.py (bit-exact digests of every tensor, plus sampled rows)."""
    p = sample_ply_scene()
    assert p.P == 531327 and p.features_rest.shape == (531327, 0, 3)
    op = torch.sigmoid(p.opacity)
    assert abs(float(op.mean()) - 0.103) < 2e-3                      # SURVEY.md 8c's measured statistics of the file
    assert abs(float(torch.exp(p.scaling).median()) - 0.0028) < 2e-4
    ply = np.load(os.path.join(ROOT, "tests", "golden", "sample_ply_check.npz"))
    rows = torch.from_numpy(ply["row_index"])
    for conv in ("training", "animation"):
        r = sample_ply_scene(convention=conv)
        for k in KEYS:
            t = getattr(r, k)
            assert list(t.shape) == ply[f"{conv}_{k}_shape"].tolist(), (conv, k)
            assert np.array_equal(t[rows].numpy(), ply[f"{conv}_{k}_rows"]), (conv, k)
            digest = hashlib.sha256(np.ascontiguousarray(t.numpy(), dtype=np.float32).tobytes()).hexdigest()
            assert digest == str(ply[f"{conv}_{k}_sha256"]), (conv, k)
    s = sample_ply_scene(300000, 3)
    assert s.P == 300000 and s.features_rest.shape == (300000, 15, 3) and abs(float(s.features_rest.std()) - 0.1) < 1e-3
