"""probreg_b200.io: readers and the voxel down-sampler (CPU; also on the reference's example data, kept under tests/golden/ref_data)."""
import os
import struct

import numpy as np
import pytest

from conftest import GOLDEN
from probreg_b200 import io as pio

REF_DATA = os.path.join(GOLDEN, "ref_data")


def test_pcd_and_txt_roundtrip(tmp_path):
    pts = np.random.default_rng(0).random((50, 3))
    p = tmp_path / "a.pcd"
    p.write_text("# .PCD v0.7\nVERSION 0.7\nFIELDS x y z intensity\nSIZE 4 4 4 4\nTYPE F F F F\nCOUNT 1 1 1 1\nWIDTH 50\nHEIGHT 1\n"
                 "POINTS 50\nDATA ascii\n" + "\n".join("%r %r %r 0" % tuple(r) for r in pts.tolist()) + "\n")
    np.testing.assert_allclose(pio.read_points(str(p)), pts, rtol=0, atol=0)
    t = tmp_path / "a.txt"
    np.savetxt(str(t), pts[:, :2])
    np.testing.assert_allclose(pio.read_points(str(t)), pts[:, :2])


@pytest.mark.parametrize("fmt,order", [("binary_big_endian", ">"), ("binary_little_endian", "<"), ("ascii", None)])
def test_ply_vertices(tmp_path, fmt, order):
    pts = np.random.default_rng(1).random((20, 3)).astype(np.float32)
    head = ("ply\nformat %s 1.0\ncomment test\nelement vertex 20\nproperty float32 x\nproperty float32 y\nproperty float32 z\n"
            "property uint8 red\nelement face 1\nproperty list uint8 int32 vertex_indices\nend_header\n" % fmt).encode()
    if order is None:
        body = "".join("%r %r %r 7\n" % tuple(float(v) for v in r) for r in pts).encode() + b"3 0 1 2\n"
    else:
        body = b"".join(struct.pack(order + "fffB", *r, 7) for r in pts.tolist()) + struct.pack(order + "Biii", 3, 0, 1, 2)
    p = tmp_path / "a.ply"
    p.write_bytes(head + body)
    np.testing.assert_allclose(pio.read_ply(str(p)), pts.astype(np.float64), rtol=1e-7)


def test_voxel_down_sample():
    pts = np.array([[0.0, 0, 0], [0.1, 0.1, 0.1], [0.9, 0.9, 0.9], [1.2, 0, 0], [1.3, 0.1, 0.0]])
    out = pio.voxel_down_sample(pts, 1.0)
    assert out.shape == (2, 3)
    np.testing.assert_allclose(sorted(out[:, 0]), [1.0 / 3, 1.25])
    rng = np.random.default_rng(2)
    cloud = rng.random((5000, 3))
    ds = pio.voxel_down_sample(cloud, 0.25)
    assert ds.shape[0] == 64 and np.all(ds >= 0) and np.all(ds <= 1)
    with pytest.raises(ValueError):
        pio.voxel_down_sample(cloud, 0.0)


def test_reference_fixtures_load():
    bunny = pio.read_points(os.path.join(REF_DATA, "bunny.pcd"))
    assert bunny.shape == (397, 3)                                            # examples/bunny.pcd:9
    assert abs(pio.voxel_down_sample(bunny, 0.005).shape[0] - 381) <= 12      # SURVEY: ~381 points at voxel 0.005
    # data/horse.ply (binary_big_endian, 48 485 vertices) shrunk to one vertex per occupied voxel of the 0.01 grid, which keeps
    # the full file's voxel count (tests/golden/make_ref_data.py)
    horse = pio.read_points(os.path.join(REF_DATA, "horse.ply"))
    assert horse.shape == (490, 3)
    assert abs(pio.voxel_down_sample(horse, 0.01).shape[0] - 480) <= 40       # tests/test_cpd.py recipe: ~480 points
    assert pio.read_points(os.path.join(REF_DATA, "cloud_0.pcd")).shape == (500, 3)      # the first 500 of 6 535 points
    assert pio.read_points(os.path.join(REF_DATA, "fish_source.txt")).shape == (91, 2)


def test_example_utils_follow_the_reference_recipes(monkeypatch):
    """examples/utils.py: numpy counterparts of the reference's examples/utils.py (rigid recipe: voxel filter, shuffle, noise,
    outliers, 30 degrees about z; non-rigid: the two text clouds, voxel-filtered)."""
    import os
    import sys

    import numpy as np

    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples"))
    import utils as ex

    r = ex.euler2mat(0.1, -0.2, 0.3)
    np.testing.assert_allclose(r.dot(r.T), np.identity(3), atol=1e-15)
    np.testing.assert_allclose(ex.euler2mat(0.0, 0.0, np.deg2rad(30.0))[:2, :2], [[np.cos(np.pi / 6), -0.5], [0.5, np.cos(np.pi / 6)]], atol=1e-15)
    monkeypatch.setenv("PROBREG_EXAMPLES", REF_DATA)
    bunny = ex.reference_file("bunny.pcd")
    assert bunny is not None
    src, tgt = ex.prepare_source_and_target_rigid_3d(bunny, rng=np.random.default_rng(0))
    assert src.shape[1] == 3 and tgt.shape == (src.shape[0] + 500, 3)
    # undo the known transform: the inliers are the (shuffled, slightly noised) source
    back = tgt[: src.shape[0]].dot(ex.euler2mat(0.0, 0.0, np.deg2rad(30.0)))
    d = np.sqrt(((back[:, None, :] - src[None, :, :]) ** 2).sum(-1)).min(axis=1)
    assert d.max() < 0.01
    fish = ex.prepare_source_and_target_nonrigid_2d(ex.reference_file("fish_source.txt"), ex.reference_file("fish_target.txt"))
    assert fish[0].shape == (91, 2) and fish[1].shape == (91, 2)


def test_ply_with_an_element_in_front_of_the_vertices(tmp_path):
    """Legal PLY: another element may precede `vertex`; its rows are skipped (ascii and binary)."""
    import struct

    pts = np.arange(15, dtype=np.float32).reshape(5, 3)
    head = ("ply\nformat %s 1.0\nelement camera 2\nproperty float32 fx\nproperty int32 id\nelement vertex 5\n"
            "property float32 x\nproperty float32 y\nproperty float32 z\nend_header\n")
    p = tmp_path / "pre_ascii.ply"
    p.write_text(head % "ascii" + "1.5 7\n2.5 8\n" + "\n".join(" ".join("%g" % v for v in r) for r in pts) + "\n")
    np.testing.assert_allclose(pio.read_ply(str(p)), pts)
    p = tmp_path / "pre_bin.ply"
    with open(str(p), "wb") as f:
        f.write((head % "binary_little_endian").encode())
        f.write(struct.pack("<fi", 1.5, 7) + struct.pack("<fi", 2.5, 8))
        f.write(pts.astype("<f4").tobytes())
    np.testing.assert_allclose(pio.read_ply(str(p)), pts)
