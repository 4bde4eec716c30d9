#!/usr/bin/env python
"""Write tests/golden/ref_data/: the reference's example data files that tests/test_io.py reads, small enough to commit.

bunny.pcd, fish_source.txt and fish_target.txt are copied unchanged.  cloud_0.pcd keeps its header and its first 500 points.
horse.ply keeps its header layout (binary_big_endian, x y z confidence red green blue, then a face list) but only the first vertex
of every occupied voxel of the 0.01 grid plus the vertices at the minimum of each axis, so that the grid (anchored at the minimum
corner) and its number of occupied voxels are those of the full file; the faces are the ones whose three vertices were kept.

Usage:  python tests/golden/make_ref_data.py <probreg checkout>
"""
import os
import re
import shutil
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "ref_data")
CLOUD_POINTS = 500
HORSE_VOXEL = 0.01


def shrink_pcd(src, dst, keep):
    lines = open(src).read().splitlines()
    start = next(i for i, l in enumerate(lines) if l.startswith("DATA")) + 1
    head = [re.sub(r"^(WIDTH|POINTS) \d+$", r"\1 %d" % keep, l) for l in lines[:start]]
    with open(dst, "w") as f:
        f.write("\n".join(head + lines[start:start + keep]) + "\n")


def shrink_horse(src, dst):
    with open(src, "rb") as f:
        head = []
        while not head or head[-1] != b"end_header\n":
            head.append(f.readline())
        body = f.read()
    n_vertex = int(next(l for l in head if l.startswith(b"element vertex")).split()[2])
    n_face = int(next(l for l in head if l.startswith(b"element face")).split()[2])
    vdt = np.dtype([("x", ">f4"), ("y", ">f4"), ("z", ">f4"), ("confidence", ">f4"), ("red", "u1"), ("green", "u1"), ("blue", "u1")])
    fdt = np.dtype([("n", "u1"), ("v", ">i4", (3,))])
    assert len(body) == vdt.itemsize * n_vertex + fdt.itemsize * n_face
    v = np.frombuffer(body, dtype=vdt, count=n_vertex)
    faces = np.frombuffer(body, dtype=fdt, count=n_face, offset=vdt.itemsize * n_vertex)
    assert np.all(faces["n"] == 3)
    xyz = np.stack([v["x"], v["y"], v["z"]], axis=1).astype(np.float64)
    key = np.floor((xyz - xyz.min(axis=0)) / HORSE_VOXEL).astype(np.int64)
    _, first = np.unique(key, axis=0, return_index=True)
    keep = np.unique(np.concatenate([first, xyz.argmin(axis=0)]))
    new_index = np.full(n_vertex, -1, dtype=np.int64)
    new_index[keep] = np.arange(keep.size)
    kept_faces = faces[np.all(new_index[faces["v"]] >= 0, axis=1)].copy()
    kept_faces["v"] = new_index[kept_faces["v"]]
    head = [b"element vertex %d\n" % keep.size if l.startswith(b"element vertex") else
            b"element face %d\n" % kept_faces.size if l.startswith(b"element face") else l for l in head]
    with open(dst, "wb") as f:
        f.write(b"".join(head) + v[keep].tobytes() + kept_faces.tobytes())
    return keep.size, kept_faces.size


def main(ref):
    os.makedirs(OUT, exist_ok=True)
    for name in ("bunny.pcd", "fish_source.txt", "fish_target.txt"):
        shutil.copyfile(os.path.join(ref, "examples", name), os.path.join(OUT, name))
    shrink_pcd(os.path.join(ref, "examples", "cloud_0.pcd"), os.path.join(OUT, "cloud_0.pcd"), CLOUD_POINTS)
    print("horse.ply: %d vertices, %d faces kept" % shrink_horse(os.path.join(ref, "data", "horse.ply"), os.path.join(OUT, "horse.ply")))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
