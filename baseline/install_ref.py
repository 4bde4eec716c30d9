#!/usr/bin/env python
"""Install the UNMODIFIED reference files of the CPD path into the git-ignored ``baseline/_ref`` (bench.py --impl reference).

``pip install /root/reference`` cannot work here: the six pybind11 extensions need Eigen, an un-vendored submodule that is
missing (SURVEY section 8c), and ``probreg/__init__.py`` imports open3d / transforms3d, which are absent.  The CPD path
itself is pure Python + numpy/scipy, so the files it consists of are copied byte for byte (checksums recorded in
``baseline/_ref/MANIFEST.json``); nothing under ``baseline/_ref`` is tracked by git, and nothing in the product imports it.
Runs only where ``/root/reference`` exists (the build container); the GPU box uses the copy that travelled with gpurun.
"""
import hashlib
import json
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
FILES = ["cpd.py", "transformation.py", "math_utils.py", "log.py", "version.py"]


def install(ref="/root/reference", force=False):
    src_dir = os.path.join(ref, "probreg")
    dst_dir = os.path.join(HERE, "_ref", "probreg")
    if not os.path.isdir(src_dir):
        return os.path.isdir(dst_dir)
    os.makedirs(dst_dir, exist_ok=True)
    manifest = {"source": src_dir, "files": {}}
    for name in FILES:
        s, d = os.path.join(src_dir, name), os.path.join(dst_dir, name)
        data = open(s, "rb").read()
        if force or not os.path.exists(d) or open(d, "rb").read() != data:
            shutil.copyfile(s, d)
        manifest["files"][name] = hashlib.sha256(data).hexdigest()
    with open(os.path.join(HERE, "_ref", "MANIFEST.json"), "w") as f:
        json.dump(manifest, f, indent=1)
    return True


if __name__ == "__main__":
    ok = install(*(sys.argv[1:2] or ["/root/reference"]))
    print("baseline/_ref:", "installed" if ok else "reference checkout not found")
