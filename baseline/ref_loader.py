"""Load the unmodified reference CPD modules from ``baseline/_ref`` (see install_ref.py) for the CPU arm of bench.py.

The parent package is planted in ``sys.modules`` so that ``probreg/__init__.py`` (which imports every algorithm and their
absent dependencies) is not needed; ``open3d`` is stubbed with the two classes the annotations / isinstance checks name;
``probreg._math`` (pybind11 + Eigen, not buildable here) is replaced by the float32 numpy restatement of
cc/math_utils.cc:5-19 held by the oracle -- it is only reached by ``_initialize`` (sigma2_0) and NonRigidCPD's G, never by the
E-step / M-step the bench times.
"""
import importlib
import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(HERE, "_ref", "probreg")


def available():
    return os.path.isfile(os.path.join(REF_DIR, "cpd.py"))


def load():
    """-> (probreg.cpd, probreg.transformation) of the reference, unmodified."""
    if not available():
        raise RuntimeError("baseline/_ref/probreg is missing: run python baseline/install_ref.py where /root/reference exists")
    if "open3d" not in sys.modules:
        o3 = types.ModuleType("open3d")
        o3.geometry = types.ModuleType("open3d.geometry")
        o3.utility = types.ModuleType("open3d.utility")
        o3.geometry.PointCloud = type("PointCloud", (), {})
        o3.utility.Vector3dVector = type("Vector3dVector", (), {})
        sys.modules["open3d"] = o3
        sys.modules["open3d.geometry"] = o3.geometry
        sys.modules["open3d.utility"] = o3.utility
    pkg = types.ModuleType("probreg")
    pkg.__path__ = [REF_DIR]
    sys.modules["probreg"] = pkg
    root = os.path.dirname(HERE)
    if root not in sys.path:
        sys.path.insert(0, root)
    from oracle import cpd_oracle as orc
    m = types.ModuleType("probreg._math")
    m.squared_kernel = orc.squared_kernel_f32
    m.rbf_kernel = orc.rbf_kernel_f32
    sys.modules["probreg._math"] = m
    pkg._math = m
    return importlib.import_module("probreg.cpd"), importlib.import_module("probreg.transformation")
