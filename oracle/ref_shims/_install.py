"""Shims that let the UNMODIFIED reference package (/root/reference/lab4d) import and run on CPU
in the build container.  TEST INFRASTRUCTURE ONLY: used by oracle/gen_golden.py to produce the
golden vectors under tests/golden/.  Nothing in lab4d_b200/ imports this.

What is stubbed (all cold-path dependencies that are absent offline, SURVEY.md §8c):
  trimesh, pysdf, skimage.measure, matplotlib(.pyplot/.cm), imageio, and the dqtorch `quaternion`
  extension, which is replaced by a pure-torch module with the CUDA kernel's semantics
  (3-vectors are pure quaternions, lab4d/third_party/quaternion/src/quaternion.cu:46-57).
"""
import sys
import types

import numpy as np
import torch

import os

# The reference checkout when it exists, else the git-ignored copy of its package
# (oracle/_ref, written by oracle/make_ref.py / __graft_entry__.build()).
_HERE = os.path.dirname(os.path.abspath(__file__))
_REF_COPY = os.path.normpath(os.path.join(_HERE, "..", "_ref"))
REF_ROOT = os.environ.get("LAB4D_REF_ROOT") or ("/root/reference" if os.path.isdir("/root/reference/lab4d") else _REF_COPY)


def available():
    return os.path.isdir(os.path.join(REF_ROOT, "lab4d"))


def _mod(name, **attrs):
    m = types.ModuleType(name)
    for k, v in attrs.items():
        setattr(m, k, v)
    sys.modules[name] = m
    return m


class _FakeMesh:
    def __init__(self, vertices=None, faces=None, **kw):
        self.vertices = np.zeros((8, 3), np.float32) if vertices is None else np.asarray(vertices)
        self.faces = np.zeros((0, 3), np.int64) if faces is None else np.asarray(faces)

    @property
    def bounds(self):
        return np.stack([self.vertices.min(0), self.vertices.max(0)], 0)

    def export(self, *a, **k):
        pass

    def apply_transform(self, *a, **k):
        return self


def _uv_sphere(radius=1.0, count=(4, 4)):
    c = np.array([[x, y, z] for x in (-1, 1) for y in (-1, 1) for z in (-1, 1)], np.float32)
    return _FakeMesh(vertices=c * radius / np.sqrt(3.0))


def _corners(bounds):
    lo, hi = np.asarray(bounds)
    return np.array([[x, y, z] for x in (lo[0], hi[0]) for y in (lo[1], hi[1]) for z in (lo[2], hi[2])])


def _qpad(x):
    if x.shape[-1] == 3:
        return torch.cat([torch.zeros_like(x[..., :1]), x], -1)
    return x


def _quaternion_mul(a, b):
    a, b = _qpad(a), _qpad(b)
    aw, ax, ay, az = a.unbind(-1)
    bw, bx, by, bz = b.unbind(-1)
    return torch.stack(
        (
            aw * bw - ax * bx - ay * by - az * bz,
            aw * bx + ax * bw + ay * bz - az * by,
            aw * by - ax * bz + ay * bw + az * bx,
            aw * bz + ax * by - ay * bx + az * bw,
        ),
        -1,
    )


def _quaternion_conjugate(q):
    return torch.cat((q[..., :1], -q[..., 1:]), -1)


def install():
    if "lab4d" in sys.modules:
        return
    tm = _mod("trimesh", Trimesh=_FakeMesh, load=lambda *a, **k: _uv_sphere(0.5))
    tm.creation = _mod("trimesh.creation", uv_sphere=_uv_sphere)
    tm.bounds = _mod("trimesh.bounds", corners=_corners)
    _mod("pysdf", SDF=lambda *a, **k: (lambda p: np.zeros(len(p))))
    sk = _mod("skimage")
    sk.measure = _mod("skimage.measure", marching_cubes=None)
    mpl = _mod("matplotlib")
    mpl.pyplot = _mod("matplotlib.pyplot")
    mpl.cm = _mod("matplotlib.cm", get_cmap=lambda *a, **k: None)
    mpl.pyplot.cm = mpl.cm
    mpl.pyplot.get_cmap = mpl.cm.get_cmap
    _mod("imageio")
    if not os.path.isdir(os.path.join(REF_ROOT, "preprocess", "third_party", "vcnplus", "flowutils")):
        # visualisation helper of the preprocessing tree (lab4d/utils/vis_utils.py:11-16); absent from the travelling copy
        fu = _mod("flowutils")
        fu.flowlib = _mod("flowutils.flowlib", flow_to_image=lambda *a, **k: None)
    _mod("quaternion", quaternion_mul=_quaternion_mul, quaternion_conjugate=_quaternion_conjugate)
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    import lab4d.utils.quat_transform as qt  # noqa: E402

    # reference CPU branch is broken for 3-vector operands (quat_transform.py:62-81,106-113)
    qt._quaternion_mul = _quaternion_mul
    qt.quaternion_mul = lambda a, b: _quaternion_mul(a, b)
