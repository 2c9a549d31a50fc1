"""Shared helpers of the GPU parity tests (test infrastructure)."""
import hashlib
import importlib.util
import os

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_ref_ext = None
_ref_tried = False

# (n -> m, radii, nsamples) of the four SA levels (reference pvn3d.py:65-111)
SA_LEVELS = [(12288, 2048, (0.0175, 0.025), (16, 32)), (2048, 1024, (0.025, 0.05), (16, 32)),
             (1024, 512, (0.05, 0.1), (16, 32)), (512, 128, (0.1, 0.2), (16, 32))]
# (batch, points) of the DenseFusion + heads parity cases (tests/test_heads_gpu.py)
HEADS_CASES = [(2, 2048), (1, 12288), (2, 1000)]


def digest(a) -> str:
    """SHA-256 of an array's dtype, shape and bytes: the stored form of reference outputs too large to keep."""
    a = np.ascontiguousarray(a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


def state_dict_digest(module) -> str:
    h = hashlib.sha256()
    for k, v in module.state_dict().items():
        h.update(k.encode())
        h.update(digest(v.detach().cpu().numpy()).encode())
    return h.hexdigest()


def sample(a, k, rows=False, seed=0):
    """A fixed, seeded sample of k elements of `a` (flattened), or of k rows of a 2-D `a`, in storage order."""
    a = np.asarray(a)
    n = a.shape[0] if rows else a.size
    pos = np.sort(np.random.default_rng(seed).choice(n, size=min(k, n), replace=False))
    return a[pos] if rows else a.reshape(-1)[pos]


def sa_autograd_inputs():
    """xyz [2,512,3] and features [2,6,512] of the SA-module gradient parity test"""
    return (np.random.default_rng(1).uniform(size=(2, 512, 3)).astype(np.float32),
            np.random.default_rng(3).uniform(size=(2, 6, 512)).astype(np.float32))


def load_ref_ext():
    """The UNMODIFIED reference op library built by oracle/build_ref_ext.sh, or None."""
    global _ref_ext, _ref_tried
    if _ref_tried:
        return _ref_ext
    _ref_tried = True
    path = os.path.join(ROOT, "oracle", "_ref", "_ext.so")
    if not os.path.exists(path):
        return None
    try:
        spec = importlib.util.spec_from_file_location("_ext", path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        _ref_ext = mod
    except Exception as e:  # pragma: no cover
        print("reference _ext not loadable:", e)
        _ref_ext = None
    return _ref_ext


def level_clouds(batch=2, seed0=500, shape="ycb", n=12288):
    """xyz of every SA level for `batch` synthetic frames, computed with the ORACLE's FPS."""
    from oracle import pn2
    from pvn3d_b200 import synth

    frames = [synth.make_frame(shape, n_points=n, seed=seed0 + i) for i in range(batch)]
    xyz = np.stack([f.pcld for f in frames])
    levels = [xyz]
    for (_, m, _, _) in SA_LEVELS:
        if levels[-1].shape[1] <= m:
            break
        idx = pn2.furthest_point_sampling(levels[-1], m)
        levels.append(np.take_along_axis(levels[-1], idx[..., None].astype(np.int64).repeat(3, -1), 1))
    return frames, levels


def t(x, dev):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


_ref_py = None
_ref_py_tried = False


def load_reference_python():
    """The UNMODIFIED reference Python staged by oracle/build_ref_ext.sh under oracle/_ref/py (lib/,
    common.py, datasets/ fixtures), imported on top of pvn3d_b200.compat.install() -- i.e. with this
    package's `_ext` bound at pointnet2_utils.py:19.  Returns a namespace of the reference modules, or
    None when the staging directory is absent."""
    global _ref_py, _ref_py_tried
    if _ref_py_tried:
        return _ref_py
    _ref_py_tried = True
    root = os.path.join(ROOT, "oracle", "_ref", "py")
    if not os.path.isdir(os.path.join(root, "lib")):
        return None
    import types

    from pvn3d_b200 import compat

    compat.install(root)
    try:
        from lib import pvn3d as ref_pvn3d
        from lib.pointnet2_utils import pointnet2_utils as ref_pn2_utils
        from lib.utils import basic_utils as ref_bu
        from lib.utils import meanshift_pytorch as ref_ms
        from lib.utils import pvn3d_eval_utils as ref_eval
    except Exception as e:  # pragma: no cover
        print("reference python not importable:", repr(e))
        return None
    _ref_py = types.SimpleNamespace(pvn3d=ref_pvn3d, pn2_utils=ref_pn2_utils, basic_utils=ref_bu,
                                    meanshift=ref_ms, eval_utils=ref_eval)
    return _ref_py
