"""This package's drop-in boundary against outputs recorded from the UNMODIFIED reference on a B200
(tests/golden/ref_modules.npz, written by tests/golden/make_golden_ref_gpu.py from the reference's own Python
and its own compiled `_ext`):

  * the reference `Pointnet2MSG` (pvn3d/lib/pvn3d.py:46-154) on the reference `_ext` with TF32 off: this
    package's mirror module with the same weights (state_dict digest of the reference model), on the drop-in
    `_ext`, must give the SAME BITS under the cuDNN build they were recorded with (every index op is bit-exact, so
    every cuDNN call sees identical operands; the reference module itself on the drop-in `_ext` gave the same bits
    when it was recorded), and agree to 1e-4 of the mean feature magnitude under any other;
  * train_*.py path: the gradients of a reference PointnetSAModuleMSG through its autograd Functions
    (pointnet2_utils.py:67-241) vs the mirror's, i.e. gather_points_grad / group_points_grad of the drop-in;
  * the reference `cal_frame_poses` / `cal_frame_poses_lm` (pvn3d_eval_utils.py:37-110,156-201), executed as
    written on CUDA tensors with the reference `MeanShiftTorch`, vs the entry points compat.patch_post_modules()
    binds in their place (what demo.py:22,98-119 would run): class ids equal, poses within 1e-4.
"""
import os

import numpy as np
import pytest
import torch

from pvn3d_b200 import eval_utils, pointnet2, synth, testing

from helpers import digest, sa_autograd_inputs, sample, state_dict_digest, t

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ref(golden_dir):
    return np.load(os.path.join(golden_dir, "ref_modules.npz"))


def _pose_close(p, q, tol=1e-4):
    dr = np.linalg.norm(p[:, :3] - q[:, :3])
    dt = np.linalg.norm(p[:, 3] - q[:, 3]) / max(np.linalg.norm(q[:, 3]), 1e-9)
    return dr <= tol * np.sqrt(3) and dt <= tol, (dr, dt)


def test_reference_pointnet2msg_on_dropin_ext_is_bit_identical(cuda_dev, ref):
    mine = testing.seeded_pointnet2msg(0, 1)
    assert state_dict_digest(mine) == str(ref["pn2msg_state_dict"]), "weights differ from the reference model's"
    mine = mine.to(cuda_dev)
    frames = synth.make_batch("ycb", 2, n_points=12288, config_id=11)
    x = torch.from_numpy(np.stack([f.cld_rgb_nrm for f in frames])).to(cuda_dev)
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            y = mine(x)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
    assert y.shape == (2, 128, 12288)
    y = y.cpu().numpy()
    s, want = sample(y, 4096), ref["pn2msg_sample"]
    assert float(np.abs(s - want).max()) <= 1e-4 * float(ref["pn2msg_abs_mean"])
    # the index ops are bit-exact, so every convolution sees the reference's operands; which fp32 algorithm cuDNN runs
    # depends on its build, so the bits themselves are asserted under the cuDNN the features were recorded with
    if torch.backends.cudnn.version() == int(ref["cudnn_version"]):
        assert np.array_equal(s, want) and digest(y) == str(ref["pn2msg_digest"])


def test_reference_sa_module_autograd_on_dropin_ext(cuda_dev, ref):
    """train_*.py path: the autograd Functions call gather_points_grad / group_points_grad of the drop-in"""
    torch.manual_seed(1)
    sa = pointnet2.PointnetSAModuleMSG(npoint=64, radii=[0.1, 0.2], nsamples=[8, 16], mlps=[[6, 16, 32], [6, 16, 32]])
    assert state_dict_digest(sa) == str(ref["sa_state_dict"]), "weights differ from the reference module's"
    sa = sa.to(cuda_dev).eval()
    xyz, feat = sa_autograd_inputs()
    feat = t(feat, cuda_dev).requires_grad_(True)
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        _, out = sa(t(xyz, cuda_dev), feat)
        out.square().sum().backward()
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    want = t(ref["sa_grad"], cuda_dev)
    # scatter-adds accumulate in a different order: float tolerance, not bits
    assert torch.allclose(feat.grad, want, rtol=1e-4, atol=1e-5 * float(want.abs().max()))


@pytest.mark.parametrize("shape", ["ycb", "linemod"])
def test_reference_cal_frame_poses_vs_patched(cuda_dev, ref, shape):
    """reference post-processing on CUDA tensors (what demo.py runs) vs the entry points compat.patch_post_modules()
    binds in its place"""
    f = synth.make_frame(shape, n_points=4096, seed=77, lm_obj_id=1 if shape == "linemod" else None)
    args = [t(a, cuda_dev) for a in (f.pcld, f.labels, f.ctr_of, f.kp_of)]
    if shape == "ycb":
        ids, poses = eval_utils.cal_frame_poses(*args, True, 22, True)
        assert np.array_equal(ids, ref["frame_poses_ycb_ids"])
    else:
        poses = eval_utils.cal_frame_poses_lm(*args, True, 2, False, 1)
    poses_ref = ref[f"frame_poses_{shape}"]
    assert len(poses) == len(poses_ref)
    for p, q in zip(poses, poses_ref):
        # the reference ran torch CUDA kernels (soft cross-check: their norm / sum may round differently from
        # the CPU kernels the contract is pinned to), still well inside the bar
        ok, err = _pose_close(np.asarray(p, np.float64), np.asarray(q, np.float64))
        assert ok, err
