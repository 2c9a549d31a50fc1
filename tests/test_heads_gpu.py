"""DenseFusion + SEG / KpOF / CtrOf heads (SURVEY section 8 f3) on the tensor-core layer kernel against the same
network evaluated in fp32 torch (TF32 off) on every output, and that evaluation against the REFERENCE modules
(pvn3d/lib/pvn3d.py:157-182,245-267,297-308): the reference's own classes, loaded with the weights of
heads.reference_layout_modules() below and run in fp32 on a B200, recorded as seeded samples of their outputs
(tests/golden/ref_modules.npz, tests/golden/make_golden_ref_gpu.py).

Tolerance: TF32 operands through 6 stacked 1x1 convolutions with K up to 1024 -> mean error <= 3e-3 and max error <=
3e-2 of the mean output magnitude per head (the class of the reference's default cuDNN TF32 path).  The fp32
evaluation here matches the recorded reference samples to 1e-4 of that magnitude (fp32 accumulation order only).
"""
import os

import numpy as np
import pytest
import torch

from pvn3d_b200 import eval_utils, fixtures, heads, testing
from pvn3d_b200.eval_utils import FramePoseSolver

from helpers import HEADS_CASES, sample

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ref_modules(cuda_dev):
    """DenseFusion + the three stacks in the reference's layout, the weights the reference modules were recorded with"""
    torch.manual_seed(3)
    mods = heads.reference_layout_modules(n_classes=22, n_kps=8)
    for i, m in enumerate(mods):
        testing.randomize_bn_(m, 10 + i)
    return [m.to(cuda_dev).eval() for m in mods]


@pytest.fixture(scope="module")
def ref(golden_dir):
    return np.load(os.path.join(golden_dir, "ref_modules.npz"))


def _fp32_forward(mods, rgb_emb, cld_emb):
    """DenseFusion.forward (pvn3d.py:166-182) and the three head stacks (:297-306) in fp32 torch, TF32 off"""
    fusion, seg, kpof, ctrof = mods
    b, _, n = cld_emb.shape
    relu = torch.relu
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            feat_1 = torch.cat((rgb_emb, cld_emb), 1)
            feat_2 = torch.cat((relu(fusion.conv2_rgb(rgb_emb)), relu(fusion.conv2_cld(cld_emb))), 1)
            rgbd = relu(fusion.conv4(relu(fusion.conv3(feat_1))))
            f = torch.cat([feat_1, feat_2, torch.nn.functional.avg_pool1d(rgbd, n).expand(-1, -1, n)], 1)
            return (kpof(f).view(b, 8, 3, n).permute(0, 1, 3, 2).contiguous(), seg(f).transpose(1, 2).contiguous(),
                    ctrof(f).view(b, 1, 3, n).permute(0, 1, 3, 2).contiguous())
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev


@pytest.mark.parametrize("b,n", HEADS_CASES)
def test_fused_heads_match_reference_modules(cuda_dev, ref_modules, ref, b, n):
    g = torch.Generator().manual_seed(n)
    rgb_emb = torch.randn(b, 128, n, generator=g).to(cuda_dev)
    cld_emb = torch.randn(b, 128, n, generator=g).abs().to(cuda_dev)          # PointNet++ features are post-ReLU
    want = _fp32_forward(ref_modules, rgb_emb, cld_emb)
    eng = heads.FusedHeads(*ref_modules, device=cuda_dev)
    got = eng(rgb_emb, cld_emb)
    key = f"heads_{b}x{n}"
    shapes = {"kp_of": (b, 8, n, 3), "seg": (b, n, 22), "ctr_of": (b, 1, n, 3)}
    for name, gt, w in zip(("kp_of", "seg", "ctr_of"), got, want):
        assert gt.shape == shapes[name] == w.shape and gt.is_contiguous(), name
        scale = float(ref[f"{key}_{name}_scale"])
        # the fp32 evaluation is the reference modules' computation: the same numbers at the recorded samples
        w_np = w.cpu().numpy()
        if name == "seg":
            rec = ref[f"{key}_seg_rows"]
            ws = sample(w_np.reshape(b * n, -1), len(rec), rows=True)
        else:
            rec = ref[f"{key}_{name}"]
            ws = sample(w_np, rec.size)
        assert float(np.abs(ws - rec).max()) <= 1e-4 * scale, name
        err = (gt - w).abs()
        print(f"{name} [{b}x{n}]: fused mean {float(err.mean()) / scale:.2e} max {float(err.max()) / scale:.2e}")
        assert float(err.mean()) <= 3e-3 * scale and float(err.max()) <= 3e-2 * scale, name
    # the predicted classes agree wherever the reference's own margin is not a rounding artefact
    top2 = want[1].topk(2, dim=-1).values
    clear = (top2[..., 0] - top2[..., 1]) > 1e-2 * float(ref[f"{key}_seg_scale"])
    assert torch.equal(got[1].argmax(-1)[clear], want[1].argmax(-1)[clear])


def test_head_outputs_feed_the_pose_solver(cuda_dev, ref_modules):
    """network output -> seg argmax -> cal_frame_poses on device (demo.py:98-119 without the CNN): shapes and dtypes fit"""
    b, n = 1, 2048
    g = torch.Generator().manual_seed(1)
    eng = heads.FusedHeads(*ref_modules, device=cuda_dev)
    kp_of, seg, ctr_of = eng(torch.randn(b, 128, n, generator=g).to(cuda_dev), torch.randn(b, 128, n, generator=g).abs().to(cuda_dev))
    mask = eval_utils.seg_argmax(seg)
    assert mask.shape == (b, n) and mask.dtype == torch.int32
    pcld = torch.rand(b, n, 3, generator=g).to(cuda_dev)
    s = FramePoseSolver(b, n, 8, 22, fixtures.mesh_kps_table_ycb(), fixtures.radius_thresholds_ycb(), True, device=cuda_dev)
    poses, present, _, _ = s.solve(pcld, mask, ctr_of[:, 0].contiguous(), kp_of)
    torch.cuda.synchronize()
    assert poses.shape == (b, 22, 3, 4) and bool(torch.isfinite(poses).all())
