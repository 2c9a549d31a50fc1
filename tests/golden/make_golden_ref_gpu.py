"""Record what the GPU parity tests compare against from the UNMODIFIED reference, on a B200.

    python tests/golden/make_golden_ref_gpu.py OUT_DIR     # writes OUT_DIR/pn2_ref_digests.json, ref_modules.npz

Needs what oracle/build_ref_ext.sh builds from a checkout of the reference: its op library
(oracle/_ref/_ext.so) and its Python (oracle/_ref/py).  The two files are committed under tests/golden/;
the tests then run without the reference:

  pn2_ref_digests.json   SHA-256 (tests/helpers.py:digest) of every reference op output tests/test_pn2_gpu.py
                         compares with, on the same seeded inputs: the sm_100a ops must match them bit for bit.
  ref_modules.npz        the reference Pointnet2MSG on the reference `_ext` (TF32 off): digest and a seeded sample
                         of its features, digest of its state_dict; gradients of a reference PointnetSAModuleMSG;
                         the reference cal_frame_poses / cal_frame_poses_lm on CUDA tensors; seeded samples of the
                         reference DenseFusion + head stacks (fp32) loaded with pvn3d_b200.heads.reference_layout_modules
                         weights -- for tests/test_reference_dropin_gpu.py and tests/test_heads_gpu.py.

Every recorded op output is also checked against this package's kernels here, so a recording that the tests
could not reproduce fails loudly instead of being committed.
"""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from helpers import (HEADS_CASES, SA_LEVELS, digest, level_clouds, load_ref_ext, load_reference_python,  # noqa: E402
                     sa_autograd_inputs, sample, state_dict_digest)
from oracle import pn2  # noqa: E402
from pvn3d_b200 import _ext as our_ext  # noqa: E402
from pvn3d_b200 import eval_utils, heads, synth, testing  # noqa: E402

dev = torch.device("cuda:0")


def t(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def record_ops(ref_ext):
    """the reference op calls of tests/test_pn2_gpu.py, inputs generated exactly as there"""
    out = {}

    def put(key, ref_out, ours):
        r, o = ref_out.cpu().numpy(), ours.cpu().numpy()
        assert r.dtype == o.dtype and np.array_equal(r, o), f"{key}: this package differs from the reference"
        out[key] = digest(r)

    _, levels = level_clouds(batch=2, seed0=500)
    for li, (_, m, _, _) in enumerate(SA_LEVELS):
        x = t(levels[li])
        put(f"fps/level{li}", ref_ext.furthest_point_sampling(x, m), our_ext.furthest_point_sampling(x, m))
    rng = np.random.default_rng(3)
    for n, m in [(512, 64), (1024, 300), (700, 128), (128, 32), (37, 20), (3000, 257), (12288, 200), (5000, 130),
                 (6100, 90)]:
        base = rng.uniform(0.2, 1.0, size=(2, max(4, n // 3), 3)).astype(np.float32)
        xyz = np.concatenate([base] * 4, 1)[:, :n].copy()
        xyz[:, 5] = [0.01, 0.01, 0.01]
        put(f"fps_ties/{n}_{m}", ref_ext.furthest_point_sampling(t(xyz), m), our_ext.furthest_point_sampling(t(xyz), m))
    for li, (_, _, radii, nss) in enumerate(SA_LEVELS):
        xyz, new = t(levels[li]), t(levels[li + 1])
        for r, ns in zip(radii, nss):
            put(f"ball_query/level{li}_{r}_{ns}", ref_ext.ball_query(new, xyz, r, ns), our_ext.ball_query(new, xyz, r, ns))
    rng = np.random.default_rng(6)
    for li, c in [(1, 96), (3, 512)]:
        xyz, new = levels[li], levels[li + 1]
        feats = rng.normal(size=(2, c, xyz.shape[1])).astype(np.float32)
        idx = t(pn2.ball_query(new, xyz, SA_LEVELS[li][2][1], 32))
        put(f"group_points/level{li}_{c}", ref_ext.group_points(t(feats), idx), our_ext.group_points(t(feats), idx))
    rng = np.random.default_rng(9)
    for lu, c in [(0, 256), (1, 512), (2, 512), (3, 1024)]:
        unknown, known = t(levels[lu]), t(levels[lu + 1])
        rd2, ridx = ref_ext.three_nn(unknown, known)
        d2, idx = our_ext.three_nn(unknown, known)
        put(f"three_nn_d2/level{lu}", rd2, d2)
        put(f"three_nn_idx/level{lu}", ridx, idx)
        feats = rng.normal(size=(2, c, known.shape[1])).astype(np.float32)
        w = rng.uniform(0, 1, size=tuple(d2.shape)).astype(np.float32)
        w /= w.sum(-1, keepdims=True)
        put(f"three_interpolate/level{lu}", ref_ext.three_interpolate(t(feats), idx, t(w)),
            our_ext.three_interpolate(t(feats), idx, t(w)))
    for m, n in [(600, 2000), (2048, 5000), (4096, 9000), (512, 1024)]:
        rng = np.random.default_rng(m + n)
        known = rng.integers(-20, 20, size=(2, m, 3)).astype(np.float32) * 0.01
        known[:, m // 2:m // 2 + m // 4] = known[:, :m // 4]
        known[1, :, 0] = 0.05
        unk = rng.integers(-25, 25, size=(2, n, 3)).astype(np.float32) * 0.01
        unk[:, :m // 8] = known[:, :m // 8]
        rd2, ridx = ref_ext.three_nn(t(unk), t(known))
        d2, idx = our_ext.three_nn(t(unk), t(known))
        put(f"three_nn_d2/slab_{m}_{n}", rd2, d2)
        put(f"three_nn_idx/slab_{m}_{n}", ridx, idx)
    return out


def no_tf32(fn):
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            return fn()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev


def record_pointnet2msg(ref, ref_ext, out):
    torch.manual_seed(0)
    model = ref.pvn3d.Pointnet2MSG(input_channels=6)
    testing.randomize_bn_(model, 1)
    model = model.to(dev).eval()
    frames = synth.make_batch("ycb", 2, n_points=12288, config_id=11)
    x = torch.from_numpy(np.stack([f.cld_rgb_nrm for f in frames])).to(dev)
    y_ours = no_tf32(lambda: model(x))
    ref.pn2_utils._ext = ref_ext
    try:
        y_ref = no_tf32(lambda: model(x))
    finally:
        ref.pn2_utils._ext = our_ext
    assert torch.equal(y_ours, y_ref), "reference Pointnet2MSG: drop-in _ext differs from the reference _ext"
    mirror = testing.seeded_pointnet2msg(0, 1).to(dev)
    assert state_dict_digest(mirror) == state_dict_digest(model), "mirror weights differ from the reference's"
    y_mirror = no_tf32(lambda: mirror(x))
    print("pn2msg: mirror module bit-identical to the reference module:", bool(torch.equal(y_mirror, y_ref)),
          "max |diff|", float((y_mirror - y_ref).abs().max()))
    y = y_ref.cpu().numpy()
    out.update(pn2msg_digest=digest(y), pn2msg_sample=sample(y, 4096), pn2msg_abs_mean=np.float64(np.abs(y).mean()),
               pn2msg_state_dict=state_dict_digest(model), cudnn_version=np.int64(torch.backends.cudnn.version()))


def record_sa_autograd(ref, ref_ext, out):
    from lib.pointnet2_utils import pointnet2_modules as ref_mod

    from pvn3d_b200 import pointnet2

    torch.manual_seed(1)
    sa = ref_mod.PointnetSAModuleMSG(npoint=64, radii=[0.1, 0.2], nsamples=[8, 16],
                                     mlps=[[6, 16, 32], [6, 16, 32]]).to(dev).eval()
    torch.manual_seed(1)
    mirror = pointnet2.PointnetSAModuleMSG(npoint=64, radii=[0.1, 0.2], nsamples=[8, 16], mlps=[[6, 16, 32], [6, 16, 32]])
    assert state_dict_digest(mirror) == state_dict_digest(sa), "mirror SA weights differ from the reference's"
    xyz_np, feat_np = sa_autograd_inputs()
    ref.pn2_utils._ext = ref_ext
    try:
        feat = t(feat_np).requires_grad_(True)
        prev = torch.backends.cudnn.allow_tf32
        torch.backends.cudnn.allow_tf32 = False
        try:
            _, o = sa(t(xyz_np), feat)
            o.square().sum().backward()
        finally:
            torch.backends.cudnn.allow_tf32 = prev
    finally:
        ref.pn2_utils._ext = our_ext
    out.update(sa_grad=feat.grad.cpu().numpy(), sa_state_dict=state_dict_digest(sa))


def record_frame_poses(ref, out):
    for shape in ("ycb", "linemod"):
        f = synth.make_frame(shape, n_points=4096, seed=77, lm_obj_id=1 if shape == "linemod" else None)
        args = [t(a) for a in (f.pcld, f.labels, f.ctr_of, f.kp_of)]
        if shape == "ycb":
            ids, poses = ref.eval_utils.cal_frame_poses(*args, True, 22, True)
            ours_ids, ours = eval_utils.cal_frame_poses(*args, True, 22, True)
            assert np.array_equal(ours_ids, ids)
            out["frame_poses_ycb_ids"] = np.asarray(ids, np.int64)
        else:
            poses = ref.eval_utils.cal_frame_poses_lm(*args, True, 2, False, 1)
            ours = eval_utils.cal_frame_poses_lm(*args, True, 2, False, 1)
        poses = np.stack([np.asarray(p, np.float64) for p in poses])
        print(f"cal_frame_poses {shape}: max |ours - reference| {float(np.abs(np.stack(ours) - poses).max()):.2e}")
        out[f"frame_poses_{shape}"] = poses


def record_heads(ref, out):
    import lib.utils.etw_pytorch_utils as pt_utils
    from torch import nn

    torch.manual_seed(3)
    mods = heads.reference_layout_modules(n_classes=22, n_kps=8)
    for i, m in enumerate(mods):
        testing.randomize_bn_(m, 10 + i)
    n_cls, n_kps = 22, 8
    # the reference classes, built as PVN3D.__init__ builds them (pvn3d.py:157-182,245-267), with the same weights
    rmods = [ref.pvn3d.DenseFusion(2048)]
    for width, n_out in ((128, n_cls), (256, n_kps * 3), (128, 3)):
        rmods.append(pt_utils.Seq(1792).conv1d(1024, bn=True, activation=nn.ReLU()).conv1d(512, bn=True, activation=nn.ReLU())
                     .conv1d(width, bn=True, activation=nn.ReLU()).conv1d(n_out, activation=None))
    for r, m in zip(rmods, mods):
        r.load_state_dict(m.state_dict(), strict=True)
    fusion, seg, kpof, ctrof = [m.to(dev).eval() for m in rmods]
    eng = heads.FusedHeads(*[m.to(dev).eval() for m in mods], device=dev)
    for b, n in HEADS_CASES:
        g = torch.Generator().manual_seed(n)
        rgb_emb = torch.randn(b, 128, n, generator=g).to(dev)
        cld_emb = torch.randn(b, 128, n, generator=g).abs().to(dev)
        fusion.ap1 = nn.AvgPool1d(n)

        def fwd():
            f = fusion(rgb_emb, cld_emb)
            return (kpof(f).view(b, n_kps, 3, n).permute(0, 1, 3, 2).contiguous(),      # pvn3d.py:297-306
                    seg(f).transpose(1, 2).contiguous(), ctrof(f).view(b, 1, 3, n).permute(0, 1, 3, 2).contiguous())

        want = [w.cpu().numpy() for w in no_tf32(fwd)]
        got = [x.cpu().numpy() for x in eng(rgb_emb, cld_emb)]
        for name, w, x in zip(("kp_of", "seg", "ctr_of"), want, got):
            scale = np.abs(w).mean()
            print(f"heads {name} [{b}x{n}]: fused mean {np.abs(x - w).mean() / scale:.2e} max {np.abs(x - w).max() / scale:.2e}")
            out[f"heads_{b}x{n}_{name}_scale"] = np.float64(scale)
        out[f"heads_{b}x{n}_kp_of"] = sample(want[0], 2048)
        out[f"heads_{b}x{n}_ctr_of"] = sample(want[2], 1024)
        out[f"heads_{b}x{n}_seg_rows"] = sample(want[1].reshape(b * n, n_cls), 256, rows=True)


def main():
    out_dir = sys.argv[1]
    ref_ext, ref = load_ref_ext(), load_reference_python()
    assert ref_ext is not None and ref is not None, "oracle/_ref/_ext.so or oracle/_ref/py missing"
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "pn2_ref_digests.json"), "w") as f:
        json.dump(record_ops(ref_ext), f, indent=1, sort_keys=True)
    out = {}
    record_pointnet2msg(ref, ref_ext, out)
    record_sa_autograd(ref, ref_ext, out)
    record_frame_poses(ref, out)
    record_heads(ref, out)
    np.savez_compressed(os.path.join(out_dir, "ref_modules.npz"), **out)
    print("wrote", out_dir, {k: getattr(v, "shape", None) for k, v in out.items()})


if __name__ == "__main__":
    main()
