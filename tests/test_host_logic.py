"""Host-side logic that needs no GPU: fixtures, synthetic data, compat shims, op argument contracts,
and the N>1 frame sharding / gather over a world_size-2 gloo group."""
import os
import sys

import numpy as np
import pytest
import torch

from pvn3d_b200 import _ext, compat, dist as pdist, fixtures, pointnet2, synth, testing


def test_fixtures_shapes_and_thresholds():
    t = fixtures.mesh_kps_table_ycb()
    assert t.shape == (22, 9, 3) and np.all(t[0] == 0)
    assert np.allclose(t[1, 8], fixtures.get_ctr(1))          # centre appended LAST (pvn3d_eval_utils.py:99-103)
    thr = fixtures.radius_thresholds_ycb()
    r = fixtures.ycb_r_lst()
    assert thr.dtype == np.float32 and thr[5] == np.float32(r[4] * 0.8)
    assert fixtures.lm_obj_dict()["ape"] == 1 and fixtures.mesh_kps_table_lm(1).shape == (2, 9, 3)


def test_synthetic_frame_contract():
    f = synth.make_frame("ycb", n_points=4096, seed=3)
    assert f.cld_rgb_nrm.shape == (4096, 9) and f.cld_rgb_nrm.dtype == np.float32
    assert f.kp_of.shape == (8, 4096, 3) and f.ctr_of.shape == (1, 4096, 3) and f.labels.dtype == np.int64
    assert np.array_equal(f.cld_rgb_nrm[:, :3], f.pcld)
    assert np.linalg.norm(f.pcld, axis=1).min() > np.sqrt(1e-3)     # no point FPS would skip
    assert set(np.unique(f.labels)) == {0, *f.cls_ids.tolist()}
    # votes of an instance cluster on its true centre
    c = int(f.cls_ids[0]); sel = f.labels == c
    votes = f.pcld[sel] - f.ctr_of[0][sel]
    assert np.linalg.norm(np.median(votes, 0) - (f.RTs[0][:, :3] @ fixtures.get_ctr(c) + f.RTs[0][:, 3])) < 2e-3
    g = synth.make_frame("ycb", n_points=4096, seed=3)
    assert np.array_equal(f.kp_of, g.kp_of), "seeded generator must be deterministic"
    lm = synth.make_frame("linemod", n_points=12288, seed=2000)
    assert 0.2 < (lm.labels == 1).mean() < 0.32


def test_ext_contract_on_cpu_tensors():
    x = torch.zeros(1, 8, 3)
    with pytest.raises(RuntimeError, match="CPU not supported"):
        _ext.ball_query(x, x, 0.1, 4)
    with pytest.raises(RuntimeError, match="must be a contiguous tensor"):
        _ext.three_nn(torch.zeros(1, 3, 8).transpose(1, 2), x)
    with pytest.raises(RuntimeError, match="must be an int tensor"):
        _ext.group_points(torch.zeros(1, 3, 8), torch.zeros(1, 2, 2))
    names = ["gather_points", "gather_points_grad", "furthest_point_sampling", "three_nn", "three_interpolate",
             "three_interpolate_grad", "ball_query", "group_points", "group_points_grad"]   # bindings.cpp:6-19
    assert all(callable(getattr(_ext, n)) for n in names)


def test_compat_install_registers_ext_module():
    compat.install()
    assert sys.modules["lib.pointnet2_utils._ext"] is _ext
    import yaml
    assert yaml.load("a: 1") == {"a": 1}                     # common.py:133 calls yaml.load without Loader
    assert "torch._six" in sys.modules and "neupeak.utils.webcv2" in sys.modules


def test_pointnet2msg_mirror_layout():
    m = testing.seeded_pointnet2msg(0, 1)
    sd = m.state_dict()
    assert "SA_modules.0.mlps.0.layer0.conv.weight" in sd
    assert "FP_modules.3.mlp.layer1.normlayer.bn.running_var" in sd
    assert sd["SA_modules.0.mlps.0.layer0.conv.weight"].shape == (16, 9, 1, 1)     # +3 xyz channels
    assert sd["SA_modules.3.mlps.1.layer2.conv.weight"].shape == (512, 384, 1, 1)
    assert sd["FP_modules.0.mlp.layer0.conv.weight"].shape == (128, 262, 1, 1)
    assert sum(p.numel() for p in m.parameters()) == 3012272 or sum(p.numel() for p in m.parameters()) > 2.9e6
    # the caller's lists are not mutated (the reference does, pointnet2_modules.py:108-110)
    spec = [[6, 16]]
    pointnet2.PointnetSAModuleMSG(npoint=4, radii=[0.1], nsamples=[2], mlps=spec)
    assert spec == [[6, 16]]


def test_shard_frames_partitions():
    for n, w in [(128, 8), (16, 4), (5, 2), (3, 4)]:
        shards = [pdist.shard_frames(n, r, w) for r in range(w)]
        assert sorted(sum(shards, [])) == list(range(n))
        assert max(len(s) for s in shards) - min(len(s) for s in shards) <= 1


def _gloo_worker(rank, world, port, n_frames, q):
    os.environ.update(RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1",
                      MASTER_PORT=str(port))
    import torch.distributed as dist
    r, _, w = pdist.init_from_env(backend="gloo")
    ids = pdist.shard_frames(n_frames, r, w)
    local = torch.stack([torch.full((2, 3, 4), float(i)) for i in ids]) if ids else torch.zeros(0, 2, 3, 4)
    full = pdist.gather_frame_results(local, n_frames, r, w)
    ok = all(bool((full[i] == float(i)).all()) for i in range(n_frames))
    mx = pdist.max_over_ranks(float(rank + 1), "cpu")
    q.put((rank, ok, mx))
    dist.destroy_process_group()


@pytest.mark.parametrize("n_frames", [5, 8])
def test_frame_shard_and_gather_gloo_world2(n_frames):
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29600 + n_frames
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, n_frames, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert all(ok for _, ok, _ in res) and all(mx == 2.0 for _, _, mx in res)


def test_unmodified_reference_binds_to_the_drop_in(tmp_path):
    """`from lib.pointnet2_utils import _ext` (reference pointnet2_utils.py:19) resolves to this package's
    module, and the post-processing names are rebound -- on a stand-in tree with the reference's module paths and
    the import lines compat.install() relies on, in a subprocess to keep sys.modules clean.  The stand-in does not
    import what the real lib/ imports, so the shims for it (torch._six, yaml.load's Loader, neupeak / plyfile / pcl)
    are exercised here only through test_compat_install_registers_ext_module; importing the real reference Python
    and running its Pointnet2MSG, SA autograd and cal_frame_poses on the drop-in is done by
    tests/golden/make_golden_ref_gpu.py when the reference outputs are recorded.  The "CPU not supported" check runs
    through this package's mirror Pointnet2MSG, which calls the same `_ext` entry points."""
    import subprocess
    tree = {
        "lib/pointnet2_utils/pointnet2_utils.py": "from lib.pointnet2_utils import _ext\n",
        "lib/utils/meanshift_pytorch.py": "class MeanShiftTorch:\n    pass\n",
        "lib/utils/pvn3d_eval_utils.py": ("from lib.utils.meanshift_pytorch import MeanShiftTorch\n"
                                          "def cal_frame_poses(*args):\n    pass\n"
                                          "def cal_frame_poses_lm(*args):\n    pass\n"),
    }
    for rel, text in tree.items():
        (tmp_path / rel).parent.mkdir(parents=True, exist_ok=True)
        (tmp_path / rel).write_text(text)
    code = (
        "import sys; sys.path.insert(0, %r)\n"
        "from pvn3d_b200 import compat, _ext, eval_utils, meanshift\n"
        "compat.install(%r, patch_post=True)\n"
        "from lib.pointnet2_utils import pointnet2_utils as pu\n"
        "from lib.utils import pvn3d_eval_utils as ev, meanshift_pytorch as ms\n"
        "from pvn3d_b200.pointnet2 import Pointnet2MSG\n"
        "import torch\n"
        "assert pu._ext is _ext and ms.MeanShiftTorch is meanshift.MeanShiftTorch\n"
        "assert ev.MeanShiftTorch is meanshift.MeanShiftTorch\n"
        "assert ev.cal_frame_poses is eval_utils.cal_frame_poses and ev.cal_frame_poses_lm is eval_utils.cal_frame_poses_lm\n"
        "m = Pointnet2MSG(input_channels=6)\n"
        "try:\n    m(torch.zeros(1, 4096, 9)); raise SystemExit(3)\n"
        "except RuntimeError as e:\n    assert 'CPU not supported' in str(e)\n"
        "print('ok')\n") % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), str(tmp_path))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-2000:]


def test_mlp_packing_folds_batchnorm_and_rounds_to_tf32():
    """Host half of the tensor-core MLP path (pvn3d_b200/mlp.py): Conv2d(1x1)+BatchNorm2d(eval) folded into one
    matrix + bias reproduces the module (pytorch_utils.py:25-50), weights are TF32 values (10-bit mantissa, ties
    away = cvt.rna) zero-padded to the kernel's k_pad % 32 / n_pad % 16 grid, and the first SA layer's xyz
    columns are moved behind the descriptor columns (the order pvn3d_mlp_sa_first's producer emits)."""
    from pvn3d_b200 import mlp
    x = torch.tensor([1.0, 1.0 + 2 ** -11, 1.0 + 2 ** -10, -3.0000002, 65504.5, 0.0, 1e-30])
    r = mlp.tf32_round(x)
    assert torch.equal(r.view(torch.int32) & 0x1FFF, torch.zeros_like(r, dtype=torch.int32))      # low 13 bits clear
    assert r[1] == 1.0 + 2 ** -10 and r[0] == 1.0 and r[2] == x[2]                                  # tie rounds away
    assert ((r - x).abs() <= x.abs() * 2 ** -11).all()

    model = testing.seeded_pointnet2msg(0, 1).eval()
    layer = model.SA_modules[1].mlps[0][0]                     # Conv2d(99 -> 64, no bias) + BN + ReLU
    w, b = mlp.fold_conv_bn(layer)
    g = torch.Generator().manual_seed(5)
    a = torch.randn(2, w.shape[1], 7, 3, generator=g)
    with torch.no_grad():
        want = layer(a)                                        # ReLU(BN(conv(a)))
    got = torch.relu(torch.einsum("nk,bkms->bnms", w, a) + b[None, :, None, None])
    assert (got - want).abs().max() <= 1e-5 * max(1.0, want.abs().max())

    pk = mlp.PackedLayer(w, b)
    assert pk.k_pad % 32 == 0 and pk.n_pad % 16 == 0 and pk.k_pad >= w.shape[1] and pk.n_pad >= w.shape[0]
    assert torch.equal(pk.w[: w.shape[0], : w.shape[1]], mlp.tf32_round(w))
    assert pk.w[w.shape[0]:].abs().sum() == 0 and pk.w[:, w.shape[1]:].abs().sum() == 0 and pk.bias[w.shape[0]:].abs().sum() == 0
    nxt = mlp.PackedLayer(torch.randn(40, w.shape[0], generator=g), torch.zeros(40), pk.n_pad)
    assert nxt.k_pad >= pk.n_pad                               # consumes the padded activations of `pk`

    eng_cols = torch.cat([w[:, 3:], w[:, :3]], dim=1)          # [xyz | feat] -> [feat | xyz]
    assert torch.equal(eng_cols[:, -3:], w[:, :3]) and torch.equal(eng_cols[:, :-3], w[:, 3:])
    assert mlp.MLP_RELU == 1 and mlp.MLP_ROUND_OUT == 2 and mlp.MLP_A_TF32 == 4          # include/pvn3d_b200.h
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "pvn3d_b200.h")).read()
    for name, val in (("PVN3D_MLP_RELU", 1), ("PVN3D_MLP_ROUND_OUT", 2), ("PVN3D_MLP_A_TF32", 4)):
        assert f"#define {name} {val}" in hdr
