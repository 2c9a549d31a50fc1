"""Parity of the sm_100a PointNet++ ops (through the C ABI) with the oracle and with the unmodified
reference op library on the same seeded inputs: the reference's outputs are stored as SHA-256 digests
(tests/golden/pn2_ref_digests.json, recorded by tests/golden/make_golden_ref_gpu.py).

Bar (BASELINE.json north_star): indices bit-exact; gathered / interpolated values bit-exact too
(pure copies and a 3-term fma chain contracted like the reference SASS).
"""
import json
import os

import numpy as np
import pytest
import torch

from helpers import SA_LEVELS, digest, level_clouds, t
from oracle import pn2
from pvn3d_b200 import _ext

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def clouds():
    return level_clouds(batch=2, seed0=500)


@pytest.fixture(scope="module")
def ref(golden_dir):
    """digests of the reference op outputs, by call"""
    with open(os.path.join(golden_dir, "pn2_ref_digests.json")) as f:
        return json.load(f)


def test_fps_all_levels_bit_exact(cuda_dev, clouds, ref):
    _, levels = clouds
    for li, (n, m, _, _) in enumerate(SA_LEVELS):
        xyz = levels[li]
        got = _ext.furthest_point_sampling(t(xyz, cuda_dev), m).cpu().numpy()
        want = pn2.furthest_point_sampling(xyz, m)
        assert np.array_equal(got, want), f"FPS level {li} differs from oracle"
        assert digest(got) == ref[f"fps/level{li}"], f"FPS differs from REFERENCE at level {li}"


def test_fps_ties_duplicates_and_origin_points(cuda_dev, ref):
    rng = np.random.default_rng(3)
    for n, m in [(512, 64), (1024, 300), (700, 128), (128, 32), (37, 20), (3000, 257), (12288, 200), (5000, 130),
                 (6100, 90)]:          # 4097..12288 points: the thread-block-cluster kernel (3 or 6 points per thread)
        base = rng.uniform(0.2, 1.0, size=(2, max(4, n // 3), 3)).astype(np.float32)
        xyz = np.concatenate([base] * 4, 1)[:, :n].copy()          # wrap-padded duplicates => exact ties
        xyz[:, 5] = [0.01, 0.01, 0.01]                              # |p|^2 <= 1e-3: never selected
        got = _ext.furthest_point_sampling(t(xyz, cuda_dev), m).cpu().numpy()
        assert np.array_equal(got, pn2.furthest_point_sampling(xyz, m)), (n, m)
        assert digest(got) == ref[f"fps_ties/{n}_{m}"], (n, m)
    # all points coincide except the start: the bit-reversed-tid tie-break of the reference tree
    xyz = np.zeros((1, 512, 3), np.float32); xyz[:] = [1, 0, 2]; xyz[0, 0] = [0, 0, 2]
    assert _ext.furthest_point_sampling(t(xyz, cuda_dev), 2).cpu().numpy().tolist() == [[0, 256]]


def test_fps_large_cloud_generic_path(cuda_dev):
    rng = np.random.default_rng(4)
    xyz = rng.uniform(0.3, 1.2, size=(1, 20000, 3)).astype(np.float32)
    got = _ext.furthest_point_sampling(t(xyz, cuda_dev), 64).cpu().numpy()
    assert np.array_equal(got, pn2.furthest_point_sampling(xyz, 64))


def test_ball_query_all_scales_bit_exact(cuda_dev, clouds, ref):
    _, levels = clouds
    for li, (n, m, radii, nss) in enumerate(SA_LEVELS):
        xyz, new = levels[li], levels[li + 1]
        for r, ns in zip(radii, nss):
            got = _ext.ball_query(t(new, cuda_dev), t(xyz, cuda_dev), r, ns).cpu().numpy()
            want = pn2.ball_query(new, xyz, float(np.float32(r)), ns)
            assert np.array_equal(got, want), (li, r, ns)
            assert digest(got) == ref[f"ball_query/level{li}_{r}_{ns}"], f"ball_query differs from REFERENCE {(li, r, ns)}"


def test_ball_query_empty_and_ragged(cuda_dev):
    rng = np.random.default_rng(5)
    xyz = rng.uniform(0, 1, size=(3, 1000, 3)).astype(np.float32)
    new = rng.uniform(0, 1, size=(3, 77, 3)).astype(np.float32)
    new[:, 0] = 9.0                                                  # empty ball -> zeros
    for r, ns in [(0.05, 16), (0.3, 32), (0.02, 5), (2.0, 64), (0.1, 1)]:
        got = _ext.ball_query(t(new, cuda_dev), t(xyz, cuda_dev), r, ns).cpu().numpy()
        assert np.array_equal(got, pn2.ball_query(new, xyz, float(np.float32(r)), ns)), (r, ns)
        assert (got[:, 0] == 0).all()


def test_group_and_gather_bit_exact(cuda_dev, clouds, ref):
    _, levels = clouds
    rng = np.random.default_rng(6)
    for li, c in [(1, 96), (3, 512)]:
        xyz, new = levels[li], levels[li + 1]
        n, m = xyz.shape[1], new.shape[1]
        feats = rng.normal(size=(2, c, n)).astype(np.float32)
        idx = pn2.ball_query(new, xyz, SA_LEVELS[li][2][1], 32)
        got = _ext.group_points(t(feats, cuda_dev), t(idx, cuda_dev)).cpu().numpy()
        assert np.array_equal(got, pn2.group_points(feats, idx))
        assert digest(got) == ref[f"group_points/level{li}_{c}"], (li, c)
        fidx = pn2.furthest_point_sampling(xyz, m)
        g2 = _ext.gather_points(t(feats, cuda_dev), t(fidx, cuda_dev)).cpu().numpy()
        assert np.array_equal(g2, pn2.gather_points(feats, fidx))
        # point-major centre gather == gather_operation(xyz^T, idx)^T (pointnet2_modules.py:47-53)
        nx = _ext.gather_xyz(t(xyz, cuda_dev), t(fidx, cuda_dev)).cpu().numpy()
        want = pn2.gather_points(np.ascontiguousarray(xyz.transpose(0, 2, 1)), fidx).transpose(0, 2, 1)
        assert np.array_equal(nx, want)


def test_query_and_group_fused_bit_exact(cuda_dev, clouds):
    _, levels = clouds
    rng = np.random.default_rng(7)
    for li, c in [(0, 6), (1, 96), (2, 256), (3, 512), (3, 0), (2, 40)]:
        xyz, new = levels[li], levels[li + 1]
        n = xyz.shape[1]
        feats = rng.normal(size=(2, c, n)).astype(np.float32) if c else None
        for r, ns in zip(SA_LEVELS[li][2], SA_LEVELS[li][3]):
            want, widx = pn2.query_and_group(xyz, new, feats, float(np.float32(r)), ns)
            feat_pm = _ext.transpose_cn_to_nc(t(feats, cuda_dev)) if c else None
            got, gidx = _ext.query_and_group(t(xyz, cuda_dev), t(new, cuda_dev), feat_pm, r, ns)
            assert np.array_equal(gidx.cpu().numpy(), widx), (li, c, r, ns)
            assert np.array_equal(got.cpu().numpy(), want), (li, c, r, ns)


def test_query_and_group_odd_sizes(cuda_dev):
    rng = np.random.default_rng(8)
    xyz = rng.uniform(0, 1, size=(2, 2500, 3)).astype(np.float32)
    new = xyz[:, ::7][:, :301].copy()
    feats = rng.normal(size=(2, 45, 2500)).astype(np.float32)
    for r, ns in [(0.08, 16), (0.15, 24), (0.05, 7), (0.3, 64), (0.3, 200)]:
        want, widx = pn2.query_and_group(xyz, new, feats, float(np.float32(r)), ns)
        got, gidx = _ext.query_and_group(t(xyz, cuda_dev), t(new, cuda_dev),
                                         _ext.transpose_cn_to_nc(t(feats, cuda_dev)), r, ns)
        assert np.array_equal(gidx.cpu().numpy(), widx), (r, ns)
        assert np.array_equal(got.cpu().numpy(), want), (r, ns)


def test_three_nn_and_interpolate_bit_exact(cuda_dev, clouds, ref):
    _, levels = clouds
    rng = np.random.default_rng(9)
    for lu, c in [(0, 256), (1, 512), (2, 512), (3, 1024)]:
        unknown, known = levels[lu], levels[lu + 1]
        d2, idx = _ext.three_nn(t(unknown, cuda_dev), t(known, cuda_dev))
        wd2, widx = pn2.three_nn(unknown, known)
        assert np.array_equal(idx.cpu().numpy(), widx) and np.array_equal(d2.cpu().numpy(), wd2), lu
        assert digest(idx.cpu().numpy()) == ref[f"three_nn_idx/level{lu}"], lu
        assert digest(d2.cpu().numpy()) == ref[f"three_nn_d2/level{lu}"], lu
        feats = rng.normal(size=(2, c, known.shape[1])).astype(np.float32)
        w = rng.uniform(0, 1, size=wd2.shape).astype(np.float32)
        w /= w.sum(-1, keepdims=True)
        got = _ext.three_interpolate(t(feats, cuda_dev), idx, t(w, cuda_dev)).cpu().numpy()
        assert np.array_equal(got, pn2.three_interpolate(feats, widx, w)), lu
        assert digest(got) == ref[f"three_interpolate/level{lu}"], lu


def test_three_nn_ties_and_small_m(cuda_dev):
    known = np.array([[[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 0, 0]]], np.float32)
    unk = np.array([[[0.9, 0, 0], [0, 0.2, 0]]], np.float32)
    d2, idx = _ext.three_nn(t(unk, cuda_dev), t(known, cuda_dev))
    wd2, widx = pn2.three_nn(unk, known)
    assert np.array_equal(idx.cpu().numpy(), widx) and idx[0, 0].tolist() == [1, 3, 0]
    d2, idx = _ext.three_nn(t(unk, cuda_dev), t(known[:, :2], cuda_dev))
    assert torch.isinf(d2[0, 0, 2]) and int(idx[0, 0, 2]) == 0


@pytest.mark.parametrize("m,n", [(600, 2000), (2048, 5000), (4096, 9000), (512, 1024)])
def test_three_nn_sorted_slab_ties_and_padding(cuda_dev, ref, m, n):
    """the x-sorted walk (m >= 512) against the oracle's index-order cascade on clouds built to tie: duplicated known
    points (equal distances -> the LOWER index must win, in all three slots), points sharing x, queries ON known
    points, m not a power of two (padding of the sort), coordinates on a lattice (many equal squared distances)"""
    rng = np.random.default_rng(m + n)
    known = rng.integers(-20, 20, size=(2, m, 3)).astype(np.float32) * 0.01          # lattice -> exact ties everywhere
    known[:, m // 2:m // 2 + m // 4] = known[:, :m // 4]                              # exact duplicates, higher indices
    known[1, :, 0] = 0.05                                                             # one frame: all known share x
    unk = rng.integers(-25, 25, size=(2, n, 3)).astype(np.float32) * 0.01
    unk[:, :m // 8] = known[:, :m // 8]                                               # queries on known points: d2 = 0 ties
    d2, idx = _ext.three_nn(t(unk, cuda_dev), t(known, cuda_dev))
    wd2, widx = pn2.three_nn(unk, known)
    assert np.array_equal(idx.cpu().numpy(), widx), int((idx.cpu().numpy() != widx).sum())
    assert np.array_equal(d2.cpu().numpy(), wd2)
    assert digest(idx.cpu().numpy()) == ref[f"three_nn_idx/slab_{m}_{n}"]
    assert digest(d2.cpu().numpy()) == ref[f"three_nn_d2/slab_{m}_{n}"]


def test_three_nn_interpolate_fused(cuda_dev, clouds):
    """fused FP front end == three_nn -> sqrt -> 1/(d+1e-8) -> normalise -> three_interpolate
    (pointnet2_modules.py:183-190) composed from the separate ops + torch."""
    _, levels = clouds
    rng = np.random.default_rng(10)
    for lu, c in [(0, 256), (2, 512)]:
        unknown, known = t(levels[lu], cuda_dev), t(levels[lu + 1], cuda_dev)
        feats = t(rng.normal(size=(2, c, levels[lu + 1].shape[1])).astype(np.float32), cuda_dev)
        d2, idx = _ext.three_nn(unknown, known)
        dist_recip = 1.0 / (torch.sqrt(d2) + 1e-8)
        weight = dist_recip / torch.sum(dist_recip, dim=2, keepdim=True)
        want = _ext.three_interpolate(feats, idx, weight)                        # [B,C,n]
        got, gd2, gidx = _ext.three_nn_interpolate(unknown, known, _ext.transpose_cn_to_nc(feats), want_nn=True)
        assert torch.equal(gidx, idx) and torch.equal(gd2, d2)
        got_cn = got.transpose(1, 2)
        # weights: same IEEE ops; bit-exact unless torch's 3-term sum orders differently
        assert torch.allclose(got_cn, want, rtol=1e-6, atol=1e-6)


def test_grad_ops_are_adjoints(cuda_dev):
    rng = np.random.default_rng(11)
    b, c, n, m, s = 2, 5, 200, 40, 8
    idx = t(rng.integers(0, n, size=(b, m, s)).astype(np.int32), cuda_dev)
    go = t(rng.normal(size=(b, c, m, s)).astype(np.float32), cuda_dev)
    got = _ext.group_points_grad(go, idx, n).cpu().numpy()
    assert np.allclose(got, pn2.group_points_grad(go.cpu().numpy(), idx.cpu().numpy(), n), atol=1e-5)
    idx2 = t(rng.integers(0, n, size=(b, m)).astype(np.int32), cuda_dev)
    go2 = t(rng.normal(size=(b, c, m)).astype(np.float32), cuda_dev)
    got = _ext.gather_points_grad(go2, idx2, n).cpu().numpy()
    assert np.allclose(got, pn2.gather_points_grad(go2.cpu().numpy(), idx2.cpu().numpy(), n), atol=1e-5)
    idx3 = t(rng.integers(0, m, size=(b, n, 3)).astype(np.int32), cuda_dev)
    w = t(rng.uniform(size=(b, n, 3)).astype(np.float32), cuda_dev)
    go3 = t(rng.normal(size=(b, c, n)).astype(np.float32), cuda_dev)
    got = _ext.three_interpolate_grad(go3, idx3, w, m).cpu().numpy()
    want = pn2.three_interpolate_grad(go3.cpu().numpy(), idx3.cpu().numpy(), w.cpu().numpy(), m)
    assert np.allclose(got, want, atol=1e-4)


def test_contract_errors(cuda_dev):
    x = torch.zeros(1, 8, 3)
    with pytest.raises(RuntimeError, match="CPU not supported"):
        _ext.furthest_point_sampling(x, 2)
    xc = torch.zeros(1, 3, 8, device=cuda_dev).transpose(1, 2)
    with pytest.raises(RuntimeError, match="must be a contiguous tensor"):
        _ext.furthest_point_sampling(xc, 2)
    with pytest.raises(RuntimeError, match="must be an int tensor"):
        _ext.gather_points(torch.zeros(1, 3, 8, device=cuda_dev), torch.zeros(1, 2, device=cuda_dev))
    with pytest.raises(RuntimeError, match="must be a float tensor"):
        _ext.ball_query(torch.zeros(1, 2, 3, device=cuda_dev).double(), torch.zeros(1, 8, 3, device=cuda_dev), 0.1, 4)


def test_query_and_group2_both_radii_in_one_launch(cuda_dev, clouds):
    """The two scales of every MSG level from ONE launch == two oracle QueryAndGroup calls, bit for bit;
    idx-only form (ball_query2) == ball_query twice."""
    _, levels = clouds
    rng = np.random.default_rng(12)
    for li, c in [(0, 6), (1, 96), (2, 256), (3, 512), (1, 40)]:
        xyz, new = levels[li], levels[li + 1]
        n = xyz.shape[1]
        feats = rng.normal(size=(2, c, n)).astype(np.float32)
        radii, nss = SA_LEVELS[li][2], SA_LEVELS[li][3]
        feat_pm = _ext.transpose_cn_to_nc(t(feats, cuda_dev))
        outs, idxs = _ext.query_and_group2(t(xyz, cuda_dev), t(new, cuda_dev), feat_pm, radii, nss)
        i0, i1 = _ext.ball_query2(t(new, cuda_dev), t(xyz, cuda_dev), radii, nss)
        for s in range(2):
            want, widx = pn2.query_and_group(xyz, new, feats, float(np.float32(radii[s])), nss[s])
            assert np.array_equal(idxs[s].cpu().numpy(), widx), (li, c, s)
            assert np.array_equal(outs[s].cpu().numpy(), want), (li, c, s)
            assert np.array_equal((i0, i1)[s].cpu().numpy(), widx), (li, c, s)
