"""The tcgen05 shared-MLP layer kernel (csrc/mlp_tc.cu) against a float64 torch reference of the same
op on TF32-rounded operands, and the fused hot path A against features recorded from the REFERENCE
Pointnet2MSG.  Tolerances: the kernel itself 2e-5 relative (fp32 accumulation order only); end to end
the TF32 class of the reference's default cuDNN path (written at the assertion)."""
import os

import numpy as np
import pytest
import torch

from oracle import pn2
from pvn3d_b200 import mlp, testing

pytestmark = pytest.mark.gpu


def ref_dense(a, w, b, relu, pool):
    y = a.double() @ w.double().t() + b.double()
    if relu:
        y = y.clamp_min(0)
    if pool:
        y = y.view(-1, pool, y.size(-1)).max(1).values
    return y.float()


@pytest.mark.parametrize("rows,k,n,relu,pool", [
    (128, 32, 16, False, 0), (300, 64, 64, True, 0), (1000, 96, 128, True, 0), (512, 128, 196, True, 0),
    (512, 256, 384, True, 0), (640, 544, 256, True, 0), (2048, 384, 512, True, 32), (1024, 64, 32, True, 16),
    (256, 32, 16, False, 8), (131, 48, 80, True, 0),
    # many tiles per persistent CTA (ring and both TMEM accumulators wrap), odd chunk counts, 2 column blocks
    (64000, 96, 128, True, 0), (70005, 32, 32, True, 0), (40960, 64, 64, True, 16), (9000, 544, 512, True, 0),
    (38400, 160, 272, True, 32),
    # wide pooled layers: transposed accumulator (channel = TMEM lane), every pool size, ragged last tile, 1 / 2 / 4 column
    # blocks, single-chunk K
    (8192, 96, 128, True, 32), (4144, 64, 128, True, 16), (8000, 224, 256, True, 8), (50016, 224, 256, True, 32),
    (2064, 256, 512, False, 16), (4096, 32, 1024, True, 32), (160, 384, 128, True, 16)])
def test_dense_layer(cuda_dev, rows, k, n, relu, pool):
    g = torch.Generator().manual_seed(rows + k + n)
    a = torch.randn(rows, k, generator=g)
    w = torch.randn(n, k, generator=g) / np.sqrt(k)
    b = torch.randn(n, generator=g)
    layer = mlp.PackedLayer(w.to(cuda_dev), b.to(cuda_dev))
    lda = (k + 15) // 16 * 16
    ad = torch.zeros(rows, lda, device=cuda_dev)
    ad[:, :k] = a.to(cuda_dev)
    out = mlp.mlp_dense(ad, layer, relu=relu, pool=pool).cpu()
    want = ref_dense(mlp.tf32_round(a), mlp.tf32_round(w), b, relu, pool)
    assert out.shape == ((rows // pool if pool else rows), layer.n_pad)
    assert (out[:, :n] - want).abs().max() <= 2e-5 * max(1.0, want.abs().max())
    if layer.n_pad > n:
        assert out[:, n:].abs().max() == 0           # pad columns are exact zeros for the next layer


@pytest.mark.parametrize("rows,k,n,pool", [(65536, 96, 128, 32), (32768, 208, 256, 16), (8192, 384, 512, 32)])
def test_pooled_layer_into_a_column_slice_of_the_level_table(cuda_dev, rows, k, n, pool):
    """the call FusedPointnet2MSG makes for the last layer of an SA scale: pre-rounded activations (cp.async producers),
    max-pool epilogue writing columns [col0, col0 + n) of a wider table, rounded output; the other columns untouched"""
    g = torch.Generator().manual_seed(rows + n)
    a = mlp.tf32_round(torch.randn(rows, k, generator=g)).to(cuda_dev)
    w = torch.randn(n, k, generator=g) / np.sqrt(k)
    b = torch.randn(n, generator=g)
    layer = mlp.PackedLayer(w.to(cuda_dev), b.to(cuda_dev), k)
    table = torch.full((rows // pool, n + 192), 7.0, device=cuda_dev)
    mlp.mlp_dense(a, layer, pool=pool, out=table, col0=64, a_tf32=True, round_out=True)
    want = mlp.tf32_round(ref_dense(a.cpu(), mlp.tf32_round(w), b, True, pool))
    got = table.cpu()
    assert (got[:, 64:64 + n] - want).abs().max() <= 1e-3 * max(1.0, want.abs().max())     # one TF32 ulp of the rounding
    assert (got[:, 64:64 + n] - want).abs().mean() <= 2e-5 * max(1.0, want.abs().max())
    assert torch.equal(got[:, 64:64 + n], mlp.tf32_round(got[:, 64:64 + n]))
    assert (got[:, :64] == 7.0).all() and (got[:, 64 + n:] == 7.0).all()


@pytest.mark.parametrize("rows,k,n1,n2", [(50000, 64, 96, 128), (3000, 256, 384, 512), (20000, 32, 16, 32)])
def test_chained_layers_take_tf32_activations_asynchronously(cuda_dev, rows, k, n1, n2):
    """layer 1 stores TF32-rounded activations (ROUND_OUT), layer 2 copies them with cp.async (A_TF32):
    same numbers as rounding while staging."""
    g = torch.Generator().manual_seed(rows + k)
    a = torch.randn(rows, k, generator=g)
    w1 = torch.randn(n1, k, generator=g) / np.sqrt(k)
    w2 = torch.randn(n2, n1, generator=g) / np.sqrt(n1)
    b1, b2 = torch.randn(n1, generator=g), torch.randn(n2, generator=g)
    l1 = mlp.PackedLayer(w1.to(cuda_dev), b1.to(cuda_dev))
    l2 = mlp.PackedLayer(w2.to(cuda_dev), b2.to(cuda_dev), l1.n_pad)
    ad = torch.zeros(rows, (k + 15) // 16 * 16, device=cuda_dev)
    ad[:, :k] = a.to(cuda_dev)
    h = mlp.mlp_dense(ad, l1, round_out=True)
    assert torch.equal(h, mlp.tf32_round(h))
    h_plain = mlp.mlp_dense(ad, l1)
    assert torch.equal(h, mlp.tf32_round(h_plain))
    out = mlp.mlp_dense(h, l2, a_tf32=True)
    out_sync = mlp.mlp_dense(h_plain, l2)
    assert torch.equal(out, out_sync)
    want = ref_dense(h.cpu()[:, :n1], mlp.tf32_round(w2), b2, True, 0)
    assert (out.cpu()[:, :n2] - want).abs().max() <= 2e-5 * max(1.0, want.abs().max())


def test_sa_first_layer_fuses_query_and_group(cuda_dev):
    rng = np.random.default_rng(1)
    b_, n_, m_, c_, ns_ = 2, 1024, 128, 96, 16
    xyz = rng.uniform(0, 1, (b_, n_, 3)).astype(np.float32)
    fidx = pn2.furthest_point_sampling(xyz, m_)
    new = np.take_along_axis(xyz, fidx[..., None].astype(np.int64).repeat(3, -1), 1)
    feats = rng.normal(size=(b_, c_, n_)).astype(np.float32)
    grouped, idx = pn2.query_and_group(xyz, new, feats, float(np.float32(0.15)), ns_)      # [B,3+C,M,S] oracle
    w = torch.from_numpy((rng.normal(size=(64, 3 + c_)) / 10).astype(np.float32))
    bias = torch.from_numpy(rng.normal(size=64).astype(np.float32))
    X = torch.from_numpy(grouped).permute(0, 2, 3, 1).reshape(-1, 3 + c_)
    want = ref_dense(mlp.tf32_round(X), mlp.tf32_round(w), bias, True, 0)
    layer = mlp.PackedLayer(torch.cat([w[:, 3:], w[:, :3]], 1).to(cuda_dev), bias.to(cuda_dev))
    feat_pm = torch.from_numpy(feats).permute(0, 2, 1).contiguous().to(cuda_dev)
    args = (torch.from_numpy(xyz).to(cuda_dev), torch.from_numpy(new).to(cuda_dev), feat_pm.data_ptr(), c_, c_,
            torch.from_numpy(idx).to(cuda_dev), layer)
    out = mlp.mlp_sa_first(*args).cpu()
    assert (out[:, :64] - want).abs().max() <= 2e-5 * want.abs().max()
    pooled = mlp.mlp_sa_first(*args, pool=ns_).cpu()
    assert (pooled[:, :64] - want.view(-1, ns_, 64).max(1).values).abs().max() <= 2e-5 * want.abs().max()


def test_fp_first_layer_fuses_interpolation(cuda_dev):
    rng = np.random.default_rng(2)
    b_, n_u, m_k, c2, c1 = 2, 512, 128, 256, 96
    unk = rng.uniform(0, 1, (b_, n_u, 3)).astype(np.float32)
    kn = rng.uniform(0, 1, (b_, m_k, 3)).astype(np.float32)
    d2, nn = pn2.three_nn(unk, kn)
    kf = torch.from_numpy(rng.normal(size=(b_, m_k, c2)).astype(np.float32))
    sk = torch.from_numpy(rng.normal(size=(b_, n_u, c1)).astype(np.float32))
    d2_dev = torch.from_numpy(d2).to(cuda_dev)
    nw = mlp.three_nn_weights(d2_dev)
    # nn_weights_kernel in exactly rounded fp32, its order of operations: r_i = 1 / (sqrt(d_i) + 1e-8),
    # w_i = r_i / ((r_1 + r_2) + r_3) -- the same bits on every host
    r = np.float32(1) / (np.sqrt(d2) + np.float32(1e-8))
    w_exact = r / ((r[..., 0] + r[..., 1]) + r[..., 2])[..., None]
    nw_h = nw.cpu().numpy()
    assert np.array_equal(nw_h, w_exact), f"{int((nw_h != w_exact).sum())} weights differ, max {np.abs(nw_h - w_exact).max():.3e}"
    dr = 1.0 / (torch.sqrt(torch.from_numpy(d2)) + 1e-8)                        # pointnet2_modules.py:184-186
    wref = dr / dr.sum(2, keepdim=True)
    # torch's CPU kernels round the reciprocal and the sum their own way (1 ulp here): a float tolerance
    assert (torch.from_numpy(nw_h) - wref).abs().max() < 2e-7
    interp = (kf[torch.arange(b_)[:, None, None], torch.from_numpy(nn).long()] * wref[..., None]).sum(2)
    X = torch.cat([interp, sk], -1).reshape(-1, c2 + c1)
    w = torch.from_numpy((rng.normal(size=(128, c2 + c1)) / 16).astype(np.float32))
    bias = torch.from_numpy(rng.normal(size=128).astype(np.float32))
    want = ref_dense(mlp.tf32_round(X), mlp.tf32_round(w), bias, True, 0)
    layer = mlp.PackedLayer(w.to(cuda_dev), bias.to(cuda_dev))
    kfd, nnd, skd = kf.to(cuda_dev), torch.from_numpy(nn).to(cuda_dev), sk.to(cuda_dev)
    out = mlp.mlp_fp_first(kfd, nnd, nw, skd.data_ptr(), c1, c1, layer).cpu()
    # same inputs, same bits: the producers' K chunks, the weight stages and the accumulators leave nothing to chance
    again = mlp.mlp_fp_first(kfd, nnd, nw, skd.data_ptr(), c1, c1, layer).cpu()
    diff = (out != again).nonzero()
    assert diff.numel() == 0, f"second launch differs in rows {diff[:, 0].unique()[:8].tolist()}, columns {diff[:, 1].unique()[:8].tolist()}"
    # interpolation rounds to TF32 after a 3-term fp32 sum: allow one TF32 ulp of the operands
    err = (out[:, :128] - want).abs()
    bad = (err > 1e-3 * want.abs().max()).nonzero()
    assert bad.numel() == 0, (f"max error {float(err.max()):.3e} vs bound {1e-3 * float(want.abs().max()):.3e}, rows "
                              f"{bad[:, 0].unique()[:8].tolist()}, columns {bad[:, 1].unique()[:8].tolist()}")


def test_fused_pointnet2msg_matches_reference_features(cuda_dev, golden_dir):
    """End to end vs the reference Pointnet2MSG (fp32 on CPU).  TF32 operands (10-bit mantissa) through
    12 shared-MLP layers on raw 0..255 colours: mean error <= 0.3 % and max error <= 5 % of the mean
    feature magnitude -- the same class as the module graph under torch's default TF32 convolutions,
    which is measured alongside."""
    z = np.load(os.path.join(golden_dir, "pn2msg.npz"))
    model = testing.seeded_pointnet2msg(0, 1)
    eng = mlp.FusedPointnet2MSG(model, cuda_dev)
    x = torch.from_numpy(z["cld_rgb_nrm"])[None].to(cuda_dev)
    y = eng(x)
    assert y.shape == (1, 128, x.size(1))
    cols = torch.from_numpy(z["cols"]).long().to(cuda_dev)
    got = y[0][:, cols].cpu().numpy()
    scale = float(z["feat_abs_mean"])
    err = np.abs(got - z["feats"])
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = True
    try:
        with torch.no_grad():
            y_mod = model.to(cuda_dev)(x)[0][:, cols].cpu().numpy()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
    err_mod = np.abs(y_mod - z["feats"])
    print(f"fused: mean {err.mean() / scale:.2e} max {err.max() / scale:.2e} | cuDNN-TF32 modules: "
          f"mean {err_mod.mean() / scale:.2e} max {err_mod.max() / scale:.2e}")
    assert err.mean() <= 3e-3 * scale and err.max() <= 5e-2 * scale


# --------------------------------------------------------------------------------------------------
# chained SharedMLP kernel (one launch per SA scale / FP module, inter-layer tiles through L2)
# --------------------------------------------------------------------------------------------------
def _sa_case(cuda_dev, b, n, m, ns, c_feat, widths, seed):
    rng = np.random.default_rng(seed)
    xyz = torch.from_numpy(rng.uniform(0, 1, (b, n, 3)).astype(np.float32)).to(cuda_dev)
    new_xyz = xyz[:, :m].contiguous()
    idx = torch.from_numpy(rng.integers(0, n, (b, m, ns)).astype(np.int32)).to(cuda_dev)
    feat = torch.from_numpy(rng.normal(size=(b, n, max(c_feat, 4))).astype(np.float32)).to(cuda_dev)
    g = torch.Generator().manual_seed(seed)
    layers, prev, k = [], None, c_feat + 3
    for w_out in widths:
        w = torch.randn(w_out, k, generator=g) / np.sqrt(k)
        bias = torch.randn(w_out, generator=g) * 0.1
        pl = mlp.PackedLayer(w.to(cuda_dev), bias.to(cuda_dev), prev)
        prev, k = pl.n_pad, w_out
        layers.append(pl)
    return xyz, new_xyz, idx, feat, layers


@pytest.mark.parametrize("b,n,m,ns,c_feat,widths", [
    (2, 4096, 1024, 16, 6, (16, 16, 32)),       # SA1 scale 0: every layer is ONE K chunk (producer groups alternate items)
    (2, 4096, 1024, 32, 6, (32, 32, 64)),       # SA1 scale 1
    (3, 2048, 777, 16, 96, (64, 64, 128)),      # ragged row count, odd number of row tiles
    (2, 1024, 512, 32, 96, (64, 96, 128)),      # n_pad 96: K of the last layer not a multiple of its input tile
    (2, 1024, 300, 16, 256, (128, 196, 256)),   # 196 -> n_pad 208, k_pad 224
    (2, 512, 128, 32, 512, (256, 384, 512)),    # two column blocks in the last layer, few row tiles per CTA
    (1, 512, 40, 8, 64, (32, 48)),              # two layers, pool 8, fewer row tiles than CTAs
    (32, 2048, 1024, 32, 6, (32, 32, 64)),      # many row-tile pairs per CTA: ring, accumulators and slots wrap
])
def test_sa_chain_equals_per_layer_launches(cuda_dev, b, n, m, ns, c_feat, widths):
    """pvn3d_mlp_sa_chain == pvn3d_mlp_sa_first -> pvn3d_mlp_dense -> pvn3d_mlp_dense(pool), bit for bit
    (same operands, same MMA order per output element)"""
    xyz, new_xyz, idx, feat, layers = _sa_case(cuda_dev, b, n, m, ns, c_feat, widths, seed=b + m + ns)
    fptr, ldf = feat.data_ptr(), feat.size(-1)
    h = mlp.mlp_sa_first(xyz, new_xyz, fptr, ldf, c_feat, idx, layers[0], round_out=True)
    for mid in layers[1:-1]:
        h = mlp.mlp_dense(h, mid, round_out=True, a_tf32=True)
    want = mlp.mlp_dense(h, layers[-1], pool=ns, a_tf32=True)
    chain = mlp.LayerChain(layers)
    got = mlp.mlp_sa_chain(xyz, new_xyz, fptr, ldf, c_feat, idx, chain, pool=ns)
    assert got.shape == want.shape == (b * m, layers[-1].n_pad)
    assert torch.equal(got, want), float((got - want).abs().max())
    # un-pooled rows (EPI_STORE as the final epilogue)
    want_rows = mlp.mlp_dense(h, layers[-1], a_tf32=True)
    got_rows = mlp.mlp_sa_chain(xyz, new_xyz, fptr, ldf, c_feat, idx, chain, pool=0)
    assert torch.equal(got_rows, want_rows)


@pytest.mark.parametrize("b,n_u,m_k,c2,c1,widths", [(2, 512, 128, 1024, 512, (512, 512)), (2, 4096, 1024, 256, 6, (128, 128)),
                                                   (3, 1000, 333, 512, 96, (256, 256)), (1, 100, 20, 64, 0, (32, 16))])
def test_fp_chain_equals_per_layer_launches(cuda_dev, b, n_u, m_k, c2, c1, widths):
    rng = np.random.default_rng(n_u)
    unk = rng.uniform(0, 1, (b, n_u, 3)).astype(np.float32)
    kn = rng.uniform(0, 1, (b, m_k, 3)).astype(np.float32)
    d2, nn = pn2.three_nn(unk, kn)
    kf = torch.from_numpy(rng.normal(size=(b, m_k, c2)).astype(np.float32)).to(cuda_dev)
    sk = torch.from_numpy(rng.normal(size=(b, n_u, max(c1, 4))).astype(np.float32)).to(cuda_dev)
    nw = mlp.three_nn_weights(torch.from_numpy(d2).to(cuda_dev))
    nn_d = torch.from_numpy(nn).to(cuda_dev)
    g = torch.Generator().manual_seed(c2)
    layers, prev, k = [], None, c2 + c1
    for w_out in widths:
        pl = mlp.PackedLayer((torch.randn(w_out, k, generator=g) / np.sqrt(k)).to(cuda_dev),
                             (torch.randn(w_out, generator=g) * 0.1).to(cuda_dev), prev)
        prev, k = pl.n_pad, w_out
        layers.append(pl)
    h = mlp.mlp_fp_first(kf, nn_d, nw, sk.data_ptr(), sk.size(-1), c1, layers[0], round_out=True)
    want = mlp.mlp_dense(h, layers[1], a_tf32=True)
    got = mlp.mlp_fp_chain(kf, nn_d, nw, sk.data_ptr(), sk.size(-1), c1, mlp.LayerChain(layers))
    assert torch.equal(got, want), float((got - want).abs().max())


def test_chain_engine_equals_layer_engine_and_is_deterministic(cuda_dev):
    """whole hot path A: chained engine == per-layer engine bit for bit, and 200 repetitions of the
    chained forward give identical bits (stress for the warp-specialised mbarrier pipeline)."""
    from pvn3d_b200 import synth

    model = testing.seeded_pointnet2msg(0, 1)
    frames = synth.make_batch("ycb", 2, n_points=12288, config_id=13)
    x = torch.from_numpy(np.stack([f.cld_rgb_nrm for f in frames])).to(cuda_dev)
    layer_eng = mlp.FusedPointnet2MSG(model, cuda_dev, chain=False)
    layer_eng.factor = False          # the chained kernel runs the unfactored first layer: same operands, same bits
    y_layer = layer_eng(x)
    eng = mlp.FusedPointnet2MSG(model, cuda_dev, chain=True)
    y0 = eng(x).clone()
    assert torch.equal(y0, y_layer), float((y0 - y_layer).abs().max())
    for i in range(200):
        assert torch.equal(eng(x), y0), f"run {i} differs"


def test_rounded_level_tables_do_not_change_the_features(cuda_dev):
    """SA1-3 level tables stored TF32-rounded (so that the next level gathers them with cp.async) vs stored in
    fp32 and rounded while staging: identical features, bit for bit"""
    from pvn3d_b200 import synth

    model = testing.seeded_pointnet2msg(0, 1)
    frames = synth.make_batch("linemod", 2, n_points=12288, config_id=14)
    x = torch.from_numpy(np.stack([f.cld_rgb_nrm for f in frames])).to(cuda_dev)
    eng = mlp.FusedPointnet2MSG(model, cuda_dev, chain=False)
    assert eng.round_tables
    y_async = eng(x).clone()
    eng.round_tables = False
    y_sync = eng(x)
    assert torch.equal(y_async, y_sync), float((y_async - y_sync).abs().max())


def test_factored_first_layer_matches_unfactored_engine(cuda_dev, golden_dir):
    """first SA layer evaluated once per point (U_j - V_i, coordinate term split hi + lo) vs once per grouped row with
    the difference x_j - c_i rounded to TF32: same function, different rounding points -> TF32-class agreement; and the
    factored engine is at least as close to the reference's fp32 features as the unfactored one"""
    from pvn3d_b200 import synth

    z = np.load(os.path.join(golden_dir, "pn2msg_big.npz"))
    model = testing.seeded_pointnet2msg(0, 1)
    x = torch.from_numpy(z["cld_rgb_nrm"])[None].to(cuda_dev)
    eng = mlp.FusedPointnet2MSG(model, cuda_dev, chain=False)
    assert eng.factor
    y_fact = eng(x).clone()
    eng.factor = False
    y_plain = eng(x)
    scale = float(y_plain.abs().mean())
    d = (y_fact - y_plain).abs()
    assert float(d.mean()) <= 3e-3 * scale and float(d.max()) <= 5e-2 * scale, (float(d.mean()) / scale, float(d.max()) / scale)
    cols = torch.from_numpy(z["cols"]).long().to(cuda_dev)
    ref = torch.from_numpy(z["feats"]).to(cuda_dev)
    e_fact = float((y_fact[0][:, cols] - ref).abs().mean())
    e_plain = float((y_plain[0][:, cols] - ref).abs().mean())
    print(f"mean |err| vs reference fp32 features: factored {e_fact / scale:.2e}, unfactored {e_plain / scale:.2e}")
    assert e_fact <= 1.2 * e_plain + 1e-6


@pytest.mark.parametrize("b,n,m,ns,c_feat,n1,n2", [(2, 1024, 300, 16, 96, 64, 96), (1, 512, 100, 32, 6, 32, 32),
                                                    (3, 700, 129, 8, 256, 128, 208), (2, 2048, 512, 32, 512, 256, 384)])
def test_factored_sa_first_layer_kernels(cuda_dev, b, n, m, ns, c_feat, n1, n2):
    """pvn3d_sa_factor_table + pvn3d_mlp_dense (U) + pvn3d_sa_centre_term (V): U[idx] - V == W1.[f | x - c] + b1 to fp32
    accuracy (the hi/lo coordinate split), and pvn3d_mlp_sa_fact == relu(tf32(relu(U[idx] - V)) . W2 + b2)"""
    rng = np.random.default_rng(b + n + ns)
    xyz = torch.from_numpy(rng.uniform(-0.5, 1.2, (b, n, 3)).astype(np.float32)).to(cuda_dev)
    sel = torch.from_numpy(np.stack([rng.choice(n, m, replace=False) for _ in range(b)])).to(cuda_dev)
    new_xyz = torch.gather(xyz, 1, sel[..., None].expand(-1, -1, 3)).contiguous()
    idx = torch.from_numpy(rng.integers(0, n, (b, m, ns)).astype(np.int32)).to(cuda_dev)
    feat = torch.from_numpy(rng.normal(size=(b, n, c_feat)).astype(np.float32)).to(cuda_dev)
    g = torch.Generator().manual_seed(n + m)
    w1 = (torch.randn(n1, c_feat + 3, generator=g) / np.sqrt(c_feat + 3)).to(cuda_dev)     # producer order [f | xyz]
    b1 = (torch.randn(n1, generator=g) * 0.1).to(cuda_dev)
    first = mlp.PackedLayer(torch.cat([w1, w1[:, c_feat:]], 1), torch.zeros_like(b1))         # [W_f | W_x | W_x]
    wx = mlp.tf32_round(w1[:, c_feat:].contiguous())
    wxp = torch.zeros((first.n_pad, 3), device=cuda_dev); wxp[:n1] = wx
    b1p = torch.zeros((first.n_pad,), device=cuda_dev); b1p[:n1] = b1
    table = mlp.sa_factor_table(xyz, feat.data_ptr(), c_feat, c_feat, first.k_pad)
    u = mlp.mlp_dense(table, first, relu=False, a_tf32=True)
    v = mlp.sa_centre_term(new_xyz, wxp, b1p)
    bi = torch.arange(b, device=cuda_dev)[:, None, None]
    got1 = (u.view(b, n, -1)[bi, idx.long()] - v.view(b, m, 1, -1))[..., :n1]                  # pre-ReLU first layer
    f64 = mlp.tf32_round(feat).double()[bi, idx.long()]
    dx = xyz.double()[bi, idx.long()] - new_xyz.double()[:, :, None, :]
    want1 = f64 @ mlp.tf32_round(w1[:, :c_feat]).double().t() + dx @ wx.double().t() + b1.double()
    assert float((got1.double() - want1).abs().max()) <= 2e-5 * max(1.0, float(want1.abs().max()))
    # second layer on relu(U[idx] - V)
    w2 = (torch.randn(n2, n1, generator=g) / np.sqrt(n1)).to(cuda_dev)
    b2 = (torch.randn(n2, generator=g) * 0.1).to(cuda_dev)
    l2 = mlp.PackedLayer(w2, b2, first.n_pad)
    got2 = mlp.mlp_sa_fact(u, v, idx, n, l2)
    a2 = mlp.tf32_round(torch.relu(u.view(b, n, -1)[bi, idx.long()] - v.view(b, m, 1, -1)).reshape(-1, first.n_pad)[:, :n1])
    want2 = ref_dense(a2.cpu(), mlp.tf32_round(w2).cpu(), b2.cpu(), True, 0)
    assert (got2.cpu()[:, :n2] - want2).abs().max() <= 2e-5 * max(1.0, float(want2.abs().max()))
    got2p = mlp.mlp_sa_fact(u, v, idx, n, l2, pool=ns)
    assert torch.equal(got2p, got2.view(b * m, ns, -1).max(1).values)


def test_factored_fp_first_layer_kernel(cuda_dev):
    rng = np.random.default_rng(9)
    b_, n_u, m_k, n1, n2 = 2, 1000, 333, 128, 128
    nn = torch.from_numpy(rng.integers(0, m_k, (b_, n_u, 3)).astype(np.int32)).to(cuda_dev)
    w = rng.uniform(0.05, 1, (b_, n_u, 3)).astype(np.float32)
    w = torch.from_numpy(w / w.sum(-1, keepdims=True)).to(cuda_dev)
    p = torch.from_numpy(rng.normal(size=(b_ * m_k, n1)).astype(np.float32)).to(cuda_dev)
    s_ = torch.from_numpy(rng.normal(size=(b_ * n_u, n1)).astype(np.float32)).to(cuda_dev)
    g = torch.Generator().manual_seed(4)
    l2 = mlp.PackedLayer((torch.randn(n2, n1, generator=g) / np.sqrt(n1)).to(cuda_dev), (torch.randn(n2, generator=g) * 0.1).to(cuda_dev), n1)
    got = mlp.mlp_fp_fact(p, s_, nn, w, m_k, l2)
    bi = torch.arange(b_, device=cuda_dev)[:, None, None]
    pg = p.view(b_, m_k, n1)[bi, nn.long()]                                                     # [b, n, 3, n1]
    a = torch.relu((pg[:, :, 2] * w[..., 2:3]).add(pg[:, :, 0] * w[..., 0:1] + pg[:, :, 1] * w[..., 1:2]) + s_.view(b_, n_u, n1))
    want = ref_dense(mlp.tf32_round(a.reshape(-1, n1)).cpu(), l2.w.cpu()[:n2, :n1], l2.bias.cpu()[:n2], True, 0)
    # interpolation order differs in the last ulp before TF32 rounding: one TF32 ulp of the operands
    assert (got.cpu()[:, :n2] - want).abs().max() <= 1e-3 * max(1.0, float(want.abs().max()))


@pytest.mark.parametrize("b_,n_u,m_k,n2", [(2, 1024, 333, 128), (3, 4128, 512, 256), (1, 96, 40, 128)])
def test_factored_fp_layer_channel_major_output(cuda_dev, b_, n_u, m_k, n2):
    """PVN3D_MLP_OUT_CN: the same numbers as the row-major call, laid out [b, n_pad, n_unknown] (what
    Pointnet2MSG.forward returns, pvn3d.py:154) -- bit for bit, ragged last tile and frames that end inside a tile"""
    rng = np.random.default_rng(b_ + n_u)
    n1 = 128
    nn = torch.from_numpy(rng.integers(0, m_k, (b_, n_u, 3)).astype(np.int32)).to(cuda_dev)
    w = rng.uniform(0.05, 1, (b_, n_u, 3)).astype(np.float32)
    w = torch.from_numpy(w / w.sum(-1, keepdims=True)).to(cuda_dev)
    p = torch.from_numpy(rng.normal(size=(b_ * m_k, n1)).astype(np.float32)).to(cuda_dev)
    s_ = torch.from_numpy(rng.normal(size=(b_ * n_u, n1)).astype(np.float32)).to(cuda_dev)
    g = torch.Generator().manual_seed(n2)
    l2 = mlp.PackedLayer((torch.randn(n2, n1, generator=g) / np.sqrt(n1)).to(cuda_dev), (torch.randn(n2, generator=g) * 0.1).to(cuda_dev), n1)
    rows = mlp.mlp_fp_fact(p, s_, nn, w, m_k, l2)
    cn = mlp.mlp_fp_fact(p, s_, nn, w, m_k, l2, out_cn=True)
    assert cn.shape == (b_, n2, n_u)
    assert torch.equal(cn, rows.view(b_, n_u, n2).transpose(1, 2))
    # unsupported shapes are refused, not mis-stored
    if n_u % 32 == 0:
        with pytest.raises(RuntimeError):
            mlp.mlp_fp_fact(p[:, :n1], s_, nn[:, :n_u - 1].contiguous(), w[:, :n_u - 1].contiguous(), m_k, l2, out_cn=True)

