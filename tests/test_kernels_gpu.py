"""GPU parity tests: every CUDA kernel called through the C ABI (tensorflow_yolo2_b200.ops ->
ctypes -> libyolo2_b200.so) against the CPU oracle on the same seeded inputs."""
import os

import numpy as np
import pytest
import torch

from oracle import yolo2_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def ops():
    from tensorflow_yolo2_b200 import ops as _ops
    from tensorflow_yolo2_b200 import _lib
    _lib.load()
    return _ops


def cu(a, dtype=None):
    t = torch.as_tensor(np.ascontiguousarray(a)).cuda()
    return t.to(dtype) if dtype is not None else t


# ---------------------------------------------------------------------------------- a10
def test_preprocess_u8_bit_exact(ops, golden_dir):
    import cv2
    im = cv2.resize(cv2.imread(os.path.join(golden_dir, 'testImg1.jpg')), (416, 416))
    want = O.preprocess_u8(im)
    got = ops.preprocess_u8(cu(im[None]), bf16c8=False).cpu().numpy()[0]
    np.testing.assert_array_equal(got, want)                 # integer/byte work: bit-exact
    got8 = ops.preprocess_u8(cu(im[None]), bf16c8=True).float().cpu().numpy()[0]
    want8 = torch.tensor(want).to(torch.bfloat16).float().numpy()
    np.testing.assert_array_equal(got8[..., :3], want8)
    assert np.all(got8[..., 3:] == 0)


# ---------------------------------------------------------------------------------- a10+a1+a2+a3 first layer fused
@pytest.mark.parametrize('N,H,W', [(2, 32, 16, ), (3, 96, 96), (1, 64, 160), (2, 416, 416)])
def test_conv1_u8_pool_vs_oracle(ops, N, H, W):
    """uint8 image -> preprocessing -> conv 3x3 3->32 (+bias, BN incl. NEGATIVE gammas) -> leaky -> 2x2 pool, one
    kernel, against the oracle's conv_bn_layer + max_pool on bf16-rounded operands (the kernel folds the BN scale into
    the bf16 weights, so the oracle's weights are rounded after the same folding)."""
    rs = np.random.RandomState(7 + H)
    img = rs.randint(0, 256, (N, H, W, 3)).astype(np.uint8)
    w = (rs.randn(3, 3, 3, 32) * 0.3).astype(np.float32)
    b = (rs.randn(32) * 0.1).astype(np.float32)
    gamma = (rs.uniform(0.5, 1.5, 32) * np.where(rs.rand(32) < 0.3, -1, 1)).astype(np.float32)
    beta, mm = (rs.randn(32) * 0.2).astype(np.float32), (rs.randn(32) * 0.2).astype(np.float32)
    mv = rs.uniform(0.5, 2.0, 32).astype(np.float32)
    scale, shift = ops.bn_fold(cu(gamma), cu(beta), cu(mm), cu(mv), cu(b))
    wp = ops.pack_weights_conv1_u8(cu(w), scale)
    got = ops.conv1_u8_pool(cu(img), wp, shift).float().cpu().numpy()
    assert got.shape == (N, H // 2, W // 2, 32)
    # oracle: same folding, operands rounded to bf16 at the same points, float64 accumulation
    x = O.bf16_round(torch.tensor(O.preprocess_u8(img))).double()
    wf = O.bf16_round(torch.tensor(w) * scale.cpu().reshape(1, 1, 1, 32)).double()
    h = O.conv2d_same(x, wf, torch.float64) + shift.cpu().double()
    want = O.max_pool_2x2(torch.maximum(O.ALPHA * h, h)).numpy()
    np.testing.assert_allclose(got, want, rtol=1e-2, atol=1e-2)        # output is bf16 (8 mantissa bits)
    assert np.linalg.norm(got - want) / np.linalg.norm(want) < 3e-3


# ---------------------------------------------------------------------------------- a1 (fp32 path)
@pytest.mark.parametrize('N,H,W,Cin,Cout,k', [(2, 13, 13, 64, 48, 3), (1, 16, 20, 3, 32, 3), (2, 7, 7, 128, 30, 1),
                                              (1, 26, 26, 32, 125, 3)])
def test_conv_f32_vs_oracle(ops, N, H, W, Cin, Cout, k):
    rs = np.random.RandomState(1)
    x = rs.randn(N, H, W, Cin).astype(np.float32)
    w = (rs.randn(k, k, Cin, Cout) * 0.1).astype(np.float32)
    b = rs.randn(Cout).astype(np.float32)
    want = (O.conv2d_same(torch.tensor(x), torch.tensor(w), torch.float64) + torch.tensor(b).double()).numpy()
    got = ops.conv_fwd_f32(cu(x), cu(w), cu(b)).cpu().numpy()
    np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-5 * np.abs(want).max())   # fp32 path: 1e-5


# ---------------------------------------------------------------------------------- a1 halo-patch path, CTA pairs
@pytest.mark.parametrize('N,H,W,Cin,Cout,pool', [(3, 72, 72, 32, 64, True),      # kw-merged stages, odd tile count (135)
                                                 (2, 64, 80, 64, 128, False),    # one chunk, 128-wide, un-pooled
                                                 (1, 104, 104, 128, 64, False),  # two chunks; 91 tiles: last pair half empty
                                                 (2, 66, 70, 64, 128, True)])    # ragged borders inside the 8x16 tiles
def test_conv_halo_pair_vs_single_cta_and_oracle(ops, monkeypatch, N, H, W, Cin, Cout, pool):
    """3x3 layers on maps >= 64x64 run as CTA pairs on cta_group::2 MMAs (each CTA its own 8x16-pixel tile and half of the
    resident filters): bit-identical to the single-CTA kernel (same products, same fp32 accumulation order per output) and
    within bf16 tolerance of the oracle, with fused scale/shift (negative scales too), leaky and 2x2 pool."""
    rs = np.random.RandomState(H + Cin)
    x = rs.randn(N, H, W, Cin).astype(np.float32)
    w = (rs.randn(3, 3, Cin, Cout) * 0.05).astype(np.float32)
    b = rs.randn(Cout).astype(np.float32)
    sc = (rs.uniform(0.5, 1.5, Cout) * np.where(rs.rand(Cout) < 0.3, -1, 1)).astype(np.float32)
    xb = cu(x, torch.bfloat16)
    wp = ops.pack_weights_bf16(cu(w))
    kw = dict(scale=cu(sc), shift=cu(b), leaky=True, pool=pool)
    monkeypatch.setenv('Y2_CONV_NO_IS', '1')         # (the 64-filter shapes would otherwise take the input-stationary kernel)
    ops.reload_env()
    got = ops.conv_fwd_bf16(xb, wp, 3, Cin, Cout, **kw)
    monkeypatch.setenv('Y2_CONV_NO_CTA2', '1')
    ops.reload_env()                     # the launchers cache the Y2_* switches
    ref = ops.conv_fwd_bf16(xb, wp, 3, Cin, Cout, **kw)
    torch.cuda.synchronize()
    assert torch.equal(got, ref)
    want = O.conv2d_same(O.bf16_round(torch.tensor(x)).double(), O.bf16_round(torch.tensor(w)).double(), torch.float64)
    want = want * torch.tensor(sc).double() + torch.tensor(b).double()
    want = torch.maximum(O.ALPHA * want, want)
    if pool:
        want = want.reshape(N, H // 2, 2, W // 2, 2, Cout).amax(dim=(2, 4))
    want = want.numpy()
    g = got.float().cpu().numpy()
    np.testing.assert_allclose(g, want, rtol=1e-2, atol=1e-2 * np.abs(want).max())
    assert np.linalg.norm(g - want) / np.linalg.norm(want) < 4e-3


@pytest.mark.parametrize('N,H,W,Cin,Cout,ld', [(2, 64, 80, 64, 128, 128),     # layer 3 / 5 shape of the training forward pass
                                               (2, 70, 68, 64, 128, 160),     # tiles clipped at the right / bottom edge, padded rows
                                               (1, 104, 104, 32, 64, 64),     # layer 2: 64-byte operand rows, 64 columns
                                               (2, 96, 64, 3, 32, 32)])       # first layer (8-channel padded input)
def test_conv_f32_rows_tma_store_equals_direct_stores(ops, monkeypatch, N, H, W, Cin, Cout, ld):
    """Training forward: conv + bias as float32 rows [N*H*W, ld].  On the halo-patch path the rows leave through swizzled smem
    and TMA box stores of 16 columns; Y2_CONV_NO_TMA_STORE_F32=1 selects the per-lane 16-byte stores: same bits, and both
    within bf16-operand tolerance of the oracle."""
    rs = np.random.RandomState(H + Cout)
    x = rs.randn(N, H, W, Cin).astype(np.float32)
    w = (rs.randn(3, 3, Cin, Cout) * 0.05).astype(np.float32)
    b = rs.randn(Cout).astype(np.float32)
    if Cin == 3:
        xb = torch.zeros((N, H, W, 8), dtype=torch.bfloat16, device='cuda')
        xb[..., :3] = cu(x, torch.bfloat16)
    else:
        xb = cu(x, torch.bfloat16)
    wp = ops.pack_weights_bf16(cu(w))
    monkeypatch.setenv('Y2_CONV_NO_IS', '1')
    ops.reload_env()
    outs = []
    for direct in (False, True):
        if direct:
            monkeypatch.setenv('Y2_CONV_NO_TMA_STORE_F32', '1')
            ops.reload_env()
        y = torch.full((N * H * W, ld), -7.0, dtype=torch.float32, device='cuda')
        ops.conv_fwd_bf16(xb, wp, 3, Cin, Cout, scale=None, shift=cu(b), leaky=False, pool=False, out_f32=True, ldy=ld, out=y)
        torch.cuda.synchronize()
        outs.append(y)
    assert torch.equal(outs[0][:, :Cout], outs[1][:, :Cout])
    want = O.conv2d_same(O.bf16_round(torch.tensor(x)).double(), O.bf16_round(torch.tensor(w)).double(), torch.float64) \
        + torch.tensor(b).double()
    g = outs[0][:, :Cout].cpu().numpy().reshape(N, H, W, Cout)
    assert np.linalg.norm(g - want.numpy()) / np.linalg.norm(want.numpy()) < 1e-5


@pytest.mark.parametrize('N,H,W,Cin,pool,out_f32,x3', [(3, 72, 72, 32, True, False, False),     # layer 2 shape: 64-byte rows, pooled epilogue
                                                         (1, 104, 104, 128, False, False, False),  # layer 4 shape: two chunks, odd tile count
                                                         (2, 70, 66, 64, False, False, False),     # ragged: W % 14 != 0, H % 8 != 0
                                                         (2, 64, 64, 64, True, True, False),       # float32 rows + pool (generic epilogue)
                                                         (2, 80, 72, 128, False, True, False),     # training forward / float32 rows
                                                         (2, 72, 72, 32, True, False, True),       # bf16x3: three K blocks, split output
                                                         (1, 72, 80, 128, False, False, True),     # bf16x3 at 128 channels: streamed filters
                                                         (1, 64, 98, 64, False, False, False)])    # exactly 7 tiles wide
def test_conv_input_stationary_vs_halo_kernel_and_oracle(ops, monkeypatch, N, H, W, Cin, pool, out_f32, x3):
    """conv_is_kernel (3x3, 64 filters, maps >= 64x64: the three horizontal taps as column blocks of one N = 192 MMA, the
    horizontal shift applied to the accumulators with warp shuffles) against the halo-patch kernel it replaces
    (Y2_CONV_NO_IS=1: same products, different fp32 summation order) and the float64 oracle on the same operands."""
    Cout = 64
    rs = np.random.RandomState(H + W + Cin)
    x = rs.randn(N, H, W, Cin).astype(np.float32)
    w = (rs.randn(3, 3, Cin, Cout) * 0.05).astype(np.float32)
    b = rs.randn(Cout).astype(np.float32)
    sc = (rs.uniform(0.5, 1.5, Cout) * np.where(rs.rand(Cout) < 0.3, -1, 1)).astype(np.float32)
    if x3:
        t = torch.tensor(x)
        hi = t.to(torch.bfloat16)
        xb = torch.cat([hi, (t - hi.float()).to(torch.bfloat16)], dim=-1).contiguous().cuda()
        wp = ops.pack_weights_bf16_split(cu(w))
        xo = (hi.float() + (t - hi.float()).to(torch.bfloat16).float()).double()
        wt = torch.tensor(w)
        wh = wt.to(torch.bfloat16).float()
        wo = (wh + (wt - wh).to(torch.bfloat16).float()).double()
    else:
        xb, wp = cu(x, torch.bfloat16), ops.pack_weights_bf16(cu(w))
        xo, wo = O.bf16_round(torch.tensor(x)).double(), O.bf16_round(torch.tensor(w)).double()
    kw = dict(scale=cu(sc), shift=cu(b), leaky=True, pool=pool, out_f32=out_f32, split_in=x3, split_out=x3 and not out_f32)
    monkeypatch.setenv('Y2_CONV_FORCE_IS', '1')        # (by default the kernel is only chosen for K >= 96 channels per tap)
    ops.reload_env()
    got = ops.conv_fwd_bf16(xb, wp, 3, Cin, Cout, **kw)
    monkeypatch.delenv('Y2_CONV_FORCE_IS')
    monkeypatch.setenv('Y2_CONV_NO_IS', '1')
    ops.reload_env()
    ref = ops.conv_fwd_bf16(xb, wp, 3, Cin, Cout, **kw)
    torch.cuda.synchronize()
    want = O.conv2d_same(xo, wo, torch.float64) * torch.tensor(sc).double() + torch.tensor(b).double()
    want = torch.maximum(O.ALPHA * want, want)
    if pool:
        want = O.max_pool_2x2(want)
    want = want.numpy()
    Ho, Wo = (H // 2, W // 2) if pool else (H, W)

    def f32(t):
        if out_f32:
            return t.view(N, Ho, Wo, Cout).cpu().numpy()
        if x3:
            return (t[..., :Cout].float() + t[..., Cout:].float()).cpu().numpy()
        return t.float().cpu().numpy()
    g, r = f32(got), f32(ref)
    tol = 3e-5 if (x3 or out_f32) else 4e-3
    e_g, e_r = np.linalg.norm(g - want) / np.linalg.norm(want), np.linalg.norm(r - want) / np.linalg.norm(want)
    print('input-stationary rel_l2 %.3g (halo kernel %.3g)' % (e_g, e_r))
    assert e_g < tol and e_r < tol
    # same products, only the fp32 summation order differs: the two kernels agree far inside the output rounding
    np.testing.assert_allclose(g, r, rtol=2e-2 if not (x3 or out_f32) else 1e-4, atol=(1e-2 if not (x3 or out_f32) else 1e-4) * np.abs(want).max())


@pytest.mark.parametrize('N,S,Cin,Cout,k,pool,out_f32', [(5, 26, 256, 512, 3, True, False),     # tiled boxes + fused pool, 256-wide, streamed B
                                                         (7, 13, 1024, 512, 1, False, False),   # 1x1, 10 tiles of 128 rows -> 5 pairs, 2 N tiles
                                                         (3, 13, 512, 256, 1, False, False),    # 1x1 with a resident half bank, 4 tiles
                                                         (3, 13, 1024, 125, 1, False, True)])   # detection layer: 125 -> 128 columns, float32 rows
def test_conv_generic_pair_vs_single_cta(ops, monkeypatch, N, S, Cin, Cout, k, pool, out_f32):
    """im2col / tiled-box layers as CTA pairs == the single-CTA kernel, bit for bit (odd tile counts, ragged last tile)."""
    rs = np.random.RandomState(S + Cout + k)
    xb = cu(rs.randn(N, S, S, Cin).astype(np.float32), torch.bfloat16)
    wp = ops.pack_weights_bf16(cu((rs.randn(k, k, Cin, Cout) * 0.05).astype(np.float32)))
    sc = cu((rs.uniform(0.5, 1.5, Cout) * np.where(rs.rand(Cout) < 0.3, -1, 1)).astype(np.float32))
    ld = (Cout + 31) // 32 * 32
    kw = dict(scale=None if out_f32 else sc, shift=cu(rs.randn(Cout).astype(np.float32)), leaky=not out_f32, pool=pool,
              out_f32=out_f32, ldy=ld if out_f32 else None)
    monkeypatch.setenv('Y2_CONV_NO_STREAMK', '1')
    ops.reload_env()                     # the launchers cache the Y2_* switches
    got = ops.conv_fwd_bf16(xb, wp, k, Cin, Cout, **kw)
    monkeypatch.setenv('Y2_CONV_NO_CTA2', '1')
    ops.reload_env()                     # the launchers cache the Y2_* switches
    ref = ops.conv_fwd_bf16(xb, wp, k, Cin, Cout, **kw)
    torch.cuda.synchronize()
    g, r = got.reshape(-1, got.shape[-1])[:, :Cout], ref.reshape(-1, ref.shape[-1])[:, :Cout]
    assert torch.equal(g, r)
    assert float(g.float().abs().sum()) > 0


# ---------------------------------------------------------------------------------- a1 stream-K 256x256 path
@pytest.mark.parametrize('N,S,Cin,Cout,k,out_f32', [(16, 13, 512, 512, 3, True), (9, 13, 1024, 256, 3, False),
                                                    (6, 19, 1024, 256, 3, True), (8, 26, 256, 512, 3, False),
                                                    # more tiles than CTA pairs: tiles are split between neighbouring pairs
                                                    # and the partial accumulators travel through the workspace
                                                    (64, 13, 512, 256, 3, False), (48, 13, 512, 512, 3, True),
                                                    # four N tiles of 256 filters, tiles split between pairs
                                                    (64, 13, 256, 1024, 3, False), (60, 13, 256, 1024, 3, True)])
def test_conv_streamk_vs_generic_and_oracle(ops, monkeypatch, N, S, Cin, Cout, k, out_f32):
    """Deep 3x3 layer on a small map: the 256x256 stream-K kernel (a tile's K range split between two CTAs, the partial
    travels through the workspace and the owner runs the fused epilogue) against the generic tcgen05 kernel and the
    oracle, for the float32 pre-BN output and for the fused scale/shift/leaky bf16 output; bit-identical across runs."""
    rs = np.random.RandomState(S + Cout)
    x = rs.randn(N, S, S, Cin).astype(np.float32)
    w = (rs.randn(k, k, Cin, Cout) * 0.05).astype(np.float32)
    b = rs.randn(Cout).astype(np.float32)
    sc = None if out_f32 else (rs.uniform(0.5, 1.5, Cout) * np.where(rs.rand(Cout) < 0.3, -1, 1)).astype(np.float32)
    xb = cu(x, torch.bfloat16)
    wp = ops.pack_weights_bf16(cu(w))
    kw = dict(scale=None if sc is None else cu(sc), shift=cu(b), leaky=not out_f32, out_f32=out_f32)
    monkeypatch.setenv('Y2_CONV_NO_STREAMK', '1')
    ops.reload_env()                     # the launchers cache the Y2_* switches
    ref = ops.conv_fwd_bf16(xb, wp, k, Cin, Cout, **kw).float().cpu().numpy().reshape(-1, Cout)
    monkeypatch.delenv('Y2_CONV_NO_STREAMK')
    monkeypatch.setenv('Y2_CONV_FORCE_STREAMK', '1')           # small test shapes have fewer tiles than the auto rule wants
    ops.reload_env()                         # the launchers cache the Y2_* switches
    got1 = ops.conv_fwd_bf16(xb, wp, k, Cin, Cout, **kw)
    got2 = ops.conv_fwd_bf16(xb, wp, k, Cin, Cout, **kw)
    torch.cuda.synchronize()
    assert torch.equal(got1, got2)
    got = got1.float().cpu().numpy().reshape(-1, Cout)
    tol = 2e-4 if out_f32 else 1e-2                             # fp32 accumulation order / one bf16 ulp
    np.testing.assert_allclose(got, ref, rtol=tol, atol=tol * np.abs(ref).max())
    if N > 16:                                                  # full-size cases: float64 oracle on a slice of the batch
        x, got = x[:4], got[:4 * S * S]
    want = O.conv2d_same(O.bf16_round(torch.tensor(x)).double(), O.bf16_round(torch.tensor(w)).double(), torch.float64)
    if sc is not None:
        want = want * torch.tensor(sc).double()
    want = want + torch.tensor(b).double()
    if not out_f32:
        want = torch.maximum(O.ALPHA * want, want)
    want = want.numpy().reshape(-1, Cout)
    tol = 1e-3 if out_f32 else 1e-2
    np.testing.assert_allclose(got, want, rtol=tol, atol=tol * np.abs(want).max())
    assert np.linalg.norm(got - want) / np.linalg.norm(want) < (1e-4 if out_f32 else 4e-3)


# ---------------------------------------------------------------------------------- a2 / a3
def test_bn_stats_fold_matches_two_step(ops):
    """y2_bn_stats_fold == y2_bn_stats followed by y2_bn_fold(mean=0, bias=None), bit for bit."""
    rs = np.random.RandomState(5)
    M, C = 5 * 13 * 13, 96
    x = cu((rs.randn(M, C) * rs.uniform(0.5, 3, C) + rs.randn(C) * 10).astype(np.float32))
    gamma, beta = cu(rs.uniform(0.5, 1.5, C).astype(np.float32)), cu(rs.randn(C).astype(np.float32))
    mean, var = ops.bn_stats(x, C)
    sc, sh = ops.bn_fold(gamma, beta, torch.zeros_like(mean), var, None)
    m2, v2, sc2, sh2 = ops.bn_stats_fold(x, C, gamma, beta)
    torch.cuda.synchronize()
    assert torch.equal(mean, m2) and torch.equal(var, v2) and torch.equal(sc, sc2) and torch.equal(sh, sh2)


@pytest.mark.parametrize('C,ld,ldo,col', [(1024, 1024, None, 0), (72, 96, 160, 8)])
def test_affine_rows_fast_path_equals_generic(ops, monkeypatch, C, ld, ldo, col):
    """The row-walking bf16 kernel of the batch-statistics head layers == the generic kernel, bit for bit (dense rows and
    a channel slice of a wider tensor)."""
    rs = np.random.RandomState(6)
    N, S = 3, 13
    x = cu((rs.randn(N * S * S, ld) * 3).astype(np.float32))
    sub, sc, sh = (cu(rs.randn(C).astype(np.float32)) for _ in range(3))
    outs = []
    for generic in (False, True):
        if generic:
            monkeypatch.setenv('Y2_AFFINE_GENERIC', '1')
            ops.reload_env()                     # the launchers cache the Y2_* switches
        out = torch.zeros((N, S, S, ldo or C), dtype=torch.bfloat16, device='cuda')
        ops.affine_leaky_pool(x, N, S, S, C, ldx=ld, sub=sub, scale=sc, shift=sh, leaky=True, out_bf16=True, out=out,
                              ldo=ldo, out_col=col)
        outs.append(out)
    torch.cuda.synchronize()
    assert torch.equal(outs[0], outs[1])
    want = (x[:, :C] - sub) * sc + sh
    want = torch.maximum(want, 0.1 * want).to(torch.bfloat16).float().reshape(N, S, S, C)
    got = outs[0][..., col:col + C].float()
    assert (got - want).abs().max() <= 2e-2 * want.abs().max()


def test_bn_stats_large_mean(ops):
    rs = np.random.RandomState(2)
    M, C = 3 * 13 * 13, 70
    x = (rs.randn(M, C) * rs.uniform(0.5, 3, C) * 1e6 + rs.randn(C) * 1e9).astype(np.float32)   # |mean| >> std
    mean, var = ops.bn_stats(cu(x), C)
    np.testing.assert_allclose(mean.cpu().numpy(), x.astype(np.float64).mean(0), rtol=1e-6)
    np.testing.assert_allclose(var.cpu().numpy(), x.astype(np.float64).var(0), rtol=1e-5)


@pytest.mark.parametrize('C,pool,bf16', [(64, True, False), (125, False, False), (32, True, True), (30, False, False)])
def test_affine_leaky_pool(ops, C, pool, bf16):
    rs = np.random.RandomState(3)
    N, H, W = 2, 8, 6
    ld = (C + 31) // 32 * 32
    x = rs.randn(N * H * W, ld).astype(np.float32)
    sub, scale, shift = [rs.randn(C).astype(np.float32) for _ in range(3)]
    y = (torch.tensor(x[:, :C]).double().reshape(N, H, W, C) - torch.tensor(sub).double()) * torch.tensor(scale).double() \
        + torch.tensor(shift).double()
    y = torch.maximum(O.ALPHA * y, y)
    if pool:
        y = O.max_pool_2x2(y)
    got = ops.affine_leaky_pool(cu(x), N, H, W, C, ldx=ld, sub=cu(sub), scale=cu(scale), shift=cu(shift), leaky=True,
                                pool=pool, out_bf16=bf16).float().cpu().numpy()
    np.testing.assert_allclose(got, y.numpy(), rtol=1e-2 if bf16 else 1e-5, atol=1e-2 if bf16 else 1e-5)


def test_affine_space_to_depth_into_concat_slice(ops):
    """Passthrough / reorg folded into the store address: the 26x26x64 branch lands space-to-depth in channels
    [1024, 1280) of a [N,13,13,1280] tensor whose first 1024 channels belong to another producer."""
    rs = np.random.RandomState(11)
    N, H, W, C = 2, 26, 26, 64
    x = rs.randn(N * H * W, C).astype(np.float32)
    scale, shift = rs.uniform(0.5, 1.5, C).astype(np.float32), rs.randn(C).astype(np.float32)
    cat = torch.full((N, H // 2, W // 2, 1280), 7.0, dtype=torch.bfloat16, device='cuda')
    ops.affine_leaky_pool(cu(x), N, H, W, C, scale=cu(scale), shift=cu(shift), leaky=True, out_bf16=True, out=cat,
                          ldo=1280, out_col=1024, space_to_depth=True)
    y = torch.tensor(x).double().reshape(N, H, W, C) * torch.tensor(scale).double() + torch.tensor(shift).double()
    y = torch.maximum(O.ALPHA * y, y)
    want = O.space_to_depth2(y).to(torch.bfloat16).float().numpy()
    got = cat.float().cpu().numpy()
    assert np.all(got[..., :1024] == 7.0)                                 # the other producer's slice is untouched
    np.testing.assert_allclose(got[..., 1024:], want, rtol=1e-2, atol=1e-2)
    # dense slice with a row stride (conv2's share of the same tensor)
    x2 = rs.randn(N * 13 * 13, 1024).astype(np.float32)
    ops.affine_leaky_pool(cu(x2), N, 13, 13, 1024, leaky=False, out_bf16=True, out=cat, ldo=1280, out_col=0)
    got = cat.float().cpu().numpy()
    np.testing.assert_array_equal(got[..., :1024], torch.tensor(x2).to(torch.bfloat16).float().numpy().reshape(N, 13, 13, 1024))
    np.testing.assert_allclose(got[..., 1024:], want, rtol=1e-2, atol=1e-2)


def test_maxpool2x2_bf16(ops):
    x = torch.randn((3, 26, 26, 512), generator=torch.Generator().manual_seed(5)).to(torch.bfloat16)
    got = ops.maxpool2x2_bf16(x.cuda()).float().cpu()
    want = O.max_pool_2x2(x.float())
    assert torch.equal(got, want)                                         # max of bf16 values: exact


def test_bn_fold_and_moving(ops):
    rs = np.random.RandomState(4)
    C = 50
    g, b, m, bias = [rs.randn(C).astype(np.float32) for _ in range(4)]
    v = rs.uniform(0.1, 2, C).astype(np.float32)
    scale, shift = ops.bn_fold(cu(g), cu(b), cu(m), cu(v), cu(bias))
    s = g / np.sqrt(v + 1e-3)
    np.testing.assert_allclose(scale.cpu().numpy(), s, rtol=1e-5)
    np.testing.assert_allclose(shift.cpu().numpy(), b + (bias - m) * s, rtol=1e-4, atol=1e-5)
    mm, mv = cu(np.zeros(C, np.float32)), cu(np.ones(C, np.float32))
    ops.bn_update_moving(mm, mv, cu(m), cu(v))
    np.testing.assert_allclose(mm.cpu().numpy(), m * 0.01, rtol=1e-4, atol=1e-7)
    np.testing.assert_allclose(mv.cpu().numpy(), 0.99 + v * 0.01, rtol=1e-5)


# ---------------------------------------------------------------------------------- a8
@pytest.mark.parametrize('name,S,B', [('s7', 7, 2), ('s13', 13, 5)])
def test_decode_ref_v1_golden(ops, golden_dir, name, S, B):
    g = np.load(os.path.join(golden_dir, 'ref_decode.npz'))
    pred = g[name + '_pred']
    boxes, conf, keep, cls = [t.cpu().numpy() for t in ops.decode_ref_v1(cu(pred), S, B, 20, 0.5)]
    dec = O.decode_ref_v1(pred[0], S, B, 20, 0.5)
    np.testing.assert_array_equal(boxes[0, ..., 0], dec['xs'])        # same fp32 op order: bit-exact
    np.testing.assert_array_equal(boxes[0, ..., 1], dec['ys'])
    np.testing.assert_array_equal(boxes[0, ..., 2], dec['ws'])
    np.testing.assert_array_equal(boxes[0, ..., 3], dec['hs'])
    np.testing.assert_array_equal(keep[0].astype(bool), dec['keep'])
    np.testing.assert_array_equal(cls[0], dec['cls'])
    # and the reference's own draw list (golden produced by the reference source)
    im_w, im_h = [int(v) for v in g['im_wh']]
    d = dict(xs=boxes[0, ..., 0], ys=boxes[0, ..., 1], ws=boxes[0, ..., 2], hs=boxes[0, ..., 3], conf=conf[0],
             keep=keep[0].astype(bool), cls=cls[0])
    rects = np.array([r[:4] for r in O.draw_list_ref_v1(d, im_w, im_h)], dtype=np.int64).reshape(-1, 4)
    np.testing.assert_array_equal(rects, g[name + '_rects'])


# ---------------------------------------------------------------------------------- a' region decode
@pytest.mark.parametrize('N,S', [(3, 13), (2, 19), (1, 7)])
def test_decode_region_vs_oracle(ops, N, S):
    net = (2.0 * np.random.RandomState(1234).randn(N, S, S, 125)).astype(np.float32)
    boxes, scores = ops.decode_region(cu(net), cu(O.VOC_ANCHORS), 20, 0.3)
    wb, ws_thr, ws = O.region_decode_v2(net, O.VOC_ANCHORS, 20, 0.3)
    np.testing.assert_allclose(boxes.cpu().numpy(), wb, rtol=1e-5, atol=1e-7)
    got = scores.cpu().numpy()
    # threshold flips are allowed only for scores within 1e-5 relative of the threshold
    near = np.abs(ws - 0.3) < 1e-5
    np.testing.assert_allclose(got[~near], ws_thr[~near], rtol=1e-5, atol=1e-7)


# ---------------------------------------------------------------------------------- a' NMS (bit-exact)
def _nms_check(ops, boxes, scores, score_thr, iou_thr):
    ki, kc = ops.nms(cu(boxes), cu(scores), score_thr, iou_thr)
    ki, kc = ki.cpu().numpy(), kc.cpu().numpy()
    for n in range(boxes.shape[0]):
        want = O.nms_per_class(boxes[n], scores[n], iou_thr, score_thr)
        for k in range(scores.shape[2]):
            assert kc[n, k] == len(want[k]), (n, k, kc[n, k], len(want[k]))
            np.testing.assert_array_equal(ki[n, k, :kc[n, k]], want[k])


def test_nms_bit_exact_decoded(ops):
    net = (2.0 * np.random.RandomState(1234).randn(4, 13, 13, 125)).astype(np.float32)
    boxes, scores = ops.decode_region(cu(net), cu(O.VOC_ANCHORS), 20, 0.3)
    _nms_check(ops, boxes.cpu().numpy(), scores.cpu().numpy(), 0.3, 0.45)


def test_nms_bit_exact_dense_overlaps(ops):
    rs = np.random.RandomState(7)
    N, nbox, C = 2, 845, 20
    boxes = np.concatenate([rs.uniform(0.3, 0.7, (N, nbox, 2)), rs.uniform(0.05, 0.5, (N, nbox, 2))], -1).astype(np.float32)
    scores = rs.uniform(0, 1, (N, nbox, C)).astype(np.float32)
    scores[scores < 0.6] = 0                         # ~40% candidates per class, heavy overlap
    scores[0, 5:40, 3] = 0.75                        # score ties -> index order
    boxes[0, 100] = boxes[0, 101]                    # identical boxes -> IoU 1
    _nms_check(ops, boxes, scores, 0.3, 0.45)


def test_nms_worst_case_all_candidates_and_empty(ops):
    rs = np.random.RandomState(8)
    N, nbox, C = 1, 845, 3
    boxes = np.concatenate([rs.uniform(0, 1, (N, nbox, 2)), rs.uniform(0.01, 0.3, (N, nbox, 2))], -1).astype(np.float32)
    scores = rs.uniform(0.01, 1, (N, nbox, C)).astype(np.float32)
    scores[:, :, 2] = 0                              # an empty class
    _nms_check(ops, boxes, scores, 0.0, 0.45)        # thresh 0: every box of classes 0,1 is a candidate


def test_nms_fallback_path_1805_boxes(ops):
    rs = np.random.RandomState(9)
    N, nbox, C = 1, 1805, 2
    boxes = np.concatenate([rs.uniform(0, 1, (N, nbox, 2)), rs.uniform(0.01, 0.2, (N, nbox, 2))], -1).astype(np.float32)
    scores = rs.uniform(0.01, 1, (N, nbox, C)).astype(np.float32)
    _nms_check(ops, boxes, scores, 0.0, 0.45)        # n > 1024 -> on-the-fly sweep


# ---------------------------------------------------------------------------------- a6 / a7 loss
@pytest.mark.parametrize('name', ['katA', 'katB', 'katC', 'rand7', 'rand13', 'rand19'])
def test_loss_v1_golden(ops, golden_dir, name):
    g = np.load(os.path.join(golden_dir, 'ref_loss.npz'))
    IS, S, B = [int(v) for v in g[name + '_cfg']]
    net, lab = g[name + '_net'], g[name + '_labels']
    terms, ious, mask, dnet = ops.loss_v1(cu(net, torch.float32), cu(lab, torch.float32), S, B, 20, IS)
    r = O.get_loss(net, lab, 20, net.shape[0], IS, S, B, with_grad=True)
    want_terms = [r['class_loss'], r['coord_loss'], r['object_loss'], r['noobject_loss'], r['loss']]
    np.testing.assert_allclose(terms.cpu().numpy(), want_terms, rtol=1e-3, atol=1e-6)      # spec: 1e-3 relative
    assert float(terms[4]) == pytest.approx(float(g[name + '_loss']), rel=1e-3)            # the reference's own graph
    np.testing.assert_allclose(ious.cpu().numpy(), r['ious'], atol=2e-6)
    np.testing.assert_array_equal(mask.cpu().numpy(), r['object_mask'])
    gmax = np.abs(r['dnet']).max()
    np.testing.assert_allclose(dnet.cpu().numpy(), r['dnet'], rtol=1e-3, atol=1e-5 * gmax)
    if name not in ('katA', 'katB'):
        np.testing.assert_allclose(dnet.cpu().numpy(), g[name + '_dnet'], rtol=1e-3, atol=1e-5 * gmax)


def test_loss_v1_batch64(ops):
    rs = np.random.RandomState(0)
    N, S, B, IS = 64, 13, 5, 416
    net = rs.uniform(-0.3, 1.0, (N, S, S, 45)).astype(np.float32)
    lab = np.zeros((N, S, S, 25), np.float32)
    for n in range(N):
        for _ in range(rs.randint(1, 4)):
            cx, cy = rs.uniform(0, IS, 2)
            j, i = int(cx * S / IS), int(cy * S / IS)
            if lab[n, i, j, 0] == 1:
                continue
            lab[n, i, j, :5] = [1, cx, cy, rs.uniform(20, 300), rs.uniform(20, 300)]
            lab[n, i, j, 5 + rs.randint(20)] = 1
    terms, ious, mask, dnet = ops.loss_v1(cu(net), cu(lab), S, B, 20, IS)
    r = O.get_loss(net, lab, 20, N, IS, S, B, with_grad=True)
    assert float(terms[4]) == pytest.approx(r['loss'], rel=1e-4)
    np.testing.assert_array_equal(mask.cpu().numpy(), r['object_mask'])
    np.testing.assert_allclose(dnet.cpu().numpy(), r['dnet'], rtol=1e-3, atol=1e-5 * np.abs(r['dnet']).max())


# ---------------------------------------------------------------------------------- a11 Adam
def test_adam_step(ops):
    rs = np.random.RandomState(5)
    n = 10007
    p, g, m, v = rs.randn(n).astype(np.float32), rs.randn(n).astype(np.float32), \
        rs.randn(n).astype(np.float32) * 0.1, rs.uniform(0, 1, n).astype(np.float32)
    pt, mt, vt = cu(p), cu(m), cu(v)
    ops.adam_step(pt, cu(g), mt, vt, step=3)
    wp, wm, wv = O.adam_step(p.astype(np.float64), g.astype(np.float64), m.astype(np.float64), v.astype(np.float64), 3)
    np.testing.assert_allclose(pt.cpu().numpy(), wp, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(mt.cpu().numpy(), wm, rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(vt.cpu().numpy(), wv, rtol=1e-5, atol=1e-7)


def test_adam_step_ex_scale_zero_and_device_lr(ops):
    """y2_adam_step_ex == Adam on grad_scale * g, with the step size read from device memory and g cleared behind the read."""
    rs = np.random.RandomState(6)
    n = 4096 * 5
    p, g, m, v = rs.randn(n).astype(np.float32), rs.randn(n).astype(np.float32) * 4, \
        rs.randn(n).astype(np.float32) * 0.1, rs.uniform(0, 1, n).astype(np.float32)
    wp, wm, wv = O.adam_step(p.astype(np.float64), 0.25 * g.astype(np.float64), m.astype(np.float64), v.astype(np.float64), 7)
    for dev_lr in (False, True):
        pt, gt, mt, vt = cu(p), cu(g), cu(m), cu(v)
        lr_t = ops.adam_lr_t(7)
        lr_dev = torch.tensor([lr_t], dtype=torch.float32).cuda() if dev_lr else None
        ops.adam_step_ex(pt, gt, mt, vt, lr_t=0.0 if dev_lr else lr_t, lr_t_dev=lr_dev, grad_scale=0.25, zero_grad=True)
        np.testing.assert_allclose(pt.cpu().numpy(), wp, rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(mt.cpu().numpy(), wm, rtol=1e-5, atol=1e-7)
        np.testing.assert_allclose(vt.cpu().numpy(), wv, rtol=1e-5, atol=1e-7)
        assert float(gt.abs().max()) == 0.0
    gt = cu(g)
    ops.adam_step_ex(cu(p), gt, cu(m), cu(v), lr_t=1e-3, zero_grad=False)
    assert torch.equal(gt, cu(g))


# ---- fused decode + NMS ---------------------------------------------------------------------------
@pytest.mark.parametrize('impl', ['detect_fused', 'detect_split'])
@pytest.mark.parametrize('N,S,thr', [(7, 13, 0.3), (3, 19, 0.2), (2, 13, 0.01), (2, 7, 0.3), (64, 13, 0.1)])
def test_detect_fused_equals_decode_plus_nms_and_oracle(ops, impl, N, S, thr):
    detect = getattr(ops, impl)          # one CTA per image / chunked decode + per-image NMS over candidate lists
    rs = np.random.RandomState(S * 10 + N)
    net = (2.0 * rs.randn(N, S, S, 125)).astype(np.float32)
    an = cu(O.VOC_ANCHORS)
    b0, s0 = ops.decode_region(cu(net), an, 20, thr)
    ki0, kc0 = ops.nms(b0, s0, thr, 0.45)
    ks = torch.zeros((N, 20, S * S * 5), dtype=torch.float32, device='cuda')
    b1, s1, ki1, kc1, _ = detect(cu(net), an, 20, thr, 0.45, keep_score=ks)
    if impl == 'detect_split':           # second call on the same (self-resetting) workspace must agree with the first
        ks2 = torch.zeros_like(ks)
        b2, s2, ki2, kc2, _ = detect(cu(net), an, 20, thr, 0.45, keep_score=ks2)
        torch.cuda.synchronize()
        assert torch.equal(kc1, kc2) and torch.equal(s1, s2) and torch.equal(b1, b2) and torch.equal(ks, ks2)
        assert int(ops.detect_workspace(N, 20, b1.device)[:N * 20 * 4].view(torch.int32).abs().sum()) == 0
    torch.cuda.synchronize()
    # the fused kernel uses the fast intrinsics (ex2.approx / rcp.approx), the two-kernel path expf and IEEE division:
    # both sit inside the spec's 1e-5; a score within that distance of the threshold may be kept by one and not the other
    np.testing.assert_allclose(b1.cpu().numpy(), b0.cpu().numpy(), rtol=1e-5, atol=1e-7)
    d = np.abs(s1.cpu().numpy() - s0.cpu().numpy())
    near = np.abs(np.maximum(s1.cpu().numpy(), s0.cpu().numpy()) - thr) < 1e-5
    assert np.all((d <= 1e-5 * np.abs(s0.cpu().numpy()) + 1e-7) | near)
    # oracle: decode parity, then NMS on the fused kernel's own boxes/scores must give its keep lists bit-exactly
    wb, wst, _ = O.region_decode_v2(net, O.VOC_ANCHORS, 20, thr)
    np.testing.assert_allclose(b1.cpu().numpy(), wb, rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(s1.cpu().numpy(), wst, rtol=1e-4, atol=1e-6)
    boxes, scores = b1.cpu().numpy(), s1.cpu().numpy()
    ki, kc, ksc = ki1.cpu().numpy(), kc1.cpu().numpy(), ks.cpu().numpy()
    total = 0
    for n in range(N):
        keeps = O.nms_per_class(boxes[n], scores[n], 0.45, thr)
        for k in range(20):
            assert kc[n, k] == len(keeps[k])
            np.testing.assert_array_equal(ki[n, k, :kc[n, k]], keeps[k])
            np.testing.assert_array_equal(ksc[n, k, :kc[n, k]], scores[n, keeps[k], k])
            total += len(keeps[k])
    assert total > 0
    if float((s0 != s1).sum()) == 0:        # identical scores -> identical keep lists from the two-kernel path
        assert torch.equal(kc0, kc1)


@pytest.mark.parametrize('impl', ['detect_fused', 'detect_split'])
def test_detect_fused_overflow_falls_back_to_bitmatrix_kernel(ops, impl):
    """threshold 0: all 845 x 20 candidates (> 2048) -> image flagged and re-done by nms_kernel; and a mixed batch."""
    detect = getattr(ops, impl)
    rs = np.random.RandomState(77)
    net = (1.0 * rs.randn(3, 13, 13, 125)).astype(np.float32)
    net[1, ..., 4::25] = -30.0                       # image 1: objectness ~ 0 -> scores underflow below any threshold
    an = cu(O.VOC_ANCHORS)
    b1, s1, ki1, kc1, _ = detect(cu(net), an, 20, 1e-12, 0.45, max_keep=845)
    torch.cuda.synchronize()
    boxes, scores = b1.cpu().numpy(), s1.cpu().numpy()
    ki, kc = ki1.cpu().numpy(), kc1.cpu().numpy()
    assert (kc >= 0).all()
    for n in range(3):
        keeps = O.nms_per_class(boxes[n], scores[n], 0.45, 1e-12)
        for k in range(20):
            assert kc[n, k] == len(keeps[k])
            np.testing.assert_array_equal(ki[n, k, :kc[n, k]], keeps[k])
    # without a scores buffer the overflowed images are reported, not silently dropped
    _, _, _, kc2, _ = detect(cu(net), an, 20, 1e-12, 0.45, max_keep=845, want_scores=False)
    torch.cuda.synchronize()
    assert (kc2.cpu().numpy()[0] == -1).all()


# ---------------------------------------------------------------------------------- a7 standalone + histogram deltas
def test_iou_vs_reference_golden(ops, golden_dir):
    """y2_iou / ops.iou / net_utils.get_iou against the golden emitted by the reference's own get_iou (net_utils.py:222-260)
    -- including the SURVEY 8c KATs baked into the fixture (1.0, 0.25, 0.0, 1/3, zero area)."""
    from tensorflow_yolo2_b200.yolo2_nets import net_utils as nu
    g = np.load(os.path.join(golden_dir, 'ref_iou.npz'))
    b1, b2 = g['boxes1'].astype(np.float32), g['boxes2'].astype(np.float32)
    got = ops.iou(cu(b1), cu(b2)).cpu().numpy()
    assert got.shape == g['iou'].shape
    np.testing.assert_allclose(got, g['iou'], atol=2e-6)                     # golden is the float64 graph
    want32 = O.get_iou(b1, b2)                                               # same op order in float32: bit-exact
    np.testing.assert_array_equal(got, want32)
    assert got[0, 0, 0, 0] == 1.0 and got[0, 0, 2, 0] == 0.0 and got[0, 1, 1, 0] == 0.0
    assert abs(got[0, 0, 1, 0] - 0.25) < 1e-6 and abs(got[0, 1, 0, 0] - 1.0 / 3.0) < 1e-6
    got2 = nu.get_iou(cu(b1), cu(b2)).cpu().numpy()                          # the drop-in entry point
    np.testing.assert_array_equal(got2, got)
    # a big ragged batch: 1e6 random pairs, property = oracle bit-exactness on a strided sample + range
    rs = np.random.RandomState(3)
    a, b = rs.uniform(0, 1, (1000003, 4)).astype(np.float32), rs.uniform(0, 1, (1000003, 4)).astype(np.float32)
    big = ops.iou(cu(a), cu(b)).cpu().numpy()
    assert big.min() >= 0.0 and big.max() <= 1.0
    np.testing.assert_array_equal(big[::997], O.get_iou(a[::997], b[::997]))


def test_loss_box_deltas_histogram_inputs(ops, golden_dir):
    """y2_loss_v1_box_deltas = the tensors behind tf.summary.histogram('boxes_delta_x' .. 'boxes_delta_h')
    (net_utils.py:337-342,366-369), against a NumPy restatement of those lines."""
    g = np.load(os.path.join(golden_dir, 'ref_loss.npz'))
    net, lab = g['rand13_net'].astype(np.float32), g['rand13_labels'].astype(np.float32)
    N, S, B, C, IS = net.shape[0], 13, 5, 20, 416.0
    got = ops.loss_v1_box_deltas(cu(net), cu(lab), S, B, C, IS).cpu().numpy()
    pb = net[..., C + B:].reshape(N, S, S, B, 4)
    gt = np.tile((lab[..., 1:5] / np.float32(IS))[:, :, :, None, :], (1, 1, 1, B, 1))
    off = np.tile(np.arange(S, dtype=np.float32)[None, None, :, None], (N, S, 1, B))      # offset[y, x, b] = x
    want = np.stack([pb[..., 0] - (gt[..., 0] * S - off), pb[..., 1] - (gt[..., 1] * S - off.transpose(0, 2, 1, 3)),
                     pb[..., 2] - np.sqrt(gt[..., 2]), pb[..., 3] - np.sqrt(gt[..., 3])], axis=-1)
    np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-6)


# ---------------------------------------------------------------------------------- a1: the call is checked before any path
def test_conv_streamk_shape_with_overlapping_output_rows_is_refused(ops):
    """A 64x13x13 1024 -> 1024 3x3 layer runs on the stream-K kernel (the default workspace is registered).  Output rows that
    overlap are refused before that kernel is planned: float32 rows of stride 256 < Cout, and hi | lo bf16 rows whose lo
    half starts at column 8, inside the hi half.  Each output holds every address such a launch would write, so a call that
    got through would still stay in bounds."""
    from tensorflow_yolo2_b200 import _lib
    N, S, C_ = 64, 13, 1024
    M = N * S * S
    x = torch.zeros((N, S, S, C_), dtype=torch.bfloat16, device='cuda')
    wp = ops.pack_weights_bf16(torch.zeros((3, 3, C_, C_), dtype=torch.float32, device='cuda'))
    y32 = torch.zeros((M * C_,), dtype=torch.float32, device='cuda')
    with pytest.raises(_lib.Y2Error, match='ldy >= c.Cout'):
        ops.conv_fwd_bf16(x, wp, 3, C_, C_, out_f32=True, ldy=256, out=y32)
    y16 = torch.zeros((M * 2 * C_,), dtype=torch.bfloat16, device='cuda')
    with pytest.raises(_lib.Y2Error, match='lo_off >= c.Cout'):
        ops.conv_fwd_bf16(x, wp, 3, C_, C_, split_out=True, lo_off=8, ldy=2 * C_, out=y16)
    torch.cuda.synchronize()
    assert not y32.any() and not y16.any()


# ---------------------------------------------------------------------------------- a10 / f2: cv2.resize on the GPU
def test_resize_bilinear_u8_bit_exact_vs_cv2(ops, golden_dir):
    """y2_resize_bilinear_u8 == cv2.resize (the call of pascal_detect_darknet.py:35 / pascal_voc.py:61), bit for bit, on the
    reference's fixtures at 224 / 416 / 608 and on random up- / down-scales incl. the exact-2x INTER_AREA switch; and the
    engine's load_images() path == host cv2.resize + copy."""
    import cv2
    rs = np.random.RandomState(1)
    cases = []
    for f in ('testImg1.jpg', 'testImg2.jpg'):
        im = cv2.imread(os.path.join(golden_dir, f))
        cases += [(im, IS, IS) for IS in (224, 416, 608)]
    cases += [(rs.randint(0, 256, (h, w, 3)).astype(np.uint8), dh, dw) for (h, w, dh, dw) in
              [(240, 352, 416, 416), (375, 500, 608, 608), (832, 832, 416, 416), (100, 100, 416, 416), (1000, 750, 416, 416),
               (123, 457, 224, 224), (37, 41, 96, 96), (416, 416, 416, 416), (333, 500, 200, 300)]]
    for im, dh, dw in cases:
        got = ops.resize_bilinear_u8(cu(im), dh, dw).cpu().numpy()
        np.testing.assert_array_equal(got, cv2.resize(im, (dw, dh)))
        np.testing.assert_array_equal(got, O.resize_bilinear_u8(im, dw, dh))
    from tensorflow_yolo2_b200.engine import Yolo2Engine
    from tests.helpers import make_store
    st, _ = make_store(125, tame=True)
    eng = Yolo2Engine(2, 96, 125, store=st, use_cuda_graph=False)
    ims = [cv2.imread(os.path.join(golden_dir, f)) for f in ('testImg1.jpg', 'testImg2.jpg')]
    eng.load_images(ims)
    want = np.stack([cv2.resize(im, (96, 96)) for im in ims])
    np.testing.assert_array_equal(eng.in_u8.cpu().numpy(), want)


@pytest.mark.parametrize('k,Cin,Cout', [(3, 32, 64), (3, 64, 125), (1, 1024, 125), (3, 512, 1024), (1, 96, 40)])
def test_pack_weights_tiled_equals_generic(ops, monkeypatch, k, Cin, Cout):
    """The transposing (coalesced) weight packer writes exactly what the element-wise one does, padding included."""
    rs = np.random.RandomState(k + Cin + Cout)
    w = cu(rs.randn(k, k, Cin, Cout).astype(np.float32))
    n = int(ops._lib.load().y2_conv_packed_weight_elems(k, Cin, Cout))
    a = torch.full((n,), 7.0, dtype=torch.bfloat16, device='cuda')
    ops.pack_weights_bf16(w, out=a)
    monkeypatch.setenv('Y2_AFFINE_GENERIC', '1')            # (the switch that forces every generic element-wise variant)
    ops.reload_env()
    b = torch.full((n,), 9.0, dtype=torch.bfloat16, device='cuda')
    ops.pack_weights_bf16(w, out=b)
    assert torch.equal(a, b)
    cout_p = (Cout + 15) // 16 * 16
    want = torch.zeros((cout_p, k * k, Cin), dtype=torch.float32, device='cuda')
    want[:Cout] = w.permute(3, 0, 1, 2).reshape(Cout, k * k, Cin)
    assert torch.equal(a.view(cout_p, k * k, Cin).float(), want.to(torch.bfloat16).float())
