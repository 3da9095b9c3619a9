"""GPU parity of the "bf16x3" precision mode and END-TO-END detection parity of the engine against the float64 oracle.

north_star (BASELINE.json): "decoded boxes and scores within 1e-3 relative (bf16 convs, fp32 accumulate) ... NMS
keep-lists bit-exact on identical inputs".  The plain bf16 tensor-core path rounds every conv operand to 8 mantissa
bits; after 22 layers the network output is ~1e-2 off (measured below and reported, not hidden).  The bf16x3 path
(hi + lo bf16 pairs, three tcgen05.mma per K step) is the one that meets the 1e-3 bar; these tests assert it at
BASELINE configs[1] (416^2, batch 64, untamed seed-0 weights -- what bench.py times) and configs[3] (608^2, batch 32).
"""
import json
import os

import numpy as np
import pytest
import torch

from oracle import yolo2_oracle as O
from tests import parity_detect as PD
from tests.helpers import rel_l2

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


def split_pair(x):
    """float32 numpy -> [.., 2C] bf16 torch tensor [hi | lo] (the Y2_CONV_IN_SPLIT layout)."""
    t = torch.tensor(x)
    hi = t.to(torch.bfloat16)
    lo = (t - hi.float()).to(torch.bfloat16)
    return torch.cat([hi, lo], dim=-1).contiguous()


def join_pair(y):
    c = y.shape[-1] // 2
    return y[..., :c].float() + y[..., c:].float()


# ---- kernel level: the split conv in every tiling mode of conv_tc_kernel / conv_streamk2_kernel --------------------------
@pytest.mark.parametrize('N,H,W,Cin,Cout,k,pool,out_f32', [
    (2, 72, 72, 32, 64, 3, True, False),        # halo-patch pair, 64-byte rows (layer 2 shape), pooled bf16 epilogue
    (2, 80, 64, 64, 128, 3, False, False),      # halo-patch, 128-wide, un-pooled (layer 3 shape): generic split epilogue
    (2, 70, 68, 64, 128, 3, False, False),      # ... with tiles clipped at the right / bottom edge
    (1, 64, 64, 128, 64, 3, False, False),      # layer 4 shape
    (3, 26, 26, 256, 512, 3, True, False),      # tiled boxes + pool, streamed B, pair
    (4, 26, 26, 512, 256, 1, False, False),     # 1x1, im2col mode
    (32, 13, 13, 512, 1024, 3, False, False),   # stream-K pair kernel, bf16 split output
    (32, 13, 13, 1024, 1024, 3, False, True),   # stream-K, float32 rows (head layers), 432 K steps per tile
    (5, 13, 13, 1024, 125, 1, False, True),     # output layer
    (2, 7, 7, 64, 48, 3, False, False),         # Cout not a multiple of 32: scalar split stores
])
def test_conv_split_vs_oracle(ops, N, H, W, Cin, Cout, k, pool, out_f32):
    """y2_conv_fwd_bf16 with IN_SPLIT (+ OUT_SPLIT) against a float64 convolution of the SAME (hi + lo) operands:
    the three-MMA scheme drops only a_lo*w_lo (2^-18) -> 2e-5 relative."""
    rs = np.random.RandomState(Cin + Cout + H)
    x = (rs.randn(N, H, W, Cin) * 2 + 0.7).astype(np.float32)
    w = (rs.randn(k, k, Cin, Cout) * 0.1).astype(np.float32)
    scale = (rs.uniform(0.5, 1.5, Cout) * np.where(rs.rand(Cout) < 0.3, -1, 1)).astype(np.float32)
    shift = (rs.randn(Cout) * 0.3).astype(np.float32)
    xs = split_pair(x).cuda()
    wp = ops.pack_weights_bf16_split(cu(w))
    ld = (Cout + 31) // 32 * 32 if out_f32 else None
    got = ops.conv_fwd_bf16(xs, wp, k, Cin, Cout, scale=cu(scale), shift=cu(shift), leaky=True, pool=pool, out_f32=out_f32,
                            ldy=ld, split_in=True, split_out=not out_f32)
    torch.cuda.synchronize()
    # oracle on the operands the kernel sees: x = hi + lo (16 bits), w = hi + lo
    xj = join_pair(xs.cpu()).double()
    wt = torch.tensor(w)
    wh = wt.to(torch.bfloat16).float()
    wj = (wh + (wt - wh).to(torch.bfloat16).float()).double()
    h = O.conv2d_same(xj, wj, torch.float64) * torch.tensor(scale).double() + torch.tensor(shift).double()
    h = torch.maximum(0.1 * h, h)
    if pool:
        h = O.max_pool_2x2(h)
    want = h.numpy()
    if out_f32:
        g = got.view(N, H, W, ld)[..., :Cout].cpu().numpy()
    else:
        assert got.shape[-1] == 2 * Cout
        g = join_pair(got.cpu()).numpy()
    e = rel_l2(g, want)
    print('split conv %s: rel_l2=%.3g' % ((N, H, W, Cin, Cout, k, pool, out_f32), e))
    assert e < 4e-5           # (measured 2.4e-5 at K = 3 * 9216: fp32 accumulation over 27 648 products)
    np.testing.assert_allclose(g, want, rtol=2e-4, atol=2e-4 * np.abs(want).max())


@pytest.mark.parametrize('N,H,W', [(2, 32, 16), (3, 96, 96), (2, 416, 416)])
def test_conv1_u8_pool_split_vs_oracle(ops, N, H, W):
    """bf16x3 first layer: exact integer pixels + ones channel, hi + lo weights with x = v*2/255 - 1 folded in, against the
    oracle's float64 preprocessing + conv + BN (negative gammas included) + leaky + pool."""
    rs = np.random.RandomState(17 + H)
    img = rs.randint(0, 256, (N, H, W, 3)).astype(np.uint8)
    w = (rs.randn(3, 3, 3, 32) * 0.3).astype(np.float32)
    b = (rs.randn(32) * 0.1).astype(np.float32)
    gamma = (rs.uniform(0.5, 1.5, 32) * np.where(rs.rand(32) < 0.3, -1, 1)).astype(np.float32)
    beta, mm = (rs.randn(32) * 0.2).astype(np.float32), (rs.randn(32) * 0.2).astype(np.float32)
    mv = rs.uniform(0.5, 2.0, 32).astype(np.float32)
    scale, shift = ops.bn_fold(cu(gamma), cu(beta), cu(mm), cu(mv), cu(b))
    wp = ops.pack_weights_conv1_u8_split(cu(w), scale)
    got = ops.conv1_u8_pool(cu(img), wp, shift, split=True)
    assert got.shape == (N, H // 2, W // 2, 64)
    g = join_pair(got.cpu()).numpy()
    p = dict(W=torch.tensor(w), b=torch.tensor(b), gamma=torch.tensor(gamma), beta=torch.tensor(beta), mm=torch.tensor(mm),
             mv=torch.tensor(mv))
    y, _, _ = O.conv_bn_layer(torch.tensor(O.preprocess_u8(img)), p, False, torch.float64)
    want = O.max_pool_2x2(y).numpy()
    e = rel_l2(g, want)
    print('split conv1 %s: rel_l2=%.3g' % ((N, H, W), e))
    assert e < 2e-5


@pytest.mark.parametrize('C,pool', [(1024, False), (64, True), (72, False)])
def test_affine_split_output(ops, C, pool):
    """y2_affine_leaky_pool_ex out_dtype 2: hi + lo == the float32 result to 2^-16."""
    rs = np.random.RandomState(C)
    N, H, W = 2, 6, 8
    x = (rs.randn(N * H * W, C) * 3).astype(np.float32)
    sub, sc, sh = [(rs.randn(C) * s).astype(np.float32) for s in (0.5, 1.0, 0.2)]
    ref = ops.affine_leaky_pool(cu(x), N, H, W, C, sub=cu(sub), scale=cu(sc), shift=cu(sh), pool=pool, out_bf16=False)
    got = ops.affine_leaky_pool(cu(x), N, H, W, C, sub=cu(sub), scale=cu(sc), shift=cu(sh), pool=pool, out_bf16=True,
                                split_out=True)
    assert got.shape[-1] == 2 * C
    hi = ops.affine_leaky_pool(cu(x), N, H, W, C, sub=cu(sub), scale=cu(sc), shift=cu(sh), pool=pool, out_bf16=True)
    assert torch.equal(got[..., :C], hi)                       # the hi half is the plain bf16 result
    np.testing.assert_allclose(join_pair(got.cpu()).numpy(), ref.cpu().numpy(), rtol=2e-5, atol=1e-30)


# ---- the drop-in builders in the bf16x3 mode (config.COMPUTE = 'bf16x3') -------------------------------------------------
@pytest.mark.parametrize('tame', [True, False])
def test_builders_bf16x3_vs_oracle(tame):
    """yolo2_nets.darknet.darknet19_core / darknet19_detection with config.COMPUTE = 'bf16x3' (float32 pixels in: exact FFMA
    first layer, then hi + lo pairs through the tensor-core kernels) against the float64 oracle -- no bf16-mirroring."""
    from tensorflow_yolo2_b200 import config, variables
    from tensorflow_yolo2_b200.yolo2_nets.darknet import darknet19_core, darknet19_detection
    from tests.helpers import make_store, oracle_params
    st, layers = make_store(125, tame=tame)
    core_p, head_p = oracle_params(st, layers)
    variables._DEFAULT_STORE = st
    st.reset_name_counters()
    x = np.random.RandomState(3).uniform(-1, 1, (4, 128, 128, 3)).astype(np.float32)
    want, inter = O.darknet19_forward(torch.tensor(x), core_p, head_p, dtype=torch.float64, return_intermediates=True)
    old = config.COMPUTE
    config.COMPUTE = 'bf16x3'
    try:
        core = darknet19_core(torch.tensor(x).cuda(), is_training=False)
        out = darknet19_detection(core, 125)
    finally:
        config.COMPUTE = old
        variables.reset_default_store(seed=0)
    assert core.dtype == torch.bfloat16 and core.shape == (4, 4, 4, 2048)            # [hi | lo]
    assert out.dtype == torch.float32 and out.shape == (4, 4, 4, 125)
    e_core = rel_l2(join_pair(core.cpu()).numpy(), inter[17].numpy())
    e_out = rel_l2(out.cpu().numpy(), want.numpy())
    print('bf16x3 builders vs float64 oracle: tame=%s core rel_l2=%.3g out rel_l2=%.3g' % (tame, e_core, e_out))
    assert e_core < 2e-4 and e_out < 5e-4


def test_get_loss_is_differentiable_like_tf_minimize(ops, golden_dir):
    """net_utils.get_loss as a torch.autograd node: loss.backward() / autograd.grad deliver the golden d loss / d net (the
    reference graph + autodiff, tests/golden/ref_loss.npz), scaled by the upstream gradient -- the minimize(loss) pattern
    of pascal_train_darknet.py:44-51."""
    from tensorflow_yolo2_b200 import config as cfg
    from tensorflow_yolo2_b200.yolo2_nets import net_utils as nu
    g = np.load(os.path.join(golden_dir, 'ref_loss.npz'))
    net = cu(g['rand7_net'].astype(np.float32)).requires_grad_(True)
    lab = g['rand7_labels']
    N = net.shape[0]
    loss, ious, mask = nu.get_loss(net, lab, 20, N, 224, 7, 2, cfg._grid_offset(7, 2))
    assert loss.requires_grad and not ious.requires_grad and not mask.requires_grad
    np.testing.assert_allclose(float(loss), float(g['rand7_loss']), rtol=1e-5)
    (3.0 * loss).backward()
    np.testing.assert_allclose(net.grad.cpu().numpy(), 3.0 * g['rand7_dnet'], rtol=1e-3, atol=1e-6)
    # composes with further torch ops upstream of net
    w = torch.ones_like(net, requires_grad=True)
    loss2 = nu.get_loss(net.detach() * w, lab, 20, N, 224, 7, 2)[0]
    (gw,) = torch.autograd.grad(loss2, w)
    np.testing.assert_allclose(gw.cpu().numpy(), g['rand7_dnet'] * g['rand7_net'], rtol=1e-3, atol=1e-6)
    # no grad required: plain forward, .dnet still available
    r = nu.get_loss(net.detach(), lab, 20, N, 224, 7, 2)
    assert not r[0].requires_grad
    np.testing.assert_allclose(r.dnet.cpu().numpy(), g['rand7_dnet'], rtol=1e-3, atol=1e-6)


# ---- end to end: engine (network + decode + NMS) vs the float64 oracle end to end ----------------------------------------
_ORACLE_CACHE = {}
_REPORT = []


def _case(batch, image_size, tame, precision, **kw):
    r = PD.run_case(batch, image_size, tame, precision, oracle_cache=_ORACLE_CACHE, **kw)
    _REPORT.append(r)
    print(json.dumps(r))
    return r


def _dump_report():
    out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'gpurun_out')
    try:
        os.makedirs(out, exist_ok=True)
        with open(os.path.join(out, 'parity_report.json'), 'w') as f:
            json.dump(_REPORT, f, indent=1)
    except OSError:
        pass


@pytest.mark.parametrize('tame', [False, True])
def test_detections_small_bf16x3_and_bf16(tame):
    """Quick case (batch 8, 160^2, low threshold so that detections exist): bf16x3 meets 1e-3; the bf16 numbers are
    printed beside it (and must at least stay within the 6e-2 the round-1 tests allowed)."""
    r3 = _case(8, 160, tame, 'bf16x3', score_thresh=0.05, per_layer=True)
    r1 = _case(8, 160, tame, 'bf16', score_thresh=0.05, per_layer=True)
    _dump_report()
    assert r3['matched'] > 0
    assert r3['score_rel_max'] < 1e-3 and r3['box_rel_max'] < 1e-3, r3
    assert r3['net_rel_l2'] < 2e-4, r3
    assert r1['net_rel_l2'] < 6e-2


@pytest.mark.parametrize('batch,image_size', [(64, 416), (32, 608)])
def test_detections_baseline_configs_bf16x3(batch, image_size):
    """BASELINE configs[1] / configs[3] with the weights bench.py times (reference initialiser, seed 0, thresh 0.3 / IoU
    0.45): every detection kept by both sides agrees to 1e-3 relative in score and box, and the keep lists are the
    oracle's except where a score sits within 2e-3 of the threshold or an IoU within 2e-3 of 0.45 (plus the boxes such a
    flip un-/suppresses): zero unexplained differences, >= 99 % identical."""
    r3 = _case(batch, image_size, False, 'bf16x3')
    r1 = _case(batch, image_size, False, 'bf16')
    _dump_report()
    assert r3['matched'] > 100, r3
    assert r3['score_rel_max'] < 1e-3 and r3['box_rel_max'] < 1e-3, r3
    assert r3['unexplained_list_differences'] == 0, r3
    assert r3['keep_lists_identical'] >= 0.99 and r3['detections_jaccard'] >= 0.995, r3
    # plain bf16: reported (see profiles/r2_parity.json); bounded so that a regression shows
    assert r1['net_rel_l2'] < 6e-2, r1
    assert r1['detections_jaccard'] > 0.5, r1


def test_detections_tame_416_bf16x3():
    r3 = _case(16, 416, True, 'bf16x3', score_thresh=0.05)
    _dump_report()
    assert r3['matched'] > 0
    assert r3['score_rel_max'] < 1e-3 and r3['box_rel_max'] < 1e-3, r3


@pytest.mark.parametrize('tame', [False, True])
def test_detections_config0_testimg1_batch1(golden_dir, tame):
    """BASELINE configs[0]: 416x416 detect on the reference's tests/testImg1.jpg, batch 1, random-init weights, 20 classes,
    5 anchors -- the image read and resized on the GPU by the engine (load_images == cv2.resize, bit-exact), bf16x3 engine
    against the float64 oracle end to end.  (Batch 1: the head's batch statistics run over 169 cells only.)"""
    import cv2
    from tensorflow_yolo2_b200.engine import Yolo2Engine
    from tests.helpers import make_store
    raw = cv2.imread(os.path.join(golden_dir, 'testImg1.jpg'))
    st, _ = make_store(125, tame=tame)
    eng = Yolo2Engine(1, 416, 125, store=st, use_cuda_graph=False, precision='bf16x3')
    eng.load_images([raw])
    img = eng.in_u8.cpu().numpy()
    np.testing.assert_array_equal(img[0], cv2.resize(raw, (416, 416)))
    del eng
    r3 = _case(1, 416, tame, 'bf16x3', score_thresh=0.1, images=img)
    r1 = _case(1, 416, tame, 'bf16', score_thresh=0.1, images=img)
    _dump_report()
    assert r3['net_rel_l2'] < 3e-4, r3
    assert r3['score_rel_max'] < 1e-3 and r3['box_rel_max'] < 1e-3 and r3['unexplained_list_differences'] == 0, r3
    assert r1['net_rel_l2'] < 8e-2, r1
