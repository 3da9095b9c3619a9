"""The inference pass at the sizes bench.py times -- Yolo2Engine at 416x416 batch 64 and 608x608 batch 32, in bf16 and in
bf16x3 -- checked layer by layer against float64.

Inference runs kernel configurations that training never does: the fused uint8 first layer, BN folded into the conv
epilogue with leaky and the 2x2 pool (negative scales flip the pooled accumulators), the pooled tiled-box mode on the 26x26
/ 38x38 maps, the single-CTA halo kernel on 608's 76x76 map, stream-K with a fused bf16 or hi|lo epilogue, bf16x3 outputs
everywhere, and detection on a real network output at full batch.  One EAGER engine step is recorded per configuration:
the input, every layer's activation, the head's pre-BN rows and batch statistics, the folded BN, the packed weights, the
moving statistics before and after, the outputs and the kernel names.  Each layer is then checked on ITS OWN recorded input
against a float64 reference computed with torch on the GPU from exactly the operands the kernel multiplies, read back from
the engine's packed buffers (test ids read `608-x3-L13-act`).

Element bound, fixed before any run:  |got - ref| <= ulp_out(ref) / 2 + tau * absref
  ulp_out  bf16 outputs: the bf16 spacing at ref; float32 outputs: 0; hi|lo outputs: instead of ulp_out / 2 the
           representation error SPLIT_REPR * (|ref| + tau * absref) (tests/helpers.py derives |v - hi - lo| <= 2^-16 |v|)
  absref   the same operation on the absolute values of the operands (pooled outputs: the window maximum -- max is
           1-Lipschitz)
plus a rel-L2 bound per tensor.  In bf16x3 the reference is the three-product sum the kernel computes, hi w_hi + lo w_hi +
hi w_lo; that the output stays close to the full product x W is checked separately."""
import os
import re

import numpy as np
import pytest
import torch

from oracle import yolo2_oracle as O
from tests.helpers import REL_L2_ELEM, TAU, _check, _images, _rel_l2, make_store, split_hi_lo

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# bf16x3: K is three times longer ([hi | lo | hi] x [w_hi | w_hi | w_lo]), so three times the float32 accumulation steps of
# the bf16 convolution (up to 1728 MMAs of K = 16 on the head layers) -- three times its tau
TAU_X3 = 3 * TAU
# what the three-product sum leaves out of the full product x W: lo * w_lo (<= 2^-16 |x| |W|) and the representation error of
# W as w_hi + w_lo (<= 2^-16 |W|): 2^-15 of absref on top of the kernel's own bound
TAU_DROPPED = 2.0 ** -15
CONFIGS = [(416, 64, 'bf16'), (416, 64, 'bf16x3'), (608, 32, 'bf16'), (608, 32, 'bf16x3')]
IDS = ['416-bf16', '416-x3', '608-bf16', '608-x3']
NUM_LAYERS = 22
HEAD = (18, 19, 20, 21)
OF = 125
SCORE_THRESH, IOU_THRESH = 0.05, 0.45
BENCH_THRESH = 0.3               # bench.py's score threshold: fewer candidates, the fast NMS path
CAND_CAP = 64                    # DF_CAPK / DS_CAPK: candidates a class keeps in the fast path before the image falls back

# Kernels the step must run (regexes over the profiler's kernel names), from the launchers (conv_tcgen05.cu launch_conv /
# conv_is_try, conv_streamk_tcgen05.cu conv_streamk_try).  If a dispatch heuristic moves a layer off one of these, the
# dispatch test fails and this table is updated on purpose.
CONV1 = {'bf16': r'conv1_u8_pool_kernel<false>', 'bf16x3': r'conv1_u8_pool_kernel<true>'}
HALO_PAIR_C32_POOLED = r'conv_tc_kernel<64, 2, 1, true, false>'          # L2 bf16 (pooled epilogue)
HALO_PAIR_TMA_STORE_BF16 = r'conv_tc_kernel<128, 2, 2, true, true>'      # L3 bf16
HALO_PAIR_128 = r'conv_tc_kernel<128, 2, 2, true, false>'                # L5 pooled; L3 too in bf16x3
HALO_SINGLE = r'conv_tc_kernel<128, 2, 2, false, false>'                 # 608 L6, L8 pooled (two N tiles)
IM2COL_PAIR = r'conv_tc_kernel<128, 0, 2, true, false>'                  # L7, L22 (1x1)
TILED_BOX_POOLED = r'conv_tc_kernel<\d+, 1, 2, true, false>'             # L8 at 416, L13: pooled maps < 64x64
INPUT_STATIONARY = r'conv_is_kernel<2>'                                  # L4 (Cin 128)
INPUT_STATIONARY_C32 = r'conv_is_kernel<1>'                              # L2 in bf16x3: 3 * 32 >= 96, pooled
STREAMK = {'bf16': r'conv_streamk2_kernel<false>', 'bf16x3': r'conv_streamk2_kernel<true>'}
DETECT = r'detect_fused_kernel'                                          # batch < 128
HEAD_BN = [r'bn_stats_partial_v4_kernel<', r'bn_stats_final_kernel', r'affine_leaky']


def _expected(IS, prec):
    e = [CONV1[prec], HALO_PAIR_128, INPUT_STATIONARY, IM2COL_PAIR, TILED_BOX_POOLED, STREAMK[prec], DETECT] + HEAD_BN
    e += [HALO_PAIR_C32_POOLED, HALO_PAIR_TMA_STORE_BF16] if prec == 'bf16' else [INPUT_STATIONARY_C32]
    if IS == 608:
        e.append(HALO_SINGLE)
    return e


EXPECTED = {(IS, p): _expected(IS, p) for IS, _, p in CONFIGS}


def _profile_step(IS, N, prec):
    """Kernel names of one eager engine step of configuration (IS, N, prec), under the torch profiler."""
    from torch.profiler import ProfilerActivity, profile
    st, _ = make_store(OF, tame=True)
    eng = _engine(dict(IS=IS, N=N, prec=prec, store=st), use_cuda_graph=False)
    eng.in_u8.copy_(torch.as_tensor(_images(IS, N, IS)))
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        eng.run()
        torch.cuda.synchronize()
    return sorted({e.key for e in prof.key_averages()})


def _step_kernel_names(IS, N, prec):
    """_profile_step in a child process.  The profiler's CUDA activity tracing keeps state across sessions: run in the test
    process, after this file's engine steps and CUDA graphs, later sessions lost kernel launches -- the first layers' here,
    and every launch of test_training_fullres_gpu.py's per-layer sessions when the two files ran in one process."""
    import json
    import subprocess
    import sys
    code = ('import json, sys; sys.path.insert(0, %r); from tests.test_inference_fullres_gpu import _profile_step; '
            'print(json.dumps(_profile_step(%d, %d, %r)))' % (ROOT, IS, N, prec))
    flags = ['-s'] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable] + flags + ['-c', code], cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, 'profiling child failed:\n%s' % r.stderr[-4000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def _engine(R, use_cuda_graph):
    from tensorflow_yolo2_b200.engine import Yolo2Engine
    return Yolo2Engine(R['N'], R['IS'], OF, store=R['store'], use_cuda_graph=use_cuda_graph, precision=R['prec'],
                       score_thresh=SCORE_THRESH, iou_thresh=IOU_THRESH, device='cuda:0')


def _outputs(eng):
    return dict(net=eng.acts[-1], boxes=eng.boxes, scores=eng.scores, keep_idx=eng.keep_idx, keep_count=eng.keep_count)


# ---- the recorded step ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module', params=CONFIGS, ids=IDS)
def rec(request):
    """One eager engine step of configuration request.param, recorded (see the module docstring); its kernel names come
    from the same step profiled in a child process.  The engine is freed before the tests run."""
    IS, N, prec = request.param
    kernels = _step_kernel_names(IS, N, prec)
    st, _ = make_store(OF, tame=True)
    R = dict(IS=IS, N=N, prec=prec, x3=prec == 'bf16x3', tag='%d-%s' % (IS, 'x3' if prec == 'bf16x3' else 'bf16'),
             images=_images(IS, N, IS), store=st)
    eng = _engine(R, use_cuda_graph=False)
    assert len(eng.layers) == NUM_LAYERS and eng.fused_conv1 and not eng.core_training and eng.head_training
    g = lambda name: st[name].detach().clone()
    R['kernels'] = kernels
    R['layers'] = eng.layers
    R['detect_impl'] = eng.detect_impl
    R['params'] = [dict(W=g(L['W']), b=g(L['b']), gamma=g(L['bn']['gamma']), beta=g(L['bn']['beta']),
                        mm=g(L['bn']['moving_mean']), mv=g(L['bn']['moving_variance'])) for L in eng.layers]
    eng.in_u8.copy_(torch.as_tensor(R['images']))
    eng.run()
    R['x_u8'] = eng.in_u8.clone()
    R['acts'] = [a.clone() for a in eng.acts]
    R['raw'] = {li: eng.raw[li].clone() for li in HEAD}
    R['stats'] = {li: dict(zip(('mean', 'var', 'scale', 'shift'), (t.clone() for t in eng.stats[li][:4]))) for li in HEAD}
    R['fold'] = {li: (s.clone(), h.clone()) for li, (s, h) in eng.fold.items()}
    R['packed'] = [p.clone() if p is not None else None for p in eng.packed]
    R['packed_c1'] = eng.packed_c1.clone()
    R['out'] = {k: (R['acts'][-1] if k == 'net' else v.clone()) for k, v in _outputs(eng).items()}
    R['moving_after'] = [(g(L['bn']['moving_mean']), g(L['bn']['moving_variance'])) for L in eng.layers]
    del eng
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    yield R
    R.clear()
    torch.cuda.empty_cache()


# ---- operands and float64 references -------------------------------------------------------------------------------------
def _bits_equal(tag, got, want):
    assert got.shape == want.shape and got.dtype == want.dtype == torch.bfloat16, (tag, got.shape, want.shape)
    diff = got.view(torch.int16) != want.view(torch.int16)
    assert not bool(diff.any()), '%s: %d of %d packed values differ from the restated packer' % (tag, int(diff.sum()),
                                                                                                diff.numel())


def _conv(x, w, dtype):
    """SAME stride-1 cross-correlation, NHWC x HWIO -> NHWC."""
    return O.conv2d_same(x.to(dtype), w.to(dtype), dtype)


def _leaky(z):
    return torch.where(z > 0, z, O.ALPHA * z)


def _pool_max(t):
    N, H, W, C = t.shape
    return t.reshape(N, H // 2, 2, W // 2, 2, C).amax(dim=(2, 4))


def _joined(t):
    """A hi | lo activation re-joined in float64 (exact)."""
    c = t.shape[-1] // 2
    return t[..., :c].double() + t[..., c:].double()


def _operands(R, li):
    """(x, w) that the conv of layer li >= 1 multiplies: x NHWC [N,H,W,K], w HWIO [k,k,K,cout], read back from the recorded
    input and the engine's packed weights, after asserting that those equal bf16(W) (bf16: [cout_p, k*k, cin]) or, per tap,
    [w_hi | w_hi | w_lo] (bf16x3: [cout_p, k*k, 3*cin]) bit for bit, zero padding rows included.  bf16x3: x = [hi | lo | hi],
    so x . w is the kernel's hi*w_hi + lo*w_hi + hi*w_lo.  Also returns W (float32 HWIO) for the full product."""
    L = R['layers'][li]
    k, cin, cout = L['k'], L['cin'], L['cout']
    cout_p = (cout + 15) // 16 * 16
    W = R['params'][li]['W']
    Wt = W.permute(3, 0, 1, 2).reshape(cout, k * k, cin)
    packed = R['packed'][li]
    a = R['acts'][li - 1]
    if not R['x3']:
        assert packed.numel() == cout_p * k * k * cin and a.shape[-1] == cin
        p = packed.view(cout_p, k * k, cin)
        _bits_equal('L%d packed' % (li + 1), p[:cout], Wt.to(torch.bfloat16))
        x = a
    else:
        assert packed.numel() == cout_p * k * k * 3 * cin and a.shape[-1] == 2 * cin
        p = packed.view(cout_p, k * k, 3, cin)
        hi, lo = split_hi_lo(Wt)
        for part, want in ((0, hi), (1, hi), (2, lo)):
            _bits_equal('L%d packed part %d' % (li + 1, part), p[:cout, :, part], want)
        p = p.reshape(cout_p, k * k, 3 * cin)
        x = torch.cat([a[..., :cin], a[..., cin:], a[..., :cin]], dim=-1)
    assert not bool((p[cout:].view(torch.int16) != 0).any()), 'L%d: packed padding rows must be 0' % (li + 1)
    w = p[:cout].reshape(cout, k, k, -1).permute(1, 2, 3, 0)
    return x, w, W


def _conv1_layout(taps):
    """The B operand of conv1_fused.cu from per-tap values taps [3,3,4,32] (kh, kw, channel, filter):
    [ty 4][k-group 2][n = window*32 + ch][8 = (tx_local 2) x (c 4)], value taps[ty-dy][tx-dx][c][ch] where the tap exists."""
    idx = torch.arange(4 * 2 * 128 * 8, device=taps.device)
    e, n, kg, ty = idx & 7, (idx >> 3) & 127, (idx >> 10) & 1, idx >> 11
    c, tx = e & 3, kg * 2 + (e >> 2)
    win, ch = n >> 5, n & 31
    kh, kw = ty - (win >> 1), tx - (win & 1)
    ok = (kh >= 0) & (kh < 3) & (kw >= 0) & (kw < 3)
    v = taps[kh.clamp(0, 2), kw.clamp(0, 2), c, ch]
    return torch.where(ok, v, torch.zeros_like(v))


def _conv1_operands(R):
    """Layer 1 (fused uint8 first layer): the packer restated in torch and checked bit for bit against the engine's buffer;
    returns (x, taps) that the kernel multiplies -- taps [3,3,4,32] float64 (bf16x3: hi + lo, exact), x NHWC with 4 channels:
    bf16: bf16(fma(v, 2/255, -1)) and a zero channel; bf16x3: the integer bytes v and a ones channel (0 in the SAME halo,
    which the zero padding of the reference conv reproduces)."""
    W, scale = R['params'][0]['W'], R['fold'][0][0]
    taps = torch.zeros((3, 3, 4, 32), dtype=torch.float64, device=W.device)
    u8 = R['x_u8']
    if not R['x3']:
        taps[:, :, :3] = (W * scale).to(torch.bfloat16).double()                    # float32 product, one rounding
        hi = taps.to(torch.bfloat16)
        _bits_equal('conv1 packed', R['packed_c1'], _conv1_layout(hi))
        kk = torch.tensor(2.0 / 255.0, dtype=torch.float32).double()
        lut = (torch.arange(256, dtype=torch.float64, device=W.device) * kk - 1.0).float().to(torch.bfloat16)  # = fmaf
        x = torch.cat([lut[u8.long()].double(), torch.zeros_like(u8[..., :1], dtype=torch.float64)], dim=-1)
    else:
        sc, wd = scale.double(), W.double()
        v = torch.empty((3, 3, 4, 32), dtype=torch.float64, device=W.device)
        v[:, :, :3] = sc * wd * (2.0 / 255.0)
        v[:, :, 3] = -sc * ((wd[:, :, 0] + wd[:, :, 1]) + wd[:, :, 2])
        hi = v.float().to(torch.bfloat16)
        lo = (v - hi.double()).float().to(torch.bfloat16)
        _bits_equal('conv1 packed hi', R['packed_c1'][:8192], _conv1_layout(hi))
        _bits_equal('conv1 packed lo', R['packed_c1'][8192:], _conv1_layout(lo))
        taps = hi.double() + lo.double()
        x = torch.cat([u8.double(), torch.ones_like(u8[..., :1], dtype=torch.float64)], dim=-1)
        return x, taps, (hi.double().abs() + lo.double().abs())
    return x, taps, taps.abs()


def _tau(R):
    return TAU_X3 if R['x3'] else TAU


def _check_out(R, tag, got, ref, absref, tau, f32_out=False):
    if f32_out:
        _check(tag, got, ref, absref, bf16_out=False, tau=tau)
    elif R['x3']:
        _check(tag, _joined(got), ref, absref, bf16_out=False, tau=tau, split_out=True)
    else:
        _check(tag, got, ref, absref, bf16_out=True, tau=tau)


def _check_full_product(R, tag, got, full, absref, tau):
    """bf16x3 only: the output against the full product, by rel-L2 -- within a quarter of the rel-L2 of the element bound
    widened by what the three products leave out."""
    g = got.double() if got.dtype == torch.float32 else _joined(got)
    bound = (tau + TAU_DROPPED) * absref.double() + 2.0 ** -16 * full.abs()
    rl, limit = _rel_l2(g, full), REL_L2_ELEM * _rel_l2(full + bound, full)
    print('%-18s rel-L2 vs full product %.3g (limit %.3g)' % (tag, rl, limit))
    assert rl <= limit, '%s: rel-L2 vs the full product %.3g > %.3g' % (tag, rl, limit)


# ---- stages ----------------------------------------------------------------------------------------------------------------
def _stage_act_core(R, li):
    """Core layers 1-18: leaky(conv * scale + shift), pooled where the layer pools, against acts[li]."""
    L = R['layers'][li]
    scale, shift = R['fold'][li]
    sc, sh = scale.double(), shift.double()
    if li == 0:
        x, w, wabs = _conv1_operands(R)
        acc = _conv(x, w, torch.float64)
        z = acc + sh                                        # the scale lives in the weights
        absref = _conv(x.abs().float(), wabs.float(), torch.float32).double() + sh.abs()
    else:
        x, w, _ = _operands(R, li)
        acc = _conv(x, w, torch.float64)
        z = acc * sc + sh
        absref = _conv(x.abs().float(), w.abs().float(), torch.float32).double() * sc.abs() + sh.abs()
        del x, w
    ref = _leaky(z)
    del acc, z
    if L['pool']:
        ref, absref = _pool_max(ref), _pool_max(absref)
    got = R['acts'][li]
    assert got.dtype == torch.bfloat16
    _check_out(R, 'bn+leaky' + ('+pool' if L['pool'] else ''), got, ref, absref, _tau(R))
    del ref
    if R['x3']:
        W = R['params'][li]['W']
        if li == 0:
            xf = R['x_u8'].double() * (2.0 / 255.0) - 1.0
            full = _conv(xf, W.double() * sc, torch.float64) + sh
        else:
            full = _conv(_joined(R['acts'][li - 1]), W.double(), torch.float64) * sc + sh
        full = _leaky(full)
        if L['pool']:
            full = _pool_max(full)
        _check_full_product(R, 'full product', got, full, absref, _tau(R))


def _stage_conv_head(R, li):
    """Head layers 19-22: conv + bias as float32 rows (zero padding columns)."""
    L = R['layers'][li]
    cout = L['cout']
    x, w, W = _operands(R, li)
    b = R['params'][li]['b']
    ref = (_conv(x, w, torch.float64) + b.double()).reshape(-1, cout)
    absref = (_conv(x.abs().float(), w.abs().float(), torch.float32) + b.abs()).reshape(-1, cout)
    raw = R['raw'][li]
    ld = (cout + 31) // 32 * 32
    assert raw.shape == (ref.shape[0], ld)
    assert torch.all(raw[:, cout:] == 0), 'padding columns %d..%d of the pre-BN rows must be 0' % (cout, ld)
    _check('conv+bias', raw[:, :cout], ref, absref, bf16_out=False, tau=_tau(R))
    if R['x3']:
        full = (_conv(_joined(R['acts'][li - 1]), W.double(), torch.float64) + b.double()).reshape(-1, cout)
        _check_full_product(R, 'full product', raw[:, :cout], full, absref, _tau(R))


def _stage_stats_head(R, li):
    """Batch statistics over the recorded rows (the training file's bounds); the store's moving statistics untouched."""
    C, s, p = R['layers'][li]['cout'], R['stats'][li], R['params'][li]
    h = R['raw'][li][:, :C].double()
    mean = h.mean(dim=0)
    var = ((h - mean) ** 2).mean(dim=0)
    em = ((s['mean'].double() - mean).abs() / (mean.abs() + var.sqrt())).max()
    ev = ((s['var'].double() - var).abs() / var).max()
    want_scale = p['gamma'].double() / (s['var'].double() + O.BN_EPS).sqrt()
    es = ((s['scale'].double() - want_scale).abs() / want_scale.abs()).max()
    print('mean err / (|mean| + std) %.3g   var rel err %.3g   scale rel err %.3g' % (em, ev, es))
    assert em <= 1e-6 and ev <= 1e-5 and es <= 1e-6, (float(em), float(ev), float(es))
    assert torch.equal(s['shift'], p['beta'])
    mm, mv = R['moving_after'][li]
    assert torch.equal(mm, p['mm']) and torch.equal(mv, p['mv']), 'inference must not update the moving statistics'


def _stage_act_head(R, li):
    """Head layers 19-22: leaky((h - mean) * scale + shift) -> bf16 / hi|lo (19-21), float32 (22)."""
    C, s = R['layers'][li]['cout'], R['stats'][li]
    N, S = R['N'], R['IS'] // 32
    h = R['raw'][li][:, :C].double()
    d = h - s['mean'].double()
    ref = _leaky(d * s['scale'].double() + s['shift'].double()).reshape(N, S, S, C)
    absref = (d.abs() * s['scale'].double().abs() + s['shift'].double().abs()).reshape(N, S, S, C)
    last = li == NUM_LAYERS - 1
    got = R['acts'][li]
    assert got.dtype == (torch.float32 if last else torch.bfloat16)
    _check_out(R, 'affine+leaky', got, ref, absref, TAU, f32_out=last)


_STAGE_FN = dict(act=_stage_act_core, conv=_stage_conv_head, stats=_stage_stats_head)
_CASES = [pytest.param(li, 'act', id='L%d-act' % (li + 1)) for li in range(18)] + \
         [pytest.param(li, st, id='L%d-%s' % (li + 1, st)) for li in HEAD for st in ('conv', 'stats', 'act')]


@pytest.mark.parametrize('li,stage', _CASES)
def test_stage_vs_float64(rec, li, stage):
    print('\n%s-L%d-%s' % (rec['tag'], li + 1, stage))
    with torch.no_grad():
        (_stage_act_head if stage == 'act' and li in HEAD else _STAGE_FN[stage])(rec, li)
    torch.cuda.empty_cache()


# ---- detection -------------------------------------------------------------------------------------------------------------
def _keep_lists_equal(a, b):
    """(keep_idx, keep_count) pairs equal in the counts and in every slot below the count."""
    ki_a, kc_a = a
    ki_b, kc_b = b
    if not torch.equal(kc_a, kc_b):
        return False
    slot = torch.arange(ki_a.shape[-1], device=ki_a.device)
    live = slot < kc_a[..., None]
    return torch.equal(torch.where(live, ki_a, -1), torch.where(live, ki_b, -1))


@pytest.mark.parametrize('thresh', [SCORE_THRESH, BENCH_THRESH], ids=['thr0.05', 'thr0.3'])
def test_detection_vs_oracle(rec, thresh):
    """Decode of the recorded network output against O.region_decode_v2 (1e-5; a score may cross the threshold only within
    1e-5 of it), keep lists bit-exact against O.nms_per_class on the kernel's own boxes and scores, and the other detection
    implementation bit-equal on the same output.  At 0.05 the engine's own outputs of the recorded step, where every image
    overflows some class's candidate list and takes the fallback NMS; at bench.py's 0.3 the engine's implementation run again
    on the recorded output, to reach the fast path too."""
    from tensorflow_yolo2_b200 import ops
    net, N = rec['out']['net'], rec['N']
    anchors = torch.as_tensor(O.VOC_ANCHORS).to(net.device)
    max_keep = rec['out']['keep_idx'].shape[-1]
    impl, other = ('detect_fused', 'detect_split') if rec['detect_impl'] == 'fused' else ('detect_split', 'detect_fused')
    keys = ('boxes', 'scores', 'keep_idx', 'keep_count')
    if thresh == SCORE_THRESH:
        out = rec['out']
    else:
        out = dict(zip(keys, getattr(ops, impl)(net, anchors, 20, thresh, IOU_THRESH, max_keep)[:4]))
        torch.cuda.synchronize()
    wb, wst, _ = O.region_decode_v2(net.cpu().numpy(), O.VOC_ANCHORS, 20, thresh)
    boxes, scores = out['boxes'].cpu().numpy(), out['scores'].cpu().numpy()
    eb = np.abs(boxes - wb) / np.maximum(np.abs(wb), 1e-300)
    print('\n%s thresh %g boxes: max rel err %.3g' % (rec['tag'], thresh, float(eb.max())))
    np.testing.assert_allclose(boxes, wb, rtol=1e-5, atol=1e-7)
    d = np.abs(scores - wst)
    close = d <= 1e-5 * np.abs(wst) + 1e-7
    near = np.abs(np.maximum(scores, wst) - thresh) < 1e-5
    print('scores: max rel err %.3g over kept scores, %d threshold flips within 1e-5' % (
        float((d / np.maximum(wst, 1e-30))[wst > 0].max()), int((~close & near).sum())))
    assert (close | near).all(), '%d scores out of bound' % int((~(close | near)).sum())
    ki, kc = out['keep_idx'].cpu().numpy(), out['keep_count'].cpu().numpy()
    total = 0
    for n in range(N):
        keeps = O.nms_per_class(boxes[n], scores[n], IOU_THRESH, thresh)
        for k in range(20):
            assert kc[n, k] == len(keeps[k]), (n, k, kc[n, k], len(keeps[k]))
            np.testing.assert_array_equal(ki[n, k, :kc[n, k]], keeps[k])
            total += len(keeps[k])
    cand = (scores > thresh).sum(axis=1)                                         # [N, C]
    print('detections %d; candidates per image %d..%d; images past the %d-candidate class lists (fallback NMS): %d of %d'
          % (total, int(cand.sum(1).min()), int(cand.sum(1).max()), CAND_CAP, int((cand > CAND_CAP).any(1).sum()), N))
    assert total > 0
    got = dict(zip(keys, getattr(ops, other)(net, anchors, 20, thresh, IOU_THRESH, max_keep)[:4]))
    torch.cuda.synchronize()
    assert torch.equal(got['boxes'], out['boxes']) and torch.equal(got['scores'], out['scores']), \
        '%s: boxes / scores differ' % other
    assert _keep_lists_equal((got['keep_idx'], got['keep_count']), (out['keep_idx'], out['keep_count'])), \
        '%s: keep lists differ' % other


# ---- dispatch, graph and pipelined paths -----------------------------------------------------------------------------------
def test_dispatch_reaches_the_covered_kernels(rec):
    """The layers above are only covered where they run the kernels this file claims: the table EXPECTED."""
    names = rec['kernels']
    missing = [pat for pat in EXPECTED[(rec['IS'], rec['prec'])] if not any(re.search(pat, n) for n in names)]
    assert not missing, 'missing %s; ran: %s' % (missing, [n[:90] for n in names if 'kernel' in n])


def _assert_outputs_equal(got, want, what):
    for k in ('net', 'boxes', 'scores', 'keep_idx', 'keep_count'):
        assert torch.equal(got[k], want[k]), '%s: %s differs from the eager step' % (what, k)


def test_graph_and_pipeline_equal_eager(rec):
    """run() with a CUDA graph -- what bench.py times -- gives the eager step's outputs bit for bit: the forward pass has no
    float atomics, and the detection kernels' atomics only order candidates before a sort.  At 416 bf16 also submit(),
    which captures one graph per staging slot (bench.py's e2e figure): two batches, one per slot."""
    eng = _engine(rec, use_cuda_graph=True)
    eng.infer(torch.as_tensor(rec['images']))
    torch.cuda.synchronize()
    assert eng.graph is not None
    _assert_outputs_equal(_outputs(eng), rec['out'], 'graph replay')
    if (rec['IS'], rec['prec']) == (416, 'bf16'):
        host = torch.as_tensor(rec['images']).pin_memory()
        outs = []
        for _ in range(2):
            o = {k: torch.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in rec['out'].items()}
            eng.submit(host, out_host=o)
            outs.append(o)
        eng.wait_outputs()
        torch.cuda.synchronize()
        assert len(eng._pipe_graphs) == 2
        want = {k: v.cpu() for k, v in rec['out'].items()}
        for i, o in enumerate(outs):
            _assert_outputs_equal(o, want, 'submit() slot %d' % i)
    del eng
    torch.cuda.empty_cache()
