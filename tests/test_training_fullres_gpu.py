"""The training step at the sizes it is run at -- 416x416 batch 64 (reference loss, 45 channels: what `bench.py --mode train`
times) and 608x608 batch 32 (region loss, 125 channels) -- checked layer by layer against float64.

At these sizes the backward pass runs kernels and configurations the small-map tests never reach: the halo-patch CTA pair
with 32 output channels, the input-stationary kernel and stream-K with no scale and no shift (the data gradient), split-K
weight gradients over millions of pixels, batch statistics over 11 M rows.  One eager step is recorded per configuration:
every layer's input, pre-BN rows, statistics, activation, incoming gradient, dh, dW / dgamma / dbeta and data gradient.
Each stage is then checked on ITS OWN recorded inputs against a float64 reference computed with torch on the GPU, so that
errors do not compound and a failure names one kernel (test ids read `416-L14-dgrad`).

Element bound, fixed before any run:  |got - ref| <= ulp_out(ref) / 2 + TAU * absref
  ulp_out  spacing of the output format at ref (bf16 for activations, dh, dx; zero for float32 outputs)
  absref   the same operation on absolute values (|x| conv |w|, ...): what a float32 accumulation error is relative to
plus a rel-L2 bound per tensor.

Half of each batch is the two golden photos letterboxed with constant gray bars, the rest random images with a constant
rectangle: constant regions give bit-identical pre-BN values, i.e. exact ties in the 2x2 max-pool windows, whose gradient
must go to the first maximum of the window."""
import os

import numpy as np
import pytest
import torch

from oracle import yolo2_oracle as O
from tests.helpers import make_store

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
TAU = 1e-5
# conv_wgrad_tc_kernel: one float32 accumulator in tensor memory takes a whole K range -- on the 13x13 and 19x19 layers all
# N*H*W pixels (64 * 169 = 10816: 676 MMAs of K = 16), each step rounding relative to a partial sum bounded by absref, so
# the worst case is 676 * 2^-24 = 4e-5 of absref (twice that if the accumulation truncates): 1e-4.
TAU_WGRAD = 1e-4
REL_L2_BF16 = 2.0 ** -8          # twice the worst relative rounding error of a bf16 output
REL_L2_ELEM = 0.25               # float32 outputs: RMS error <= a quarter of the RMS element bound
CONFIGS = {416: dict(IS=416, N=64, loss='v1', OF=45), 608: dict(IS=608, N=32, loss='region', OF=125)}
NUM_LAYERS = 22
STAGES = ('conv', 'stats', 'act', 'bnbwd', 'wgrad', 'dgrad')
TIED_LAYERS = (0, 1, 4)          # pooled layers that must see >= 1000 exactly tied windows
MIN_TIED = 1000
# Share of windows whose top candidates are within the float32 error of the affine.  Inside constant image regions the rows of
# a window are the same exact sum; on stream-K layers (maps < 64x64 with Cout % 256 == 0) a tile shared by two CTA pairs
# rounds it in another order than its neighbours, which leaves such windows a few ulps apart: 0.26 % at 416x416 layer 8,
# 0.12 % at 608x608 layer 13, <= 0.02 % on every other pooled layer.
MAX_AMBIGUOUS = 5e-3

# Kernel families the backward pass of a layer must reach (1-based layer -> regexes over the profiler's kernel names).
# If a dispatch heuristic moves a layer off one of these, the test below fails and this table is updated on purpose.
HALO_PAIR = r'conv_tc_kernel<\d+, 2, \d+, true, (true|false)>'
HALO_PAIR_TMA_STORE = r'conv_tc_kernel<\d+, 2, \d+, true, true>'
IM2COL_PAIR = r'conv_tc_kernel<\d+, 0, \d+, true, (true|false)>'
INPUT_STATIONARY = r'conv_is_kernel<'
STREAMK = r'conv_streamk2_kernel<'
WGRAD_TC = r'conv_wgrad_tc_kernel<'
WGRAD_C3 = r'conv_wgrad_c3_mma_kernel'
BN_BWD_POOL_ROWS = r'bn_bwd_apply_rows_kernel<true>'
BN_STATS_8ROW = r'bn_stats_partial_v4_kernel<\d+, 8>'
_COMMON = {1: [WGRAD_C3, BN_BWD_POOL_ROWS], 2: [HALO_PAIR, WGRAD_TC, BN_BWD_POOL_ROWS], 3: [INPUT_STATIONARY, WGRAD_TC],
           4: [HALO_PAIR_TMA_STORE], 5: [INPUT_STATIONARY, BN_BWD_POOL_ROWS], 9: [STREAMK], 11: [STREAMK], 13: [STREAMK],
           14: [STREAMK], 16: [STREAMK], 18: [STREAMK], 19: [STREAMK], 20: [STREAMK], 21: [STREAMK], 22: [IM2COL_PAIR]}
EXPECTED_BWD = {416: dict(_COMMON), 608: {**_COMMON, 6: [HALO_PAIR], 7: [IM2COL_PAIR], 8: [HALO_PAIR, BN_BWD_POOL_ROWS]}}
EXPECTED_FWD = {416: [BN_STATS_8ROW], 608: [BN_STATS_8ROW]}


# ---- inputs ------------------------------------------------------------------------------------------------------------
def _images(IS, N, seed):
    """uint8 BGR [N,IS,IS,3]: the first half letterboxed golden photos (constant gray bars), the rest random noise with a
    constant-colour rectangle of at least 160 x 160."""
    import cv2
    rs = np.random.RandomState(seed)
    photos = [cv2.imread(os.path.join(GOLDEN, f)) for f in ('testImg1.jpg', 'testImg2.jpg')]
    out = np.empty((N, IS, IS, 3), dtype=np.uint8)
    for i in range(N):
        if i < N // 2:
            im = photos[i % 2]
            h, w = im.shape[:2]
            s = IS / max(h, w) * rs.uniform(0.7, 1.0)
            nh, nw = int(h * s), int(w * s)
            img = np.full((IS, IS, 3), (114, 128)[rs.randint(2)], dtype=np.uint8)
            y0, x0 = rs.randint(0, IS - nh + 1), rs.randint(0, IS - nw + 1)
            img[y0:y0 + nh, x0:x0 + nw] = cv2.resize(im, (nw, nh))
            if rs.rand() < 0.5:
                img = img[:, ::-1]
        else:
            img = rs.randint(0, 256, (IS, IS, 3)).astype(np.uint8)
            hh, ww = rs.randint(160, IS // 2 + 1, 2)
            y0, x0 = rs.randint(0, IS - hh + 1), rs.randint(0, IS - ww + 1)
            img[y0:y0 + hh, x0:x0 + ww] = rs.randint(0, 256, 3)
        out[i] = img
    return out


def _labels_v1(rs, N, S, IS, C=20):
    lab = np.zeros((N, S, S, 5 + C), dtype=np.float32)
    for n in range(N):
        for _ in range(rs.randint(1, 4)):
            cx, cy = rs.uniform(0, IS, 2)
            w, h = rs.uniform(20, IS * 0.7, 2)
            j, i = int(cx * S / IS), int(cy * S / IS)
            if lab[n, i, j, 0] == 1:
                continue
            lab[n, i, j, 0] = 1
            lab[n, i, j, 1:5] = [cx, cy, w, h]
            lab[n, i, j, 5 + rs.randint(0, C)] = 1
    return lab


def _random_gt(rs, N, G, S):
    counts = rs.randint(0, min(G, 6) + 1, N).astype(np.int32)
    boxes = np.zeros((N, G, 4), dtype=np.float32)
    classes = np.zeros((N, G), dtype=np.int32)
    for n in range(N):
        for g in range(counts[n]):
            boxes[n, g] = [rs.uniform(0.02, 0.98), rs.uniform(0.02, 0.98), rs.uniform(0.05, 0.7), rs.uniform(0.05, 0.7)]
            classes[n, g] = rs.randint(0, 20)
        if counts[n] >= 2:          # two ground truths in the same cell with similar shapes: slot collision
            boxes[n, 1] = boxes[n, 0] + np.array([0.001, 0.001, 0.01, 0.01], dtype=np.float32)
    return boxes, classes, counts


def _trainer(cfg, use_cuda_graph=False):
    from tensorflow_yolo2_b200.trainer import Yolo2Trainer
    c = CONFIGS[cfg]
    st, _ = make_store(c['OF'], tame=True)
    return Yolo2Trainer(c['N'], c['IS'], c['OF'], store=st, loss=c['loss'], device='cuda:0', use_cuda_graph=use_cuda_graph)


def _set_targets(tr, targets):
    if tr.loss_kind == 'v1':
        tr.set_labels(targets)
    else:
        tr.set_ground_truth(*targets)


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sorted({e.key for e in prof.key_averages()})


# ---- the recorded step ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module', params=list(CONFIGS), ids=[str(c) for c in CONFIGS])
def rec(request):
    """One eager training step of configuration request.param, recorded layer by layer (see the module docstring); the
    forward pass and every layer's backward run under the profiler, so the kernel names are recorded too.  The trainer is
    freed before the tests run."""
    from tensorflow_yolo2_b200 import ops
    cfg = request.param
    c = CONFIGS[cfg]
    N, IS = c['N'], c['IS']
    S = IS // 32
    rs = np.random.RandomState(cfg)
    images = _images(IS, N, cfg)
    targets = _labels_v1(rs, N, S, IS) if c['loss'] == 'v1' else _random_gt(rs, N, 32, S)
    tr = _trainer(cfg)
    _set_targets(tr, targets)
    tr.in_u8.copy_(torch.as_tensor(images))
    nl = len(tr.layers)
    assert nl == NUM_LAYERS
    R = dict(cfg=cfg, N=N, images=images, targets=targets, layers=tr.layers, geom=tr.geom, x0=tr.x0, acts=tr.acts,
             raw=tr.raw, stats=tr.stats, kernels_bwd={}, dy={}, dh={}, dx={}, grads={})
    R['params'] = [{k: v.clone() for k, v in tr.P[li].items()} for li in range(nl)]
    R['moving_before'] = [(tr.store[L['bn']['moving_mean']].clone(), tr.store[L['bn']['moving_variance']].clone())
                          for L in tr.layers]
    tr.iteration += 1
    tr._set_lr()
    with ops.conv_workspace_scope(tr.conv_ws):
        R['kernels_fwd'] = _kernel_names(tr.forward)
        tr.loss()
        # what backward() does, one layer at a time (at world size 1 the reducer calls are no-ops)
        for li in reversed(range(nl)):
            R['dy'][li] = tr._dy_of(li).clone()
            R['kernels_bwd'][li] = _kernel_names(lambda: tr._backward_layer(li))
            g = tr.geom[li]
            R['dh'][li] = tr.dh[:g['M'] * g['ld_dh']].view(g['M'], g['ld_dh']).clone()
            if li > 0:
                R['dx'][li] = tr.dx[li & 1][:g['M'] * tr.layers[li]['cin']].clone()
            R['grads'][li] = {k: v.clone() for k, v in tr.G[li].items()}
        tr.update(_lr_set=True, zero_grad=False)
    torch.cuda.synchronize()
    R['terms'] = tr.terms.clone()
    R['params_after'] = tr.params.clone()
    R['moving_after'] = [(tr.store[L['bn']['moving_mean']].clone(), tr.store[L['bn']['moving_variance']].clone())
                         for L in tr.layers]
    del tr
    torch.cuda.empty_cache()
    yield R
    R.clear()
    torch.cuda.empty_cache()


# ---- float64 references and the element check ----------------------------------------------------------------------------
def _ulp(x, bits):
    """Spacing of a float format with `bits` significant bits at |x| (0 at x == 0)."""
    _, e = torch.frexp(x)
    return torch.where(x == 0, torch.zeros_like(x), torch.ldexp(torch.ones_like(x), e - bits))


def _rel_l2(got, ref):
    return float(torch.linalg.vector_norm(got.double() - ref) / torch.linalg.vector_norm(ref).clamp_min(1e-300))


def _check(tag, got, ref, absref, bf16_out, tau=TAU):
    """Every element within ulp_out(ref)/2 + tau * absref; rel-L2 within 2^-8 for bf16 outputs, and for float32 outputs
    within a quarter of the element bound's own rel-L2 (float32 results carry cancellation: |ref| << absref)."""
    got, ref = got.double(), ref.double()
    bound = tau * absref.double()
    if bf16_out:
        bound = bound + 0.5 * _ulp(ref, 8)
    err = (got - ref).abs()
    bad = err > bound
    worst = float((err / bound.clamp_min(1e-300)).max())
    rl = _rel_l2(got, ref)
    print('%-18s max err / bound %.3f   rel-L2 %.3g' % (tag, worst, rl))
    nbad = int(bad.sum())
    if nbad:
        i = int(torch.argmax((err - bound).flatten()))
        raise AssertionError('%s: %d of %d elements out of bound; worst at flat index %d (of shape %s): got %.9g ref %.9g '
                             'absref %.4g' % (tag, nbad, got.numel(), i, tuple(got.shape), float(got.flatten()[i]),
                                              float(ref.flatten()[i]), float(absref.flatten()[i])))
    limit = REL_L2_BF16 if bf16_out else REL_L2_ELEM * _rel_l2(ref + bound, ref)
    assert rl <= limit, '%s: rel-L2 %.3g > %.3g' % (tag, rl, limit)


def _nchw(t):
    return t.permute(0, 3, 1, 2).contiguous()


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


def _layer_input(R, li):
    return R['x0'][..., :3] if li == 0 else R['acts'][li - 1]


def _w_bf16(R, li):
    return R['params'][li]['W'].to(torch.bfloat16)


def _conv(x, w, dtype):
    """SAME stride-1 cross-correlation, NHWC x HWIO -> NHWC."""
    return O.conv2d_same(x.to(dtype), w.to(dtype), dtype)


def _stage_conv(R, li):
    L, g = R['layers'][li], R['geom'][li]
    cout = L['cout']
    x, w, b = _layer_input(R, li), _w_bf16(R, li), R['params'][li]['b']
    ref = (_conv(x, w, torch.float64) + b.double()).reshape(-1, cout)
    absref = (_conv(x.abs(), w.abs(), torch.float32) + b.abs()).reshape(-1, cout)       # (a magnitude: float32 is plenty)
    raw = R['raw'][li]
    assert raw.shape == (g['M'], g['ldh'])
    assert torch.all(raw[:, cout:] == 0), 'padding columns %d..%d of the pre-BN rows must be 0' % (cout, g['ldh'])
    _check('conv+bias', raw[:, :cout], ref, absref, bf16_out=False)


def _stage_stats(R, li):
    L, s = R['layers'][li], R['stats'][li]
    C = L['cout']
    h = R['raw'][li][:, :C].double()
    mean = h.mean(dim=0)
    var = ((h - mean) ** 2).mean(dim=0)
    std = var.sqrt()
    em = ((s['mean'].double() - mean).abs() / (mean.abs() + std)).max()
    ev = ((s['var'].double() - var).abs() / var).max()
    print('mean err / (|mean| + std) %.3g   var rel err %.3g' % (em, ev))
    assert em <= 1e-6 and ev <= 1e-5, (float(em), float(ev))
    # the folded affine the activation pass uses: scale = gamma * rsqrt(var + eps), shift = beta (centred form)
    p = R['params'][li]
    want_scale = p['gamma'].double() / (s['var'].double() + O.BN_EPS).sqrt()
    es = ((s['scale'].double() - want_scale).abs() / want_scale.abs()).max()
    print('scale rel err %.3g' % es)
    assert es <= 1e-6 and torch.equal(s['shift'], p['beta'])
    # UPDATE_OPS: moving = moving * 0.99 + batch * 0.01
    for (m0, m1), bv in zip(zip(R['moving_before'][li], R['moving_after'][li]), (s['mean'], s['var'])):
        want = m0.double() * O.BN_MOMENTUM + bv.double() * (1 - O.BN_MOMENTUM)
        assert torch.all((m1.double() - want).abs() <= 1e-6 * (m0.double().abs() + bv.double().abs()))


def _pool_max(t, N, H):
    C = t.shape[-1]
    return t.reshape(N, H // 2, 2, H // 2, 2, C).amax(dim=(2, 4))


def _stage_act(R, li):
    L, g, s = R['layers'][li], R['geom'][li], R['stats'][li]
    N, H, C = R['N'], g['H'], L['cout']
    h = R['raw'][li][:, :C].double().reshape(N, H, H, C)
    d = h - s['mean'].double()
    z = d * s['scale'].double() + s['shift'].double()
    ref = torch.where(z > 0, z, O.ALPHA * z)
    absref = d.abs() * s['scale'].double().abs() + s['shift'].double().abs()
    if L['pool']:
        ref, absref = O.max_pool_2x2(ref), _pool_max(absref, N, H)
    last = li == NUM_LAYERS - 1
    got = R['acts'][li]
    assert got.dtype == (torch.float32 if last else torch.bfloat16)
    _check('affine+leaky' + ('+pool' if L['pool'] else ''), got, ref, absref, bf16_out=not last)


def _windows(t, N, H, pool):
    """[M, C] rows of an NHWC map -> [units, positions, C]: 2x2 windows in the order (0,0), (0,1), (1,0), (1,1)."""
    C = t.shape[-1]
    if not pool:
        return t.reshape(-1, 1, C)
    return t.reshape(N, H // 2, 2, H // 2, 2, C).permute(0, 1, 3, 2, 4, 5).reshape(-1, 4, C)


def _stage_bnbwd(R, li):
    """Pooled batch-norm backward.  Routing: the first maximum of the window's pre-BN rows in window order (the arg-max for
    gamma > 0, the arg-min for gamma < 0).  The kernel decides on its float32 recomputation of the affine + leaky, so where
    the top candidates are within 4 float32 ulps of the affine's terms (|xhat * gamma| + |beta|) it may pick any of them --
    such a window is 'ambiguous' and either routing is accepted; likewise the leaky slope where |z| is within that error."""
    L, g, s = R['layers'][li], R['geom'][li], R['stats'][li]
    N, H, C, M = R['N'], g['H'], L['cout'], g['M']
    pool = L['pool']
    p = R['params'][li]
    gamma, beta = p['gamma'].double(), p['beta'].double()
    mean, var = s['mean'].double(), s['var'].double()
    inv = (var + O.BN_EPS).rsqrt()
    hw = _windows(R['raw'][li][:, :C].double(), N, H, pool)                  # [U, P, C]
    dy = R['dy'][li].double().reshape(-1, C)                                 # [U, C]
    U, P = hw.shape[0], hw.shape[1]
    xh = (hw - mean) * inv
    z = xh * gamma + beta
    a = torch.where(z > 0, z, O.ALPHA * z)
    slope = torch.where(z > 0, torch.ones_like(z), torch.full_like(z, O.ALPHA))
    err_aff = 4 * _ulp((xh * gamma).abs() + beta.abs(), 24)                 # float32 error scale of the recomputed affine
    pos = torch.arange(P, device=hw.device).view(1, P, 1)
    key = hw * torch.sign(gamma)
    first = torch.where(key == key.amax(dim=1, keepdim=True), pos, P).amin(dim=1)          # [U, C]
    h_first = hw.gather(1, first[:, None]).squeeze(1)
    a_top = a.amax(dim=1, keepdim=True)
    cand = a >= a_top - err_aff.amax(dim=1, keepdim=True)                   # positions the kernel may legitimately pick
    ambiguous = (cand & (hw != h_first[:, None])).any(dim=1)
    z_amb = z.abs() <= err_aff                                              # leaky slope undecided in float32
    tied = (hw == h_first[:, None]).sum(dim=1) >= 2
    n_tied, n_amb = int(tied.sum()), int(ambiguous.sum())
    print('windows %d  exactly tied %d  ambiguous %d' % (U * C, n_tied, n_amb))
    if pool:
        assert n_amb <= MAX_AMBIGUOUS * U * C, 'ambiguous windows %d of %d' % (n_amb, U * C)
        if li in TIED_LAYERS:
            assert n_tied >= MIN_TIED, 'layer %d: only %d exactly tied windows' % (li + 1, n_tied)

    # dbeta = sum dz, dgamma = sum dz * xhat over the routed entries
    take = lambda t: t.gather(1, first[:, None]).squeeze(1)
    dz = dy * take(slope)
    xr = take(xh)
    dbeta_ref, dgamma_ref = dz.sum(0), (dz * xr).sum(0)
    # what an ambiguous window or an undecided slope may change
    spread = torch.where(ambiguous, xh.masked_fill(~cand, -np.inf).amax(1) - xh.masked_fill(~cand, np.inf).amin(1), 0.0)
    slope_amb = (cand & z_amb).any(dim=1)
    slack_b = torch.where(slope_amb, (1 - O.ALPHA) * dy.abs(), 0.0).sum(0)
    slack_g = (dz.abs() * spread).sum(0) + torch.where(slope_amb, (1 - O.ALPHA) * dy.abs() * xh.abs().amax(1), 0.0).sum(0)
    gr = R['grads'][li]
    for nm, got, ref, tol in (('dbeta', gr['beta'], dbeta_ref, TAU * dz.abs().sum(0) + slack_b),
                              ('dgamma', gr['gamma'], dgamma_ref, TAU * (dz * xr).abs().sum(0) + slack_g)):
        e = (got.double() - ref).abs()
        rl = _rel_l2(got, ref)
        print('%-18s max err / bound %.3f   rel-L2 %.3g' % (nm, float((e / tol).max()), rl))
        assert torch.all(e <= tol), '%s: %d of %d channels out of bound' % (nm, int((e > tol).sum()), C)
        limit = REL_L2_ELEM * _rel_l2(ref + tol, ref)
        assert rl <= limit, '%s: rel-L2 %.3g > %.3g' % (nm, rl, limit)

    # dh = gamma * inv * (dz at the routed entry - dbeta / M - xhat * dgamma / M), from the recorded dgamma / dbeta
    dh_all = R['dh'][li]
    assert torch.all(dh_all[:, C:] == 0), 'padding columns %d..%d of dh must be 0' % (C, g['ld_dh'])
    got = _windows(dh_all[:, :C].double(), N, H, pool)
    gi = gamma * inv
    m1, m2 = gr['beta'].double() / M, gr['gamma'].double() / M
    base = gi * (-m1 - xh * m2)
    abs_base = gi.abs() * (m1.abs() + (xh * m2).abs())

    def ok(gv, ref, absref):
        return (gv - ref).abs() <= 0.5 * _ulp(ref, 8) + TAU * absref

    ok_base = ok(got, base, abs_base)                                       # [U, P, C]: entry not routed
    route_ok = []                                                           # [U, C] per routing choice r
    for r in range(P):
        d_r = dy * slope[:, r]
        ok_r = ok(got[:, r], base[:, r] + gi * d_r, abs_base[:, r] + (gi * d_r).abs())
        alt = dy * (1.0 + O.ALPHA - slope[:, r])                            # the other leaky slope
        ok_r |= z_amb[:, r] & ok(got[:, r], base[:, r] + gi * alt, abs_base[:, r] + (gi * alt).abs())
        others = torch.cat([ok_base[:, :r], ok_base[:, r + 1:]], dim=1).all(dim=1) if P > 1 else torch.ones_like(ok_r)
        route_ok.append(ok_r & others)
    route_ok = torch.stack(route_ok, dim=1)                                 # [U, P, C]
    passed = route_ok.gather(1, first[:, None]).squeeze(1) | (ambiguous & (route_ok & cand).any(dim=1))
    nbad = int((~passed).sum())
    ref_first = base.clone()
    ref_first.scatter_add_(1, first[:, None], (gi * dz)[:, None])
    abs_first = abs_base.clone()
    abs_first.scatter_add_(1, first[:, None], (gi * dz).abs()[:, None])
    sel = ~ambiguous[:, None, :].expand_as(got)
    ratio = ((got - ref_first).abs() / (0.5 * _ulp(ref_first, 8) + TAU * abs_first).clamp_min(1e-300))[sel]
    rl = _rel_l2(got[sel], ref_first[sel])
    print('%-18s max err / bound %.3f   rel-L2 %.3g (unambiguous windows)' % ('dh', float(ratio.max()), rl))
    if nbad:
        bad = ~passed
        last_tied = torch.where(hw == h_first[:, None], pos, -1).amax(dim=1)
        later = int((bad & tied & route_ok.gather(1, last_tied[:, None]).squeeze(1)).sum())
        raise AssertionError('dh: %d of %d windows match no admissible routing (%d of them exactly tied; %d routed to the '
                             'LAST tied maximum instead of the first)' % (nbad, U * C, int((bad & tied).sum()), later))
    assert rl <= REL_L2_BF16, 'dh: rel-L2 %.3g' % rl


def _stage_wgrad(R, li):
    L = R['layers'][li]
    k, cin, cout = L['k'], L['cin'], L['cout']
    x = _nchw(_layer_input(R, li))
    dh = _nchw(R['dh'][li][:, :cout].reshape(R['N'], R['geom'][li]['H'], R['geom'][li]['H'], cout))
    wshape = (cout, cin, k, k)
    ref = torch.nn.grad.conv2d_weight(x.double(), wshape, dh.double(), padding=k // 2).permute(2, 3, 1, 0)
    absref = torch.nn.grad.conv2d_weight(x.float().abs(), wshape, dh.float().abs(), padding=k // 2).permute(2, 3, 1, 0)
    gr = R['grads'][li]
    _check('wgrad', gr['W'], ref, absref, bf16_out=False, tau=TAU_WGRAD)
    assert float(gr['b'].abs().max()) == 0.0                 # bias in front of batch-statistics BN: gradient exactly 0


def _stage_dgrad(R, li):
    L, g = R['layers'][li], R['geom'][li]
    k, cin, cout = L['k'], L['cin'], L['cout']
    N, H = R['N'], g['H']
    dh = _nchw(R['dh'][li][:, :cout].reshape(N, H, H, cout))
    w = _w_bf16(R, li).permute(3, 2, 0, 1)                  # HWIO -> OIHW
    ref = _nhwc(torch.nn.grad.conv2d_input((N, cin, H, H), w.double(), dh.double(), padding=k // 2))
    absref = _nhwc(torch.nn.grad.conv2d_input((N, cin, H, H), w.float().abs(), dh.float().abs(), padding=k // 2))
    got = R['dx'][li].view(N, H, H, cin)
    _check('dgrad', got, ref, absref, bf16_out=True)


_STAGE_FN = dict(conv=_stage_conv, stats=_stage_stats, act=_stage_act, bnbwd=_stage_bnbwd, wgrad=_stage_wgrad,
                 dgrad=_stage_dgrad)
_CASES = [pytest.param(li, st, id='L%d-%s' % (li + 1, st))
          for li in range(NUM_LAYERS) for st in STAGES if not (st == 'dgrad' and li == 0)]


@pytest.mark.parametrize('li,stage', _CASES)
def test_stage_vs_float64(rec, li, stage):
    print('\n%d-L%d-%s' % (rec['cfg'], li + 1, stage))
    with torch.no_grad():
        _STAGE_FN[stage](rec, li)
    torch.cuda.empty_cache()


def test_dispatch_reaches_the_covered_kernels(rec):
    """The layers above are only covered where they run the kernels this file claims: the table EXPECTED_BWD."""
    import re
    cfg = rec['cfg']
    missing = []
    for pat in EXPECTED_FWD[cfg]:
        if not any(re.search(pat, n) for n in rec['kernels_fwd']):
            missing.append('forward: %s' % pat)
    for layer, pats in sorted(EXPECTED_BWD[cfg].items()):
        names = rec['kernels_bwd'][layer - 1]
        for pat in pats:
            if not any(re.search(pat, n) for n in names):
                missing.append('backward L%d: %s   (ran: %s)' % (layer, pat, [n[:90] for n in names if 'kernel' in n]))
    assert not missing, '\n'.join(missing)


@pytest.mark.parametrize('rec', [pytest.param(416, id='416')], indirect=True)
def test_graph_step_equals_eager(rec):
    """The same step as one CUDA graph: the forward pass is deterministic, so the loss terms and the BN moving statistics
    are bit-equal to the eager step's; the weights agree up to the float atomics of the weight gradient (the bound of
    test_training_step_cuda_graph_equals_eager)."""
    tr = _trainer(rec['cfg'], use_cuda_graph=True)
    _set_targets(tr, rec['targets'])
    tr.step(torch.as_tensor(rec['images']))
    torch.cuda.synchronize()
    assert tr.graph is not None and tr.iteration == 1
    assert torch.equal(tr.terms, rec['terms']), (tr.terms, rec['terms'])
    for L, (mm, mv) in zip(tr.layers, rec['moving_after']):
        assert torch.equal(tr.store[L['bn']['moving_mean']], mm) and torch.equal(tr.store[L['bn']['moving_variance']], mv)
    dp = (tr.params - rec['params_after']).abs()
    print('params |diff| mean %.3g max %.3g' % (float(dp.mean()), float(dp.max())))
    assert float(dp.mean()) < 3e-4 and float(dp.max()) < 1e-2
    del tr
    torch.cuda.empty_cache()
