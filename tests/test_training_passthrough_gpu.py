"""Training the YOLOv2 passthrough graph (Yolo2Trainer(passthrough=True)): the batch-norm backward's three dy read modes
(row stride, depth-to-space, un-pooled addend) against float64 autograd, one small step layer by layer and as a whole
against the oracle, the new backward stages of a full-size step against float64, the CUDA-graph step, convergence and the
checkpoint -> Yolo2Engine(passthrough=True) round trip.  The whole-chain reference is the oracle's training step restated
over the passthrough graph (train_step_reference below); the last test is its CPU check."""
import numpy as np
import pytest
import torch

from oracle import yolo2_oracle as O
from tests.helpers import TAU, _check, _images, make_store, oracle_params, rel_l2

TAU_WGRAD = 1e-4                 # as in test_training_fullres_gpu.py: one float32 accumulator over K = N*H*W pixels


@pytest.fixture(scope='module')
def ops():
    from tensorflow_yolo2_b200 import ops as _ops
    return _ops


def cu(a, dtype=None):
    t = torch.as_tensor(np.asarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda().contiguous()


def bf16r(a):
    return torch.as_tensor(np.asarray(a), dtype=torch.float32).to(torch.bfloat16).to(torch.float64).numpy()


def _d2s(v, C):
    """depth_to_space(2) of [N,h,w,4C] -> [N,2h,2w,C] (the inverse of O.space_to_depth2)."""
    n, h, w, _ = v.shape
    return v.reshape(n, h, w, 2, 2, C).permute(0, 1, 3, 2, 4, 5).reshape(n, 2 * h, 2 * w, C)


def _random_gt(rs, N, G):
    counts = rs.randint(1, min(G, 6) + 1, N).astype(np.int32)
    boxes = np.zeros((N, G, 4), dtype=np.float32)
    classes = np.zeros((N, G), dtype=np.int32)
    for n in range(N):
        for g in range(counts[n]):
            boxes[n, g] = [rs.uniform(0.02, 0.98), rs.uniform(0.02, 0.98), rs.uniform(0.05, 0.7), rs.uniform(0.05, 0.7)]
            classes[n, g] = rs.randint(0, 20)
    return boxes, classes, counts


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


def train_step_reference(x_nhwc, params_core, params_head, loss_fn, params_passthrough=None, bf16_operands=True,
                         dtype=torch.float64):
    """The oracle's train_step_reference (one training iteration up to the gradients: every layer with batch statistics,
    loss, torch autograd) over the YOLOv2 passthrough graph of O.darknet19_forward: a 1x1 conv_bn_layer on the un-pooled
    output of core layer O.PASSTHROUGH_LAYER, space_to_depth(2), concatenated after head conv2's channels.  Built from the
    oracle's own primitives.  Returns (loss, grads, stats, net) like O.train_step_reference, the passthrough conv's entries
    between conv2's and conv3's (the layer order of create_variables(..., passthrough=True)); params_passthrough=None is the
    reference's graph."""
    plist = list(params_core) + list(params_head)
    nc = len(params_core)
    ip = None
    if params_passthrough is not None:
        ip = nc + 2
        plist.insert(ip, params_passthrough)
    leaves = []
    for p in plist:
        q = {k: torch.as_tensor(np.asarray(v), dtype=dtype).clone() for k, v in p.items()}
        for k in ('W', 'b', 'gamma', 'beta'):
            q[k].requires_grad_(True)
        leaves.append(q)
    x = torch.as_tensor(np.asarray(x_nhwc), dtype=dtype)
    stats, pt_src = [], None
    for li, q in enumerate(leaves):
        if li == ip:
            pt, h, _ = O.conv_bn_layer(pt_src, q, True, dtype, bf16_operands)
            x = torch.cat([x, O.space_to_depth2(pt)], dim=-1)
        else:
            x, h, _ = O.conv_bn_layer(x, q, True, dtype, bf16_operands)
        stats.append((h.detach().mean(dim=(0, 1, 2)).numpy(), h.detach().var(dim=(0, 1, 2), unbiased=False).numpy()))
        if li == O.PASSTHROUGH_LAYER:
            pt_src = x
        if li < nc and O.CORE_PLAN[li][3]:
            x = O.max_pool_2x2(x)
    loss = loss_fn(x)
    loss.backward()
    grads = [{k: q[k].grad.numpy() for k in ('W', 'b', 'gamma', 'beta')} for q in leaves]
    return float(loss.detach()), grads, stats, x.detach().numpy()


def _trainer(N, IS, loss, **kw):
    from tensorflow_yolo2_b200.trainer import Yolo2Trainer
    OF = 125 if loss == 'region' else 30
    st, layers = make_store(OF, tame=True, passthrough=True)
    tr = Yolo2Trainer(N, IS, OF, store=st, loss=loss, B=2, device='cuda:0', passthrough=True, **kw)
    return st, layers, tr


# ---- 1. the dy read modes of the batch-norm backward ------------------------------------------------------------------------
# mode, N, H, C, pool, ldy, col: 'rows' reads columns [col, col + C) of rows of stride ldy, 's2d' the same through
# depth_to_space(2), 'add' a pooled layer with an un-pooled bf16 addend (windows with exactly tied maxima included)
BWD_CASES = [('rows', 2, 6, 1024, False, 1280, 0), ('rows', 2, 8, 64, True, 192, 64), ('rows', 2, 6, 30, False, 40, 3),
             ('s2d', 2, 8, 64, False, 1280, 1024), ('s2d', 1, 6, 30, False, 124, 2),
             ('add', 2, 8, 64, True, None, 0), ('add', 2, 12, 512, True, None, 0), ('add', 2, 8, 30, True, None, 0)]


@pytest.mark.gpu
@pytest.mark.parametrize('generic', [False, True], ids=['fast', 'generic'])
@pytest.mark.parametrize('dy_bf16', [True, False], ids=['dy_bf16', 'dy_f32'])
@pytest.mark.parametrize('mode,N,H,C,pool,ldy,col', BWD_CASES)
def test_bn_bwd_dy_modes_vs_autograd(ops, monkeypatch, mode, N, H, C, pool, ldy, col, dy_bf16, generic):
    if generic:
        monkeypatch.setenv('Y2_BN_BWD_GENERIC', '1')
        ops.reload_env()
    rs = np.random.RandomState(C + H + len(mode))
    ldh = (C + 31) // 32 * 32
    h = rs.randn(N, H, H, ldh).astype(np.float32) * 2 + 0.5
    h[:, 2:6, 2:6, :] = h[:, 2:3, 2:3, :]                   # a constant region: 2x2 windows with exactly tied maxima
    h = h.reshape(N * H * H, ldh)
    gamma = (rs.uniform(0.5, 1.5, C) * np.where(rs.rand(C) < 0.2, -1, 1)).astype(np.float32)
    beta = (rs.randn(C) * 0.3).astype(np.float32)
    Ho = H // 2 if pool else H
    rnd = (lambda a: bf16r(a).astype(np.float32)) if dy_bf16 else (lambda a: a.astype(np.float32))
    add = None
    if mode == 'add':
        wide = rnd(rs.randn(N, Ho, Ho, C))
        dy_dense = wide
        add = bf16r(rs.randn(N, H, H, C)).astype(np.float32)
    elif mode == 'rows':
        wide = rnd(rs.randn(N, Ho, Ho, ldy))
        dy_dense = wide[..., col:col + C]
    else:
        wide = rnd(rs.randn(N, H // 2, H // 2, ldy))
        dy_dense = _d2s(torch.tensor(wide[..., col:col + 4 * C]), C).numpy()
    # float64 autograd through batch_norm -> leaky (-> pool), plus the un-pooled consumer
    ht = torch.tensor(h[:, :C].reshape(N, H, H, C), dtype=torch.float64, requires_grad=True)
    gt_, bt = torch.tensor(gamma, dtype=torch.float64, requires_grad=True), torch.tensor(beta, dtype=torch.float64, requires_grad=True)
    z, _, _ = O.batch_norm(ht, gt_, bt, torch.zeros(C, dtype=torch.float64), torch.ones(C, dtype=torch.float64), True)
    y = torch.maximum(O.ALPHA * z, z)
    obj = ((O.max_pool_2x2(y) if pool else y) * torch.tensor(dy_dense, dtype=torch.float64)).sum()
    if add is not None:
        obj = obj + (y * torch.tensor(add, dtype=torch.float64)).sum()
    obj.backward()
    hd = cu(h)
    mean, var = ops.bn_stats(hd, C, ld=ldh)
    ld_dh = (C + 63) // 64 * 64
    dyt = cu(wide, torch.bfloat16 if dy_bf16 else torch.float32)
    dgamma, dbeta, dh = ops.bn_leaky_pool_bwd(hd, dyt, mean, var, cu(gamma), cu(beta), N, H, H, C, ldh=ldh, leaky=True,
                                              pool=pool, ld_dh=ld_dh, ldy=ldy, dy_col=col, dy_s2d=mode == 's2d',
                                              dy_add=None if add is None else cu(add, torch.bfloat16))
    torch.cuda.synchronize()
    assert rel_l2(dgamma.cpu().numpy(), gt_.grad.numpy()) < 1e-4
    assert rel_l2(dbeta.cpu().numpy(), bt.grad.numpy()) < 1e-4
    got = dh.float().cpu().numpy()
    assert np.all(got[:, C:] == 0), 'padding columns of dh must be zero'
    assert rel_l2(got[:, :C], ht.grad.numpy().reshape(-1, C)) < 6e-3


@pytest.mark.gpu
@pytest.mark.parametrize('generic', [False, True], ids=['fast', 'generic'])
@pytest.mark.parametrize('N,H,C,pool,dy_bf16', [(2, 8, 64, True, True), (3, 6, 125, False, False), (1, 4, 1024, False, True),
                                                 (2, 12, 32, True, False)])
def test_bn_bwd_ex_defaults_bit_identical(ops, monkeypatch, N, H, C, pool, dy_bf16, generic):
    """y2_bn_leaky_pool_bwd_ex with ldy = C, no depth-to-space and no addend gives y2_bn_leaky_pool_bwd's bits."""
    if generic:
        monkeypatch.setenv('Y2_BN_BWD_GENERIC', '1')
        ops.reload_env()
    rs = np.random.RandomState(C + H)
    ldh = (C + 31) // 32 * 32
    h = cu(rs.randn(N * H * H, ldh).astype(np.float32) * 2)
    Ho = H // 2 if pool else H
    dy = cu(rs.randn(N, Ho, Ho, C).astype(np.float32), torch.bfloat16 if dy_bf16 else torch.float32)
    mean, var = ops.bn_stats(h, C, ld=ldh)
    gamma, beta = cu(rs.uniform(-1.5, 1.5, C).astype(np.float32)), cu(rs.randn(C).astype(np.float32))
    outs = [ops.bn_leaky_pool_bwd(h, dy, mean, var, gamma, beta, N, H, H, C, ldh=ldh, pool=pool, ldy=ldy)
            for ldy in (None, C)]
    torch.cuda.synchronize()
    for a, b in zip(*outs):
        assert torch.equal(a.view(torch.int16) if a.dtype == torch.bfloat16 else a.view(torch.int32),
                           b.view(torch.int16) if b.dtype == torch.bfloat16 else b.view(torch.int32))


# ---- 2. one small step, layer-local and whole-chain ---------------------------------------------------------------------------
def _layer_input(tr, li):
    L = tr.layers[li]
    if li == 0:
        return tr.x0[..., :3]
    return tr.pt_src if L.get('role') == 'passthrough' else tr.acts[li - 1]


@pytest.mark.gpu
@pytest.mark.parametrize('loss', ['region', 'v1'])
def test_passthrough_step_vs_oracle(ops, loss):
    """96x96, batch 6, 23 layers.  Layer-locally (the method of test_training_step_vs_oracle): float64 autograd on the
    product's own saved layer input and incoming gradient reproduces dW, dgamma, dbeta and the outgoing data gradient of
    every layer -- the passthrough conv (input: layer 13 un-pooled; gradient: depth_to_space of the concat gradient),
    conv2 (the concat gradient's first 1024 columns) and layer 13 (the sum of its two consumers).  Whole chain against the
    oracle's training step over the passthrough graph (train_step_reference above): the net output and the direction of dW.  With the region loss, the oracle's chain is seeded with the
    loss gradient at the product's net output (the oracle restates the region loss forward + gradient, not as a graph)."""
    N, IS = 6, 96
    S = IS // 32
    rs = np.random.RandomState(7)
    img = rs.randint(0, 256, (N, IS, IS, 3)).astype(np.uint8)
    st, layers, tr = _trainer(N, IS, loss)
    core_p, head_p, pt_p = oracle_params(st, layers, with_passthrough=True)
    assert len(tr.layers) == 23 and tr.layers[20]['role'] == 'passthrough'
    if loss == 'region':
        gt = _random_gt(rs, N, 32)
        tr.set_ground_truth(*gt)
    else:
        labels = _labels_v1(rs, N, S, IS)
        tr.set_labels(labels)
    p_before = [{k: v.clone() for k, v in tr.P[li].items()} for li in range(23)]
    cap = {}
    tr.step(torch.tensor(img), capture=cap)
    torch.cuda.synchronize()
    got_net = tr.acts[-1].cpu().numpy()

    # loss gradient on the product's own net output
    if loss == 'region':
        _, dnet_want, _ = O.region_loss_torch(got_net, *gt)
        seed = torch.tensor(dnet_want, dtype=torch.float64)
        loss_fn = lambda net: (net * seed).sum()
    else:
        _, dnet_want = O.get_loss_torch(got_net, labels, 20, N, IS, S, 2)
        lab_t = torch.tensor(labels, dtype=torch.float64)
        loss_fn = lambda net: O.loss_v1_graph(net, lab_t, 20, N, IS, S, 2)[0]
    assert rel_l2(cap[22].cpu().numpy(), dnet_want) < 1e-4

    # whole chain
    _, grads, _, net = train_step_reference(O.preprocess_u8(img), core_p, head_p, loss_fn, params_passthrough=pt_p)
    print('net rel_l2 %.3g' % rel_l2(got_net, net))
    assert rel_l2(got_net, net) < 8e-2
    for li in (22, 20, 12, 0):
        a, b = tr.G[li]['W'].cpu().numpy().ravel().astype(np.float64), grads[li]['W'].ravel()
        cos = float(a @ b / (np.linalg.norm(a) * np.linalg.norm(b)))
        print('layer %2d dW cosine vs whole-chain oracle %.3f' % (li + 1, cos))
        assert cos > 0.8

    # layer-local
    for li in reversed(range(23)):
        L = layers[li]
        x = _layer_input(tr, li).double().cpu().requires_grad_(True)
        q = {k: p_before[li][k].double().cpu().requires_grad_(True) for k in ('W', 'b', 'gamma', 'beta')}
        q['mm'], q['mv'] = torch.zeros(L['cout'], dtype=torch.float64), torch.ones(L['cout'], dtype=torch.float64)
        y, _, _ = O.conv_bn_layer(x, q, True, torch.float64, bf16_operands=True)
        obj = ((O.max_pool_2x2(y) if L['pool'] else y) * cap[li].double().cpu()).sum()
        if li == 12:                                            # the passthrough conv's gradient of the un-pooled output
            obj = obj + (y * cap['d_pt'].double().cpu()).sum()
        obj.backward()
        if li == 21:
            dx_got = tr.d_cat
        elif li == 20:
            dx_got = cap['d_pt']
        else:
            dx_got = cap.get(li - 1)
        eW = rel_l2(tr.G[li]['W'].cpu().numpy(), q['W'].grad.numpy())
        eg = rel_l2(tr.G[li]['gamma'].cpu().numpy(), q['gamma'].grad.numpy())
        eb = rel_l2(tr.G[li]['beta'].cpu().numpy(), q['beta'].grad.numpy())
        ex = rel_l2(dx_got.float().cpu().numpy(), x.grad.numpy()) if li > 0 else 0.0
        print('layer %2d local: dW %.3g dgamma %.3g dbeta %.3g dx %.3g' % (li + 1, eW, eg, eb, ex))
        assert eW < 1e-2 and eg < 1e-2 and eb < 1e-2 and ex < 1e-2, (li, eW, eg, eb, ex)
        assert float(tr.G[li]['b'].abs().max()) == 0.0


# ---- 3. the new backward stages of a full-size step ---------------------------------------------------------------------------
@pytest.fixture(scope='module')
def rec416():
    """One eager 416x416 batch-64 region-loss step of the passthrough graph, recorded at the layers whose backward is new:
    layer 13 (index 12), conv2 (19), the passthrough conv (20) and conv3 (21)."""
    from tensorflow_yolo2_b200 import ops
    N, IS = 64, 416
    rs = np.random.RandomState(416)
    images = _images(IS, N, 416)
    st, layers, tr = _trainer(N, IS, 'region')
    tr.set_ground_truth(*_random_gt(rs, N, 32))
    tr.in_u8.copy_(torch.as_tensor(images))
    keep = (12, 19, 20, 21)
    R = dict(N=N, layers=tr.layers, geom=tr.geom, dy={}, dh={}, dx={}, grads={}, raw={}, stats={}, x={})
    R['params'] = {li: {k: v.clone() for k, v in tr.P[li].items()} for li in keep}
    tr.iteration += 1
    tr._set_lr()
    with ops.conv_workspace_scope(tr.conv_ws):
        tr.forward()
        tr.loss()
        for li in keep:
            R['raw'][li] = tr.raw[li].clone()
            R['stats'][li] = {k: v.clone() for k, v in tr.stats[li].items()}
            R['x'][li] = _layer_input(tr, li).clone()
        for li in reversed(range(len(tr.layers))):
            if li in keep:
                R['dy'][li] = tr._dy_of(li).clone()
                if li == 12:
                    R['d_pt'] = tr.d_pt.clone()
            tr._backward_layer(li)
            if li in keep:
                g = tr.geom[li]
                R['dh'][li] = tr.dh[:g['M'] * g['ld_dh']].view(g['M'], g['ld_dh']).clone()
                R['dx'][li] = tr.dx_out[li].clone()
                R['grads'][li] = {k: v.clone() for k, v in tr.G[li].items()}
    torch.cuda.synchronize()
    del tr
    torch.cuda.empty_cache()
    yield R
    R.clear()
    torch.cuda.empty_cache()


def _nchw(t):
    return t.permute(0, 3, 1, 2).contiguous()


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


def _stage_wgrad(R, li):
    L, H = R['layers'][li], R['geom'][li]['H']
    k, cin, cout = L['k'], L['cin'], L['cout']
    x = _nchw(R['x'][li])
    dh = _nchw(R['dh'][li][:, :cout].reshape(R['N'], H, H, cout))
    ref = torch.nn.grad.conv2d_weight(x.double(), (cout, cin, k, k), dh.double(), padding=k // 2).permute(2, 3, 1, 0)
    absref = torch.nn.grad.conv2d_weight(x.float().abs(), (cout, cin, k, k), dh.float().abs(), padding=k // 2).permute(2, 3, 1, 0)
    _check('wgrad', R['grads'][li]['W'], ref, absref, bf16_out=False, tau=TAU_WGRAD)
    assert float(R['grads'][li]['b'].abs().max()) == 0.0


def _stage_dgrad(R, li):
    L, H = R['layers'][li], R['geom'][li]['H']
    k, cin, cout = L['k'], L['cin'], L['cout']
    N = R['N']
    dh = _nchw(R['dh'][li][:, :cout].reshape(N, H, H, cout))
    w = R['params'][li]['W'].to(torch.bfloat16).permute(3, 2, 0, 1)
    ref = _nhwc(torch.nn.grad.conv2d_input((N, cin, H, H), w.double(), dh.double(), padding=k // 2))
    absref = _nhwc(torch.nn.grad.conv2d_input((N, cin, H, H), w.float().abs(), dh.float().abs(), padding=k // 2))
    got = R['dx'][li].view(N, H, H, cin)
    _check('dgrad', got, ref, absref, bf16_out=True)


def _stage_bnbwd(R, li):
    """Batch-norm backward of one recorded layer against float64, routing the pooled gradient to the first maximum of each
    window; the un-pooled addend (layer 13) reaches every row.  Where the float32 recomputation of the affine cannot decide
    the routing (top candidates within 4 float32 ulps) or the leaky slope (|z| within that error), the window is left out of
    the dh element check and its possible effect is added to the dgamma / dbeta bound (the rule of
    test_training_fullres_gpu.py)."""
    from tests.helpers import REL_L2_BF16, REL_L2_ELEM, _rel_l2, _ulp
    L, g, s, p = R['layers'][li], R['geom'][li], R['stats'][li], R['params'][li]
    N, H, C, M, pool = R['N'], g['H'], L['cout'], g['M'], L['pool']
    P = 4 if pool else 1
    win = lambda t: (t.reshape(N, H // 2, 2, H // 2, 2, C).permute(0, 1, 3, 2, 4, 5).reshape(-1, 4, C) if pool
                     else t.reshape(-1, 1, C))
    gamma, beta, mean = p['gamma'].double(), p['beta'].double(), s['mean'].double()
    inv = (s['var'].double() + O.BN_EPS).rsqrt()
    hw = win(R['raw'][li][:, :C].double())
    xh = (hw - mean) * inv
    z = xh * gamma + beta
    a = torch.where(z > 0, z, O.ALPHA * z)
    slope = torch.where(z > 0, torch.ones_like(z), torch.full_like(z, O.ALPHA))
    err_aff = 4 * _ulp((xh * gamma).abs() + beta.abs(), 24)
    pos = torch.arange(P, device=hw.device).view(1, P, 1)
    key = hw * torch.sign(gamma)
    first = torch.where(key == key.amax(dim=1, keepdim=True), pos, P).amin(dim=1)
    h_first = hw.gather(1, first[:, None]).squeeze(1)
    cand = a >= a.amax(dim=1, keepdim=True) - err_aff.amax(dim=1, keepdim=True)
    ambiguous = (cand & (hw != h_first[:, None])).any(dim=1)                    # [U, C]
    z_amb = z.abs() <= err_aff                                                  # [U, P, C]
    dy = R['dy'][li].double().reshape(-1, C)
    dA = (pos == first[:, None]).double() * dy[:, None]
    if li == 12:
        dA = dA + win(R['d_pt'].double().reshape(-1, C))
    dz = dA * slope
    n_amb = int(ambiguous.sum())
    print('windows %d  ambiguous %d  undecided slopes %d' % (dy.numel(), n_amb, int(z_amb.sum())))
    assert n_amb <= 5e-3 * dy.numel()
    slack_b = (torch.where(ambiguous, 2 * dy.abs(), 0.0) + ((1 - O.ALPHA) * dA.abs() * z_amb).sum(1)).sum(0)
    slack_g = (torch.where(ambiguous, 2 * dy.abs() * xh.abs().amax(1), 0.0)
               + ((1 - O.ALPHA) * (dA * xh).abs() * z_amb).sum(1)).sum(0)
    gr = R['grads'][li]
    for nm, got, ref, tol in (('dbeta', gr['beta'], dz.sum((0, 1)), TAU * dz.abs().sum((0, 1)) + slack_b),
                              ('dgamma', gr['gamma'], (dz * xh).sum((0, 1)), TAU * (dz * xh).abs().sum((0, 1)) + slack_g)):
        e = (got.double() - ref).abs()
        print('%-8s max err / bound %.3f   rel-L2 %.3g' % (nm, float((e / tol).max()), _rel_l2(got, ref)))
        assert torch.all(e <= tol), '%s: %d of %d channels out of bound' % (nm, int((e > tol).sum()), C)
        assert _rel_l2(got, ref) <= REL_L2_ELEM * _rel_l2(ref + tol, ref)
    dh_all = R['dh'][li]
    assert torch.all(dh_all[:, C:] == 0)
    got = win(dh_all[:, :C].double())
    gi = gamma * inv
    m1, m2 = gr['beta'].double() / M, gr['gamma'].double() / M
    ref = gi * (dz - m1 - xh * m2)
    absref = gi.abs() * (dz.abs() + m1.abs() + (xh * m2).abs())
    sel = ~(ambiguous[:, None, :] | z_amb.any(dim=1, keepdim=True)).expand_as(got)
    _check('dh', got[sel], ref[sel], absref[sel], bf16_out=True)
    assert _rel_l2(got, ref) <= REL_L2_BF16 * 1.5


_FULL_STAGES = [(21, 'dgrad'), (21, 'wgrad'), (20, 'bnbwd'), (20, 'wgrad'), (20, 'dgrad'), (19, 'bnbwd'), (12, 'bnbwd')]


@pytest.mark.gpu
@pytest.mark.parametrize('li,stage', [pytest.param(li, st, id='L%d-%s' % (li + 1, st)) for li, st in _FULL_STAGES])
def test_fullsize_passthrough_stage_vs_float64(rec416, li, stage):
    with torch.no_grad():
        dict(dgrad=_stage_dgrad, wgrad=_stage_wgrad, bnbwd=_stage_bnbwd)[stage](rec416, li)
    torch.cuda.empty_cache()


# ---- 4.-6. CUDA graph, convergence, checkpoint -> inference -------------------------------------------------------------------
@pytest.mark.gpu
def test_passthrough_cuda_graph_equals_eager(ops):
    N, IS = 4, 96
    rs = np.random.RandomState(4)
    img = torch.tensor(rs.randint(0, 256, (N, IS, IS, 3)).astype(np.uint8))
    gt = _random_gt(rs, N, 32)
    res = []
    for graph in (False, True):
        st, _, tr = _trainer(N, IS, 'region', use_cuda_graph=graph)
        tr.set_ground_truth(*gt)
        losses = [float(tr.step(img)[4]) for _ in range(3)]
        torch.cuda.synchronize()
        assert (tr.graph is not None) == graph and tr.iteration == 3
        assert float(tr.grads.abs().max()) == 0.0
        res.append((losses, tr.params.clone(), st[tr.layers[20]['bn']['moving_mean']].clone()))
    (l0, p0, mm0), (l1, p1, mm1) = res
    print(l0, l1)
    np.testing.assert_allclose(l0, l1, rtol=2e-2)
    assert float((p0 - p1).abs().mean()) < 3e-4 and float((p0 - p1).abs().max()) < 1e-2
    np.testing.assert_allclose(mm0.cpu().numpy(), mm1.cpu().numpy(), rtol=2e-2, atol=1e-3)


@pytest.mark.gpu
def test_passthrough_training_loss_decreases(ops):
    N, IS = 4, 96
    rs = np.random.RandomState(3)
    img = torch.tensor(rs.randint(0, 256, (N, IS, IS, 3)).astype(np.uint8))
    st, _, tr = _trainer(N, IS, 'region')
    tr.set_ground_truth(*_random_gt(rs, N, 32))
    w0 = tr.P[20]['W'].clone()
    losses = [float(tr.step(img)[4]) for _ in range(12)]
    print(losses)
    # measured on a B200: 29.9 -> 21.5 (0.72x), falling every step after the second; the region loss of this batch (3x3 grid,
    # 45 anchors per image, mostly no-object terms) comes down more slowly than the v1 loss of test_training_loss_decreases
    assert all(b < a for a, b in zip(losses[2:], losses[3:]))
    assert losses[-1] < 0.75 * losses[0]
    assert float((tr.P[20]['W'] - w0).abs().max()) > 0


@pytest.mark.gpu
def test_passthrough_checkpoint_serves_in_engine(ops, tmp_path):
    from tensorflow_yolo2_b200.engine import Yolo2Engine
    from tensorflow_yolo2_b200.variables import VariableStore
    from tensorflow_yolo2_b200.yolo2_nets import net_utils
    N, IS = 4, 96
    rs = np.random.RandomState(5)
    img = torch.tensor(rs.randint(0, 256, (N, IS, IS, 3)).astype(np.uint8))
    st, _, tr = _trainer(N, IS, 'region')
    tr.set_ground_truth(*_random_gt(rs, N, 32))
    for _ in range(2):
        tr.step(img)
    with ops.conv_workspace_scope(tr.conv_ws):
        net = tr.forward().clone()                          # the trained weights' forward pass (batch statistics)
    torch.cuda.synchronize()
    path = str(tmp_path / 'yolo2_pt')
    net_utils.save_checkpoint(path, st, extra=tr.optimizer_state())
    st2 = VariableStore(seed=123)
    eng = Yolo2Engine(N, IS, 125, store=st2, passthrough=True, core_training=True, fused_conv1=False, use_cuda_graph=False,
                      device='cuda:0')
    restored, missing = net_utils.restore_checkpoint(path, st2)
    assert not missing and any('passthrough' in k for k in restored)
    eng.refresh_weights()
    got = eng.infer(img)['net']
    torch.cuda.synchronize()
    e = rel_l2(got.cpu().numpy(), net.cpu().numpy())
    print('engine vs trainer forward: rel_l2 %.3g' % e)
    assert e < 1e-2
    # Adam's slots of the passthrough variables round-trip
    _, _, tr2 = _trainer(N, IS, 'region')
    found = tr2.load_optimizer_state(path + '.npz')
    pt_slots = [k for k in found if '/passthrough/' in k]
    assert len(pt_slots) == 8 and tr2.iteration == tr.iteration
    assert torch.equal(tr2.adam_m, tr.adam_m) and torch.equal(tr2.adam_v, tr.adam_v)


# ---- 7. CPU: the reference training step of the passthrough graph ----------------------------------------------------------
def test_train_step_reference_passthrough_forward_matches_darknet19_forward():
    """train_step_reference above runs O.darknet19_forward's passthrough graph; without the branch it is the oracle's
    O.train_step_reference, value for value."""
    st, layers = make_store(125, tame=True, passthrough=True)
    core_p, head_p, pt_p = oracle_params(st, layers, with_passthrough=True)
    x = O.preprocess_u8(np.random.RandomState(0).randint(0, 256, (2, 64, 64, 3)).astype(np.uint8))
    loss_fn = lambda net: (net ** 2).mean()
    loss, grads, stats, net = train_step_reference(x, core_p, head_p, loss_fn, params_passthrough=pt_p, bf16_operands=False)
    want = O.darknet19_forward(torch.as_tensor(x), core_p, head_p, core_training=True, params_passthrough=pt_p).numpy()
    assert len(grads) == 23 and len(stats) == 23 and grads[20]['W'].shape == (1, 1, 512, 64)
    np.testing.assert_array_equal(net, want)
    # without the branch: the oracle's own training step
    st0, layers0 = make_store(125, tame=True)
    c0, h0 = oracle_params(st0, layers0)
    mine = train_step_reference(x, c0, h0, loss_fn, bf16_operands=False)
    ref = O.train_step_reference(x, c0, h0, loss_fn, bf16_operands=False)
    assert mine[0] == ref[0] and len(mine[1]) == 22
    np.testing.assert_array_equal(mine[3], ref[3])
    for a, b in zip(mine[1], ref[1]):
        for k in a:
            np.testing.assert_array_equal(a[k], b[k])
    for a, b in zip(mine[2], ref[2]):
        np.testing.assert_array_equal(a[0], b[0])
        np.testing.assert_array_equal(a[1], b[1])
