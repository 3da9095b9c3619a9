"""CPU oracle for the tensorflow_yolo2 detection hot path.  TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl reference``
legs may import this module, and only as the checker.  The product
(``tensorflow_yolo2_b200``) never imports it and has no CPU fallback.

What it is: a restatement in NumPy / PyTorch-CPU of the reference's algorithm for the path
(reference = /root/reference, a Python-2 / TensorFlow-1.x repo that cannot run in this image).
Every function cites the reference file:line it follows.  TensorFlow primitive semantics (SAME
padding, BN defaults eps=1e-3 / momentum=0.99, max/min gradient tie rules) are *TF knowledge*,
not code in the reference tree.  Max-pool ties: the gradient of a 2x2 window goes whole to its first
maximum in the order (0,0), (0,1), (1,0), (1,1) (max_pool_2x2), as the training kernels route it.

Pinning status (see DESIGN.md "Oracle"):
  * get_iou / get_loss / decode / label encoder / darknet19 builders are pinned against golden
    vectors produced by executing the reference's OWN source (py2->py3 token fixes in memory,
    nothing copied) over a torch-backed TF1 shim: tests/golden/make_golden.py ->
    tests/golden/ref_*.npz.  The structure (slicing, offsets, masks, layer plan) is therefore the
    reference's; the primitive semantics are the shim's.
  * SURVEY.md section 8(c) hand-derived KATs (IoU values, loss KAT-A/B/C) are checked too.
  * region decode (sigmoid/exp/softmax + anchors), per-class NMS and the region loss do NOT exist
    in the reference -> "parity unpinned" for those: this file is their definition
    (SURVEY.md Appendix A).
"""
from __future__ import annotations

import numpy as np

try:  # torch is only needed for the conv stack and autograd cross-checks
    import torch
    import torch.nn.functional as F
except Exception:  # pragma: no cover
    torch = None

ALPHA = 0.1           # darknet.py:5
BN_EPS = 1e-3         # tf.layers.batch_normalization default [TF-knowledge]
BN_MOMENTUM = 0.99    # tf.layers.batch_normalization default [TF-knowledge]
LAMBDA_COORD = 5.0    # config.py:44
LAMBDA_NOOBJ = 0.5    # config.py:45

VOC_ANCHORS = np.array([[1.3221, 1.73145], [3.19275, 4.00944], [5.05587, 8.09892],
                        [9.47112, 4.84053], [11.2364, 10.0071]], dtype=np.float32)

VOC_CLASSES = ('aeroplane', 'bicycle', 'bird', 'boat', 'bottle', 'bus', 'car', 'cat', 'chair',
               'cow', 'diningtable', 'dog', 'horse', 'motorbike', 'person', 'pottedplant',
               'sheep', 'sofa', 'train', 'tvmonitor')     # pascal_voc.py:24-29

# (ksize, cin, cout, pool_after) -- darknet.py:150-177 (darknet19_core)
CORE_PLAN = [
    (3, 3, 32, True), (3, 32, 64, True),
    (3, 64, 128, False), (3, 128, 64, False), (3, 64, 128, True),
    (3, 128, 256, False), (1, 256, 128, False), (3, 128, 256, True),
    (3, 256, 512, False), (1, 512, 256, False), (3, 256, 512, False), (1, 512, 256, False),
    (3, 256, 512, True),
    (3, 512, 1024, False), (1, 1024, 512, False), (3, 512, 1024, False), (1, 1024, 512, False),
    (3, 512, 1024, False),
]
# NB: layer 4 (darknet.py:156) is conv_bn_layer(h_conv3, 3, 128, 64, ...): a THREE-by-three conv
# (canonical Darknet19 uses 1x1 there; the reference does not) -> ksize 3 above.


def head_plan(output_filter):
    """darknet.py:189-200 (darknet19_detection): 3x(3x3,1024->1024) + 1x1 -> output_filter."""
    return [(3, 1024, 1024, False), (3, 1024, 1024, False), (3, 1024, 1024, False),
            (1, 1024, output_filter, False)]


# ----------------------------------------------------------------------------------------------
# config.py:40-42  YOLO_GRID_OFFSET  (py2: np.array(range(S) * S * B) -> reshape(B,S,S) -> [Y,X,B])
# ----------------------------------------------------------------------------------------------
def yolo_grid_offset(S, B):
    off = np.array(list(range(S)) * S * B)
    off = np.reshape(off, (B, S, S))
    return np.transpose(off, (1, 2, 0))       # off[i, j, b] == j (column index)


# ----------------------------------------------------------------------------------------------
# Convolution stack (darknet.py:20-46) on torch CPU
# ----------------------------------------------------------------------------------------------
def bf16_round(x):
    """Round-to-nearest-even to bfloat16 and back (models the bf16 operand path).  Straight-through for autograd:
    the gradient is NOT rounded (a plain .to(bfloat16) would quantise the gradient flowing back as well)."""
    r = x.detach().to(torch.bfloat16).to(x.dtype)
    return x + (r - x.detach()) if x.requires_grad else r


def conv2d_same(x_nhwc, w_hwio, dtype=None):
    """darknet.py:20-21: tf.nn.conv2d(x, W, strides 1, padding='SAME') -- cross-correlation,
    zero pad floor(k/2) for odd k, stride 1 [TF-knowledge]."""
    dtype = dtype or x_nhwc.dtype
    k = w_hwio.shape[0]
    x = x_nhwc.permute(0, 3, 1, 2).to(dtype)
    w = w_hwio.permute(3, 2, 0, 1).to(dtype)
    y = F.conv2d(x, w, bias=None, stride=1, padding=k // 2)
    return y.permute(0, 2, 3, 1).contiguous()


def max_pool_2x2(x_nhwc):
    """darknet.py:24-25: tf.nn.max_pool 2x2 stride 2 SAME (even maps -> no padding).
    Gradient: the whole incoming gradient goes to the FIRST maximum of each window in the order (0,0), (0,1), (1,0),
    (1,1) [TF-knowledge: MaxPoolGrad routes to the arg-max the forward recorded, the first one it met], never split
    between tied entries (torch's amax would split it evenly)."""
    n, h, w, c = x_nhwc.shape
    assert h % 2 == 0 and w % 2 == 0
    win = x_nhwc.reshape(n, h // 2, 2, w // 2, 2, c).permute(0, 1, 3, 5, 2, 4).reshape(n, h // 2, w // 2, c, 4)
    v = win.detach()
    pos = torch.arange(4, device=v.device)
    first = torch.where(v == v.amax(dim=-1, keepdim=True), pos, 4).amin(dim=-1, keepdim=True)
    return win.gather(-1, first).squeeze(-1)


def batch_norm(h, gamma, beta, moving_mean, moving_var, training):
    """darknet.py:42-44: tf.layers.batch_normalization(center, scale, training).
    training -> biased batch variance over (N,H,W), and the moving stats are updated with
    momentum 0.99 (UPDATE_OPS, pascal_train_darknet.py:49-50) [TF-knowledge].
    Returns (y, new_moving_mean, new_moving_var)."""
    if training:
        mean = h.mean(dim=(0, 1, 2))
        var = h.var(dim=(0, 1, 2), unbiased=False)
        new_mm = moving_mean * BN_MOMENTUM + mean * (1 - BN_MOMENTUM)
        new_mv = moving_var * BN_MOMENTUM + var * (1 - BN_MOMENTUM)
    else:
        mean, var = moving_mean, moving_var
        new_mm, new_mv = moving_mean, moving_var
    y = (h - mean) * torch.rsqrt(var + BN_EPS) * gamma + beta
    return y, new_mm, new_mv


def conv_bn_layer(x, p, training, dtype, bf16_operands=False):
    """darknet.py:39-46: conv + bias -> BN -> leaky(0.1).  p = dict(W,b,gamma,beta,mm,mv).
    bf16_operands=True rounds the conv operands (activation and weight) to bf16 first, which is
    what the tcgen05 path feeds the tensor cores (accumulation stays wide)."""
    W = p['W'].to(dtype)
    xin = x.to(dtype)
    if bf16_operands:
        W = bf16_round(W)
        xin = bf16_round(xin)
    h = conv2d_same(xin, W, dtype) + p['b'].to(dtype)                     # darknet.py:35
    y, mm, mv = batch_norm(h, p['gamma'].to(dtype), p['beta'].to(dtype),
                           p['mm'].to(dtype), p['mv'].to(dtype), training)
    y = torch.maximum(ALPHA * y, y)                                       # darknet.py:45
    return y, h, (mm, mv)


def space_to_depth2(x_nhwc):
    """Passthrough / reorg layer (ABSENT from the reference -- SURVEY Appendix A; parity unpinned): tf.space_to_depth
    with block_size 2 on NHWC, out[n, i, j, (di*2 + dj)*C + c] = x[n, 2i+di, 2j+dj, c]."""
    n, h, w, c = x_nhwc.shape
    assert h % 2 == 0 and w % 2 == 0
    return x_nhwc.reshape(n, h // 2, 2, w // 2, 2, c).permute(0, 1, 3, 2, 4, 5).reshape(n, h // 2, w // 2, 4 * c)


PASSTHROUGH_LAYER = 12          # CORE_PLAN index of the 26x26x512 layer (darknet.py:170), taken BEFORE its max-pool


def darknet19_forward(x_nhwc, params_core, params_head, core_training=False, head_training=True,
                      dtype=None, bf16_operands=False, return_intermediates=False, params_passthrough=None):
    """darknet.py:126-179 (core) + :182-201 (head).  Defaults reproduce the detect script:
    core is_training=False (pascal_detect_darknet.py:41), head is_training=True (darknet.py:184
    default, not overridden at pascal_detect_darknet.py:42).

    params_passthrough (extension, SURVEY Appendix A, default off = the reference's graph): a 1x1 conv_bn_layer
    (512 -> F) on the un-pooled output of core layer 13, space_to_depth(2), channel-concatenated AFTER the 1024
    channels of head conv2; head conv3 then has 1024 + 4F input channels."""
    dtype = dtype or torch.float64
    x = x_nhwc.to(dtype)
    inter = []
    pt_src = None
    for li, ((k, cin, cout, pool), p) in enumerate(zip(CORE_PLAN, params_core)):
        x, _, _ = conv_bn_layer(x, p, core_training, dtype, bf16_operands)
        if li == PASSTHROUGH_LAYER:
            pt_src = x
        if pool:
            x = max_pool_2x2(x)
        inter.append(x)
    for hi, p in enumerate(params_head):
        if hi == 2 and params_passthrough is not None:
            pt, _, _ = conv_bn_layer(pt_src, params_passthrough, head_training, dtype, bf16_operands)
            x = torch.cat([x, space_to_depth2(pt)], dim=-1)
        x, _, _ = conv_bn_layer(x, p, head_training, dtype, bf16_operands)
        inter.append(x)
    if return_intermediates:
        return x, inter
    return x


def avg_pool_kxk(x_nhwc, k):
    """darknet.py:28-29 / :116: k x k, stride k average pool on an evenly divisible map."""
    n, h, w, c = x_nhwc.shape
    return x_nhwc.reshape(n, h // k, k, w // k, k, c).mean(dim=(2, 4))


def darknet19_classifier_forward(x_nhwc, params_core, param_cls, training=False, dtype=None, bf16_operands=False):
    """darknet.py:61-123: core layers + conv_bn_layer(1x1, 1024 -> 1000) + 7x7 average pool + reshape -> logits [N, 1000]."""
    dtype = dtype or torch.float64
    x = x_nhwc.to(dtype)
    for (k, cin, cout, pool), p in zip(CORE_PLAN, params_core):
        x, _, _ = conv_bn_layer(x, p, training, dtype, bf16_operands)
        if pool:
            x = max_pool_2x2(x)
    x, _, _ = conv_bn_layer(x, param_cls, training, dtype, bf16_operands)
    return avg_pool_kxk(x, 7).reshape(-1, x.shape[-1])


# ----------------------------------------------------------------------------------------------
# net_utils.py:222-260  get_iou      (numpy; dtype follows the inputs)
# ----------------------------------------------------------------------------------------------
def get_iou(boxes1, boxes2):
    """boxes*: [..., 4] (cx, cy, w, h) -> iou [...].  Op order follows net_utils.py:231-260
    exactly so that a float32 evaluation is bit-reproducible on the GPU (no FMA contraction)."""
    b1 = np.asarray(boxes1)
    b2 = np.asarray(boxes2)
    dt = np.result_type(b1.dtype, b2.dtype)
    two = dt.type(2.0)
    x1a = b1[..., 0] - b1[..., 2] / two
    y1a = b1[..., 1] - b1[..., 3] / two
    x2a = b1[..., 0] + b1[..., 2] / two
    y2a = b1[..., 1] + b1[..., 3] / two
    x1b = b2[..., 0] - b2[..., 2] / two
    y1b = b2[..., 1] - b2[..., 3] / two
    x2b = b2[..., 0] + b2[..., 2] / two
    y2b = b2[..., 1] + b2[..., 3] / two
    lu_x = np.maximum(x1a, x1b)
    lu_y = np.maximum(y1a, y1b)
    rd_x = np.minimum(x2a, x2b)
    rd_y = np.minimum(y2a, y2b)
    iw = np.maximum(dt.type(0.0), rd_x - lu_x)
    ih = np.maximum(dt.type(0.0), rd_y - lu_y)
    inter = iw * ih
    sq1 = (x2a - x1a) * (y2a - y1a)
    sq2 = (x2b - x1b) * (y2b - y1b)
    union = np.maximum(sq1 + sq2 - inter, dt.type(1e-10))
    return np.clip(inter / union, dt.type(0.0), dt.type(1.0))


# ----------------------------------------------------------------------------------------------
# net_utils.py:263-372  get_loss  (YOLOv1 SSE loss, layout [C | B conf | B x (x,y,sqrt w,sqrt h)])
# ----------------------------------------------------------------------------------------------
def get_loss(net, labels, num_class, batch_size, image_size, S, B, OFFSET=None,
             lambda_coord=LAMBDA_COORD, lambda_noobj=LAMBDA_NOOBJ, with_grad=False,
             dtype=np.float64):
    """Returns dict(loss, class_loss, coord_loss, object_loss, noobject_loss, ious, object_mask
    [, dnet]).  dnet is the analytic gradient TF autodiff would produce: the graph has no
    stop_gradient, so the object term back-propagates through `ious` into the predicted box
    (through max/min/clip, the division and w^2); the masks come from a compare+cast and carry
    no gradient.  Tie rules follow TF: maximum(x,y) routes the gradient to x when x >= y,
    minimum(x,y) to x when x <= y [TF-knowledge]."""
    net = np.asarray(net, dtype=dtype)
    labels = np.asarray(labels, dtype=dtype)
    N, C = batch_size, num_class
    if OFFSET is None:
        OFFSET = yolo_grid_offset(S, B)
    assert net.shape == (N, S, S, C + 5 * B) and labels.shape == (N, S, S, 5 + C)
    t = dtype
    p_cls = net[..., :C]                                                  # :279
    p_conf = net[..., C:C + B]                                            # :281
    p_box = net[..., C + B:].reshape(N, S, S, B, 4)                       # :284-285

    resp = labels[..., 0].reshape(N, S, S, 1)                             # :290-291
    classes = labels[..., 5:]                                             # :292
    class_delta = resp * (p_cls - classes)                                # :294-295
    class_loss = np.mean(np.sum(class_delta ** 2, axis=(1, 2, 3)))        # :296-297

    gt = labels[..., 1:5].reshape(N, S, S, 1, 4)                          # :302
    gt = np.tile(gt, (1, 1, 1, B, 1)) / t(float(image_size))              # :303
    off = np.asarray(OFFSET, dtype=dtype).reshape(1, S, S, B)             # :307-309
    off = np.tile(off, (N, 1, 1, 1))
    off_t = np.transpose(off, (0, 2, 1, 3))
    px = (p_box[..., 0] + off) / t(float(S))                              # :310
    py = (p_box[..., 1] + off_t) / t(float(S))                            # :311-312
    pw = p_box[..., 2] ** 2                                               # :313
    ph = p_box[..., 3] ** 2                                               # :314
    pred_abs = np.stack([px, py, pw, ph], axis=4)                         # :315-316
    ious = get_iou(pred_abs, gt)                                          # :320

    omax = np.max(ious, axis=3, keepdims=True)                            # :323
    object_mask = (ious >= omax).astype(dtype) * resp                     # :324
    noobject_mask = np.ones_like(object_mask) - object_mask               # :325-326

    gx = gt[..., 0] * t(S) - off                                          # :330
    gy = gt[..., 1] * t(S) - off_t                                        # :331-332
    gw = np.sqrt(gt[..., 2])                                              # :333
    gh = np.sqrt(gt[..., 3])                                              # :334
    dxs = p_box[..., 0] - gx                                              # :338
    dys = p_box[..., 1] - gy
    dws = p_box[..., 2] - gw                                              # :341 (sqrt-space)
    dhs = p_box[..., 3] - gh
    boxes_delta = np.stack([dxs, dys, dws, dhs], axis=4) * object_mask[..., None]  # :343-345
    coord_loss = np.mean(np.sum(boxes_delta ** 2, axis=(1, 2, 3, 4))) * t(lambda_coord)  # :346

    object_delta = object_mask * (p_conf - ious)                          # :353
    object_loss = np.mean(np.sum(object_delta ** 2, axis=(1, 2, 3)))      # :354-355
    noobject_delta = noobject_mask * p_conf                               # :357
    noobject_loss = np.mean(np.sum(noobject_delta ** 2, axis=(1, 2, 3))) * t(lambda_noobj)  # :358

    out = dict(loss=class_loss + object_loss + noobject_loss + coord_loss,   # :372
               class_loss=class_loss, coord_loss=coord_loss, object_loss=object_loss,
               noobject_loss=noobject_loss, ious=ious, object_mask=object_mask)
    if not with_grad:
        return out

    # ---- analytic backward (what TF autodiff computes for this graph) ----
    invN = t(1.0) / t(N)
    d_cls = 2.0 * resp * resp * (p_cls - classes) * invN
    d_conf = (2.0 * object_mask ** 2 * (p_conf - ious)
              + 2.0 * t(lambda_noobj) * noobject_mask ** 2 * p_conf) * invN
    m2 = object_mask ** 2
    d_box = np.stack([dxs, dys, dws, dhs], axis=4) * (2.0 * t(lambda_coord) * invN) * m2[..., None]
    # gradient through ious (object term): dL/diou = -2 m^2 (conf - iou)/N
    d_iou = -2.0 * m2 * (p_conf - ious) * invN
    d_abs = _iou_backward(pred_abs, gt, d_iou)                            # d wrt (px,py,pw,ph)
    d_box[..., 0] += d_abs[..., 0] / t(float(S))
    d_box[..., 1] += d_abs[..., 1] / t(float(S))
    d_box[..., 2] += d_abs[..., 2] * 2.0 * p_box[..., 2]
    d_box[..., 3] += d_abs[..., 3] * 2.0 * p_box[..., 3]
    dnet = np.concatenate([d_cls, d_conf, d_box.reshape(N, S, S, 4 * B)], axis=3)
    out['dnet'] = dnet
    return out


def _iou_backward(b1, b2, d_iou):
    """Gradient of get_iou w.r.t. boxes1 (cx,cy,w,h), TF tie semantics."""
    t = b1.dtype.type
    cx, cy, w, h = b1[..., 0], b1[..., 1], b1[..., 2], b1[..., 3]
    x1a, y1a, x2a, y2a = cx - w / 2.0, cy - h / 2.0, cx + w / 2.0, cy + h / 2.0
    x1b = b2[..., 0] - b2[..., 2] / 2.0
    y1b = b2[..., 1] - b2[..., 3] / 2.0
    x2b = b2[..., 0] + b2[..., 2] / 2.0
    y2b = b2[..., 1] + b2[..., 3] / 2.0
    lu_x, lu_y = np.maximum(x1a, x1b), np.maximum(y1a, y1b)
    rd_x, rd_y = np.minimum(x2a, x2b), np.minimum(y2a, y2b)
    dw_, dh_ = rd_x - lu_x, rd_y - lu_y
    iw, ih = np.maximum(0.0, dw_), np.maximum(0.0, dh_)
    inter = iw * ih
    sq1 = (x2a - x1a) * (y2a - y1a)
    sq2 = (x2b - x1b) * (y2b - y1b)
    u_raw = sq1 + sq2 - inter
    union = np.maximum(u_raw, 1e-10)
    q = inter / union
    # clip_by_value(q,0,1) = minimum(maximum(q,0),1): gradient passes when 0 <= q <= 1
    g_q = d_iou * ((q >= 0.0) & (q <= 1.0)).astype(b1.dtype)
    g_inter = g_q / union
    g_union = -g_q * inter / (union * union)
    g_uraw = g_union * (u_raw >= 1e-10).astype(b1.dtype)          # maximum(u_raw, 1e-10): x first
    g_sq1 = g_uraw
    g_inter = g_inter - g_uraw
    g_iw = g_inter * ih
    g_ih = g_inter * iw
    # maximum(0.0, d): constant is the FIRST argument -> on a tie (d == 0) the constant wins
    g_dw = g_iw * (dw_ > 0.0).astype(b1.dtype)
    g_dh = g_ih * (dh_ > 0.0).astype(b1.dtype)
    g_rdx, g_lux = g_dw, -g_dw
    g_rdy, g_luy = g_dh, -g_dh
    # lu = maximum(boxes1, boxes2): boxes1 first -> gets gradient when >=
    g_x1a = g_lux * (x1a >= x1b).astype(b1.dtype)
    g_y1a = g_luy * (y1a >= y1b).astype(b1.dtype)
    # rd = minimum(boxes1, boxes2): boxes1 gets gradient when <=
    g_x2a = g_rdx * (x2a <= x2b).astype(b1.dtype)
    g_y2a = g_rdy * (y2a <= y2b).astype(b1.dtype)
    # square1 = (x2a-x1a)*(y2a-y1a)
    g_x2a = g_x2a + g_sq1 * (y2a - y1a)
    g_x1a = g_x1a - g_sq1 * (y2a - y1a)
    g_y2a = g_y2a + g_sq1 * (x2a - x1a)
    g_y1a = g_y1a - g_sq1 * (x2a - x1a)
    g = np.zeros_like(b1)
    g[..., 0] = g_x1a + g_x2a
    g[..., 1] = g_y1a + g_y2a
    g[..., 2] = (g_x2a - g_x1a) * 0.5
    g[..., 3] = (g_y2a - g_y1a) * 0.5
    return g


def loss_v1_graph(net, labels, num_class, batch_size, image_size, S, B,
                  lambda_coord=LAMBDA_COORD, lambda_noobj=LAMBDA_NOOBJ):
    """get_loss (net_utils.py:263-372) as a differentiable torch float64 graph; returns the scalar loss tensor
    and the four terms (class, coord, object, noobject)."""
    N, C = batch_size, num_class
    net = net.reshape(N, S, S, C + 5 * B)
    p_cls, p_conf = net[..., :C], net[..., C:C + B]
    p_box = net[..., C + B:].reshape(N, S, S, B, 4)
    resp = labels[..., 0].reshape(N, S, S, 1)
    class_loss = ((resp * (p_cls - labels[..., 5:])) ** 2).sum(dim=(1, 2, 3)).mean()
    gt = labels[..., 1:5].reshape(N, S, S, 1, 4).repeat(1, 1, 1, B, 1) / float(image_size)
    off = torch.as_tensor(yolo_grid_offset(S, B), dtype=torch.float64).reshape(1, S, S, B)
    off_t = off.permute(0, 2, 1, 3)
    pa = torch.stack([(p_box[..., 0] + off) / S, (p_box[..., 1] + off_t) / S,
                      p_box[..., 2] ** 2, p_box[..., 3] ** 2], dim=4)

    def corners(b):
        return (b[..., 0] - b[..., 2] / 2, b[..., 1] - b[..., 3] / 2,
                b[..., 0] + b[..., 2] / 2, b[..., 1] + b[..., 3] / 2)
    x1a, y1a, x2a, y2a = corners(pa)
    x1b, y1b, x2b, y2b = corners(gt)
    iw = torch.clamp(torch.minimum(x2a, x2b) - torch.maximum(x1a, x1b), min=0)
    ih = torch.clamp(torch.minimum(y2a, y2b) - torch.maximum(y1a, y1b), min=0)
    inter = iw * ih
    union = torch.clamp((x2a - x1a) * (y2a - y1a) + (x2b - x1b) * (y2b - y1b) - inter, min=1e-10)
    ious = torch.clamp(inter / union, 0, 1)
    mask = ((ious >= ious.max(dim=3, keepdim=True).values).double() * resp).detach()
    nomask = 1 - mask
    gx, gy = gt[..., 0] * S - off, gt[..., 1] * S - off_t
    gw, gh = gt[..., 2].sqrt(), gt[..., 3].sqrt()
    delta = torch.stack([p_box[..., 0] - gx, p_box[..., 1] - gy,
                         p_box[..., 2] - gw, p_box[..., 3] - gh], dim=4) * mask[..., None]
    coord = (delta ** 2).sum(dim=(1, 2, 3, 4)).mean() * lambda_coord
    obj = ((mask * (p_conf - ious)) ** 2).sum(dim=(1, 2, 3)).mean()
    noobj = ((nomask * p_conf) ** 2).sum(dim=(1, 2, 3)).mean() * lambda_noobj
    return class_loss + obj + noobj + coord, (class_loss, coord, obj, noobj)


def get_loss_torch(net, labels, num_class, batch_size, image_size, S, B,
                   lambda_coord=LAMBDA_COORD, lambda_noobj=LAMBDA_NOOBJ):
    """Same graph as get_loss on torch float64 with autograd -- an independent check of the
    analytic gradient (torch splits max/min ties evenly, so only tie-free inputs compare)."""
    net = torch.as_tensor(np.asarray(net), dtype=torch.float64).clone().requires_grad_(True)
    labels = torch.as_tensor(np.asarray(labels), dtype=torch.float64)
    loss, _ = loss_v1_graph(net, labels, num_class, batch_size, image_size, S, B, lambda_coord, lambda_noobj)
    loss.backward()
    return float(loss), net.grad.numpy()


def train_step_reference(x_nhwc, params_core, params_head, loss_fn, bf16_operands=True, dtype=torch.float64):
    """One iteration of pascal_train_darknet.py:96-102 up to the gradients: forward with is_training=True in
    every layer (:36,39-40 feed is_training=True), loss, backward (TF autodiff == torch autograd on the same
    graph).  loss_fn(net float64 tensor) -> scalar tensor.  Returns (loss, grads) with grads a list (layer order)
    of dict(W, b, gamma, beta) float64 numpy arrays, plus the per-layer batch (mean, var)."""
    leaves = []
    for p in list(params_core) + list(params_head):
        q = {k: torch.as_tensor(np.asarray(v), dtype=dtype).clone() for k, v in p.items()}
        for k in ('W', 'b', 'gamma', 'beta'):
            q[k].requires_grad_(True)
        leaves.append(q)
    nc = len(params_core)
    x = torch.as_tensor(np.asarray(x_nhwc), dtype=dtype)
    stats = []
    for li, q in enumerate(leaves):
        x, h, _ = conv_bn_layer(x, q, True, dtype, bf16_operands)
        stats.append((h.detach().mean(dim=(0, 1, 2)).numpy(), h.detach().var(dim=(0, 1, 2), unbiased=False).numpy()))
        if li < nc and CORE_PLAN[li][3]:
            x = max_pool_2x2(x)
    loss = loss_fn(x)
    loss.backward()
    grads = [{k: q[k].grad.numpy() for k in ('W', 'b', 'gamma', 'beta')} for q in leaves]
    return float(loss.detach()), grads, stats, x.detach().numpy()


# ----------------------------------------------------------------------------------------------
# net_utils.py:387-421  decode half of show_yolo_detection  (REF_V1)
# ----------------------------------------------------------------------------------------------
def decode_ref_v1(predict_output, S, B, num_class, object_thresh=0.5, dtype=np.float32):
    """predict_output: one image [S,S,C+5B].  Returns the dense decode the reference computes
    before its draw loop: dict(xs, ys, ws, hs [S,S,B] normalised to the image, conf [S,S,B],
    keep [S,S,B] bool, cls [S,S] argmax of the CELL's class vector)."""
    p = np.asarray(predict_output, dtype=dtype).reshape(S, S, num_class + B * 5)   # :393
    cls = p[:, :, :num_class]                                                     # :394
    conf = p[:, :, num_class:num_class + B]                                       # :395
    box = p[:, :, num_class + B:].reshape(S, S, B, 4)                             # :396-397
    keep = conf > dtype(object_thresh)                                            # :398
    off = yolo_grid_offset(S, B).astype(dtype)
    xs = (box[..., 0] + off) / dtype(float(S))                                    # :403
    ys = (box[..., 1] + np.transpose(off, (1, 0, 2))) / dtype(float(S))           # :404-405
    ws = np.square(box[..., 2])                                                   # :406
    hs = np.square(box[..., 3])                                                   # :407
    return dict(xs=xs, ys=ys, ws=ws, hs=hs, conf=conf, keep=keep,
                cls=np.argmax(cls, axis=2))                                       # :418


def draw_list_ref_v1(dec, im_w, im_h):
    """net_utils.py:410-421: the per-box integer pixel math of the draw loop (py2 semantics:
    int() truncation, `predict_w / 2` floor division).  Returns a list of
    (upper_left_x, upper_left_y, w, h, class, conf) in the reference's loop order."""
    out = []
    S, _, B = dec['keep'].shape
    for c in range(S):
        for r in range(S):
            for i in range(B):
                if dec['keep'][c, r, i]:
                    px = int(dec['xs'][c, r, i] * im_w)
                    py = int(dec['ys'][c, r, i] * im_h)
                    pw = int(dec['ws'][c, r, i] * im_w)
                    ph = int(dec['hs'][c, r, i] * im_h)
                    out.append((px - pw // 2, py - ph // 2, pw, ph,
                                int(dec['cls'][c, r]), float(dec['conf'][c, r, i])))
    return out


# ----------------------------------------------------------------------------------------------
# Appendix A (ABSENT from the reference; parity unpinned): region decode, per-class NMS
# ----------------------------------------------------------------------------------------------
def region_decode_v2(net, anchors=VOC_ANCHORS, num_class=20, thresh=0.3):
    """net [N,S,S,A*(5+C)] fp32 -> boxes [N,S*S*A,4] (cx,cy,w,h normalised), scores
    [N,S*S*A,C] = sigmoid(to)*softmax(c), zeroed where <= thresh.  Box index = (i*S+j)*A+a."""
    net = np.asarray(net, dtype=np.float32)
    N, S = net.shape[0], net.shape[1]
    A = len(anchors)
    C = num_class
    v = net.reshape(N, S, S, A, 5 + C).astype(np.float64)
    jj = np.arange(S).reshape(1, 1, S, 1)
    ii = np.arange(S).reshape(1, S, 1, 1)
    sig = lambda z: 1.0 / (1.0 + np.exp(-z))
    bx = (jj + sig(v[..., 0])) / S
    by = (ii + sig(v[..., 1])) / S
    an = np.asarray(anchors, dtype=np.float64)
    bw = an[:, 0].reshape(1, 1, 1, A) * np.exp(v[..., 2]) / S
    bh = an[:, 1].reshape(1, 1, 1, A) * np.exp(v[..., 3]) / S
    obj = sig(v[..., 4])
    c = v[..., 5:]
    e = np.exp(c - c.max(axis=-1, keepdims=True))
    p = e / e.sum(axis=-1, keepdims=True)
    scores = (obj[..., None] * p)
    boxes = np.stack([bx, by, bw, bh], axis=-1).reshape(N, S * S * A, 4).astype(np.float32)
    scores = scores.reshape(N, S * S * A, C).astype(np.float32)
    scores_thr = np.where(scores > np.float32(thresh), scores, np.float32(0.0))
    return boxes, scores_thr, scores


def nms_per_class(boxes, scores, iou_thresh=0.45, score_thresh=0.0):
    """Greedy per-class NMS (Darknet do_nms_sort semantics; SURVEY Appendix A).
    boxes [nbox,4] fp32 (cx,cy,w,h), scores [nbox,C] fp32.  For every class: candidates are the
    boxes with score > score_thresh, ordered by (score desc, box index asc); a candidate is
    suppressed iff an earlier KEPT candidate has IoU > iou_thresh (strict), IoU evaluated in
    float32 with get_iou's op order.  Returns list over classes of int32 arrays of kept box
    indices in visiting order."""
    boxes = np.asarray(boxes, dtype=np.float32)
    scores = np.asarray(scores, dtype=np.float32)
    thr = np.float32(iou_thresh)
    keeps = []
    for k in range(scores.shape[1]):
        s = scores[:, k]
        cand = np.nonzero(s > np.float32(score_thresh))[0]
        order = cand[np.lexsort((cand, -s[cand].astype(np.float64)))]
        kept = []
        alive = np.ones(len(order), dtype=bool)
        for a in range(len(order)):
            if not alive[a]:
                continue
            kept.append(order[a])
            if a + 1 < len(order):
                rest = order[a + 1:]
                iou = get_iou(np.broadcast_to(boxes[order[a]], (len(rest), 4)), boxes[rest])
                alive[a + 1:] &= ~(iou > thr)
        keeps.append(np.asarray(kept, dtype=np.int32))
    return keeps


# ----------------------------------------------------------------------------------------------
# Region (YOLOv2) loss -- Appendix A, absent from the reference; torch float64 + autograd
# ----------------------------------------------------------------------------------------------
def region_loss_torch(net, gt_boxes, gt_classes, gt_counts, anchors=VOC_ANCHORS, num_class=20,
                      lambda_coord=1.0, lambda_obj=5.0, lambda_noobj=1.0, lambda_class=1.0,
                      ignore_thresh=0.6):
    """net [N,S,S,A*(5+C)]; gt_boxes [N,G,4] normalised (cx,cy,w,h); gt_classes [N,G] int;
    gt_counts [N].  Returns (loss, dnet, terms[4]=(coord,obj,noobj,class)).  Loss = mean over the
    batch of per-image sums, like get_loss (net_utils.py:296)."""
    net_t = torch.as_tensor(np.asarray(net), dtype=torch.float64).clone().requires_grad_(True)
    N, S = net_t.shape[0], net_t.shape[1]
    A, C = len(anchors), num_class
    an = torch.as_tensor(np.asarray(anchors, dtype=np.float64))
    v = net_t.reshape(N, S, S, A, 5 + C)
    sx, sy = torch.sigmoid(v[..., 0]), torch.sigmoid(v[..., 1])
    tw, th = v[..., 2], v[..., 3]
    so = torch.sigmoid(v[..., 4])
    pc = torch.softmax(v[..., 5:], dim=-1)
    jj = torch.arange(S, dtype=torch.float64).reshape(1, 1, S, 1)
    ii = torch.arange(S, dtype=torch.float64).reshape(1, S, 1, 1)
    bx, by = (jj + sx) / S, (ii + sy) / S
    bw = an[:, 0].reshape(1, 1, 1, A) * torch.exp(tw) / S
    bh = an[:, 1].reshape(1, 1, 1, A) * torch.exp(th) / S
    pred = torch.stack([bx, by, bw, bh], dim=-1)

    def iou_t(b1, b2):
        x1a, y1a = b1[..., 0] - b1[..., 2] / 2, b1[..., 1] - b1[..., 3] / 2
        x2a, y2a = b1[..., 0] + b1[..., 2] / 2, b1[..., 1] + b1[..., 3] / 2
        x1b, y1b = b2[..., 0] - b2[..., 2] / 2, b2[..., 1] - b2[..., 3] / 2
        x2b, y2b = b2[..., 0] + b2[..., 2] / 2, b2[..., 1] + b2[..., 3] / 2
        iw = torch.clamp(torch.minimum(x2a, x2b) - torch.maximum(x1a, x1b), min=0)
        ih = torch.clamp(torch.minimum(y2a, y2b) - torch.maximum(y1a, y1b), min=0)
        inter = iw * ih
        union = torch.clamp((x2a - x1a) * (y2a - y1a) + (x2b - x1b) * (y2b - y1b) - inter,
                            min=1e-10)
        return torch.clamp(inter / union, 0, 1)

    gtb = torch.as_tensor(np.asarray(gt_boxes), dtype=torch.float64)
    coord = obj = noobj = cls = 0.0
    for n in range(N):
        G = int(gt_counts[n])
        noobj_mask = torch.ones(S, S, A, dtype=torch.float64)
        if G > 0:
            ious_all = iou_t(pred[n].detach().unsqueeze(3), gtb[n, :G].reshape(1, 1, 1, G, 4))
            best = ious_all.max(dim=3).values
            noobj_mask = (best < ignore_thresh).double()
        assigned = {}
        for g in range(G):
            gx, gy, gw, gh = [float(z) for z in gtb[n, g]]
            j, i = min(int(gx * S), S - 1), min(int(gy * S), S - 1)
            # responsible anchor: arg-max IoU of (0,0,pw,ph) vs (0,0,gw,gh) -- first max wins
            best_a, best_iou = 0, -1.0
            for a in range(A):
                pw_, ph_ = float(an[a, 0]) / S, float(an[a, 1]) / S
                inter = min(pw_, gw) * min(ph_, gh)
                u = pw_ * ph_ + gw * gh - inter
                v_ = inter / u
                if v_ > best_iou:
                    best_iou, best_a = v_, a
            if (i, j, best_a) in assigned:       # first GT wins a (cell, anchor) slot
                continue
            assigned[(i, j, best_a)] = g
            a = best_a
            noobj_mask[i, j, a] = 0.0
            scale = lambda_coord * (2.0 - gw * gh)
            tx_t, ty_t = gx * S - j, gy * S - i
            tw_t = np.log(gw * S / float(an[a, 0]))
            th_t = np.log(gh * S / float(an[a, 1]))
            coord = coord + scale * ((sx[n, i, j, a] - tx_t) ** 2 + (sy[n, i, j, a] - ty_t) ** 2
                                     + (tw[n, i, j, a] - tw_t) ** 2 + (th[n, i, j, a] - th_t) ** 2)
            iou_g = iou_t(pred[n, i, j, a], gtb[n, g]).detach()
            obj = obj + lambda_obj * (so[n, i, j, a] - iou_g) ** 2
            onehot = torch.zeros(C, dtype=torch.float64)
            onehot[int(gt_classes[n, g])] = 1.0
            cls = cls + lambda_class * ((pc[n, i, j, a] - onehot) ** 2).sum()
        noobj = noobj + lambda_noobj * ((noobj_mask * so[n]) ** 2).sum()
    loss = (coord + obj + noobj + cls) / N
    loss.backward()
    terms = [float(z) / N for z in (coord, obj, noobj, cls)]
    return float(loss), net_t.grad.numpy(), terms


# ----------------------------------------------------------------------------------------------
# pascal_voc.py:125-165  label encoder; :60-67 / pascal_detect_darknet.py:34-38 preprocessing
# ----------------------------------------------------------------------------------------------
def encode_labels(objects, im_h, im_w, image_size, S, num_class=20):
    """objects: list of (class_index, xmin, ymin, xmax, ymax) 1-based VOC pixels.
    Returns label [S,S,5+C] float64 (pascal_voc.py:137-163): first object wins a cell."""
    h_ratio = 1.0 * image_size / im_h                                      # :133
    w_ratio = 1.0 * image_size / im_w                                      # :134
    label = np.zeros((S, S, 5 + num_class))                                # :137
    for cls_ind, xmin, ymin, xmax, ymax in objects:
        x1 = max(min((float(xmin) - 1) * w_ratio, image_size - 1), 0)      # :146-147
        y1 = max(min((float(ymin) - 1) * h_ratio, image_size - 1), 0)
        x2 = max(min((float(xmax) - 1) * w_ratio, image_size - 1), 0)
        y2 = max(min((float(ymax) - 1) * h_ratio, image_size - 1), 0)
        boxes = [(x2 + x1) / 2.0, (y2 + y1) / 2.0, x2 - x1, y2 - y1]       # :156
        x_ind = int(boxes[0] * S / image_size)                             # :157
        y_ind = int(boxes[1] * S / image_size)                             # :158
        if label[y_ind, x_ind, 0] == 1:                                    # :159-160
            continue
        label[y_ind, x_ind, 0] = 1
        label[y_ind, x_ind, 1:5] = boxes
        label[y_ind, x_ind, 5 + cls_ind] = 1
    return label


def parse_voc_xml(path):
    import xml.etree.ElementTree as ET
    tree = ET.parse(path)
    size = tree.find('size')
    im_w, im_h = int(size.find('width').text), int(size.find('height').text)
    objs = []
    for obj in tree.findall('object'):
        bb = obj.find('bndbox')
        cls = VOC_CLASSES.index(obj.find('name').text.lower().strip())
        objs.append((cls, float(bb.find('xmin').text), float(bb.find('ymin').text),
                     float(bb.find('xmax').text), float(bb.find('ymax').text)))
    return objs, im_h, im_w


def resize_bilinear_u8(src, dst_w, dst_h):
    """cv2.resize(src, (dst_w, dst_h)) for an 8-bit image, default INTER_LINEAR (pascal_detect_darknet.py:35,
    pascal_voc.py:61).  The arithmetic lives in a third-party dependency that is not in /root/reference: OpenCV
    (opencv-python 4.13.0 in this image; unpinned by the reference).  Restated from OpenCV's published fixed-point algorithm
    (modules/imgproc/src/resize.cpp: 2048-scaled short coefficients; columns clamped with the weight zeroed, rows clamped
    with the weights kept; vertical pass ((b*(R>>4))>>16), then (+2)>>2; exact 2x down-scale -> INTER_AREA) and pinned
    against cv2.resize itself in tests/test_oracle.py."""
    src = np.asarray(src)
    sh, sw = src.shape[:2]
    s = src.reshape(sh, sw, -1).astype(np.int64)
    if sw == 2 * dst_w and sh == 2 * dst_h:
        out = (s[0::2, 0::2] + s[0::2, 1::2] + s[1::2, 0::2] + s[1::2, 1::2] + 2) >> 2
        return out.astype(np.uint8).reshape((dst_h, dst_w) + src.shape[2:])

    def coef(dn, sn, clamp):
        scale = 1.0 / (float(dn) / float(sn))
        f = ((np.arange(dn, dtype=np.float64) + 0.5) * scale - 0.5).astype(np.float32)
        s0 = np.floor(f).astype(np.int64)
        f = (f - s0.astype(np.float32)).astype(np.float32)
        if clamp:
            lo, hi = s0 < 0, s0 >= sn - 1
            f[lo | hi] = 0.0
            s0 = np.where(lo, 0, np.where(hi, sn - 1, s0))
        c0 = np.rint((np.float32(1.0) - f) * np.float32(2048.0)).astype(np.int64)
        c1 = np.rint(f * np.float32(2048.0)).astype(np.int64)
        return s0, c0, c1
    xi, a0, a1 = coef(dst_w, sw, True)
    yi, b0, b1 = coef(dst_h, sh, False)
    x1 = np.minimum(xi + 1, sw - 1)
    rows = s[:, xi, :] * a0[None, :, None] + s[:, x1, :] * a1[None, :, None]
    y0, y1 = np.clip(yi, 0, sh - 1), np.clip(yi + 1, 0, sh - 1)
    out = (((b0[:, None, None] * (rows[y0] >> 4)) >> 16) + ((b1[:, None, None] * (rows[y1] >> 4)) >> 16) + 2) >> 2
    return np.clip(out, 0, 255).astype(np.uint8).reshape((dst_h, dst_w) + src.shape[2:])


def preprocess_u8(image_u8_bgr_resized):
    """pascal_voc.py:62-64 / pascal_detect_darknet.py:36-37 on an already-resized uint8 BGR
    image: float32, (x / 255.0) * 2.0 - 1.0."""
    x = np.asarray(image_u8_bgr_resized).astype(np.float32)
    return (x / np.float32(255.0)) * np.float32(2.0) - np.float32(1.0)


# ----------------------------------------------------------------------------------------------
# Adam (tf.train.AdamOptimizer defaults, pascal_train_darknet.py:51) [TF-knowledge]
# ----------------------------------------------------------------------------------------------
def adam_step(p, g, m, v, step, lr=1e-3, b1=0.9, b2=0.999, eps=1e-8):
    """TF1 Adam: lr_t = lr*sqrt(1-b2^t)/(1-b1^t); p -= lr_t * m / (sqrt(v) + eps)."""
    m = b1 * m + (1 - b1) * g
    v = b2 * v + (1 - b2) * g * g
    lr_t = lr * np.sqrt(1 - b2 ** step) / (1 - b1 ** step)
    p = p - lr_t * m / (np.sqrt(v) + eps)
    return p, m, v
