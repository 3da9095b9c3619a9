"""Darknet19 network builders with the reference's interface (src/yolo2_nets/darknet.py), running on
the B200 kernels of libyolo2_b200.so.

Same names, positional/keyword arguments and defaults as the reference:
    alpha, weight_variable, bias_variable, conv2d, max_pool, conv_layer, conv_bn_layer,
    darknet19_core, darknet19_detection
Tensors are CUDA torch tensors in NHWC (float32 in, bf16 between layers on the tensor-core path,
float32 out of the detection head).  Where the reference builds a TF graph, these functions execute
eagerly; variables live in a VariableStore that reproduces TF's auto-generated names
(`darknet19/Variable_3`, `darknet19/batch_normalization_1/gamma`, ...), created on first use and
found again under `reuse=True`.

Compute path (config.COMPUTE): 'bf16' -> tcgen05 implicit-GEMM conv with BN/leaky/pool fused in the
epilogue; 'bf16x3' -> the same kernels on hi + lo bf16 operand pairs (three MMAs per K step; activations travel as
[N,H,W,2C] = [hi | lo] bf16 tensors) -- the mode that meets the 1e-3 detections bar; 'fp32' -> exact FFMA conv +
separate BN/leaky/pool kernels.  No CPU / cuDNN fallback, and no torch library kernel on the path (casts, pools,
concat and space_to_depth are y2_* kernels / store addresses).
"""
from __future__ import annotations

import numpy as np
import torch

from .. import config as cfg
from .. import ops
from ..variables import default_store

alpha = 0.1                       # darknet.py:5

# The reference's UPDATE_OPS only run as a dependency of train_op (pascal_train_darknet.py:49-50);
# a plain sess.run(grid_net) with is_training=True normalises with batch statistics but leaves the
# moving averages untouched.  The training harness flips this flag.
UPDATE_MOVING_AVERAGES = False

# (ksize, cin, cout, pool_after): darknet.py:150-177
CORE_PLAN = [
    (3, 3, 32, True), (3, 32, 64, True),
    (3, 64, 128, False), (3, 128, 64, False), (3, 64, 128, True),
    (3, 128, 256, False), (1, 256, 128, False), (3, 128, 256, True),
    (3, 256, 512, False), (1, 512, 256, False), (3, 256, 512, False), (1, 512, 256, False), (3, 256, 512, True),
    (3, 512, 1024, False), (1, 1024, 512, False), (3, 512, 1024, False), (1, 1024, 512, False),
    (3, 512, 1024, False),
]

PASSTHROUGH_LAYER = 12            # CORE_PLAN index of the 26x26x512 layer (darknet.py:170); its UN-pooled output is the source
PASSTHROUGH_FILTERS = 64


def head_plan(output_filter, passthrough_filters=0):
    """darknet.py:182-201, the detection head as (scope, ksize, cin, cout) in creation order: conv1..conv3 (3x3, 1024->1024)
    and output (1x1 -> output_filter).  passthrough_filters > 0 adds the YOLOv2 passthrough branch (absent from the
    reference, SURVEY Appendix A): a 1x1 conv (scope `passthrough`) on the un-pooled output of CORE_PLAN[PASSTHROUGH_LAYER],
    whose space_to_depth(2) is concatenated after conv2's 1024 channels, so conv3 takes 1024 + 4 * passthrough_filters."""
    plan = [('conv1', 3, 1024, 1024), ('conv2', 3, 1024, 1024)]
    if passthrough_filters:
        plan.append(('passthrough', 1, CORE_PLAN[PASSTHROUGH_LAYER][2], passthrough_filters))
    return plan + [('conv3', 3, 1024 + 4 * passthrough_filters, 1024), ('output', 1, 1024, output_filter)]


def classifier_plan(num_classes=1000):
    """The 19th layer of the `darknet19` ImageNet classifier (darknet.py:61-123), as a CORE_PLAN entry: 1x1, 1024 -> classes."""
    return (1, 1024, int(num_classes), False)


def _device():
    return torch.device('cuda', torch.cuda.current_device())


def _as_param(store, name):
    """Variables are created as numpy arrays by the store; move them to the GPU on first touch."""
    v = store[name]
    if isinstance(v, np.ndarray):
        v = torch.from_numpy(v).to(_device())
        store.vars[name] = v
    return v


# ---------------------------------------------------------------------------------------------
# packed-weight cache (invalidated when the store changes)
# ---------------------------------------------------------------------------------------------
_pack_cache = {}


def _packed(store, wname, split):
    """pack_weights_bf16 of the variable, or pack_weights_bf16_split (bf16x3) with split=True."""
    key = (id(store), wname, split)
    hit = _pack_cache.get(key)
    w = _as_param(store, wname)
    if hit is None or hit[0] != store.version or hit[1] != w.data_ptr():
        hit = (store.version, w.data_ptr(), (ops.pack_weights_bf16_split if split else ops.pack_weights_bf16)(w))
        _pack_cache[key] = hit
    return hit[2]


# ---------------------------------------------------------------------------------------------
# building blocks (darknet.py:10-46)
# ---------------------------------------------------------------------------------------------
def weight_variable(shape):
    """darknet.py:10-12 -- truncated normal, stddev 0.1."""
    store = default_store()
    name, _ = store.weight_variable(list(shape))
    return _as_param(store, name)


def bias_variable(shape):
    """darknet.py:15-17 -- constant 0.1."""
    store = default_store()
    name, _ = store.bias_variable(list(shape))
    return _as_param(store, name)


def _f32(x):
    """float32, contiguous view of an activation (bf16 -> float32 through y2_cast)."""
    x = x if x.dtype == torch.float32 else ops.cast(x, torch.float32)
    return x if x.is_contiguous() else x.contiguous()


def conv2d(x, W, stride):
    """darknet.py:20-21: SAME, stride 1 cross-correlation (exact fp32 kernel, no bias)."""
    assert stride == 1
    return ops.conv_fwd_f32(_f32(x), W, None)


def max_pool(x, pool_size, stride):
    """darknet.py:24-25: 2x2/2 max-pool."""
    assert pool_size == 2 and stride == 2
    N, H, W, C = x.shape
    if x.dtype == torch.bfloat16 and C % 8 == 0:
        return ops.maxpool2x2_bf16(x if x.is_contiguous() else x.contiguous())
    return ops.affine_leaky_pool(_f32(x), N, H, W, C, leaky=False, pool=True, out_bf16=x.dtype == torch.bfloat16)


def avg_pool(x, pool_size, stride):
    """darknet.py:28-29: tf.nn.avg_pool(SAME) -- with pool_size == stride on an evenly divisible map, as every use in the
    reference (the 7x7 global pool, darknet.py:116), SAME and VALID coincide.  Returns float32."""
    assert pool_size == stride and x.shape[1] % stride == 0 and x.shape[2] % stride == 0
    return ops.avg_pool(x, pool_size)


def fc_layer(x, input_dim, output_dim, flat=False, linear=False):
    """darknet.py:49-57: x @ W + b (exact fp32 kernel: a 1x1 convolution over a 1x1 map), leaky(0.1) unless linear."""
    W_fc = weight_variable([input_dim, output_dim])
    b_fc = bias_variable([output_dim])
    if flat:
        x = x.reshape(-1, input_dim)
    n = x.shape[0]
    h = ops.conv_fwd_f32(_f32(x).view(n, 1, 1, input_dim), W_fc.view(1, 1, input_dim, output_dim), b_fc)
    if not linear:                                     # tf.maximum(alpha * h, h) (darknet.py:57)
        h = ops.affine_leaky_pool(h, n, 1, 1, output_dim, leaky=True, pool=False, out_bf16=False)
    return h.view(n, output_dim)


def conv_layer(x, filter_size, input_chl, output_chl, stride):
    """darknet.py:32-36: conv + bias (fp32)."""
    assert stride == 1
    W_conv = weight_variable([filter_size, filter_size, input_chl, output_chl])
    b_conv = bias_variable([output_chl])
    return ops.conv_fwd_f32(_f32(x), W_conv, b_conv)


def conv_bn_layer(x, filter_size, input_chl, output_chl, stride, is_training, _pool=False, _out_f32=None, _out=None,
                  _ldo=None, _col=0, _s2d=False):
    """darknet.py:39-46: conv + bias -> batch norm -> leaky(0.1).

    Extensions (defaults reproduce the reference call): `_pool` fuses the 2x2 max-pool that follows the layer in the
    builders (darknet.py:151,154,...); `_out_f32` forces a float32 result (the detection output); `_out` / `_ldo` /
    `_col` / `_s2d` write the activation into channels [_col, _col + output_chl) of a wider (concatenated) tensor of
    row stride `_ldo`, optionally through tf.space_to_depth(2) -- the passthrough branch, never a copy.

    config.COMPUTE: 'fp32' exact FFMA conv; 'bf16' one tcgen05.mma per K step on bf16-rounded operands; 'bf16x3' hi + lo
    bf16 pairs, three MMAs per K step (activations then travel as [N,H,W,2C] = [hi | lo] bf16 tensors between layers)."""
    assert stride == 1
    store = default_store()
    wname, _ = store.weight_variable([filter_size, filter_size, input_chl, output_chl])
    bname, _ = store.bias_variable([output_chl])
    bn = store.batch_norm_variables(output_chl)
    W, b = _as_param(store, wname), _as_param(store, bname)
    gamma, beta = _as_param(store, bn['gamma']), _as_param(store, bn['beta'])
    mm, mv = _as_param(store, bn['moving_mean']), _as_param(store, bn['moving_variance'])
    training = bool(is_training)
    moving = (mm, mv) if UPDATE_MOVING_AVERAGES else None
    N, H, Wd, _ = x.shape
    mode = cfg.COMPUTE
    if mode not in ('fp32', 'bf16', 'bf16x3'):
        raise ValueError('config.COMPUTE must be "fp32", "bf16" or "bf16x3"')
    x3 = mode == 'bf16x3'
    if x3 and (_out is not None or _s2d):
        raise NotImplementedError('the passthrough branch has no bf16x3 path yet')
    out_f32 = bool(_out_f32) or mode == 'fp32'
    # the exact FFMA route: the fp32 mode, and the first layer of the bf16x3 mode when it is fed float32 pixels (the batch
    # engine's fused uint8 first layer is the fast bf16x3 route; this eager path keeps the 16-bit accuracy with no tensor core)
    if mode == 'fp32' or (x3 and x.dtype == torch.float32 and input_chl == 3):
        h = ops.conv_fwd_f32(_f32(x), W, b)
        if training:
            mean, _, scale, shift = _batch_norm(h.view(-1, output_chl), output_chl, output_chl, gamma, beta, moving)
        else:                                        # the centred form of _batch_norm, on the moving statistics
            scale, _ = ops.bn_fold(gamma, beta, mm, mv)
            mean, shift = mm, beta
        return ops.affine_leaky_pool(h, N, H, Wd, output_chl, sub=mean, scale=scale, shift=shift, leaky=True,
                                     pool=_pool, out_bf16=not out_f32, out=_out, ldo=_ldo, out_col=_col, space_to_depth=_s2d,
                                     split_out=x3)
    # ---- tensor-core path ----
    if x.dtype == torch.float32:
        if input_chl == 3:
            xb = ops.pad_cast_f32_to_bf16c8(x.contiguous())
        elif x3:                                     # float32 fed mid-network: split it into the [hi | lo] pair
            xb = ops.affine_leaky_pool(x.contiguous(), N, H, Wd, input_chl, leaky=False, pool=False, out_bf16=True, split_out=True)
        else:
            xb = ops.cast(x, torch.bfloat16)
    else:
        xb = x
    if x3:
        assert xb.shape[-1] == 2 * input_chl, 'bf16x3: expected a [hi | lo] activation with %d channels' % (2 * input_chl)
    wp = _packed(store, wname, x3)
    fold = None if training else ops.bn_fold(gamma, beta, mm, mv, b)          # inference: bias folded, acc has no bias
    return conv_bn_tc(xb, wp, filter_size, input_chl, output_chl, fold=fold, bias=b, gamma=gamma, beta=beta, moving=moving,
                      pool=_pool, out_f32=out_f32, out=_out, ldo=_ldo, col=_col, s2d=_s2d, x3=x3)


def raw_ld(cout):
    """Row stride of the float32 conv rows of conv_bn_tc: cout rounded up to 32 columns."""
    return (cout + 31) // 32 * 32


def _batch_norm(rows, cout, ld, gamma, beta, moving=None, stats=None, workspace=None):
    """Batch statistics of the float32 conv rows [M, ld] and the affine of the centred form y = (x - mean) * scale + shift
    (scale = gamma * rsqrt(var + eps), shift = beta), plus the moving-average update (UPDATE_OPS) of
    moving=(moving_mean, moving_variance) when given: two launches either way.  Returns stats=(mean, var, scale, shift)."""
    if stats is None:
        stats = tuple(torch.empty((cout,), dtype=torch.float32, device=rows.device) for _ in range(4))
    mean, var, scale, shift = stats
    if moving is None:
        ops.bn_stats_fold(rows, cout, gamma, beta, ld=ld, workspace=workspace, mean=mean, var=var, scale=scale, shift=shift)
    else:
        ops.bn_stats_fold_train(rows, cout, gamma, beta, *moving, ld=ld, workspace=workspace, mean=mean, var=var, scale=scale,
                                shift=shift)
    return stats


def conv_bn_tc(x, wp, k, cin, cout, fold=None, bias=None, gamma=None, beta=None, moving=None, stats=None, workspace=None,
               pool=False, out_f32=False, out=None, ldo=None, col=0, s2d=False, x3=False, raw=None):
    """One conv + BN + leaky(0.1) (+ 2x2 max-pool) layer on the tensor cores: the kernels that conv_bn_layer, Yolo2Engine
    and Yolo2Trainer issue for it.

    x: bf16 [N,H,W,Cin_p] ([N,H,W,2*cin] = [hi | lo] with x3); wp: pack_weights_bf16 (pack_weights_bf16_split with x3).
    BN: fold=(scale, shift) of bn_fold with the conv bias folded in (inference), or fold=None: batch statistics of conv +
    `bias`, normalised with `gamma` / `beta` (see _batch_norm for `moving`, `stats` and `workspace`).
    Output: bf16 [N,Ho,Wo,cout] ([hi | lo] with x3; float32 with out_f32) in `out`, or in channels [col, col + cout) of
    the rows of stride ldo of `out`, stored space-to-depth(2) with s2d.  raw: the float32 [N*H*W, raw_ld(cout)] conv
    rows, written unless BN, leaky and pool run in the conv epilogue.  Buffers left None are allocated.  Returns the output."""
    N, H, W = x.shape[:3]
    if fold is not None and not (out_f32 or s2d):
        return ops.conv_fwd_bf16(x, wp, k, cin, cout, scale=fold[0], shift=fold[1], leaky=True, pool=pool, out=out, ldy=ldo,
                                 out_col=col, split_in=x3, split_out=x3)
    # float32 rows -- normalised (inference) or conv + bias (batch statistics) -- then one pass that normalises them (batch
    # statistics), compacts the padded rows, pools and / or scatters them space-to-depth into `out`
    ld = raw_ld(cout)
    assert raw is None or tuple(raw.shape) == (N * H * W, ld)
    batch = fold is None
    scale, shift = (None, bias) if batch else fold
    raw = ops.conv_fwd_bf16(x, wp, k, cin, cout, scale=scale, shift=shift, leaky=not batch, pool=False, out_f32=True, ldy=ld,
                            out=raw, split_in=x3)
    mean = scale = shift = None
    if batch:
        mean, _, scale, shift = _batch_norm(raw, cout, ld, gamma, beta, moving, stats, workspace)
    return ops.affine_leaky_pool(raw, N, H, W, cout, ldx=ld, sub=mean, scale=scale, shift=shift, leaky=batch, pool=pool,
                                 out_bf16=not out_f32, out=out, ldo=ldo, out_col=col, space_to_depth=s2d, split_out=x3)


def layer_route(L, li, x, out, pt_src=None):
    """Where layer li of create_variables' list reads and writes in the YOLOv2 graph -- the routing Yolo2Engine and
    Yolo2Trainer share.  x: the previous layer's activation; out: this layer's activation buffer (for conv2 and the
    passthrough conv: the [N,S,S,1280] concat buffer, which both fill); pt_src: the un-pooled bf16 [N,2S,2S,512] output of
    layer PASSTHROUGH_LAYER when the passthrough branch is on, else None.

    Returns dict(x, out, ldo, col, s2d, pool, pooled): conv_bn_tc's input, output and store address, and whether it pools.
    `pooled` is None, or -- layer PASSTHROUGH_LAYER -- the buffer maxpool2x2_bf16(pt_src) must fill after the layer, because
    conv_bn_tc then writes the un-pooled activation to pt_src."""
    r = dict(x=x, out=out, ldo=None, col=0, s2d=False, pool=L['pool'], pooled=None)
    if pt_src is None:
        return r
    role = L.get('role')
    if li == PASSTHROUGH_LAYER:
        r.update(out=pt_src, pool=False, pooled=out)
    elif role == 'conv2':                            # channels [0, 1024) of the concat
        r.update(ldo=out.shape[-1])
    elif role == 'passthrough':                      # space_to_depth(2) into channels [1024, 1280) of the concat
        r.update(x=pt_src, ldo=out.shape[-1], col=out.shape[-1] - 4 * L['cout'], s2d=True)
    return r


# ---------------------------------------------------------------------------------------------
# builders (darknet.py:126-201)
# ---------------------------------------------------------------------------------------------
class _variable_scope:
    """tf.variable_scope(scope, default, [inputs], reuse=reuse) for the reference's UNNAMED variables (tf.Variable(initial),
    darknet.py:12,17), whose names come from the name scope: entering the same scope a second time without reuse opens
    `<scope>_1/` in TF (so a second darknet19_core call creates darknet19_1/Variable, ...), and so it does here.
    reuse=True replays the auto-generated names of the first pass so that the existing variables are found (the
    drop-in scripts build once, restore the checkpoint, then run with reuse=True)."""

    def __init__(self, name, reuse=None):
        self.name, self.reuse = name, reuse
        self.store = default_store()

    def __enter__(self):
        name = self.name
        if not self.reuse:
            uses = self.store.__dict__.setdefault('_scope_uses', {})
            full = (self.store._prefix(), name)
            k = uses.get(full, 0)
            uses[full] = k + 1
            if k:
                name = '%s_%d' % (name, k)
        self.ctx = self.store.scope(name)
        self.ctx.__enter__()
        if self.reuse:
            prefix = self.store._prefix()
            for key in [k for k in self.store._counters if k[0] == prefix or k[0].startswith(prefix + '/')]:
                del self.store._counters[key]
        return self

    def __exit__(self, *exc):
        return self.ctx.__exit__(*exc)


def space_to_depth(x, block_size=2):
    """tf.space_to_depth on NHWC (the YOLOv2 reorg layer; absent from the reference, SURVEY Appendix A).  Pure data
    movement, done with torch views here; the batch engine folds it into the producer's store address instead."""
    assert block_size == 2
    n, h, w, c = x.shape
    return x.reshape(n, h // 2, 2, w // 2, 2, c).permute(0, 1, 3, 2, 4, 5).reshape(n, h // 2, w // 2, 4 * c).contiguous()


def darknet19_core(inputs, num_classes=None, is_training=True, global_pool=True, output_stride=None, reuse=None,
                   scope='darknet19', return_passthrough=False):
    """darknet.py:126-179.  `num_classes`, `global_pool`, `output_stride` are accepted and ignored,
    exactly like the reference.  Fully convolutional: 224 -> 7x7, 416 -> 13x13, 608 -> 19x19.

    return_passthrough=True (extension; default reproduces the reference) also returns the un-pooled 26x26x512
    output of layer 13 (darknet.py:170), the source of the YOLOv2 passthrough branch: -> (net, passthrough)."""
    net = inputs
    pt = None
    if return_passthrough and cfg.COMPUTE == 'bf16x3':
        raise NotImplementedError('the passthrough branch has no bf16x3 path yet')
    with _variable_scope(scope, reuse=reuse):
        for li, (k, cin, cout, pool) in enumerate(CORE_PLAN):
            if return_passthrough and li == PASSTHROUGH_LAYER:
                pt = conv_bn_layer(net, k, cin, cout, 1, is_training)
                net = ops.maxpool2x2_bf16(pt) if pt.dtype == torch.bfloat16 else max_pool(pt, 2, 2)
            else:
                net = conv_bn_layer(net, k, cin, cout, 1, is_training, _pool=pool)
    return (net, pt) if return_passthrough else net


def darknet19(inputs, num_classes=None, is_training=True, global_pool=True, output_stride=None, reuse=None,
              scope='darknet19'):
    """darknet.py:61-123, the ImageNet classifier: the 18 core layers, a 19th conv_bn_layer (1x1, 1024 -> 1000) in the SAME
    variable scope (so its variables continue the core's numbering: Variable_36/37, batch_normalization_18), the 7x7 average
    pool (darknet.py:116) and the reshape to [N, 1000].  224x224 input only, like the reference (7x7 final map)."""
    net = inputs
    with _variable_scope(scope, reuse=reuse):
        for (k, cin, cout, pool) in CORE_PLAN:
            net = conv_bn_layer(net, k, cin, cout, 1, is_training, _pool=pool)
        k, cin, cout, _ = classifier_plan()
        net = conv_bn_layer(net, k, cin, cout, 1, is_training, _out_f32=(cfg.COMPUTE == 'bf16x3'))
        assert net.shape[1] == 7 and net.shape[2] == 7, 'darknet19 classifier expects a 224x224 input (darknet.py:116)'
        logits = avg_pool(net, 7, 7).reshape(-1, cout)
    return logits


def darknet19_detection(net, output_filter, is_training=True, scope='darknet19_detection', reuse=None,
                        passthrough=None, passthrough_filters=64):
    """darknet.py:182-201: conv1..conv3 (3x3, 1024->1024) + output (1x1 -> output_filter), every
    layer conv+BN+leaky, `is_training` defaulting to True (so the head normalises with batch
    statistics unless the caller says otherwise -- the reference's scripts never do).

    passthrough (extension, SURVEY Appendix A; default None = the reference's graph): the 26x26x512 tensor from
    darknet19_core(return_passthrough=True).  It goes through a 1x1 conv_bn_layer (scope `passthrough`, 512 ->
    passthrough_filters), space_to_depth(2), and is concatenated after conv2's 1024 channels; conv3 then takes
    1024 + 4*passthrough_filters input channels."""
    filters = 0 if passthrough is None else passthrough_filters
    with _variable_scope(scope, reuse=reuse):
        for sc, k, cin, cout in head_plan(output_filter, filters):
            with _variable_scope(sc):
                if sc == 'conv2' and filters:
                    # conv2's 1024 channels and the reorganised passthrough's 4 * filters share ONE [N,S,S,cat] tensor: the
                    # concat and tf.space_to_depth are the two producers' store addresses (as in the batch engine), never a copy
                    N, S, cat = int(net.shape[0]), int(net.shape[1]), cout + 4 * filters
                    buf = torch.empty((N, S, S, cat), dtype=torch.float32 if cfg.COMPUTE == 'fp32' else torch.bfloat16,
                                      device=net.device)
                    conv_bn_layer(net, k, cin, cout, 1, is_training, _out=buf, _ldo=cat)
                    net = buf
                elif sc == 'passthrough':
                    conv_bn_layer(passthrough, k, cin, cout, 1, is_training, _out=net, _ldo=cat, _col=1024, _s2d=True)
                else:
                    net = conv_bn_layer(net, k, cin, cout, 1, is_training, _out_f32=sc == 'output')
    return net
