"""Thin torch-tensor front end over the C ABI (include/yolo2_b200.h).

torch is plumbing here: device memory, streams.  Every function enqueues on the current torch
CUDA stream and raises (never falls back) if a tensor is not a contiguous CUDA tensor of the
expected dtype or if the library call fails.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from ._lib import ConvParams, Y2_CONV_LEAKY, Y2_CONV_POOL2, Y2_CONV_OUT_F32, Y2_CONV_IN_SPLIT, Y2_CONV_OUT_SPLIT, check

ALPHA = 0.1        # yolo2_nets/darknet.py:5
BN_EPS = 1e-3      # tf.layers.batch_normalization default
BN_MOMENTUM = 0.99


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t, dtype=None):
    if t is None:
        return None
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise _lib.Y2Error('expected a CUDA tensor (no CPU fallback exists)')
    if not t.is_contiguous():
        raise _lib.Y2Error('expected a contiguous tensor')
    if dtype is not None and t.dtype != dtype:
        raise _lib.Y2Error('expected dtype %s, got %s' % (dtype, t.dtype))
    return C.c_void_p(t.data_ptr())


def launch_count():
    return int(_lib.load().y2_launch_count())


# ---- a10 -----------------------------------------------------------------------------------
def preprocess_u8(img_u8, bf16c8=True, out=None):
    """[N,H,W,3] uint8 BGR (already resized) -> (x/255)*2-1 as bf16 [N,H,W,8] or f32 [N,H,W,3]."""
    N, H, W, c = img_u8.shape
    assert c == 3
    if out is None:
        out = torch.empty((N, H, W, 8), dtype=torch.bfloat16, device=img_u8.device) if bf16c8 else \
            torch.empty((N, H, W, 3), dtype=torch.float32, device=img_u8.device)
    check(_lib.load().y2_preprocess_u8(_p(img_u8, torch.uint8), _p(out), N, H, W, 1 if bf16c8 else 0, _stream()),
          'y2_preprocess_u8')
    return out


def resize_bilinear_u8(img_u8, dst_h, dst_w, out=None):
    """cv2.resize(img, (dst_w, dst_h)) of an 8-bit BGR image [H,W,3] on the GPU, bit-exact (INTER_LINEAR fixed point)."""
    H, W, c = img_u8.shape
    assert c == 3
    if out is None:
        out = torch.empty((dst_h, dst_w, 3), dtype=torch.uint8, device=img_u8.device)
    assert tuple(out.shape) == (dst_h, dst_w, 3)
    check(_lib.load().y2_resize_bilinear_u8(_p(img_u8, torch.uint8), H, W, _p(out, torch.uint8), dst_h, dst_w, _stream()),
          'y2_resize_bilinear_u8')
    return out


def pad_cast_f32_to_bf16c8(x, out=None):
    N, H, W, c = x.shape
    assert c == 3
    if out is None:
        out = torch.empty((N, H, W, 8), dtype=torch.bfloat16, device=x.device)
    check(_lib.load().y2_pad_cast_f32_to_bf16c8(_p(x, torch.float32), _p(out, torch.bfloat16), N, H, W, _stream()),
          'y2_pad_cast_f32_to_bf16c8')
    return out


# ---- a1 ------------------------------------------------------------------------------------
def conv_fwd_f32(x, w_hwio, bias, out=None):
    N, H, W, Cin = x.shape
    k, k2, cin2, Cout = w_hwio.shape
    assert k == k2 and cin2 == Cin
    if out is None:
        out = torch.empty((N, H, W, Cout), dtype=torch.float32, device=x.device)
    check(_lib.load().y2_conv_fwd_f32(_p(x, torch.float32), _p(w_hwio, torch.float32), _p(bias, torch.float32),
                                      _p(out, torch.float32), N, H, W, Cin, Cout, k, _stream()), 'y2_conv_fwd_f32')
    return out


def conv_cin_padded(cin):
    return int(_lib.load().y2_conv_cin_padded(cin))


def pack_weights_bf16(w_hwio, out=None):
    k, _, Cin, Cout = w_hwio.shape
    n = int(_lib.load().y2_conv_packed_weight_elems(k, Cin, Cout))
    if out is None:
        out = torch.empty((n,), dtype=torch.bfloat16, device=w_hwio.device)
    assert out.numel() >= n
    check(_lib.load().y2_pack_weights_bf16(_p(w_hwio, torch.float32), _p(out), k, Cin, Cout, _stream()),
          'y2_pack_weights_bf16')
    return out


def pack_weights_bf16_split(w_hwio, out=None):
    """bf16x3 operand of conv_fwd_bf16(split_in=True): per tap [w_hi | w_hi | w_lo] (include/yolo2_b200.h)."""
    k, _, Cin, Cout = w_hwio.shape
    n = int(_lib.load().y2_conv_packed_weight_split_elems(k, Cin, Cout))
    if out is None:
        out = torch.empty((n,), dtype=torch.bfloat16, device=w_hwio.device)
    assert out.numel() >= n
    check(_lib.load().y2_pack_weights_bf16_split(_p(w_hwio, torch.float32), _p(out), k, Cin, Cout, _stream()),
          'y2_pack_weights_bf16_split')
    return out


def conv_fwd_bf16(x, w_packed, ksize, cin, cout, scale=None, shift=None, leaky=True, pool=False, out_f32=False,
                  ldy=None, out=None, alpha=ALPHA, out_col=0, split_in=False, split_out=False, lo_off=0):
    """x bf16 [N,H,W,Cin_p]; returns bf16 [N,Ho,Wo,Cout] or (out_f32) f32 [N*H*W, ldy].
    bf16x3 mode: split_in -> x is [N,H,W,2*Cin] = [hi | lo] and w_packed comes from pack_weights_bf16_split;
    split_out -> the bf16 result is [N,Ho,Wo,2*Cout] = [hi | lo] (lo at column lo_off or Cout of a row of stride ldy)."""
    N, H, W, cin_p = x.shape
    assert cin_p == (2 * cin if split_in else conv_cin_padded(cin)), (cin_p, cin, split_in)
    _ensure_conv_workspace(x.device)
    split_out = bool(split_out) and not out_f32
    flags = (Y2_CONV_LEAKY if leaky else 0) | (Y2_CONV_POOL2 if pool else 0) | (Y2_CONV_OUT_F32 if out_f32 else 0) | \
        (Y2_CONV_IN_SPLIT if split_in else 0) | (Y2_CONV_OUT_SPLIT if split_out else 0)
    ld = int(ldy) if ldy else (2 * cout if split_out else cout)
    Ho, Wo = (H // 2, W // 2) if pool else (H, W)
    if out is None:
        if out_f32:
            out = torch.empty((N * Ho * Wo, ld), dtype=torch.float32, device=x.device)
        else:
            assert ld == (2 * cout if split_out else cout)
            out = torch.empty((N, Ho, Wo, ld), dtype=torch.bfloat16, device=x.device)
    prm = ConvParams(x=_p(x, torch.bfloat16), w_packed=_p(w_packed, torch.bfloat16), scale=_p(scale, torch.float32),
                     shift=_p(shift, torch.float32), y=_p_off(out, out_col), N=N, H=H, W=W, Cin=cin, Cout=cout, ksize=ksize,
                     flags=flags, alpha=alpha, ldy=ld, lo_off=int(lo_off) if split_out else 0)
    check(_lib.load().y2_conv_fwd_bf16(C.byref(prm), _stream()), 'y2_conv_fwd_bf16')
    return out


import contextlib as _contextlib
import threading as _threading

_conv_ws = {}
_tls = _threading.local()


def new_conv_workspace(device=None):
    """A fresh, zero-filled stream-K scratch buffer (hand-over flags + partial accumulators) for y2_conv_fwd_bf16.  The
    kernels leave the flags zero after every launch, so one buffer serves any number of launches -- as long as they are
    serialised: launches that may run CONCURRENTLY (different streams, an engine next to a trainer) need different buffers."""
    device = torch.device(device) if device is not None else torch.device('cuda', torch.cuda.current_device())
    with torch.cuda.device(device):
        return torch.zeros((int(_lib.load().y2_conv_workspace_bytes()),), dtype=torch.uint8, device=device)


def _register_conv_workspace(ws):
    """The C ABI keeps the registered scratch per calling thread."""
    key = None if ws is None else (ws.data_ptr(), ws.numel())
    if getattr(_tls, 'conv_ws_key', False) != key:
        check(_lib.load().y2_conv_set_workspace(_p(ws), ws.numel() if ws is not None else 0), 'y2_conv_set_workspace')
        _tls.conv_ws_key = key


def conv_workspace(device=None):
    """The default scratch of the calling context: one zero-filled buffer per (device, stream), registered for the thread."""
    device = torch.device(device) if device is not None else torch.device('cuda', torch.cuda.current_device())
    key = (device, torch.cuda.current_stream(device).cuda_stream)
    ws = _conv_ws.get(key)
    if ws is None:
        ws = new_conv_workspace(device)
        _conv_ws[key] = ws
    _register_conv_workspace(ws)
    return ws


@_contextlib.contextmanager
def conv_workspace_scope(ws):
    """Issue the convolutions of the block with `ws` (from new_conv_workspace) as their scratch -- an engine or a trainer
    owns one, whatever stream (or CUDA-graph capture) it is enqueued on."""
    prev = getattr(_tls, 'conv_ws_pinned', None)
    _tls.conv_ws_pinned = ws
    _register_conv_workspace(ws)
    try:
        yield ws
    finally:
        _tls.conv_ws_pinned = prev
        if prev is not None:
            _register_conv_workspace(prev)


def reload_env():
    """Re-read the Y2_* environment switches of the launchers (they are cached once per process)."""
    check(_lib.load().y2_reload_env(), 'y2_reload_env')


def _ensure_conv_workspace(device):
    if getattr(_tls, 'conv_ws_pinned', None) is not None:
        _register_conv_workspace(_tls.conv_ws_pinned)
    else:
        conv_workspace(device)


def pack_weights_conv1_u8(w_hwio, scale=None, out=None):
    """First-layer weights [3,3,3,32] (TF HWIO) with the BN scale folded in -> operand of conv1_u8_pool."""
    assert tuple(w_hwio.shape) == (3, 3, 3, 32), 'the fused first layer is Darknet19\'s 3x3 3->32 conv'
    n = int(_lib.load().y2_conv1_u8_packed_weight_elems())
    if out is None:
        out = torch.empty((n,), dtype=torch.bfloat16, device=w_hwio.device)
    check(_lib.load().y2_pack_weights_conv1_u8(_p(w_hwio, torch.float32), _p(scale, torch.float32), _p(out), _stream()),
          'y2_pack_weights_conv1_u8')
    return out


def pack_weights_conv1_u8_split(w_hwio, scale=None, out=None):
    """bf16x3 operand of conv1_u8_pool(split=True): hi + lo halves of the weights with x = v*2/255 - 1 folded in."""
    assert tuple(w_hwio.shape) == (3, 3, 3, 32), 'the fused first layer is Darknet19\'s 3x3 3->32 conv'
    n = 2 * int(_lib.load().y2_conv1_u8_packed_weight_elems())
    if out is None:
        out = torch.empty((n,), dtype=torch.bfloat16, device=w_hwio.device)
    check(_lib.load().y2_pack_weights_conv1_u8_split(_p(w_hwio, torch.float32), _p(scale, torch.float32), _p(out), _stream()),
          'y2_pack_weights_conv1_u8_split')
    return out


def conv1_u8_pool(img_u8, w_packed_c1, shift, out=None, alpha=ALPHA, split=False):
    """uint8 [N,H,W,3] BGR -> bf16 [N,H/2,W/2,32]: preprocessing + conv1 + BN(scale folded, +shift) + leaky + pool.
    split=True (bf16x3): w_packed_c1 from pack_weights_conv1_u8_split, result [N,H/2,W/2,64] = [hi | lo]."""
    N, H, W, c = img_u8.shape
    assert c == 3
    if out is None:
        out = torch.empty((N, H // 2, W // 2, 64 if split else 32), dtype=torch.bfloat16, device=img_u8.device)
    fn = _lib.load().y2_conv1_u8_pool_fwd_split if split else _lib.load().y2_conv1_u8_pool_fwd
    check(fn(_p(img_u8, torch.uint8), _p(w_packed_c1, torch.bfloat16), _p(shift, torch.float32), _p(out, torch.bfloat16),
             N, H, W, alpha, _stream()), 'y2_conv1_u8_pool_fwd')
    return out


# ---- a2 / a3 -------------------------------------------------------------------------------
_ws_cache = {}


def _workspace(nbytes, device):
    key = (device, torch.cuda.current_stream().cuda_stream)
    ws = _ws_cache.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty((max(int(nbytes), 1 << 16),), dtype=torch.uint8, device=device)
        _ws_cache[key] = ws
    return ws


def bn_stats_workspace_bytes(M, C_):
    return int(_lib.load().y2_bn_stats_workspace_bytes(M, C_))


def bn_stats(x2d, C_, ld=None, workspace=None, mean=None, var=None):
    """x2d f32 [M, ld]; returns (mean[C], biased var[C])."""
    M = x2d.shape[0]
    ld = ld or x2d.shape[1]
    lib = _lib.load()
    need = int(lib.y2_bn_stats_workspace_bytes(M, C_))
    ws = workspace if workspace is not None else _workspace(need, x2d.device)
    if mean is None:
        mean = torch.empty((C_,), dtype=torch.float32, device=x2d.device)
    if var is None:
        var = torch.empty((C_,), dtype=torch.float32, device=x2d.device)
    check(lib.y2_bn_stats(_p(x2d, torch.float32), M, C_, ld, _p(mean), _p(var), _p(ws), ws.numel(), _stream()),
          'y2_bn_stats')
    return mean, var


def bn_stats_fold(x2d, C_, gamma, beta, ld=None, workspace=None, mean=None, var=None, scale=None, shift=None, eps=BN_EPS):
    """bn_stats + the folded affine of the centred form y = (x - mean) * scale + shift, in the same two launches.
    Returns (mean, var, scale, shift)."""
    M = x2d.shape[0]
    ld = ld or x2d.shape[1]
    lib = _lib.load()
    need = int(lib.y2_bn_stats_workspace_bytes(M, C_))
    ws = workspace if workspace is not None else _workspace(need, x2d.device)
    new = lambda: torch.empty((C_,), dtype=torch.float32, device=x2d.device)
    mean = new() if mean is None else mean
    var = new() if var is None else var
    scale = new() if scale is None else scale
    shift = new() if shift is None else shift
    check(lib.y2_bn_stats_fold(_p(x2d, torch.float32), M, C_, ld, _p(mean), _p(var), _p(gamma, torch.float32),
                               _p(beta, torch.float32), eps, _p(scale), _p(shift), _p(ws), ws.numel(), _stream()),
          'y2_bn_stats_fold')
    return mean, var, scale, shift


def bn_stats_fold_train(x2d, C_, gamma, beta, moving_mean, moving_var, ld=None, workspace=None, mean=None, var=None, scale=None,
                        shift=None, eps=BN_EPS, momentum=BN_MOMENTUM):
    """bn_stats_fold + the moving-average update (UPDATE_OPS) in the same two launches."""
    M = x2d.shape[0]
    ld = ld or x2d.shape[1]
    lib = _lib.load()
    need = int(lib.y2_bn_stats_workspace_bytes(M, C_))
    ws = workspace if workspace is not None else _workspace(need, x2d.device)
    check(lib.y2_bn_stats_fold_train(_p(x2d, torch.float32), M, C_, ld, _p(mean), _p(var), _p(gamma, torch.float32),
                                     _p(beta, torch.float32), eps, _p(scale), _p(shift), _p(moving_mean, torch.float32),
                                     _p(moving_var, torch.float32), momentum, _p(ws), ws.numel(), _stream()),
          'y2_bn_stats_fold_train')
    return mean, var, scale, shift


def bn_fold(gamma, beta, mean, var, conv_bias=None, eps=BN_EPS, scale=None, shift=None):
    C_ = gamma.numel()
    if scale is None:
        scale = torch.empty((C_,), dtype=torch.float32, device=gamma.device)
    if shift is None:
        shift = torch.empty((C_,), dtype=torch.float32, device=gamma.device)
    check(_lib.load().y2_bn_fold(_p(gamma, torch.float32), _p(beta, torch.float32), _p(mean, torch.float32),
                                 _p(var, torch.float32), _p(conv_bias, torch.float32), eps, _p(scale), _p(shift),
                                 C_, _stream()), 'y2_bn_fold')
    return scale, shift


def bn_update_moving(mm, mv, mean, var, momentum=BN_MOMENTUM):
    check(_lib.load().y2_bn_update_moving(_p(mm, torch.float32), _p(mv, torch.float32), _p(mean, torch.float32),
                                          _p(var, torch.float32), momentum, mm.numel(), _stream()),
          'y2_bn_update_moving')


def _p_off(t, col):
    """Pointer to channel `col` of the first row of a contiguous tensor (a channel slice of a concatenated buffer)."""
    base = _p(t)
    return C.c_void_p(base.value + int(col) * t.element_size()) if col else base


def affine_leaky_pool(x, N, H, W, C_, ldx=None, sub=None, scale=None, shift=None, leaky=True, pool=False,
                      out_bf16=False, alpha=ALPHA, out=None, ldo=None, out_col=0, space_to_depth=False, split_out=False,
                      lo_off=0):
    """x f32 rows [N*H*W, ldx] (or [N,H,W,C]); y = leaky((x-sub)*scale+shift), optional 2x2 pool.
    ldo / out_col: write into channels [out_col, out_col+C) of rows of stride ldo (`out` = the whole wider tensor);
    space_to_depth: the passthrough reorg (block 2) folded into the store address (out = [N,H/2,W/2,ldo])."""
    ldx = ldx or C_
    Ho, Wo = (H // 2, W // 2) if pool else (H, W)
    split_out = bool(split_out) and out_bf16          # bf16x3: [hi | lo] rows (lo at column lo_off, default C / ldo/2)
    if out is None:
        assert not ldo and not space_to_depth
        out = torch.empty((N, Ho, Wo, 2 * C_ if split_out else C_), dtype=torch.bfloat16 if out_bf16 else torch.float32,
                          device=x.device)
    assert out.dtype == (torch.bfloat16 if out_bf16 else torch.float32)
    check(_lib.load().y2_affine_leaky_pool_ex(_p(x, torch.float32), ldx, _p(sub, torch.float32), _p(scale, torch.float32),
                                              _p(shift, torch.float32), alpha, 1 if leaky else 0, 1 if pool else 0,
                                              _p_off(out, out_col), 2 if split_out else (1 if out_bf16 else 0),
                                              int(ldo or (2 * C_ if split_out else C_)), 1 if space_to_depth else 0,
                                              int(lo_off) if split_out else 0, N, H, W, C_, _stream()),
          'y2_affine_leaky_pool_ex')
    return out


def maxpool2x2_bf16(x, out=None):
    """bf16 [N,H,W,C] -> [N,H/2,W/2,C] (darknet.py:24-25) for the layer whose un-pooled output is the passthrough source."""
    N, H, W, C_ = x.shape
    if out is None:
        out = torch.empty((N, H // 2, W // 2, C_), dtype=torch.bfloat16, device=x.device)
    check(_lib.load().y2_maxpool2x2_bf16(_p(x, torch.bfloat16), _p(out, torch.bfloat16), N, H, W, C_, _stream()),
          'y2_maxpool2x2_bf16')
    return out


def avg_pool(x, k):
    """[N,H,W,C] bf16 or f32 -> f32 [N,H/k,W/k,C]: k x k / stride k average pool (darknet.py:28-29,116)."""
    N, H, W, C_ = x.shape
    assert H % k == 0 and W % k == 0
    if x.dtype not in (torch.float32, torch.bfloat16):
        x = x.float()
    x = x.contiguous()
    out = torch.empty((N, H // k, W // k, C_), dtype=torch.float32, device=x.device)
    check(_lib.load().y2_avgpool(_p(x), 1 if x.dtype == torch.bfloat16 else 0, _p(out), N, H, W, C_, k, _stream()), 'y2_avgpool')
    return out


def cast(x, dtype):
    """float32 <-> bfloat16 through y2_cast (the builders' dtype plumbing; no library kernel on the path)."""
    if x.dtype == dtype:
        return x
    code = {torch.float32: 0, torch.bfloat16: 1}
    if x.dtype not in code or dtype not in code:
        raise _lib.Y2Error('cast: only float32 <-> bfloat16')
    x = x if x.is_contiguous() else x.contiguous()
    out = torch.empty(x.shape, dtype=dtype, device=x.device)
    check(_lib.load().y2_cast(_p(x), code[x.dtype], _p(out), code[dtype], x.numel(), _stream()), 'y2_cast')
    return out


def scale_by_device_scalar(x, scalar, out=None):
    """x * scalar with the scalar (a 0-d / 1-element float32 CUDA tensor) read on the device."""
    if out is None:
        out = torch.empty_like(x)
    check(_lib.load().y2_scale_by_device_scalar(_p(x, torch.float32), _p(scalar.reshape(1), torch.float32), _p(out, torch.float32),
                                                x.numel(), _stream()), 'y2_scale_by_device_scalar')
    return out


# ---- a8 / a' -------------------------------------------------------------------------------
def decode_ref_v1(net, S, B, C_, thresh=0.5):
    N = net.shape[0]
    assert net.numel() == N * S * S * (C_ + 5 * B)
    dev = net.device
    boxes = torch.empty((N, S, S, B, 4), dtype=torch.float32, device=dev)
    conf = torch.empty((N, S, S, B), dtype=torch.float32, device=dev)
    keep = torch.empty((N, S, S, B), dtype=torch.uint8, device=dev)
    cls = torch.empty((N, S, S), dtype=torch.int32, device=dev)
    check(_lib.load().y2_decode_ref_v1(_p(net, torch.float32), N, S, B, C_, thresh, _p(boxes), _p(conf), _p(keep),
                                       _p(cls), _stream()), 'y2_decode_ref_v1')
    return boxes, conf, keep, cls


def decode_region(net, anchors, C_=20, thresh=0.3, boxes=None, scores=None):
    N, S = net.shape[0], net.shape[1]
    A = anchors.shape[0]
    assert net.numel() == N * S * S * A * (5 + C_)
    dev = net.device
    if boxes is None:
        boxes = torch.empty((N, S * S * A, 4), dtype=torch.float32, device=dev)
    if scores is None:
        scores = torch.empty((N, S * S * A, C_), dtype=torch.float32, device=dev)
    check(_lib.load().y2_decode_region(_p(net, torch.float32), _p(anchors, torch.float32), N, S, A, C_, thresh,
                                       _p(boxes), _p(scores), _stream()), 'y2_decode_region')
    return boxes, scores


def nms(boxes, scores, score_thresh=0.3, iou_thresh=0.45, max_keep=None, keep_idx=None, keep_count=None):
    N, nbox, _ = boxes.shape
    C_ = scores.shape[2]
    max_keep = max_keep or nbox
    dev = boxes.device
    if keep_idx is None:
        keep_idx = torch.full((N, C_, max_keep), -1, dtype=torch.int32, device=dev)
    if keep_count is None:
        keep_count = torch.empty((N, C_), dtype=torch.int32, device=dev)
    check(_lib.load().y2_nms(_p(boxes, torch.float32), _p(scores, torch.float32), N, nbox, C_, score_thresh,
                             iou_thresh, _p(keep_idx), _p(keep_count), max_keep, None, 0, _stream()), 'y2_nms')
    return keep_idx, keep_count


def detect_fused(net, anchors, C_=20, score_thresh=0.3, iou_thresh=0.45, max_keep=None, boxes=None, scores=None,
                 keep_idx=None, keep_count=None, keep_score=None, want_scores=True):
    """Region decode + per-class NMS in one kernel (one CTA per image).  Returns (boxes, scores or None, keep_idx,
    keep_count, keep_score)."""
    N, S = net.shape[0], net.shape[1]
    A = anchors.shape[0]
    nbox = S * S * A
    assert net.numel() == N * nbox * (5 + C_)
    max_keep = max_keep or nbox
    dev = net.device
    if boxes is None:
        boxes = torch.empty((N, nbox, 4), dtype=torch.float32, device=dev)
    if scores is None and want_scores:
        scores = torch.empty((N, nbox, C_), dtype=torch.float32, device=dev)
    if keep_idx is None:
        keep_idx = torch.full((N, C_, max_keep), -1, dtype=torch.int32, device=dev)
    if keep_count is None:
        keep_count = torch.empty((N, C_), dtype=torch.int32, device=dev)
    check(_lib.load().y2_detect_fused(_p(net, torch.float32), _p(anchors, torch.float32), N, S, A, C_, score_thresh,
                                      iou_thresh, _p(boxes, torch.float32), _p(scores, torch.float32),
                                      _p(keep_idx, torch.int32), _p(keep_count, torch.int32), _p(keep_score, torch.float32),
                                      max_keep, _stream()), 'y2_detect_fused')
    return boxes, scores, keep_idx, keep_count, keep_score


_detect_ws = {}


def detect_workspace_bytes(N, C_):
    return int(_lib.load().y2_detect_workspace_bytes(N, C_))


def detect_workspace(N, C_, device):
    """Zero-filled candidate-list workspace of y2_detect_split for (N, C) on `device` (cached: every call leaves it
    zero-filled again, so one buffer per shape and device serves all calls on a stream)."""
    key = (str(device), int(N), int(C_))
    ws = _detect_ws.get(key)
    if ws is None:
        need = int(_lib.load().y2_detect_workspace_bytes(N, C_))
        ws = torch.zeros((need,), dtype=torch.uint8, device=device)
        _detect_ws[key] = ws
    return ws


def detect_split(net, anchors, C_=20, score_thresh=0.3, iou_thresh=0.45, max_keep=None, boxes=None, scores=None,
                 keep_idx=None, keep_count=None, keep_score=None, want_scores=True, workspace=None):
    """Region decode + per-class NMS as two launches (chunked bulk-copy decode over the whole batch, per-image NMS over
    candidate lists) -- same results as detect_fused.  Returns (boxes, scores or None, keep_idx, keep_count, keep_score)."""
    N, S = net.shape[0], net.shape[1]
    A = anchors.shape[0]
    nbox = S * S * A
    assert net.numel() == N * nbox * (5 + C_)
    max_keep = max_keep or nbox
    dev = net.device
    if boxes is None:
        boxes = torch.empty((N, nbox, 4), dtype=torch.float32, device=dev)
    if scores is None and want_scores:
        scores = torch.empty((N, nbox, C_), dtype=torch.float32, device=dev)
    if keep_idx is None:
        keep_idx = torch.full((N, C_, max_keep), -1, dtype=torch.int32, device=dev)
    if keep_count is None:
        keep_count = torch.empty((N, C_), dtype=torch.int32, device=dev)
    ws = workspace if workspace is not None else detect_workspace(N, C_, dev)
    check(_lib.load().y2_detect_split(_p(net, torch.float32), _p(anchors, torch.float32), N, S, A, C_, score_thresh,
                                      iou_thresh, _p(boxes, torch.float32), _p(scores, torch.float32),
                                      _p(keep_idx, torch.int32), _p(keep_count, torch.int32), _p(keep_score, torch.float32),
                                      max_keep, _p(ws), ws.numel(), _stream()), 'y2_detect_split')
    return boxes, scores, keep_idx, keep_count, keep_score


# ---- a6 / a7 -------------------------------------------------------------------------------
def iou(boxes1, boxes2):
    """[..., 4] x [..., 4] (cx,cy,w,h) f32 -> [...] IoU (net_utils.get_iou arithmetic)."""
    assert boxes1.shape == boxes2.shape and boxes1.shape[-1] == 4
    out = torch.empty(boxes1.shape[:-1], dtype=torch.float32, device=boxes1.device)
    check(_lib.load().y2_iou(_p(boxes1, torch.float32), _p(boxes2, torch.float32), _p(out), out.numel(), _stream()),
          'y2_iou')
    return out


def loss_v1(net, labels, S, B, C_, image_size, lambda_coord=5.0, lambda_noobj=0.5, want_grad=True, terms=None,
            ious=None, object_mask=None, dnet=None):
    """Returns (terms[5] = class, coord, object, noobject, total; ious; object_mask; dnet)."""
    N = net.shape[0]
    dev = net.device
    lib = _lib.load()
    if terms is None:
        terms = torch.empty((5,), dtype=torch.float32, device=dev)
    if ious is None:
        ious = torch.empty((N, S, S, B), dtype=torch.float32, device=dev)
    if object_mask is None:
        object_mask = torch.empty((N, S, S, B), dtype=torch.float32, device=dev)
    if dnet is None and want_grad:
        dnet = torch.empty_like(net)
    need = int(lib.y2_loss_v1_workspace_bytes(N, S))
    ws = _workspace(need, dev)
    check(lib.y2_loss_v1_fwd_bwd(_p(net, torch.float32), _p(labels, torch.float32), N, S, B, C_, float(image_size),
                                 lambda_coord, lambda_noobj, _p(terms), _p(ious), _p(object_mask), _p(dnet), _p(ws),
                                 ws.numel(), _stream()), 'y2_loss_v1_fwd_bwd')
    return terms, ious, object_mask, dnet


def loss_v1_box_deltas(net, labels, S, B, C_, image_size, out=None):
    """[N,S,S,B,4] unmasked (dx, dy, dw, dh) of get_loss (net_utils.py:337-342) -- the histogram summaries of :366-369."""
    N = net.shape[0]
    if out is None:
        out = torch.empty((N, S, S, B, 4), dtype=torch.float32, device=net.device)
    check(_lib.load().y2_loss_v1_box_deltas(_p(net, torch.float32), _p(labels, torch.float32), N, S, B, C_, float(image_size),
                                            _p(out, torch.float32), _stream()), 'y2_loss_v1_box_deltas')
    return out


def region_loss(net, anchors, gt_boxes, gt_classes, gt_counts, C_=20, lambda_coord=1.0, lambda_obj=5.0, lambda_noobj=1.0,
                lambda_class=1.0, ignore_thresh=0.6, want_grad=True, terms=None, dnet=None):
    """YOLOv2 region loss (SURVEY Appendix A).  net f32 [N,S,S,A*(5+C)]; gt_boxes f32 [N,G,4] normalised
    (cx,cy,w,h); gt_classes int32 [N,G]; gt_counts int32 [N].  Returns (terms[5] = coord, obj, noobj, class,
    total; dnet)."""
    N, S = net.shape[0], net.shape[1]
    A = anchors.shape[0]
    G = gt_boxes.shape[1]
    assert net.numel() == N * S * S * A * (5 + C_)
    dev = net.device
    lib = _lib.load()
    if terms is None:
        terms = torch.empty((5,), dtype=torch.float32, device=dev)
    if dnet is None and want_grad:
        dnet = torch.empty_like(net)
    need = int(lib.y2_region_loss_workspace_bytes(N, S))
    ws = _workspace(need, dev)
    check(lib.y2_region_loss_fwd_bwd(_p(net, torch.float32), _p(anchors, torch.float32), _p(gt_boxes, torch.float32),
                                     _p(gt_classes, torch.int32), _p(gt_counts, torch.int32), N, S, A, C_, G,
                                     lambda_coord, lambda_obj, lambda_noobj, lambda_class, ignore_thresh, _p(terms),
                                     _p(dnet), _p(ws), ws.numel(), _stream()), 'y2_region_loss_fwd_bwd')
    return terms, dnet


# ---- a11: backward --------------------------------------------------------------------------
def bn_bwd_workspace_bytes(M, C_):
    return int(_lib.load().y2_bn_bwd_workspace_bytes(M, C_))


def bn_leaky_pool_bwd(h_raw, dy, mean, var, gamma, beta, N, H, W, C_, ldh=None, leaky=True, pool=False, ld_dh=None,
                      dgamma=None, dbeta=None, dh=None, workspace=None, alpha=ALPHA, eps=BN_EPS, ldy=None, dy_col=0,
                      dy_s2d=False, dy_add=None):
    """Backward of max_pool(leaky(batch_norm(h_raw))) (batch statistics).  dy: grad of the layer output
    [N,Ho,Wo,C] (f32 or bf16).  Returns (dgamma[C], dbeta[C], dh bf16 [N*H*W, ld_dh]).

    The defaults read dy as dense [N,Ho,Wo,C] rows.  Otherwise (y2_bn_leaky_pool_bwd_ex): dy is a wider tensor whose rows
    of stride `ldy` hold the layer's gradient from column `dy_col` on; dy_s2d=True reads it through depth_to_space(2)
    (the layer's output was stored space_to_depth(2) there: the passthrough branch); dy_add (bf16 [N,H,W,C], pooled layers)
    is the gradient of the un-pooled output from a second consumer, added to every input row before the leaky slope."""
    ldh = ldh or C_
    ld_dh = ld_dh or (C_ + 63) // 64 * 64
    dev = h_raw.device
    if dy.dtype not in (torch.float32, torch.bfloat16):
        raise _lib.Y2Error('dy must be float32 or bfloat16')
    if dgamma is None:
        dgamma = torch.empty((C_,), dtype=torch.float32, device=dev)
    if dbeta is None:
        dbeta = torch.empty((C_,), dtype=torch.float32, device=dev)
    M = N * H * W
    if dh is None:
        dh = torch.empty((M, ld_dh), dtype=torch.bfloat16, device=dev)
    assert dh.numel() >= M * ld_dh
    lib = _lib.load()
    need = int(lib.y2_bn_bwd_workspace_bytes(M, C_))
    ws = workspace if workspace is not None else _workspace(need, dev)
    args = (_p(mean, torch.float32), _p(var, torch.float32), _p(gamma, torch.float32), _p(beta, torch.float32), eps, alpha,
            1 if leaky else 0, 1 if pool else 0, N, H, W, C_, _p(dgamma, torch.float32), _p(dbeta, torch.float32),
            _p(dh, torch.bfloat16), ld_dh, _p(ws), ws.numel(), _stream())
    dy_code = 0 if dy.dtype == torch.float32 else 1
    if ldy is None and not dy_col and not dy_s2d and dy_add is None:
        check(lib.y2_bn_leaky_pool_bwd(_p(h_raw, torch.float32), ldh, _p(dy), dy_code, *args), 'y2_bn_leaky_pool_bwd')
    else:
        ldy = ldy or dy.shape[-1]
        assert dy.numel() % ldy == 0 and (dy_add is None or dy_add.numel() == M * C_)
        check(lib.y2_bn_leaky_pool_bwd_ex(_p(h_raw, torch.float32), ldh, _p_off(dy, dy_col), dy_code, int(ldy),
                                          1 if dy_s2d else 0, _p(dy_add, torch.bfloat16), *args), 'y2_bn_leaky_pool_bwd_ex')
    return dgamma, dbeta, dh


def pack_weights_dgrad_bf16(w_hwio, ld_dh, out=None):
    """Weights for the data-gradient convolution (transposed + flipped), to be used with
    conv_fwd_bf16(dh, packed, ksize, cin=ld_dh, cout=Cin, leaky=False)."""
    k, _, Cin, Cout = w_hwio.shape
    lib = _lib.load()
    n = int(lib.y2_conv_packed_weight_dgrad_elems(k, Cin, ld_dh))
    if out is None:
        out = torch.empty((n,), dtype=torch.bfloat16, device=w_hwio.device)
    assert out.numel() >= n
    check(lib.y2_pack_weights_dgrad_bf16(_p(w_hwio, torch.float32), _p(out), k, Cin, Cout, ld_dh, _stream()),
          'y2_pack_weights_dgrad_bf16')
    return out


def conv_wgrad_bf16(x, dh, ksize, cin, cout, dw):
    """dw (HWIO f32, pre-zeroed) += weight gradient; x bf16 [N,H,W,cin], dh bf16 [N*H*W, ld_dh]."""
    N, H, W, cx = x.shape
    assert cx == cin
    ld_dh = dh.shape[-1]
    check(_lib.load().y2_conv_wgrad_bf16(_p(x, torch.bfloat16), _p(dh, torch.bfloat16), ld_dh, _p(dw, torch.float32), N, H,
                                         W, cin, cout, ksize, _stream()), 'y2_conv_wgrad_bf16')
    return dw


def conv_wgrad_c3(x8, dh, cout, dw):
    """First layer: x bf16 [N,H,W,8] (3 real channels), dh bf16 [N*H*W, ld_dh]; dw [3,3,3,cout] f32 +=."""
    N, H, W, c8 = x8.shape
    assert c8 == 8
    check(_lib.load().y2_conv_wgrad_c3(_p(x8, torch.bfloat16), _p(dh, torch.bfloat16), dh.shape[-1], N, H, W, cout,
                                       _p(dw, torch.float32), _stream()), 'y2_conv_wgrad_c3')
    return dw


def sum_rows_bf16(a, C_, out):
    M, ld = a.shape
    check(_lib.load().y2_sum_rows_bf16(_p(a, torch.bfloat16), ld, M, C_, _p(out, torch.float32), _stream()),
          'y2_sum_rows_bf16')
    return out


# ---- a11 -----------------------------------------------------------------------------------
def adam_step(p, g, m, v, step, lr=1e-3, b1=0.9, b2=0.999, eps=1e-8):
    lr_t = lr * (1.0 - b2 ** step) ** 0.5 / (1.0 - b1 ** step)
    check(_lib.load().y2_adam_step(_p(p, torch.float32), _p(g, torch.float32), _p(m, torch.float32),
                                   _p(v, torch.float32), p.numel(), lr_t, b1, b2, eps, _stream()), 'y2_adam_step')


def adam_lr_t(step, lr=1e-3, b1=0.9, b2=0.999):
    """TF's AdamOptimizer step size at iteration `step` (1-based): lr * sqrt(1 - b2^t) / (1 - b1^t)."""
    return lr * (1.0 - b2 ** step) ** 0.5 / (1.0 - b1 ** step)


def adam_step_ex(p, g, m, v, lr_t=0.0, lr_t_dev=None, b1=0.9, b2=0.999, eps=1e-8, grad_scale=1.0, zero_grad=False):
    """y2_adam_step_ex: Adam with the gradient scaled on the fly, the step size optionally read from a device scalar, and the
    gradient arena cleared behind the read."""
    check(_lib.load().y2_adam_step_ex(_p(p, torch.float32), _p(g, torch.float32), _p(m, torch.float32), _p(v, torch.float32),
                                      p.numel(), float(lr_t), _p(lr_t_dev, torch.float32), b1, b2, eps, float(grad_scale),
                                      1 if zero_grad else 0, _stream()), 'y2_adam_step_ex')


def momentum_step(p, g, accum, lr, momentum, grad_scale=1.0, zero_grad=False):
    """y2_momentum_step: tf.train.MomentumOptimizer's update (imagenet_train_darknet.py:58) over a flat fp32 arena."""
    check(_lib.load().y2_momentum_step(_p(p, torch.float32), _p(g, torch.float32), _p(accum, torch.float32), p.numel(), float(lr),
                                       float(momentum), float(grad_scale), 1 if zero_grad else 0, _stream()), 'y2_momentum_step')


def softmax_xent(net, labels, want_grad=False, terms=None, logits=None, losses=None, correct=None, dnet=None):
    """y2_softmax_xent_fwd_bwd.  net: fp32 [N,H,W,C] (average-pooled over H*W first, darknet.py:116-117) or [N,C] logits;
    labels: int32 [N].  Returns dict(terms=[mean loss, accuracy], logits [N,C], losses [N], correct [N], dnet or None)."""
    assert net.dtype == torch.float32 and net.dim() in (2, 4)
    N, C = net.shape[0], net.shape[-1]
    HW = 1 if net.dim() == 2 else net.shape[1] * net.shape[2]
    f32 = dict(dtype=torch.float32, device=net.device)
    terms = torch.empty((2,), **f32) if terms is None else terms
    logits = torch.empty((N, C), **f32) if logits is None else logits
    losses = torch.empty((N,), **f32) if losses is None else losses
    correct = torch.empty((N,), **f32) if correct is None else correct
    if want_grad and dnet is None:
        dnet = torch.empty_like(net)
    assert labels.dtype == torch.int32 and labels.numel() == N
    check(_lib.load().y2_softmax_xent_fwd_bwd(_p(net, torch.float32), _p(labels, torch.int32), N, HW, C, _p(logits, torch.float32),
                                              _p(losses, torch.float32), _p(correct, torch.float32), _p(terms, torch.float32),
                                              _p(dnet, torch.float32) if dnet is not None else None, _stream()),
          'y2_softmax_xent_fwd_bwd')
    return dict(terms=terms, logits=logits, losses=losses, correct=correct, dnet=dnet)
