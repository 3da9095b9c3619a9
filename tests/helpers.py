"""Shared test helpers: move variables between the product's VariableStore and the oracle; the inputs and the element check
of the full-size layer-by-layer tests (test_training_fullres_gpu.py, test_inference_fullres_gpu.py)."""
import os

import numpy as np
import torch

from tensorflow_yolo2_b200.engine import create_classifier_variables, create_variables
from tensorflow_yolo2_b200.variables import VariableStore, _to_numpy


def make_store(output_filter, seed=0, tame=False, passthrough=False, classifier=False):
    """Variables in the reference's order/naming.  tame=True rescales W to He-init magnitude
    (sqrt(2/fan_in)) so activations stay O(1) instead of exploding to 1e9+ (SURVEY 8d, config 1)."""
    st = VariableStore(seed=seed)
    layers = (create_classifier_variables(st, output_filter) if classifier      # darknet19 classifier: 18 core layers + logits conv
              else create_variables(st, output_filter, passthrough=passthrough))
    if tame:
        rs = np.random.RandomState(seed + 1)
        for L in layers:
            fan_in = L['k'] * L['k'] * L['cin']
            st[L['W']] = (st[L['W']] * (np.sqrt(2.0 / fan_in) / 0.1)).astype(np.float32)
            st[L['b']] = (rs.randn(L['cout']) * 0.1).astype(np.float32)
            bn = L['bn']
            st[bn['gamma']] = rs.uniform(0.5, 1.5, L['cout']).astype(np.float32) * np.where(rs.rand(L['cout']) < 0.2, -1, 1).astype(np.float32)
            st[bn['beta']] = (rs.randn(L['cout']) * 0.2).astype(np.float32)
            st[bn['moving_mean']] = (rs.randn(L['cout']) * 0.2).astype(np.float32)
            st[bn['moving_variance']] = rs.uniform(0.5, 2.0, L['cout']).astype(np.float32)
    return st, layers


def oracle_params(st, layers, with_passthrough=False):
    """-> (core, head) parameter lists for the oracle; with_passthrough=True -> (core, head, passthrough_params)."""
    core, head, pt = [], [], None
    for L in layers:
        bn = L['bn']
        g = lambda n: torch.tensor(_to_numpy(st[n]))
        p = dict(W=g(L['W']), b=g(L['b']), gamma=g(bn['gamma']), beta=g(bn['beta']), mm=g(bn['moving_mean']),
                 mv=g(bn['moving_variance']))
        if L.get('role') == 'passthrough':
            pt = p
        else:
            (head if L['head'] else core).append(p)
    return (core, head, pt) if with_passthrough else (core, head)


def rel_l2(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30))


# ---- full-size layer-by-layer checks -------------------------------------------------------------------------------------
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
TAU = 1e-5                       # float32 accumulation error of a bf16 convolution, relative to absref
REL_L2_BF16 = 2.0 ** -8          # twice the worst relative rounding error of a bf16 output
REL_L2_ELEM = 0.25               # float32 outputs: RMS error <= a quarter of the RMS element bound
# A bf16x3 value v (float32) is stored as hi = bf16(v), lo = bf16(v - hi).  bf16 keeps 8 significant bits, so rounding to
# nearest moves a value by at most half an ulp, i.e. by at most 2^-8 of its magnitude: |v - hi| <= 2^-8 |v|.  v - hi is exact
# in float32 (it is the low 16 bits of v's 24-bit significand), so |v - hi - lo| <= 2^-8 |v - hi| <= 2^-16 |v| -- as long as
# lo is a normal bf16 number (|v| >= 2^-110 or so; see test_split_hi_lo_representation_bound).
SPLIT_REPR = 2.0 ** -16


def split_hi_lo(v):
    """float32 -> (hi, lo) bf16, the way the kernels store a bf16x3 value (split8_bf16, pack_weights_split_kernel)."""
    v = v.float()
    hi = v.to(torch.bfloat16)
    return hi, (v - hi.float()).to(torch.bfloat16)


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


def _ulp(x, bits):
    """Spacing of a float format with `bits` significant bits at |x| (0 at x == 0)."""
    _, e = torch.frexp(x)
    return torch.where(x == 0, torch.zeros_like(x), torch.ldexp(torch.ones_like(x), e - bits))


def _rel_l2(got, ref):
    return float(torch.linalg.vector_norm(got.double() - ref) / torch.linalg.vector_norm(ref).clamp_min(1e-300))


def _check(tag, got, ref, absref, bf16_out, tau=TAU, split_out=False):
    """Every element within ulp_out(ref)/2 + tau * absref; rel-L2 within 2^-8 for bf16 outputs, and for float32 outputs
    within a quarter of the element bound's own rel-L2 (float32 results carry cancellation: |ref| << absref).
    split_out: `got` is a bf16x3 output re-joined (hi + lo): its representation error is SPLIT_REPR * |v| instead of half a
    bf16 ulp, and its rel-L2 is held to a quarter of the element bound's, as for float32 outputs."""
    got, ref = got.double(), ref.double()
    bound = tau * absref.double()
    if split_out:
        bound = bound + SPLIT_REPR * (ref.abs() + bound)          # |v| <= |ref| + tau * absref
    elif bf16_out:
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
    limit = REL_L2_BF16 if bf16_out and not split_out else REL_L2_ELEM * _rel_l2(ref + bound, ref)
    assert rl <= limit, '%s: rel-L2 %.3g > %.3g' % (tag, rl, limit)
