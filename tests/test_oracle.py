"""CPU: the oracle (oracle/yolo2_oracle.py) against (a) goldens produced by executing the
reference's own source over the TF1 shim (tests/golden/make_golden.py) and (b) the hand-derived
KATs of SURVEY.md section 8(c)."""
import os

import numpy as np
import pytest
import torch

from oracle import yolo2_oracle as O
from tensorflow_yolo2_b200.variables import VariableStore


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name), allow_pickle=False)


def test_iou_golden_and_kats(golden_dir):
    g = _load(golden_dir, 'ref_iou.npz')
    iou = O.get_iou(g['boxes1'], g['boxes2'])
    np.testing.assert_allclose(iou, g['iou'], rtol=0, atol=1e-15)
    # SURVEY 8(c) KATs
    f = lambda a, b: float(O.get_iou(np.array(a, dtype=np.float64), np.array(b, dtype=np.float64)))
    assert f([.3, .4, .2, .1], [.3, .4, .2, .1]) == pytest.approx(1.0)
    assert f([.5, .5, 1, 1], [.5, .5, .5, .5]) == pytest.approx(0.25)
    assert f([.1, .1, .1, .1], [.8, .8, .1, .1]) == 0.0
    assert f([.5, .5, .2, .2], [.6, .5, .2, .2]) == pytest.approx(1.0 / 3.0)
    assert f([.5, .5, 0, 0], [.5, .5, .3, .3]) == 0.0


def test_label_encoder_golden(golden_dir):
    g = _load(golden_dir, 'ref_labels.npz')
    objs, im_h, im_w = O.parse_voc_xml(os.path.join(golden_dir, 'testImg2Anno.xml'))
    assert (im_h, im_w) == (500, 353)
    for IS, S, cells in ((224, 7, {(4, 2), (3, 3)}), (416, 13, {(7, 4), (6, 6)}), (608, 19, {(11, 6), (9, 9)})):
        lab = O.encode_labels(objs, im_h, im_w, IS, S)
        np.testing.assert_allclose(lab, g['label_%d_%d' % (IS, S)], rtol=0, atol=1e-12)
        assert {tuple(c) for c in np.argwhere(lab[..., 0] == 1)} == cells     # SURVEY 8(c)
    np.testing.assert_allclose(O.encode_labels(objs, im_h, im_w, 224, 7)[4, 2, 1:5],
                               [76.465, 136.416, 93.280, 58.688], atol=1e-3)


def test_preprocess_golden(golden_dir):
    import cv2
    g = _load(golden_dir, 'ref_labels.npz')
    im = cv2.resize(cv2.imread(os.path.join(golden_dir, 'testImg2.jpg')), (224, 224))
    np.testing.assert_array_equal(O.preprocess_u8(im), g['image_224'])


@pytest.mark.parametrize('name', ['katA', 'katB', 'katC', 'rand7', 'rand13', 'rand19'])
def test_loss_golden(golden_dir, name):
    g = _load(golden_dir, 'ref_loss.npz')
    IS, S, B = [int(v) for v in g[name + '_cfg']]
    net, lab = g[name + '_net'], g[name + '_labels']
    r = O.get_loss(net, lab, 20, net.shape[0], IS, S, B, with_grad=True)
    assert r['loss'] == pytest.approx(float(g[name + '_loss']), rel=1e-13)
    np.testing.assert_allclose(r['ious'], g[name + '_ious'], atol=1e-14)
    np.testing.assert_array_equal(r['object_mask'], g[name + '_mask'])
    if name not in ('katA', 'katB'):      # A/B sit on max/min ties where torch splits the gradient
        np.testing.assert_allclose(r['dnet'], g[name + '_dnet'], atol=1e-12)


def test_loss_survey_kats(golden_dir):
    g = _load(golden_dir, 'ref_loss.npz')
    want = {'katA': (2.0, 34.569972, 0.0, 0.0, 36.569972, 4),
            'katB': (10.0, 5.686596, 0.377669, 11.75, 27.814265, 4),
            'katC': (14.288050, 4.450934, 0.629178, 15.577960, 34.946123, 2)}
    for name, (cl, co, ob, no, tot, msum) in want.items():
        r = O.get_loss(g[name + '_net'], g[name + '_labels'], 20, 1, 224, 7, 2)
        assert r['class_loss'] == pytest.approx(cl, abs=2e-6)
        assert r['coord_loss'] == pytest.approx(co, abs=2e-6)
        assert r['object_loss'] == pytest.approx(ob, abs=2e-6)
        assert r['noobject_loss'] == pytest.approx(no, abs=2e-6)
        assert r['loss'] == pytest.approx(tot, abs=2e-6)
        assert r['object_mask'].sum() == msum
    rB = O.get_loss(g['katB_net'], g['katB_labels'], 20, 1, 224, 7, 2)
    assert rB['ious'][0, 4, 2, 0] == pytest.approx(0.47847113, abs=1e-7)
    assert rB['ious'][0, 3, 3, 0] == pytest.approx(0.06598269, abs=1e-7)


def test_loss_grad_matches_autograd():
    rs = np.random.RandomState(3)
    N, S, B = 3, 13, 5
    net = rs.uniform(-0.3, 1.1, (N, S, S, 20 + 5 * B))
    lab = np.zeros((N, S, S, 25))
    for n in range(N):
        for _ in range(3):
            i, j = rs.randint(0, S, 2)
            lab[n, i, j, 0] = 1
            lab[n, i, j, 1:5] = [(j + rs.rand()) * 32, (i + rs.rand()) * 32, rs.uniform(20, 300), rs.uniform(20, 300)]
            lab[n, i, j, 5:] = 0
            lab[n, i, j, 5 + rs.randint(20)] = 1
    r = O.get_loss(net, lab, 20, N, 416, S, B, with_grad=True)
    loss_t, g_t = O.get_loss_torch(net, lab, 20, N, 416, S, B)
    assert r['loss'] == pytest.approx(loss_t, rel=1e-13)
    np.testing.assert_allclose(r['dnet'], g_t, atol=1e-12)


@pytest.mark.parametrize('name,S,B', [('s7', 7, 2), ('s13', 13, 5)])
def test_decode_golden(golden_dir, name, S, B):
    g = _load(golden_dir, 'ref_decode.npz')
    im_w, im_h = [int(v) for v in g['im_wh']]
    dec = O.decode_ref_v1(g[name + '_pred'][0], S, B, 20, 0.5)
    draws = O.draw_list_ref_v1(dec, im_w, im_h)
    rects = np.array([d[:4] for d in draws], dtype=np.int64).reshape(-1, 4)
    np.testing.assert_array_equal(rects, g[name + '_rects'])
    texts = [O.VOC_CLASSES[d[4]] + ':' + str(np.float32(d[5])) for d in draws]
    assert texts == [str(t) for t in g[name + '_texts']]


def build_params(output_filter, seed=0):
    """Create variables in the reference's order through the product's VariableStore and hand
    them to the oracle as torch tensors."""
    st = VariableStore(seed=seed)
    core, head = [], []

    def layer(k, cin, cout):
        wn, W = st.weight_variable([k, k, cin, cout])
        bn_, b = st.bias_variable([cout])
        bn = st.batch_norm_variables(cout)
        return dict(W=torch.tensor(W), b=torch.tensor(b), gamma=torch.tensor(st[bn['gamma']]),
                    beta=torch.tensor(st[bn['beta']]), mm=torch.tensor(st[bn['moving_mean']]),
                    mv=torch.tensor(st[bn['moving_variance']]))
    with st.scope('darknet19'):
        for (k, cin, cout, pool) in O.CORE_PLAN:
            core.append(layer(k, cin, cout))
    with st.scope('darknet19_detection'):
        for sc, (k, cin, cout, pool) in zip(('conv1', 'conv2', 'conv3', 'output'), O.head_plan(output_filter)):
            with st.scope(sc):
                head.append(layer(k, cin, cout))
    return st, core, head


@pytest.mark.parametrize('name,of', [('d64_30', 30), ('d96_125', 125)])
def test_darknet_golden(golden_dir, name, of):
    g = _load(golden_dir, 'ref_darknet.npz')
    st, core, head = build_params(of)
    assert st.names() == [str(s) for s in g[name + '_varnames']]          # TF auto-naming + order
    np.testing.assert_array_equal(st['darknet19/Variable'], g[name + '_w0'].astype(np.float32))
    x = torch.tensor(g[name + '_x'])
    out, inter = O.darknet19_forward(x, core, head, core_training=False, head_training=True,
                                     dtype=torch.float64, return_intermediates=True)
    np.testing.assert_allclose(inter[17].numpy(), g[name + '_core'], rtol=1e-10)
    np.testing.assert_allclose(out.numpy(), g[name + '_out'], rtol=1e-7, atol=1e-9)


def test_darknet_training_mode_golden(golden_dir):
    g = _load(golden_dir, 'ref_darknet.npz')
    st, core, head = build_params(30)
    out, inter = O.darknet19_forward(torch.tensor(g['t32_x']), core, head, core_training=True,
                                     head_training=True, dtype=torch.float64, return_intermediates=True)
    np.testing.assert_allclose(inter[17].numpy(), g['t32_core'], rtol=1e-6, atol=1e-8)
    np.testing.assert_allclose(out.numpy(), g['t32_out'], rtol=1e-5, atol=1e-7)


def test_nms_oracle_basic():
    boxes = np.array([[.5, .5, .2, .2], [.51, .5, .2, .2], [.8, .8, .1, .1], [.5, .5, .2, .2]], dtype=np.float32)
    scores = np.array([[.9, 0], [.8, 0], [.7, .6], [.9, .5]], dtype=np.float32)
    keeps = O.nms_per_class(boxes, scores, 0.45, 0.3)
    assert keeps[0].tolist() == [0, 2]          # tie on score broken by index; 1 and 3 suppressed
    assert keeps[1].tolist() == [2, 3]


def test_region_decode_shapes():
    net = np.random.RandomState(0).randn(2, 13, 13, 125).astype(np.float32)
    boxes, sthr, s = O.region_decode_v2(net, thresh=0.3)
    assert boxes.shape == (2, 845, 4) and s.shape == (2, 845, 20)
    assert np.all(s.sum(-1) <= 1.0 + 1e-6)
    assert np.all((sthr == 0) | (sthr > 0.3))


def test_space_to_depth_matches_definition():
    """Appendix A reorg: out[n,i,j,(di*2+dj)*C + c] = x[n,2i+di,2j+dj,c] (tf.space_to_depth, block 2)."""
    import torch
    x = torch.arange(2 * 4 * 6 * 3, dtype=torch.float64).reshape(2, 4, 6, 3)
    y = O.space_to_depth2(x)
    assert y.shape == (2, 2, 3, 12)
    for n in range(2):
        for i in range(2):
            for j in range(3):
                for di in range(2):
                    for dj in range(2):
                        for c in range(3):
                            assert y[n, i, j, (di * 2 + dj) * 3 + c] == x[n, 2 * i + di, 2 * j + dj, c]


def test_avg_pool_and_classifier_shapes():
    """darknet.py:28-29,116: k x k / stride k average pool; classifier forward returns [N, 1000] logits."""
    x = torch.arange(2 * 4 * 4 * 3, dtype=torch.float64).reshape(2, 4, 4, 3)
    y = O.avg_pool_kxk(x, 2)
    assert y.shape == (2, 2, 2, 3)
    np.testing.assert_allclose(y[0, 0, 0].numpy(), x[0, :2, :2].reshape(4, 3).mean(0).numpy())
    np.testing.assert_allclose(O.avg_pool_kxk(x, 4)[1, 0, 0].numpy(), x[1].reshape(16, 3).mean(0).numpy())


def test_resize_restatement_pinned_to_cv2(golden_dir):
    """oracle.resize_bilinear_u8 restates OpenCV's fixed-point INTER_LINEAR (a third-party dependency of the reference,
    pascal_detect_darknet.py:35): bit-exact against cv2.resize on the fixtures and on random images -- up- and down-scales,
    the exact-2x INTER_AREA switch, non-square sources."""
    import cv2
    rs = np.random.RandomState(0)
    cases = [(rs.randint(0, 256, (h, w, 3)).astype(np.uint8), IS) for (h, w, IS) in
             [(240, 352, 416), (500, 353, 224), (375, 500, 608), (832, 832, 416), (100, 100, 416), (416, 416, 416),
              (1000, 750, 416), (123, 457, 224), (37, 41, 96), (448, 448, 224)]]
    for f in ('testImg1.jpg', 'testImg2.jpg'):
        im = cv2.imread(os.path.join(golden_dir, f))
        cases += [(im, IS) for IS in (224, 416, 608)]
    for im, IS in cases:
        np.testing.assert_array_equal(O.resize_bilinear_u8(im, IS, IS), cv2.resize(im, (IS, IS)))
    im = cases[0][0]
    np.testing.assert_array_equal(O.resize_bilinear_u8(im, 300, 200), cv2.resize(im, (300, 200)))     # non-square target


def test_max_pool_routes_ties_to_first_maximum():
    """max_pool_2x2's gradient goes whole to the first maximum of each window, in the order (0,0), (0,1), (1,0), (1,1), like
    the training kernels' arg-max routing (constant image regions give bit-identical pre-BN values, so exact ties are common);
    the forward value is the plain maximum."""
    x = torch.zeros((1, 4, 6, 2), dtype=torch.float64)
    wins = {(0, 0): [[5, 5], [5, 5]],          # four-way tie -> (0,0)
            (0, 1): [[1, 7], [7, 7]],          # three-way tie after the first entry -> (0,1)
            (0, 2): [[2, 3], [9, 9]],          # tie in the bottom row -> (1,0)
            (1, 0): [[-4, -4], [-4, -4]],      # negative ties
            (1, 1): [[0, 2], [1, 3]],          # no tie -> (1,1)
            (1, 2): [[6, 1], [6, 0]]}          # tie down the first column -> (0,0)
    for (i, j), w in wins.items():
        x[0, 2 * i:2 * i + 2, 2 * j:2 * j + 2, 0] = torch.tensor(w, dtype=torch.float64)
        x[0, 2 * i:2 * i + 2, 2 * j:2 * j + 2, 1] = -torch.tensor(w, dtype=torch.float64)   # channel 1: the mirror image
    x.requires_grad_(True)
    y = O.max_pool_2x2(x)
    np.testing.assert_array_equal(y.detach().numpy(), x.detach().reshape(1, 2, 2, 3, 2, 2).amax(dim=(2, 4)).numpy())
    dy = torch.arange(1, 13, dtype=torch.float64).reshape(1, 2, 3, 2)
    (y * dy).sum().backward()
    want = torch.zeros_like(x)
    xd = x.detach()
    for i in range(2):
        for j in range(3):
            for c in range(2):
                w = xd[0, 2 * i:2 * i + 2, 2 * j:2 * j + 2, c].reshape(4)
                k = int(next(k for k in range(4) if w[k] == w.max()))
                want[0, 2 * i + k // 2, 2 * j + k % 2, c] = dy[0, i, j, c]
    np.testing.assert_array_equal(x.grad.numpy(), want.numpy())
    assert want[0, 0, 0, 0] == dy[0, 0, 0, 0] and want[0, 0, 3, 0] == dy[0, 0, 1, 0] and want[0, 1, 4, 0] == dy[0, 0, 2, 0]


def test_split_hi_lo_representation_bound():
    """The bound the full-size inference test allows a bf16x3 output (tests/helpers.py SPLIT_REPR): hi + lo of split_hi_lo(v)
    is within 2^-16 |v| of v, over every binade of normal bf16 lo parts and at bf16 rounding ties of hi and of lo.  It is
    within a factor 2 of tight: lo rounds |v - hi| < 2^-8 |v| to 8 bits, so the error reaches 2^-17 |v| when lo is a tie."""
    from tests.helpers import SPLIT_REPR, split_hi_lo
    rs = np.random.RandomState(5)
    mant = rs.uniform(1.0, 2.0, 200000)
    expo = rs.randint(-100, 120, mant.size)
    v = (mant * np.exp2(expo) * rs.choice([-1.0, 1.0], mant.size)).astype(np.float32)
    bits = rs.randint(0, 1 << 23, 4096).astype(np.uint32) | np.uint32(127 << 23)
    ties = ((bits & ~np.uint32(0xFFFF)) | np.uint32(0x8000)).view(np.float32)       # exactly halfway between two bf16
    worst = ((bits & ~np.uint32(0xFFFF)) | np.uint32(0x4040)).view(np.float32)      # v - hi = 0x4040 units: lo is a tie
    v = torch.from_numpy(np.concatenate([v, ties, -ties, worst, np.float32([0.0, 1.0, -2.5, 1e38, 2.0 ** -100])]))
    hi, lo = split_hi_lo(v)
    assert hi.dtype == lo.dtype == torch.bfloat16
    assert torch.equal(hi, v.to(torch.bfloat16))
    err = (v.double() - hi.double() - lo.double()).abs()
    ratio = err / (SPLIT_REPR * v.double().abs()).clamp_min(1e-300)
    assert torch.all(err <= SPLIT_REPR * v.double().abs()), float(ratio.max())
    assert float(ratio.max()) > 0.45
