"""Training step of the reference's Pascal script on the B200 kernels.

What the reference runs per iteration (src/pascal/pascal_train_darknet.py:96-102) is one
``sess.run([loss, train_op, ious, object_mask], feed_dict)``: forward of darknet19_core +
darknet19_detection with batch-statistics batch norm in all 22 layers, the BN moving-average
UPDATE_OPS (:49-50), get_loss (:44-46), TF autodiff, and ``AdamOptimizer().minimize`` (:51, TF defaults
lr 1e-3, beta 0.9/0.999, eps 1e-8).  ``Yolo2Trainer.step`` enqueues exactly that on the current CUDA stream:

  forward   conv_tc_kernel (tcgen05) -> fp32 pre-BN rows, bn_stats, affine_leaky_pool -> bf16 activation
  loss      loss_v1 (the reference's get_loss, C+5B channels) or region_loss (YOLOv2, A*(5+C) channels): loss terms
            and d loss / d net in one kernel
  backward  per layer, last to first: y2_bn_leaky_pool_bwd -> (dgamma, dbeta, dh bf16);
            y2_conv_wgrad_bf16 (tcgen05, MN-major operands, split-K) / y2_conv_wgrad_c3 (first layer);
            data gradient = conv_tc_kernel on dh with transposed+flipped packed weights
  all-reduce (world > 1) NCCL, bucketed in reverse layer order, each bucket issued as soon as its layers'
            gradients are enqueued so it overlaps the rest of the backward pass; gradients are averaged
            (each rank's loss is the mean over its local batch, net_utils.py:296)
  update    one y2_adam_step over the flat parameter arena

Parameters, gradients and Adam moments live in flat fp32 arenas (layers in REVERSE order so that a bucket is a
contiguous slice that becomes ready early); the VariableStore entries are views into the parameter arena, so
checkpoints (net_utils.save_checkpoint) see the live weights under their TF names.
The conv bias sits in front of a batch-statistics BN, so its gradient is identically zero (TF computes rounding
noise there); it is left at exactly 0.

Yolo2Trainer(passthrough=True) trains the YOLOv2 graph instead (23 layers, the passthrough conv between conv2 and conv3, see
the constructor): the forward pass routes every layer through darknet.layer_route, as Yolo2Engine does, and the backward pass
reads each layer's incoming gradient where its consumer wrote it (dy_src).
"""
from __future__ import annotations

import numpy as np
import torch

from . import ops
from .engine import create_classifier_variables, create_variables
from .parallel import BucketedAllReduce, bucket_segments, make_buckets
from .variables import VariableStore
from .yolo2_nets.darknet import PASSTHROUGH_FILTERS, PASSTHROUGH_LAYER, conv_bn_tc, layer_route, raw_ld
from .yolo2_nets.net_utils import VOC_ANCHORS


def _round_up(v, m):
    return (v + m - 1) // m * m


class Yolo2Trainer:
    def __init__(self, batch, image_size=416, output_filter=None, store=None, loss='v1', num_class=20, B=5,
                 anchors=VOC_ANCHORS, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8, lambda_coord=None, lambda_noobj=None,
                 max_gt=32, device=None, seed=0, process_group=None, bucket_bytes=48 << 20, update_moving=True,
                 use_cuda_graph=False, optimizer='adam', momentum=0.9, passthrough=False):
        """loss: 'v1' (the reference's get_loss), 'region' (YOLOv2 region loss) or 'softmax' -- the ImageNet classifier of
        imagenet_train_darknet.py:46-58: the 18 core layers + the 1x1 conv to `num_class` logits maps + 7x7 average pool,
        sparse softmax cross-entropy (image_size 224, num_class 1000 there).  optimizer: 'adam' (pascal_train_darknet.py:51)
        or 'momentum' (tf.train.MomentumOptimizer(lr, momentum), imagenet_train_darknet.py:58).

        passthrough=True trains the YOLOv2 graph of head_plan(OF, 64) (23 layers; the detection losses only): the un-pooled
        output of layer 13 goes through a 1x1 conv (512 -> 64) whose space_to_depth(2) fills channels [1024, 1280) of a
        [N,S,S,1280] concat after conv2's 1024, and conv3 reads all 1280 -- the graph Yolo2Engine(passthrough=True) serves,
        under the same variable names.  Backward: conv3's data gradient is the [N,S,S,1280] concat gradient; conv2 reads its
        first 1024 columns in place (row stride 1280), the passthrough conv the last 256 through depth_to_space(2); the
        passthrough conv's data gradient (the un-pooled [N,2S,2S,512] `d_pt`) is added to every pre-pool row of layer 13
        inside its batch-norm backward, next to the pooled gradient of layer 14."""
        self.device = torch.device(device) if device is not None else torch.device('cuda', torch.cuda.current_device())
        self.N, self.IS = int(batch), int(image_size)
        assert self.IS % 32 == 0
        self.S = self.IS // 32
        self.C = int(num_class)
        self.loss_kind = loss
        if loss == 'v1':
            self.B = int(B)
            of = self.C + 5 * self.B                     # net_utils.py:279-285 channel layout
            self.lambda_coord = 5.0 if lambda_coord is None else lambda_coord      # config.py:44
            self.lambda_noobj = 0.5 if lambda_noobj is None else lambda_noobj      # config.py:45
        elif loss == 'region':
            self.anchors_np = np.asarray(anchors, dtype=np.float32)
            self.A = self.anchors_np.shape[0]
            of = self.A * (5 + self.C)
            self.lambda_coord = 1.0 if lambda_coord is None else lambda_coord
            self.lambda_noobj = 1.0 if lambda_noobj is None else lambda_noobj
            self.max_gt = int(max_gt)
        elif loss == 'softmax':
            of = self.C
        else:
            raise ValueError('loss must be "v1", "region" or "softmax"')
        if passthrough and loss == 'softmax':
            raise ValueError('passthrough=True is the YOLOv2 detection graph: use loss="region" or "v1"')
        self.passthrough = bool(passthrough)
        if optimizer not in ('adam', 'momentum'):
            raise ValueError('optimizer must be "adam" or "momentum"')
        self.optimizer, self.momentum = optimizer, float(momentum)
        self.OF = int(output_filter) if output_filter is not None else of
        assert self.OF == of, 'output_filter %d does not match the %s loss layout (%d)' % (self.OF, loss, of)
        self.lr, self.beta1, self.beta2, self.eps = lr, beta1, beta2, eps
        self.pg = process_group
        self.world = 1
        if process_group is not None or (torch.distributed.is_available() and torch.distributed.is_initialized()):
            self.world = torch.distributed.get_world_size(process_group)
        self.update_moving = update_moving
        self.store = store if store is not None else VariableStore(seed=seed)
        self.layers = (create_classifier_variables(self.store, self.OF) if loss == 'softmax'
                       else create_variables(self.store, self.OF, passthrough=self.passthrough))
        self.iteration = 0
        # the whole step (forward, loss, backward, Adam: ~245 launches) replayed as ONE CUDA graph.  With world > 1 the NCCL
        # buckets stay eager launches on NCCL's stream (capturing them too dead-locked in a 2-GPU trial) and the step is cut
        # into one graph per stretch between two bucket launches: [forward, loss, backward down to the first bucket's last
        # layer], [... to the second bucket], ..., [update] -- see _enqueue_segment / step.
        import os as _os
        self.use_cuda_graph = bool(use_cuda_graph)
        if _os.environ.get('Y2_BUCKET_MB'):
            bucket_bytes = int(float(_os.environ['Y2_BUCKET_MB']) * (1 << 20))
        self.graph = None
        self.seg_graphs = None
        self.launches_per_step = 0
        self._grads_clean = True                    # the gradient arena is all zero (fresh, or cleared by the last update)
        dev = self.device
        with torch.cuda.device(dev):
            self._build_arenas()
            self._build_buffers()
            self._build_buckets(bucket_bytes)

    # ------------------------------------------------------------------------------------------
    def _build_arenas(self):
        """Flat fp32 arenas, layers in reverse order, per layer [W | b | gamma | beta], 64-float aligned."""
        st, dev = self.store, self.device
        off = 0
        self.slots = [None] * len(self.layers)
        for li in reversed(range(len(self.layers))):
            L = self.layers[li]
            names = (L['W'], L['b'], L['bn']['gamma'], L['bn']['beta'])
            sl = {}
            start = off
            for key, nm in zip(('W', 'b', 'gamma', 'beta'), names):
                n = int(np.prod(np.shape(st[nm])))
                sl[key] = (off, n, tuple(np.shape(st[nm])))
                off = _round_up(off + n, 64)
            sl['range'] = (start, off)
            self.slots[li] = sl
        self.arena_elems = off
        f32 = dict(dtype=torch.float32, device=dev)
        self.params = torch.zeros((off,), **f32)
        self.grads = torch.zeros((off,), **f32)
        self.adam_m = torch.zeros((off,), **f32)           # (momentum optimizer: the accumulator slot)
        self.adam_v = torch.zeros((off if self.optimizer == 'adam' else 4,), **f32)
        self.P, self.G = [], []
        for li, L in enumerate(self.layers):
            sl = self.slots[li]
            pv, gv = {}, {}
            for key, nm in zip(('W', 'b', 'gamma', 'beta'), (L['W'], L['b'], L['bn']['gamma'], L['bn']['beta'])):
                o, n, shp = sl[key]
                pv[key] = self.params[o:o + n].view(shp)
                gv[key] = self.grads[o:o + n].view(shp)
                src = st[nm]
                pv[key].copy_(torch.as_tensor(src).to(dev) if not isinstance(src, torch.Tensor) else src.to(dev))
                st.vars[nm] = pv[key]                       # the store now aliases the arena
            for nm in (L['bn']['moving_mean'], L['bn']['moving_variance']):
                v = st[nm]
                st.vars[nm] = (torch.as_tensor(v) if not isinstance(v, torch.Tensor) else v).to(dev).contiguous()
            self.P.append(pv)
            self.G.append(gv)
        st.version += 1

    def _build_buffers(self):
        N, IS, dev = self.N, self.IS, self.device
        f32 = dict(dtype=torch.float32, device=dev)
        bf16 = dict(dtype=torch.bfloat16, device=dev)
        self.in_u8 = torch.zeros((N, IS, IS, 3), dtype=torch.uint8, device=dev)
        self.in_f32 = None
        self.x0 = torch.empty((N, IS, IS, 8), **bf16)
        self.acts, self.raw, self.stats, self.geom = [], [], [], []
        self.packed, self.packed_dgrad = [], []
        self.pt_src = self.d_cat = self.d_pt = None
        H = IS
        max_ws, max_dh, max_dx = 1, 1, 1
        nl = len(self.layers)
        for li, L in enumerate(self.layers):
            role = L.get('role')
            Ho = H // 2 if L['pool'] else H
            Hc = 2 * H if role == 'passthrough' else H          # the map the conv runs on: the passthrough conv's is 2S x 2S
            last = li == nl - 1
            cout, cin, k = L['cout'], L['cin'], L['k']
            ldh = raw_ld(cout)
            ld_dh = 32 if li == 0 else _round_up(cout, 64)
            self.geom.append(dict(H=Hc, Ho=Ho if role != 'passthrough' else Hc, ldh=ldh, ld_dh=ld_dh, M=N * Hc * Hc))
            if self.passthrough and role == 'conv2':
                # conv2's 1024 channels and the passthrough branch's 4 * 64 share one [N,S,S,1280] activation (conv3's input)
                self.acts.append(torch.empty((N, Ho, Ho, cout + 4 * PASSTHROUGH_FILTERS), **bf16))
            elif role == 'passthrough':
                self.acts.append(self.acts[-1])
            else:
                self.acts.append(torch.empty((N, Ho, Ho, cout), **(f32 if last else bf16)))
            if self.passthrough and li == PASSTHROUGH_LAYER:
                self.pt_src = torch.empty((N, H, H, cout), **bf16)             # layer 13 before its pool
                self.d_pt = torch.empty((N, H, H, cout), **bf16)               # its gradient from the passthrough conv
            self.raw.append(torch.empty((N * Hc * Hc, ldh), **f32))
            self.stats.append(dict(mean=torch.empty((cout,), **f32), var=torch.empty((cout,), **f32),
                                   scale=torch.empty((cout,), **f32), shift=torch.empty((cout,), **f32)))
            max_ws = max(max_ws, ops.bn_stats_workspace_bytes(N * Hc * Hc, cout), ops.bn_bwd_workspace_bytes(N * Hc * Hc, cout))
            max_dh = max(max_dh, N * Hc * Hc * ld_dh)
            if li > 0 and not (self.passthrough and role in ('passthrough', 'conv3')):      # (those two: d_pt, d_cat)
                max_dx = max(max_dx, N * Hc * Hc * cin)
            self.packed.append(torch.empty((int(ops._lib.load().y2_conv_packed_weight_elems(k, cin, cout)),), **bf16))
            self.packed_dgrad.append(None if li == 0 else torch.empty(
                (int(ops._lib.load().y2_conv_packed_weight_dgrad_elems(k, cin, ld_dh)),), **bf16))
            H = Ho
        self.ws = torch.empty((max_ws,), dtype=torch.uint8, device=dev)
        self.conv_ws = ops.new_conv_workspace(dev)          # this trainer's own stream-K scratch (see ops.conv_workspace_scope)
        self.dh = torch.empty((max_dh,), **bf16)
        self.dx = [torch.empty((max_dx,), **bf16), torch.empty((max_dx,), **bf16)]
        if self.passthrough:
            self.d_cat = torch.empty(tuple(self.acts[self._index('conv3') - 1].shape), **bf16)     # conv3's data gradient
        S = self.S
        self.terms = torch.zeros((2 if self.loss_kind == 'softmax' else 5,), **f32)
        self.lr_dev = torch.zeros((1,), **f32)              # Adam step size of the current iteration (read by the update kernel)
        self._lr_host = torch.zeros((1,), dtype=torch.float32).pin_memory()
        self.dnet = torch.empty((N, S, S, self.OF), **f32)
        if self.loss_kind == 'v1':
            self.labels = torch.zeros((N, S, S, 5 + self.C), **f32)
            self.ious = torch.empty((N, S, S, self.B), **f32)
            self.object_mask = torch.empty((N, S, S, self.B), **f32)
        elif self.loss_kind == 'softmax':
            self.class_labels = torch.zeros((N,), dtype=torch.int32, device=dev)
            self.logits = torch.empty((N, self.OF), **f32)
            self.losses = torch.empty((N,), **f32)
            self.correct = torch.empty((N,), **f32)
        else:
            self.anchors = torch.as_tensor(self.anchors_np).to(dev).contiguous()
            self.gt_boxes = torch.zeros((N, self.max_gt, 4), **f32)
            self.gt_classes = torch.zeros((N, self.max_gt), dtype=torch.int32, device=dev)
            self.gt_counts = torch.zeros((N,), dtype=torch.int32, device=dev)
        self._build_gradient_routes()

    def _index(self, role):
        return next(li for li, L in enumerate(self.layers) if L.get('role') == role)

    def _build_gradient_routes(self):
        """Per layer: where its data gradient goes (dx_out) and where the gradient of its output is read (dy_src: the
        consumer's data gradient as (tensor, ldy, column, depth_to_space, un-pooled addend), or the loss gradient).  In the
        chain, layer li writes the ping-pong buffer dx[li & 1] and layer li - 1 reads it; the passthrough graph adds the
        concat gradient d_cat (conv3 -> conv2 and the passthrough conv) and d_pt (passthrough conv -> layer 13)."""
        N, nl = self.N, len(self.layers)
        self.dx_out, self.dy_src = [None] * nl, [None] * nl
        for li in range(1, nl):
            g, L = self.geom[li], self.layers[li]
            if self.passthrough and L.get('role') in ('passthrough', 'conv3'):
                self.dx_out[li] = self.d_pt if L['role'] == 'passthrough' else self.d_cat
            else:
                self.dx_out[li] = self.dx[li & 1][:g['M'] * L['cin']].view(N, g['H'], g['H'], L['cin'])
        for li in range(nl - 1):
            self.dy_src[li] = dict(t=self.dx_out[li + 1], ldy=None, col=0, s2d=False, add=None)
        self.dy_src[nl - 1] = dict(t=self.dnet, ldy=None, col=0, s2d=False, add=None)
        if not self.passthrough:
            return
        i2, ip = self._index('conv2'), self._index('passthrough')
        ldc = self.d_cat.shape[-1]
        self.dy_src[i2] = dict(t=self.d_cat, ldy=ldc, col=0, s2d=False, add=None)
        self.dy_src[ip] = dict(t=self.d_cat, ldy=ldc, col=ldc - 4 * self.layers[ip]['cout'], s2d=True, add=None)
        self.dy_src[PASSTHROUGH_LAYER]['add'] = self.d_pt

    def _build_buckets(self, bucket_bytes):
        """Contiguous arena slices in backward order; a bucket is launched once its last layer's gradients are enqueued."""
        ranges = [(li,) + self.slots[li]['range'] for li in reversed(range(len(self.layers)))]
        self.buckets = make_buckets(ranges, bucket_bytes)
        self.reducer = BucketedAllReduce(self.grads, self.buckets, self.pg, self.world)

    # ------------------------------------------------------------------------------------------
    def set_labels(self, labels):
        """v1 loss: labels [N,S,S,5+C] as produced by pascal_voc.get() (float64 numpy in the reference,
        pascal_voc.py:43-46; cast to float32 at the feed like the TF placeholder does)."""
        assert self.loss_kind == 'v1'
        self.labels.copy_(torch.as_tensor(np.asarray(labels), dtype=torch.float32), non_blocking=True)

    def set_class_labels(self, labels):
        """softmax loss: int class index per image (the int32 `label_data` placeholder, imagenet_train_darknet.py:47)."""
        assert self.loss_kind == 'softmax'
        self.class_labels.copy_(torch.as_tensor(np.asarray(labels).astype(np.int32)), non_blocking=True)

    def set_ground_truth(self, gt_boxes, gt_classes, gt_counts):
        assert self.loss_kind == 'region'
        self.gt_boxes.copy_(torch.as_tensor(np.asarray(gt_boxes), dtype=torch.float32), non_blocking=True)
        self.gt_classes.copy_(torch.as_tensor(np.asarray(gt_classes), dtype=torch.int32), non_blocking=True)
        self.gt_counts.copy_(torch.as_tensor(np.asarray(gt_counts), dtype=torch.int32), non_blocking=True)

    # ------------------------------------------------------------------------------------------
    def forward(self):
        if self.in_f32 is not None:
            ops.pad_cast_f32_to_bf16c8(self.in_f32, out=self.x0)        # pascal_voc.get() images: already x/255*2-1
        else:
            ops.preprocess_u8(self.in_u8, bf16c8=True, out=self.x0)
        x = self.x0
        nl = len(self.layers)
        for li, L in enumerate(self.layers):
            s, P, bn = self.stats[li], self.P[li], L['bn']
            ops.pack_weights_bf16(P['W'], out=self.packed[li])
            moving = (self.store[bn['moving_mean']], self.store[bn['moving_variance']]) if self.update_moving else None
            r = layer_route(L, li, x, self.acts[li], self.pt_src)
            conv_bn_tc(r['x'], self.packed[li], L['k'], L['cin'], L['cout'], bias=P['b'], gamma=P['gamma'], beta=P['beta'],
                       moving=moving, stats=(s['mean'], s['var'], s['scale'], s['shift']), workspace=self.ws, pool=r['pool'],
                       out_f32=li == nl - 1, out=r['out'], ldo=r['ldo'], col=r['col'], s2d=r['s2d'], raw=self.raw[li])
            if r['pooled'] is not None:
                ops.maxpool2x2_bf16(self.pt_src, out=r['pooled'])
            x = self.acts[li]
        return self.acts[-1]

    def loss(self):
        net = self.acts[-1]
        if self.loss_kind == 'v1':
            ops.loss_v1(net, self.labels, self.S, self.B, self.C, float(self.IS), self.lambda_coord, self.lambda_noobj,
                        want_grad=True, terms=self.terms, ious=self.ious, object_mask=self.object_mask, dnet=self.dnet)
        elif self.loss_kind == 'softmax':
            ops.softmax_xent(net, self.class_labels, terms=self.terms, logits=self.logits, losses=self.losses,
                             correct=self.correct, dnet=self.dnet)
        else:
            ops.region_loss(net, self.anchors, self.gt_boxes, self.gt_classes, self.gt_counts, self.C,
                            lambda_coord=self.lambda_coord, lambda_noobj=self.lambda_noobj, terms=self.terms,
                            dnet=self.dnet)
        return self.terms

    def backward(self, capture=None):
        """capture: optional dict; receives {layer index: clone of the gradient w.r.t. that layer's output} (tests)."""
        if not self._grads_clean:                   # (only when backward runs twice without an update in between: the
            self.grads.zero_()                      #  update kernel leaves the arena cleared)
        self._grads_clean = False
        self.reducer.begin()
        for li in reversed(range(len(self.layers))):
            self._backward_layer(li, capture)
            self.reducer.layer_done(li)
        self.reducer.finish(scale=False)            # sums; the 1/world of the mean is applied inside the update kernel

    def _dy_of(self, li):
        """Gradient w.r.t. layer li's output as a dense [N,Ho,Wo,C] tensor: the loss gradient for the last layer, else the
        data gradient of its consumer -- for the passthrough graph's conv2 a view of the concat gradient's first 1024
        columns, for the passthrough conv a depth_to_space copy of its last 256 (tests and tools; the backward pass reads
        them in place).  Layer 13's second, un-pooled gradient (passthrough graph) is self.d_pt."""
        d = self.dy_src[li]
        L, t = self.layers[li], d['t']
        c = L['cout']
        if d['ldy'] is None:
            return t
        v = t[..., d['col']:d['col'] + (4 * c if d['s2d'] else c)]
        if not d['s2d']:
            return v
        n, h, w, _ = v.shape                                    # depth_to_space(2): [N,S,S,4C] -> [N,2S,2S,C]
        return v.reshape(n, h, w, 2, 2, c).permute(0, 1, 3, 2, 4, 5).reshape(n, 2 * h, 2 * w, c)

    def _backward_layer(self, li, capture=None):
        L, g, s, P, G = self.layers[li], self.geom[li], self.stats[li], self.P[li], self.G[li]
        H, M, cout, cin, k = g['H'], g['M'], L['cout'], L['cin'], L['k']
        d = self.dy_src[li]
        if capture is not None:
            capture[li] = self._dy_of(li).clone()
            if d['add'] is not None:
                capture['d_pt'] = d['add'].clone()
        dh = self.dh[:M * g['ld_dh']].view(M, g['ld_dh'])
        ops.bn_leaky_pool_bwd(self.raw[li], d['t'], s['mean'], s['var'], P['gamma'], P['beta'], self.N, H, H, cout,
                              ldh=g['ldh'], leaky=True, pool=L['pool'], ld_dh=g['ld_dh'], dgamma=G['gamma'],
                              dbeta=G['beta'], dh=dh, workspace=self.ws, ldy=d['ldy'], dy_col=d['col'], dy_s2d=d['s2d'],
                              dy_add=d['add'])
        if L.get('role') == 'passthrough':
            xin = self.pt_src
        else:
            xin = self.x0 if li == 0 else self.acts[li - 1]
        if li == 0:
            ops.conv_wgrad_c3(xin, dh, cout, G['W'])
        else:
            ops.conv_wgrad_bf16(xin, dh, k, cin, cout, G['W'])
            ops.pack_weights_dgrad_bf16(P['W'], g['ld_dh'], out=self.packed_dgrad[li])
            ops.conv_fwd_bf16(dh.view(self.N, H, H, g['ld_dh']), self.packed_dgrad[li], k, g['ld_dh'], cin, scale=None,
                              shift=None, leaky=False, pool=False, out=self.dx_out[li])

    def _set_lr(self):
        """TF's bias-corrected step size of iteration self.iteration -> device scalar (a 4-byte async copy, outside the graph)."""
        self._lr_host[0] = ops.adam_lr_t(self.iteration, self.lr, self.beta1, self.beta2)
        self.lr_dev.copy_(self._lr_host, non_blocking=True)

    def update(self, _lr_set=False, zero_grad=True):
        """Adam on the (summed) gradients scaled by 1/world; clears the gradient arena behind the read (zero_grad=False keeps
        the gradients readable -- tests; the next backward then clears the arena itself)."""
        if not _lr_set:
            self.iteration += 1
            self._set_lr()
        if self.optimizer == 'momentum':
            ops.momentum_step(self.params, self.grads, self.adam_m, self.lr, self.momentum, grad_scale=1.0 / self.world,
                              zero_grad=zero_grad)
        else:
            ops.adam_step_ex(self.params, self.grads, self.adam_m, self.adam_v, lr_t_dev=self.lr_dev, b1=self.beta1,
                             b2=self.beta2, eps=self.eps, grad_scale=1.0 / self.world, zero_grad=zero_grad)
        self._grads_clean = bool(zero_grad)
        self.store.version += 1

    def _enqueue_step(self):
        self.forward()
        self.loss()
        self.backward()
        self.update(_lr_set=True)

    # ---- data parallel: one graph per stretch between two bucket launches ----
    def _segments(self):
        return bucket_segments(self.buckets, len(self.layers))

    def _enqueue_segment(self, i, seg):
        if i == 0:
            self.forward()
            self.loss()
        for li in range(seg[0], seg[1] - 1, -1):
            self._backward_layer(li)

    def _step_segmented(self):
        """world > 1 with CUDA graphs: replay stretch i, launch bucket i's all-reduce (eager, NCCL's stream, overlapping the
        next stretch), ..., wait for the buckets, replay the update."""
        segs = self._segments()
        if self.seg_graphs is None:
            if not self._grads_clean:
                self.grads.zero_()
                self._grads_clean = True
            # warm-up outside the capture (every rank runs it, collectives included), then restore what it changed
            snap = [t.clone() for t in self._graph_state()]
            self._enqueue_step()
            torch.cuda.synchronize(self.device)
            for t, c in zip(self._graph_state(), snap):
                t.copy_(c)
            self.grads.zero_()
            n0 = ops.launch_count()
            pool = torch.cuda.graph_pool_handle()
            graphs = []
            for i, seg in enumerate(segs):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, pool=pool):
                    self._enqueue_segment(i, seg)
                graphs.append(g)
            gu = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gu, pool=pool):
                self.update(_lr_set=True)
            self.launches_per_step = ops.launch_count() - n0
            for t, c in zip(self._graph_state(), snap):       # (capture does not execute, but keep the invariant explicit)
                t.copy_(c)
            self.seg_graphs = (graphs, gu)
        graphs, gu = self.seg_graphs
        self.reducer.begin()
        for g, seg in zip(graphs, segs):
            g.replay()
            self.reducer.layer_done(seg[1])
        self.reducer.finish(scale=False)
        gu.replay()
        self._grads_clean = True
        self.store.version += 1

    def step(self, images=None, capture=None):
        """One training iteration on the current stream.  images: uint8 [N,IS,IS,3] BGR (host or device) or None
        to reuse self.in_u8.  Returns the device tensor terms[5] (the loss is terms[4])."""
        if images is not None:
            t = torch.as_tensor(images)
            if t.dtype == torch.uint8:
                if self.in_f32 is not None:                 # the input kind is baked into a captured step
                    self.in_f32, self.graph, self.seg_graphs = None, None, None
                self.in_u8.copy_(t, non_blocking=True)
            else:       # float images as produced by pascal_voc.get() (float64 in the reference, cast at the feed)
                if self.in_f32 is None:
                    self.graph, self.seg_graphs = None, None
                    self.in_f32 = torch.empty((self.N, self.IS, self.IS, 3), dtype=torch.float32, device=self.device)
                self.in_f32.copy_(t.to(torch.float32), non_blocking=True)
        self.iteration += 1
        self._set_lr()
        with ops.conv_workspace_scope(self.conv_ws):
            if not self.use_cuda_graph or capture is not None:
                self.forward()
                self.loss()
                self.backward(capture)
                self.update(_lr_set=True, zero_grad=capture is None)      # (a capturing caller reads the gradients afterwards)
                return self.terms
            if self.world > 1:
                self._step_segmented()
                return self.terms
            if self.graph is None:
                if not self._grads_clean:
                    self.grads.zero_()
                    self._grads_clean = True
                # warm-up outside the capture (function attributes, workspaces), then restore what it changed: the weights,
                # the Adam moments and the BN moving statistics must see this iteration exactly once
                snap = [t.clone() for t in self._graph_state()]
                s = torch.cuda.Stream(device=self.device)
                s.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(s):
                    self._enqueue_step()
                torch.cuda.current_stream().wait_stream(s)
                torch.cuda.synchronize(self.device)
                for t, c in zip(self._graph_state(), snap):
                    t.copy_(c)
                n0 = ops.launch_count()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._enqueue_step()
                self.launches_per_step = ops.launch_count() - n0
                for t, c in zip(self._graph_state(), snap):       # (capture does not execute, but keep the invariant explicit)
                    t.copy_(c)
                self.graph = g
            self.graph.replay()
            self._grads_clean = True
            self.store.version += 1
        return self.terms

    def _graph_state(self):
        st = [self.params, self.adam_m, self.adam_v, self.grads]
        for L in self.layers:
            st += [self.store[L['bn']['moving_mean']], self.store[L['bn']['moving_variance']]]
        return st

    def phase_times(self, iters=3):
        """Device time (ms) of the phases of one eager step -- forward / loss / backward (+ all-reduce) / update -- and, with
        world > 1, the part of the all-reduce that the overlap with backward does NOT hide (backward timed with and without
        the collectives).  Weights / moments are restored afterwards."""
        snap = [t.clone() for t in self._graph_state()]
        it0 = self.iteration
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        acc = np.zeros(4)
        bwd_local = 0.0
        with ops.conv_workspace_scope(self.conv_ws):
            for k in range(iters + 1):
                self.iteration += 1
                self._set_lr()
                ev[0].record(); self.forward(); ev[1].record(); self.loss(); ev[2].record(); self.backward(); ev[3].record()
                self.update(_lr_set=True); ev[4].record()
                ev[4].synchronize()
                if k:
                    acc += [ev[i].elapsed_time(ev[i + 1]) for i in range(4)]
            out = dict(zip(('forward', 'loss', 'backward', 'update'), (acc / iters).round(4).tolist()))
            if self.world > 1:
                w = self.reducer.world
                self.reducer.world = 1                  # same kernels, no collectives
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                for k in range(iters + 1):
                    self.forward(); self.loss()
                    if torch.distributed.is_initialized():
                        torch.cuda.synchronize()
                        torch.distributed.barrier(group=self.pg)
                    e0.record(); self.backward(); e1.record()
                    e1.synchronize()
                    self.grads.zero_(); self._grads_clean = True
                    if k:
                        bwd_local += e0.elapsed_time(e1) / iters
                self.reducer.world = w
                out['backward_without_allreduce'] = round(bwd_local, 4)
                out['allreduce_exposed'] = round(out['backward'] - bwd_local, 4)
        for t, c in zip(self._graph_state(), snap):
            t.copy_(c)
        self.iteration = it0
        return out


    # ---- checkpoint state beyond the variables (tf.train.Saver() saves ALL global variables: pascal_train_darknet.py:54,111) ----
    def optimizer_state(self):
        """Adam's slot variables under the names TF gives them (`<var>/Adam` = m, `<var>/Adam_1` = v) plus `beta1_power`,
        `beta2_power` -- what the reference's Saver writes next to the weights -- and the iteration count.  Pass the dict as
        `extra=` to net_utils.save_checkpoint; `load_optimizer_state` is the inverse.  Without them a resumed run would
        restart Adam from zero moments and a bias correction at t = 1."""
        out = {}
        for li, L in enumerate(self.layers):
            sl = self.slots[li]
            for key, nm in zip(('W', 'b', 'gamma', 'beta'), (L['W'], L['b'], L['bn']['gamma'], L['bn']['beta'])):
                o, n, shp = sl[key]
                if self.optimizer == 'momentum':            # MomentumOptimizer's one slot: `<var>/Momentum`
                    out[nm + '/Momentum'] = self.adam_m[o:o + n].view(shp).detach().cpu().numpy()
                    continue
                out[nm + '/Adam'] = self.adam_m[o:o + n].view(shp).detach().cpu().numpy()
                out[nm + '/Adam_1'] = self.adam_v[o:o + n].view(shp).detach().cpu().numpy()
        if self.optimizer == 'adam':
            out['beta1_power'] = np.float32(self.beta1 ** (self.iteration + 1))      # TF holds beta^(t+1) after t updates
            out['beta2_power'] = np.float32(self.beta2 ** (self.iteration + 1))
        out['y2_iteration'] = np.int64(self.iteration)
        return out

    def load_optimizer_state(self, npz_path, iteration=None):
        """Restore what optimizer_state() saved.  Returns the list of slot names found; slots absent from the file (a
        warm start from an ImageNet snapshot, a weights-only file) keep their zero initial value."""
        data = np.load(npz_path)
        found = []
        for li, L in enumerate(self.layers):
            sl = self.slots[li]
            for key, nm in zip(('W', 'b', 'gamma', 'beta'), (L['W'], L['b'], L['bn']['gamma'], L['bn']['beta'])):
                o, n, shp = sl[key]
                slots_ = ((('/Momentum', self.adam_m),) if self.optimizer == 'momentum'
                          else (('/Adam', self.adam_m), ('/Adam_1', self.adam_v)))
                for suffix, arena in slots_:
                    if nm + suffix in data.files:
                        arena[o:o + n].view(shp).copy_(torch.as_tensor(data[nm + suffix], dtype=torch.float32))
                        found.append(nm + suffix)
        if iteration is not None:
            self.iteration = int(iteration)
        elif 'y2_iteration' in data.files:
            self.iteration = int(data['y2_iteration'])
        elif 'beta1_power' in data.files:
            self.iteration = int(round(np.log(float(data['beta1_power'])) / np.log(self.beta1))) - 1
        return found

    def sync_moving_statistics(self):
        """Average the BN moving means / variances over the ranks (each rank tracks its own shard's statistics; the
        reference is single-device, so any consistent choice is an extension).  Called before rank 0 writes a snapshot."""
        if self.world <= 1:
            return
        for L in self.layers:
            for nm in (L['bn']['moving_mean'], L['bn']['moving_variance']):
                t = self.store[nm]
                torch.distributed.all_reduce(t, group=self.pg)
                t.mul_(1.0 / self.world)

    # helpers for tests / checkpoints
    def gradient(self, li, key):
        return self.G[li][key]

    def num_parameters(self):
        return sum(sl[k][1] for sl in self.slots for k in ('W', 'b', 'gamma', 'beta'))
