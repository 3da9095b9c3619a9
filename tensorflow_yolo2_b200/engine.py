"""Batch inference engine: Darknet19 + detection head -> decode -> per-class NMS, all buffers
pre-allocated, weights pre-packed, inference-mode BN pre-folded, the whole step captured in one
CUDA graph.  Every conv layer except the fused uint8 first one (conv1_u8_pool) goes through
yolo2_nets.darknet.conv_bn_tc, the routine behind the eager builders' tensor-core path, so the
engine issues the builders' kernels into its own buffers.  It exists because a 22-layer network at
>10 k images/s is launch-bound from Python otherwise.

The layer semantics follow the reference scripts (src/pascal/pascal_detect_darknet.py:41-43):
core with is_training=False (moving statistics), head with is_training=True (batch statistics
over the batch the engine is given) unless overridden.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from . import ops
from .variables import VariableStore
from .yolo2_nets.darknet import (CORE_PLAN, PASSTHROUGH_FILTERS, PASSTHROUGH_LAYER, classifier_plan, conv_bn_tc,
                                  head_plan, layer_route, raw_ld)
from .yolo2_nets.net_utils import VOC_ANCHORS


def _layer_variables(store, k, cin, cout, pool=False, **kw):
    wn, _ = store.weight_variable([k, k, cin, cout])
    bn_, _ = store.bias_variable([cout])
    return dict(k=k, cin=cin, cout=cout, pool=pool, W=wn, b=bn_, bn=store.batch_norm_variables(cout), **kw)


def create_variables(store, output_filter, passthrough=False):
    """Create (or find) every variable of darknet19_core + darknet19_detection in the reference's creation order and naming.
    passthrough=True adds the YOLOv2 passthrough branch of yolo2_nets.darknet.head_plan."""
    store.reset_name_counters()
    with store.scope('darknet19'):
        layers = [_layer_variables(store, *p, head=False) for p in CORE_PLAN]
    with store.scope('darknet19_detection'):
        for sc, k, cin, cout in head_plan(output_filter, PASSTHROUGH_FILTERS if passthrough else 0):
            with store.scope(sc):
                layers.append(_layer_variables(store, k, cin, cout, head=True, role=sc))
    return layers


def create_classifier_variables(store, num_classes=1000):
    """The variables of the `darknet19` ImageNet classifier (darknet.py:61-123) in creation order: the 18 core layers and the
    19th conv_bn_layer (1x1, 1024 -> num_classes) in the SAME scope, so its names continue the core's numbering
    (darknet19/Variable_36, Variable_37, batch_normalization_18)."""
    store.reset_name_counters()
    with store.scope('darknet19'):
        layers = [_layer_variables(store, *p, head=False, role=None) for p in CORE_PLAN]
        layers.append(_layer_variables(store, *classifier_plan(num_classes), head=True, role='logits'))
    return layers


class Yolo2Engine:
    def __init__(self, batch, image_size=416, output_filter=125, store=None, core_training=False, head_training=True,
                 anchors=VOC_ANCHORS, num_class=20, score_thresh=0.3, iou_thresh=0.45, max_keep=None,
                 input_kind='u8', decode='region', use_cuda_graph=True, device=None, seed=0, fused_detect=True,
                 fused_conv1=True, passthrough=False, precision='bf16'):
        """precision: 'bf16' -- every conv operand rounded once to bf16 (one tcgen05.mma per K step; ~1e-2 on the network
        output after 22 layers); 'bf16x3' -- activations and weights travel as hi + lo bf16 pairs and every product is
        a_hi*w_hi + a_lo*w_hi + a_hi*w_lo (three MMAs per K step, fp32 accumulate): the mode that meets the spec's 1e-3
        bar on decoded boxes / scores (tests/test_parity_gpu.py)."""
        if precision not in ('bf16', 'bf16x3'):
            raise ValueError("precision must be 'bf16' or 'bf16x3'")
        self.precision = precision
        self.x3 = precision == 'bf16x3'
        self.device = torch.device(device) if device is not None else torch.device('cuda', torch.cuda.current_device())
        self.N, self.IS, self.OF = int(batch), int(image_size), int(output_filter)
        assert self.IS % 32 == 0
        self.S = self.IS // 32
        self.C = num_class
        self.core_training, self.head_training = bool(core_training), bool(head_training)
        self.score_thresh, self.iou_thresh = float(score_thresh), float(iou_thresh)
        self.input_kind = input_kind
        self.decode = decode
        self.fused_detect = bool(fused_detect)
        # 'split': chunked decode over the whole batch + per-image NMS over candidate lists (detect_split.cu);
        # 'fused': one CTA per image (detect_fused.cu).  Same results.
        # Same results; measured on B200: at batch 64 the single launch wins (1.990 vs 2.008 ms per step), at batch 256
        # the split pair does (27.6 vs 30.7 us for decode + NMS alone)
        self.detect_impl = os.environ.get('Y2_DETECT_IMPL', 'split' if self.N >= 128 else 'fused')
        # first layer fused with the uint8 preprocessing and the pool (conv1_fused.cu): inference-mode BN, u8 input
        self.fused_conv1 = bool(fused_conv1) and input_kind == 'u8' and not self.core_training
        self.store = store if store is not None else VariableStore(seed=seed)
        self.passthrough = bool(passthrough)
        if self.x3 and (self.passthrough or not self.fused_conv1):
            raise NotImplementedError("precision='bf16x3' needs the fused uint8 first layer (input_kind='u8', inference-mode "
                                      "core) and has no passthrough branch yet")
        self.layers = create_variables(self.store, self.OF, passthrough=self.passthrough)
        dev = self.device
        f32 = dict(dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            self._to_device()
            # ---- buffers ----
            N, IS = self.N, self.IS
            self.in_u8 = torch.zeros((N, IS, IS, 3), dtype=torch.uint8, device=dev)
            self.in_f32 = torch.zeros((N, IS, IS, 3), **f32) if input_kind == 'f32' else None
            self.x0 = torch.empty((N, IS, IS, 8), dtype=torch.bfloat16, device=dev)
            self.acts, self.raw, self.stats = [], {}, {}
            H = IS
            max_ws = 1
            self.pt_src = None
            for li, L in enumerate(self.layers):
                Ho = H // 2 if L['pool'] else H
                training = self.head_training if L['head'] else self.core_training
                last = li == len(self.layers) - 1
                role = L.get('role')
                Hin = 2 * H if role == 'passthrough' else H           # the passthrough conv runs on the 26x26 map
                cm = 2 if self.x3 else 1                  # bf16x3: rows are [hi | lo]
                if last:
                    self.acts.append(torch.empty((N, Ho, Ho, L['cout']), **f32))
                elif self.passthrough and role == 'conv2':
                    # conv2's 1024 channels and the reorganised passthrough's 256 share one [N,S,S,1280] tensor: the
                    # concat is the two producers' store addresses, never a copy
                    self.acts.append(torch.empty((N, Ho, Ho, L['cout'] + 4 * PASSTHROUGH_FILTERS), dtype=torch.bfloat16,
                                                 device=dev))
                elif role == 'passthrough':
                    self.acts.append(self.acts[-1])
                else:
                    self.acts.append(torch.empty((N, Ho, Ho, cm * L['cout']), dtype=torch.bfloat16, device=dev))
                if self.passthrough and li == PASSTHROUGH_LAYER:
                    self.pt_src = torch.empty((N, H, H, L['cout']), dtype=torch.bfloat16, device=dev)
                if training or last or role == 'passthrough':                # conv_bn_tc writes float32 conv rows
                    self.raw[li] = torch.empty((N * Hin * Hin, raw_ld(L['cout'])), **f32)
                if training:
                    self.stats[li] = tuple(torch.empty((L['cout'],), **f32) for _ in range(4))     # mean, var, scale, shift
                    max_ws = max(max_ws, ops.bn_stats_workspace_bytes(N * Hin * Hin, L['cout']))
                H = Ho
            self.ws = torch.empty((max_ws,), dtype=torch.uint8, device=dev)
            # this engine's own stream-K scratch (zero-filled flags): engines / trainers on other streams have theirs
            self.conv_ws = ops.new_conv_workspace(dev)
            if decode == 'region':
                assert self.OF % (5 + self.C) == 0
                self.A = self.OF // (5 + self.C)
                self.anchors = torch.as_tensor(np.asarray(anchors, dtype=np.float32)[:self.A]).to(dev).contiguous()
                self.nbox = self.S * self.S * self.A
                self.max_keep = int(max_keep or self.nbox)
                self.boxes = torch.empty((N, self.nbox, 4), **f32)
                self.scores = torch.empty((N, self.nbox, self.C), **f32)
                self.keep_idx = torch.full((N, self.C, self.max_keep), -1, dtype=torch.int32, device=dev)
                self.keep_count = torch.zeros((N, self.C), dtype=torch.int32, device=dev)
                # candidate lists of the split detection path: zero-filled once, every call leaves it zero-filled
                self.detect_ws = torch.zeros((ops.detect_workspace_bytes(N, self.C),), dtype=torch.uint8, device=dev)
            self.refresh_weights()
            self.graph = None
            self.use_cuda_graph = use_cuda_graph

    # ------------------------------------------------------------------------------------------
    def _to_device(self):
        for k, v in list(self.store.vars.items()):
            if isinstance(v, np.ndarray):
                self.store.vars[k] = torch.from_numpy(v).to(self.device)
            elif v.device != self.device:
                self.store.vars[k] = v.to(self.device)

    def refresh_weights(self):
        """(Re)pack weights and fold inference-mode BN; call after the store changes."""
        st = self.store
        self.packed, self.fold = [], {}
        for li, L in enumerate(self.layers):
            if self.x3:
                self.packed.append(ops.pack_weights_bf16_split(st[L['W']]) if li > 0 else None)
            else:
                self.packed.append(ops.pack_weights_bf16(st[L['W']]))
            training = self.head_training if L['head'] else self.core_training
            if not training:
                bn = L['bn']
                self.fold[li] = ops.bn_fold(st[bn['gamma']], st[bn['beta']], st[bn['moving_mean']],
                                            st[bn['moving_variance']], st[L['b']])
        if self.fused_conv1:
            pack_c1 = ops.pack_weights_conv1_u8_split if self.x3 else ops.pack_weights_conv1_u8
            self.packed_c1 = pack_c1(st[self.layers[0]['W']], self.fold[0][0])
        self.graph = None
        self._pipe_graphs = {}
        self._version = st.version

    # ------------------------------------------------------------------------------------------
    def _enqueue(self):
        with ops.conv_workspace_scope(self.conv_ws):
            self._enqueue_body()

    def _enqueue_body(self):
        st = self.store
        if self.fused_conv1:
            pass                                     # the first conv reads self.in_u8 directly
        elif self.input_kind == 'u8':
            ops.preprocess_u8(self.in_u8, bf16c8=True, out=self.x0)
        else:
            ops.pad_cast_f32_to_bf16c8(self.in_f32, out=self.x0)
        x = self.x0
        nl = len(self.layers)
        for li, L in enumerate(self.layers):
            training = self.head_training if L['head'] else self.core_training
            out = self.acts[li]
            if li == 0 and self.fused_conv1:
                ops.conv1_u8_pool(self.in_u8, self.packed_c1, self.fold[0][1], out=out, split=self.x3)
            else:
                # where the layer reads and writes: dense, a channel slice of the concat buffer, or un-pooled to pt_src
                r = layer_route(L, li, x, out, self.pt_src)
                bn = L['bn']
                conv_bn_tc(r['x'], self.packed[li], L['k'], L['cin'], L['cout'], fold=None if training else self.fold[li],
                           bias=st[L['b']], gamma=st[bn['gamma']], beta=st[bn['beta']], stats=self.stats.get(li),
                           workspace=self.ws, pool=r['pool'], out_f32=li == nl - 1, out=r['out'], ldo=r['ldo'], col=r['col'],
                           s2d=r['s2d'], x3=self.x3, raw=self.raw.get(li))
                if r['pooled'] is not None:
                    ops.maxpool2x2_bf16(self.pt_src, out=r['pooled'])
            x = self.acts[li]
        if self.decode == 'region':
            if self.C == 20 and self.nbox <= 4095 and self.fused_detect:
                if self.detect_impl == 'split' and self.A == 5:
                    ops.detect_split(self.acts[-1], self.anchors, self.C, self.score_thresh, self.iou_thresh, self.max_keep,
                                     boxes=self.boxes, scores=self.scores, keep_idx=self.keep_idx, keep_count=self.keep_count,
                                     workspace=self.detect_ws)
                else:
                    ops.detect_fused(self.acts[-1], self.anchors, self.C, self.score_thresh, self.iou_thresh, self.max_keep,
                                     boxes=self.boxes, scores=self.scores, keep_idx=self.keep_idx, keep_count=self.keep_count)
            else:
                ops.decode_region(self.acts[-1], self.anchors, self.C, self.score_thresh, boxes=self.boxes,
                                  scores=self.scores)
                ops.nms(self.boxes, self.scores, self.score_thresh, self.iou_thresh, self.max_keep,
                        keep_idx=self.keep_idx, keep_count=self.keep_count)

    def run(self):
        """Enqueue one step (input already in self.in_u8 / self.in_f32) on the current stream."""
        if self._version != self.store.version:
            self.refresh_weights()
        if not self.use_cuda_graph:
            self._enqueue()
            return
        if self.graph is None:
            s = torch.cuda.Stream(device=self.device)
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                self._enqueue()            # warm-up: sets func attributes, primes caches
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize(self.device)
            n0 = ops.launch_count()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._enqueue()
            self.launches_per_step = ops.launch_count() - n0
            self.graph = g
        self.graph.replay()

    # ------------------------------------------------------------------------------------------
    # pipelined serving path: H2D of batch i+1 overlaps the compute of batch i
    # ------------------------------------------------------------------------------------------
    def _pipeline_init(self):
        dev = self.device
        self._copy_stream = torch.cuda.Stream(device=dev)
        src = self.in_u8 if self.input_kind == 'u8' else self.in_f32
        self._staging = [torch.empty_like(src) for _ in range(2)]
        self._ready = [torch.cuda.Event() for _ in range(2)]
        self._free = [torch.cuda.Event() for _ in range(2)]
        self._slot = 0
        for e in self._free:
            e.record(torch.cuda.current_stream(dev))
        # results leave through a second side stream: a small device-side snapshot of the outputs (two buffers), then the
        # device->host copy runs while the NEXT batch computes (the outputs themselves are overwritten by it)
        self._out_stream = torch.cuda.Stream(device=dev)
        self._out_stage = [dict(), dict()]
        self._out_ready = [torch.cuda.Event() for _ in range(2)]
        self._out_free = [torch.cuda.Event() for _ in range(2)]
        self._out_slot = 0
        for e in self._out_free:
            e.record(torch.cuda.current_stream(dev))

    def submit(self, host_images, out_host=None):
        """Enqueue one batch from (pinned) host memory: the host->device copy runs on a copy stream into one of two
        staging buffers, so it overlaps the previous batch's kernels; the step itself and the device->host copy of
        the detections (into `out_host`: dict of pinned tensors keyed keep_idx / keep_count / boxes / scores / net)
        runs on the current stream; the results are snapshotted on the device and copied to the host on a second side
        stream, behind the next batch's kernels.  Returns immediately; call wait_outputs() + synchronise the current stream
        (or torch.cuda.synchronize()) before reading `out_host`.  Successive calls that pass the SAME host buffers
        overwrite them in submission order."""
        if not hasattr(self, '_copy_stream'):
            self._pipeline_init()
        cur = torch.cuda.current_stream(self.device)
        i = self._slot
        self._slot ^= 1
        with torch.cuda.stream(self._copy_stream):
            self._copy_stream.wait_event(self._free[i])
            self._staging[i].copy_(torch.as_tensor(host_images), non_blocking=True)
            self._ready[i].record(self._copy_stream)
        cur.wait_event(self._ready[i])
        srcs = dict(net=self.acts[-1])
        if self.decode == 'region':
            srcs.update(boxes=self.boxes, scores=self.scores, keep_idx=self.keep_idx, keep_count=self.keep_count)
        j = stage = None
        if out_host is not None:
            j = self._out_slot
            self._out_slot ^= 1
            stage = self._out_stage[j]
            for k in out_host:
                if k not in stage:
                    stage[k] = torch.empty_like(srcs[k])
            cur.wait_event(self._out_free[j])                   # the D2H that last read this snapshot has finished
        if self.use_cuda_graph and self.input_kind == 'u8':
            # one CUDA graph per staging slot: the first conv reads the staging buffer DIRECTLY (no device-side copy of the
            # 33 MB batch) and the snapshot of the results is part of the graph -- one launch per batch on the compute stream
            if self._version != self.store.version:
                self.refresh_weights()
            key = (i, j, tuple(sorted(out_host)) if out_host is not None else ())
            g = self._pipe_graphs.get(key)
            if g is None:
                if self.graph is None:
                    self.run()                                  # warm-up + the plain graph (sets launches_per_step)
                saved, self.in_u8 = self.in_u8, self._staging[i]
                try:
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        self._enqueue()
                        for k in (out_host or ()):
                            stage[k].copy_(srcs[k], non_blocking=True)
                finally:
                    self.in_u8 = saved
                self._pipe_graphs[key] = g
            g.replay()
            self._free[i].record(cur)
        else:
            (self.in_u8 if self.input_kind == 'u8' else self.in_f32).copy_(self._staging[i], non_blocking=True)
            self._free[i].record(cur)
            self.run()
            for k in (out_host or ()):
                stage[k].copy_(srcs[k], non_blocking=True)      # device-side snapshot (on the compute stream)
        if out_host is not None:
            self._out_ready[j].record(cur)
            with torch.cuda.stream(self._out_stream):
                self._out_stream.wait_event(self._out_ready[j])
                for k, dst in out_host.items():
                    dst.copy_(stage[k], non_blocking=True)
                self._out_free[j].record(self._out_stream)
            self._last_out_event = self._out_free[j]

    def wait_outputs(self):
        """Make the current stream wait for the device->host copies of every submit() so far (then synchronise the stream,
        or use torch.cuda.synchronize(), before reading the host buffers)."""
        ev = getattr(self, '_last_out_event', None)
        if ev is not None:
            torch.cuda.current_stream(self.device).wait_event(ev)

    def load_images(self, images_bgr_u8):
        """Fill the input batch from RAW decoded images of any size (list of uint8 [H,W,3] BGR arrays / tensors, host or
        device): each is copied to the device as it is and resized there by y2_resize_bilinear_u8 -- bit-identical to the
        cv2.resize((IS, IS)) of pascal_detect_darknet.py:35 -- straight into its row of the uint8 batch (the /255*2-1 is
        fused into the first conv).  At tens of thousands of images per second the host-side cv2.resize is the bottleneck."""
        assert self.input_kind == 'u8' and len(images_bgr_u8) <= self.N
        for n, im in enumerate(images_bgr_u8):
            t = torch.as_tensor(im)
            assert t.dtype == torch.uint8 and t.dim() == 3 and t.shape[2] == 3
            t = t.to(self.device, non_blocking=True).contiguous()
            ops.resize_bilinear_u8(t, self.IS, self.IS, out=self.in_u8[n])
        return self.in_u8

    @property
    def net_out(self):
        return self.acts[-1]

    def layer_activation(self, li):
        """Layer li's activation as float32 [N,H,W,C] (bf16x3: hi + lo re-joined) -- for parity tests / error attribution."""
        a = self.acts[li]
        if a.dtype == torch.float32:
            return a
        if self.x3:
            c = a.shape[-1] // 2
            return a[..., :c].float() + a[..., c:].float()
        return a.float()

    def infer(self, images):
        """images: uint8 [N,IS,IS,3] BGR (host or device) or float32 (input_kind='f32').
        Returns dict(net, boxes, scores, keep_idx, keep_count) of device tensors."""
        dst = self.in_u8 if self.input_kind == 'u8' else self.in_f32
        dst.copy_(torch.as_tensor(images), non_blocking=True)
        self.run()
        out = dict(net=self.acts[-1])
        if self.decode == 'region':
            out.update(boxes=self.boxes, scores=self.scores, keep_idx=self.keep_idx, keep_count=self.keep_count)
        return out
