#!/usr/bin/env python
"""bench.py -- images/sec of Darknet19-YOLO2 416x416 inference (forward + region decode + per-class
NMS), the metric BASELINE.json names, on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--precision bf16|bf16x3]   # this repo's CUDA path
    python bench.py --impl reference [--steps K] [--warmup W]        # CPU restatement of the reference
    python bench.py --mode train [...]                               # one training step (BASELINE configs[4])
    torchrun ... bench.py --gpus N ...                               # N > 1: one rank per GPU

One "step" = one pass of the hot path over one synthetic batch (64 images of 416x416x3 uint8 per
GPU, random-init weights of the reference's initialiser, core BN in inference mode, head BN in
batch-statistics mode -- the reference detect script's graph).  Prints ONE JSON line (rank 0).

precision  BOTH modes are timed in one invocation (--single-mode: only the selected one).  `--precision` (default bf16, the
           dtype north_star names for the convs) picks the mode behind value / e2e / roofline and is printed as
           config.precision; the other one is summarised under precision_modes.  bf16x3 is the mode that meets the 1e-3
           detections bar (tests/test_parity_gpu.py, profiles/r2*_parity.json); plain bf16 measures 4e-2 on the net output.
value      device-timed throughput of exactly K steps with the batch already resident in HBM (CUDA events per step on
           the launching stream, L2 flushed between steps, max over ranks).
e2e        same metric through Yolo2Engine.submit(): pinned host uint8 batch -> H2D -> step -> D2H of the
           detections, every copy inside the timed region (H2D of batch i+1 on a copy stream, D2H of batch i-1 on a
           second one, both behind the kernels of batch i, as a serving loop would).
roofline   tensor-core bound, recomputable by hand: achieved = batch x algorithmic conv FLOPs / (conv_share_of_step x
           ms_per_step); conv_share_of_step = time of the 22 conv launches / time of the step, both from CUDA-event NODES
           inside a graph replay of the step (live, this run); peak = the burst figure of MEASURED_PEAKS.json when the K
           timed steps took < 1 s of wall clock, the sustained one otherwise (regime + all three fractions printed).
           roofline.traffic = DRAM bytes of the conv launches from the ncu launch list tools/profile_step.sh committed
           (profiles/r2*_traffic_<mode>.json, with the git HEAD it was taken at).
sustained  the same step back to back for >= --sustain-seconds (3 s): value of the last quarter of the run + its clocks.
cpu_baseline  the oracle (CPU restatement of the reference, PyTorch-CPU fp32) on a bounded sample.

    --image-size 608 --batch 32    BASELINE.json configs[3] (19x19 grid) instead of the headline 416 / 64
    --no-graph                     eager launches (for ncu launch lists);  --no-cpu-baseline skips the CPU leg
    --dump-outputs DIR             after the K timed steps, write what the last one computed (rank 0, --precision mode) as
                                   DIR/<name>.npy: infer -> net, boxes, scores, keep_idx, keep_count (what Yolo2Engine.infer
                                   returns); train -> loss_terms (what Yolo2Trainer.step returns) and params_strided (every
                                   k-th weight after the update).  Inputs and weights are seeded, so the same arguments give
                                   the same inputs on every run and two builds can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH_PER_GPU = 64
IMAGE_SIZE = 416
OUTPUT_FILTER = 125
SCORE_THRESH, IOU_THRESH = 0.3, 0.45
METRIC = 'images/sec Darknet19-YOLO2 416x416 (fwd+decode+NMS)'

# (k, cin, cout, out_hw) at 416^2 -> algorithmic FLOPs = 2*k*k*cin*cout*hw*hw   (SURVEY 8d)
def conv_flops_per_image(image_size, output_filter):
    from tensorflow_yolo2_b200.yolo2_nets.darknet import CORE_PLAN
    h = image_size
    total, per = 0.0, []
    plan = list(CORE_PLAN) + [(3, 1024, 1024, False)] * 3 + [(1, 1024, output_filter, False)]
    for (k, cin, cout, pool) in plan:
        f = 2.0 * k * k * cin * cout * h * h
        per.append(f)
        total += f
        if pool:
            h //= 2
    return total, per


def make_config(world, precision='bf16', extra=None):
    """config of the bench line -- the reference arm prints the same one (it is the driver's join key)."""
    cfg = dict(workload='Darknet19-YOLO2 %dx%d inference, fwd + region decode + per-class NMS, synthetic uint8 batch ' % (IMAGE_SIZE, IMAGE_SIZE) +
                        '%d per GPU (BASELINE.json configs[%d])' % (BATCH_PER_GPU, 1 if IMAGE_SIZE == 416 else 3),
               global_batch=world * BATCH_PER_GPU, image_size=IMAGE_SIZE, output_filter=OUTPUT_FILTER,
               score_thresh=SCORE_THRESH, iou_thresh=IOU_THRESH, head_bn='batch statistics',
               l2='flushed (256 MiB memset) between timed steps', parallelism='batch sharding x%d' % world,
               precision=precision)
    if extra:
        cfg.update(extra)
    return cfg


PRECISION_NOTE = {
    'bf16': 'every conv operand rounded once to bf16, fp32 accumulate (one tcgen05.mma per K step); detections vs the float64 '
            'oracle: see profiles/r2_parity.json (net rel-L2 ~4e-2, scores up to 1e-1 off)',
    'bf16x3': 'hi+lo bf16 operand pairs, a_hi*w_hi + a_lo*w_hi + a_hi*w_lo (three tcgen05.mma per K step), fp32 accumulate; '
              'meets the 1e-3 bar on decoded boxes / scores (tests/test_parity_gpu.py, profiles/r2_parity.json)',
}


def load_traffic(precision):
    """DRAM bytes (read + write) of the 22 conv launches of one step, from the ncu launch list of this same command
    committed by tools/profile_step.sh (ncu numbers are never taken live inside a timed run).  Returns (bytes, source, head)."""
    import glob
    cands = sorted(glob.glob(os.path.join(ROOT, 'profiles', 'r2*_traffic_%s.json' % precision)))
    for p in reversed(cands):
        try:
            d = json.load(open(p))
            return float(d['conv_dram_bytes_per_step']), os.path.relpath(p, ROOT), d.get('head'), d.get('conv_share_of_step_under_ncu')
        except Exception:  # noqa: BLE001
            continue
    return None, None, None, None


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(burst=d.get('bf16_tflops', 1590.0), sustained=d.get('bf16_tflops_sustained', 1400.0),
                    hbm=d.get('hbm_gbs', 6650.0), which='measured (MEASURED_PEAKS.json)')
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, which='fallback (B200_PROFILING.md)')


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays, batch_major=True):
    """Write arrays as out_dir/<name>.npy: floating ones as float32, integer ones as float64 (exact for int32).  When
    batch-major arrays together exceed DUMP_LIMIT_BYTES, the same seeded sample of images (rows of axis 0) is kept from
    each, and its row numbers are written as sampled_rows.npy."""
    import numpy as np
    arrays = {k: a.astype(np.float32 if np.issubdtype(a.dtype, np.floating) else np.float64) for k, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if batch_major and total > DUMP_LIMIT_BYTES:
        n = next(iter(arrays.values())).shape[0]
        keep = max(1, n * DUMP_LIMIT_BYTES // (total + 8 * n))
        rows = np.sort(np.random.RandomState(0).choice(n, keep, replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays['sampled_rows'] = rows.astype(np.float64)
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_LIMIT_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + '.npy'), a)


def engine_outputs(eng):
    """What Yolo2Engine.infer() hands its caller, as numpy.  Slots of keep_idx past keep_count still hold what an earlier
    step left there, so they are written as -1."""
    import numpy as np
    out = {k: t.cpu().numpy() for k, t in dict(net=eng.net_out, boxes=eng.boxes, scores=eng.scores, keep_idx=eng.keep_idx,
                                                keep_count=eng.keep_count).items()}
    slot = np.arange(out['keep_idx'].shape[-1])
    out['keep_idx'] = np.where(slot < out['keep_count'][..., None], out['keep_idx'], -1)
    return out


class ClockSampler:
    """SM clock / throttle reasons DURING the timed region, sampled in-process through NVML every 20 ms (the
    B200_PROFILING.md recipe's nvidia-smi query, without a subprocess' start-up latency)."""

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.maxclk = index, [], set(), None
        self._stop = None
        self._thr = None

    def start(self):
        import threading
        try:
            import pynvml
            pynvml.nvmlInit()
            try:
                import torch
                uuid = 'GPU-' + str(torch.cuda.get_device_properties(self.index).uuid)
                h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.maxclk = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception:
            return
        names = dict(hw_slowdown=0x8, hw_thermal_slowdown=0x40, sw_thermal_slowdown=0x20, sw_power_cap=0x4)   # NVML reason bits
        self._stop = threading.Event()

        def loop():
            while not self._stop.is_set():
                try:
                    self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                    try:
                        r = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                    except Exception:
                        r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for k, bit in names.items():
                        if r & bit:
                            self.reasons.add(k)
                except Exception:
                    pass
                self._stop.wait(0.02)
        self._thr = threading.Thread(target=loop, daemon=True)
        self._thr.start()

    def stop(self):
        if self._thr is None:
            return None
        self._stop.set()
        self._thr.join(timeout=2)
        if not self.samples:
            return None
        return dict(sm_mhz=statistics.median(self.samples), sm_min_mhz=min(self.samples), sm_max_mhz=self.maxclk,
                    reasons=sorted(self.reasons), samples=len(self.samples))


# ------------------------------------------------------------------------------------------------
# CPU restatement of the reference (oracle) -- used ONLY for cpu_baseline / --impl reference
# ------------------------------------------------------------------------------------------------
def cpu_reference_step(batch, threads=None, reps=1, seed=0):
    import numpy as np
    import torch
    from oracle import yolo2_oracle as O
    from tests.helpers import make_store, oracle_params
    if threads:
        torch.set_num_threads(threads)
    st, layers = make_store(OUTPUT_FILTER, seed=seed)
    core_p, head_p = oracle_params(st, layers)
    img = np.random.RandomState(seed).randint(0, 256, (batch, IMAGE_SIZE, IMAGE_SIZE, 3)).astype(np.uint8)
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        x = torch.tensor(O.preprocess_u8(img))
        with torch.no_grad():
            net = O.darknet19_forward(x, core_p, head_p, core_training=False, head_training=True,
                                      dtype=torch.float32).numpy()
        boxes, sthr, _ = O.region_decode_v2(net, O.VOC_ANCHORS, 20, SCORE_THRESH)
        for n in range(batch):
            O.nms_per_class(boxes[n], sthr[n], IOU_THRESH, SCORE_THRESH)
        times.append(time.perf_counter() - t0)
    return times, torch.get_num_threads()


def run_reference(args):
    """Reference arm: the CPU restatement of the reference's path (the reference itself cannot run: DESIGN.md section 2) on
    the box's host cores, the SAME workload per step (batch 64 of 416x416: forward + decode + NMS)."""
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sample_batch = BATCH_PER_GPU
    t_all, threads = cpu_reference_step(sample_batch, threads=cores, reps=args.warmup + args.steps)
    timed = t_all[args.warmup:]
    total = sum(timed)
    value = sample_batch * len(timed) / total
    sample = 'the whole batch of %d x %dx%d per step, torch-CPU fp32 restatement of the reference' % (sample_batch, IMAGE_SIZE, IMAGE_SIZE)
    line = dict(metric=METRIC.replace('416x416', '%dx%d' % (IMAGE_SIZE, IMAGE_SIZE)), value=value, unit='images/s', n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * total / len(timed), higher_is_better=True, scaling='weak', vs_baseline=None,
                dtype='f32', data='synthetic', impl='reference',
                config=make_config(max(args.gpus, 1), args.precision),
                cpu_baseline=dict(value=value, unit='images/s', cores=threads, kind='port', sample=sample),
                e2e=dict(value=value, unit='images/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def measure_mode(precision, args, world, rank, dev, dist, sampler_index):
    """Time one precision mode: device-timed value (K steps, L2 flushed between them), e2e from pinned host memory, a
    >= 3 s sustained run, and the conv kernels' share of the step timed live inside an instrumented graph replay."""
    import torch
    from tensorflow_yolo2_b200 import ops
    from tensorflow_yolo2_b200.engine import Yolo2Engine

    N = BATCH_PER_GPU
    eng = Yolo2Engine(N, IMAGE_SIZE, OUTPUT_FILTER, score_thresh=SCORE_THRESH, iou_thresh=IOU_THRESH, max_keep=64,
                      use_cuda_graph=not args.no_graph, device=dev, seed=0, precision=precision)
    g = torch.Generator(device='cpu').manual_seed(1234 + rank)
    host_batches = [torch.randint(0, 256, (N, IMAGE_SIZE, IMAGE_SIZE, 3), dtype=torch.uint8, generator=g).pin_memory()
                    for _ in range(2)]
    dev_batches = [b.to(dev) for b in host_batches]
    flush = torch.empty((256 << 20,), dtype=torch.uint8, device=dev)      # > 126 MB L2
    stream = torch.cuda.current_stream()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(ms):
        tt = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    def one_step(i, timed):
        eng.in_u8.copy_(dev_batches[i % len(dev_batches)])       # device->device, outside the events
        flush.zero_()                                            # L2 flush, outside the events
        if timed:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            eng.run()
            e1.record(stream)
            return e0, e1
        eng.run()
        return None

    # ---- value: exactly K timed steps ----
    for i in range(max(args.warmup, 3)):
        one_step(i, False)
    barrier()
    sampler = ClockSampler(sampler_index)
    if rank == 0:
        sampler.start()
    n_launch0 = ops.launch_count()
    t_wall0 = time.perf_counter()
    evs = [one_step(i, True) for i in range(args.steps)]
    eager_launches = ops.launch_count() - n_launch0          # 0 under CUDA-graph replay (counted at capture)
    barrier()
    timed_region_s = time.perf_counter() - t_wall0
    clocks = sampler.stop() if rank == 0 else None
    t_ms = allmax(sum(a.elapsed_time(b) for a, b in evs))
    value = world * N * args.steps / (t_ms * 1e-3)
    ms_per_step = t_ms / args.steps
    cand = int((eng.scores > 0).sum().item())
    kept = int(eng.keep_count.sum().item())
    if args.dump_outputs and rank == 0 and precision == args.precision:
        dump_outputs(args.dump_outputs, engine_outputs(eng))

    # ---- e2e: pinned host uint8 -> H2D -> step -> D2H (keep lists + boxes of the batch) ----
    res_host = dict(keep_idx=torch.empty(eng.keep_idx.shape, dtype=torch.int32).pin_memory(),
                    keep_count=torch.empty(eng.keep_count.shape, dtype=torch.int32).pin_memory(),
                    boxes=torch.empty(eng.boxes.shape, dtype=torch.float32).pin_memory())
    h2d = host_batches[0].numel()
    d2h = sum(t.numel() * t.element_size() for t in res_host.values())
    for i in range(3):
        eng.submit(host_batches[i % 2], res_host)                 # H2D (copy stream) | step | D2H, pipelined
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(args.steps):
        eng.submit(host_batches[i % 2], res_host)
    eng.wait_outputs()                                            # the last batch's results have reached the host buffers
    e1.record(stream)
    barrier()
    e2e_value = world * N * args.steps / (allmax(e0.elapsed_time(e1)) * 1e-3)

    # ---- sustained: the same step back to back for >= 3 s (power-capped clocks), same flush between steps ----
    sustained = None
    if args.sustain_seconds > 0 and not args.no_graph:
        n_sus = max(args.steps, int(args.sustain_seconds / max(ms_per_step * 1e-3 + 6e-5, 1e-5)))
        barrier()
        samp2 = ClockSampler(sampler_index)
        if rank == 0:
            samp2.start()
        evs2 = [one_step(i, True) for i in range(n_sus)]
        barrier()
        clk2 = samp2.stop() if rank == 0 else None
        # the last quarter of the run: clocks have settled under the power cap
        tail = evs2[-max(1, n_sus // 4):]
        t_tail = allmax(sum(a.elapsed_time(b) for a, b in tail))
        sustained = dict(value=world * N * len(tail) / (t_tail * 1e-3), ms_per_step=t_tail / len(tail), steps_run=n_sus,
                         steps_counted=len(tail), clocks=clk2)

    out = dict(precision=precision, value=value, ms_per_step=ms_per_step, t_ms=t_ms, timed_region_s=timed_region_s, clocks=clocks,
               e2e=dict(value=e2e_value, unit='images/s', h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h), sustained=sustained,
               nms_candidates=cand, nms_kept=kept,
               launches_per_step=int(eng.launches_per_step if not args.no_graph else eager_launches // max(args.steps, 1)))
    if rank == 0:
        out['conv'] = conv_share_live(eng, ops, flush, iters=max(3, min(args.steps, 10)))
    del eng
    torch.cuda.empty_cache()
    return out


def build_roofline(m, peaks):
    """Tensor-core roofline of the conv kernels of one mode, recomputable by hand from the line:
        achieved = batch * algorithmic conv FLOPs per image / (conv_share * ms_per_step)       [TFLOP/s]
        frac     = achieved / peak,  peak = burst figure when the K timed steps took < 1 s of wall clock (a kernel timed
                   alone / a short region runs at full clocks), the sustained one otherwise (MEASURED_PEAKS.json's definition)
    conv_share = time of the 22 conv launches / time of the whole step, both measured LIVE with CUDA events recorded as
    nodes inside a graph replay of the step."""
    N = BATCH_PER_GPU
    flops_img, per_layer = conv_flops_per_image(IMAGE_SIZE, OUTPUT_FILTER)
    conv = m['conv']
    conv_ms = conv['share'] * m['ms_per_step']
    achieved = N * flops_img / (conv_ms * 1e-3) / 1e12
    regime = 'burst' if m['timed_region_s'] < 1.0 else 'sustained'
    peak = peaks[regime]
    traffic, tsrc, thead, _ = load_traffic(m['precision'])
    if not (IMAGE_SIZE == 416 and N == 64):
        traffic, tsrc, thead = None, None, None
    mma_mult = 3 if m['precision'] == 'bf16x3' else 1
    roof = dict(bound='tensor', achieved=achieved, peak=peak, unit='TFLOP/s', frac=achieved / peak, regime=regime,
                frac_vs_burst=achieved / peaks['burst'], frac_vs_sustained=achieved / peaks['sustained'],
                frac_vs_nominal_2250=achieved / 2250.0, peak_source=peaks['which'] + ' ' + regime + ' bf16',
                traffic=traffic, traffic_source=tsrc, traffic_head=thead,
                algorithmic_bytes=N * 35.0e6 * IMAGE_SIZE * IMAGE_SIZE / (416.0 * 416.0),
                algorithmic_flops_per_step=N * flops_img, executed_mma_flops_per_step=N * flops_img * mma_mult,
                executed_tflops=achieved * mma_mult,
                kernel='conv_tc_kernel / conv_streamk2_kernel x21 + conv1_u8_pool_kernel (22 conv launches/step)',
                conv_ms_per_step=conv_ms, conv_share_of_step=conv['share'],
                conv_ms_source='share of the step taken by the 22 conv launches, CUDA-event nodes inside a graph replay '
                               '(instrumented step %.3f ms vs %.3f ms un-instrumented) x the device-timed ms_per_step'
                               % (conv['instrumented_step_ms'], m['ms_per_step']),
                per_layer_tflops=[round(N * f / (ms * 1e-3) / 1e12, 1) if ms > 0 else None for f, ms in zip(per_layer, conv['per_layer_ms'])])
    if m.get('sustained'):
        sus = m['sustained']
        roof['sustained_achieved'] = N * flops_img / (conv['share'] * sus['ms_per_step'] * 1e-3) / 1e12
        roof['sustained_frac'] = roof['sustained_achieved'] / peaks['sustained']
    return roof


def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get('WORLD_SIZE', 1))
    rank = int(os.environ.get('RANK', 0))
    local = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)

    modes = [args.precision] + ([] if args.single_mode else [p for p in ('bf16', 'bf16x3') if p != args.precision])
    results = {p: measure_mode(p, args, world, rank, dev, dist, local) for p in modes}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = load_peaks()
    main_m = results[args.precision]
    roofline = build_roofline(main_m, peaks)

    # ---- CPU baseline: oracle on a bounded sample ----
    cpu = None
    if not args.no_cpu_baseline:
        try:
            times, threads = cpu_reference_step(4, threads=os.cpu_count(), reps=2)
            cpu = dict(value=4 / min(times), unit='images/s', cores=threads, kind='port',
                       sample='batch 4 of %dx%d (fwd+decode+NMS), best of 2, torch-CPU fp32 restatement of the reference' % (IMAGE_SIZE, IMAGE_SIZE))
        except Exception as e:  # noqa: BLE001
            cpu = dict(value=None, unit='images/s', cores=os.cpu_count(), kind='port', sample='failed: %r' % (e,))

    def summary(m):
        r = build_roofline(m, peaks)
        return dict(value=m['value'], ms_per_step=m['ms_per_step'], e2e=m['e2e']['value'],
                    sustained_value=(m['sustained'] or {}).get('value'), roofline_frac=r['frac'], regime=r['regime'],
                    executed_tflops=r['executed_tflops'], conv_share_of_step=r['conv_share_of_step'],
                    per_layer_ms=[round(v, 4) for v in m['conv']['per_layer_ms']], nms_kept=m['nms_kept'], launches_per_step=m['launches_per_step'],
                    note=PRECISION_NOTE[m['precision']])

    line = dict(metric=METRIC.replace('416x416', '%dx%d' % (IMAGE_SIZE, IMAGE_SIZE)), value=main_m['value'], unit='images/s', n_gpus=world,
                steps=args.steps, warmup=max(args.warmup, 3), ms_per_step=main_m['ms_per_step'], higher_is_better=True, scaling='weak',
                vs_baseline=None, dtype='bf16', data='synthetic',
                config=make_config(world, args.precision),
                e2e=main_m['e2e'],
                gpu_launches=int(main_m['launches_per_step'] * args.steps), launches_per_step=main_m['launches_per_step'],
                roofline=roofline, cpu_baseline=cpu, clocks=main_m['clocks'],
                sustained=main_m['sustained'], detections=dict(nms_candidates=main_m['nms_candidates'], nms_kept=main_m['nms_kept']),
                precision_modes={p: summary(m) for p, m in results.items()})
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# --mode train: BASELINE.json configs[4] -- one training step (forward with batch-statistics BN in all 22 layers, the
# reference's get_loss, backward, [N > 1: bucketed NCCL gradient all-reduce overlapped with backward], Adam)
# ------------------------------------------------------------------------------------------------
TRAIN_METRIC = 'images/sec Darknet19-YOLO2 416x416 training step (fwd+loss+bwd+allreduce+Adam)'


def train_config(world, loss):
    return dict(workload='Darknet19-YOLO2 %dx%d training step, fused %s loss fwd/bwd, synthetic uint8 batch %d per GPU, '
                         'data-parallel NCCL gradient all-reduce (BASELINE.json configs[4])'
                         % (IMAGE_SIZE, IMAGE_SIZE, 'YOLO (net_utils.get_loss, C+5B = 45 channels)' if loss == 'v1' else 'region (125 channels)',
                            BATCH_PER_GPU),
                global_batch=world * BATCH_PER_GPU, image_size=IMAGE_SIZE, loss=loss, optimizer='Adam (TF defaults)',
                bn='batch statistics in all 22 layers, per-rank', l2='flushed (256 MiB memset) between timed steps',
                parallelism='data parallel x%d' % world, precision='bf16')


def synthetic_labels(rs, N, S, IS, loss, max_gt=32):
    """SURVEY 8(d) config 5: per image 1-3 GT boxes, cx,cy ~ U(0,IS), w,h ~ U(20,300), class ~ U{0..19}."""
    import numpy as np
    if loss == 'v1':
        lab = np.zeros((N, S, S, 25), dtype=np.float32)
        for n in range(N):
            for _ in range(rs.randint(1, 4)):
                cx, cy = rs.uniform(0, IS, 2)
                w, h = rs.uniform(20, 300, 2)
                j, i = min(int(cx * S / IS), S - 1), min(int(cy * S / IS), S - 1)
                if lab[n, i, j, 0] == 0:                       # first object wins a cell (pascal_voc.py:159-160)
                    lab[n, i, j, 0] = 1
                    lab[n, i, j, 1:5] = [cx, cy, w, h]
                    lab[n, i, j, 5 + rs.randint(0, 20)] = 1
        return lab
    cnt = rs.randint(1, 4, N).astype(np.int32)
    bx = np.zeros((N, max_gt, 4), dtype=np.float32)
    bx[:, :3] = np.stack([rs.uniform(0.05, 0.95, (N, 3)), rs.uniform(0.05, 0.95, (N, 3)), rs.uniform(0.05, 0.7, (N, 3)),
                          rs.uniform(0.05, 0.7, (N, 3))], axis=-1)
    return bx, rs.randint(0, 20, (N, max_gt)).astype(np.int32), cnt


def cpu_train_step(batch, threads, reps=1, seed=0):
    """The oracle's restatement of one reference training iteration (forward is_training=True, get_loss, autograd backward;
    pascal_train_darknet.py:96-102) on torch-CPU float32 -- cpu_baseline / --impl reference only."""
    import numpy as np
    import torch
    from oracle import yolo2_oracle as O
    from tests.helpers import make_store, oracle_params
    torch.set_num_threads(threads)
    S = IMAGE_SIZE // 32
    st, layers = make_store(45, seed=seed, tame=True)
    core_p, head_p = oracle_params(st, layers)
    rs = np.random.RandomState(seed)
    img = rs.randint(0, 256, (batch, IMAGE_SIZE, IMAGE_SIZE, 3)).astype(np.uint8)
    lab = torch.tensor(synthetic_labels(rs, batch, S, IMAGE_SIZE, 'v1'))
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        O.train_step_reference(O.preprocess_u8(img), core_p, head_p,
                               lambda net: O.loss_v1_graph(net, lab.to(net.dtype), 20, batch, IMAGE_SIZE, S, 5)[0],
                               bf16_operands=False, dtype=torch.float32)
        times.append(time.perf_counter() - t0)
    return times, torch.get_num_threads()


def run_reference_train(args):
    if int(os.environ.get('RANK', 0)) != 0:
        return
    cores = os.cpu_count() or 1
    sample_batch = 4
    t_all, threads = cpu_train_step(sample_batch, cores, reps=args.warmup + args.steps)
    timed = t_all[args.warmup:]
    value = sample_batch * len(timed) / sum(timed)
    sample = 'batch %d of %dx%d per step (bounded sample of the batch-%d step), torch-CPU fp32 autograd restatement' % (
        sample_batch, IMAGE_SIZE, IMAGE_SIZE, BATCH_PER_GPU)
    line = dict(metric=TRAIN_METRIC.replace('416x416', '%dx%d' % (IMAGE_SIZE, IMAGE_SIZE)), value=value, unit='images/s',
                n_gpus=args.gpus, steps=args.steps, warmup=args.warmup, ms_per_step=1e3 * sum(timed) / len(timed),
                higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f32', data='synthetic', impl='reference',
                config=train_config(max(args.gpus, 1), args.loss),
                cpu_baseline=dict(value=value, unit='images/s', cores=threads, kind='port', sample=sample),
                e2e=dict(value=value, unit='images/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


def run_train(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from tensorflow_yolo2_b200 import ops
    from tensorflow_yolo2_b200.trainer import Yolo2Trainer
    from tests.helpers import make_store

    world = int(os.environ.get('WORLD_SIZE', 1))
    rank = int(os.environ.get('RANK', 0))
    local = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    N, IS = BATCH_PER_GPU, IMAGE_SIZE
    S = IS // 32
    of = 45 if args.loss == 'v1' else 125
    st, _ = make_store(of, tame=True)                 # He-scaled weights: a training run that does not overflow in step 1
    tr = Yolo2Trainer(N, IS, of, store=st, loss=args.loss, B=5, device=dev, use_cuda_graph=not args.no_graph)
    rs = np.random.RandomState(1234 + rank)
    host_imgs = [torch.tensor(rs.randint(0, 256, (N, IS, IS, 3)).astype(np.uint8)).pin_memory() for _ in range(2)]
    dev_imgs = [b.to(dev) for b in host_imgs]
    labs = synthetic_labels(rs, N, S, IS, args.loss)
    if args.loss == 'v1':
        host_lab = torch.tensor(labs).pin_memory()
        tr.set_labels(host_lab)
    else:
        tr.set_ground_truth(*labs)
    flush = torch.empty((256 << 20,), dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(ms):
        tt = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    def one_step(i, timed):
        tr.in_u8.copy_(dev_imgs[i % 2])
        flush.zero_()
        if not timed:
            tr.step()
            return None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        tr.step()
        e1.record(stream)
        return e0, e1

    for i in range(max(args.warmup, 3)):
        one_step(i, False)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    n0 = ops.launch_count()
    t_wall0 = time.perf_counter()
    evs = [one_step(i, True) for i in range(args.steps)]
    launches = ops.launch_count() - n0
    barrier()
    timed_region_s = time.perf_counter() - t_wall0
    clocks = sampler.stop() if rank == 0 else None
    t_ms = allmax(sum(a.elapsed_time(b) for a, b in evs))
    ms_per_step = t_ms / args.steps
    value = world * N * args.steps / (t_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        params = tr.params.cpu().numpy()
        stride = -(-params.size // (4 << 20))                 # at most 4 Mi weights (16 MiB)
        dump_outputs(args.dump_outputs, dict(loss_terms=tr.terms.cpu().numpy(), params_strided=params[::stride]),
                     batch_major=False)

    # ---- e2e: pinned host images (+ labels) -> H2D -> step -> D2H of the five loss terms, every step ----
    terms_host = torch.empty((5,), dtype=torch.float32).pin_memory()
    h2d = host_imgs[0].numel() + (host_lab.numel() * 4 if args.loss == 'v1' else 0)

    def e2e_step(i):
        if args.loss == 'v1':
            tr.labels.copy_(host_lab, non_blocking=True)
        terms = tr.step(host_imgs[i % 2])
        terms_host.copy_(terms, non_blocking=True)

    for i in range(3):
        e2e_step(i)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(args.steps):
        e2e_step(i)
    e1.record(stream)
    barrier()
    e2e_value = world * N * args.steps / (allmax(e0.elapsed_time(e1)) * 1e-3)
    final_loss = float(terms_host[4])

    # ---- phases (eager, events between them) and the exposed part of the all-reduce ----
    phases = tr.phase_times(iters=3)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    graphed = tr.graph is not None or tr.seg_graphs is not None
    peaks = load_peaks()
    flops_img, _ = conv_flops_per_image(IS, of)
    alg = 3.0 * N * flops_img                                   # forward + data gradient + weight gradient
    regime = 'burst' if timed_region_s < 1.0 else 'sustained'
    achieved = alg / (ms_per_step * 1e-3) / 1e12
    roofline = dict(bound='tensor', achieved=achieved, peak=peaks[regime], unit='TFLOP/s', frac=achieved / peaks[regime], regime=regime,
                    frac_vs_burst=achieved / peaks['burst'], frac_vs_sustained=achieved / peaks['sustained'],
                    peak_source=peaks['which'] + ' ' + regime + ' bf16', traffic=None,
                    algorithmic_flops_per_step=alg,
                    kernel='conv_tc / conv_streamk2 (forward + dgrad) + conv_wgrad_tc; whole step in the denominator',
                    note='achieved = 3 x forward conv FLOPs of the batch / device-timed step (BN, loss, Adam and the all-reduce included)')
    cpu = None
    if not args.no_cpu_baseline:
        try:
            times, threads = cpu_train_step(2, os.cpu_count() or 1, reps=2)
            cpu = dict(value=2 / min(times), unit='images/s', cores=threads, kind='port',
                       sample='batch 2 of %dx%d, one training iteration (fwd + get_loss + autograd bwd), best of 2, torch-CPU fp32' % (IS, IS))
        except Exception as e:  # noqa: BLE001
            cpu = dict(value=None, unit='images/s', cores=os.cpu_count(), kind='port', sample='failed: %r' % (e,))
    line = dict(metric=TRAIN_METRIC.replace('416x416', '%dx%d' % (IS, IS)), value=value, unit='images/s', n_gpus=world,
                steps=args.steps, warmup=max(args.warmup, 3), ms_per_step=ms_per_step, higher_is_better=True, scaling='weak',
                vs_baseline=None, dtype='bf16', data='synthetic', config=train_config(world, args.loss),
                e2e=dict(value=e2e_value, unit='images/s', h2d_bytes_per_step=h2d, d2h_bytes_per_step=20),
                gpu_launches=int(tr.launches_per_step * args.steps if graphed else launches),
                launches_per_step=int(tr.launches_per_step if graphed else launches // max(args.steps, 1)),
                cuda_graph=('one graph' if tr.graph is not None else '%d graphs (one per stretch between bucket launches) + update'
                            % len(tr.seg_graphs[0])) if graphed else False, roofline=roofline, cpu_baseline=cpu, clocks=clocks, phases_ms=phases,
                allreduce=dict(bytes_per_step=int(tr.arena_elems * 4) if world > 1 else 0, buckets=len(tr.buckets) if world > 1 else 0,
                               exposed_ms=phases.get('allreduce_exposed')),
                final_loss=final_loss)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def conv_share_live(eng, ops, flush, iters=5):
    """Share of the step spent in the 22 conv launches, measured live: the step is captured into a CUDA graph with
    event-record NODES (torch.cuda.Event(external=True)) before and after every conv launch and at both ends, replayed
    `iters` times with the L2 flushed in between, and the events read back.  (The event nodes cut the programmatic-dependent-
    launch edges between consecutive kernels, so the instrumented step is a few per cent slower than the real one -- which is
    why only the SHARE is taken from it, and applied to the un-instrumented device-timed step.)"""
    import torch
    real, real1 = ops.conv_fwd_bf16, ops.conv1_u8_pool
    nl = len(eng.layers)
    ev = lambda: torch.cuda.Event(enable_timing=True, external=True)
    pairs = []
    t_begin, t_end = ev(), ev()

    def timed(fn):
        def wrapper(*a, **k):
            e0, e1 = ev(), ev()
            e0.record()
            out = fn(*a, **k)
            e1.record()
            pairs.append((e0, e1))
            return out
        return wrapper

    s = torch.cuda.Stream(device=eng.device)
    s.wait_stream(torch.cuda.current_stream())
    ops.conv_fwd_bf16, ops.conv1_u8_pool = timed(real), timed(real1)     # the engine calls them in layer order
    try:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            t_begin.record()
            eng._enqueue()
            t_end.record()
    finally:
        ops.conv_fwd_bf16, ops.conv1_u8_pool = real, real1
    assert len(pairs) == nl, (len(pairs), nl)
    per_layer = [0.0] * nl
    step_ms = 0.0
    for _ in range(iters + 1):
        flush.zero_()
        g.replay()
        torch.cuda.synchronize()
        if _ == 0:
            continue                                   # first replay: warm-up
        step_ms += t_begin.elapsed_time(t_end) / iters
        for i, (a, b) in enumerate(pairs):
            per_layer[i] += a.elapsed_time(b) / iters
    return dict(share=min(1.0, sum(per_layer) / step_ms), instrumented_step_ms=step_ms, per_layer_ms=per_layer)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--mode', default='infer', choices=['infer', 'train'],
                    help='infer: the headline metric (BASELINE configs[1]/[3]); train: one training step (configs[4])')
    ap.add_argument('--loss', default='v1', choices=['v1', 'region'], help='--mode train: the reference get_loss (45 ch) or the region loss (125 ch)')
    ap.add_argument('--precision', default='bf16', choices=['bf16', 'bf16x3'],
                    help="mode that produces value / e2e / roofline (config.precision); the other mode is timed too and "
                         "reported under precision_modes unless --single-mode")
    ap.add_argument('--single-mode', action='store_true')
    ap.add_argument('--sustain-seconds', type=float, default=3.0, help='length of the sustained run (0 = skip)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-graph', action='store_true', help='eager launches (for ncu launch lists)')
    ap.add_argument('--image-size', type=int, default=None, help='416 (headline, BASELINE configs[1]) or 608 (configs[3])')
    ap.add_argument('--batch', type=int, default=None, help='images per GPU (default 64; configs[3] uses 32 at 608)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the outputs of the last timed step as DIR/<name>.npy (float32 / float64, <= 64 MiB in all)')
    args = ap.parse_args()
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the CUDA path (--impl ours)')
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    global IMAGE_SIZE, BATCH_PER_GPU
    if args.image_size:
        IMAGE_SIZE = args.image_size
    if args.batch:
        BATCH_PER_GPU = args.batch
    if args.mode == 'train':
        (run_reference_train if args.impl == 'reference' else run_train)(args)
    elif args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
