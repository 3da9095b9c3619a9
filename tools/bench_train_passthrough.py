"""Cost of training the YOLOv2 passthrough graph: the CUDA-graphed region-loss training step with and without the passthrough
branch (Yolo2Trainer(passthrough=False / True)), in one process, the two trainers alternated round by round so that both see
the same clocks and neighbours.  Prints one JSON line: the median device time per step of each (CUDA events around K replays
per round), their ratio, the eager phase times (phase_times) of each, and the card's name and power limit.

    python tools/bench_train_passthrough.py [--batch 64] [--image-size 416] [--steps 20] [--rounds 5]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))
from tensorflow_yolo2_b200.trainer import Yolo2Trainer                 # noqa: E402


def card():
    """Name and power limit of GPU 0 (a read-only nvidia-smi query)."""
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()[0]
        name, limit = [s.strip() for s in out.split(',')]
        return dict(name=name, power_limit=limit)
    except Exception as e:  # noqa: BLE001
        return dict(name=torch.cuda.get_device_name(0), power_limit='unknown (%s)' % type(e).__name__)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batch', type=int, default=64)
    ap.add_argument('--image-size', type=int, default=416)
    ap.add_argument('--steps', type=int, default=20, help='replays per round and trainer')
    ap.add_argument('--rounds', type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('bench_train_passthrough.py needs a CUDA device')
    torch.cuda.set_device(0)
    N, IS = args.batch, args.image_size
    rs = np.random.RandomState(0)
    images = torch.as_tensor(rs.randint(0, 256, (N, IS, IS, 3)).astype(np.uint8)).cuda()
    counts = rs.randint(1, 7, N).astype(np.int32)
    boxes = np.zeros((N, 32, 4), dtype=np.float32)
    classes = np.zeros((N, 32), dtype=np.int32)
    for n in range(N):
        for g in range(counts[n]):
            boxes[n, g] = [rs.uniform(0.05, 0.95), rs.uniform(0.05, 0.95), rs.uniform(0.05, 0.7), rs.uniform(0.05, 0.7)]
            classes[n, g] = rs.randint(0, 20)
    trainers = {}
    for pt in (False, True):
        tr = Yolo2Trainer(N, IS, loss='region', device='cuda:0', use_cuda_graph=True, passthrough=pt, seed=1)
        tr.set_ground_truth(boxes, classes, counts)
        tr.step(images)                                  # capture + warm-up
        for _ in range(3):
            tr.step()
        trainers[pt] = tr
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = {False: [], True: []}
    for _ in range(args.rounds):
        for pt in (False, True):
            tr = trainers[pt]
            e0.record()
            for _ in range(args.steps):
                tr.step()
            e1.record()
            e1.synchronize()
            times[pt].append(e0.elapsed_time(e1) / args.steps)
    med = {pt: float(np.median(v)) for pt, v in times.items()}
    phases = {pt: trainers[pt].phase_times(iters=3) for pt in (False, True)}
    out = dict(metric='train_step_ms', image_size=IS, batch=N, loss='region', cuda_graph=True, steps_per_round=args.steps,
               rounds=args.rounds, plain_ms=round(med[False], 4), passthrough_ms=round(med[True], 4),
               ratio=round(med[True] / med[False], 4), plain_ms_rounds=[round(t, 4) for t in times[False]],
               passthrough_ms_rounds=[round(t, 4) for t in times[True]], phases_plain=phases[False],
               phases_passthrough=phases[True], launches_per_step=dict(plain=trainers[False].launches_per_step,
                                                                        passthrough=trainers[True].launches_per_step),
               gpu=card())
    print(json.dumps(out))


if __name__ == '__main__':
    main()
