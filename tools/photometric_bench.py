#!/usr/bin/env python
"""Time the reference's full photometric `image_train` chain (RandomBlur .. RandomGamma) as one `yb_photometric_u8` launch.

    python tools/photometric_bench.py [--batch 64] [--size 416] [--iters 200] [--out profiles/photometric_bench.json]

B uint8 [H, W, 3] frames per launch, every image with its own draws from the reference config's ranges.  Four input batches rotate so
the working set (4 x B x H x W x 3 bytes in, the same out) is not served from L2 alone; CUDA events over `--iters` launches after a
warm-up.  Reports us per batch and the achieved bytes/s (one read and one write of every frame) as a fraction of 7.7 TB/s (the HBM3e
data-sheet figure for one B200), beside the card name and power limit read in the same run, and the host cost of the same chain in
ms/image on one core: cv2 when it is installed (the reference's own arithmetic), the numpy oracle otherwise."""
import argparse
import configparser
import json
import os
import random
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'yolo2-pytorch_b200'))
sys.path.insert(0, ROOT)
import transform  # noqa: E402
import transform.image as TI  # noqa: E402
from b200 import ops as _ops  # noqa: E402
from oracle import photometric as P  # noqa: E402
from oracle import yolo2_oracle as O  # noqa: E402

CHAIN = ['RandomBlur', 'BGR2HSV', 'RandomHue', 'RandomSaturation', 'RandomBrightness', 'HSV2RGB', 'RandomGamma']
AUG = {'random_blur': '5 5', 'random_hue': '0 25', 'random_saturation': '0.5 1.5', 'random_brightness': '0.5 1.5', 'random_gamma': '0.9 1.5'}
PEAK_BPS = 7.7e12


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', str(torch.cuda.current_device())],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ''
    return q or torch.cuda.get_device_name()


def host_ms_per_image(frame, n=8):
    """One core, the same chain with the reference's draws: cv2 (the reference's arithmetic) when present, else the numpy oracle."""
    try:
        import cv2
        cv2.setNumThreads(1)

        def run(img):
            img = cv2.blur(img, (random.randint(1, 5), random.randint(1, 5)))
            hsv = cv2.cvtColor(img, cv2.COLOR_BGR2HSV)
            h, s, v = cv2.split(hsv)
            h = np.clip(h.astype(int) + random.randint(0, 25), 0, 179).astype(np.uint8)
            s = np.clip(s * random.uniform(0.5, 1.5), 0, 255).astype(np.uint8)
            v = np.clip(v * random.uniform(0.5, 1.5), 0, 255).astype(np.uint8)
            rgb = cv2.cvtColor(cv2.merge((h, s, v)), cv2.COLOR_HSV2RGB)
            return P.gamma_table(random.uniform(0.9, 1.5))[rgb]
        how = 'cv2 %s, one thread' % cv2.__version__
    except ImportError:
        def run(img):
            return P.chain(img, (random.randint(1, 5), random.randint(1, 5)), random.randint(0, 25), random.uniform(0.5, 1.5),
                           random.uniform(0.5, 1.5), random.uniform(0.9, 1.5))
        how = 'numpy oracle (cv2 not installed)'
    run(frame)
    t = time.perf_counter()
    for _ in range(n):
        run(frame)
    return (time.perf_counter() - t) * 1e3 / n, how


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batch', type=int, default=64)
    ap.add_argument('--size', type=int, default=416)
    ap.add_argument('--iters', type=int, default=200)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('photometric_bench needs a CUDA device')
    b, h, w = a.batch, a.size, a.size
    cfg = configparser.ConfigParser()
    cfg.read_dict({'augmentation': AUG})
    comp = transform.get_transform(cfg, ['transform.image.' + n for n in CHAIN])
    groups = TI.split_chain(comp.transforms)
    assert len(groups) == 1
    random.seed(0)
    g = torch.Generator(device='cuda').manual_seed(0)
    inputs = [torch.randint(0, 256, (b, h, w, 3), dtype=torch.uint8, device='cuda', generator=g) for _ in range(4)]
    # one plan per input batch, built once: the timed loop is the launch alone
    plans = []
    for _ in inputs:
        launch = TI.Launch(b)
        draws = [[op.draw() for op in comp.transforms] for _ in range(b)]
        for j, op in enumerate(comp.transforms):
            for i in range(b):
                op.plan(launch, i, draws[i][j])
        plans.append(launch)

    def dev(x):
        return torch.from_numpy(np.ascontiguousarray(x)).cuda()
    args = [(dev(p._blur), dev(p._lut_hsv), dev(p._lut_out)) for p in plans]
    outs = [torch.empty_like(x) for x in inputs]

    def kernel(i):
        k = i % 4
        _ops.call('yb_photometric_u8', inputs[k], outs[k], b, h, w, args[k][0], 1, args[k][1], 1, args[k][2])
    for i in range(8):
        kernel(i)
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for i in range(a.iters):
        kernel(i)
    stop.record()
    torch.cuda.synchronize()
    us = start.elapsed_time(stop) * 1e3 / a.iters
    # the whole host-facing call as Collate makes it: draws, tables, upload, launch (host clock around a synchronised loop)
    n_e2e = max(a.iters // 10, 5)
    t = time.perf_counter()
    for i in range(n_e2e):
        comp(inputs[i % 4])
    torch.cuda.synchronize()
    us_e2e = (time.perf_counter() - t) * 1e6 / n_e2e
    nbytes = 2 * b * h * w * 3
    host_ms, how = host_ms_per_image(O.synth_frame(0, h, w))
    res = dict(card=card(), batch=b, height=h, width=w, iters=a.iters, us_per_batch=round(us, 2), us_per_image=round(us / b, 3),
               bytes_per_batch=nbytes, achieved_TBps=round(nbytes / us / 1e6, 3), fraction_of_7p7TBps=round(nbytes / (us * 1e-6) / PEAK_BPS, 3),
               us_per_batch_with_draws_and_upload=round(us_e2e, 1), host_ms_per_image=round(host_ms, 3), host=how, working_set_MB=round(4 * nbytes / 1e6, 1))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
