#!/usr/bin/env python
"""Time the DenseNet backbones (model/densenet.py) on the B200 kernels, eager and CUDA-graph replayed.

    python tools/densenet_bench.py [--batch 32] [--size 416] [--names densenet121,...] [--out profiles/r04_densenet_bench.json]

Per variant: the oracle's seeded synthetic weights, seeded inputs, every shape warmed up; then the forward timed with CUDA events over a
window of at least --seconds, eagerly and as a replayed CUDA graph.  Also reported, per forward and from shapes: the launches, the conv
FLOPs (at the padded Cin the kernels execute), and the norm+relu passes (yb_bn_relu_f16 / yb_bn_relu_avgpool2x2_f16) replayed alone on the
same shapes with their bytes moved; a pass whose source block buffer and destination fit the 126 MB L2 together is marked l2_resident (by
size, which is when its reads can be served from L2 -- not a measurement).  The card name and power limit are read in the same run."""
import argparse
import json
import math
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'yolo2-pytorch_b200'))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
import model  # noqa: E402
import model.densenet as D  # noqa: E402
from b200 import ops as _ops  # noqa: E402
import densenet_oracle as DO  # noqa: E402
from oracle import yolo2_oracle as O  # noqa: E402

L2_BYTES = 126e6


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', str(torch.cuda.current_device())],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ''
    return q or torch.cuda.get_device_name()


def timed(fn, seconds):
    """ms per call of fn, from device events around one window of at least `seconds` (grown until it is that long)."""
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 3
    while True:
        start.record()
        for _ in range(n):
            fn()
        stop.record()
        torch.cuda.synchronize()
        ms = start.elapsed_time(stop)
        if ms >= seconds * 1e3:
            return ms / n, n
        n = math.ceil(n * 1.2 * seconds * 1e3 / max(ms, 1e-3))


def shape_counts(pl, batch):
    flops = 0
    norm_passes = []
    for op in pl['launches']:
        if op['op'] in ('conv', 'head'):
            flops += 2 * batch * op['height'] * op['width'] * op['cin'] * op['cout'] * op['ksize'] ** 2
        elif op['op'] in ('bn_relu', 'bn_relu_avgpool'):
            pix = batch * op['height'] * op['width']
            src = batch * op['height'] * op['width'] * op['x_ld'] * 2
            if op['op'] == 'bn_relu':
                moved = pix * (op['channels'] + op['channels_padded']) * 2
                dst = pix * op['channels_padded'] * 2
            else:
                moved = pix * op['channels'] * 2 + (pix // 4) * op['channels'] * 2
                dst = (pix // 4) * op['channels'] * 2
            norm_passes.append(dict(op=op, bytes=moved, l2_resident=src + dst <= L2_BYTES))
    return flops, norm_passes


def norm_passes_alone(net, pl, passes, batch, seconds):
    """The plan's norm+relu launches on buffers of the forward's shapes (random block contents), in plan order, timed alone."""
    dev = torch.device('cuda')
    g = torch.Generator(device='cuda').manual_seed(1)
    bufs = {k: torch.randn((batch,) + v, generator=g, device=dev).half() for k, v in pl['buffers'].items() if isinstance(v, tuple)}
    scratch = torch.empty(batch * pl['buffers']['scratch'], dtype=torch.float16, device=dev)
    calls = []
    for p in passes:
        op = p['op']
        scale, shift = net._fold(op['bn'])
        h, w = op['height'], op['width']
        if op['op'] == 'bn_relu':
            calls.append(('yb_bn_relu_f16', bufs[op['src']], op['x_ld'], scale, shift, scratch, op['channels_padded'], batch * h * w,
                          op['channels'], op['channels_padded']))
        else:
            calls.append(('yb_bn_relu_avgpool2x2_f16', bufs[op['src']], op['x_ld'], scale, shift, scratch, batch, h, w, op['channels']))

    def run():
        for c in calls:
            _ops.call(*c)
    run()
    torch.cuda.synchronize()
    return timed(run, seconds)[0]


def bench(name, batch, size, seconds):
    net = getattr(D, name)(model.ConfigChannels(None), O.anchors_yolo_voc(), 20)
    net.load_state_dict(DO.make_densenet_state_dict(name, 0), strict=False)
    net = net.cuda().eval()
    x = O.synth_images(batch, size, size, seed=3).cuda()
    pl = net.plan(size, size)
    with torch.no_grad():
        net(x)
        net(x)
        torch.cuda.synchronize()
        before = _ops.launch_count
        net(x)
        launches = _ops.launch_count - before
        eager_ms, eager_n = timed(lambda: net(x), seconds)
        stream = torch.cuda.Stream()
        stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(stream):
            net(x)
        torch.cuda.current_stream().wait_stream(stream)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            net(x)
        graph.replay()
        torch.cuda.synchronize()
        graph_ms, graph_n = timed(graph.replay, seconds)
        flops, passes = shape_counts(pl, batch)
        norm_ms = norm_passes_alone(net, pl, passes, batch, seconds)
    del graph
    norm_bytes = sum(p['bytes'] for p in passes)
    resident = [p for p in passes if p['l2_resident']]
    return dict(
        batch=batch, size=size, launches_per_forward=launches, planned_launches=len(pl['launches']),
        eager=dict(ms=eager_ms, img_per_s=batch * 1e3 / eager_ms, iters=eager_n),
        graph=dict(ms=graph_ms, img_per_s=batch * 1e3 / graph_ms, iters=graph_n),
        conv_gflop=flops / 1e9, conv_tflop_per_s_over_whole_graph_forward=flops / graph_ms / 1e9,
        norm_relu=dict(passes=len(passes), ms_alone=norm_ms, share_of_graph_forward=norm_ms / graph_ms, gbytes=norm_bytes / 1e9,
                       tb_per_s=norm_bytes / norm_ms / 1e9, l2_resident_passes=len(resident),
                       l2_resident_gbytes=sum(p['bytes'] for p in resident) / 1e9,
                       l2_resident_blocks=sorted({p['op']['src'] for p in resident}),
                       dram_blocks=sorted({p['op']['src'] for p in passes if not p['l2_resident']})))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batch', type=int, default=32)
    ap.add_argument('--size', type=int, default=416)
    ap.add_argument('--names', default=','.join(D.CONFIGS))
    ap.add_argument('--seconds', type=float, default=1.0)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('densenet_bench needs a CUDA device')
    res = dict(gpu=card(), note='CUDA events over >= %.1f s windows; norm_relu passes timed alone on the forward shapes' % a.seconds, variants={})
    for name in a.names.split(','):
        res['variants'][name] = bench(name, a.batch, a.size, a.seconds)
        print(name, json.dumps(res['variants'][name]), flush=True)
    res['gpu_after'] = card()
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
