#!/usr/bin/env python
"""bench.py -- 416x416 images/sec of the YOLOv2 hot path on B200 (BASELINE.json metric).

Workload (BASELINE.json configs[1], "C2"): Darknet-19 416x416 batch-32 inference + anchor decode +
class softmax + threshold filter + NMS + per-class expansion, synthetic images, random-init
weights.  One "step" = one batch of 32 images through the whole chain.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # B200 arm (prints ONE JSON line)
    python bench.py --impl reference [--steps K] [--warmup W]      # the reference's CPU implementation of the same chain
    python bench.py --steps K --dump-outputs DIR                   # also writes what the last of the K timed steps returned

The inputs and weights are seeded, so two runs with the same arguments see the same data and their --dump-outputs files compare
output for output.  The bench writes nothing into the source tree; its scratch files go to the temporary directory.

N > 1: launched by torch.distributed.run, one rank per GPU; the inference path shards by image with no
data-path collective (replicas), so scaling is "weak" and `value` is the whole-job rate
(N * 32 * K images / max-over-ranks device time).  The training records below DO carry the path's one
exchange step (the NCCL gradient all-reduce).

Numbers in the JSON line:
  value      images/s, inputs resident in HBM (4 rotating input batches = 265 MB > 126 MB L2), CUDA-graph
             replay of the kernel chain, 2 batches in flight, CUDA events on the launching stream, max over ranks.
  one_lane   the same with ONE batch in flight (what a latency-bound caller sees); the per-kernel figures below are
             fractions of THIS step time.
  e2e        same metric through the serving API with HOST (pinned) fp32 batches: H2D copy of every
             batch and D2H of the detection arrays inside the timed region (double-buffered).
  strict     the same chain with precision='strict' (split fp16 operands; the mode whose head feature is inside the
             reference's 1e-3 contract) -- its cost next to the default 'fast' mode's measured error.
  roofline   tensor-core roofline of the dominant kernel family (the tcgen05 implicit-GEMM conv, 22 launches/step):
             algorithmic FLOPs of those launches / (their share of the step's kernel time x the one-lane step time), against
             MEASURED_PEAKS.json bf16_tflops (the BURST figure: the timed region is tens of milliseconds).
  train      BASELINE configs[2]: 416x416 batch-64 training step per GPU (train-mode fwd, region loss, bwd, Adam), with the
             gradient all-reduce when N > 1 (plus the same step with the exchange switched off = exposed communication).
  train_ddp  N > 1, BASELINE configs[3]: 16 images per GPU, sizes cycling {320, 416, 608}.
  mobilenet  BASELINE configs[4]: MobileNet backbone 416x416 batch-32 + decode + NMS.
  cpu_baseline  the reference's CPU path on all host cores on a bounded sample of the same workload; rank 0, N=1 only.
"""
import argparse
import configparser
import json
import os
import signal
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, 'yolo2-pytorch_b200')
for _p in (PKG, ROOT):
    if _p not in sys.path:
        sys.path.insert(0, _p)

GFLOP_PER_IMAGE_416 = 29.360334848          # SURVEY 8d: sum 2*Cin*Cout*k^2*H*W over the 23 convs
GFLOP_LAYER0_416 = 0.299040768              # layers1.0 (direct CUDA-core kernel, not tcgen05)
METRIC = '416x416 images/sec'


def make_config():
    config = configparser.ConfigParser()
    config.read_dict({'batch_norm': {'enable': '1'}, 'model': {'threshold': '0.6'},
                      'detect': {'threshold': '0.3', 'threshold_cls': '0.005', 'fix': '1', 'overlap': '0.45'}})
    return config


ANCHORS_HW = [[1.73145, 1.3221], [4.00944, 3.19275], [8.09892, 5.05587], [4.84053, 9.47112], [10.0071, 11.2364]]


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        # the timed regions here last tens of milliseconds at full clocks: the BURST figure is the honest denominator
        return dict(tflops=float(d.get('bf16_tflops', 1700.0)), tflops_sustained=float(d.get('bf16_tflops_sustained', 1460.0)),
                    hbm=float(d.get('hbm_gbs', 6650.0)), source='MEASURED_PEAKS.json (bf16_tflops, burst)')
    return dict(tflops=1700.0, tflops_sustained=1460.0, hbm=6650.0, source='fallback (B200_PROFILING.md)')


def committed_traffic():
    """DRAM bytes per launch of the conv family from the committed `ncu --set full` summary (profiles/traffic.json)."""
    path = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return d.get('conv_family_dram_bytes_per_launch'), d.get('source')
    return None, None


class ClockSampler(object):
    """SM clock / throttle reasons / power sampled through NVML every ~2 ms by a thread, so that even a 20 ms timed region
    holds several samples (nvidia-smi's 200 ms loop saw one).  Falls back to an nvidia-smi loop when pynvml is missing."""

    def __init__(self, index):
        self.rows = []          # (sm_mhz, max_mhz, power_w, reasons bitmask)
        self._stop = False
        self.smi = None
        try:
            import pynvml
            pynvml.nvmlInit()
            from b200 import hostbind
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(hostbind.physical_index(index))
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
        except Exception:
            self.nv = None
            self._start_smi(index)

    def _poll(self):
        nv = self.nv
        while not self._stop:
            try:
                self.rows.append((float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)), self.max_mhz,
                                  nv.nvmlDeviceGetPowerUsage(self.h) / 1e3, int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))))
            except Exception:
                pass
            time.sleep(0.002)

    def _start_smi(self, index):
        q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        try:
            self.smi = subprocess.Popen(['nvidia-smi', '-i', str(index), '--query-gpu=' + q, '--format=csv,noheader,nounits', '-lms', '100'],
                                        stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.smi_rows = []
            threading.Thread(target=lambda: [self.smi_rows.append(l.strip()) for l in self.smi.stdout], daemon=True).start()
        except Exception:
            self.smi = None

    def stop(self):
        if self.nv is not None:
            self._stop = True
            self.thread.join(timeout=1.0)
            nv = self.nv
            names = (('hw_slowdown', nv.nvmlClocksEventReasonHwSlowdown), ('hw_thermal_slowdown', nv.nvmlClocksEventReasonHwThermalSlowdown),
                     ('sw_thermal_slowdown', nv.nvmlClocksEventReasonSwThermalSlowdown), ('sw_power_cap', nv.nvmlClocksEventReasonSwPowerCap))
            sm = sorted(r[0] for r in self.rows)
            mask = 0
            for r in self.rows:
                mask |= r[3]
            return dict(sm_mhz=(sm[len(sm) // 2] if sm else None), sm_max_mhz=self.max_mhz, samples=len(sm),
                        power_w_max=(max(r[2] for r in self.rows) if self.rows else None), reasons=[n for n, bit in names if mask & bit], source='nvml')
        if self.smi is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        time.sleep(0.15)
        self.smi.terminate()
        sm, mx, reasons = [], [], set()
        names = ('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap')
        for r in self.smi_rows:
            parts = [x.strip() for x in r.split(',')]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        sm.sort()
        return dict(sm_mhz=(sm[len(sm) // 2] if sm else None), sm_max_mhz=(max(mx) if mx else None), samples=len(sm), reasons=sorted(reasons), source='nvidia-smi')


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port on the host cores
# ------------------------------------------------------------------------------------------------
def make_cpu_chain():
    """The CPU implementation of the C2 chain: the UNMODIFIED reference staged under baseline/_ref (kind 'reference') when present,
    else the oracle port (kind 'port').  Returns (chain(x) -> (feature, detections), kind, image generator)."""
    import torch
    from oracle import yolo2_oracle as O      # seeded input / weight generators (and the port when the reference is not staged)
    sd = O.make_state_dict(0)
    anchors = O.anchors_yolo_voc()
    try:
        from baseline import ref_runner
        if ref_runner.available():
            return ref_runner.build_chain(sd, anchors), 'reference', O.synth_images
    except Exception as ex:
        sys.stderr.write('bench.py: staged reference unusable (%s); timing the oracle port\n' % ex)

    def chain(x):
        with torch.no_grad():
            feature = O.darknet_forward(sd, x)
            pred = O.decode(feature, anchors)
            prob = O.class_prob(pred)
            out = []
            for bi in range(x.size(0)):
                out.append(O.postprocess(pred['iou'][bi].reshape(-1), pred['yx_min'][bi].reshape(-1, 2), pred['yx_max'][bi].reshape(-1, 2),
                                         prob[bi].reshape(-1, prob.size(-1)), True, 0.3, 0.005, 0.45))
        return feature, out
    return chain, 'port', O.synth_images


def cpu_measure(batch, steps, warmup, budget_s, keep_features=0):
    """The reference's CPU path timed on all host cores.  Returns (images/s, cores, sample description, ms/step, kind, features):
    `features` = (images, head features) of the first `keep_features` sample images for the precision record."""
    import torch
    chain, kind, synth_images = make_cpu_chain()
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    # calibrate on 4 images: give the CPU path its best thread count (all cores is torch's default,
    # but oversubscription can hurt), then size the per-step sample so the whole run fits the budget
    x2 = synth_images(4, 416, 416, seed=0)
    best = None
    for th in sorted({ncpu, min(ncpu, 64), min(ncpu, 32), min(ncpu, 16)}, reverse=True):
        torch.set_num_threads(th)
        chain(x2)
        t0 = time.perf_counter()
        chain(x2)
        dt = (time.perf_counter() - t0) / 4
        if best is None or dt < best[0]:
            best = (dt, th)
    per_img, cores = best
    torch.set_num_threads(cores)
    sample = int(max(1, min(batch, budget_s / max(1, steps + warmup) / per_img)))
    x = synth_images(sample, 416, 416, seed=0)
    for _ in range(warmup):
        chain(x)
    t0 = time.perf_counter()
    for _ in range(steps):
        feature, _ = chain(x)
    dt = time.perf_counter() - t0
    feats = None
    if keep_features:
        n = min(keep_features, sample)
        feats = (x[:n].clone(), feature[:n].clone())
    what = "the reference's own modules (baseline/_ref)" if kind == 'reference' else 'oracle port of the reference'
    return (sample * steps / dt, cores, '%d steps x %d images (of the %d-image batch), fp32, %s, torch %d threads' % (steps, sample, batch, what, cores),
            dt / steps * 1e3, kind, feats)


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    value, cores, sample, ms, kind, feats = cpu_measure(args.batch, args.steps, args.warmup, budget_s=args.cpu_budget, keep_features=args.keep_features)
    if args.features_out and feats is not None:
        import numpy as np
        np.savez(args.features_out, x=feats[0].numpy(), feature=feats[1].numpy())
    line = dict(impl='reference', metric=METRIC, value=value, unit='images/s', n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=ms, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f32', data='synthetic',
                config=dict(workload='Darknet-19 416x416 batch-%d inference + decode + softmax + filter + NMS (BASELINE configs[1])' % args.batch,
                            global_batch=args.batch,
                            note=('CPU: the unmodified reference (model.yolo2.Darknet + model.Inference + detect.postprocess from baseline/_ref), torch fp32'
                                  if kind == 'reference' else 'CPU: oracle port of the reference algorithm (torch fp32)') + ', bounded sample per step'),
                cpu_baseline=dict(value=value, unit='images/s', cores=cores, kind=kind, sample=sample),
                e2e=dict(value=value, unit='images/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line))


def cpu_leg_subprocess(batch, budget_s, keep_features):
    """cpu_baseline of the B200 arm: the CPU path in a child process (the reference's packages are called `model` / `utils` like
    this repository's own, so the two cannot share an interpreter).  Returns (cpu_baseline dict, (images, features) or None)."""
    import tempfile
    import numpy as np
    import torch
    feat_path = os.path.join(tempfile.gettempdir(), 'yb_cpu_leg_%d.npz' % os.getpid())
    cmd = [sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--steps', '3', '--warmup', '1', '--batch', str(batch),
           '--cpu-budget', str(budget_s), '--keep-features', str(keep_features), '--features-out', feat_path]
    env = {k: v for k, v in os.environ.items() if k not in ('RANK', 'LOCAL_RANK', 'WORLD_SIZE')}
    env['CUDA_VISIBLE_DEVICES'] = ''
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    line = None
    for l in r.stdout.splitlines():
        if l.startswith('{'):
            line = json.loads(l)
    if line is None:
        return dict(error='cpu leg failed: %s' % (r.stderr or '')[-300:]), None
    feats = None
    if os.path.exists(feat_path):
        d = np.load(feat_path)
        feats = (torch.from_numpy(d['x']), torch.from_numpy(d['feature']))
        os.remove(feat_path)
    return line['cpu_baseline'], feats


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def build_model(device):
    import torch
    import model
    import model.yolo2
    config = make_config()
    anchors = torch.tensor(ANCHORS_HW, dtype=torch.float32)
    torch.manual_seed(0)
    dnn = model.yolo2.Darknet(model.ConfigChannels(config), anchors, 20)
    g = torch.Generator().manual_seed(1)
    for m in dnn.modules():
        if isinstance(m, torch.nn.BatchNorm2d):      # non-trivial BN so the fused scale/shift is exercised
            m.weight.data = torch.rand(m.num_features, generator=g) + 0.5
            m.bias.data = torch.randn(m.num_features, generator=g) * 0.1
            m.running_mean = torch.randn(m.num_features, generator=g) * 0.1
            m.running_var = torch.rand(m.num_features, generator=g) + 0.5
    dnn = dnn.to(device).eval()
    inference = model.Inference(config, dnn, anchors).eval()
    return config, dnn, inference


def profile_layers(pipe, steps):
    """Instrumented eager pass: CUDA events around every tcgen05 conv launch (a long spin kernel in
    front of each step lets the host run ahead so the events bracket back-to-back kernels)."""
    import torch
    from b200 import ops
    records = []
    orig = ops.conv_bn_act

    def timed(x, w, *a, **kw):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        y = orig(x, w, *a, **kw)
        e.record()
        b, h, wd, _ = x.shape
        cout, k, _, cin = w.shape
        records.append((s, e, 2.0 * b * h * wd * cin * cout * k * k, (h, cin, cout, k)))
        return y

    ops.conv_bn_act = timed
    other_records = []
    originals = {}

    def wrap_other(name):
        fn = getattr(ops, name)
        originals[name] = fn

        def timed_other(*a, **kw):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            y = fn(*a, **kw)
            e.record()
            other_records.append((name, s, e))
            return y
        setattr(ops, name, timed_other)

    for name in ('conv0_bn_leaky_pool', 'conv0_u8_bn_leaky_pool', 'maxpool2x2', 'reorg_f16', 'decode', 'filter_nms'):
        wrap_other(name)
    step_events = []
    try:
        pipe._forward(pipe.x[0])          # un-timed: allocator and lazy-init effects stay out of the events
        torch.cuda.synchronize()
        del records[:], other_records[:]
        for _ in range(steps):
            torch.cuda._sleep(int(6e7))   # ~30 ms head start: the host enqueues the whole eager step while the GPU spins
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            pipe._forward(pipe.x[0])
            e.record()
            step_events.append((s, e))
        torch.cuda.synchronize()
    finally:
        ops.conv_bn_act = orig
        for name, fn in originals.items():
            setattr(ops, name, fn)
    others = {}
    for name, s, e in other_records:
        others.setdefault(name, []).append(s.elapsed_time(e) * 1e3)
    others = {k: dict(launches_per_step=len(v) // steps, us_per_step=sum(v) / steps) for k, v in others.items()}
    per_step = len(records) // steps
    layers = []
    for i in range(per_step):
        ms = sum(records[j * per_step + i][0].elapsed_time(records[j * per_step + i][1]) for j in range(steps)) / steps
        fl = records[i][2]
        layers.append(dict(shape='%dx%d cin%d cout%d k%d' % ((records[i][3][0],) * 2 + records[i][3][1:]), us=ms * 1e3, tflops=fl / ms / 1e9))
    conv_ms = sum(l['us'] for l in layers) / 1e3
    conv_flops = sum(records[i][2] for i in range(per_step))
    step_ms = sum(s.elapsed_time(e) for s, e in step_events) / steps
    kernels_ms = conv_ms + sum(v['us_per_step'] for v in others.values()) / 1e3
    return dict(layers=layers, others=others, conv_ms=conv_ms, conv_flops=conv_flops, eager_step_ms=step_ms, kernels_ms=kernels_ms, launches=per_step)


def timed_steps(pipe, steps, warmup, slots, cur, barrier, world, device):
    """W warm-up + K timed graph replays rotating over the resident input slots.  Returns ms for K steps (max over ranks)."""
    import torch
    import torch.distributed as dist
    for i in range(warmup):
        pipe.run(i % slots)
    barrier()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record(cur)
    pipe.start_after(start)
    for i in range(steps):
        pipe.run(i % slots)
    pipe.wait_all(cur)
    end.record(cur)
    torch.cuda.synchronize()
    ms = start.elapsed_time(end)
    barrier()
    if world > 1:
        t = torch.tensor([ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms


def dump_outputs(pipe, slot, out_dir, budget=64 << 20):
    """Writes what the caller of the timed path received from its last step (input slot `slot`) as out_dir/<name>.npy: the decoded
    head (feature, iou, yx_min, yx_max, prob) and every image's detections in the form detect.postprocess returns them (keep_iou,
    det_yx_min, det_yx_max, det_cls, det_score), concatenated over images; n_keep / n_det per image split them.  Float arrays are
    float32, counts and classes float64 (exact).  Images are taken in batch order while the files fit in `budget` bytes."""
    import numpy as np
    import torch
    host = pipe.fetch(slot)
    torch.cuda.synchronize()
    dense = {k: pipe.out[slot][k].float().cpu().numpy() for k in ('feature', 'iou', 'yx_min', 'yx_max', 'prob')}
    parts = {k: [] for k in ('n_keep', 'n_det', 'keep_iou', 'det_yx_min', 'det_yx_max', 'det_cls', 'det_score')}
    used = 128 * (len(dense) + len(parts))         # .npy headers
    for bi in range(pipe.batch):
        d = pipe.detections(host, bi)
        iou, yx_min, yx_max, cls, score = (torch.zeros(0), torch.zeros(0, 2), torch.zeros(0, 2), torch.zeros(0), torch.zeros(0)) if d is None else d
        size = sum(v[bi].nbytes for v in dense.values()) + 8 * (2 + iou.numel() + 6 * cls.numel())
        if used + size > budget:
            break
        used += size
        parts['n_keep'].append(np.array([iou.numel()], np.float64))
        parts['n_det'].append(np.array([cls.numel()], np.float64))
        parts['keep_iou'].append(iou.float().numpy())
        parts['det_yx_min'].append(yx_min.float().numpy())
        parts['det_yx_max'].append(yx_max.float().numpy())
        parts['det_cls'].append(cls.double().numpy())
        parts['det_score'].append(score.float().numpy())
    n = len(parts['n_keep'])
    os.makedirs(out_dir, exist_ok=True)
    for k, v in dense.items():
        np.save(os.path.join(out_dir, k + '.npy'), v[:n])
    for k, v in parts.items():
        np.save(os.path.join(out_dir, k + '.npy'), np.concatenate(v))


def mobilenet_record(args, device, peaks):
    """BASELINE configs[4]: MobileNet backbone 416x416 batch-32 + decode + filter + NMS through the plugin surface, one CUDA graph."""
    import torch
    import detect
    import model
    import model.mobilenet
    from b200 import ops
    config = make_config()
    anchors = torch.tensor(ANCHORS_HW, dtype=torch.float32)
    torch.manual_seed(0)
    dnn = model.mobilenet.MobileNet(model.ConfigChannels(config), anchors, 20)
    g = torch.Generator().manual_seed(1)
    for m in dnn.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.weight.data = torch.rand(m.num_features, generator=g) + 0.5
            m.bias.data = torch.randn(m.num_features, generator=g) * 0.1
            m.running_mean = torch.randn(m.num_features, generator=g) * 0.1
            m.running_var = torch.rand(m.num_features, generator=g) + 0.5
    dnn = dnn.to(device).eval()
    inference = model.Inference(config, dnn, anchors).eval()
    B, H, W = args.batch, args.size, args.size
    xs = [torch.rand(B, 3, H, W, generator=g).to(device) for _ in range(4)]      # 266 MB > L2

    def chain(x):
        pred = model._inference(inference, x)
        return detect._run(config, pred['iou'], pred['yx_min'], pred['yx_max'], detect.get_prob(pred), True, True)[1]

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            n0 = ops.launch_count
            chain(xs[0])
            launches = ops.launch_count - n0
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graphs = []
    for x in xs:
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            chain(x)
        graphs.append(gr)
    steps = max(10, args.steps)
    for i in range(max(3, args.warmup)):
        graphs[i % 4].replay()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for i in range(steps):
        graphs[i % 4].replay()
    e.record()
    torch.cuda.synchronize()
    ms = s.elapsed_time(e) / steps
    # instrumented eager pass: pointwise (tcgen05) vs depthwise / first conv (HBM-bound) kernel time
    recs = []
    orig_conv, orig_call = ops.conv_bn_act, ops.call

    def t_conv(x, w, *a, **kw):
        s1, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s1.record(); y = orig_conv(x, w, *a, **kw); e1.record()
        b, h, wd, _ = x.shape
        cout, k, _, cin = w.shape
        recs.append(('pw', s1, e1, 2.0 * b * h * wd * cin * cout * k * k, 2.0 * (b * h * wd * (cin + cout) + cin * cout)))
        return y

    def t_call(name, *a):
        s1, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s1.record(); orig_call(name, *a); e1.record()
        if name == 'yb_dwconv3x3_bn_relu_fwd':
            x, _, _, _, out = a[:5]
            recs.append(('dw', s1, e1, 2.0 * 9 * out.numel(), 2.0 * (x.numel() + out.numel())))
        elif name == 'yb_mb_conv0_bn_relu_fwd':
            x, out = a[0], a[4]
            recs.append(('conv0', s1, e1, 2.0 * 27 * out.numel(), 4.0 * x.numel() + 2.0 * out.numel()))

    ops.conv_bn_act, ops.call = t_conv, t_call
    try:
        reps = 3
        for _ in range(reps):
            torch.cuda._sleep(int(4e7))
            dnn(xs[0])
        torch.cuda.synchronize()
    finally:
        ops.conv_bn_act, ops.call = orig_conv, orig_call
    agg = {}
    for kind, s1, e1, fl, by in recs:
        d = agg.setdefault(kind, [0.0, 0.0, 0.0, 0])
        d[0] += s1.elapsed_time(e1) / reps; d[1] += fl / reps; d[2] += by / reps; d[3] += 1
    out = dict(metric=METRIC, value=B / (ms / 1e3), unit='images/s', ms_per_step=ms, batch=B, gpu_launches_per_step=launches,
               workload='MobileNet 416x416 batch-%d inference + decode + softmax + filter + NMS (BASELINE configs[4]), CUDA graph, 1 batch in flight' % B,
               gflop_per_image=3.959)
    if 'pw' in agg:
        t, fl, by, n = agg['pw']
        out['pointwise'] = dict(launches=n // reps, us=t * 1e3, tflops=fl / t / 1e9, frac_of_tensor_peak=fl / t / 1e9 / peaks['tflops'],
                                alg_gbs=by / t / 1e6, note='1x1 convs + head on the tcgen05 kernel; arithmetic intensity 30-250 FLOP/B: HBM/latency-bound at batch 32')
    for kind in ('dw', 'conv0'):
        if kind in agg:
            t, fl, by, n = agg[kind]
            out['depthwise' if kind == 'dw' else 'first_conv'] = dict(launches=n // reps, us=t * 1e3, alg_bytes=by, achieved_gbs=by / t / 1e6,
                                                                        frac_of_hbm_peak=by / t / 1e6 / peaks['hbm'])
    # strict precision ([hi | lo] activations, split-precision pointwise convs; 1e-3 contract, tests/test_gpu_parity.py): cost of the mode
    try:
        f_fast = dnn(xs[0]).clone()
        dnn.set_precision('strict')
        f_strict = dnn(xs[0]).clone()
        torch.cuda.synchronize()
        gs = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gs):
            chain(xs[1])
        for _ in range(3):
            gs.replay()
        s.record()
        for _ in range(steps):
            gs.replay()
        e.record()
        torch.cuda.synchronize()
        ms_s = s.elapsed_time(e) / steps
        out['strict'] = dict(value=B / (ms_s / 1e3), ms_per_step=ms_s, cost_vs_fast=ms_s / ms,
                             fast_vs_strict_feature_rel_err=float(((f_fast - f_strict).abs().max() / f_strict.abs().max()).item()))
    except Exception as ex:     # the headline record must not depend on the optional mode
        out['strict'] = dict(error='%s: %s' % (type(ex).__name__, ex))
    finally:
        dnn.set_precision('fast')
    return out


def train_records_subprocess(args, world, rank, local):
    """Training records (C3, and C4 when N > 1) measured by a child process per rank with its own rendezvous: a fault or a hang in
    the multi-GPU training path cannot take the headline line down with it.  Returns dict or {'error': ...} (rank 0), None elsewhere."""
    import tempfile
    out_path = os.path.join(tempfile.gettempdir(), 'yb_train_records_%d_%d.json' % (os.getpid(), rank))
    env = dict(os.environ)
    env['RANK'], env['LOCAL_RANK'], env['WORLD_SIZE'] = str(rank), str(local), str(world)
    env.setdefault('MASTER_ADDR', '127.0.0.1')
    env['MASTER_PORT'] = str(int(os.environ.get('MASTER_PORT', '29500')) + 1)
    env['TORCHELASTIC_USE_AGENT_STORE'] = 'False'          # the child group hosts its own store on MASTER_PORT + 1
    for k in ('TORCHELASTIC_RUN_ID', 'TORCHELASTIC_RESTART_COUNT', 'TORCHELASTIC_MAX_RESTARTS'):
        env.pop(k, None)
    cmd = [sys.executable, os.path.abspath(__file__), '--mode', 'train_records', '--gpus', str(world), '--steps', str(args.steps), '--warmup', str(args.warmup),
           '--json-out', out_path]
    err = None
    proc = subprocess.Popen(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, start_new_session=True)
    try:
        _, errtxt = proc.communicate(timeout=args.train_timeout)
        if proc.returncode != 0:
            err = 'child rc %d: %s' % (proc.returncode, (errtxt or '')[-600:])
    except subprocess.TimeoutExpired:
        err = 'child exceeded %d s' % args.train_timeout
        try:
            os.killpg(proc.pid, signal.SIGKILL)       # its own session: exactly the group we started
        except Exception:
            pass
        proc.communicate()
    if rank != 0:
        return None
    if err is None and os.path.exists(out_path):
        with open(out_path) as f:
            rec = json.load(f)
        os.remove(out_path)
        return rec
    return dict(error=err or 'no output')


def run_b200(args):
    import torch
    import torch.distributed as dist
    from b200 import hostbind, ops
    from b200.pipeline import DetectPipeline

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: the B200 arm needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm')
    # launching thread + the pinned staging buffers it allocates live on the GPU's own NUMA node (e2e is PCIe-bound)
    affinity_before, affinity_now = hostbind.bind_to_gpu(local)
    torch.cuda.set_device(local)
    device = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=device)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    config, dnn, inference = build_model(device)
    B, H, W = args.batch, args.size, args.size
    slots = 4
    pipe = DetectPipeline(inference, config, B, H, W, slots=slots, lanes=args.lanes, use_graph=not args.no_graph).prepare()
    cur = torch.cuda.current_stream()
    g = torch.Generator().manual_seed(100 + rank)
    host = [torch.rand(B, 3, H, W, generator=g).pin_memory() for _ in range(2)]
    resident = [torch.rand(B, 3, H, W, generator=g) for _ in range(slots)]
    for s in range(slots):
        pipe.x[s].copy_(resident[s])
    torch.cuda.synchronize()

    # ---- device-resident throughput (the headline `value`) ----
    # clocks / throttle reasons are sampled from here to the end of the last timed inference region (headline, one lane, e2e x2, strict:
    # ~0.2 s under load); an NVML query takes several ms, so the 20 ms headline region alone would hold one or two samples
    sampler = ClockSampler(local) if rank == 0 else None
    t_wall = time.perf_counter()
    ms = timed_steps(pipe, args.steps, args.warmup, slots, cur, barrier, world, device)
    wall_ms = (time.perf_counter() - t_wall) * 1e3
    if args.dump_outputs and rank == 0:
        # now: the pipelines timed next share the engine's per-lane activation plans, where the head feature lives
        dump_outputs(pipe, (args.steps - 1) % slots, args.dump_outputs)
    graph_launches = pipe.launches_per_run * args.steps
    value = world * B * args.steps / (ms / 1e3)

    # ---- the same with one batch in flight: the per-kernel figures below are fractions of THIS step ----
    pipe1 = DetectPipeline(inference, config, B, H, W, slots=slots, lanes=1, use_graph=not args.no_graph).prepare()
    for s in range(slots):
        pipe1.x[s].copy_(resident[s])
    ms1 = timed_steps(pipe1, args.steps, args.warmup, slots, cur, barrier, world, device)
    one_lane = dict(value=world * B * args.steps / (ms1 / 1e3), unit='images/s', ms_per_step=ms1 / args.steps, lanes=1)

    # ---- end to end through the serving API: pinned host batches in, detection arrays out ----
    def measure_e2e(pp, host_batches):
        for i in range(max(4, args.warmup)):
            pp.load(i % slots, host_batches[i % 2]); pp.run(i % slots, fetch=True)
        barrier()
        s2, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s2.record(cur)
        pp.start_after(s2)
        pp.load(0, host_batches[0])
        for i in range(args.steps):
            if i + 1 < args.steps:
                pp.load((i + 1) % slots, host_batches[(i + 1) % 2])
            pp.run(i % slots, fetch=True)
        pp.wait_all(cur)
        e2.record(cur)
        torch.cuda.synchronize()
        t_ms = s2.elapsed_time(e2)
        barrier()
        if world > 1:
            t = torch.tensor([t_ms], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            t_ms = float(t.item())
        return t_ms

    ms_e2e = measure_e2e(pipe, host)
    e2e_value = world * B * args.steps / (ms_e2e / 1e3)
    h2d = B * 3 * H * W * 4
    d2h = pipe.result_bytes()
    # same call with the frames as the reference's data loader holds them before ToTensor (uint8 HWC, detect.py:142-146):
    # the first conv kernel applies the 1/255 and the layout change, so the host->device copy is 4x smaller
    pipe_u8 = DetectPipeline(inference, config, B, H, W, slots=slots, lanes=args.lanes, use_graph=not args.no_graph, uint8_input=True).prepare()
    host_u8 = [torch.randint(0, 256, (B, H, W, 3), dtype=torch.uint8, generator=g).pin_memory() for _ in range(2)]
    ms_e2e_u8 = measure_e2e(pipe_u8, host_u8)
    e2e_u8 = dict(value=world * B * args.steps / (ms_e2e_u8 / 1e3), unit='images/s', h2d_bytes_per_step=B * 3 * H * W, d2h_bytes_per_step=d2h,
                  ms_per_step=ms_e2e_u8 / args.steps, input='uint8 NHWC frames (ToTensor fused into the first conv kernel)')
    del pipe_u8

    # ---- strict precision: the mode the reference's 1e-3 contract is asserted in (tests), and what it costs ----
    _, dnn_s, inference_s = build_model(device)
    dnn_s.engine.set_precision('strict')
    pipe_s = DetectPipeline(inference_s, config, B, H, W, slots=slots, lanes=args.lanes, use_graph=not args.no_graph).prepare()
    for s in range(slots):
        pipe_s.x[s].copy_(resident[s])
    ms_s = timed_steps(pipe_s, args.steps, args.warmup, slots, cur, barrier, world, device)
    clocks = sampler.stop() if sampler else None
    if clocks is not None:
        clocks['window'] = 'all timed inference regions of this run (headline, one lane, e2e, e2e_u8, strict)'
    strict = dict(value=world * B * args.steps / (ms_s / 1e3), unit='images/s', ms_per_step=ms_s / args.steps, gpu_launches_per_step=pipe_s.launches_per_run,
                  note="precision='strict': split fp16 hi+lo operands on all units but layers1.0/1.2, passthrough, layers3.0 (b200.engine.STRICT_KEEP)")

    # ---- training records (C3; C4 under N > 1) in a child process per rank ----
    train_rec = None
    if not args.no_train:
        barrier()
        train_rec = train_records_subprocess(args, world, rank, local)
        barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel family (tcgen05 convs): share of the step from an instrumented pass x the one-lane step ----
    peaks = measured_peaks()
    prof = profile_layers(pipe1, max(3, min(args.steps, 10)))
    step1_ms = ms1 / args.steps
    share = prof['conv_ms'] / prof['kernels_ms']
    conv_ms = share * step1_ms                        # conv-family time inside the timed one-lane step (sum of kernel times == step time)
    achieved = prof['conv_flops'] / (conv_ms / 1e3) / 1e12
    graph_step_ms = ms / args.steps
    traffic, traffic_source = committed_traffic()
    roofline = dict(bound='tensor', achieved=achieved, peak=peaks['tflops'], unit='TFLOP/s', frac=achieved / peaks['tflops'],
                    frac_of_sustained_peak=achieved / peaks['tflops_sustained'],
                    traffic=traffic, traffic_source=traffic_source,
                    kernel='conv_igemm_kernel x21 + conv_c32_kernel x1 (the tcgen05 implicit-GEMM conv family, 22 launches/step)', peak_source=peaks['source'],
                    flops_per_launch=prof['conv_flops'] / prof['launches'], us_per_launch=conv_ms * 1e3 / prof['launches'],
                    share_of_step=share, step_ms=step1_ms,
                    how='share = conv CUDA-event time / all kernels\' CUDA-event time in an instrumented eager pass of this run; us_per_launch = share x one_lane.ms_per_step / 22',
                    eager_event_sum=dict(conv_ms=prof['conv_ms'], all_kernels_ms=prof['kernels_ms'], note='isolated CUDA events add ~2-4 us per kernel: only the ratio is used'),
                    layers=prof['layers'],
                    whole_step_two_lanes=dict(tflops=(B * GFLOP_PER_IMAGE_416 / 1e3) / (graph_step_ms / 1e3),
                                              frac=(B * GFLOP_PER_IMAGE_416 / 1e3) / (graph_step_ms / 1e3) / peaks['tflops']))
    # HBM-bound kernels of the step: algorithmic bytes (SURVEY 8d, fp16 activations inside the backbone) / their slice of the one-lane step
    S = H // 32
    boxes = B * S * S * len(ANCHORS_HW)
    alg_bytes = {
        'conv0_bn_leaky_pool': B * 3 * H * W * 4 + B * (H // 2) * (W // 2) * 32 * 2,
        'maxpool2x2': int(1.25 * 2 * B * ((H // 4) ** 2 * 128 + (H // 8) ** 2 * 256 + (H // 16) ** 2 * 512)),
        'reorg_f16': 2 * B * (H // 16) ** 2 * 64 * 2,
        'decode': B * 125 * S * S * 4 + boxes * (1 + 8 + 20 + 20) * 4,
        'filter_nms': boxes * (1 + 4 + 20) * 4,
    }
    hbm_kernels = {}
    for name, nbytes in alg_bytes.items():
        rec = prof['others'].get(name)
        if rec and rec['us_per_step'] > 0:
            us = rec['us_per_step'] / (prof['kernels_ms'] * 1e3) * step1_ms * 1e3
            gbs = nbytes / (us * 1e-6) / 1e9
            hbm_kernels[name] = dict(us=us, alg_bytes=nbytes, achieved_gbs=gbs, frac_of_hbm_peak=gbs / peaks['hbm'])

    mobilenet = None
    if not args.no_mobilenet:
        try:
            mobilenet = mobilenet_record(args, device, peaks)
        except Exception as ex:      # a secondary record must not cost the headline
            mobilenet = dict(error='%s: %s' % (type(ex).__name__, ex))

    cpu = None
    precision = None
    if world == 1 and not args.no_cpu:
        hostbind.restore(affinity_before)             # the CPU arm gets every host core back
        cpu, feats = cpu_leg_subprocess(B, 20.0, 2)
        if feats is not None:
            # the checker's fp32 features of the first two sample images vs both GPU precisions: same seeded images, and the CPU arm's
            # weights (the seeded generator it used) loaded into the GPU models for this comparison
            from oracle import yolo2_oracle as O
            xs, ref = feats
            precision = {}
            sd = O.make_state_dict(0)
            for name, d in (('fast', dnn), ('strict', dnn_s)):
                d.load_state_dict(sd, strict=False)
                f = d(xs.to(device)).float().cpu()
                precision[name] = dict(feature_max_rel_err=float(((f - ref).abs().max() / ref.abs().max()).item()))
            precision['contract'] = 1e-3
            precision['note'] = "max|d|/max|ref| of the head feature vs the CPU reference on 2 images; tests assert strict <= 1e-3 on BASELINE's configs"

    line = dict(metric=METRIC, value=value, unit='images/s', n_gpus=world, steps=args.steps, warmup=args.warmup, ms_per_step=ms / args.steps,
                higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f16', data='synthetic',
                config=dict(workload='Darknet-19 416x416 batch-%d inference + decode + softmax + filter + NMS (BASELINE configs[1])' % B,
                            global_batch=B * world, per_gpu_batch=B, parallelism='replicas x%d (images shard, no collective)' % world,
                            l2='inputs rotate over %d resident batches (%.0f MB > 126 MB L2); ~0.6 GB of activations streamed per step' % (slots, slots * h2d / 1e6),
                            cuda_graph=not args.no_graph, lanes=pipe.lanes, precision='fast', weights='random-init (kaiming) + random BN statistics',
                            host_affinity=(sorted(affinity_now)[:1] + sorted(affinity_now)[-1:] + [len(affinity_now)]) if affinity_now else None),
                clocks=clocks, e2e=dict(value=e2e_value, unit='images/s', h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h, ms_per_step=ms_e2e / args.steps,
                         input='fp32 NCHW tensors (the reference forward() signature)'),
                e2e_u8=e2e_u8, one_lane=one_lane, strict=strict, precision=precision,
                gpu_launches=graph_launches, roofline=roofline, hbm_kernels=hbm_kernels, cpu_baseline=cpu, wall_ms=wall_ms)
    if train_rec is not None:
        for k in ('train', 'train_ddp', 'error'):
            if k in train_rec:
                line['train_error' if k == 'error' else k] = train_rec[k]
    if mobilenet is not None:
        line['mobilenet'] = mobilenet
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def synth_targets(batch, height, width, slots, generator):
    import torch
    yx_min = torch.zeros(batch, slots, 2)
    yx_max = torch.zeros(batch, slots, 2)
    cls = torch.zeros(batch, slots, dtype=torch.long)
    for b in range(batch):
        n = int(torch.randint(1, slots + 1, (1,), generator=generator))
        hw = torch.rand(n, 2, generator=generator) * torch.tensor([height / 2 - 16.0, width / 2 - 16.0]) + 16.0
        lo, hi = hw / 2, torch.tensor([float(height), float(width)]) - hw / 2
        c = lo + torch.rand(n, 2, generator=generator) * (hi - lo)
        yx_min[b, :n], yx_max[b, :n] = c - hw / 2, c + hw / 2
        cls[b, :n] = torch.randint(0, 20, (n,), generator=generator)
    return yx_min, yx_max, cls


def _train_setup(device, capturable):
    import torch
    config, dnn, inference = build_model(device)
    config.read_dict({'hparam': {'foreground': '5', 'background': '1', 'center': '1', 'size': '1', 'cls': '1'},
                      'train': {'cross_entropy': '1'}})
    dnn.train(); inference.train()
    anchors = torch.tensor(ANCHORS_HW, dtype=torch.float32)
    optimizer = torch.optim.Adam(dnn.parameters(), 1e-5, betas=(0.9, 0.999), eps=1e-8, capturable=capturable, fused=os.environ.get('YB_ADAM_FUSED', '1') != '0')
    return config, dnn, inference, anchors, optimizer


def _train_batches(B, H, W, device, generator, count=2):
    import torch
    batches = []
    for _ in range(count):
        yx_min, yx_max, cls = synth_targets(B, H, W, 16, generator)
        batches.append(dict(tensor=torch.rand(B, 3, H, W, generator=generator).to(device), yx_min=yx_min.to(device), yx_max=yx_max.to(device),
                            cls=cls.to(device)))
    return batches


def _gflop_train(H, W):
    return (3 * GFLOP_PER_IMAGE_416 - GFLOP_LAYER0_416) * (H * W) / (416.0 * 416.0)   # SURVEY 8d: 87.78 GFLOP / image at 416x416


def run_train_records(args):
    """Child of the default bench run (also callable directly): BASELINE configs[2] and, under N > 1, configs[3].

    train      416x416, 64 images per GPU: train-mode forward (batch-statistics BN), region loss, full backward, gradient
               all-reduce over the library's NCCL communicator when N > 1, Adam -- one CUDA graph per step.
    train_ddp  N > 1: 16 images per GPU (global batch 16 N; 128 on 8 GPUs), input size cycling {320, 416, 608} on every rank together
               (utils.data.SizeSchedule semantics), one CUDA graph per size.
    For N > 1 every configuration is also timed with the exchange switched off (same kernels, no collective):
    exposed communication = step - compute-only step."""
    import gc
    import torch
    import torch.distributed as dist
    import train as yb_train
    from b200 import ddp
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    device = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=device)
    peaks = measured_peaks()
    steps = max(5, min(args.steps, 20))
    warmup = max(3, args.warmup)
    g = torch.Generator().manual_seed(200 + rank)
    config, dnn, inference, anchors, optimizer = _train_setup(device, capturable=True)
    reducer = ddp.default_reducer() if world > 1 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def time_steps(step_fn, batches, n):
        for i in range(warmup):
            step_fn(batches[i % len(batches)])
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(n):
            out = step_fn(batches[i % len(batches)])
        e.record()
        torch.cuda.synchronize()
        ms = s.elapsed_time(e)
        barrier()
        if world > 1:
            t = torch.tensor([ms], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / n, out

    graphed = yb_train.GraphedStep(inference, optimizer, anchors, config, reducer)                # data parallel (or single GPU)
    graphed_local = yb_train.GraphedStep(inference, optimizer, anchors, config, False) if world > 1 else None
    records = {}
    # ---- configs[2]: 64 images per GPU at 416 ----
    B, H = 64, 416
    batches = _train_batches(B, H, H, device, g)
    bytes0 = reducer.bytes_reduced if reducer else 0
    sampler = ClockSampler(local) if rank == 0 else None
    ms, out = time_steps(graphed, batches, steps)
    clocks = sampler.stop() if sampler else None
    value = world * B / (ms / 1e3)
    tfl = value * _gflop_train(H, H) / 1e3
    rec = dict(metric='416x416 training images/sec', value=value, unit='images/s', n_gpus=world, ms_per_step=ms, steps=steps, warmup=warmup,
               per_gpu_batch=B, global_batch=B * world, tflops=tfl, frac_of_tensor_peak=tfl / world / peaks['tflops'],
               frac_of_sustained_peak=tfl / world / peaks['tflops_sustained'], gflop_per_image=_gflop_train(H, H),
               loss_total=float(out['loss_total'].item()), cuda_graph=True, clocks=clocks,
               workload='Darknet-19 416x416 batch-64/GPU training step: train-mode fwd + region loss + bwd%s + Adam (BASELINE configs[2])'
                        % (' + NCCL gradient all-reduce' if world > 1 else ''))
    if world > 1:
        arena = dnn.trainer.arena
        ms_local, _ = time_steps(graphed_local, batches, steps)
        rec.update(allreduce_bytes_per_step=int(arena.flat.numel() * 4), allreduce_buckets=len(arena.buckets), allreduce_dtype='f32',
                   collective='ncclAllReduce(sum) per bucket on a communication stream, captured in the step graph (yb_allreduce_bucket)',
                   compute_only_ms=ms_local, exposed_comm_ms=ms - ms_local, efficiency_vs_compute_only=ms_local / ms)
    records['train'] = rec
    # ---- configs[3]: 16 images per GPU, sizes cycling {320, 416, 608} ----
    if world > 1:
        Bs, sizes, maintain = 16, (320, 416, 608), max(4, steps // 2)
        per_size = {}
        tot_ms = tot_local = 0.0
        for size in sizes:
            bt = _train_batches(Bs, size, size, device, g)
            ms_s, _ = time_steps(graphed, bt, maintain)
            ms_l, _ = time_steps(graphed_local, bt, maintain)
            per_size[str(size)] = dict(ms_per_step=ms_s, compute_only_ms=ms_l, exposed_comm_ms=ms_s - ms_l, images_per_s=world * Bs / (ms_s / 1e3),
                                       tflops_per_gpu=Bs / (ms_s / 1e3) * _gflop_train(size, size) / 1e3)
            tot_ms += ms_s * maintain
            tot_local += ms_l * maintain
        nsteps = maintain * len(sizes)
        arena = dnn.trainer.arena
        records['train_ddp'] = dict(metric='multi-scale training images/sec', value=world * Bs * nsteps / (tot_ms / 1e3), unit='images/s', n_gpus=world,
                                    per_gpu_batch=Bs, global_batch=Bs * world, sizes=list(sizes), steps_per_size=maintain, per_size=per_size,
                                    allreduce_bytes_per_step=int(arena.flat.numel() * 4), allreduce_buckets=len(arena.buckets),
                                    exposed_comm_ms=(tot_ms - tot_local) / nsteps, efficiency_vs_compute_only=tot_local / tot_ms,
                                    workload='Darknet-19 multi-scale {320,416,608} training, %d images per GPU (global batch %d), NCCL data parallel '
                                             '(BASELINE configs[3])' % (Bs, Bs * world))
    if rank == 0 and args.json_out:
        with open(args.json_out, 'w') as f:
            json.dump(records, f)
    if rank == 0 and not args.json_out:
        print(json.dumps(records))
    # teardown in dependency order: graphs that captured collectives -> the library communicator -> torch.distributed
    graphed.close()
    if graphed_local is not None:
        graphed_local.close()
    del graphed, graphed_local
    gc.collect()
    torch.cuda.synchronize()
    ddp.shutdown()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=300)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--batch', type=int, default=32)
    ap.add_argument('--size', type=int, default=416)
    ap.add_argument('--no-graph', action='store_true')
    ap.add_argument('--mode', default='infer', choices=['infer', 'train_records'],
                    help='train_records: only the training records (what the default run measures in a child process)')
    ap.add_argument('--lanes', type=int, default=2, help='batches in flight per GPU (one CUDA stream + activation plan each)')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-train', action='store_true', help='skip the training records (configs[2]/[3])')
    ap.add_argument('--no-mobilenet', action='store_true', help='skip the MobileNet record (configs[4])')
    ap.add_argument('--train-timeout', type=int, default=420, help='seconds the training-record child may take before it is killed')
    ap.add_argument('--json-out', default=None, help='train_records mode: write the records here instead of stdout')
    ap.add_argument('--cpu-budget', type=float, default=150.0, help='reference arm: seconds of CPU work for the whole run')
    ap.add_argument('--keep-features', type=int, default=0, help=argparse.SUPPRESS)
    ap.add_argument('--features-out', default=None, help=argparse.SUPPRESS)
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the arrays the last timed step returned (detections, decoded head) as DIR/<name>.npy')
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != 'b200' or args.mode != 'infer'):
        ap.error('--dump-outputs applies to the B200 inference arm')
    if args.impl == 'reference':
        # the reference moves tensors to a GPU whenever it sees one (utils/__init__.py:104-111); this arm is its CPU path
        os.environ['CUDA_VISIBLE_DEVICES'] = ''
        args.warmup = max(args.warmup, 1)
        run_reference(args)
    elif args.mode == 'train_records':
        run_train_records(args)
    else:
        args.warmup = max(args.warmup, 3)
        run_b200(args)


if __name__ == '__main__':
    main()
