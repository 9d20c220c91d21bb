"""Error budget of the TRAIN-mode forward under fp16 storage, in pure CPU fp32 arithmetic (the oracle's ops) with only the roundings
of the GPU path added: weights -> fp16, raw conv output z -> fp16, activation -> fp16.  Shows that batch-statistics BatchNorm amplifies
a relative perturbation by ~sqrt(1 + mu^2/sigma^2) per layer (the batch mean it removes carried part of the signal, the error stays), so
the head feature of this untrained network moves by 3.7e-2 although every layer adds only ~1e-3 -- the reason the end-to-end training
test (tests/test_gpu_parity.py: C3) asserts losses / statistics and the per-layer test asserts activations.

    python tools/train_error_budget.py 8 416     # batch, size  ->  profiles/r02_train_error_budget.txt
"""
import os, sys, time, torch, torch.nn.functional as F
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import yolo2_oracle as O
torch.set_num_threads(8)
sd = O.make_state_dict(0)
layers = O.darknet19_layers()
B = int(sys.argv[1]); S = int(sys.argv[2])
x = O.synth_images(B, S, S, seed=64)
def r16(t): return t.half().float()
def fwd(round_w, round_z, round_a, stats=None, collect=None):
    by = {}
    for l in layers: by.setdefault(l['group'], []).append(l)
    def unit(x, l):
        k = l['key']
        w = sd[k + '.conv.weight']
        if round_w and k != 'layers1.0': w = r16(w)
        if k == 'layers1.0' and round_w: w = r16(w); x = r16(x)
        bias = None if l['bn'] else sd.get(k + '.conv.bias')
        y = F.conv2d(x, w, bias, padding=(l['k'] - 1) // 2)
        if l['bn']:
            if round_z: y = r16(y)
            m = y.mean(dim=(0, 2, 3)); v = y.var(dim=(0, 2, 3), unbiased=False)
            if stats is not None: stats[k] = (m, v)
            y = F.batch_norm(y, None, None, sd[k + '.bn.weight'], sd[k + '.bn.bias'], True, 0.0, 1e-5)
        if l['act']: y = F.leaky_relu(y, 0.1)
        if round_a and l['bn']: y = r16(y)
        if collect is not None: collect[k] = y
        return y
    def run(g, x, pre=False):
        if pre: x = F.max_pool2d(x, 2)
        for l in by[g]:
            x = unit(x, l)
            if l['pool_after']: x = F.max_pool2d(x, 2)
        return x
    x1 = run('layers1', x)
    _x = O.reorg(run('passthrough', x1))
    x2 = run('layers2', x1, True)
    return run('layers3', torch.cat([_x, x2], 1))
with torch.no_grad():
    c0, c1 = {}, {}
    s0 = {}
    t = time.time(); ref = fwd(False, False, False, s0, c0); print('ref', time.time() - t, flush=True)
    for name, cfg in (('w only', (True, False, False)), ('z only', (False, True, False)), ('a only', (False, False, True)), ('all', (True, True, True))):
        c1 = {}
        y = fwd(*cfg, collect=c1)
        print(name, 'feature rel %.3e' % ((y - ref).abs().max() / ref.abs().max()).item(), flush=True)
        if name == 'all':
            for k in c0:
                print('  %-12s rel %.2e   mean/std of z-stats: |mu|/sigma max %.1f' % (k, ((c1[k] - c0[k]).abs().max() / c0[k].abs().max()).item(),
                      (s0[k][0].abs() / s0[k][1].sqrt()).max().item() if k in s0 else 0))
