"""Error budget of the EVAL-mode backbone under fp16 operands, in pure CPU fp32 arithmetic with one rounding switched on at a time:
for every unit, round only its weights (w) or only its input activation (a) to fp16 and measure the head feature against the fp32
forward.  Result (profiles/r02_error_budget.txt): all 46 roundings contribute alike (~2e-4 relative rms each; the first two layers and
the passthrough half of that), they add in quadrature to 1.3e-3 rms = 1.7e-3 max-norm -- there is no offending layer, so reaching the
reference's 1e-3 contract needs ~3/4 of the roundings removed: b200.engine.STRICT_KEEP.

    python tools/error_budget.py
"""
import os, sys, time, torch, torch.nn.functional as F
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import yolo2_oracle as O
torch.set_num_threads(8)
sd = O.make_state_dict(0)
x = O.synth_images(2, 416, 416, seed=0)
layers = O.darknet19_layers()
def r16(t): return t.half().float()
def fwd(rw, ra):
    """rw, ra: sets of layer keys whose weights / input activations are fp16-rounded"""
    by = {}
    for l in layers: by.setdefault(l['group'], []).append(l)
    def unit(x, l):
        k = l['key']
        w = sd[k + '.conv.weight']
        if k in rw: w = r16(w)
        if k in ra: x = r16(x)
        bias = None if l['bn'] else sd.get(k + '.conv.bias')
        y = F.conv2d(x, w, bias, padding=(l['k'] - 1) // 2)
        if l['bn']:
            y = F.batch_norm(y, sd[k + '.bn.running_mean'], sd[k + '.bn.running_var'], sd[k + '.bn.weight'], sd[k + '.bn.bias'], False, 0.0, 1e-5)
        if l['act']: y = F.leaky_relu(y, 0.1)
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
    ref = fwd(set(), set())
    keys = [l['key'] for l in layers]
    def err(y): return ((y - ref).abs().max() / ref.abs().max()).item()
    t = time.time(); full = fwd(set(keys), set(keys)); print('full fp16', err(full), time.time() - t)
    print('weights only', err(fwd(set(keys), set())))
    print('acts only', err(fwd(set(), set(keys))))
    tot = 0
    for k in keys:
        ew = err(fwd({k}, set())); ea = err(fwd(set(), {k}))
        rms_w = ((fwd({k}, set()) - ref).pow(2).mean().sqrt() / ref.pow(2).mean().sqrt()).item()
        rms_a = ((fwd(set(), {k}) - ref).pow(2).mean().sqrt() / ref.pow(2).mean().sqrt()).item()
        tot += rms_w ** 2 + rms_a ** 2
        print('%-12s w %.2e (rms %.2e)  a %.2e (rms %.2e)' % (k, ew, rms_w, ea, rms_a))
    print('rss rms', tot ** 0.5, 'full rms', ((full - ref).pow(2).mean().sqrt() / ref.pow(2).mean().sqrt()).item())
