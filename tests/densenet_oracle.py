"""CPU oracle of the DenseNet plugin -- TEST INFRASTRUCTURE ONLY (the product never imports it).

A restatement of the reference's eval-mode `model/densenet.py:29-117` (torchvision's _DenseLayer / _Transition) with torch ops on CPU, pinned
to the executed reference by tests/golden/make_golden_densenet.py (1e-5), plus the fp16 error model of the B200 path that the GPU tolerances
of tests/test_densenet.py come from.  Inputs come from oracle/yolo2_oracle.py's generators.
"""
import math

import torch
import torch.nn.functional as F

from oracle.yolo2_oracle import synth_images

DENSENET_CONFIGS = {'densenet121': (64, 32, (6, 12, 24, 16)), 'densenet169': (64, 32, (6, 12, 32, 32)),
                    'densenet201': (64, 32, (6, 12, 48, 32)), 'densenet161': (96, 48, (6, 12, 36, 24))}   # (init, growth, blocks), :68-117
DENSENET_BN_SIZE = 4


def densenet_blocks(name='densenet121'):
    """Per dense block, in forward order (model/densenet.py:42-50): prefix, input channels, growth, the layers as (prefix, C_l) where C_l
    is the layer's input width, output channels, and the transition that follows it (None after the last block)."""
    init, growth, counts = DENSENET_CONFIGS[name]
    out, c = [], init
    for i, n in enumerate(counts, 1):
        layers = [('features.denseblock%d.denselayer%d' % (i, l + 1), c + l * growth) for l in range(n)]
        cout = c + n * growth
        trans = 'features.transition%d' % i if i < len(counts) else None
        out.append(dict(prefix='features.denseblock%d' % i, cin=c, growth=growth, layers=layers, cout=cout, transition=trans))
        c = cout // 2 if trans else cout
    return out


def _densenet_run(sd, x, name, collect=None, fp16=False, calibrate=False):
    """model/densenet.py:64-65 (features: conv0 norm0 relu0 pool0, dense blocks, transitions, norm5, conv), in fp32 as the reference runs.
    fp16: float64, rounded to fp16 where the B200 kernels store fp16, each transition pooled before its conv as the kernels do.
    calibrate: float64, normalising with (and storing into sd) each BatchNorm's batch statistics instead of its running ones."""
    dt = torch.float64 if (fp16 or calibrate) else torch.float32
    r = (lambda t: t.half().to(dt)) if fp16 else (lambda t: t)

    def p(key):
        return sd[key].to(dt)

    def bn(y, prefix):
        if calibrate:
            sd[prefix + '.running_mean'] = y.mean((0, 2, 3)).float()
            sd[prefix + '.running_var'] = y.var((0, 2, 3), unbiased=False).float()
        return F.batch_norm(y, p(prefix + '.running_mean'), p(prefix + '.running_var'), p(prefix + '.weight'), p(prefix + '.bias'), False, 0.0, 1e-5)

    x = r(F.relu(bn(F.conv2d(x.to(dt), p('features.conv0.weight'), None, 2, 3), 'features.norm0')))
    x = F.max_pool2d(x, 3, 2, 1)
    if collect is not None:
        collect['features.pool0'] = x.float()
    for blk in densenet_blocks(name):
        feats = [x]
        for lp, _ in blk['layers']:
            a = r(F.relu(bn(torch.cat(feats, 1), lp + '.norm1')))
            bott = r(F.relu(bn(F.conv2d(a, r(p(lp + '.conv1.weight'))), lp + '.norm2')))
            feats.append(r(F.conv2d(bott, r(p(lp + '.conv2.weight')), None, 1, 1)))
        x = torch.cat(feats, 1)
        if collect is not None:
            collect[blk['prefix']] = x.float()
        t = blk['transition']
        if t is not None:
            a = F.relu(bn(x, t + '.norm'))
            if fp16:
                x = r(F.conv2d(r(F.avg_pool2d(a, 2)), r(p(t + '.conv.weight'))))
            else:
                x = F.avg_pool2d(F.conv2d(a, p(t + '.conv.weight')), 2)
            if collect is not None:
                collect[t] = x.float()
    n5 = bn(x, 'features.norm5')
    if collect is not None:
        collect['features.norm5'] = n5.float()
    w, b = p('features.conv.weight'), p('features.conv.bias')
    if not fp16:
        return F.conv2d(n5, w, b).float()
    # the head folds norm5 (no ReLU follows it, :53-54): W' = W diag(s), b' = b + W t, W' stored fp16
    s = p('features.norm5.weight') / torch.sqrt(p('features.norm5.running_var') + 1e-5)
    shift = p('features.norm5.bias') - p('features.norm5.running_mean') * s
    return F.conv2d(x, r(w * s[None, :, None, None]), b + (w[:, :, 0, 0] * shift[None, :]).sum(1)).float()


def make_densenet_state_dict(name='densenet121', seed=0, num_anchors=5, num_cls=20):
    """Deterministic synthetic DenseNet state_dict with torchvision's current key names: kaiming-normal convs as model/densenet.py:57-62,
    BatchNorm gamma / beta randomised so folding is exercised, and every running mean / variance set to the batch statistics of one
    float64 pass over two 128x128 synth_images, which keeps each stage's activations O(1) through the 58..98 layers."""
    init, growth, _ = DENSENET_CONFIGS[name]
    g = torch.Generator().manual_seed(seed)
    sd = {}

    def conv(key, cout, cin, k):
        sd[key + '.weight'] = torch.randn(cout, cin, k, k, generator=g) * math.sqrt(2.0 / (cin * k * k))

    def bn(prefix, c):
        sd[prefix + '.weight'] = torch.rand(c, generator=g) + 0.5
        sd[prefix + '.bias'] = torch.randn(c, generator=g) * 0.1
        sd[prefix + '.running_mean'] = torch.zeros(c)
        sd[prefix + '.running_var'] = torch.ones(c)

    conv('features.conv0', init, 3, 7)
    bn('features.norm0', init)
    for blk in densenet_blocks(name):
        for lp, c in blk['layers']:
            bn(lp + '.norm1', c)
            conv(lp + '.conv1', DENSENET_BN_SIZE * growth, c, 1)
            bn(lp + '.norm2', DENSENET_BN_SIZE * growth)
            conv(lp + '.conv2', growth, DENSENET_BN_SIZE * growth, 3)
        if blk['transition'] is not None:
            bn(blk['transition'] + '.norm', blk['cout'])
            conv(blk['transition'] + '.conv', blk['cout'] // 2, blk['cout'], 1)
    cin = densenet_blocks(name)[-1]['cout']
    bn('features.norm5', cin)
    ch = num_anchors * (5 + num_cls) if num_cls > 1 else num_anchors * 5
    sd['features.conv.weight'] = torch.randn(ch, cin, 1, 1, generator=g) * math.sqrt(1.0 / cin)
    sd['features.conv.bias'] = torch.randn(ch, generator=g) * 0.1
    with torch.no_grad():
        _densenet_run(sd, synth_images(2, 128, 128, seed=7), name, calibrate=True)
    return sd


def densenet_forward(sd, x, name='densenet121', collect=None, fp16=False):
    """Eval-mode DenseNet (model/densenet.py:64-65): x [B,3,H,W] -> [B, A*(5+C), H/32, W/32] fp32.  `collect`
    receives features.pool0, every denseblockN / transitionN output and features.norm5.  fp16=True is the error model of the B200
    path: fp16 at the stem output, every norm1+relu1 output, bottleneck output, growth-conv output, pooled transition input and
    transition output, every packed conv weight and the norm5-folded head weight; all other arithmetic float64."""
    with torch.no_grad():
        return _densenet_run(sd, x, name, collect, fp16)
