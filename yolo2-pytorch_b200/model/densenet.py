"""model.densenet -- DenseNet backbone plugin on the B200 kernels (inference).

Drop-in for the reference's `model/densenet.py` (file:line cited per item): same constructors `densenet121 / densenet169 / densenet201 /
densenet161 (config_channels, anchors, num_cls)` (:68-117), same state_dict keys as torchvision's DenseNet (`features.conv0.weight`,
`features.denseblockN.denselayerL.norm1.*`, `features.transitionN.conv.weight`, `features.norm5.*`) plus the 1x1 detection head
`features.conv.{weight,bias}` (:54), same forward contract x[B,3,H,W] fp32 -> [B, A*(5+C), H/32, W/32] fp32 (:64-65).  Checkpoints with
the torchvision 0.2 dense-layer names (`denselayerL.norm.1.weight`, `conv.2.weight`, ...) load too.

Modules only hold parameters; `DenseNet.plan(height, width)` is the whole forward as a launch list, and the forward executes it on fp16 NHWC
activations.  Each dense block owns one concatenation buffer [B, h, w, C_block_out]; every layer appends its growth channels in place:
  conv0 7x7 s2 + norm0 + relu0   -> yb_stem7x7_bn_relu_fwd (64 wide) / yb_stem7x7_96_bn_relu_fwd (densenet161)
  pool0 max 3x3 s2 p1            -> yb_maxpool3x3_s2_strided_f16 into channels [0, C0) of block 1's buffer
  dense layer (input C_l)        -> yb_bn_relu_f16 (norm1 + relu1 into a scratch buffer zero-padded to a multiple of 32 channels)
                                    -> 1x1 conv to 4g with norm2 + relu2 folded into its epilogue
                                    -> 3x3 conv to g, written at channels [C_l, C_l + g) of the block buffer
  transition                     -> yb_bn_relu_avgpool2x2_f16, then the 1x1 conv into channels [0, C/2) of the next block's buffer (pooling
                                    before a 1x1 conv is exact in real arithmetic; it does 4x fewer MMAs -- only the fp16 rounding order differs)
  norm5 + head conv              -> one 1x1 conv with norm5 folded into its weight and bias (no ReLU follows norm5, :53-54), fp32 NCHW out.
Training this plugin is not on the B200 path (train() forward raises).
"""
import re

import torch
import torch.nn as nn
import torch.nn.functional as F

import model
from b200 import ops as _ops

CONFIGS = {'densenet121': (64, 32, (6, 12, 24, 16)), 'densenet169': (64, 32, (6, 12, 32, 32)),
           'densenet201': (64, 32, (6, 12, 48, 32)), 'densenet161': (96, 48, (6, 12, 36, 24))}
STEMS = {64: 'yb_stem7x7_bn_relu_fwd', 96: 'yb_stem7x7_96_bn_relu_fwd'}

# torchvision < 0.3 named the dense-layer modules 'norm.1', 'relu.1', 'conv.1', 'norm.2', ...; its hosted ImageNet files still do
_LEGACY_KEY = re.compile(r'^(.*denselayer\d+\.(?:norm|relu|conv))\.((?:[12])\.(?:weight|bias|running_mean|running_var|num_batches_tracked))$')


def rename_legacy_keys(state_dict):
    """Rename `denselayerL.norm.1.weight` -> `denselayerL.norm1.weight` (and conv.1, norm.2, conv.2) in place; returns state_dict."""
    for key in list(state_dict.keys()):
        m = _LEGACY_KEY.match(key)
        if m is not None:
            state_dict[m.group(1) + m.group(2)] = state_dict.pop(key)
    return state_dict


def _roundup32(c):
    return (c + 31) // 32 * 32


class _DenseLayer(nn.Module):
    def __init__(self, channels_in, growth_rate, bn_size):
        nn.Module.__init__(self)
        self.norm1 = nn.BatchNorm2d(channels_in)
        self.relu1 = nn.ReLU(inplace=True)
        self.conv1 = nn.Conv2d(channels_in, bn_size * growth_rate, kernel_size=1, bias=False)
        self.norm2 = nn.BatchNorm2d(bn_size * growth_rate)
        self.relu2 = nn.ReLU(inplace=True)
        self.conv2 = nn.Conv2d(bn_size * growth_rate, growth_rate, kernel_size=3, padding=1, bias=False)


class _DenseBlock(nn.Module):
    def __init__(self, num_layers, channels_in, growth_rate, bn_size):
        nn.Module.__init__(self)
        for i in range(num_layers):
            self.add_module('denselayer%d' % (i + 1), _DenseLayer(channels_in + i * growth_rate, growth_rate, bn_size))


class _Transition(nn.Module):
    def __init__(self, channels_in, channels_out):
        nn.Module.__init__(self)
        self.norm = nn.BatchNorm2d(channels_in)
        self.relu = nn.ReLU(inplace=True)
        self.conv = nn.Conv2d(channels_in, channels_out, kernel_size=1, bias=False)
        self.pool = nn.AvgPool2d(kernel_size=2, stride=2)


class DenseNet(nn.Module):
    def __init__(self, config_channels, anchors, num_cls, growth_rate=32, block_config=(6, 12, 24, 16), num_init_features=64, bn_size=4, drop_rate=0):
        nn.Module.__init__(self)                # drop_rate only acts in training, which this plugin does not run
        self.growth_rate, self.block_config, self.num_init_features, self.bn_size = growth_rate, tuple(block_config), num_init_features, bn_size
        self.features = nn.Sequential()
        self.features.add_module('conv0', nn.Conv2d(3, num_init_features, kernel_size=7, stride=2, padding=3, bias=False))
        self.features.add_module('norm0', nn.BatchNorm2d(num_init_features))
        self.features.add_module('relu0', nn.ReLU(inplace=True))
        self.features.add_module('pool0', nn.MaxPool2d(kernel_size=3, stride=2, padding=1))
        c = num_init_features
        for i, n in enumerate(block_config):
            self.features.add_module('denseblock%d' % (i + 1), _DenseBlock(n, c, growth_rate, bn_size))
            c += n * growth_rate
            if i != len(block_config) - 1:
                self.features.add_module('transition%d' % (i + 1), _Transition(c, c // 2))
                c //= 2
        self.features.add_module('norm5', nn.BatchNorm2d(c))
        self.features.add_module('conv', nn.Conv2d(c, model.output_channels(len(anchors), num_cls), 1))
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight)
            elif isinstance(m, nn.BatchNorm2d):
                nn.init.ones_(m.weight)
                nn.init.zeros_(m.bias)
        self.register_load_state_dict_pre_hook(lambda module, state_dict, *args: rename_legacy_keys(state_dict))
        self._cache = {}
        self._plans = {}

    def train(self, mode=True):
        if bool(mode) != self.training:
            self._cache = {}
        return nn.Module.train(self, mode)

    # ---- the launch plan ------------------------------------------------------------------------------
    def plan(self, height, width):
        """The forward at input size height x width as data (no tensors, no side effects): `buffers` maps each activation buffer to its
        per-image (h, w, channels) -- 'stem', 'blockN' -- or, for the two buffers reused across layers in stream order ('scratch': norm1
        outputs and pooled transition inputs, 'bottleneck': the 4g-wide 1x1 outputs), to its per-image element count; `launches` lists
        every kernel launch in order with its parameter keys, source / destination buffer, channel counts, pitches and offsets."""
        c0, g, nb = self.num_init_features, self.growth_rate, len(self.block_config)
        widths, c = [], c0                      # (input, output) channels of each dense block
        for i, n in enumerate(self.block_config):
            widths.append((c, c + n * g))
            c = (c + n * g) // 2 if i < nb - 1 else c + n * g
        h, w = height // 4, width // 4
        buffers = {'stem': (height // 2, width // 2, c0)}
        launches = [dict(op='stem', params='features.conv0', bn='features.norm0', dst='stem', height=height, width=width, cout=c0),
                    dict(op='maxpool', src='stem', dst='block1', height=height // 2, width=width // 2, channels=c0, y_ld=widths[0][1], y_ch_off=0)]
        scratch = bottleneck = 0
        for i, (n, (c_in, c_out)) in enumerate(zip(self.block_config, widths), 1):
            block = 'block%d' % i
            buffers[block] = (h, w, c_out)
            bottleneck = max(bottleneck, h * w * self.bn_size * g)
            for l in range(n):
                p = 'features.denseblock%d.denselayer%d' % (i, l + 1)
                c_l, c_pad = c_in + l * g, _roundup32(c_in + l * g)
                scratch = max(scratch, h * w * c_pad)
                launches += [
                    dict(op='bn_relu', bn=p + '.norm1', src=block, x_ld=c_out, dst='scratch', height=h, width=w, channels=c_l, channels_padded=c_pad),
                    dict(op='conv', params=p + '.conv1', bn=p + '.norm2', src='scratch', x_ld=c_pad, cin=c_pad, ksize=1, height=h, width=w,
                         dst='bottleneck', cout=self.bn_size * g, y_ld=self.bn_size * g, y_ch_off=0, slope=0.0),
                    dict(op='conv', params=p + '.conv2', bn=None, src='bottleneck', x_ld=self.bn_size * g, cin=self.bn_size * g, ksize=3, height=h,
                         width=w, dst=block, cout=g, y_ld=c_out, y_ch_off=c_l, slope=1.0)]
            if i < nb:
                t = 'features.transition%d' % i
                scratch = max(scratch, (h // 2) * (w // 2) * c_out)
                launches += [dict(op='bn_relu_avgpool', bn=t + '.norm', src=block, x_ld=c_out, dst='scratch', height=h, width=w, channels=c_out),
                             dict(op='conv', params=t + '.conv', bn=None, src='scratch', x_ld=c_out, cin=c_out, ksize=1, height=h // 2, width=w // 2,
                                  dst='block%d' % (i + 1), cout=c_out // 2, y_ld=widths[i][1], y_ch_off=0, slope=1.0)]
                h, w = h // 2, w // 2
        c_last = widths[-1][1]
        launches.append(dict(op='head', params='features.conv', bn='features.norm5', src='block%d' % nb, x_ld=c_last, cin=c_last, ksize=1,
                             height=h, width=w, cout=self.features.conv.weight.shape[0]))
        buffers['scratch'], buffers['bottleneck'] = scratch, bottleneck
        return dict(buffers=buffers, launches=launches)

    # ---- operand preparation (cached per parameter version) ------------------------------------------
    def _cached(self, key, tensors, make):
        ver = tuple((t.data_ptr(), t._version) for t in tensors)
        hit = self._cache.get(key)
        if hit is None or hit[0] != ver:
            hit = (ver, make())
            self._cache[key] = hit
        return hit[1]

    def _fold(self, key):
        bn = self.get_submodule(key)
        ts = (bn.weight, bn.bias, bn.running_mean, bn.running_var)
        return self._cached(key, ts, lambda: _ops.bn_fold(*(t.detach().contiguous() for t in ts), eps=bn.eps))

    def _packed(self, key, cin):
        """fp16 [Cout, k, k, cin] weight, input channels zero-padded from the module's Cin up to cin."""
        wt = self.get_submodule(key).weight
        return self._cached(key, (wt,), lambda: _ops.pack_weight_f16(F.pad(wt.detach(), (0, 0, 0, 0, 0, cin - wt.shape[1])).contiguous(), 0))

    def _identity(self, cout, device):
        """scale 1 / shift 0 of the convs without a BatchNorm after them."""
        key = ('identity', cout, device)
        hit = self._cache.get(key)
        if hit is None:
            hit = self._cache[key] = (torch.ones(cout, dtype=torch.float32, device=device), torch.zeros(cout, dtype=torch.float32, device=device))
        return hit

    def _head(self):
        """norm5 folded into the head conv in fp32: W' = W diag(s), b' = b + W t; returns (fp16 packed W', b')."""
        conv, bn = self.features.conv, self.features.norm5

        def make():
            s, t = _ops.bn_fold(*(v.detach().contiguous() for v in (bn.weight, bn.bias, bn.running_mean, bn.running_var)), eps=bn.eps)
            wt = conv.weight.detach().float()
            folded = (wt * s[None, :, None, None]).contiguous()
            peak = folded.abs().max().item()
            if not peak <= 65504.0:
                raise ValueError('DenseNet (B200): the norm5-folded head weight reaches %g, beyond fp16' % peak)
            bias = (conv.bias.detach().float() + (wt[:, :, 0, 0] * t[None, :]).sum(1)).contiguous()
            return _ops.pack_weight_f16(folded, 0), bias
        return self._cached('head', (conv.weight, conv.bias, bn.weight, bn.bias, bn.running_mean, bn.running_var), make)

    # ---- forward ---------------------------------------------------------------------------------------
    def forward(self, x):
        if self.training:
            raise NotImplementedError('DenseNet (B200): the training step of this plugin is not built; use eval() -- Darknet, Tiny and MobileNet train')
        if not x.is_cuda:
            raise RuntimeError('DenseNet (B200): input must be a CUDA tensor; there is no CPU fallback')
        b, c, h, w = x.shape
        if c != 3 or h % 32 or w % 32:
            raise ValueError('DenseNet expects [B,3,H,W] with H, W multiples of 32')
        if self.num_init_features not in STEMS:
            raise ValueError('DenseNet (B200): the stem has a kernel for %s output channels, not %d' % (sorted(STEMS), self.num_init_features))
        return self.run(x.contiguous().float())

    def run(self, x, stages=None):
        """Execute plan(H, W) on x (fp32 NCHW, CUDA).  `stages`, when a dict, receives every block buffer ('blockN', fp16 NHWC): after the
        forward, blockN holds denseblockN's output, and its channels [0, C0) the output of the transition before it."""
        b, _, height, width = x.shape
        pl = self._plans.get((height, width))
        if pl is None:
            pl = self._plans[(height, width)] = self.plan(height, width)
        dev = x.device
        bufs = {}
        for name, shape in pl['buffers'].items():
            if isinstance(shape, tuple):
                bufs[name] = torch.empty((b,) + shape, dtype=torch.float16, device=dev)
            else:
                bufs[name] = torch.empty(b * shape, dtype=torch.float16, device=dev)

        def view(name, h, w, ld):
            buf = bufs[name]
            return buf if buf.dim() == 4 else buf[:b * h * w * ld].view(b, h, w, ld)

        out = None
        for op in pl['launches']:
            kind = op['op']
            if kind == 'stem':
                scale, shift = self._fold(op['bn'])
                _ops.call(STEMS[op['cout']], x, self.features.conv0.weight.detach().contiguous(), scale, shift, bufs['stem'], b, height, width)
            elif kind == 'maxpool':
                _ops.call('yb_maxpool3x3_s2_strided_f16', bufs['stem'], bufs[op['dst']], b, op['height'], op['width'], op['channels'], op['y_ld'],
                          op['y_ch_off'])
            elif kind == 'bn_relu':
                scale, shift = self._fold(op['bn'])
                h, w = op['height'], op['width']
                _ops.call('yb_bn_relu_f16', bufs[op['src']], op['x_ld'], scale, shift, view('scratch', h, w, op['channels_padded']),
                          op['channels_padded'], b * h * w, op['channels'], op['channels_padded'])
            elif kind == 'bn_relu_avgpool':
                scale, shift = self._fold(op['bn'])
                h, w = op['height'], op['width']
                _ops.call('yb_bn_relu_avgpool2x2_f16', bufs[op['src']], op['x_ld'], scale, shift, view('scratch', h // 2, w // 2, op['channels']),
                          b, h, w, op['channels'])
            elif kind == 'conv':
                h, w = op['height'], op['width']
                scale, shift = self._fold(op['bn']) if op['bn'] else self._identity(op['cout'], dev)
                _ops.conv_bn_act(view(op['src'], h, w, op['x_ld']), self._packed(op['params'], op['cin']), scale, shift, op['slope'],
                                 out=view(op['dst'], h, w, op['y_ld']), y_ch_off=op['y_ch_off'])
            else:
                weight, bias = self._head()
                ones, _ = self._identity(op['cout'], dev)
                out = _ops.conv_bn_act(bufs[op['src']], weight, ones, bias, 1.0, out_mode=_ops.OUT_F32_NCHW)
        if stages is not None:
            stages.update({k: v for k, v in bufs.items() if k.startswith('block')})
        return out


def _pretrained(net, config_channels, name):
    """`[model] pretrained` (model/densenet.py:70-77): copy the torchvision ImageNet weights whose keys exist in this model, after renaming
    the files' legacy dense-layer keys."""
    config = getattr(config_channels, 'config', None)
    if config is None or not config.getboolean('model', 'pretrained', fallback=False):
        return net
    import torchvision.models as tvm
    weights = getattr(tvm, 'DenseNet%s_Weights' % name[len('densenet'):]).IMAGENET1K_V1
    state_dict = net.state_dict()
    for key, value in rename_legacy_keys(dict(weights.get_state_dict(progress=False))).items():
        if key in state_dict:
            state_dict[key] = value
    net.load_state_dict(state_dict)
    return net


def _make(name, config_channels, anchors, num_cls, **kwargs):
    init, growth, blocks = CONFIGS[name]
    net = DenseNet(config_channels, anchors, num_cls, num_init_features=init, growth_rate=growth, block_config=blocks, **kwargs)
    return _pretrained(net, config_channels, name)


def densenet121(config_channels, anchors, num_cls, **kwargs):
    return _make('densenet121', config_channels, anchors, num_cls, **kwargs)


def densenet169(config_channels, anchors, num_cls, **kwargs):
    return _make('densenet169', config_channels, anchors, num_cls, **kwargs)


def densenet201(config_channels, anchors, num_cls, **kwargs):
    return _make('densenet201', config_channels, anchors, num_cls, **kwargs)


def densenet161(config_channels, anchors, num_cls, **kwargs):
    return _make('densenet161', config_channels, anchors, num_cls, **kwargs)
