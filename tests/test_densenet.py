"""DenseNet plugin (model/densenet.py): the oracle against the executed reference (tests/golden/make_golden_densenet.py), the module surface,
legacy checkpoint keys and the launch plan on CPU; on the GPU the new kernels against float64 torch, the concatenation-buffer writes with
canaries, the plugin against the golden at every stage, detection on top, and CUDA-graph replay.

The GPU bound of each stage is max(2 x EMULATED[stage], 5e-4) in relative L2 error against the golden.  EMULATED is the error of the
oracle's fp16 error model (densenet_oracle.densenet_forward(fp16=True): fp16 exactly where the kernels store fp16, float64 elsewhere)
against the same golden, with the committed synthetic weights; test_emulated_errors_have_not_drifted recomputes it."""
import configparser
import os
import sys

import numpy as np
import pytest
import torch

from oracle import yolo2_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import densenet_oracle as DO  # noqa: E402

NAMES = ('densenet121', 'densenet169', 'densenet201', 'densenet161')
STAGES = ('features.denseblock1', 'features.transition1', 'features.denseblock2', 'features.transition2', 'features.denseblock3',
          'features.transition3', 'features.denseblock4')
EMULATED = {
    'features.denseblock1': 9.90e-04,
    'features.transition1': 1.05e-03,
    'features.denseblock2': 2.72e-03,
    'features.transition2': 2.15e-03,
    'features.denseblock3': 5.93e-03,
    'features.transition3': 4.67e-03,
    'features.denseblock4': 8.35e-03,
    'densenet121_feature64': 9.62e-03,
    'densenet169_feature64': 9.62e-03,
    'densenet201_feature64': 1.22e-02,
    'densenet161_feature64': 9.83e-03,
    'densenet121_feature416': 1.57e-02,
}
DEV = 'cuda'


def rel_l2(got, ref):
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    return ((got - ref).norm() / ref.norm().clamp_min(1e-30)).item()


def bound(key):
    return max(2.0 * EMULATED[key], 5e-4)


@pytest.fixture(scope='module')
def golden(golden_dir):
    return np.load(os.path.join(golden_dir, 'densenet.npz'))


def make_config():
    config = configparser.ConfigParser()
    config.read_dict({'model': {'dnn': 'model.densenet.densenet121', 'pretrained': '0'},
                      'batch_norm': {'enable': '1'},
                      'detect': {'threshold': '0.3', 'threshold_cls': '0.005', 'fix': '1', 'overlap': '0.45'}})
    return config


def build(name):
    import model
    import model.densenet  # noqa: F401
    import utils
    return utils.parse_attr('model.densenet.' + name)(model.ConfigChannels(make_config()), O.anchors_yolo_voc(), 20)


def legacy_names(sd):
    """The torchvision 0.2 / torch 0.3.1 spelling of dense-layer keys: denselayerL.norm1.weight -> denselayerL.norm.1.weight."""
    out = {}
    for k, v in sd.items():
        if '.denselayer' in k:
            head, mod, param = k.rsplit('.', 2)
            k = '%s.%s.%s.%s' % (head, mod[:-1], mod[-1], param)
        out[k] = v
    return out


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
def test_densenet_oracle_matches_reference_golden(golden):
    sd = DO.make_densenet_state_dict('densenet121', 0)
    collect = {}
    f64 = DO.densenet_forward(sd, O.synth_images(1, 64, 64, seed=10), 'densenet121', collect=collect)
    assert rel_l2(f64, torch.from_numpy(golden['densenet121_feature64'])) <= 1e-5
    for key in STAGES + ('features.norm5',):
        assert rel_l2(collect[key], torch.from_numpy(golden['densenet121_act_' + key])) <= 1e-5, key
    f416 = DO.densenet_forward(sd, O.synth_images(1, 416, 416, seed=0), 'densenet121')
    assert f416.shape == (1, 125, 13, 13) and rel_l2(f416, torch.from_numpy(golden['densenet121_feature416'])) <= 1e-5
    for name in NAMES[1:]:
        f = DO.densenet_forward(DO.make_densenet_state_dict(name, 0), O.synth_images(1, 64, 64, seed=10), name)
        assert rel_l2(f, torch.from_numpy(golden[name + '_feature64'])) <= 1e-5, name


def test_emulated_errors_have_not_drifted(golden):
    sd = DO.make_densenet_state_dict('densenet121', 0)
    collect = {}
    got = {'densenet121_feature64': rel_l2(DO.densenet_forward(sd, O.synth_images(1, 64, 64, seed=10), 'densenet121', collect, fp16=True),
                                           torch.from_numpy(golden['densenet121_feature64']))}
    got.update({k: rel_l2(collect[k], torch.from_numpy(golden['densenet121_act_' + k])) for k in STAGES})
    got['densenet121_feature416'] = rel_l2(DO.densenet_forward(sd, O.synth_images(1, 416, 416, seed=0), 'densenet121', fp16=True),
                                           torch.from_numpy(golden['densenet121_feature416']))
    for name in NAMES[1:]:
        got[name + '_feature64'] = rel_l2(DO.densenet_forward(DO.make_densenet_state_dict(name, 0), O.synth_images(1, 64, 64, seed=10), name, fp16=True),
                                          torch.from_numpy(golden[name + '_feature64']))
    assert set(got) == set(EMULATED)
    for k, v in got.items():
        assert abs(v - EMULATED[k]) <= 0.05 * EMULATED[k], (k, v, EMULATED[k])
    assert got['densenet121_feature416'] <= 3e-2


def test_densenet_state_dict_keys(golden):
    net = build('densenet121')
    sd = net.state_dict()
    assert list(sd) == list(golden['densenet121_keys']) and len(sd) == 727
    assert [str(tuple(v.shape)) for v in sd.values()] == list(golden['densenet121_shapes'])
    for name in NAMES:
        sd = build(name).state_dict()
        ref = DO.make_densenet_state_dict(name, 0)
        assert set(ref) == {k for k in sd if not k.endswith('num_batches_tracked')}, name
        assert all(tuple(sd[k].shape) == tuple(ref[k].shape) for k in ref), name


def test_densenet_loads_legacy_key_names():
    import utils.train
    sd = DO.make_densenet_state_dict('densenet121', 0)
    legacy = legacy_names(sd)
    assert 'features.denseblock1.denselayer1.norm.1.weight' in legacy and 'features.denseblock4.denselayer16.conv.2.weight' in legacy
    net = build('densenet121')
    utils.train.load_state_dict(net, legacy)
    state = net.state_dict()
    assert all(torch.equal(state[k], v) for k, v in sd.items())
    assert 'features.denseblock1.denselayer1.norm.1.weight' in legacy        # the caller's dict is not renamed
    net2 = build('densenet121')
    res = net2.load_state_dict(legacy, strict=False)
    assert not res.unexpected_keys and all(k.endswith('num_batches_tracked') for k in res.missing_keys)
    assert all(torch.equal(net2.state_dict()[k], v) for k, v in sd.items())
    bad = dict(legacy)
    bad['features.denseblock1.denselayer1.norm.3.weight'] = bad.pop('features.denseblock1.denselayer1.norm.1.weight')
    with pytest.raises(RuntimeError):
        utils.train.load_state_dict(build('densenet121'), bad)


def test_densenet_plan():
    for name in NAMES:
        net = build(name)
        pl = net.plan(416, 416)
        launches = pl['launches']
        init, growth, blocks = DO.DENSENET_CONFIGS[name]
        assert len(launches) == 1 + 1 + 3 * sum(blocks) + 2 * (len(blocks) - 1) + 1, name
        assert [l['op'] for l in launches[:2]] == ['stem', 'maxpool'] and launches[-1]['op'] == 'head'
        convs = [l for l in launches if l['op'] in ('conv', 'head')]
        assert all(l['cin'] % 32 == 0 and l['x_ld'] >= l['cin'] for l in convs), name
        for l in convs:
            assert tuple(net.get_submodule(l['params']).weight.shape[:1]) == (l['cout'],)
        for blk, ob in zip(DO.densenet_blocks(name), range(1, len(blocks) + 1)):
            key = 'block%d' % ob
            h, w, c_out = pl['buffers'][key]
            assert c_out == blk['cout'] and (h, w) == (416 // (4 << (ob - 1)),) * 2
            # every channel of the block buffer is written exactly once: the pool / transition at [0, C0), one growth conv per layer after it
            writes = [(l['y_ch_off'], l['y_ch_off'] + (l['channels'] if l['op'] == 'maxpool' else l['cout'])) for l in launches
                      if l.get('dst') == key]
            assert all(l['y_ld'] == c_out for l in launches if l.get('dst') == key)
            assert sorted(writes) == writes and writes[0][0] == 0 and writes[-1][1] == c_out
            assert all(a[1] == b[0] for a, b in zip(writes, writes[1:])), (name, key)
            norms = [l for l in launches if l['op'] == 'bn_relu' and l['src'] == key]
            assert [l['channels'] for l in norms] == [c for _, c in blk['layers']]
            assert all(l['channels_padded'] % 32 == 0 and 0 <= l['channels_padded'] - l['channels'] < 32 for l in norms)
            assert all(pl['buffers']['scratch'] >= h * w * l['channels_padded'] for l in norms)
        if name == 'densenet121':
            assert len(launches) == 183
        if name == 'densenet161':
            pads = [l['channels_padded'] for l in launches if l['op'] == 'bn_relu'][:3]
            assert pads == [96, 160, 192]                       # C_l = 96, 144, 192
            assert [l['channels'] for l in launches if l['op'] == 'bn_relu'][6 + 1] == 240   # block 2, layer 2: 192 + 48
            assert [l['channels_padded'] for l in launches if l['op'] == 'bn_relu'][6 + 1] == 256


def test_densenet_module_surface():
    net = build('densenet121')
    assert net.features.conv.weight.shape == (125, 1024, 1, 1) and net.features.norm5.num_features == 1024
    assert build('densenet161').features.conv0.weight.shape == (96, 3, 7, 7)
    with pytest.raises(RuntimeError):
        net.eval()(torch.zeros(1, 3, 32, 32))           # CPU tensor: no fallback
    with pytest.raises(NotImplementedError):
        net.train()(torch.zeros(1, 3, 32, 32))


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
CANARY = 0x5A5A          # an fp16 bit pattern no kernel output here can take (~203.25; outputs are O(1))


def _canary(n):
    return torch.full((n,), CANARY, dtype=torch.int16, device=DEV)


def _ulp_distance(got, ref64):
    """Distance in fp16 units of the last place between non-negative fp16 results and float64 references."""
    return (got.view(torch.int16).int() - ref64.half().view(torch.int16).int()).abs()


@pytest.mark.gpu
def test_bn_relu_kernels_vs_float64():
    from b200 import ops
    g = torch.Generator().manual_seed(11)
    for c in (64, 144, 1024, 2208):
        scale = (torch.rand(c, generator=g) + 0.5).to(DEV)
        shift = (torch.randn(c, generator=g) * 0.5).to(DEV)
        for (b, h, w) in ((1, 104, 104), (2, 13, 27), (3, 1, 1)):
            x_ld = c + 16
            x = (torch.randn(b, h, w, x_ld, generator=g) * 2).half().to(DEV)
            ref = torch.relu(x[..., :c].double() * scale.double() + shift.double())
            # norm1 + relu1 into a padded scratch: channels [c, c_pad) are zeros, [c_pad, y_ld) and everything around y untouched
            c_pad = (c + 31) // 32 * 32
            y_ld = c_pad + 8
            n = b * h * w * y_ld
            flat = _canary(n + 128)
            y = flat[64:64 + n].view(torch.float16).view(b, h, w, y_ld)
            ops.call('yb_bn_relu_f16', x, x_ld, scale, shift, y, y_ld, b * h * w, c, c_pad)
            assert int(_ulp_distance(y[..., :c], ref).max()) <= 1, (c, h, w)
            assert bool((y[..., c:c_pad] == 0).all()) and bool((y[..., c:c_pad].view(torch.int16) == 0).all())
            assert bool((y[..., c_pad:].view(torch.int16) == CANARY).all())
            assert bool((flat[:64] == CANARY).all()) and bool((flat[64 + n:] == CANARY).all())
            # norm + relu + 2x2 average, odd sizes floored
            if h < 2:
                with pytest.raises(RuntimeError):
                    ops.call('yb_bn_relu_avgpool2x2_f16', x, x_ld, scale, shift, y, b, h, w, c)
                continue
            oh, ow = h // 2, w // 2
            n = b * oh * ow * c
            flat = _canary(n + 128)
            y = flat[64:64 + n].view(torch.float16).view(b, oh, ow, c)
            ops.call('yb_bn_relu_avgpool2x2_f16', x, x_ld, scale, shift, y, b, h, w, c)
            ref_p = torch.nn.functional.avg_pool2d(ref.permute(0, 3, 1, 2), 2).permute(0, 2, 3, 1)
            assert int(_ulp_distance(y, ref_p).max()) <= 1, (c, h, w)
            assert bool((flat[:64] == CANARY).all()) and bool((flat[64 + n:] == CANARY).all())
    x = torch.zeros(1, 4, 4, 64, dtype=torch.float16, device=DEV)
    s = torch.ones(64, device=DEV)
    y = torch.empty_like(x)
    for bad in ((x, 64, s, s, y, 64, 16, 60, 64), (x, 60, s, s, y, 64, 16, 64, 64), (x, 64, s, s, y, 64, 16, 64, 32)):
        with pytest.raises(RuntimeError):
            ops.call('yb_bn_relu_f16', *bad)
    with pytest.raises(RuntimeError):
        ops.call('yb_bn_relu_f16', x.view(-1)[1:], 64, s, s, y, 64, 15, 64, 64)   # 2-byte aligned input


@pytest.mark.gpu
def test_strided_maxpool_into_block_buffer():
    from b200 import ops
    g = torch.Generator().manual_seed(12)
    for (b, h, w, c, y_ld, off) in ((2, 208, 208, 64, 256, 0), (1, 13, 27, 96, 384, 96), (2, 32, 48, 64, 256, 64)):
        x = torch.randn(b, h, w, c, generator=g).half().to(DEV)
        oh, ow = (h + 1) // 2, (w + 1) // 2
        plain = torch.empty(b, oh, ow, c, dtype=torch.float16, device=DEV)
        ops.call('yb_maxpool3x3_s2_f16', x, plain, b, h, w, c)
        y = _canary(b * oh * ow * y_ld).view(torch.float16).view(b, oh, ow, y_ld)
        ops.call('yb_maxpool3x3_s2_strided_f16', x, y, b, h, w, c, y_ld, off)
        ref = torch.nn.functional.max_pool2d(x.permute(0, 3, 1, 2).float(), 3, 2, 1).permute(0, 2, 3, 1)
        assert torch.equal(y[..., off:off + c], plain) and torch.equal(plain.float(), ref)
        rest = torch.cat([y[..., :off], y[..., off + c:]], -1)
        assert bool((rest.view(torch.int16) == CANARY).all())
    with pytest.raises(RuntimeError):
        ops.call('yb_maxpool3x3_s2_strided_f16', x, y, b, h, w, c, y_ld, y_ld - 32)   # slice past the pitch


@pytest.mark.gpu
def test_growth_conv_writes_only_its_slice():
    """A 3x3 conv with Cout 32 / 48 into a 256-channel buffer: the 64-wide output tile is clipped at Cout, so every channel outside
    [y_ch_off, y_ch_off + Cout) stays byte-identical to the canary, and the slice equals the conv written on its own."""
    from b200 import ops
    g = torch.Generator().manual_seed(13)
    for (b, h, w) in ((2, 26, 26), (1, 104, 104)):
        x = torch.randn(b, h, w, 128, generator=g).half().to(DEV)
        for cout in (32, 48):
            wt = ops.pack_weight_f16((torch.randn(cout, 128, 3, 3, generator=g) * 0.05).to(DEV), 0)
            one, zero = torch.ones(cout, device=DEV), torch.zeros(cout, device=DEV)
            alone = ops.conv_bn_act(x, wt, one, zero, 1.0)
            for off in (64, 208):
                buf = _canary(b * h * w * 256).view(torch.float16).view(b, h, w, 256)
                ops.conv_bn_act(x, wt, one, zero, 1.0, out=buf, y_ch_off=off)
                assert torch.equal(buf[..., off:off + cout], alone), (cout, off)
                rest = torch.cat([buf[..., :off], buf[..., off + cout:]], -1)
                assert bool((rest.view(torch.int16) == CANARY).all()), (cout, off)


def _gpu_net(name):
    net = build(name)
    res = net.load_state_dict(DO.make_densenet_state_dict(name, 0), strict=False)
    assert not res.unexpected_keys and all(k.endswith('num_batches_tracked') for k in res.missing_keys)
    return net.to(DEV).eval()


@pytest.mark.gpu
def test_densenet_plugin_vs_reference_golden(golden):
    rec = {}
    net = _gpu_net('densenet121')
    stages = {}
    with torch.no_grad():
        f64 = net.run(O.synth_images(1, 64, 64, seed=10).to(DEV), stages)
    for i, key in enumerate(STAGES):
        n = int(key[-1])
        if 'denseblock' in key:
            got = stages['block%d' % n]
        else:
            c0 = golden['densenet121_act_' + key].shape[1]
            got = stages['block%d' % (n + 1)][..., :c0]
        rec[key] = rel_l2(got.permute(0, 3, 1, 2), torch.from_numpy(golden['densenet121_act_' + key]))
    rec['densenet121_feature64'] = rel_l2(f64, torch.from_numpy(golden['densenet121_feature64']))
    with torch.no_grad():
        f416 = net(O.synth_images(1, 416, 416, seed=0).to(DEV))
    assert f416.shape == (1, 125, 13, 13) and f416.dtype == torch.float32
    rec['densenet121_feature416'] = rel_l2(f416, torch.from_numpy(golden['densenet121_feature416']))
    for name in NAMES[1:]:
        with torch.no_grad():
            f = _gpu_net(name)(O.synth_images(1, 64, 64, seed=10).to(DEV))
        rec[name + '_feature64'] = rel_l2(f, torch.from_numpy(golden[name + '_feature64']))
    print('densenet rel L2 vs golden (bound):', {k: '%.2e (%.2e)' % (v, bound(k)) for k, v in rec.items()})
    for k, v in rec.items():
        assert v <= bound(k), (k, v, bound(k))


@pytest.mark.gpu
def test_densenet_detection_graph_and_surface():
    import detect
    import model
    import utils
    from b200 import ops
    cfg = make_config()
    anchors = O.anchors_yolo_voc()
    net = utils.parse_attr(cfg.get('model', 'dnn'))(model.ConfigChannels(cfg), anchors, 20)
    net.load_state_dict(DO.make_densenet_state_dict('densenet121', 0), strict=False)
    net = net.to(DEV).eval()
    inference = model.Inference(cfg, net, anchors).eval()
    x = O.synth_images(3, 416, 416, seed=2).to(DEV)
    pred = model._inference(inference, x)
    assert pred['feature'].shape == (3, 125, 13, 13) and bool(torch.isfinite(pred['feature']).all())
    assert len(detect.postprocess_batch(cfg, pred)) == 3
    # one launch per plan entry once the folded operands are cached
    with torch.no_grad():
        eager = net(x)
        before = ops.launch_count
        eager = net(x)
        assert ops.launch_count - before == len(net.plan(416, 416)['launches']) == 183
    # no host synchronisation or allocation outside the caching allocator: the forward captures and replays
    static_x = x.clone()
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream), torch.no_grad():
        net(static_x)
    torch.cuda.current_stream().wait_stream(stream)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph), torch.no_grad():
        static_out = net(static_x)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(static_out, eager)
    with pytest.raises(ValueError):
        net(torch.zeros(1, 3, 48, 64, device=DEV))
    with pytest.raises(NotImplementedError):
        net.train()(x)
