"""Photometric training augmentations (reference transform/image.py:32-99): the numpy oracle against cv2 and the fixture made by
executing the reference's classes (tests/golden/make_golden_photometric.py), the host-side draws / tables / chain planning, and on the
GPU `yb_photometric_u8`, the `transform.image` classes and `Collate(..., transform_image=...)`.

Where cv2 4.13 disagrees with itself the oracle and the kernel take one side: cv2.blur with an area-2 kernel, (1, 2) or (2, 1),
wraps a window of two 255s to 0 in its scalar tail loop and saturates it in its vectorised body (here: 255); COLOR_HSV2RGB rounds
x * 255 in its per-pixel path and truncates it in its vectorised body (here: rounds).  The fixture stores each chain both ways and the
device must match the restored one."""
import configparser
import hashlib
import os
import random

import numpy as np
import pytest
import torch

from oracle import photometric as P
from oracle import yolo2_oracle as O

try:
    import cv2
except ImportError:  # the SHA half of the exhaustive checks still runs
    cv2 = None

CHAIN = ['RandomBlur', 'BGR2HSV', 'RandomHue', 'RandomSaturation', 'RandomBrightness', 'HSV2RGB', 'RandomGamma']
IMAGE_TRAIN = ' '.join('transform.image.' + n for n in CHAIN)   # the reference config.ini's commented `image_train` line
AUG = {'random_blur': '5 5', 'random_hue': '0 25', 'random_saturation': '0.5 1.5', 'random_brightness': '0.5 1.5', 'random_gamma': '0.9 1.5'}


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest()


@pytest.fixture(scope='module')
def G(golden_dir):
    return dict(np.load(os.path.join(golden_dir, 'photometric.npz')))


def config():
    cfg = configparser.ConfigParser()
    cfg.read_dict({'augmentation': AUG})
    return cfg


def oracle_chain(img, draws):
    kx, ky, hue, sat, bri, gam = draws
    return P.chain(img, blur=(int(kx), int(ky)), hue=int(hue), saturation=sat, brightness=bri, gamma=gam)


def flat_draws(ops):
    """One image's draws, in chain order, flattened as the fixture stores them."""
    out = []
    for op in ops:
        d = op.draw()
        out += [] if d is None else list(d) if isinstance(d, tuple) else [d]
    return out


def tables_for(draws):
    """(blur_k [2], lut_hsv [3, 256], lut_out [3, 256]) of one image of the full chain."""
    kx, ky, hue, sat, bri, gam = draws
    return ((int(kx), int(ky)), np.stack([P.hue_table(int(hue)), P.scale_table(sat), P.scale_table(bri)]), np.stack([P.gamma_table(gam)] * 3))


# ---------------------------------------------------------------- CPU


def test_oracle_hsv_conversions_exhaustive(G):
    fa = P.all_colours_frame()
    hsv = P.bgr2hsv(fa)
    assert sha(hsv) == G['bgr2hsv_all_sha'].tobytes()
    ft = P.hsv_triples_frame()
    rgb = P.hsv2rgb(ft)
    assert sha(rgb) == G['hsv2rgb_all_sha'].tobytes()
    if cv2 is not None:
        assert np.array_equal(hsv, cv2.cvtColor(fa, cv2.COLOR_BGR2HSV))
        assert np.array_equal(rgb, P.cv2_per_pixel(lambda x: cv2.cvtColor(x, cv2.COLOR_HSV2RGB), ft))


@pytest.mark.skipif(cv2 is None, reason='cv2 not installed')
def test_oracle_blur_matches_cv2_except_area2_wrap(G):
    frames = [G['s%d_src' % i] for i in range(int(G['small_count']))] + [G['cls_src'], O.synth_frame(1, 64, 80),
                                                                         (np.random.RandomState(0).rand(30, 31, 3) > 0.5).astype(np.uint8) * 255]
    wrapped_white = 0
    for fi, f in enumerate(frames):
        for kx in range(1, 6):
            for ky in range(1, 6):
                a, b = P.box_blur(f, kx, ky), cv2.blur(f, (kx, ky))
                d = a != b
                if d.any():
                    assert kx * ky == 2 and (b[d] == 0).all() and (a[d] == 255).all(), (f.shape, kx, ky)
                    if fi == 0:
                        wrapped_white += int(d.sum())
    assert wrapped_white > 0, 'the all-white frame must exercise the area-2 exception'


def test_oracle_chain_reproduces_fixture(G):
    for i in range(int(G['small_count'])):
        out = oracle_chain(G['s%d_src' % i], G['s%d_draws' % i])
        assert np.array_equal(out, G['s%d_out' % i]), i
    assert int(G['s0_restored']) > 0 and not np.array_equal(G['s0_out'], G['s0_out_cv2'])
    for name, (h, w) in (('b416', (416, 416)), ('b320x608', (320, 608))):
        for j, sd in enumerate(G[name + '_seeds']):
            f = O.synth_frame(int(sd), h, w)
            assert sha(f) == G[name + '_frame_sha'][j].tobytes()
            assert sha(oracle_chain(f, G[name + '_draws'][j])) == G[name + '_sha'][j].tobytes(), (name, j)


def test_draws_and_tables_match_reference_classes(G):
    import transform.image as TI
    cfg = config()
    ops = [getattr(TI, n)(cfg) if n.startswith('Random') else getattr(TI, n)() for n in CHAIN]
    for i in range(int(G['small_count'])):
        random.seed(int(G['s%d_seed' % i]))
        assert np.array_equal(np.array(flat_draws(ops), np.float64), G['s%d_draws' % i]), i
    # each class alone: host draw + host table == the reference class's output
    src, hsv = G['cls_src'], G['cls_src_hsv']
    for name, ch in (('RandomHue', 0), ('RandomSaturation', 1), ('RandomBrightness', 2)):
        random.seed(int(G['cls_%s_seed' % name]))
        op = getattr(TI, name)(cfg)
        d = op.draw()
        assert d == G['cls_%s_draws' % name][0]
        exp = hsv.copy()
        exp[..., ch] = op.table(d)[hsv[..., ch]]
        assert np.array_equal(exp, G['cls_' + name])
    random.seed(int(G['cls_RandomGamma_seed']))
    g = TI.RandomGamma(cfg).draw()
    assert np.array_equal(TI.gamma_table(g)[src], G['cls_RandomGamma'])
    assert np.array_equal(TI.gamma_table(g), P.gamma_table(g))
    random.seed(int(G['cls_RandomBlur_seed']))
    k = TI.RandomBlur(cfg).draw()
    assert np.array_equal(P.box_blur(src, *k), G['cls_RandomBlur'])
    assert np.array_equal(P.bgr2hsv(src), G['cls_BGR2HSV'])
    assert np.array_equal(P.hsv2rgb(hsv), G['cls_HSV2RGB'])


def test_get_transform_and_chain_plan():
    import transform
    import transform.image as TI
    from utils.data import Collate
    cfg = config()
    comp = transform.get_transform(cfg, IMAGE_TRAIN.split())
    assert [type(t).__name__ for t in comp.transforms] == CHAIN
    assert [len(g) for g in TI.split_chain(comp.transforms)] == [7]              # the reference chain is one launch
    assert [len(g) for g in TI.split_chain([TI.RandomGamma(cfg), TI.RandomBlur(cfg)])] == [1, 1]
    assert [len(g) for g in TI.split_chain([TI.RandomHue(cfg), TI.RandomHue(cfg), TI.RandomGamma(cfg)])] == [3]
    c = Collate([(416, 416)], seed=0, transform_image=comp)
    assert c.chain is not None and not c.bgr2rgb
    plain = Collate([(416, 416)], seed=0, transform_image=transform.get_transform(cfg, ['transform.image.BGR2RGB']))
    assert plain.chain is None and plain.bgr2rgb
    with pytest.raises(TypeError):
        Collate([(416, 416)], transform_image=[TI.RandomGamma(cfg), lambda x: x])
    bad = configparser.ConfigParser()
    bad.read_dict({'augmentation': {'random_blur': '16 5'}})
    with pytest.raises(ValueError):
        TI.RandomBlur(bad)


# ---------------------------------------------------------------- GPU

CANARY = 4096


def guarded(n):
    """A uint8 CUDA buffer with random canary bands of CANARY bytes around an n-byte middle -> (buffer, middle view, band copy)."""
    g = torch.Generator().manual_seed(n)
    buf = torch.randint(0, 256, (n + 2 * CANARY,), dtype=torch.uint8, generator=g).cuda()
    return buf, buf[CANARY:CANARY + n], buf.clone()


def bands_intact(buf, ref):
    return torch.equal(buf[:CANARY], ref[:CANARY]) and torch.equal(buf[-CANARY:], ref[-CANARY:])


def launch(src, dst, b, h, w, blur=None, to_hsv=0, lut_hsv=None, to_rgb=0, lut_out=None):
    from b200 import ops

    def up(a):
        return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()
    ops.call('yb_photometric_u8', src, dst, b, h, w, up(blur), int(to_hsv), up(lut_hsv), int(to_rgb), up(lut_out))


@pytest.mark.gpu
def test_gpu_hsv_conversions_exhaustive(G):
    for frame, key, flags in ((P.all_colours_frame(), 'bgr2hsv_all_sha', dict(to_hsv=1)), (P.hsv_triples_frame(), 'hsv2rgb_all_sha', dict(to_rgb=1))):
        h, w = frame.shape[:2]
        sbuf, src, sref = guarded(frame.size)
        src.copy_(torch.from_numpy(frame.reshape(-1)))
        sref = sbuf.clone()
        dbuf, dst, dref = guarded(frame.size)
        launch(src, dst, 1, h, w, **flags)
        torch.cuda.synchronize()
        assert sha(dst.cpu().numpy()) == G[key].tobytes(), key
        assert bands_intact(dbuf, dref) and torch.equal(sbuf, sref)


def run_batch(frames, draws):
    b, h, w, _ = frames.shape
    tabs = [tables_for(d) for d in draws]
    sbuf, src, _ = guarded(frames.size)
    src.copy_(torch.from_numpy(frames.reshape(-1)))
    dbuf, dst, dref = guarded(frames.size)
    launch(src, dst, b, h, w, blur=np.array([t[0] for t in tabs], np.int32), to_hsv=1, lut_hsv=np.stack([t[1] for t in tabs]), to_rgb=1,
           lut_out=np.stack([t[2] for t in tabs]))
    torch.cuda.synchronize()
    assert bands_intact(dbuf, dref), 'write outside the output'
    return dst.cpu().numpy().reshape(b, h, w, 3)


@pytest.mark.gpu
def test_gpu_full_chain_batches_and_small_frames(G):
    for name, (h, w) in (('b416', (416, 416)), ('b320x608', (320, 608))):
        frames = np.stack([O.synth_frame(int(sd), h, w) for sd in G[name + '_seeds']])
        out = run_batch(frames, G[name + '_draws'])
        for j in range(len(frames)):
            assert sha(out[j]) == G[name + '_sha'][j].tobytes(), (name, j, G[name + '_draws'][j][:2])
    for i in range(int(G['small_count'])):
        out = run_batch(G['s%d_src' % i][None], G['s%d_draws' % i][None])
        assert np.array_equal(out[0], G['s%d_out' % i]), (i, G['s%d_src' % i].shape)
    # k up to 15, odd and even, on a frame narrower and shorter than the window
    f = O.synth_frame(5, 6, 9)
    for k in ((15, 15), (14, 3), (1, 15), (8, 2)):
        out = run_batch(f[None], [(k[0], k[1], 0, 1.0, 1.0, 1.0)])
        assert np.array_equal(out[0], P.chain(f, blur=k, hue=0, saturation=1.0, brightness=1.0, gamma=1.0)), k


@pytest.mark.gpu
def test_gpu_each_class_alone(G):
    import transform.image as TI
    cfg = config()
    for name in CHAIN:
        op = getattr(TI, name)(cfg) if name.startswith('Random') else getattr(TI, name)()
        src = G['cls_src_hsv'] if name in ('RandomHue', 'RandomSaturation', 'RandomBrightness', 'HSV2RGB') else G['cls_src']
        random.seed(int(G['cls_%s_seed' % name]))
        out = op(src)
        assert out.is_cuda and tuple(out.shape) == src.shape
        assert np.array_equal(out.cpu().numpy(), G['cls_' + name]), name


@pytest.mark.gpu
def test_gpu_collate_chain_one_launch_and_training_step():
    import transform
    import train as yb_train
    import model
    import model.yolo2
    from b200 import ops
    from utils.data import Collate
    cfg = config()
    comp = transform.get_transform(cfg, IMAGE_TRAIN.split())
    rng = np.random.RandomState(3)
    batch = []
    for i, (h0, w0) in enumerate(((375, 500), (120, 90), (333, 500), (97, 131))):
        n = 1 + i % 3
        yx_min = (rng.rand(n, 2) * np.array([h0 * 0.5, w0 * 0.5])).astype(np.float32)
        batch.append(dict(image=O.synth_frame(80 + i, h0, w0), yx_min=yx_min, yx_max=yx_min + 8, cls=np.arange(n) % 20))
    collate = Collate([(128, 128)], seed=0, transform_image=comp)
    random.seed(77)
    n0 = ops.launch_count
    out = collate(batch)
    torch.cuda.synchronize()
    launches = ops.launch_count - n0
    assert launches == 2, 'resize + one photometric launch, got %d' % launches
    # the same draws on the host: image by image, chain order
    random.seed(77)
    got = out['tensor'].cpu().numpy()
    for i, d in enumerate(batch):
        draws = flat_draws(comp.transforms)
        resized = O.rescale_label(d['image'], d['yx_min'], d['yx_max'], 128, 128)[0]
        assert np.array_equal(got[i], oracle_chain(resized, draws)), i
    # the augmented batch drives a training step to a finite loss
    mcfg = configparser.ConfigParser()
    mcfg.read_dict({'batch_norm': {'enable': '1'}, 'model': {'threshold': '0.6'},
                    'hparam': {'foreground': '5', 'background': '1', 'center': '1', 'size': '1', 'cls': '1'}, 'train': {'cross_entropy': '1'}})
    anchors = O.anchors_yolo_voc()
    dnn = model.yolo2.Darknet(model.ConfigChannels(mcfg), anchors, 20)
    dnn.load_state_dict(O.make_state_dict(0), strict=False)
    dnn = dnn.cuda().train()
    inference = model.Inference(mcfg, dnn, anchors).train()
    opt = torch.optim.SGD(dnn.parameters(), 1e-4)
    step = yb_train.iterate(inference, opt, anchors, mcfg, out)
    torch.cuda.synchronize()
    loss = float(step['loss_total'].item())
    assert np.isfinite(loss) and loss > 0
