#!/usr/bin/env python
"""Generate the golden fixtures in tests/golden/*.npz by EXECUTING THE REFERENCE'S OWN CODE.

Run in the build container only (needs /root/reference; the GPU box has no reference):

    python tests/golden/make_golden.py

The reference (ruiminshen/yolo2-pytorch @ 146ebdf) is imported from /root/reference, never copied.
Two shims are applied in memory, nothing else is changed:
  * utils/__init__.py:109 uses `async` as a parameter name (SyntaxError on Python >= 3.7); the
    source text is loaded with that identifier renamed to `non_blocking` before exec.
  * detect.py cannot be imported (humanize / pybenchmark / cv2 GUI imports, detect.py:28-32), so
    the three pure functions on the path (get_logits, filter_visible, postprocess;
    detect.py:43-80) are extracted from its source by `ast` and exec'd with a no-op
    `pybenchmark.profile`.
Inputs are the deterministic synthetic generators of oracle/yolo2_oracle.py (weights are
regenerated from the seed on every machine, only the reference's OUTPUTS are stored).
"""
import ast
import configparser
import os
import sys
import types
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = '/root/reference'
sys.path.insert(0, ROOT)
warnings.filterwarnings('ignore')

from oracle import yolo2_oracle as O  # noqa: E402  (input generators only)


def import_reference():
    sys.path.insert(0, REF)
    src = open(os.path.join(REF, 'utils', '__init__.py')).read()
    src = src.replace('async=False', 'non_blocking=False').replace('device_id, async)', 'device_id, non_blocking)')
    mod = types.ModuleType('utils')
    mod.__path__ = [os.path.join(REF, 'utils')]
    mod.__file__ = os.path.join(REF, 'utils', '__init__.py')
    sys.modules['utils'] = mod
    exec(compile(src, mod.__file__, 'exec'), mod.__dict__)
    import model  # noqa
    import model.yolo2  # noqa
    import model.mobilenet  # noqa
    import utils.postprocess  # noqa
    import utils.iou.torch  # noqa
    # detect.py pure functions
    tree = ast.parse(open(os.path.join(REF, 'detect.py')).read())
    wanted = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in ('get_logits', 'filter_visible', 'postprocess')]
    pyb = types.SimpleNamespace(profile=lambda name: (lambda fn: fn))
    ns = dict(torch=torch, utils=sys.modules['utils'], pybenchmark=pyb)
    exec(compile(ast.Module(body=wanted, type_ignores=[]), os.path.join(REF, 'detect.py'), 'exec'), ns)
    return sys.modules['model'], sys.modules['utils'], types.SimpleNamespace(**{k: ns[k] for k in ('get_logits', 'filter_visible', 'postprocess')})


def make_config(fix):
    config = configparser.ConfigParser()
    config.read_dict({
        'batch_norm': {'enable': '1'},
        'detect': {'threshold': '0.3', 'threshold_cls': '0.005', 'fix': str(int(fix)), 'overlap': '0.45'},
    })
    return config


def box_indices(all_yx_min, all_yx_max, det_yx_min, det_yx_max):
    """Index (among the image's predictions) of every detection the reference returned: postprocess copies box rows, so the rows are
    bit-identical to exactly one prediction."""
    table = {}
    a, b = all_yx_min.numpy(), all_yx_max.numpy()
    for i in range(a.shape[0]):
        table.setdefault(a[i].tobytes() + b[i].tobytes(), []).append(i)
    out = []
    for lo, hi in zip(det_yx_min.numpy(), det_yx_max.numpy()):
        hit = table[lo.tobytes() + hi.tobytes()]
        assert len(hit) == 1, 'ambiguous box'
        out.append(hit[0])
    return np.array(out, dtype=np.int64)


def build_ref_darknet(model, sd):
    config = make_config(1)
    anchors = O.anchors_yolo_voc()
    dnn = model.yolo2.Darknet(model.ConfigChannels(config), anchors, 20)
    missing = dnn.load_state_dict(sd, strict=False)
    assert not missing.unexpected_keys, missing
    assert all(k.endswith('num_batches_tracked') for k in missing.missing_keys), missing
    dnn.eval()
    return dnn, anchors, config


def main():
    model, utils, detect = import_reference()
    sd = O.make_state_dict(seed=0)
    dnn, anchors, config = build_ref_darknet(model, sd)

    # ---- 1. backbone at 64x64: every conv unit's output ------------------------------------
    outs = {}
    hooks = []
    for name, m in dnn.named_modules():
        if isinstance(m, model.yolo2.Conv2d):
            hooks.append(m.register_forward_hook(lambda mod, inp, out, name=name: outs.__setitem__(name, out.detach().clone())))
    x64 = O.synth_images(1, 64, 64, seed=10)
    with torch.no_grad():
        f64 = dnn(x64)
    np.savez_compressed(os.path.join(HERE, 'darknet_64.npz'), feature=f64.numpy(),
                        **{'act_' + k: v.numpy() for k, v in outs.items()})

    # ---- 2. backbone at 416x416: feature + per-layer checksums ------------------------------
    # evaluated in float64 and stored rounded to float32: fp32 sums over 23 layers differ from CPU to CPU (vector ISA, thread
    # count) by more than the test's tolerances, so the fixture holds the exact values, which the test's float64 oracle meets anywhere
    outs.clear()
    x416 = O.synth_images(1, 416, 416, seed=0)
    with torch.no_grad():
        f416 = dnn.double()(x416.double())
    dnn.float()
    np.savez_compressed(os.path.join(HERE, 'darknet_416.npz'), feature=f416.float().numpy(),
                        **{'absmean_' + k: np.float64(v.abs().mean().item()) for k, v in outs.items()},
                        **{'head_' + k: v.flatten()[:64].float().numpy() for k, v in outs.items()})
    for h in hooks:
        h.remove()

    # ---- 3. reorg ---------------------------------------------------------------------------
    g = torch.Generator().manual_seed(5)
    xr = torch.randn(2, 8, 6, 4, generator=g)
    np.savez_compressed(os.path.join(HERE, 'reorg.npz'), x=xr.numpy(), y=model.yolo2.reorg(xr, 2, 2).numpy())

    # ---- 4. decode (+softmax) on a wide-range synthetic feature -----------------------------
    g = torch.Generator().manual_seed(6)
    feat = torch.randn(2, 125, 13, 13, generator=g) * 1.5
    inference = model.Inference(config, lambda t: t, anchors)
    with torch.no_grad():
        pred = model._inference(inference, feat)
        prob = torch.nn.functional.softmax(detect.get_logits(pred), -1)
    dec = {k: v.numpy() for k, v in pred.items()}
    dec['prob'] = prob.numpy()
    dec['anchors'] = anchors.numpy()
    np.savez_compressed(os.path.join(HERE, 'decode.npz'), **dec)

    # ---- 5. NMS -----------------------------------------------------------------------------
    nms = {}
    for tag, n, seed, overlap in (('a', 300, 3, 0.45), ('b', 1000, 4, 0.45), ('c', 64, 7, 0.3), ('d', 1, 8, 0.45), ('e', 2, 9, 0.45)):
        score, a, b = O.synth_boxes(n, seed)
        keep = utils.postprocess.nms(score, a, b, overlap)
        nms['score_' + tag], nms['yx_min_' + tag], nms['yx_max_' + tag] = score.numpy(), a.numpy(), b.numpy()
        nms['overlap_' + tag] = np.float64(overlap)
        nms['keep_' + tag] = np.array([int(i) for i in keep], dtype=np.int64)
    # decode-derived candidates (image 0, all 845 boxes)
    score, a, b = pred['iou'][0].reshape(-1), pred['yx_min'][0].reshape(-1, 2), pred['yx_max'][0].reshape(-1, 2)
    keep = utils.postprocess.nms(score, a, b, 0.45)
    nms['score_f'], nms['yx_min_f'], nms['yx_max_f'] = score.numpy(), a.numpy(), b.numpy()
    nms['overlap_f'] = np.float64(0.45)
    nms['keep_f'] = np.array([int(i) for i in keep], dtype=np.int64)
    assert utils.postprocess.nms(torch.zeros(0), torch.zeros(0, 2), torch.zeros(0, 2)) == []
    np.savez_compressed(os.path.join(HERE, 'nms.npz'), **nms)

    # ---- 6. detect.postprocess, fix=1 and fix=0, per image ----------------------------------
    post = {}
    for fix in (1, 0):
        cfg = make_config(fix)
        for bi in range(feat.size(0)):
            iou, yx_min, yx_max, p = (t[bi].reshape(-1, *t.shape[3:]) if t.dim() > 3 else t[bi].reshape(-1)
                                      for t in (pred['iou'], pred['yx_min'], pred['yx_max'], prob))
            # filter_visible alone
            fv = detect.filter_visible(cfg, iou, yx_min, yx_max, p)
            tag = 'fix%d_img%d_' % (fix, bi)
            for name, t in zip(('iou', 'yx_min', 'yx_max', 'prob', 'prob_cls', 'cls'), fv):
                post[tag + 'fv_' + name] = t.numpy()
            res = detect.postprocess(cfg, iou, yx_min, yx_max, p)
            post[tag + 'none'] = np.array(res is None)
            if res is not None:
                for name, t in zip(('iou', 'yx_min', 'yx_max', 'cls', 'score'), res):
                    post[tag + name] = t.numpy()
    # an image where nothing survives -> None
    cfg = make_config(0)
    res = detect.postprocess(cfg, torch.full((845,), 0.1), torch.zeros(845, 2), torch.ones(845, 2), torch.full((845, 20), 0.05))
    post['empty_none'] = np.array(res is None)
    np.savez_compressed(os.path.join(HERE, 'postprocess.npz'), **post)

    # ---- 7. IoU known-answer tests: run the reference's functions on its own test inputs ----
    # utils/iou/torch.py:79-113 (test0: unit neighbours -> 0; test1: 1/7 and 1/4)
    a_min = torch.tensor([[1., 1.], [0., 0.]]); a_max = torch.tensor([[3., 3.], [4., 4.]])
    b_min = torch.tensor([[0., 0.], [0., 2.], [2., 0.], [2., 2.]]); b_max = torch.tensor([[2., 2.], [2., 4.], [4., 2.], [4., 4.]])
    m1 = utils.iou.torch.iou_matrix(a_min, a_max, b_min, b_max)
    c_min = torch.tensor([[1., 1.]]); c_max = torch.tensor([[2., 2.]])
    nb = [(0, 0), (0, 1), (0, 2), (1, 0), (1, 2), (2, 0), (2, 1), (2, 2)]
    d_min = torch.tensor([[float(y), float(x)] for y, x in nb]); d_max = d_min + 1
    m0 = utils.iou.torch.iou_matrix(c_min, c_max, d_min, d_max)
    g = torch.Generator().manual_seed(11)
    r_min = torch.rand(3, 40, 2, generator=g) * 10; r_max = r_min + torch.rand(3, 40, 2, generator=g) * 5
    s_min = torch.rand(3, 7, 2, generator=g) * 10; s_max = s_min + torch.rand(3, 7, 2, generator=g) * 5
    mb = utils.iou.torch.batch_iou_matrix(r_min, r_max, s_min, s_max)
    np.savez_compressed(os.path.join(HERE, 'iou.npz'),
                        a_min=a_min.numpy(), a_max=a_max.numpy(), b_min=b_min.numpy(), b_max=b_max.numpy(), m1=m1.numpy(),
                        c_min=c_min.numpy(), c_max=c_max.numpy(), d_min=d_min.numpy(), d_max=d_max.numpy(), m0=m0.numpy(),
                        r_min=r_min.numpy(), r_max=r_max.numpy(), s_min=s_min.numpy(), s_max=s_max.numpy(), mb=mb.numpy())
    # ---- 8. MobileNet plugin (BASELINE configs[4]): feature at 64x64 and 416x416 + per-unit checksums ----
    msd = O.make_mobilenet_state_dict(seed=0)
    mnet = model.mobilenet.MobileNet(model.ConfigChannels(config), anchors, 20)
    res = mnet.load_state_dict(msd, strict=False)
    assert not res.unexpected_keys and all(k.endswith('num_batches_tracked') for k in res.missing_keys), res
    mnet.eval()
    mouts = {}
    hooks = [m.register_forward_hook(lambda mod, inp, out, name=name: mouts.__setitem__(name, out.detach().clone()))
             for name, m in mnet.layers.named_children()]
    with torch.no_grad():
        mf64 = mnet(O.synth_images(1, 64, 64, seed=10))
        acts64 = {'act_layers.' + k: v.numpy() for k, v in mouts.items() if k != '14'}
        mf416 = mnet(O.synth_images(1, 416, 416, seed=0))
    np.savez_compressed(os.path.join(HERE, 'mobilenet.npz'), feature64=mf64.numpy(), feature416=mf416.numpy(), **acts64,
                        **{'absmean416_layers.' + k: np.float64(v.double().abs().mean().item()) for k, v in mouts.items()})
    for h in hooks:
        h.remove()
    for f in sorted(os.listdir(HERE)):
        if f.endswith('.npz'):
            print('%-20s %8.1f KB' % (f, os.path.getsize(os.path.join(HERE, f)) / 1024))


if __name__ == '__main__':
    main()
