"""CPU: pin the oracle (oracle/yolo2_oracle.py) against fixtures produced by executing the
reference's own code (tests/golden/make_golden.py) and against the reference's embedded IoU
known-answer tests (utils/iou/torch.py:79-113,179-213)."""
import os

import numpy as np
import pytest
import torch

from oracle import yolo2_oracle as O


def load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


def test_topology_matches_reference_keys():
    sd = O.make_state_dict(0)
    layers = O.darknet19_layers()
    assert len(layers) == 23
    assert sum(v.numel() for k, v in sd.items() if 'running' not in k) == 50655389 - 0  # SURVEY 8a row 4 (params)
    assert layers[-1]['cout'] == 125 and layers[-2]['cin'] == 1280


def test_backbone_64_every_layer(golden_dir):
    g = load(golden_dir, 'darknet_64.npz')
    sd = O.make_state_dict(0)
    x = O.synth_images(1, 64, 64, seed=10)
    collect = {}
    with torch.no_grad():
        f = O.darknet_forward(sd, x, collect=collect)
    for key, act in collect.items():
        ref = g['act_' + key]
        np.testing.assert_allclose(act.numpy(), ref, rtol=0, atol=2e-5 * max(1.0, np.abs(ref).max()), err_msg=key)
    np.testing.assert_allclose(f.numpy(), g['feature'], rtol=0, atol=2e-5 * np.abs(g['feature']).max())


def _double(sd):
    return {k: v.double() if v.is_floating_point() else v for k, v in sd.items()}


def test_backbone_416_feature(golden_dir):
    """Both sides in float64 (the fixture rounded to float32): fp32 sums over 23 layers depend on the CPU's vector ISA and thread
    count by more than these tolerances."""
    g = load(golden_dir, 'darknet_416.npz')
    sd = _double(O.make_state_dict(0))
    x = O.synth_images(1, 416, 416, seed=0).double()
    collect = {}
    with torch.no_grad():
        f = O.darknet_forward(sd, x, collect=collect)
    ref = g['feature']
    assert np.abs(f.numpy() - ref).max() <= 2e-5 * np.abs(ref).max()
    for key, act in collect.items():
        assert abs(act.double().abs().mean().item() - float(g['absmean_' + key])) <= 1e-5 * float(g['absmean_' + key]), key
        np.testing.assert_allclose(act.flatten()[:64].numpy(), g['head_' + key], rtol=1e-4, atol=1e-5)


def test_reorg_bit_exact(golden_dir):
    g = load(golden_dir, 'reorg.npz')
    assert np.array_equal(O.reorg(torch.from_numpy(g['x'])).numpy(), g['y'])


def test_decode_and_softmax(golden_dir):
    g = load(golden_dir, 'decode.npz')
    pred = O.decode(torch.from_numpy(g['feature']), torch.from_numpy(g['anchors']))
    for k in ('iou', 'center_offset', 'size_norm', 'yx_min', 'yx_max', 'logits'):
        np.testing.assert_allclose(pred[k].numpy(), g[k], rtol=1e-6, atol=1e-6, err_msg=k)
    np.testing.assert_allclose(O.class_prob(pred).numpy(), g['prob'], rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize('tag', list('abcdef'))
def test_nms_indices_exact(golden_dir, tag):
    g = load(golden_dir, 'nms.npz')
    keep = O.nms(g['score_' + tag], g['yx_min_' + tag], g['yx_max_' + tag], float(g['overlap_' + tag]))
    assert keep == g['keep_' + tag].tolist()


def test_nms_empty():
    assert O.nms(np.zeros(0), np.zeros((0, 2)), np.zeros((0, 2))) == []


@pytest.mark.parametrize('fix', [1, 0])
@pytest.mark.parametrize('img', [0, 1])
def test_postprocess(golden_dir, fix, img):
    g = load(golden_dir, 'postprocess.npz')
    d = load(golden_dir, 'decode.npz')
    iou = torch.from_numpy(d['iou'][img]).reshape(-1)
    yx_min = torch.from_numpy(d['yx_min'][img]).reshape(-1, 2)
    yx_max = torch.from_numpy(d['yx_max'][img]).reshape(-1, 2)
    prob = torch.from_numpy(d['prob'][img]).reshape(-1, 20)
    tag = 'fix%d_img%d_' % (fix, img)
    fv = O.filter_visible(iou, yx_min, yx_max, prob, fix, 0.3, 0.005)
    for name, t in zip(('iou', 'yx_min', 'yx_max', 'prob', 'prob_cls', 'cls'), fv):
        assert np.array_equal(t.numpy(), g[tag + 'fv_' + name]), name
    res = O.postprocess(iou, yx_min, yx_max, prob, fix, 0.3, 0.005, 0.45)
    assert (res is None) == bool(g[tag + 'none'])
    if res is not None:
        for name, t in zip(('iou', 'yx_min', 'yx_max', 'cls', 'score'), res):
            np.testing.assert_allclose(t.numpy(), g[tag + name], rtol=1e-6, atol=0, err_msg=name)


def test_postprocess_none(golden_dir):
    g = load(golden_dir, 'postprocess.npz')
    assert bool(g['empty_none'])
    res = O.postprocess(torch.full((845,), 0.1), torch.zeros(845, 2), torch.ones(845, 2), torch.full((845, 20), 0.05), 0, 0.3, 0.005, 0.45)
    assert res is None


def test_iou_known_answers(golden_dir):
    g = load(golden_dir, 'iou.npz')
    t = lambda k: torch.from_numpy(g[k])
    m0 = O.iou_matrix(t('c_min'), t('c_max'), t('d_min'), t('d_max'))
    np.testing.assert_almost_equal(m0.numpy(), np.zeros((1, 8), np.float32))      # utils/iou/torch.py:79-95 (test0)
    np.testing.assert_almost_equal(m0.numpy(), g['m0'])
    m1 = O.iou_matrix(t('a_min'), t('a_max'), t('b_min'), t('b_max'))
    np.testing.assert_almost_equal(m1.numpy(), np.array([[1 / 7] * 4, [4 / 16] * 4], np.float32))  # :97-113 (test1)
    assert np.array_equal(m1.numpy(), g['m1'])
    mb = O.batch_iou_matrix(t('r_min'), t('r_max'), t('s_min'), t('s_max'))
    assert np.array_equal(mb.numpy(), g['mb'])


def test_loss_restatement_self_consistency():
    """Self-consistency of the restated loss (it is also pinned against the executed reference below); check its closed-form gradient
    (SURVEY 8a derived spec) against autograd and basic invariants."""
    torch.manual_seed(0)
    anchors = O.anchors_yolo_voc()
    B, S, G = 3, 13, 6
    feature = (torch.randn(B, 125, S, S) * 0.5).requires_grad_(True)
    data = O.norm_data(O.synth_targets(B, 416, 416, slots=G), 416, 416, S, S)
    pred = O.decode(feature, anchors)
    losses, dbg = O.loss(anchors, data, pred, 0.6)
    total = O.loss_total(losses)
    total.backward()
    pos, neg = dbg['positive'], dbg['negative']
    assert pos.sum() > 0 and not (pos & neg).any()
    cnt = B * S * S * 5
    f = feature.detach().permute(0, 2, 3, 1).reshape(B, S * S, 5, 25)
    sig = torch.sigmoid(f[..., :3])
    t_c, t_s = O.fill_norm(dbg['data']['yx_min'], dbg['data']['yx_max'], anchors)
    gexp = torch.zeros_like(f)
    p = pos.float(); n = neg.float()
    gexp[..., 0] = (5 * 2 * (sig[..., 0] - dbg['iou']) * p + 2 * sig[..., 0] * n) * sig[..., 0] * (1 - sig[..., 0]) / cnt
    gexp[..., 1:3] = 2 * (sig[..., 1:3] - t_c) * sig[..., 1:3] * (1 - sig[..., 1:3]) * p[..., None] / cnt
    gexp[..., 3:5] = torch.where(pos[..., None], 2 * (f[..., 3:5] - t_s) / cnt, torch.zeros(()))
    onehot = torch.nn.functional.one_hot(dbg['data']['cls'], 20).float()
    gexp[..., 5:] = (torch.softmax(f[..., 5:], -1) - onehot) * p[..., None] / (pos.sum() * cnt)
    gexp = gexp.reshape(B, S, S, 125).permute(0, 3, 1, 2)
    np.testing.assert_allclose(feature.grad.numpy(), gexp.numpy(), rtol=1e-4, atol=1e-9)


def test_mobilenet_oracle_matches_reference(golden_dir):
    """BASELINE configs[4]: the MobileNet restatement vs the reference's own model.mobilenet.MobileNet outputs."""
    g = load(golden_dir, 'mobilenet.npz')
    sd = O.make_mobilenet_state_dict(0)
    collect = {}
    with torch.no_grad():
        f64 = O.mobilenet_forward(sd, O.synth_images(1, 64, 64, seed=10), collect=collect)
        f416 = O.mobilenet_forward(sd, O.synth_images(1, 416, 416, seed=0))
    for k, v in collect.items():
        ref = g['act_' + k]
        assert np.abs(v.numpy() - ref).max() <= 2e-5 * max(1.0, np.abs(ref).max()), k
    assert np.abs(f64.numpy() - g['feature64']).max() <= 2e-5 * np.abs(g['feature64']).max()
    assert np.abs(f416.numpy() - g['feature416']).max() <= 2e-5 * np.abs(g['feature416']).max()
    assert sum(v.numel() for k, v in sd.items() if 'running' not in k) == 3335101          # SURVEY 8a row 23


def test_resnet_oracle_matches_reference_golden(golden_dir):
    """oracle.resnet_forward (restating model/resnet.py:28-142) against outputs of the reference's own resnet18 (BasicBlock) and
    resnet50 (Bottleneck) modules (tests/golden/make_golden_resnet.py): stem pool + every block at 64x64, the feature at 64 and 416."""
    g = np.load(os.path.join(golden_dir, 'resnet.npz'))
    sd = O.make_resnet_state_dict('resnet18', 0)
    collect = {}
    with torch.no_grad():
        f64 = O.resnet_forward(sd, O.synth_images(1, 64, 64, seed=10), 'resnet18', collect=collect)
        f416 = O.resnet_forward(sd, O.synth_images(1, 416, 416, seed=0), 'resnet18')
        g64 = O.resnet_forward(O.make_resnet_state_dict('resnet50', 0), O.synth_images(1, 64, 64, seed=10), 'resnet50')
    assert f64.shape == (1, 125, 2, 2) and f416.shape == (1, 125, 13, 13)
    np.testing.assert_allclose(f64.numpy(), g['resnet18_feature64'], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(f416.numpy(), g['resnet18_feature416'], rtol=1e-4, atol=2e-5)
    np.testing.assert_allclose(g64.numpy(), g['resnet50_feature64'], rtol=1e-4, atol=1e-5)
    keys = [k for k in g.files if k.startswith('resnet18_act_')]
    assert len(keys) == 9
    for k in keys:
        np.testing.assert_allclose(collect[k[len('resnet18_act_'):]].numpy(), g[k], rtol=1e-4, atol=1e-5, err_msg=k)


def test_tiny_oracle_matches_reference_golden(golden_dir):
    """oracle.tiny_forward (restating model/yolo2.py:140-173) against outputs of the reference's own Tiny module
    (tests/golden/make_golden_tiny.py): every conv unit at 64x64 and the 416x416 feature map."""
    g = np.load(os.path.join(golden_dir, 'tiny.npz'))
    sd = O.make_tiny_state_dict(seed=0)
    collect = {}
    with torch.no_grad():
        f64 = O.tiny_forward(sd, O.synth_images(1, 64, 64, seed=10), collect=collect)
        f416 = O.tiny_forward(sd, O.synth_images(1, 416, 416, seed=0))
    assert f64.shape == (1, 125, 2, 2) and f416.shape == (1, 125, 13, 13)
    np.testing.assert_allclose(f64.numpy(), g['feature64'], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(f416.numpy(), g['feature416'], rtol=1e-4, atol=1e-5)
    keys = [k for k in g.files if k.startswith('act_')]
    assert len(keys) == 9
    for k in keys:
        np.testing.assert_allclose(collect[k[4:]].numpy(), g[k], rtol=1e-4, atol=1e-5, err_msg=k)


def _eval_cases(g):
    tags = sorted({k.split('_')[0] for k in g.files if k.startswith('case')})
    for tag in tags:
        yield tag, {k[len(tag) + 1:]: g[k] for k in g.files if k.startswith(tag + '_')}


def test_eval_matching_and_ap_oracle_matches_reference_golden(golden_dir):
    """oracle eval_matching / average_precision (restating eval.py:57-121) against outputs of the reference's own
    functions (tests/golden/make_golden_eval.py), including the no-ground-truth and no-detection cases."""
    g = load(golden_dir, 'eval.npz')
    for tag, case in _eval_cases(g):
        tp = np.zeros(case['det_cls'].shape[0], dtype=bool)
        for c in range(int(case['num_cls'])):
            dm, gm = case['det_cls'] == c, case['gt_cls'] == c
            tp[dm] = O.eval_matching(torch.from_numpy(case['gt_min'][gm]), torch.from_numpy(case['gt_max'][gm]),
                                     torch.from_numpy(case['det_min'][dm]), torch.from_numpy(case['det_max'][dm]), 0.5)
        assert np.array_equal(tp, case['tp']), tag
    for c in range(20):
        for metric07 in (0, 1):
            ap = O.average_precision(g['sorted_tp_cls%d' % c], int(g['num_cls%d' % c]), bool(metric07))
            assert abs(ap - float(g['ap%d_cls%d' % (metric07, c)])) <= 1e-12, (c, metric07)


def test_resize_oracle_matches_cv2_golden(golden_dir):
    """oracle.resize_u8 / rescale_label (OpenCV's 8-bit INTER_LINEAR restated) against outputs of the reference's
    transform.resize.label.rescale run with cv2 itself (tests/golden/make_golden_resize.py): bit-exact."""
    import hashlib
    g = load(golden_dir, 'resize.npz')
    assert np.array_equal(O.resize_u8(g['small_src'], 64, 96), g['small_out'])
    for seed in range(8):
        h0, w0, h, w = (int(v) for v in g['case%d_dims' % seed])
        out = O.resize_u8(O.synth_frame(seed, h0, w0), h, w)
        assert out.shape == (h, w, 3)
        assert hashlib.sha256(out.tobytes()).digest() == g['case%d_sha' % seed].tobytes(), seed
    # the reference's own sample image (tests/golden/image.jpg), decoded as the golden script decoded it
    import cv2
    img = cv2.imread(os.path.join(golden_dir, 'image.jpg'))
    assert hashlib.sha256(img.tobytes()).digest() == g['jpg_src_sha'].tobytes()
    r, a, b = O.rescale_label(img, g['jpg_yx_min_in'].copy(), g['jpg_yx_max_in'].copy(), 416, 416)
    assert hashlib.sha256(r.tobytes()).digest() == g['jpg_sha_bgr'].tobytes()
    assert hashlib.sha256(r[..., ::-1].tobytes()).digest() == g['jpg_sha_rgb'].tobytes()
    assert np.array_equal(a, g['jpg_yx_min']) and np.array_equal(b, g['jpg_yx_max'])
    assert np.array_equal(r[100:132, 200:232], g['jpg_crop'])


@pytest.mark.parametrize('tag', list('abcd'))
def test_region_loss_oracle_matches_executed_reference(golden_dir, tag):
    """oracle.loss (the restatement the CUDA kernels are checked against) vs the reference's OWN model.loss executed on CPU
    under the two documented torch-0.3.1 shims (tests/golden/make_golden_loss.py): the five terms, the positive / negative
    masks, the matched IoU and the gradient w.r.t. the head feature map; case d is the one-hot (train/cross_entropy = 0)
    branch, b a 19x19 grid, c a single ground-truth slot."""
    g = load(golden_dir, 'loss.npz')
    b, s, slots, seed, one_hot = (int(v) for v in g[tag + '_dims'])
    anchors = O.anchors_yolo_voc()
    feature = torch.from_numpy(g[tag + '_feature']).clone().requires_grad_(True)
    pred = O.decode(feature, anchors)
    pred['feature'] = feature
    data = O.norm_data(O.synth_targets(b, s * 32, s * 32, slots=slots, seed=20 + seed), s * 32, s * 32, s, s)
    losses, debug = O.loss(anchors, data, pred, 0.6, cross_entropy=not one_hot)
    for k, v in losses.items():
        ref = float(g[tag + '_loss_' + k])
        assert abs(v.item() - ref) <= 1e-5 * abs(ref) + 1e-9, (k, v.item(), ref)
    assert np.array_equal(debug['positive'].numpy().astype(np.uint8), g[tag + '_positive'])
    assert np.array_equal(debug['negative'].numpy().astype(np.uint8), g[tag + '_negative'])
    np.testing.assert_allclose(debug['iou'].numpy(), g[tag + '_iou'], rtol=1e-6, atol=1e-7)
    grad, = torch.autograd.grad(O.loss_total(losses), feature)
    np.testing.assert_allclose(grad.numpy(), g[tag + '_grad'], rtol=1e-4, atol=1e-8)


def test_training_step_oracle_matches_executed_reference(golden_dir):
    """One whole training step of the oracle (train-mode Darknet with batch-statistics BatchNorm, decode, region loss,
    hparam-weighted sum, autograd) against the same step executed with the reference's own modules
    (tests/golden/make_golden_train.py): head feature, loss terms, every parameter gradient (norm + first elements,
    small tensors in full) and the BatchNorm running statistics after the step (momentum 0.01, unbiased variance)."""
    g = load(golden_dir, 'train_step.npz')
    sd0 = O.make_state_dict(seed=0)
    anchors = O.anchors_yolo_voc()
    b, size = 4, 128
    s = size // 32
    x = O.synth_images(b, size, size, seed=12)
    data = O.norm_data(O.synth_targets(b, size, size, slots=6, seed=13), size, size, s, s)
    sd = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and 'running' not in k else v.clone()) for k, v in sd0.items()}
    stats, collect = {}, {}
    feature = O.darknet_forward(sd, x, train=True, stats=stats, collect=collect)
    pred = O.decode(feature, anchors)
    pred['feature'] = feature
    losses, _ = O.loss(anchors, data, pred, 0.6)
    O.loss_total(losses).backward()
    np.testing.assert_allclose(feature.detach().numpy(), g['feature'], rtol=2e-3, atol=2e-4)
    for k, v in losses.items():
        assert abs(v.item() - float(g['loss_' + k])) <= 1e-3 * abs(float(g['loss_' + k])), k
    for name, p in sd.items():
        if not p.requires_grad:
            continue
        gr = p.grad
        ref_norm = float(g['gnorm_' + name])
        assert abs(gr.double().norm().item() - ref_norm) <= 5e-3 * ref_norm + 1e-12, name
        head = g['ghead_' + name]
        np.testing.assert_allclose(gr.flatten()[:16].numpy(), head, rtol=2e-2, atol=2e-3 * float(np.abs(head).max()) + 1e-9, err_msg=name)
        if 'gfull_' + name in g.files:
            full = g['gfull_' + name]
            assert np.linalg.norm(gr.numpy() - full) <= 1e-2 * np.linalg.norm(full) + 1e-9, name
    # running statistics after one step: 0.99 * old + 0.01 * batch statistic (unbiased variance), model/yolo2.py:58
    for key, (mean, var) in stats.items():
        n = collect[key].numel() // collect[key].shape[1]
        exp_mean = 0.99 * sd0[key + '.bn.running_mean'] + 0.01 * mean.detach()
        exp_var = 0.99 * sd0[key + '.bn.running_var'] + 0.01 * var.detach() * n / (n - 1)
        np.testing.assert_allclose(exp_mean.numpy(), g['buf_' + key + '.bn.running_mean'], rtol=1e-3, atol=1e-5, err_msg=key)
        np.testing.assert_allclose(exp_var.numpy(), g['buf_' + key + '.bn.running_var'], rtol=1e-3, atol=1e-6, err_msg=key)


def test_c1_single_image_chain_oracle_matches_executed_reference(golden_dir):
    """BASELINE configs[0]: the reference's detect.py chain on its own image.jpg (resize, BGR2RGB, ToTensor, Darknet-19,
    decode, softmax, postprocess with detect/fix = 1), executed by tests/golden/make_golden_c1.py, against the oracle on the
    stored 416x416 RGB network input: feature map, and the detection tuple with exact class / box-index agreement.  The backbone runs
    in float64 on both sides, its feature rounded to float32 for the rest of the chain (as in test_backbone_416_feature)."""
    g = load(golden_dir, 'c1_image.npz')
    sd = _double(O.make_state_dict(seed=0))
    anchors = O.anchors_yolo_voc()
    x = torch.from_numpy(g['rgb'].transpose(2, 0, 1).copy()).float().div(255).unsqueeze(0).double()
    with torch.no_grad():
        feature = O.darknet_forward(sd, x).float()
        pred = O.decode(feature, anchors)
        prob = O.class_prob(pred)
        res = O.postprocess(pred['iou'][0].reshape(-1), pred['yx_min'][0].reshape(-1, 2), pred['yx_max'][0].reshape(-1, 2),
                            prob[0].reshape(-1, prob.size(-1)), True, 0.3, 0.005, 0.45)
    np.testing.assert_allclose(feature.numpy(), g['feature'], rtol=1e-4, atol=1e-5)
    assert (res is None) == bool(g['none'])
    if res is not None:
        assert res[3].tolist() == g['det_cls'].tolist()
        np.testing.assert_allclose(res[0].numpy(), g['det_iou'], rtol=1e-5, atol=1e-7)
        np.testing.assert_allclose(res[1].numpy(), g['det_yx_min'], rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose(res[4].numpy(), g['det_score'], rtol=1e-5, atol=1e-8)
    # the stored network input is what the oracle's cv2-exact resize produces from the reference's sample image
    import cv2
    assert np.array_equal(O.resize_u8(cv2.imread(os.path.join(golden_dir, 'image.jpg')), 416, 416)[..., ::-1], g['rgb'])


def test_c2_batch32_oracle_matches_executed_reference(golden_dir):
    """BASELINE configs[1] at its real size (32 x 3 x 416 x 416): the oracle chain against the reference's own modules executed on
    the same batch (tests/golden/make_golden_c2.py): three head features, every image's max|feature|, kept-box and detection counts,
    and the detections themselves (classes exact, boxes / scores to float tolerance)."""
    g = load(golden_dir, 'c2_batch32.npz')
    b = int(g['batch'])
    sd = O.make_state_dict(seed=0)
    anchors = O.anchors_yolo_voc()
    x = O.synth_images(b, 416, 416, seed=int(g['seed']))
    with torch.no_grad():
        feature = O.darknet_forward(sd, x)
        pred = O.decode(feature, anchors)
        prob = O.class_prob(pred)
    for slot, bi in enumerate(g['images']):
        np.testing.assert_allclose(feature[bi].numpy(), g['feature'][slot], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(feature.abs().reshape(b, -1).max(1).values.numpy(), g['feature_absmax'], rtol=1e-5)
    off = np.concatenate([[0], np.cumsum(g['n_det'])])
    for bi in range(b):
        res = O.postprocess(pred['iou'][bi].reshape(-1), pred['yx_min'][bi].reshape(-1, 2), pred['yx_max'][bi].reshape(-1, 2),
                            prob[bi].reshape(-1, prob.size(-1)), True, 0.3, 0.005, 0.45)
        assert (res is None) == (int(g['n_det'][bi]) == 0)
        if res is None:
            continue
        assert len(res[0]) == int(g['n_keep'][bi]) and len(res[3]) == int(g['n_det'][bi]), bi
        sl = slice(off[bi], off[bi + 1])
        assert np.array_equal(res[3].numpy(), g['det_cls'][sl])
        np.testing.assert_allclose(res[1].numpy(), g['det_yx_min'][sl], rtol=1e-4, atol=1e-4)
        np.testing.assert_allclose(res[4].numpy(), g['det_score'][sl], rtol=1e-3, atol=1e-6)
