#!/usr/bin/env python
"""Golden fixture for the DenseNet plugin, produced by EXECUTING the reference's `model.densenet` (model/densenet.py:29-117) on CPU with the
oracle's deterministic synthetic weights:

    python tests/golden/make_golden_densenet.py        # build container only (needs /root/reference)

Stores the densenet121 head feature at 64x64 and 416x416, every denseblockN / transitionN / norm5 output of densenet121 at 64x64, the
64x64 head of densenet169, densenet201 and densenet161, and densenet121's state_dict key names and shapes.  The reference is imported
with make_golden.py's in-memory shims plus two for the installed torchvision / torch: `torchvision.models.densenet.model_urls` (removed
from torchvision, imported at densenet.py:24) and the `nn.init.kaiming_normal` alias (densenet.py:59); nothing is copied."""
import os
import sys

import numpy as np
import torch
import torch.nn as nn
import torchvision.models.densenet

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))
import densenet_oracle as DO  # noqa: E402
import make_golden as G  # noqa: E402
from oracle import yolo2_oracle as O  # noqa: E402

STAGES = ['features.denseblock1', 'features.transition1', 'features.denseblock2', 'features.transition2', 'features.denseblock3',
          'features.transition3', 'features.denseblock4', 'features.norm5']


def run(model, config, anchors, name, sizes, acts_at):
    import model.densenet
    sd = DO.make_densenet_state_dict(name, seed=0)
    net = getattr(model.densenet, name)(model.ConfigChannels(config), anchors, 20)
    res = net.load_state_dict(sd, strict=False)
    assert not res.unexpected_keys and all(k.endswith('num_batches_tracked') for k in res.missing_keys), res
    net.eval()
    outs = {}
    hooks = [net.features.get_submodule(k[len('features.'):]).register_forward_hook(
        lambda mod, inp, out, key=k: outs.__setitem__(key, out.detach().clone())) for k in STAGES]
    rec = {}
    with torch.no_grad():
        for size, seed in sizes:
            x = O.synth_images(1, size, size, seed=seed)
            f = net(x)
            rec['%s_feature%d' % (name, size)] = f.numpy()
            if size == acts_at:
                rec.update({'%s_act_%s' % (name, k): v.numpy() for k, v in outs.items()})
            # the restatement must agree with the executed reference to fp32 rounding
            o = DO.densenet_forward(sd, x, name)
            err = ((o - f).norm() / f.norm()).item()
            assert err < 1e-5, (name, size, err)
    for h in hooks:
        h.remove()
    if name == 'densenet121':
        state = net.state_dict()
        rec['densenet121_keys'] = np.array(list(state.keys()))
        rec['densenet121_shapes'] = np.array([str(tuple(v.shape)) for v in state.values()])
    return rec


def main():
    torchvision.models.densenet.model_urls = {}
    if not hasattr(nn.init, 'kaiming_normal'):
        nn.init.kaiming_normal = nn.init.kaiming_normal_
    model, utils, detect = G.import_reference()
    config = G.make_config(1)
    config.read_dict({'model': {'pretrained': '0'}})
    anchors = O.anchors_yolo_voc()
    rec = {}
    rec.update(run(model, config, anchors, 'densenet121', [(64, 10), (416, 0)], 64))
    for name in ('densenet169', 'densenet201', 'densenet161'):
        rec.update(run(model, config, anchors, name, [(64, 10)], None))
    path = os.path.join(HERE, 'densenet.npz')
    np.savez_compressed(path, **rec)
    print('densenet.npz %.1f KB' % (os.path.getsize(path) / 1024), sorted(rec))


if __name__ == '__main__':
    main()
