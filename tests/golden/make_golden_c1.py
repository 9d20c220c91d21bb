#!/usr/bin/env python
"""Golden fixture for BASELINE configs[0] ("C1": single-image inference, detect.py on image.jpg), produced by EXECUTING the
reference's own chain on CPU: cv2.imread -> transform.resize.image.rescale (cv2.resize) -> BGR2RGB -> ToTensor
(detect.py:142-146, config/darknet/yolo-voc.ini:10 drops Normalize) -> model.yolo2.Darknet (eval) -> model.Inference decode ->
softmax -> detect.postprocess (fix = 1).  Weights are the oracle's deterministic synthetic state_dict (no pretrained file
exists offline).  The 416x416 RGB uint8 network input (an OUTPUT of the reference's transform) is stored so the tests do
not need /root/reference.

    python tests/golden/make_golden_c1.py          # build container only (needs /root/reference + cv2)
"""
import os
import sys
import warnings

import cv2
import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
warnings.filterwarnings('ignore')
import make_golden as G  # noqa: E402
from oracle import yolo2_oracle as O  # noqa: E402


def main():
    model, utils, detect = G.import_reference()
    sd = O.make_state_dict(seed=0)
    dnn, anchors, config = G.build_ref_darknet(model, sd)
    image_bgr = cv2.imread(os.path.join(G.REF, 'image.jpg'))
    resized = cv2.resize(image_bgr, (416, 416))                         # transform/resize/image.py:23-24
    rgb = cv2.cvtColor(resized, cv2.COLOR_BGR2RGB)                      # transform/image.py:27-29
    tensor = torch.from_numpy(rgb.transpose(2, 0, 1).copy()).float().div(255).unsqueeze(0)     # torchvision ToTensor
    # the backbone in float64, its output rounded once to float32 (fp32 sums differ from CPU to CPU by more than the test's
    # tolerances); decode, softmax and postprocess run in float32 on that feature as in detect.py
    inference = model.Inference(config, lambda t: t, anchors)
    inference.eval()
    with torch.no_grad():
        pred = model._inference(inference, dnn.double()(tensor.double()).float())
        prob = torch.nn.functional.softmax(detect.get_logits(pred), -1)
        iou, yx_min, yx_max, p = (t[0].reshape(-1, *t.shape[3:]) if t.dim() > 3 else t[0].reshape(-1) for t in (pred['iou'], pred['yx_min'], pred['yx_max'], prob))
        res = detect.postprocess(config, iou, yx_min, yx_max, p)
    out = dict(rgb=rgb, feature=pred['feature'].numpy(), none=np.array(res is None))
    if res is not None:
        for name, t in zip(('iou', 'yx_min', 'yx_max', 'cls', 'score'), res):
            out['det_' + name] = t.numpy()
        out['det_box'] = G.box_indices(yx_min, yx_max, res[1], res[2])     # which of the 845 predictions each detection is a copy of
    path = os.path.join(HERE, 'c1_image.npz')
    np.savez_compressed(path, **out)
    print('c1_image.npz %.1f KB, detections: %s' % (os.path.getsize(path) / 1024, None if res is None else len(res[3])))


if __name__ == '__main__':
    main()
