#!/usr/bin/env python
"""Golden fixture for the photometric training augmentations, produced by EXECUTING the reference's own classes (transform/image.py:32-99:
BGR2HSV, HSV2RGB, RandomBlur, RandomHue, RandomSaturation, RandomBrightness, RandomGamma) with cv2 4.13 -- the full commented
`image_train` chain of the reference's config.ini, with its `[augmentation]` ranges.  The module imports packages that are absent or
changed, so the classes are extracted with `ast` and run with three shims:
  - `inflection.underscore` (CamelCase -> snake_case) is restated;
  - `np.int` (removed in numpy 2) is set to `int`;
  - `skimage.exposure.adjust_gamma` (scikit-image is not installed) is restated in its current form,
    np.minimum(np.rint(255 * gain * np.linspace(0, 1, 256) ** gamma), 255) as a uint8 lookup table.
`random.seed` is fixed per image and every draw is stored, so the GPU test replays the same parameters.

cv2 4.13 is inconsistent with itself in two places, and the device follows one side of each:
  - blur: an area-2 kernel ((1, 2) or (2, 1)) wraps a window of two 255s to 0 in cv2's scalar tail loop and saturates it in the
    vectorised body.  The device saturates.
  - HSV2RGB: the vectorised body truncates x * 255, the per-pixel path rounds it.  The device rounds.
Each chain is therefore run twice from the same random state: as cv2 gives it, and "restored": the blur output's wrapped pixels set
back to 255 and HSV2RGB run through cv2's per-pixel path (a one-pixel-wide frame).  The number of restored blur pixels is stored.
The device must match the restored run.

Also stored: SHA-256 of cv2's BGR2HSV over all 2^24 colours and of its per-pixel HSV2RGB over all 180 * 256 * 256 valid triples (the
frames of oracle/photometric.py), so the GPU test needs neither cv2 nor the reference.

    python tests/golden/make_golden_photometric.py          # needs the reference checkout + cv2
"""
import ast
import configparser
import hashlib
import os
import random
import re
import sys
import types

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import photometric as P  # noqa: E402
from oracle import yolo2_oracle as O  # noqa: E402

REF = '/root/reference'
CHAIN = ['RandomBlur', 'BGR2HSV', 'RandomHue', 'RandomSaturation', 'RandomBrightness', 'HSV2RGB', 'RandomGamma']
AUG = {'random_blur': '5 5', 'random_hue': '0 25', 'random_saturation': '0.5 1.5', 'random_brightness': '0.5 1.5', 'random_gamma': '0.9 1.5'}


def sha(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), np.uint8)


class Recorder(object):
    """The `random` module, recording every randint / uniform result."""

    def __init__(self):
        self.draws = []

    def randint(self, a, b):
        v = random.randint(a, b)
        self.draws.append(float(v))
        return v

    def uniform(self, a, b):
        v = random.uniform(a, b)
        self.draws.append(float(v))
        return v


def adjust_gamma(image, gamma=1, gain=1):
    table = np.minimum(np.rint(255 * gain * np.linspace(0, 1, 256) ** gamma), 255).astype(np.uint8)
    return table[image]


def load_classes(rec):
    path = os.path.join(REF, 'transform', 'image.py')
    tree = ast.parse(open(path).read())
    nodes = [n for n in tree.body if isinstance(n, ast.ClassDef) and n.name in CHAIN]
    np.int = int                                                   # numpy 2 removed the alias RandomHue uses
    inflection = types.SimpleNamespace(underscore=lambda s: re.sub(r'(?<=[a-z0-9])([A-Z])', r'_\1', s).lower())
    skimage = types.SimpleNamespace(exposure=types.SimpleNamespace(adjust_gamma=adjust_gamma))
    ns = dict(np=np, cv2=cv2, random=rec, inflection=inflection, skimage=skimage)
    exec(compile(ast.Module(body=nodes, type_ignores=[]), path, 'exec'), ns)
    config = configparser.ConfigParser()
    config.read_dict({'augmentation': AUG})
    return {name: (ns[name](config) if name.startswith('Random') else ns[name]()) for name in CHAIN}


def run_chain(ops, rec, image, seed):
    """-> (cv2 output, restored output, draws, restored pixel count)."""
    random.seed(seed)
    rec.draws = []
    blurred = ops['RandomBlur'](image)
    kx, ky = int(rec.draws[0]), int(rec.draws[1])
    wrapped = (blurred != P.box_blur(image, kx, ky))
    assert not wrapped.any() or (kx * ky == 2 and (blurred[wrapped] == 0).all()), 'unexpected cv2.blur difference'
    restored = blurred.copy()
    restored[wrapped] = 255
    state = random.getstate()
    outs = []
    for start, per_pixel in ((blurred, False), (restored, True)):
        random.setstate(state)
        del rec.draws[2:]
        x = start
        for name in CHAIN[1:]:
            x = P.cv2_per_pixel(ops[name], x) if per_pixel and name == 'HSV2RGB' else ops[name](x)
        outs.append(x)
    return outs[0], outs[1], np.array(rec.draws), int(wrapped.sum())


def first_seed(start, k):
    """The first seed from `start` up whose blur draw (randint(1, 5), randint(1, 5)) is k."""
    sd = start
    while True:
        random.seed(sd)
        if (random.randint(1, 5), random.randint(1, 5)) == k:
            return sd
        sd += 1


def main():
    rec = Recorder()
    ops = load_classes(rec)
    out = {}
    out['bgr2hsv_all_sha'] = sha(cv2.cvtColor(P.all_colours_frame(), cv2.COLOR_BGR2HSV))
    out['hsv2rgb_all_sha'] = sha(P.cv2_per_pixel(lambda x: cv2.cvtColor(x, cv2.COLOR_HSV2RGB), P.hsv_triples_frame()))
    # batches: 8 images each at 416 x 416 and 320 x 608; each holds both area-2 blur draws, (1, 2) and (2, 1)
    for name, (h, w) in (('b416', (416, 416)), ('b320x608', (320, 608))):
        base = 1000 if name == 'b416' else 2000
        seeds = [first_seed(base, k) for k in ((1, 2), (2, 1))]
        seeds += [sd for sd in range(base, base + 8) if sd not in seeds][:6]
        frames = np.stack([O.synth_frame(sd, h, w) for sd in seeds])
        res = [run_chain(ops, rec, f, sd) for f, sd in zip(frames, seeds)]
        out[name + '_seeds'] = np.array(seeds)
        out[name + '_frame_sha'] = np.stack([sha(f) for f in frames])
        out[name + '_draws'] = np.stack([r[2] for r in res])
        out[name + '_sha_cv2'] = np.stack([sha(r[0]) for r in res])
        out[name + '_sha'] = np.stack([sha(r[1]) for r in res])
        out[name + '_restored'] = np.array([r[3] for r in res])
        print(name, 'blur draws', [tuple(map(int, r[2][:2])) for r in res], 'restored', [r[3] for r in res])
    # small frames, stored in full: all-white 9 x 7 (every area-2 window wraps in cv2), 1 x 5, 5 x 1, 2 x 2, 37 x 53
    small = [np.full((9, 7, 3), 255, np.uint8), O.synth_frame(61, 1, 5), O.synth_frame(62, 5, 1), O.synth_frame(63, 2, 2),
             O.synth_frame(64, 37, 53)]
    seeds = [3000, 3001, 3002, 3003, 3004]
    seeds[0] = first_seed(seeds[0], (1, 2))           # the white frame gets an area-2 blur
    for i, (f, sd) in enumerate(zip(small, seeds)):
        a, b, d, n = run_chain(ops, rec, f, sd)
        out['s%d_src' % i], out['s%d_seed' % i], out['s%d_draws' % i] = f, np.array(sd), d
        out['s%d_out_cv2' % i], out['s%d_out' % i], out['s%d_restored' % i] = a, b, np.array(n)
        print('small', f.shape, 'draws', d, 'restored', n)
    out['small_count'] = np.array(len(small))
    # each class alone on one frame (its own seed); the HSV stages take cv2's HSV of the frame
    frame = O.synth_frame(70, 37, 53)
    hsv = cv2.cvtColor(frame, cv2.COLOR_BGR2HSV)
    out['cls_src'], out['cls_src_hsv'] = frame, hsv
    for j, name in enumerate(CHAIN):
        src = hsv if name in ('RandomHue', 'RandomSaturation', 'RandomBrightness', 'HSV2RGB') else frame
        random.seed(4000 + j)
        rec.draws = []
        out['cls_%s' % name] = P.cv2_per_pixel(ops[name], src) if name == 'HSV2RGB' else ops[name](src)
        out['cls_%s_seed' % name] = np.array(4000 + j)
        out['cls_%s_draws' % name] = np.array(rec.draws)
    path = os.path.join(HERE, 'photometric.npz')
    np.savez_compressed(path, **out)
    print('photometric.npz %.1f KB' % (os.path.getsize(path) / 1024))


if __name__ == '__main__':
    main()
