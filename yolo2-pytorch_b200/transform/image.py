"""transform.image -- the reference's transform/image.py:27-99 for uint8 HWC frames on the GPU.

`BGR2RGB` (:27-29): inside `transform.resize_batch` the swap is fused into the resize kernel; this stand-alone form is a strided
view (no copy).

The photometric augmentations (:32-99) -- `RandomBlur`, `BGR2HSV`, `RandomHue`, `RandomSaturation`, `RandomBrightness`, `HSV2RGB`,
`RandomGamma` -- take the reference's config keys (`augmentation/random_blur`, ...) and make the reference's `random` draws per call.
Each accepts a uint8 [h, w, 3] frame (numpy, CPU or CUDA tensor) or a uint8 [B, H, W, 3] CUDA batch (one draw per image) and returns
a CUDA tensor of the same shape from one `yb_photometric_u8` launch.  The kernel runs five stages in a fixed order -- box blur,
BGR->HSV, a per-channel HSV table, HSV->RGB, a per-channel output table -- so every random draw becomes host-built data: the blur's
(kx, ky), or a 256-entry table built with the reference's own numpy expression (hue, saturation, brightness on one channel each,
gamma on all three).  `apply_chain` runs a whole sequence: draws image by image in chain order (the reference's `Collate` order), and
each maximal run of ops that fits the stage order is one launch, tables on the same channel composed -- the reference's full
`image_train` chain is exactly one launch.

Pixels are cv2 4.13's 8-bit arithmetic bit for bit, with one intended difference: cv2.blur with an area-2 kernel, (1, 2) or (2, 1),
wraps a window of two 255s to 0 in its scalar tail loop; here it saturates to 255.  Gamma is restated from current scikit-image
(`adjust_gamma`'s uint8 table, `gamma_table`), which is not executed anywhere in this project."""
import random
import re

import numpy as np
import torch

from b200 import ops as _ops

STAGE_BLUR, STAGE_TO_HSV, STAGE_HSV_TABLE, STAGE_TO_RGB, STAGE_OUT_TABLE = range(5)
MAX_BLUR = 15


def _underscore(name):
    """inflection.underscore for the CamelCase class names here: 'RandomBlur' -> 'random_blur'."""
    return re.sub(r'(?<=[a-z0-9])([A-Z])', r'_\1', name).lower()


def hue_table(adjust):
    """RandomHue (:57-62): h -> clip(h.astype(int) + adjust, 0, 179), no wrap-around."""
    return np.clip(np.arange(256) + int(adjust), 0, 179).astype(np.uint8)


def scale_table(adjust):
    """RandomSaturation / RandomBrightness (:70-88): x -> clip(x * adjust, 0, 255).astype(uint8), a float64 product truncated."""
    return np.clip(np.arange(256, dtype=np.uint8) * float(adjust), 0, 255).astype(np.uint8)


def gamma_table(gamma, gain=1.0):
    """RandomGamma (:96-98): skimage.exposure.adjust_gamma(image, gamma) on uint8 is a lookup in this table (current scikit-image;
    the 2017 releases computed ((image / 255) ** gamma) * 255 in float64 and truncated)."""
    return np.minimum(np.rint(255 * gain * np.linspace(0, 1, 256) ** gamma), 255).astype(np.uint8)


class BGR2RGB(object):
    def __call__(self, image):
        return image.flip(-1)


class Photometric(object):
    """One stage of `yb_photometric_u8`.  `draw()` makes the reference's random draws for one image; `plan()` records them."""
    stage = None

    def draw(self):
        return None

    def plan(self, launch, i, param):
        raise NotImplementedError

    def __call__(self, image):
        return apply_chain([self], image)


class _Configured(Photometric):
    parse = float

    def __init__(self, config):
        self.adjust = tuple(map(self.parse, config.get('augmentation', _underscore(type(self).__name__)).split()))


class BGR2HSV(Photometric):
    stage = STAGE_TO_HSV

    def plan(self, launch, i, param):
        launch.to_hsv = True


class HSV2RGB(Photometric):
    stage = STAGE_TO_RGB

    def plan(self, launch, i, param):
        launch.to_rgb = True


class RandomBlur(_Configured):
    stage = STAGE_BLUR
    parse = int

    def __init__(self, config):
        _Configured.__init__(self, config)
        if len(self.adjust) != 2 or not all(1 <= a <= MAX_BLUR for a in self.adjust):
            raise ValueError('augmentation/random_blur must be two kernel sizes in 1..%d, got %r' % (MAX_BLUR, self.adjust))

    def draw(self):
        return tuple(random.randint(1, adjust) for adjust in self.adjust)

    def plan(self, launch, i, param):
        launch.blur_k()[i] = param


class _ChannelTable(_Configured):
    stage = STAGE_HSV_TABLE
    channel = None

    def table(self, param):
        return scale_table(param)

    def draw(self):
        return random.uniform(*self.adjust)

    def plan(self, launch, i, param):
        t = launch.lut_hsv()[i]
        t[self.channel] = self.table(param)[t[self.channel]]


class RandomHue(_ChannelTable):
    parse = int
    channel = 0

    def table(self, param):
        return hue_table(param)

    def draw(self):
        return random.randint(*self.adjust)


class RandomSaturation(_ChannelTable):
    channel = 1


class RandomBrightness(_ChannelTable):
    channel = 2


class RandomGamma(_Configured):
    stage = STAGE_OUT_TABLE

    def draw(self):
        return random.uniform(*self.adjust)

    def plan(self, launch, i, param):
        t = launch.lut_out()[i]
        t[:] = gamma_table(param)[t]


class Launch(object):
    """The arguments of one `yb_photometric_u8` launch for a batch of `batch` images."""

    def __init__(self, batch):
        self.batch = batch
        self.to_hsv = self.to_rgb = False
        self._blur = self._lut_hsv = self._lut_out = None

    def blur_k(self):
        if self._blur is None:
            self._blur = np.ones((self.batch, 2), np.int32)
        return self._blur

    def lut_hsv(self):
        if self._lut_hsv is None:
            self._lut_hsv = np.tile(np.arange(256, dtype=np.uint8), (self.batch, 3, 1))
        return self._lut_hsv

    def lut_out(self):
        if self._lut_out is None:
            self._lut_out = np.tile(np.arange(256, dtype=np.uint8), (self.batch, 3, 1))
        return self._lut_out

    def __call__(self, frames):
        """frames: uint8 CUDA [B, H, W, 3], contiguous -> a new tensor."""
        b, h, w, _ = frames.shape
        dev = frames.device
        if self._blur is not None and not ((self._blur >= 1) & (self._blur <= MAX_BLUR)).all():
            raise ValueError('blur kernel sizes must lie in 1..%d' % MAX_BLUR)

        def up(a):
            return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(dev, non_blocking=True)
        out = torch.empty_like(frames)
        _ops.call('yb_photometric_u8', frames, out, b, h, w, up(self._blur), int(self.to_hsv), up(self._lut_hsv), int(self.to_rgb),
                  up(self._lut_out))
        return out


def split_chain(ops):
    """ops -> list of launches (lists of ops): each maximal run whose stages ascend (equal table stages compose) is one launch."""
    groups, last = [], None
    for op in ops:
        if not isinstance(op, Photometric):
            raise TypeError('%r is not a photometric transform.image op (RandomBlur, BGR2HSV, RandomHue, RandomSaturation, '
                            'RandomBrightness, HSV2RGB, RandomGamma)' % (op,))
        s = op.stage
        if groups and (s > last or (s == last and s in (STAGE_HSV_TABLE, STAGE_OUT_TABLE))):
            groups[-1].append(op)
        else:
            groups.append([op])
        last = s
    return groups


def as_batch(image):
    """uint8 [h, w, 3] (numpy / CPU / CUDA) or CUDA [B, H, W, 3] -> (contiguous CUDA [B, H, W, 3], was_single)."""
    if not torch.is_tensor(image):
        image = torch.from_numpy(np.ascontiguousarray(image))
    if image.dtype != torch.uint8 or image.dim() not in (3, 4) or image.shape[-1] != 3:
        raise ValueError('expected a uint8 [h, w, 3] frame or a uint8 [B, H, W, 3] CUDA batch, got %s %s' % (image.dtype, tuple(image.shape)))
    if image.dim() == 4 and not image.is_cuda:
        raise ValueError('a [B, H, W, 3] batch must be a CUDA tensor')
    single = image.dim() == 3
    if not image.is_cuda:
        image = image.to(torch.device('cuda', torch.cuda.current_device()))
    image = image.contiguous()
    return (image[None] if single else image), single


def apply_chain(ops, image):
    """Apply the photometric ops in order to a frame or a batch.  Draws are made image by image, in chain order within an image."""
    groups = split_chain(ops)
    frames, single = as_batch(image)
    n = frames.shape[0]
    draws = [[op.draw() for op in ops] for _ in range(n)]
    k = 0
    for group in groups:
        launch = Launch(n)
        for j, op in enumerate(group):
            for i in range(n):
                op.plan(launch, i, draws[i][k + j])
        frames = launch(frames)
        k += len(group)
    return frames[0] if single else frames
