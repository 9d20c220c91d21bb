"""utils.data -- the batch-forming step of the reference's loader (utils/data.py:28-41,88-141), with the per-image CPU
work moved to the GPU: `padding_labels` (same function), the multi-scale `SizeSchedule` (`Collate.next_size`,
:135-141) and `Collate`, which turns a list of decoded samples into one batch -- size choice, label padding and ONE
kernel launch for resize + BGR->RGB + box scaling (`transform.resize_batch`) instead of a cv2 call per image inside
DataLoader workers.  `load_sizes` mirrors utils/train.py:129-131.

Multi-GPU note (SURVEY 8e / appendix B.12): in the reference every DataLoader worker keeps its own `next_size` state, so
consecutive batches can differ in size even inside a `maintain` window.  Here one SizeSchedule per process draws from a
`random.Random(seed)`: give every rank the same seed and all ranks step through the same sizes (no stragglers)."""
import random

import numpy as np
import torch


def padding_labels(data, dim, labels='yx_min, yx_max, cls, difficult'.split(', ')):
    """Zero-pad every label array of one sample to `dim` rows (reference utils/data.py:28-41)."""
    pad = dim - len(data[labels[0]])
    for key in labels:
        if key in data:
            label = np.asarray(data[key])
            data[key] = np.pad(label, [(0, pad)] + [(0, 0)] * (label.ndim - 1), 'constant')
    return data


def load_sizes(config):
    """`data/sizes` = "320,320 352,352 ..." -> [(height, width), ...] (reference utils/train.py:129-131)."""
    return [tuple(int(v) for v in s.split(',')) for s in config.get('data', 'sizes').split()]


class SizeSchedule(object):
    """`Collate.next_size` of the reference (utils/data.py:135-141): a size is drawn with random.choice and then kept
    for `maintain` further batches.  `seed` makes the sequence reproducible and identical across ranks."""

    def __init__(self, sizes, maintain=1, seed=None):
        assert maintain > 0 and len(sizes) > 0
        self.sizes = [tuple(s) for s in sizes]
        self.maintain = maintain
        self._maintain = maintain
        self.rng = random.Random(seed) if seed is not None else random
        self.size = None

    def next_size(self):
        if self._maintain < self.maintain:
            self._maintain += 1
        else:
            self.size = self.rng.choice(self.sizes)
            self._maintain = 0
        return self.size


class Collate(object):
    """samples (dicts with `image` uint8 [h, w, 3] BGR as cv2.imread gives it, `yx_min`/`yx_max` float32 [n, 2] in source
    pixels, `cls` int [n], optional `difficult`) -> one batch dict on the GPU:
        tensor   uint8 [B, H, W, 3] RGB at the scheduled size (feed it to the model as is: ToTensor's 1/255 is fused
                 into the first conv kernel)
        yx_min / yx_max float32 [B, G, 2] in pixels of the resized image, zero-padded (train.norm_data scales to grid units)
        cls int64 [B, G], difficult uint8 [B, G], size int64 [B, 2] (original sizes), height, width
    The reference's `resize` config choice maps to `rescale` (the default, transform/resize/label.py:25-31).
    `transform_image` is the reference's keyword (utils/data.py:94,121), typically
    `transform.get_transform(config, config.get('transform', 'image_train').split())`.  None or exactly [BGR2RGB] keeps the swap fused
    into the resize.  Otherwise the resize runs without the swap (`image_train` replaces BGR2RGB, as in the reference) and the chain
    -- photometric `transform.image` ops -- runs on the whole batch: draws image by image in chain order, as the reference's loop
    makes them, and one launch per run of ops that fits the kernel's stage order (the full reference chain is one launch)."""

    def __init__(self, sizes, maintain=1, seed=None, bgr2rgb=True, transform_image=None):
        self.schedule = SizeSchedule(sizes, maintain, seed)
        self.bgr2rgb = bgr2rgb
        self.chain = None
        if transform_image is not None:
            from transform import image as _image
            if isinstance(transform_image, _image.Photometric):
                chain = [transform_image]
            else:
                chain = list(getattr(transform_image, 'transforms', transform_image))
            if not (len(chain) == 1 and isinstance(chain[0], _image.BGR2RGB)):
                _image.split_chain(chain)          # TypeError for anything but photometric ops
                self.bgr2rgb = False
                self.chain = chain

    def __call__(self, batch):
        import transform.image
        height, width = self.schedule.next_size()
        dim = max(max(len(d['cls']) for d in batch), 1)
        frames, rows = [], []
        for d in batch:
            d = dict(d)
            img = d['image']
            frames.append(img if torch.is_tensor(img) else torch.from_numpy(np.ascontiguousarray(img)))
            d['size'] = np.array(frames[-1].shape[:2])
            if 'difficult' not in d:
                d['difficult'] = np.zeros(len(d['cls']), np.uint8)
            for k in ('yx_min', 'yx_max'):
                d[k] = np.asarray(d[k], np.float32).reshape(-1, 2)
            rows.append(padding_labels(d, dim))
        yx_min = torch.from_numpy(np.stack([r['yx_min'] for r in rows]).astype(np.float32))
        yx_max = torch.from_numpy(np.stack([r['yx_max'] for r in rows]).astype(np.float32))
        tensor, yx_min, yx_max = transform.resize_batch(frames, height, width, bgr2rgb=self.bgr2rgb, yx_min=yx_min, yx_max=yx_max)
        if self.chain is not None:
            tensor = transform.image.apply_chain(self.chain, tensor)
        dev = tensor.device
        return dict(tensor=tensor, yx_min=yx_min, yx_max=yx_max,
                    cls=torch.from_numpy(np.stack([np.asarray(r['cls']) for r in rows]).astype(np.int64)).to(dev),
                    difficult=torch.from_numpy(np.stack([np.asarray(r['difficult']) for r in rows]).astype(np.uint8)).to(dev),
                    size=torch.from_numpy(np.stack([r['size'] for r in rows]).astype(np.int64)), height=height, width=width)
