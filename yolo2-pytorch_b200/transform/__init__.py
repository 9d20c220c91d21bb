"""transform -- the part of the reference's `transform/` package that sits immediately upstream of the network input
(SURVEY 8f rank 2), on the GPU: `transform.resize.image.rescale`, `transform.resize.label.rescale`,
`transform.image.BGR2RGB`, and the batched `transform.resize_batch` that does all three for a whole batch of decoded
frames in one launch -- optionally through the horizontal flip and the random-crop window of the reference's training pipeline
(`transform.augmentation.flip_horizontally`, `transform.resize.label.random_crop`), which are index transforms on the source of the same
resize; `transform.augmentation.random_rotate` / `Rotator` and `transform.resize.image.fixed` (shrinking) run cv2.warpAffine's bilinear path in
one kernel.  The photometric augmentations of `transform/image.py` (`RandomBlur`, `BGR2HSV`, `RandomHue`, `RandomSaturation`,
`RandomBrightness`, `HSV2RGB`, `RandomGamma`) run as one batched kernel (`transform.image.apply_chain`, yb_photometric_u8); `get_transform`
builds the reference's `image_train` chain from its config line, and `utils.data.Collate(..., transform_image=...)` applies it to the
resized batch."""
import inspect

import torch

from b200 import ops as _ops


def resize_batch(frames, height, width, bgr2rgb=True, yx_min=None, yx_max=None, flip=None, crop=None, margin=None):
    """frames: list of uint8 [h_i, w_i, 3] tensors (CPU or CUDA; BGR as cv2.imread gives them) -> uint8 CUDA tensor
    [B, height, width, 3], cv2.resize-exact, RGB when `bgr2rgb`.  Optional padded boxes yx_min / yx_max [B, G, 2] (source
    pixels) are returned scaled by (height / h_i, width / w_i) like transform.resize.label.rescale.  One kernel launch;
    the result can be fed straight to the model (`Darknet.forward` accepts uint8 NHWC frames).
    Training form: `flip` (B booleans: cv2.flip(frame, 1) first), `crop` ([B][4] ints (y0, x0, y1, x1): frame[y0:y1, x0:x1] next) and
    `margin` ([B][2] float32: what the reference subtracts from the boxes for that crop) -- see transform.resize.label.random_crop."""
    dev = torch.device('cuda', torch.cuda.current_device())
    sizes, offs, total = [], [], 0
    for f in frames:
        if f.dtype != torch.uint8 or f.dim() != 3 or f.shape[2] != 3:
            raise ValueError('frames must be uint8 [h, w, 3]')
        sizes += [int(f.shape[0]), int(f.shape[1])]
        offs.append(total)
        total += f.numel()
    packed = torch.empty(total, dtype=torch.uint8, device=dev)
    for f, o in zip(frames, offs):
        packed[o:o + f.numel()].copy_(f.reshape(-1), non_blocking=True)
    src_off = torch.tensor(offs, dtype=torch.int64).to(dev, non_blocking=True)
    src_hw = torch.tensor(sizes, dtype=torch.int32).to(dev, non_blocking=True)
    out = torch.empty(len(frames), height, width, 3, dtype=torch.uint8, device=dev)
    slots = 0
    if yx_min is not None:
        yx_min = yx_min.to(device=dev, dtype=torch.float32).contiguous().clone()
        yx_max = yx_max.to(device=dev, dtype=torch.float32).contiguous().clone()
        slots = yx_min.shape[1]
    if flip is None and crop is None:
        _ops.call('yb_resize_batch_u8', packed, src_off, src_hw, out, len(frames), int(height), int(width), int(bool(bgr2rgb)), yx_min, yx_max, slots)
        return (out, yx_min, yx_max) if yx_min is not None else out
    flip_t = crop_t = margin_t = None
    if flip is not None:
        flip_t = torch.tensor([int(bool(f)) for f in flip], dtype=torch.uint8).to(dev, non_blocking=True)
    if crop is not None:
        crop_t = torch.as_tensor(crop, dtype=torch.int32).reshape(len(frames), 4).to(dev, non_blocking=True)
        if margin is None:
            margin = [[c[0], c[1]] for c in crop_t.tolist()]
        margin_t = torch.as_tensor(margin, dtype=torch.float32).reshape(len(frames), 2).to(dev, non_blocking=True)
        for (y0, x0, y1, x1), (h, w) in zip(torch.as_tensor(crop).reshape(-1, 4).tolist(), zip(sizes[0::2], sizes[1::2])):
            if not (0 <= y0 < y1 <= h and 0 <= x0 < x1 <= w):
                raise ValueError('crop window (%d, %d, %d, %d) outside a %d x %d frame' % (y0, x0, y1, x1, h, w))
    _ops.call('yb_resize_aug_batch_u8', packed, src_off, src_hw, crop_t, margin_t, flip_t, out, len(frames), int(height), int(width), int(bool(bgr2rgb)),
              yx_min, yx_max, slots)
    return (out, yx_min, yx_max) if yx_min is not None else out


def to_tensor(frames_u8):
    """uint8 CUDA tensor [B, H, W, 3] -> float32 [B, 3, H, W] in [0, 1] (torchvision ToTensor, one kernel).  The training
    forward needs this form; inference takes the uint8 batch directly."""
    if not (isinstance(frames_u8, torch.Tensor) and frames_u8.is_cuda and frames_u8.dtype == torch.uint8 and frames_u8.dim() == 4 and frames_u8.shape[3] == 3):
        raise RuntimeError('transform.to_tensor (B200): expected a uint8 CUDA tensor [B, H, W, 3]')
    frames_u8 = frames_u8.contiguous()
    b, h, w, _ = frames_u8.shape
    out = torch.empty(b, 3, h, w, dtype=torch.float32, device=frames_u8.device)
    _ops.call('yb_totensor_u8', frames_u8, out, b, h, w)
    return out


class Compose(object):
    """torchvision.transforms.Compose: apply `transforms` in order.  A chain made only of photometric `transform.image` ops runs
    through `transform.image.apply_chain` (the reference's draw order, one launch per run of ascending kernel stages)."""

    def __init__(self, transforms):
        self.transforms = list(transforms)

    def __call__(self, image):
        from transform import image as _image
        if self.transforms and all(isinstance(t, _image.Photometric) for t in self.transforms):
            return _image.apply_chain(self.transforms, image)
        for t in self.transforms:
            image = t(image)
        return image


def parse_transform(config, method):
    """A dotted name -> `cls(config)` when the constructor takes one argument, `cls()` otherwise (reference transform/__init__.py:25-34);
    anything else is returned as is."""
    if isinstance(method, str):
        import utils
        attr = utils.parse_attr(method)
        if len(inspect.signature(attr).parameters) == 1:
            return attr(config)
        return attr()
    return method


def get_transform(config, sequence, compose=Compose):
    """e.g. get_transform(config, config.get('transform', 'image_train').split()) (reference transform/__init__.py:37-38)."""
    return compose([parse_transform(config, method) for method in sequence])
