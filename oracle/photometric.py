"""numpy restatement of the reference's photometric training augmentations (transform/image.py:32-99) and of the cv2 8-bit
arithmetic under them -- test infrastructure only, the checker of `yb_photometric_u8`.

    box_blur      cv2.blur(img, (kx, ky)), BORDER_REFLECT_101, anchor (kx // 2, ky // 2): out = (S + a // 2) // a for a window
                  area a that is not a power of two, (S + a // 2 + 1) // a for a = 2, 4, 8, 16 (cv2's fixed-point divide rounds
                  exact ties up there), saturated to 255.  cv2 wraps an area-2 sum of 510 to 0 in its scalar tail loop; this
                  restatement (like the kernel) gives 255.
    bgr2hsv       cv2 COLOR_BGR2HSV, 8-bit: integer arithmetic with cv2's 12-bit reciprocal tables, H in 0..179.
    hsv2rgb       cv2 COLOR_HSV2RGB, 8-bit, as cv2 4.13's per-pixel path computes it: float32, s and v scaled by 1/255, h by
                  6/180, the sector table with the two `1 - s * f` terms as fused multiply-adds, then rint(x * 255).  cv2's
                  vectorised body truncates x * 255 instead, so its result depends on where a pixel falls in its row; the
                  rounding path is the one restated here (and in the kernel).
    *_table       the per-image 256-entry maps of RandomHue / RandomSaturation / RandomBrightness / RandomGamma."""
import numpy as np

F32 = np.float32


def reflect101(p, n):
    """cv2.borderInterpolate(p, n, BORDER_REFLECT_101) for an int array p."""
    p = np.asarray(p, np.int64).copy()
    if n == 1:
        return np.zeros_like(p)
    while True:
        lo, hi = p < 0, p >= n
        if not (lo.any() or hi.any()):
            return p
        p[lo] = -p[lo]
        p[hi] = 2 * n - 2 - p[hi]


def box_blur(img, kx, ky):
    """uint8 [h, w, 3] -> cv2.blur(img, (kx, ky)) with the area-2 saturation described above."""
    h, w = img.shape[:2]
    rows = reflect101(np.arange(h)[:, None] - ky // 2 + np.arange(ky)[None, :], h)     # [h, ky]
    cols = reflect101(np.arange(w)[:, None] - kx // 2 + np.arange(kx)[None, :], w)     # [w, kx]
    x = img.astype(np.int64)
    v = x[rows].sum(1)                       # [h, w, 3] vertical window sums
    s = v[:, cols].sum(2)                    # [h, w, 3]
    a = kx * ky
    bump = 1 if a in (2, 4, 8, 16) else 0
    return np.minimum((s + a // 2 + bump) // a, 255).astype(np.uint8)


def hsv_div_tables():
    i = np.maximum(np.arange(256, dtype=np.float64), 1.0)
    sdiv = np.rint((255 << 12) / i).astype(np.int64)
    hdiv = np.rint((180 << 12) / (6.0 * i)).astype(np.int64)
    sdiv[0] = hdiv[0] = 0
    return sdiv, hdiv


def bgr2hsv(img):
    sdiv, hdiv = hsv_div_tables()
    b, g, r = [img[..., c].astype(np.int64) for c in range(3)]
    v = np.maximum(np.maximum(b, g), r)
    diff = v - np.minimum(np.minimum(b, g), r)
    s = (diff * sdiv[v] + (1 << 11)) >> 12
    h = np.where(v == r, g - b, np.where(v == g, b - r + 2 * diff, r - g + 4 * diff))
    h = (h * hdiv[diff] + (1 << 11)) >> 12
    h = np.where(h < 0, h + 180, h)
    return np.stack([h, s, v], -1).astype(np.uint8)


def _fma(a, b, c):
    # a * b is exact in float64 for float32 operands; the sum is rounded once to float64, then to float32
    return (a.astype(np.float64) * b.astype(np.float64) + c).astype(F32)


def hsv2rgb(img):
    """uint8 [..., 3] HSV (H in 0..179) -> uint8 RGB."""
    flat = img.reshape(-1, 3)
    h = flat[:, 0].astype(F32) * (F32(6) / F32(180))
    s = flat[:, 1].astype(F32) * (F32(1) / F32(255))
    v = flat[:, 2].astype(F32) * (F32(1) / F32(255))
    sector = np.trunc(h)
    f = h - sector
    one = F32(1)
    tab = np.stack([v, v * (one - s), v * _fma(-s, f, 1.0), v * _fma(-s, one - f, 1.0)], -1)
    sector_data = np.array([[1, 3, 0], [1, 0, 2], [3, 0, 1], [0, 2, 1], [0, 1, 3], [2, 1, 0]])
    sec = sector.astype(np.int64)
    sec[(sec < 0) | (sec >= 6)] = 0
    bgr = np.take_along_axis(tab, sector_data[sec], 1)
    rgb = np.rint(bgr[:, ::-1] * F32(255))
    return np.clip(rgb, 0, 255).astype(np.uint8).reshape(img.shape)


def hue_table(adjust):
    """RandomHue: clip(h.astype(int) + adjust, 0, 179), no wrap-around."""
    return np.clip(np.arange(256) + int(adjust), 0, 179).astype(np.uint8)


def scale_table(adjust):
    """RandomSaturation / RandomBrightness: clip(x * adjust, 0, 255).astype(uint8) (float64 product, truncation)."""
    return np.clip(np.arange(256, dtype=np.uint8) * float(adjust), 0, 255).astype(np.uint8)


def gamma_table(gamma, gain=1.0):
    """RandomGamma: skimage.exposure.adjust_gamma's uint8 table, restated (current scikit-image form)."""
    return np.minimum(np.rint(255 * gain * np.linspace(0, 1, 256) ** gamma), 255).astype(np.uint8)


def apply_tables(img, tables):
    """tables: [3][256] uint8, one per channel."""
    return np.stack([tables[c][img[..., c]] for c in range(3)], -1)


def chain(img, blur=None, hue=None, saturation=None, brightness=None, gamma=None):
    """The reference's full `image_train` chain with given draws: RandomBlur, BGR2HSV, RandomHue, RandomSaturation,
    RandomBrightness, HSV2RGB, RandomGamma (a stage whose draw is None is left out, except the two conversions)."""
    if blur is not None:
        img = box_blur(img, *blur)
    hsv = bgr2hsv(img)
    ident = np.arange(256, dtype=np.uint8)
    hsv = apply_tables(hsv, [hue_table(hue) if hue is not None else ident,
                             scale_table(saturation) if saturation is not None else ident,
                             scale_table(brightness) if brightness is not None else ident])
    rgb = hsv2rgb(hsv)
    if gamma is not None:
        rgb = apply_tables(rgb, [gamma_table(gamma)] * 3)
    return rgb


def cv2_per_pixel(convert, img):
    """Run a cv2 colour conversion through its per-pixel path: as a one-pixel-wide frame no vectorised body applies."""
    return convert(np.ascontiguousarray(img).reshape(-1, 1, 3)).reshape(img.shape)


def all_colours_frame():
    """4096 x 4096 BGR frame holding every 24-bit colour once (b fastest)."""
    i = np.arange(1 << 24, dtype=np.uint32)
    return np.stack([i & 255, (i >> 8) & 255, i >> 16], -1).astype(np.uint8).reshape(4096, 4096, 3)


def hsv_triples_frame():
    """2880 x 4096 HSV frame holding every valid 8-bit triple (h < 180) once (v fastest)."""
    i = np.arange(180 * 65536, dtype=np.uint32)
    return np.stack([i >> 16, (i >> 8) & 255, i & 255], -1).astype(np.uint8).reshape(2880, 4096, 3)
