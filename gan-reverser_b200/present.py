"""Result presentation of apply_r.lua (SURVEY.md section 8f, rank 2): colour-space lifting, borders,
`image.toDisplayTensor` grids and the JPEG files the reference writes.  Pure host-side data movement
on the outputs of the library; nothing here touches the GPU.

Mirrors, with the reference's names and argument meaning:
  NN_UTILS.toRgb / toRgbSingle                         utils/nn_utils.lua:146-189 ("y" and "rgb" only)
  image.toDisplayTensor{input, nrow, padding, min, max} and image.save   [upstream torch/image, not vendored]
  the four writers of apply_r.lua: cluster grids :245-259, search grids :284-298,
  fixed pairs / fixed images :325-351, anomalies :375-389.

[upstream] behaviour restated here (PARITY UNPINNED: torch/image cannot run in this image):
  * toDisplayTensor lays N x C x H x W out on a grid of xmaps = min(nrow, N) columns and
    ceil(N / xmaps) rows of (H + padding) x (W + padding) cells, each image offset by padding/2,
    cells without an image filled with the input's maximum, then min/max-normalises with saturation:
    (x - min) / (max - min) clamped to [0, 1].
  * image.save scales [0, 1] to bytes (x * 255, clamped) and writes a JPEG of quality 75.
JPEG bytes depend on the encoder, so tests pin the float grids and the decoded size, not file bytes.
"""
import math
import os

import numpy as np


def toRgb(images, colorSpace):
    """NN_UTILS.toRgb (nn_utils.lua:146-167): N x C x H x W -> N x 3 x H x W."""
    images = np.asarray(images, np.float32)
    if images.ndim == 3:
        images = images[None]
    if colorSpace == "rgb":
        return images
    if colorSpace == "y":
        return np.tile(images, (1, 3, 1, 1))                 # torch.repeatTensor(images, 1, 3, 1, 1)
    if colorSpace == "hsl":
        return np.stack([hsl2rgb(im) for im in images]) if len(images) else images
    if colorSpace == "yuv":
        return np.stack([yuv2rgb(im) for im in images]) if len(images) else images
    raise ValueError(f"Unknown color space <from>: '{colorSpace}'")   # nn_utils.lua:165


def hsl2rgb(image):
    """image.hsl2rgb [upstream torch/image, not vendored: restated from its published algorithm -- the CSS3 / "hue2rgb"
    conversion with h, s, l in [0, 1]; s == 0 gives grey]: 3 x H x W -> 3 x H x W."""
    h, s, l = (np.asarray(image[c], np.float32) for c in range(3))
    q = np.where(l < 0.5, l * (1.0 + s), l + s - l * s)
    p = 2.0 * l - q

    def hue2rgb(t):
        t = np.where(t < 0.0, t + 1.0, t)
        t = np.where(t > 1.0, t - 1.0, t)
        return np.where(t < 1.0 / 6.0, p + (q - p) * 6.0 * t,
                        np.where(t < 0.5, q, np.where(t < 2.0 / 3.0, p + (q - p) * (2.0 / 3.0 - t) * 6.0, p)))

    rgb = np.stack([hue2rgb(h + 1.0 / 3.0), hue2rgb(h), hue2rgb(h - 1.0 / 3.0)])
    return np.where(s[None] == 0.0, np.stack([l, l, l]), rgb).astype(np.float32)


def yuv2rgb(image):
    """image.yuv2rgb [upstream torch/image, not vendored: restated from its published coefficients, the inverse of
    y = 0.299 r + 0.587 g + 0.114 b, u = -0.14713 r - 0.28886 g + 0.436 b, v = 0.615 r - 0.51499 g - 0.10001 b]."""
    y, u, v = (np.asarray(image[c], np.float32) for c in range(3))
    return np.stack([y + 1.13983 * v, y - 0.39465 * u - 0.58060 * v, y + 2.03211 * u]).astype(np.float32)


def toRgbSingle(image, colorSpace):
    """NN_UTILS.toRgbSingle (nn_utils.lua:169-189): C x H x W -> 3 x H x W."""
    return toRgb(np.asarray(image, np.float32)[None], colorSpace)[0]


def toDisplayTensor(input, nrow=6, padding=0, min=None, max=None, saturate=True):
    """image.toDisplayTensor for a batch of 1- or 3-channel images [upstream torch/image]."""
    x = np.asarray(input, np.float32)
    if x.ndim == 3:
        x = x[None]
    n, c, h, w = x.shape
    xmaps = builtins_min(nrow, n)
    ymaps = int(math.ceil(n / xmaps))
    height, width = h + padding, w + padding
    grid = np.full((c, height * ymaps, width * xmaps), x.max() if n else 0.0, np.float32)
    k = 0
    for y in range(ymaps):
        for xx in range(xmaps):
            if k >= n:
                break
            y0, x0 = y * height + padding // 2, xx * width + padding // 2
            grid[:, y0:y0 + h, x0:x0 + w] = x[k]
            k += 1
    lo = float(grid.min()) if min is None else float(min)
    grid = grid - lo
    span = float(grid.max()) if max is None else float(max) - lo
    if span != 0.0:
        grid = grid / span
    if saturate:
        grid = np.clip(grid, 0.0, 1.0)
    return grid.astype(np.float32)


builtins_min = min   # `min` / `max` are keyword names of toDisplayTensor, as in the Lua call sites


def to_bytes(tensor):
    """C x H x W floats in [0, 1] -> H x W x C uint8, the conversion image.save applies before encoding."""
    t = np.clip(np.asarray(tensor, np.float32) * 255.0, 0.0, 255.0)
    return np.ascontiguousarray(np.moveaxis(t, 0, -1).astype(np.uint8))


def save(path, tensor, quality=75):
    """image.save(path, tensor): JPEG (or whatever the extension says) through Pillow; fails loudly without it."""
    from PIL import Image   # imported here: only the file writers need it
    arr = to_bytes(tensor)
    img = Image.fromarray(arr[:, :, 0], "L") if arr.shape[2] == 1 else Image.fromarray(arr, "RGB")
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    img.save(path, quality=quality)
    return path


# ---------------------------------------------------------------------------------------------
# the four artefacts of apply_r.lua
# ---------------------------------------------------------------------------------------------
def clusterGrid(average_face, member_images, colorSpace):
    """apply_r.lua:247-257: the cluster's mean face followed by its members, nrow = ceil(sqrt(1 + #members))."""
    tnsr = np.concatenate([np.asarray(average_face, np.float32)[None], np.asarray(member_images, np.float32)], axis=0)
    tnsr = toRgb(tnsr, colorSpace)
    return toDisplayTensor(tnsr, nrow=int(math.ceil(math.sqrt(tnsr.shape[0]))), min=0, max=1.0)


def saveClusterImages(result, images, colorSpace, writeTo, filenamePattern="cluster_%02d.jpg"):
    """Writes one grid per non-empty cluster from createClusterImages' result (apply_r.lua:245-259)."""
    paths_out = []
    images = np.asarray(images, np.float32)
    for i in range(result["member_ids"].shape[0]):
        cnt = int(result["member_counts"][i])
        if cnt > 0:
            ids = result["member_ids"][i, :cnt]
            grid = clusterGrid(result["average_faces"][i], images[ids], colorSpace)
            paths_out.append(save(os.path.join(writeTo, filenamePattern % (i + 1)), grid))
    return paths_out


def searchGrid(found_images, colorSpace):
    """apply_r.lua:284-298: the n most similar faces (the needle itself first) with a blue 1-pixel border on image 1."""
    tnsr = toRgb(found_images, colorSpace).copy()
    first = tnsr[0]
    for ch, val in ((2, 1.0), (0, 0.0), (1, 0.0)):           # blue channel to 1, red and green to 0, on the frame
        first[ch, :, 0] = val; first[ch, :, -1] = val; first[ch, 0, :] = val; first[ch, -1, :] = val
    return toDisplayTensor(tnsr, nrow=int(math.ceil(math.sqrt(tnsr.shape[0]))), min=0, max=1.0)


def saveSimilaritySearchImages(result, images, colorSpace, writeTo):
    """Writes similar_<measure>_<needle>.jpg for createSimilaritySearchImages' result (apply_r.lua:300-317)."""
    images = np.asarray(images, np.float32)
    out = []
    for measure, pattern in (("attributes", "similar_attributes_%02d.jpg"), ("pixelwise", "similar_pixelwise_%02d.jpg")):
        ids, _ = result[measure]
        for i in range(ids.shape[0]):
            row = ids[i][ids[i] >= 0]
            out.append(save(os.path.join(writeTo, pattern % (i + 1)), searchGrid(images[row], colorSpace)))
    return out


def fixedPairsGrid(images, fixed, colorSpace):
    """apply_r.lua:325-345: N pairs (original | fixed) on a blue background with 1-pixel borders, 4 per row."""
    images, fixed = np.asarray(images, np.float32), np.asarray(fixed, np.float32)
    n, _, h, w = images.shape
    pairs = np.zeros((n, 3, 1 + h + 1, 1 + 2 * w + 1), np.float32)
    pairs[:, 2] = 1.0
    pairs[:, :, 1:1 + h, 1:1 + w] = toRgb(images, colorSpace)
    pairs[:, :, 1:1 + h, 1 + w:1 + 2 * w] = toRgb(fixed, colorSpace)
    return toDisplayTensor(pairs, nrow=4, min=0, max=1.0)


def completionGrid(columns, colorSpace, perRow=4):
    """New work (face completion, apply_r.completeFaces): one strip per face with the images of `columns` (a list of N x C x H x W
    arrays, e.g. damaged input | G(R_fixer(x, m)) | G(z_refined) | composite | original) side by side, on a blue background with
    1-pixel borders as in fixedPairsGrid, perRow strips per row."""
    cols = [toRgb(np.asarray(c, np.float32), colorSpace) for c in columns]
    n, _, h, w = cols[0].shape
    k = len(cols)
    strips = np.zeros((n, 3, 1 + h + 1, 1 + k * w + 1), np.float32)
    strips[:, 2] = 1.0
    for j, c in enumerate(cols):
        strips[:, :, 1:1 + h, 1 + j * w:1 + (j + 1) * w] = c
    return toDisplayTensor(strips, nrow=perRow, min=0, max=1.0)


def saveFixedFaces(result, colorSpace, writeTo):
    """fixed_pairs.jpg, fixed_images_<N>_unfixed.jpg, fixed_images_<N>.jpg from fixFaces' result (apply_r.lua:344-351)."""
    orig, fixed_pairs = result["pairs"]
    n = result["unfixed"].shape[0]
    nrow = int(math.floor(math.sqrt(n)))
    return [
        save(os.path.join(writeTo, "fixed_pairs.jpg"), fixedPairsGrid(orig, fixed_pairs, colorSpace)),
        save(os.path.join(writeTo, "fixed_images_%d_unfixed.jpg" % n), toDisplayTensor(result["unfixed"], nrow=nrow, min=0, max=1.0)),
        save(os.path.join(writeTo, "fixed_images_%d.jpg" % n), toDisplayTensor(result["fixed"], nrow=nrow, min=0, max=1.0)),
    ]


def anomalyGrid(images, flags, colorSpace):
    """apply_r.lua:375-388: each face inside a 1-pixel frame that is red where flagged, floor(sqrt(N)) per row."""
    images = np.asarray(images, np.float32)
    n, _, h, w = images.shape
    out = np.zeros((n, 3, 1 + h + 1, 1 + w + 1), np.float32)
    out[np.asarray(flags, bool), 0] = 1.0
    out[:, :, 1:1 + h, 1:1 + w] = toRgb(images, colorSpace)
    return toDisplayTensor(out, nrow=int(math.floor(math.sqrt(n))), min=0, max=1.0)


def saveAnomalies(images, flags, colorSpace, writeTo):
    n = len(flags)
    return save(os.path.join(writeTo, "anomalies.jpg"), anomalyGrid(np.asarray(images)[:n], flags, colorSpace))
