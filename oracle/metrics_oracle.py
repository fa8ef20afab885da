"""NumPy fp64 restatement of the held-out image metrics (oracle/METRICS_SPEC.md): the per-channel sums that
gs_metrics_batched produces, both input modes, and the two protocols' derivations.  Test infrastructure, not product.

  utils/image_utils.py:19-21   psnr: mse over view(C, -1), 20 log10(1 / sqrt(mse))
  utils/loss_utils.py:18-85    l1_loss, the 11x11 Gaussian window (sigma 1.5, fp32), _ssim with zero padding
  train_internal.py:466-479    training_report: clamp(image, 0, 1), gt / 255, l1_loss and psnr of the (3,H,W) image
  render.py:120-138            save_image of the clamped image (8-bit PNG)
  metrics.py:26-36             to_tensor of the PNG, ssim / psnr of the (1,3,H,W) tensors
"""
import math

import numpy as np

HALF = 5


def gaussian_window():
    """The 11 taps of create_window: exp() in Python doubles, stored and normalised in fp32; returned as float64."""
    g = np.array([math.exp(-((x - HALF) ** 2) / float(2 * 1.5 ** 2)) for x in range(2 * HALF + 1)], dtype=np.float32)
    return (g / g.sum(dtype=np.float32)).astype(np.float64)


def quantise_saved(x):
    """torchvision.utils.save_image's 8-bit values of a clamped fp32 image: mul(255).add_(0.5).clamp_(0, 255).to(uint8),
    each operation rounded to fp32 on its own."""
    x = np.asarray(x, dtype=np.float32)
    q = (x * np.float32(255.0)).astype(np.float32) + np.float32(0.5)
    return np.clip(q, np.float32(0.0), np.float32(255.0)).astype(np.uint8)


def metric_input(image, saved=False):
    """x of the metrics: clamp(image, 0, 1) in fp32; saved=True: the PNG round trip, quantised / 255 (to_tensor)."""
    x = np.clip(np.asarray(image, dtype=np.float32), np.float32(0.0), np.float32(1.0))
    if saved:
        x = quantise_saved(x).astype(np.float32) / np.float32(255.0)
    return x


def _filter(a, g):
    """Separable 11x11 window with zero padding over the last two axes (F.conv2d, padding 5)."""
    h, w = a.shape[-2:]
    p = np.zeros(a.shape[:-2] + (h + 2 * HALF, w + 2 * HALF))
    p[..., HALF:HALF + h, HALF:HALF + w] = a
    r = sum(g[t] * p[..., :, t:t + w] for t in range(2 * HALF + 1))
    return sum(g[t] * r[..., t:t + h, :] for t in range(2 * HALF + 1))


def ssim_map(x, y):
    """_ssim's per-pixel map of (C, h, w) images in fp64 (utils/loss_utils.py:52-85)."""
    g = gaussian_window()
    x, y = np.asarray(x, np.float64), np.asarray(y, np.float64)
    mu1, mu2 = _filter(x, g), _filter(y, g)
    s1 = _filter(x * x, g) - mu1 * mu1
    s2 = _filter(y * y, g) - mu2 * mu2
    s12 = _filter(x * y, g) - mu1 * mu2
    C1, C2 = 0.01 ** 2, 0.03 ** 2
    return ((2 * mu1 * mu2 + C1) * (2 * s12 + C2)) / ((mu1 * mu1 + mu2 * mu2 + C1) * (s1 + s2 + C2))


def metric_sums(image, gt_u8, saved=False, row0=0, row1=None, count_row0=None, count_row1=None):
    """(3,3) fp64 sums of one view, as gs_metrics_batched: [0][c] = sum |x-y|, [1][c] = sum (x-y)^2, [2][c] = sum ssim_map
    over channel c.  image (3,H,W) float (the full image); gt_u8 (3, row1-row0, W) uint8 of the window rows [row0, row1)
    (the window is zero-padded at its edges); only rows [count_row0, count_row1) are summed (default: the window)."""
    image = np.asarray(image)
    H = image.shape[1]
    row1 = H if row1 is None else row1
    c0 = row0 if count_row0 is None else count_row0
    c1 = row1 if count_row1 is None else count_row1
    x = metric_input(image[:, row0:row1], saved)
    y = np.asarray(gt_u8).astype(np.float32) / np.float32(255.0)
    d = (x - y).astype(np.float64)                   # the difference is formed in fp32, as torch does
    sl = slice(c0 - row0, c1 - row0)
    m = ssim_map(x, y)
    out = np.zeros((3, 3))
    out[0] = np.abs(d[:, sl]).sum(axis=(1, 2))
    out[1] = (d[:, sl] ** 2).sum(axis=(1, 2))
    out[2] = m[:, sl].sum(axis=(1, 2))
    return out


def derive(sums, image_height, image_width, protocol="report"):
    """(3,3) sums of one view -> {"l1", "psnr", "ssim"}.  report: mean over channels of per-channel PSNR (psnr() of a
    (3,H,W) tensor); saved: PSNR of the whole image (psnr() of a (1,3,H,W) tensor)."""
    s = np.asarray(sums, dtype=np.float64)
    hw = float(image_height) * float(image_width)
    with np.errstate(divide="ignore"):
        if protocol == "report":
            psnr = float(np.mean(20.0 * np.log10(1.0 / np.sqrt(s[1] / hw))))
        elif protocol == "saved":
            psnr = float(20.0 * np.log10(1.0 / np.sqrt(s[1].sum() / (3.0 * hw))))
        else:
            raise ValueError(protocol)
    return {"l1": float(s[0].sum() / (3 * hw)), "psnr": psnr, "ssim": float(s[2].sum() / (3 * hw))}
