"""Generates tests/golden/metrics.npz by IMPORTING the reference's own Python (run once against a reference checkout,
on a CPU with torchvision; no test reads the reference):
  utils/loss_utils.py:l1_loss, ssim        -> L1 and SSIM
  utils/image_utils.py:psnr                -> PSNR of a (3,H,W) image (per channel, then averaged, as
                                              train_internal.py:466-479 uses it) and of a (1,3,H,W) one (metrics.py)
  render.py:127-138 -> metrics.py:26-36    -> torchvision.utils.save_image to PNG, PIL + to_tensor back
Images are seeded, include values outside [0,1] and odd sizes.
Usage: python tests/golden/make_metrics_golden.py
"""
import importlib.util
import os
import tempfile

import numpy as np
import torch

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))
SIZES = [(37, 53), (67, 93), (16, 16)]


def load(path, name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(REF, path))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def make_pair(rng, H, W):
    """A smooth ground truth and a rendering of it with noise, an offset and values beyond [0,1]."""
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float64)
    base = np.stack([0.5 + 0.45 * np.sin(xx / (3 + c) + yy / (5 + c) + c) for c in range(3)])
    gt = np.clip(np.round(255 * (base + rng.normal(0, 0.03, base.shape))), 0, 255).astype(np.uint8)
    img = (base + rng.normal(0, 0.08, base.shape) + 0.02).astype(np.float32)
    img[:, :3, :5] = 1.3          # saturated block
    img[:, -2:, -4:] = -0.2       # negative block
    return img, gt


def main():
    import torchvision
    from PIL import Image
    import torchvision.transforms.functional as tf
    loss_utils = load("utils/loss_utils.py", "ref_loss_utils")
    image_utils = load("utils/image_utils.py", "ref_image_utils")
    rng = np.random.default_rng(2024)
    out = {"n": np.int64(len(SIZES))}
    with tempfile.TemporaryDirectory() as tmp:
        for i, (H, W) in enumerate(SIZES):
            img, gt = make_pair(rng, H, W)
            image = torch.clamp(torch.from_numpy(img), 0.0, 1.0)                 # train_internal.py:477-478
            gt_image = torch.clamp(torch.from_numpy(gt).float() / 255.0, 0.0, 1.0)
            out[f"image{i}"], out[f"gt{i}"] = img, gt
            # training_report
            out[f"report_l1_{i}"] = np.float64(loss_utils.l1_loss(image, gt_image).mean().double())
            out[f"report_psnr_{i}"] = np.float64(image_utils.psnr(image, gt_image).mean().double())
            out[f"report_ssim_{i}"] = np.float64(loss_utils.ssim(image, gt_image).double())
            # render.py -> PNG -> metrics.py
            pr, pg = os.path.join(tmp, f"r{i}.png"), os.path.join(tmp, f"g{i}.png")
            torchvision.utils.save_image(image, pr)
            torchvision.utils.save_image(gt_image, pg)
            render = tf.to_tensor(Image.open(pr)).unsqueeze(0)[:, :3, :, :]
            gtr = tf.to_tensor(Image.open(pg)).unsqueeze(0)[:, :3, :, :]
            out[f"saved_q{i}"] = np.asarray(Image.open(pr)).transpose(2, 0, 1).copy()   # (3,H,W) uint8 as written
            out[f"saved_gt_q{i}"] = np.asarray(Image.open(pg)).transpose(2, 0, 1).copy()
            out[f"saved_l1_{i}"] = np.float64(loss_utils.l1_loss(render, gtr).mean().double())
            out[f"saved_psnr_{i}"] = np.float64(image_utils.psnr(render, gtr).mean().double())
            out[f"saved_ssim_{i}"] = np.float64(loss_utils.ssim(render, gtr).double())
    np.savez_compressed(os.path.join(HERE, "metrics.npz"), **out)
    print("wrote", os.path.join(HERE, "metrics.npz"), {k: v for k, v in out.items() if np.ndim(v) == 0})


if __name__ == "__main__":
    main()
