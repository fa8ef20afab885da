"""Held-out evaluation throughput on one GPU (not collected by pytest): c2 (2 M Gaussians, 1920x1080), 16 held-out views.

  fused      Trainer.evaluate(protocol="report") at batch_size 4 and 8: batched preprocess + render, one metrics launch per
             batch, one host read per call
  reference  train_internal.py:466-479 restated: per view a forward render through the per-camera operator, then torch
             clamp, fp32 L1 / PSNR (utils/image_utils.py) / SSIM (utils/loss_utils.py, five 11x11 depthwise convolutions)

Each arm is warmed up, then timed as the median of --repeats calls, each ending in a device synchronise.  Prints one JSON
line: views/s per arm, the largest per-view metric difference between the arms, the device name and its power limit.
Usage: python tests/eval_bench.py [--repeats 7]
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "grendel-gs_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from gs_b200 import ops, pipeline, synthetic as syn  # noqa: E402


def _window(dev):
    g = torch.tensor([math.exp(-((x - 5) ** 2) / float(2 * 1.5 ** 2)) for x in range(11)])
    g = g / g.sum()
    return (g[:, None] @ g[None, :]).float()[None, None].expand(3, 1, 11, 11).contiguous().to(dev)


def reference_arm(params, dcams, gts_dev, window):
    """-> (N,3) device tensor of (l1, psnr, ssim) per view, as training_report computes them (plus SSIM)."""
    out = []
    conv = lambda t: F.conv2d(t, window, padding=5, groups=3)
    with torch.no_grad():
        for dcam, gt in zip(dcams, gts_dev):
            rs = dcam.settings(params.active_sh_degree)
            m2, rgb, co, radii, depths = ops.preprocess_gaussians_raw(params._xyz, params._features_dc,
                                                                      params._features_rest, params._scaling,
                                                                      params._rotation, params._opacity, rs)
            image, *_ = ops.render_gaussians(m2, co, rgb, depths, radii, None, rs)
            image = torch.clamp(image, 0.0, 1.0)
            gt_image = torch.clamp(gt / 255.0, 0.0, 1.0)
            l1 = torch.abs(image - gt_image).mean().double()
            mse = ((image - gt_image) ** 2).view(3, -1).mean(1, keepdim=True)
            psnr = (20 * torch.log10(1.0 / torch.sqrt(mse))).mean().double()
            a, b = image[None], gt_image[None]
            mu1, mu2 = conv(a), conv(b)
            s1, s2, s12 = conv(a * a) - mu1.pow(2), conv(b * b) - mu2.pow(2), conv(a * b) - mu1 * mu2
            C1, C2 = 0.01 ** 2, 0.03 ** 2
            ssim = (((2 * mu1 * mu2 + C1) * (2 * s12 + C2)) /
                    ((mu1.pow(2) + mu2.pow(2) + C1) * (s1 + s2 + C2))).mean().double()
            out.append(torch.stack([l1, psnr, ssim]))
    return torch.stack(out)


def timed(fn, warmup, repeats):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), ts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--views", type=int, default=16)
    ap.add_argument("--n", type=int, default=2_000_000)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("eval_bench.py needs a CUDA device")
    dev = "cuda"
    W, H = 1920, 1080
    scene = syn.make_scene(args.n, W, H, seed=0)
    train_cams = syn.make_batch_cameras(W, H, 4)
    tgts = [torch.from_numpy(syn.make_gt_image(W, H, seed=1 + k)).pin_memory() for k in range(4)]
    tr = pipeline.Trainer(scene, train_cams, tgts, dev)
    cams = [syn.make_camera(W, H, yaw_deg=1.5 * k - 11.0, uid=1000 + k) for k in range(args.views)]
    dcams = [pipeline.DeviceCamera(c, dev) for c in cams]
    gts = [torch.from_numpy(syn.make_gt_image(W, H, seed=300 + k)) for k in range(args.views)]
    gts_dev = [g.to(dev) for g in gts]
    window = _window(dev)
    res = {"workload": "c2", "n_gaussians": args.n, "width": W, "height": H, "views": args.views,
           "repeats": args.repeats, "warmup": args.warmup}
    ref_out = {}
    med, ts = timed(lambda: ref_out.__setitem__("m", reference_arm(tr.params, dcams, gts_dev, window)), args.warmup,
                    args.repeats)
    res["reference_views_per_s"] = args.views / med
    res["reference_ms"] = [round(t * 1e3, 3) for t in ts]
    ref = ref_out["m"].cpu().numpy()
    worst = {"l1_rel": 0.0, "psnr_db": 0.0, "ssim": 0.0}
    for bs in (4, 8):
        out = {}
        med, ts = timed(lambda: out.__setitem__("r", tr.evaluate(dcams, gts_dev, batch_size=bs)), args.warmup,
                        args.repeats)
        res[f"fused_bs{bs}_views_per_s"] = args.views / med
        res[f"fused_bs{bs}_ms"] = [round(t * 1e3, 3) for t in ts]
        for v, r in zip(out["r"]["per_view"], ref):
            worst["l1_rel"] = max(worst["l1_rel"], abs(v["l1"] / r[0] - 1))
            worst["psnr_db"] = max(worst["psnr_db"], abs(v["psnr"] - r[1]))
            worst["ssim"] = max(worst["ssim"], abs(v["ssim"] - r[2]))
    res["max_metric_difference"] = worst
    # the metrics launch alone (gs_metrics_batched, report mode) on 8 full views: CUDA events over 20 launches
    imgs = torch.rand((8, 3, H, W), device=dev)
    rows4 = [(0, H, 0, H)] * 8
    for _ in range(3):
        ops.image_metrics_batched(imgs, gts_dev[:8], rows4)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        ops.image_metrics_batched(imgs, gts_dev[:8], rows4)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 20 / 8
    res["metrics_kernel_ms_per_view"] = ms
    res["metrics_kernel_hbm_GBps"] = 15 * H * W / (ms * 1e-3) / 1e9     # 12 B image + 3 B ground truth per pixel
    res["device"] = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        res["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        res["power_limit_and_max_sm_clock"] = f"unavailable ({e})"
    print(json.dumps(res))


if __name__ == "__main__":
    main()
