"""-m gpu: held-out evaluation on the device.  gs_metrics_batched against the golden data of the reference's own metrics
and the fp64 oracle, strip windows with halos, Trainer.evaluate against the reference protocol restated in torch,
absence of side effects on training, convergence of a student towards a teacher on held-out views, rejections, and the
multi-GPU harness tests/mgpu_eval.py (2 and 4 GPUs, skipped below)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from gs_b200 import ops, pipeline, synthetic as syn
from oracle import metrics_oracle as mo

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "metrics.npz")


def _metrics(img, gt, saved, rows4=None):
    H = img.shape[1]
    rows4 = rows4 or [(0, H, 0, H)]
    gts = [torch.from_numpy(np.ascontiguousarray(gt[:, r[0]:r[1]])).cuda() for r in rows4]
    imgs = torch.from_numpy(img).cuda().unsqueeze(0).expand(len(rows4), -1, -1, -1).contiguous()
    return ops.image_metrics_batched(imgs, gts, rows4, saved=saved).cpu().numpy()


def _check_sums(got, ref, HW):
    np.testing.assert_allclose(got[:2], ref[:2], rtol=1e-6, atol=0)
    assert np.abs(got[2] - ref[2]).max() / HW <= 2e-6          # mean SSIM per channel


def _random_pair(H, W, seed):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
    base = 0.5 + 0.4 * np.sin(xx / 17.0 + yy / 23.0)[None] * np.array([1.0, 0.8, 0.6], np.float32)[:, None, None]
    gt = np.clip(np.round(255 * (base + rng.normal(0, 0.02, (3, H, W)))), 0, 255).astype(np.uint8)
    img = (base + rng.normal(0, 0.06, (3, H, W))).astype(np.float32)
    return img, gt


@pytest.mark.parametrize("saved", [False, True])
def test_metrics_kernel_matches_golden_and_oracle(saved):
    g = np.load(GOLDEN)
    proto = "saved" if saved else "report"
    for i in range(int(g["n"])):
        img, gt = g[f"image{i}"], g[f"gt{i}"]
        H, W = gt.shape[1:]
        got = _metrics(img, gt, saved)[0]
        _check_sums(got, mo.metric_sums(img, gt, saved), H * W)
        m = mo.derive(got, H, W, proto)
        assert abs(m["l1"] / float(g[f"{proto}_l1_{i}"]) - 1) <= 1e-6
        assert abs(m["psnr"] - float(g[f"{proto}_psnr_{i}"])) <= 1e-4
        assert abs(m["ssim"] - float(g[f"{proto}_ssim_{i}"])) <= 1e-5
    img, gt = _random_pair(1080, 1920, 5)
    _check_sums(_metrics(img, gt, saved)[0], mo.metric_sums(img, gt, saved), 1080 * 1920)


def test_saved_mode_quantises_exactly_like_torch():
    """Values on and next to every rounding boundary of save_image's mul(255).add_(0.5): the kernel's saved mode equals
    report mode on the image quantised by torch's own expression on the device, to fp64 summation order (one pixel
    quantised differently would move the sums by ~1e-9 relative)."""
    H, W = 1080, 1920
    k = torch.arange(H * W, device="cuda", dtype=torch.float32).reshape(1, H, W) % 256
    base = (k - 0.5) / 255.0
    img = torch.cat([base, torch.nextafter(base, torch.full_like(base, 2.0)),
                     torch.nextafter(base, torch.full_like(base, -2.0))]).contiguous()
    img = torch.where(torch.rand_like(img) < 0.01, img * 3 - 1, img)      # some values outside [0, 1]
    q = img.clamp(0.0, 1.0).mul(255).add_(0.5).clamp_(0, 255).to(torch.uint8).float()
    # to_tensor divides on the host (metrics.py:31-32); a CUDA division by a Python scalar multiplies by the rounded
    # reciprocal instead, so divide by a tensor to get the true quotient on the device
    q = q / torch.full_like(q, 255.0)
    gt = torch.randint(0, 256, (3, H, W), dtype=torch.uint8, device="cuda")
    rows4 = [(0, H, 0, H)]
    a = ops.image_metrics_batched(img[None], [gt], rows4, saved=True).cpu().numpy()
    b = ops.image_metrics_batched(q[None].contiguous(), [gt], rows4, saved=False).cpu().numpy()
    np.testing.assert_allclose(a, b, rtol=1e-12, atol=0)


@pytest.mark.parametrize("H,division_pos", [(1080, [0, 20, 45, 68]), (1060, [0, 66, 67]), (400, [0, 7, 13, 19, 25])])
def test_strip_windows_with_halos_equal_full_image_sums(H, division_pos):
    from gs_b200 import division, evaluate
    W = 640
    img, gt = _random_pair(H, W, H)
    world = len(division_pos) - 1
    wins = [evaluate.plan_window(division.DivisionStrategy(0, list(range(world)), division_pos, (H + 15) // 16, r), H)
            for r in range(world)]
    for saved in (False, True):
        full = _metrics(img, gt, saved)[0]
        parts = _metrics(img, gt, saved, [w.rows4() for w in wins]).sum(axis=0)
        np.testing.assert_allclose(parts, full, rtol=1e-12, atol=0)


# ---------------------------------------------------------------------------------------------------------
# Trainer.evaluate
# ---------------------------------------------------------------------------------------------------------
C1_N, C1_W, C1_H = 50_000, 400, 400


def _ssim_torch(img, gt):
    """utils/loss_utils.py:39-85 in fp32 torch (11x11 window, sigma 1.5, zero padding)."""
    import math
    g = torch.tensor([math.exp(-((x - 5) ** 2) / float(2 * 1.5 ** 2)) for x in range(11)])
    g = g / g.sum()
    w = (g[:, None] @ g[None, :]).float()[None, None].expand(3, 1, 11, 11).contiguous().to(img.device)
    conv = lambda t: F.conv2d(t, w, padding=5, groups=3)
    mu1, mu2 = conv(img), conv(gt)
    s1, s2, s12 = conv(img * img) - mu1 ** 2, conv(gt * gt) - mu2 ** 2, conv(img * gt) - mu1 * mu2
    C1, C2 = 0.01 ** 2, 0.03 ** 2
    return (((2 * mu1 * mu2 + C1) * (2 * s12 + C2)) / ((mu1 ** 2 + mu2 ** 2 + C1) * (s1 + s2 + C2))).mean()


def _psnr_torch(img, gt):   # utils/image_utils.py:19-21
    mse = ((img - gt) ** 2).view(img.shape[0], -1).mean(1, keepdim=True)
    return 20 * torch.log10(1.0 / torch.sqrt(mse))


def reference_protocol(params, cams, gts, protocol):
    """train_internal.py:466-479 / render.py + metrics.py restated: one render per camera, clamp, fp32 torch metrics."""
    out = []
    with torch.no_grad():
        for cam, gt in zip(cams, gts):
            dcam = pipeline.DeviceCamera(cam, "cuda")
            rs = dcam.settings(params.active_sh_degree)
            m2, rgb, co, radii, depths = ops.preprocess_gaussians_raw(params._xyz, params._features_dc,
                                                                      params._features_rest, params._scaling,
                                                                      params._rotation, params._opacity, rs)
            image, *_ = ops.render_gaussians(m2, co, rgb, depths, radii, None, rs)
            image = torch.clamp(image, 0.0, 1.0)
            gt_image = torch.clamp(gt.cuda().float() / 255.0, 0.0, 1.0)
            if protocol == "saved":
                q = image.mul(255).add_(0.5).clamp_(0, 255).to(torch.uint8).float()
                image = q / torch.full_like(q, 255.0)      # to_tensor's true division (metrics.py:31-32)
                psnr = float(_psnr_torch(image[None], gt_image[None]).mean())
            else:
                psnr = float(_psnr_torch(image, gt_image).mean())
            out.append(dict(l1=float(torch.abs(image - gt_image).mean()), psnr=psnr, ssim=float(_ssim_torch(image[None], gt_image[None]))))
    return out


def _c1(nviews=6, seed=0):
    scene = syn.make_scene(C1_N, C1_W, C1_H, seed=seed)
    cams = [syn.make_camera(C1_W, C1_H, yaw_deg=3.0 * k - 7.0, uid=100 + k) for k in range(nviews)]
    gts = [torch.from_numpy(syn.make_gt_image(C1_W, C1_H, seed=20 + k)) for k in range(nviews)]
    return scene, cams, gts


@pytest.mark.parametrize("protocol", ["report", "saved"])
def test_evaluate_matches_the_reference_protocol(protocol):
    scene, cams, gts = _c1()
    train_cams = syn.make_batch_cameras(C1_W, C1_H, 4)
    tr = pipeline.Trainer(scene, train_cams, [torch.from_numpy(syn.make_gt_image(C1_W, C1_H, seed=k)).pin_memory()
                                              for k in range(4)], "cuda")
    for views, bs in ((6, 1), (6, 4), (5, 4)):
        got = tr.evaluate(cams[:views], gts[:views], batch_size=bs, protocol=protocol)
        ref = reference_protocol(tr.params, cams[:views], gts[:views], protocol)
        assert [v["uid"] for v in got["per_view"]] == [c["uid"] for c in cams[:views]]
        for g, r in zip(got["per_view"], ref):
            assert abs(g["l1"] / r["l1"] - 1) <= 1e-6, (bs, g, r)
            assert abs(g["psnr"] - r["psnr"]) <= 1e-4, (bs, g, r)
            assert abs(g["ssim"] - r["ssim"]) <= 2e-6, (bs, g, r)
        for key in ("l1", "psnr", "ssim"):
            assert abs(got[key] - np.mean([v[key] for v in got["per_view"]])) <= 1e-12
    # gts already on the device give the same numbers
    dev_gts = [g.cuda() for g in gts]
    a = tr.evaluate(cams, gts, batch_size=4, protocol=protocol)
    b = tr.evaluate(cams, dev_gts, batch_size=4, protocol=protocol)
    for x, y in zip(a["per_view"], b["per_view"]):
        assert abs(x["l1"] - y["l1"]) <= 1e-12 * x["l1"] and abs(x["ssim"] - y["ssim"]) <= 1e-12


def test_evaluate_has_no_side_effects_on_training():
    scene, cams, gts = _c1(nviews=3, seed=2)
    train_cams = syn.make_batch_cameras(C1_W, C1_H, 4)
    tgts = [torch.from_numpy(syn.make_gt_image(C1_W, C1_H, seed=k)).pin_memory() for k in range(4)]

    def run(with_eval):
        tr = pipeline.Trainer(scene, train_cams, tgts, "cuda")
        l0 = tr.step(resident=False)
        if with_eval:
            before = (len(tr.history.history), list(tr.balance_log), tr.iteration, list(tr._pending_feedback),
                      tr.last_info(), tr.io_bytes_per_step(), tr.means2D, tr._radii_local,
                      [t.grad.clone() for t in tr.params.raw_parameters()])
            tr.evaluate(cams, gts, protocol="report")
            after = (len(tr.history.history), list(tr.balance_log), tr.iteration, list(tr._pending_feedback),
                     tr.last_info(), tr.io_bytes_per_step(), tr.means2D, tr._radii_local)
            assert before[:6] == after[:6]
            assert before[6] is after[6] and before[7] is after[7]
            assert all(torch.equal(a, t.grad) for a, t in zip(before[8], tr.params.raw_parameters()))
            assert tr._ex.PIGGYBACK_IN is None
        l1 = tr.step(resident=False)
        torch.cuda.synchronize()
        grads = [t.grad.clone() for t in tr.params.raw_parameters()] + [tr.means2D.grad.clone()]
        return (l0, l1), tr.last_info(), grads

    # The blend backward accumulates with float atomics, so gradients vary from run to run.  The spread of plain runs is
    # taken over three of them (three pairs): one pair is too small a sample of the atomics' ordering noise.
    a, plain = run(True), [run(False) for _ in range(3)]
    assert all(a[0] == p[0] for p in plain)
    assert all(a[1] == p[1] for p in plain)
    pairs = [(0, 1), (0, 2), (1, 2)]
    for q, ga in enumerate(a[2]):
        gp = [p[2][q] for p in plain]
        dmax = lambda x, y: float((x - y).abs().max())
        drms = lambda x, y: float((x - y).double().pow(2).mean().sqrt())
        spread_max, spread_rms = max(dmax(gp[i], gp[j]) for i, j in pairs), max(drms(gp[i], gp[j]) for i, j in pairs)
        diff_max, diff_rms = min(dmax(ga, g) for g in gp), min(drms(ga, g) for g in gp)
        floor = 1e-7 * float(gp[0].double().pow(2).mean().sqrt())
        assert diff_max <= 2 * spread_max + floor, (q, diff_max, spread_max)
        assert diff_rms <= 2 * spread_rms + floor, (q, diff_rms, spread_rms)


# Held-out "report" PSNR of the student measured by the first device run of this test (one B200, 1000 W power limit):
# 15.170 / 23.339 / 29.342 / 35.660 dB at steps 0 / 50 / 100 / 200, a gain of 20.49 dB.  The test asks for at least half
# of that gain.
FIRST_RUN_GAIN_DB = 20.49


def test_training_improves_held_out_views():
    """Teacher: make_scene(50 000, 400, 400); ground truth = the teacher rendered by the library, rounded to uint8, for 4
    training yaws and 3 held-out yaws.  Student: the teacher with its SH coefficients re-drawn from a seeded generator,
    trained 200 steps with FusedAdam.  The held-out report PSNR is non-decreasing (within 0.05 dB) at steps 0 / 50 / 100
    / 200, and gains at least half of the first device run's 20.49 dB (15.17 -> 35.66 dB on one B200)."""
    from gs_b200.optim import FusedAdam
    teacher = syn.make_scene(C1_N, C1_W, C1_H, seed=11)
    train_cams = [syn.make_camera(C1_W, C1_H, yaw_deg=y, uid=k) for k, y in enumerate((-9.0, -3.0, 3.0, 9.0))]
    held = [syn.make_camera(C1_W, C1_H, yaw_deg=y, uid=10 + k) for k, y in enumerate((-6.0, 0.0, 6.0))]
    tp = pipeline.GaussianParams(teacher, "cuda")

    def render_u8(cam):
        with torch.no_grad():
            rs = pipeline.DeviceCamera(cam, "cuda").settings(3)
            m2, rgb, co, radii, depths = ops.preprocess_gaussians_raw(tp._xyz, tp._features_dc, tp._features_rest,
                                                                      tp._scaling, tp._rotation, tp._opacity, rs)
            img, *_ = ops.render_gaussians(m2, co, rgb, depths, radii, None, rs)
            return (img.clamp(0, 1) * 255).round().to(torch.uint8).cpu()

    train_gts = [render_u8(c).pin_memory() for c in train_cams]
    held_gts = [render_u8(c) for c in held]
    student = dict(teacher)
    rng = np.random.default_rng(12)
    student["shs"] = np.concatenate([rng.normal(0.0, 1.0, (C1_N, 1, 3)), rng.normal(0.0, 0.1, (C1_N, 15, 3))],
                                    1).astype(np.float32)
    tr = pipeline.Trainer(student, train_cams, train_gts, "cuda")
    opt = FusedAdam(tr.optimizer_groups(), eps=1e-15)
    psnr = {0: tr.evaluate(held, held_gts)["psnr"]}
    for it in range(1, 201):
        tr.step()
        opt.step()
        if it in (50, 100, 200):
            psnr[it] = tr.evaluate(held, held_gts)["psnr"]
    gain = psnr[200] - psnr[0]
    print(f"[convergence] held-out report PSNR by step: {psnr}; gain {gain:.3f} dB")
    steps = sorted(psnr)
    assert all(psnr[b] >= psnr[a] - 0.05 for a, b in zip(steps, steps[1:])), psnr
    assert gain >= 0.5 * FIRST_RUN_GAIN_DB, (gain, FIRST_RUN_GAIN_DB)


def test_evaluate_rejects_bad_input():
    scene, cams, gts = _c1(nviews=3)
    tr = pipeline.Trainer(scene, syn.make_batch_cameras(C1_W, C1_H, 2),
                          [torch.from_numpy(syn.make_gt_image(C1_W, C1_H, seed=k)) for k in range(2)], "cuda")
    with pytest.raises(ValueError):
        tr.evaluate([], [])
    with pytest.raises(ValueError):
        tr.evaluate(cams, gts, batch_size=ops.MAX_VIEWS + 1)
    with pytest.raises(ValueError):
        tr.evaluate(cams, gts[:2])
    with pytest.raises(ValueError):
        tr.evaluate(cams, [gts[0], gts[1], gts[2][:, :-1]])
    with pytest.raises(TypeError):
        tr.evaluate(cams, [gts[0], gts[1], gts[2].float()])
    with pytest.raises(ValueError):
        tr.evaluate(cams[:2] + [syn.make_camera(C1_W + 16, C1_H)], gts[:2] + [torch.zeros((3, C1_H, C1_W + 16), dtype=torch.uint8)])
    with pytest.raises(ValueError):
        tr.evaluate(cams, gts, protocol="lpips")
    with pytest.raises(ValueError):
        ops.image_metrics_batched(torch.zeros((1, 3, 8, 8), device="cuda"), [None], [(0, 9, 0, 9)])
    with pytest.raises(TypeError):
        ops.image_metrics_batched(torch.zeros((1, 3, 8, 8), device="cuda"), [torch.zeros((3, 8, 8), device="cuda")],
                                  [(0, 8, 0, 8)])


@pytest.mark.parametrize("world", [2, 4])
def test_multi_gpu_evaluate_matches_one_rank(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(29600 + 7 * world), os.path.join(ROOT, "tests", "mgpu_eval.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    print(r.stdout[-4000:])
    assert r.returncode == 0, r.stderr[-4000:]
    assert "[mgpu-eval] PASS" in r.stdout
