"""The REFERENCE's own step functions over the drop-in boundary (VERDICT r1 #10), replayed from a recording.

tests/golden/make_dropin_golden.py ran `distributed_preprocess3dgs_and_all2all_final` -> `render_final` ->
`batched_loss_computation` -> `loss.backward()` -> `finish_strategy_final` (gaussian_renderer/__init__.py:878-1037,
1217-1288; loss_distribution.py:2536-2637; workload_division.py:944-998; train_internal.py:139-196) -- and then the
LEGACY sequence `replicated_preprocess3dgs` -> `render` with a flat `DivisionStrategy` and its `extended_compute_locally`
mask (:66-174, :458-507) -- UNMODIFIED on CPU tensors with W = 1, a real reference `GaussianModel` holding the parameters
and a real `DivisionStrategyFinal`.  The two operator methods of OUR `diff_gaussian_rasterization.GaussianRasterizer` were
recorders that kept every argument the reference passed and answered with the CPU oracle wrapped in an autograd
function; tests/golden/{dropin.json,l3_step.npz} hold those arguments and what the reference computed from the answers
(its L1+SSIM loss, the chain rule to its raw parameters, the legacy image), the per-Gaussian arrays and the image for a
seeded sample of rows and pixels.  Here (a) every recorded argument is checked against the contract of SURVEY.md 8b
(keyword names, dtypes, shapes, the 12 settings fields, the cuda_args keys) and our operator's own argument validation,
and (b) the oracle's own training step must reproduce the reference's loss and parameter gradients.  That pins the conventions that only the caller knows: transposed matrices, SH layout (N,16,3),
pre-applied activations, bool (TY,TX) mask, extended_compute_locally = None, the stats_collector keys
finish_strategy_final reads.
"""
import inspect
import json
import os

import numpy as np
import pytest
import torch

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

CUDA_ARGS_KEYS = {"mode", "world_size", "global_rank", "local_rank", "mp_world_size", "mp_rank", "log_folder",
                  "log_interval", "iteration", "zhx_debug", "zhx_time", "avoid_pixel_all2all", "stats_collector"}
INPUTS = ("means3D", "scales", "rotations", "shs", "opacities")


def _close(got, want, tol=2e-4):
    """All but 0.1 % of the elements within tol relative to themselves plus tol of the array's rms."""
    rms = float(np.sqrt((want.astype(np.float64) ** 2).mean()))
    return (np.abs(got - want) <= tol * np.abs(want) + tol * rms).mean() > 0.999


def test_reference_step_functions_run_over_the_dropin_boundary():
    import diff_gaussian_rasterization as dgr
    from gs_b200 import division, ops, synthetic as syn
    from oracle.oracle import Oracle
    rec = json.load(open(os.path.join(G, "dropin.json")))
    z = np.load(os.path.join(G, "l3_step.npz"))
    s = rec["scene"]
    W, H, N = s["W"], s["H"], s["N"]
    cam = syn.make_camera(W, H, yaw_deg=s["camera"]["yaw_deg"])
    scene = syn.make_scene(N, W, H, seed=s["scene_seed"], radius_px=s["radius_px"])
    gt = syn.make_gt_image(W, H, seed=s["gt_seed"])
    ty, tx = (H + 15) // 16, (W + 15) // 16

    # ---- (a) what the reference passed to preprocess_gaussians / render_gaussians, live step and legacy sequence ----
    for phase in ("", "legacy_"):
        assert set(rec[phase + "preprocess_keywords"]) == {*INPUTS, "cuda_args"}
        assert set(rec[phase + "render_keywords"]) == {"means2D", "conic_opacity", "rgb", "depths", "radii", "compute_locally",
                                                       "extended_compute_locally", "cuda_args"}
        inspect.signature(dgr.GaussianRasterizer.preprocess_gaussians).bind(None, **dict.fromkeys(rec[phase + "preprocess_keywords"]))
        inspect.signature(dgr.GaussianRasterizer.render_gaussians).bind(None, **dict.fromkeys(rec[phase + "render_keywords"]))
        assert tuple(rec[phase + "raster_settings_fields"]) == dgr.GaussianRasterizationSettings._fields
        rs = rec[phase + "raster_settings"]
        assert (rs["image_height"], rs["image_width"], rs["sh_degree"]) == (H, W, 3)
        assert rs["prefiltered"] is False and rs["debug"] is False and rs["scale_modifier"] == 1.0 and rs["bg"] == [0, 0, 0]
        for k in ("viewmatrix", "projmatrix", "campos"):     # the transposed (row-vector) storage of scene/cameras.py
            np.testing.assert_array_equal(np.asarray(rs[k], np.float32), np.asarray(cam[k], np.float32), err_msg=k)
        assert abs(rs["tanfovx"] - cam["tanfovx"]) < 1e-12 and abs(rs["tanfovy"] - cam["tanfovy"]) < 1e-12
        for call in ("preprocess", "render"):
            ca = rec[f"{phase}{call}_cuda_args"]
            assert set(ca) == CUDA_ARGS_KEYS | ({"dist_global_strategy"} if phase else set()), sorted(ca)
            for k, t in ca.items():                                           # all str (SURVEY 8b)
                assert t == {"stats_collector": "dict", "avoid_pixel_all2all": "bool"}.get(k, "str"), (k, t)
        for name in INPUTS:
            assert rec[phase + "preprocess_inputs"][name] == {"dtype": "torch.float32", "requires_grad": True}, name
        assert rec[phase + "compute_locally"] == {"dtype": "torch.bool", "shape": [ty, tx]}
        assert z[phase + "compute_locally"].all()                             # W = 1: everything is local
    assert "extended_compute_locally" not in rec                              # workload_division.py:802-803
    ext, cl = z["legacy_extended_compute_locally"], z["legacy_compute_locally"]
    assert rec["legacy_extended_compute_locally"] == {"dtype": "torch.bool", "shape": [ty, tx]}
    assert (ext | ~cl).all() and ext.all()                                    # the dilated region covers the local one
    # pre-applied activations (scene/gaussian_model.py:109-129): exp'd scales, unit quaternions, sigmoid'd opacity
    rows, pix = z["rows"], z["pixels"]
    n = len(rows)
    for name, shape in zip(INPUTS, ((n, 3), (n, 3), (n, 4), (n, 16, 3), (n, 1))):
        assert z[f"in_{name}"].shape == shape, name
    op = np.clip(scene["opacities"], 1e-6, 1 - 1e-6)
    assert np.array_equal(z["in_means3D"], scene["means3D"][rows]) and np.array_equal(z["in_shs"], scene["shs"][rows])
    np.testing.assert_allclose(z["in_scales"], scene["scales"][rows], rtol=1e-6)
    np.testing.assert_allclose(np.linalg.norm(z["in_rotations"], axis=1), 1.0, atol=1e-5)
    q = scene["rotations"][rows]
    np.testing.assert_allclose(z["in_rotations"], q / np.linalg.norm(q, axis=1, keepdims=True), atol=1e-6)
    np.testing.assert_allclose(z["in_opacities"], op[rows], rtol=1e-5, atol=1e-7)
    # the stats_collector keys finish_strategy_final reads are all there after the step, and our restatement of its cost
    # (division.running_time_of) needs no other
    assert set(rec["stats_collector_keys_read"]) <= set(rec["stats_collector_keys_after_step"])
    assert division.running_time_of({k: 1.0 for k in rec["stats_collector_keys_read"]}) > 0

    orc = Oracle(np.float32)
    ref = orc.train_step(scene, cam, gt)
    pre = ref["pre"]
    # the drop-in's own validation of the legacy mask (gs_b200.ops.render_gaussians) on exactly these arguments: a covering
    # mask gets as far as the device check ("no CPU path"), a mask that does not cover compute_locally is rejected
    rs = rec["legacy_raster_settings"]
    settings = dgr.GaussianRasterizationSettings(**{k: torch.tensor(v) if isinstance(v, list) else v for k, v in rs.items()})
    cuda_args = {k: {"dict": {}, "bool": False}.get(t, "0") for k, t in rec["legacy_render_cuda_args"].items()}
    a = (torch.tensor(pre["means2D"]), torch.tensor(pre["conic_opacity"]), torch.tensor(pre["rgb"]), torch.tensor(pre["depths"]),
         torch.tensor(pre["radii"]), torch.tensor(cl), settings, cuda_args)
    with pytest.raises(ValueError, match="CUDA tensor"):
        ops.render_gaussians(*a, extended_compute_locally=torch.tensor(ext))
    with pytest.raises(ValueError, match="cover"):
        ops.render_gaussians(*a, extended_compute_locally=torch.zeros_like(torch.tensor(ext)))

    # ---- (b) the same step by the oracle's own harness ------------------------------------------------------------------
    assert abs(rec["loss"] - ref["loss"]) <= 2e-6 * abs(ref["loss"]), (rec["loss"], ref["loss"])
    e = ref["grads"]
    q, gq = scene["rotations"], e["rotations"]
    raw = {"_xyz": e["means3D"], "_features_dc": e["shs"][:, :1], "_features_rest": e["shs"][:, 1:],
           "_scaling": e["scales"] * scene["scales"], "_opacity": e["opacities"] * op * (1 - op),
           "_rotation": gq - q * (q * gq).sum(1, keepdims=True)}
    for name, r in raw.items():
        assert _close(z[f"grad{name}"], r[rows]), (name, float(np.abs(z[f"grad{name}"] - r[rows]).max()))
    assert _close(z["grad_means2D"], ref["render_grads"]["means2D"][rows])
    # the legacy sequence: the reference's image, and the screen-space gradient of a weighted sum of it
    np.testing.assert_allclose(z["legacy_image"], ref["fwd"]["image"].reshape(3, -1)[:, pix], rtol=0, atol=2e-6)
    rb = orc.render_backward(H, W, ref["pre"]["means2D"], ref["pre"]["conic_opacity"], ref["pre"]["rgb"], (0.0, 0.0, 0.0),
                             ref["fwd"], z["legacy_weights"].astype(np.float32))
    assert _close(z["legacy_grad_means2D"], rb["means2D"][rows])
