"""Records tests/golden/dropin.json and tests/golden/l3_step.npz by running the reference's OWN Python over the drop-in
boundary on CPU.  Needs a checkout of nyu-systems/Grendel-GS; the tests read only the recorded files.

  python tests/golden/make_dropin_golden.py <path to a Grendel-GS checkout>

1. The names the reference reaches in the drop-in packages (an AST scan of its sources), the keywords it builds
   GaussianRasterizationSettings with, and the tile grid its utils derive from our get_block_XY().
2. `distributed_preprocess3dgs_and_all2all_final` -> `render_final` -> `batched_loss_computation` -> `loss.backward()` ->
   `finish_strategy_final` (gaussian_renderer/__init__.py:878-1037, 1217-1288; loss_distribution.py:2536-2637;
   workload_division.py:944-998; train_internal.py:139-196), then the LEGACY sequence `replicated_preprocess3dgs` ->
   `render` with a flat `DivisionStrategy` and its `extended_compute_locally` mask (:66-174, :458-507), run UNMODIFIED on
   CPU tensors with W = 1, a real reference `GaussianModel` holding the parameters and a real `DivisionStrategyFinal`.
   The two operator methods of our `diff_gaussian_rasterization.GaussianRasterizer` are replaced by recorders that keep
   every argument the reference passes (keyword names, raster settings, cuda_args, the activated inputs, the masks) and
   answer with the CPU oracle wrapped in an autograd function.  The reference's loss, the gradients of its raw
   parameters and its legacy image are stored (for a seeded sample of the Gaussians and pixels);
   tests/test_reference_l3_drive.py checks them against the oracle's own
   training step, and the recorded arguments against our operator's contract.
"""
import ast
import json
import os
import re
import sys
import types
from argparse import Namespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
PKG = os.path.join(ROOT, "grendel-gs_b200")
DROPIN_MODULES = ("diff_gaussian_rasterization", "simple_knn._C", "plyfile", "gsplat")


def names_used(ref):
    """{module: sorted dotted names} the reference's sources reach in each drop-in module."""
    used = {m: set() for m in DROPIN_MODULES}
    for d, _, files in os.walk(ref):
        if os.sep + "submodules" in d or os.sep + ".git" in d:
            continue
        for f in files:
            if not f.endswith(".py"):
                continue
            tree = ast.parse(open(os.path.join(d, f), encoding="utf-8").read())
            for node in ast.walk(tree):
                if isinstance(node, ast.ImportFrom) and node.module in used:
                    used[node.module].update(a.name for a in node.names)
                elif isinstance(node, ast.Attribute) and not isinstance(getattr(node, "_parent_attr", None), ast.Attribute):
                    chain, n = [], node
                    while isinstance(n, ast.Attribute):
                        chain.append(n.attr)
                        n = n.value
                    if isinstance(n, ast.Name) and n.id == "diff_gaussian_rasterization":
                        used[n.id].add(".".join(reversed(chain)))
                for child in ast.iter_child_nodes(node):
                    child._parent_attr = node
    return {m: sorted(v) for m, v in used.items()}


def main(ref):
    if not os.path.isdir(os.path.join(ref, "gaussian_renderer")):
        raise SystemExit(f"{ref} is not a Grendel-GS checkout")
    record = {"names_used": names_used(ref)}

    # ---- no GPU needed: "cuda" placement requests of the reference land on the CPU ---------------------------------
    def _cpuify(fn):
        def w(*a, **k):
            if str(k.get("device", "")).startswith("cuda"):
                k["device"] = "cpu"
            return fn(*a, **k)
        return w
    for name in ("zeros", "ones", "empty", "tensor", "arange", "full"):
        setattr(torch, name, _cpuify(getattr(torch, name)))
    torch.cuda.synchronize = lambda *a, **k: None
    torch.Tensor.cuda = lambda self, *a, **k: self

    sys.path[:0] = [PKG, ROOT, os.path.join(PKG, "shims"), ref]
    import diff_gaussian_rasterization as dgr
    import utils.general_utils as utils
    import gaussian_renderer as gr
    import gaussian_renderer.workload_division as wd
    import gaussian_renderer.loss_distribution as ld
    from scene.gaussian_model import GaussianModel
    from gs_b200 import synthetic as syn
    from oracle.oracle import Oracle

    # ---- settings keywords and tile grid of the reference (arguments/__init__.py:254-257, __init__.py:930-943) -------
    src = open(os.path.join(ref, "gaussian_renderer", "__init__.py"), encoding="utf-8").read()
    a = src.index("def distributed_preprocess3dgs_and_all2all_final")
    body = src[a:]
    kw = re.findall(r"^\s+(\w+)=", body[body.index("GaussianRasterizationSettings("):body.index("rasterizer = GaussianRasterizer")],
                    flags=re.M)
    record["settings_keywords"] = kw
    bx, by, one = dgr._C.get_block_XY()
    utils.set_block_size(bx, by, one)
    utils.set_img_size(1080, 1920)
    record["grid_1080p"] = dict(BLOCK_X=utils.BLOCK_X, BLOCK_Y=utils.BLOCK_Y, ONE_DIM_BLOCK_SIZE=utils.ONE_DIM_BLOCK_SIZE,
                                TILE_Y=utils.TILE_Y, TILE_X=utils.TILE_X)

    # ---- the training step -------------------------------------------------------------------------------------------
    W, H, N = 96, 64, 1500
    orc = Oracle(np.float32)
    utils.set_block_size(bx, by, one)
    utils.set_img_size(H, W)
    args = Namespace(bsz=1, log_interval=50, log_folder="logs", zhx_debug=False, zhx_time=False, lambda_dssim=0.2,
                     lr_scale_loss=1.0, gaussians_distribution=True, image_distribution=True, local_sampling=False,
                     border_divpos_coeff=1.0, heuristic_decay=0.0, no_heuristics_update=False,
                     adjust_strategy_warmup_iterations=-1, adjust_strategy_warmp_iterations=-1, backend="default")
    utils.set_args(args)
    utils.set_cur_iter(1)
    utils.GLOBAL_RANK, utils.LOCAL_RANK, utils.WORLD_SIZE = 0, 0, 1

    class _Group:
        def size(self): return 1
        def rank(self): return 0
    utils.DEFAULT_GROUP = utils.DP_GROUP = utils.MP_GROUP = utils.IN_NODE_GROUP = _Group()

    class _Timers:
        def start(self, *a, **k): pass
        def stop(self, *a, **k): pass
    utils.set_timers(_Timers())
    utils.check_initial_gpu_memory_usage = lambda *a, **k: None

    cam_d = syn.make_camera(W, H, yaw_deg=3.0)
    scene = syn.make_scene(N, W, H, seed=11, radius_px=9.0)
    gt = syn.make_gt_image(W, H, seed=5)
    camera = types.SimpleNamespace(uid=0, image_height=H, image_width=W, FoVx=cam_d["FoVx"], FoVy=cam_d["FoVy"],
                                   world_view_transform=torch.tensor(cam_d["viewmatrix"]),
                                   full_proj_transform=torch.tensor(cam_d["projmatrix"]),
                                   camera_center=torch.tensor(cam_d["campos"]), original_image=torch.tensor(gt))

    # a real reference GaussianModel with the raw parameter layout (scene/gaussian_model.py:219-228)
    pc = GaussianModel(3)
    pc.active_sh_degree = 3
    op = np.clip(scene["opacities"], 1e-6, 1 - 1e-6)
    P = torch.nn.Parameter
    pc._xyz = P(torch.tensor(scene["means3D"]))
    pc._features_dc = P(torch.tensor(scene["shs"][:, :1].copy()))
    pc._features_rest = P(torch.tensor(scene["shs"][:, 1:].copy()))
    pc._scaling = P(torch.log(torch.tensor(scene["scales"])))
    pc._rotation = P(torch.tensor(scene["rotations"]))
    pc._opacity = P(torch.log(torch.tensor(op) / (1 - torch.tensor(op))))

    # ---- the operator boundary: recorders + oracle-backed autograd ---------------------------------------------------
    arrays, calls = {}, []
    phase = [""]     # "" = the live step, "legacy_" = the legacy sequence

    def cam_of(rs):
        return dict(image_height=rs.image_height, image_width=rs.image_width, tanfovx=rs.tanfovx, tanfovy=rs.tanfovy,
                    viewmatrix=rs.viewmatrix.numpy(), projmatrix=rs.projmatrix.numpy(), campos=rs.campos.numpy(),
                    sh_degree=rs.sh_degree)

    class _Pre(torch.autograd.Function):
        @staticmethod
        def forward(ctx, means3D, scales, rotations, shs, opacities, rs):
            a = [t.detach().numpy() for t in (means3D, scales, rotations, shs, opacities)]
            pre = orc.preprocess_forward(*a, cam_of(rs), scale_modifier=rs.scale_modifier)
            ctx.a, ctx.rs, ctx.pre = a, rs, pre
            outs = (torch.tensor(pre["means2D"]), torch.tensor(pre["rgb"]), torch.tensor(pre["conic_opacity"]),
                    torch.tensor(pre["radii"]), torch.tensor(pre["depths"]))
            ctx.mark_non_differentiable(outs[3], outs[4])
            return outs

        @staticmethod
        def backward(ctx, g_m2, g_rgb, g_co, *_):
            z = lambda g, s: np.zeros(s, np.float32) if g is None else g.numpy()
            n = ctx.a[0].shape[0]
            pb = orc.preprocess_backward(*ctx.a, cam_of(ctx.rs), ctx.pre["radii"], ctx.pre["clamped"], z(g_m2, (n, 2)),
                                         z(g_co, (n, 4)), z(g_rgb, (n, 3)))
            return (torch.tensor(pb["means3D"]), torch.tensor(pb["scales"]), torch.tensor(pb["rotations"]),
                    torch.tensor(pb["shs"]), torch.tensor(pb["opacities"]), None)

    class _Render(torch.autograd.Function):
        @staticmethod
        def forward(ctx, means2D, conic_opacity, rgb, depths, radii, cl, rs):
            a = [t.detach().numpy() for t in (means2D, conic_opacity, rgb, depths, radii)]
            bg = tuple(float(v) for v in rs.bg)
            fwd = orc.render_forward(rs.image_height, rs.image_width, *a, cl.numpy().reshape(-1).astype(np.uint8), bg)
            ctx.a, ctx.rs, ctx.fwd, ctx.bg = a, rs, fwd, bg
            return torch.tensor(fwd["image"])

        @staticmethod
        def backward(ctx, g):
            rb = orc.render_backward(ctx.rs.image_height, ctx.rs.image_width, ctx.a[0], ctx.a[1], ctx.a[2], ctx.bg,
                                     ctx.fwd, g.contiguous().numpy())
            return (torch.tensor(rb["means2D"]), torch.tensor(rb["conic_opacity"]), torch.tensor(rb["rgb"]),
                    None, None, None, None)

    def cuda_args_types(ca):
        return {k: type(v).__name__ for k, v in sorted(ca.items())}

    def preprocess_gaussians(self, *pos, **kw):
        assert not pos, pos
        rs = self.raster_settings
        record[phase[0] + "preprocess_keywords"] = sorted(kw)
        record[phase[0] + "preprocess_cuda_args"] = cuda_args_types(kw["cuda_args"])
        record[phase[0] + "raster_settings"] = {f: (v.tolist() if torch.is_tensor(v) else v) for f, v in rs._asdict().items()}
        record[phase[0] + "raster_settings_fields"] = list(rs._fields)
        for name in ("means3D", "scales", "rotations", "shs", "opacities"):
            t = kw[name]
            record.setdefault(phase[0] + "preprocess_inputs", {})[name] = dict(dtype=str(t.dtype), requires_grad=t.requires_grad)
            if not phase[0]:
                arrays[f"in_{name}"] = t.detach().numpy().copy()
        calls.append("preprocess")
        return _Pre.apply(kw["means3D"], kw["scales"], kw["rotations"], kw["shs"], kw["opacities"], rs)

    def render_gaussians(self, *pos, **kw):
        assert not pos, pos
        record[phase[0] + "render_keywords"] = sorted(kw)
        record[phase[0] + "render_cuda_args"] = cuda_args_types(kw["cuda_args"])
        ext, cl = kw["extended_compute_locally"], kw["compute_locally"]
        record[phase[0] + "compute_locally"] = dict(dtype=str(cl.dtype), shape=list(cl.shape))
        arrays[phase[0] + "compute_locally"] = cl.numpy().copy()
        if ext is not None:
            record[phase[0] + "extended_compute_locally"] = dict(dtype=str(ext.dtype), shape=list(ext.shape))
            arrays[phase[0] + "extended_compute_locally"] = ext.numpy().copy()
        calls.append("render")
        img = _Render.apply(kw["means2D"], kw["conic_opacity"], kw["rgb"], kw["depths"], kw["radii"], cl,
                            self.raster_settings)
        sc = kw["cuda_args"]["stats_collector"]                              # mandatory even at W = 1 (:953-957)
        sc["forward_render_time"], sc["backward_render_time"] = 1.25, 2.5
        z = torch.zeros((), dtype=torch.int64)
        return img, z, z, z

    dgr.GaussianRasterizer.preprocess_gaussians = preprocess_gaussians
    dgr.GaussianRasterizer.render_gaussians = render_gaussians
    assert gr.GaussianRasterizer is dgr.GaussianRasterizer

    # ---- the reference's step, unmodified (train_internal.py:139-196) -------------------------------------------------
    dataset = types.SimpleNamespace(cameras=[camera])
    history = wd.DivisionStrategyHistoryFinal(dataset, 1, 0)
    strategies, _ = wd.start_strategy_final([camera], history)
    assert strategies[0].gpu_ids == [0] and list(strategies[0].division_pos) == [0, utils.TILE_Y]
    pipe = Namespace(debug=False)
    bg = torch.zeros(3)
    pkg = gr.distributed_preprocess3dgs_and_all2all_final([camera], pc, pipe, bg, batched_strategies=strategies, mode="train")
    imgs, cls = gr.render_final(pkg, strategies)
    collectors = [ca["stats_collector"] for ca in pkg["batched_cuda_args"]]
    loss_sum, _ = ld.batched_loss_computation(imgs, [camera], cls, strategies, collectors)
    loss_sum.backward()
    assert calls == ["preprocess", "render"], calls

    class _Reads(dict):                       # the stats_collector keys finish_strategy_final reads
        read = set()

        def __getitem__(self, k):
            _Reads.read.add(k)
            return super().__getitem__(k)

        def get(self, k, *d):
            _Reads.read.add(k)
            return super().get(k, *d)
    wd.finish_strategy_final([camera], history, strategies, [_Reads(c) for c in collectors])
    record["stats_collector_keys_read"] = sorted(_Reads.read)
    record["stats_collector_keys_after_step"] = sorted(collectors[0])
    record["loss"] = loss_sum.item()
    for name in ("_xyz", "_features_dc", "_features_rest", "_scaling", "_rotation", "_opacity"):
        arrays[f"grad{name}"] = getattr(pc, name).grad.numpy().copy()
    arrays["grad_means2D"] = pkg["batched_locally_preprocessed_mean2D"][0].grad.numpy().copy()

    # ---- the LEGACY single-camera sequence (gaussian_renderer/__init__.py:66-174 replicated_preprocess3dgs, :458-507
    #      render; workload_division.py:100-199 DivisionStrategy): flat tile-range division, dist_global_strategy in
    #      cuda_args, and an extended_compute_locally mask handed to render_gaussians -----------------------------------
    from gaussian_renderer.distribution_config import ImageDistributionConfig
    args.image_distribution_config = ImageDistributionConfig("replicated_loss_computation", "DivisionStrategyUniform", False,
                                                             ["backward_render_time"])
    for t in (pc._xyz, pc._features_dc, pc._features_rest, pc._scaling, pc._rotation, pc._opacity):
        t.grad = None

    phase[0] = "legacy_"
    calls.clear()
    legacy_strategy = wd.DivisionStrategy(camera, 1, 0, utils.TILE_X, utils.TILE_Y,
                                          torch.ones((utils.TILE_Y, utils.TILE_X)), "DivisionStrategyUniform")
    pkg1 = gr.replicated_preprocess3dgs(camera, pc, pipe, bg, strategy=legacy_strategy, mode="train")
    img1, _ = gr.render(pkg1, legacy_strategy)
    assert calls == ["preprocess", "render"], calls
    wgt = torch.tensor(np.random.default_rng(2).normal(size=(3, H, W)).astype(np.float16).astype(np.float32))
    (img1 * wgt).sum().backward()
    arrays["legacy_image"] = img1.detach().numpy().copy()
    arrays["legacy_weights"] = wgt.numpy().astype(np.float16)   # exact: the weights are float16 values
    arrays["legacy_grad_means2D"] = pkg1["locally_preprocessed_mean2D"].grad.numpy().copy()

    # a seeded sample of the Gaussians and of the legacy image's pixels keeps the fixture small
    rng = np.random.default_rng(0)
    rows, pix = np.sort(rng.choice(N, 300, replace=False)), np.sort(rng.choice(H * W, 2048, replace=False))
    for k, v in list(arrays.items()):
        if v.shape[:1] == (N,):
            arrays[k] = v[rows]
    arrays["legacy_image"] = arrays["legacy_image"].reshape(3, -1)[:, pix]
    arrays["rows"], arrays["pixels"] = rows, pix
    record["scene"] = dict(W=W, H=H, N=N, camera=dict(yaw_deg=3.0), scene_seed=11, radius_px=9.0, gt_seed=5)
    with open(os.path.join(HERE, "dropin.json"), "w") as f:
        json.dump(record, f, indent=1, sort_keys=True)
        f.write("\n")
    np.savez_compressed(os.path.join(HERE, "l3_step.npz"), **arrays)
    print("written:", os.path.join(HERE, "dropin.json"), os.path.join(HERE, "l3_step.npz"), "loss", record["loss"])


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(os.path.abspath(sys.argv[1]))
