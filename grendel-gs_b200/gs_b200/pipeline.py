"""Host-side training-step pipeline around the operators: the call sequence of
/root/reference/train_internal.py:139-196 (strategy -> GT load -> preprocess (+ all-to-all) -> render ->
loss -> backward) written against our C-ABI operators, for bench.py, smoke() and the tests.

The reference's own Python (gaussian_renderer/*.py) runs unchanged on top of the drop-in
`diff_gaussian_rasterization` package; this module is the equivalent harness for environments where
/root/reference is not present (the GPU box), with the same partitioning rules:
  * Gaussians sharded evenly across ranks (scene/gaussian_model.py:181-194),
  * pixels sharded by contiguous tile rows per camera (workload_division.py:852-941),
  * one sparse all-to-all of projected splats per step and its mirror in backward
    (gaussian_renderer/__init__.py:542-698).
"""

import torch
import torch.nn as nn

from . import ops
from .division import (DivisionStrategy, StrategyHistory, finish_strategy, heuristics_update_enabled,  # noqa: F401
                       start_strategy)


class RasterSettings:
    """Attribute bag with the 12 fields of GaussianRasterizationSettings (gaussian_renderer/__init__.py:930-943)."""
    __slots__ = ("image_height", "image_width", "tanfovx", "tanfovy", "bg", "scale_modifier", "viewmatrix",
                 "projmatrix", "sh_degree", "campos", "prefiltered", "debug")

    def __init__(self, **kw):
        for k in self.__slots__:
            setattr(self, k, kw[k])


class DeviceCamera:
    """Camera constants resident on the GPU (scene/cameras.py:84-100 keeps them as cuda tensors too)."""

    def __init__(self, cam, device, bg=(0.0, 0.0, 0.0)):
        self.uid = cam.get("uid", 0)
        self.image_height, self.image_width = int(cam["image_height"]), int(cam["image_width"])
        self.tanfovx, self.tanfovy = float(cam["tanfovx"]), float(cam["tanfovy"])
        self.sh_degree = int(cam["sh_degree"])
        self.viewmatrix = torch.as_tensor(cam["viewmatrix"], dtype=torch.float32).to(device)
        self.projmatrix = torch.as_tensor(cam["projmatrix"], dtype=torch.float32).to(device)
        self.campos = torch.as_tensor(cam["campos"], dtype=torch.float32).to(device)
        self.bg_host = tuple(float(v) for v in bg)
        self.bg = torch.tensor(self.bg_host, dtype=torch.float32, device=device)

    def settings(self, sh_degree=None):
        return RasterSettings(image_height=self.image_height, image_width=self.image_width, tanfovx=self.tanfovx,
                              tanfovy=self.tanfovy, bg=self.bg, scale_modifier=1.0, viewmatrix=self.viewmatrix,
                              projmatrix=self.projmatrix, sh_degree=self.sh_degree if sh_degree is None else sh_degree,
                              campos=self.campos, prefiltered=False, debug=False)


class GaussianParams(nn.Module):
    """The six raw nn.Parameter tensors of GaussianModel (scene/gaussian_model.py:219-228) with its
    activations (:109-129).  Built from an ACTIVATED synthetic scene by inverting the activations."""

    def __init__(self, scene, device):
        super().__init__()
        t = lambda a: torch.as_tensor(a, dtype=torch.float32).to(device)
        shs = t(scene["shs"])
        op = t(scene["opacities"]).clamp(1e-6, 1 - 1e-6)
        self._xyz = nn.Parameter(t(scene["means3D"]).contiguous())
        self._features_dc = nn.Parameter(shs[:, :1, :].contiguous())
        self._features_rest = nn.Parameter(shs[:, 1:, :].contiguous())
        self._scaling = nn.Parameter(torch.log(t(scene["scales"])).contiguous())
        self._rotation = nn.Parameter(t(scene["rotations"]).contiguous())
        self._opacity = nn.Parameter(torch.log(op / (1 - op)).contiguous())
        self.active_sh_degree = 3

    @property
    def get_xyz(self):
        return self._xyz

    @property
    def get_scaling(self):
        return torch.exp(self._scaling)

    @property
    def get_rotation(self):
        return torch.nn.functional.normalize(self._rotation)

    @property
    def get_opacity(self):
        return torch.sigmoid(self._opacity)

    @property
    def get_features(self):
        return torch.cat((self._features_dc, self._features_rest), dim=1)

    def raw_parameters(self):
        return [self._xyz, self._features_dc, self._features_rest, self._scaling, self._rotation, self._opacity]


def train_step_single(params, dcam, gt_u8_dev, lambda_dssim=0.2, collector=None, compute_locally=None):
    """One camera on one rank: preprocess -> render -> fused L1+SSIM -> backward.  Returns the loss tensor
    (gradients land in params.*.grad) and the projected means2D (its .grad feeds densification)."""
    rs = dcam.settings(params.active_sh_degree)
    cuda_args = {"stats_collector": collector if collector is not None else {}}
    means2D, rgb, conic_opacity, radii, depths = ops.preprocess_gaussians(
        params.get_xyz, params.get_scaling, params.get_rotation, params.get_features, params.get_opacity, rs, cuda_args)
    means2D.retain_grad()
    image, *_ = ops.render_gaussians(means2D, conic_opacity, rgb, depths, radii, compute_locally, rs, cuda_args)
    loss = ops.fused_loss(image, gt_u8_dev, 0, dcam.image_height, lambda_dssim)
    loss.backward()
    return loss, means2D, radii


class Trainer:
    """Distributed training-step harness (one process per GPU).

    Gaussians are sharded evenly by contiguous chunks (scene/gaussian_model.py:181-194); the B cameras of a
    step are divided into tile-row strips over the W ranks (division.start_strategy); projected splats reach
    their strip owners through exchange.exchange (skipped when W == 1, like gaussian_renderer/__init__.py:968).
    """

    def __init__(self, scene, cams, gts_pinned, device, rank=0, world=1, lambda_dssim=0.2, group=None,
                 fused_activations=True, border_exchange=False, batched_render=True, peer_exchange=None,
                 peer_cap_rows=None, shard=None, load_balance=True, heuristic_decay=0.0,
                 distributed_dataset_storage=False, feedback_lag=None):
        """scene: the WHOLE scene (sliced here into this rank's contiguous shard), or -- shard=(lo, hi, n_total) -- only
        this rank's Gaussians [lo, hi) of an n_total-Gaussian scene (synthetic.make_scene_shard).
        load_balance: feed the measured render times back into the strip division after every step
        (finish_strategy_final, workload_division.py:944-998; only where the reference's gate enables it).
        distributed_dataset_storage: only rank 0 holds the ground-truth images (gts_pinned may be None elsewhere); the
        strips of a resident=False step are scattered from rank 0's GPU (loss_distribution.py:2395-2533, gt_scatter.py)
        instead of being read from every rank's own host copy.
        feedback_lag: 0 = the reference's sequencing (finish_strategy_final right after the step: the render times are
        read, all-gathered and applied before the next step starts, so the host waits for the device at the end of every
        step and cannot enqueue ahead).  > 0 (default 2, GS_B200_FEEDBACK_LAG) = the times of the step `feedback_lag`
        steps back, whose events have long completed, ride on the NEXT exchange's size all-gather (exchange.PIGGYBACK_IN):
        no collective of their own, no host sync; the strips move the same way, `feedback_lag` steps later."""
        from . import exchange as _ex
        self._ex = _ex
        # splat / gradient rows travel by direct NVLink stores from the pack kernels (exchange.PeerBuffers) instead of
        # all_to_all_single; peer_exchange=None: on unless GS_B200_EXCHANGE=nccl.  Buffers hold peer_cap_rows rows
        # (default 1.25 x the scene's Gaussians); a step that needs more falls back to all_to_all_single.
        if peer_exchange is None:
            import os as _os
            peer_exchange = _os.environ.get("GS_B200_EXCHANGE", "p2p") != "nccl"
        self._peer = None
        n = scene["means3D"].shape[0] if shard is None else int(shard[2])
        if world > 1 and peer_exchange:
            # every splat of every local camera can land on one rank (bsz views of the scene): rows of the largest
            # receive / send total.  1.25 x the scene per view, capped by what a step can produce.
            cap = int(peer_cap_rows) if peer_cap_rows else int(1.25 * n) + 65536
            self._peer = _ex.open_peer_buffers(world, rank, cap, device, group)
        if world > 1:
            # NCCL connects the point-to-point channels of all_to_all_single lazily, on first use: ~7 s on an 8-GPU box.  The
            # exchange needs them only when a step exceeds the peer buffers (and the redistribution after densification
            # always does): pay for the set-up here, not inside whichever training step happens to be the first.
            import torch.distributed as _dist
            if _dist.get_backend(group) == "nccl":
                _w = torch.zeros((world,), dtype=torch.float32, device=device)
                _dist.all_to_all_single(torch.empty_like(_w), _w, group=group)
        # bin + blend + loss of all B cameras in one pass (ops.render_gaussians_batched) instead of the reference's
        # per-camera loop (render_final, gaussian_renderer/__init__.py:1217-1288); False keeps the per-camera calls
        self.batched_render = batched_render
        self.device, self.rank, self.world, self.group = device, rank, world, group
        self.lambda_dssim = lambda_dssim
        self.fused_activations = fused_activations
        self.border_exchange = border_exchange   # legacy row L1: exchange 5 halo rows so strip losses sum to the full-image loss
        if shard is None:
            lo, hi = n * rank // world, n * (rank + 1) // world
            self.params = GaussianParams({k: v[lo:hi] for k, v in scene.items()}, device)
        else:
            lo, hi = int(shard[0]), int(shard[1])
            if scene["means3D"].shape[0] != hi - lo:
                raise ValueError("shard=(lo, hi, n_total) does not match the scene passed")
            self.params = GaussianParams(scene, device)
        self.n_local, self.n_total = hi - lo, n
        self.load_balance, self.heuristic_decay = load_balance, heuristic_decay
        if feedback_lag is None:
            import os as _os
            feedback_lag = int(_os.environ.get("GS_B200_FEEDBACK_LAG", "2"))
        self.feedback_lag = max(0, int(feedback_lag))
        self._pending_feedback = []     # steps whose render times have not been fed back yet, oldest first
        self._sent_feedback = None      # the step whose times ride on the exchange of the current step
        self.iteration = 0
        self.balance_log = []      # (iteration, division rows of camera 0) whenever the division moved
        self.dcams = [DeviceCamera(c, device) for c in cams]
        self.H, self.W = self.dcams[0].image_height, self.dcams[0].image_width
        self.tile_y, self.tile_x = (self.H + 15) // 16, (self.W + 15) // 16
        self.distributed_dataset_storage = bool(distributed_dataset_storage) and world > 1
        self.gts_host = gts_pinned                      # uint8 (3,H,W) pinned host tensors
        # copies for the "inputs resident" leg (not needed by ranks without pixels in distributed-storage mode)
        self.gts_dev = [g.to(device) for g in gts_pinned] if gts_pinned is not None else None
        self.history = StrategyHistory([c.uid for c in self.dcams], self.tile_y, world)
        self._strip_cache = {}
        self._cams_packed = None   # (B,40) camera table of the batched preprocess (cameras are fixed per Trainer)
        self._strategy_cache = None
        self._mask_cache = {}
        self._bmask_cache = {}
        self._n_renders = 0
        self._copy_stream = None
        self._loss_host = torch.zeros((1,), dtype=torch.float32).pin_memory()
        self._info = {}
        self._h2d = 0

    # -- ground truth strips (load_camera_from_cpu_to_all_gpu, loss_distribution.py:2395-2533) ------------
    def _gt_strip(self, k, y0, y1, resident):
        key = (k, y0, y1, resident)
        if resident:
            if key not in self._strip_cache:
                self._strip_cache[key] = self.gts_dev[k][:, y0:y1, :].contiguous()
            return self._strip_cache[key]
        return self._strip_h2d(k, y0, y1)

    def _strip_h2d(self, k, y0, y1):
        """Rows [y0, y1) of the pinned (3,H,W) uint8 ground truth -> a (3, rows, W) device strip: the rows of one channel
        are contiguous in the pinned image, so the strip is three asynchronous copies straight out of it -- no staging
        copy, and nothing to re-pin when the load balancer moves the strip boundaries (a pinned staging strip per
        division cost several ms of cudaHostAlloc every time the strips of a 4K view moved)."""
        host = self.gts_host[k]
        if not host.is_pinned():
            key = (k, y0, y1, False)
            if key not in self._strip_cache:
                self._strip_cache[key] = host[:, y0:y1, :].contiguous().pin_memory()
            h = self._strip_cache[key]
            self._h2d += h.numel()
            return h.to(self.device, non_blocking=True)
        d = torch.empty((3, y1 - y0, self.W), dtype=torch.uint8, device=self.device)
        for c in range(3):
            d[c].copy_(host[c, y0:y1, :], non_blocking=True)
        self._h2d += d.numel()
        return d

    def _mark(self, name):
        """GS_B200_TRACE=1: synchronise and accumulate wall-clock per phase (diagnostics only)."""
        if not self._trace_on:
            return
        import time
        torch.cuda.synchronize()
        now = time.perf_counter()
        self.trace[name] = self.trace.get(name, 0.0) + (now - self._t_last) * 1e3
        self._t_last = now

    def step(self, resident=True):
        """One forward + loss + backward over the batch.  resident=False copies the GT strips from pinned host
        memory inside the step and reads the loss back (the end-to-end leg); returns the loss as a float then."""
        ops.STEP_STREAM = torch.cuda.current_stream().cuda_stream   # every kernel of the step goes to this stream
        try:
            return self._step(resident)
        finally:
            ops.STEP_STREAM = None

    def _step(self, resident):
        import os as _os, time as _time
        self._trace_on = _os.environ.get("GS_B200_TRACE") == "1"
        self._ex.TRACE = self._mark if self._trace_on else None
        if self._trace_on:
            if not hasattr(self, "trace"):
                self.trace = {}
            torch.cuda.synchronize()
            self._t_last = _time.perf_counter()
        ops_ = ops
        p = self.params
        for t in p.raw_parameters():
            t.grad = None
        self._h2d = 0
        ops.LAST_R_TOTAL = 0
        uids = [c.uid for c in self.dcams]
        ver = len(self.history.history)   # the division only changes when the cost heuristic is updated
        if self._strategy_cache is None or self._strategy_cache[0] != ver:
            new = start_strategy(uids, self.history, self.world, self.rank)[0]
            moved = self._strategy_cache is None or any(
                a.gpu_ids != b.gpu_ids or a.division_pos != b.division_pos for a, b in zip(new, self._strategy_cache[1]))
            self._strategy_cache = (ver, new)
            if moved:   # per-division caches (masks, pinned GT strips) belong to the old boundaries
                self._strip_cache.clear(); self._mask_cache.clear(); self._bmask_cache.clear()
                self.balance_log.append((self.iteration, [list(st.division_pos) for st in new],
                                         [list(st.gpu_ids) for st in new]))
        strategies = self._strategy_cache[1]
        self._tasks = [[(k, st.division_pos[st.gpu_ids.index(g)], st.division_pos[st.gpu_ids.index(g) + 1])
                        for k, st in enumerate(strategies) if g in st.gpu_ids] for g in range(self.world)]
        settings = [c.settings(p.active_sh_degree) for c in self.dcams]
        # "Asynchronously load ground-truth image to GPU" (loss_distribution.py:2399): the strips this rank needs are
        # copied from pinned host memory on a side stream while preprocess / binning / blend run, and the loss waits
        # on the copy's event.
        gt_ready = {}
        if not resident and self.distributed_dataset_storage:
            from . import gt_scatter
            strips, h2d = gt_scatter.scatter_gt_strips(self.gts_host if self.rank == 0 else self.W, self._tasks, self.H,
                                                       self.device, self.rank, self.world, self.group)
            self._h2d += h2d
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream())
            gt_ready = {k: (t, ev) for k, t in strips.items()}
        elif not resident:
            if self._copy_stream is None:
                self._copy_stream = torch.cuda.Stream(device=self.device)
            for k, st in enumerate(strategies):
                rows = st.local_pixel_rows(self.H)
                if rows is None:
                    continue
                with torch.cuda.stream(self._copy_stream):
                    d = self._strip_h2d(k, rows[0], rows[1])
                    ev = torch.cuda.Event()
                    ev.record(self._copy_stream)
                gt_ready[k] = (d, ev)
        if not self.fused_activations:  # the reference's five activation kernels + cat (__init__.py:902-906)
            xyz, scaling, rotation, feats, opacity = p.get_xyz, p.get_scaling, p.get_rotation, p.get_features, p.get_opacity
        collectors = [{} for _ in self.dcams]
        screen = []
        B = len(settings)
        use_batched = self.batched_render and B > 1 and not self.border_exchange
        if self.fused_activations and len(settings) > 1:
            # all B cameras in ONE launch: every Gaussian is read once and projected into each camera
            if self._cams_packed is None:
                self._cams_packed = ops_.pack_cameras(settings)
            bm2, brgb, bco, bradii, bdepths = ops_.preprocess_gaussians_batched(
                p._xyz, p._features_dc, p._features_rest, p._scaling, p._rotation, p._opacity, self._cams_packed,
                self.W, self.H, p.active_sh_degree)
            bm2.retain_grad()   # (B,P,2): densification reads bm2.grad[k] (means2D.grad of camera k, densification.py:24)
            batched = (bm2, brgb, bco, bradii, bdepths)
            if self.world == 1 and not use_batched:
                for k in range(len(settings)):
                    screen.append((bm2[k], brgb[k], bco[k], bradii[k], bdepths[k]))
            settings_loop = []
        else:
            batched = None
            settings_loop = settings
        for k, rs in enumerate(settings_loop):
            if self.fused_activations:
                out = ops_.preprocess_gaussians_raw(p._xyz, p._features_dc, p._features_rest, p._scaling, p._rotation,
                                                    p._opacity, rs)
            else:
                out = ops_.preprocess_gaussians(xyz, scaling, rotation, feats, opacity, rs,
                                                {"stats_collector": collectors[k]})
            out[0].retain_grad()
            screen.append(out)
        self.means2D = batched[0] if batched is not None else [s[0] for s in screen]
        self._mark("p preprocess")
        if batched is None and (self.world > 1 or use_batched):
            # per-camera results (B == 1 or unfused activations): stack into (B,P,.)
            batched = tuple(torch.stack([s[q] for s in screen]) for q in range(5))
        cat = view_start = None
        if self.world > 1:
            self._feedback_before_exchange()
            if use_batched:
                cat, view_start, cnt = self._ex.exchange_cat(*batched, strategies, settings, self.world, self.rank,
                                                             self.group, self._peer)
            else:
                redistributed, cnt = self._ex.exchange(*batched, strategies, settings, self.world, self.rank, self.group,
                                                       self._peer)
            self._feedback_after_exchange()
        elif use_batched:   # (B,P,.) stacked IS the concatenation: camera k = rows [k P, (k+1) P)
            Pn = batched[0].shape[1]
            cat = (batched[0].reshape(-1, 2), batched[1].reshape(-1, 3), batched[2].reshape(-1, 4),
                   batched[3].reshape(-1), batched[4].reshape(-1))
            view_start = [k * Pn for k in range(B + 1)]
        else:
            redistributed = screen
        self._radii_local = (batched[3] if batched is not None else
                             screen[0][3].unsqueeze(0) if len(screen) == 1 else torch.stack([s[3] for s in screen]))
        self._mark("x5 unpack")
        loss_sum = None
        Vp = Pl = 0
        self._n_renders = 0
        if use_batched:
            mk = tuple((tuple(st.gpu_ids), tuple(st.division_pos), st.rank) for st in strategies)
            if mk not in self._bmask_cache:
                m = torch.zeros((B, self.tile_y, self.tile_x), dtype=torch.uint8, device=self.device)
                rows4, coef, const = [], [], 0.0
                for k, st in enumerate(strategies):
                    r = st.local_rows()
                    if r is None:   # no strip of this camera here: no tiles, no loss term
                        rows4.append((0, 0, 0, 0))
                        coef += [0.0, 0.0]
                        continue
                    m[k, r[0]:r[1]] = 1
                    y0, y1 = st.local_pixel_rows(self.H)
                    rows4.append((y0, y1, y0, y1))
                    coef += [1.0 - self.lambda_dssim, -self.lambda_dssim]
                    const += self.lambda_dssim
                self._bmask_cache[mk] = (m.reshape(B, -1), rows4,
                                         torch.tensor(coef, dtype=torch.float32, device=self.device), const)
            cl, rows4, coef, const = self._bmask_cache[mk]
            m2, rgb, co, radii, depths = cat
            images, _stats = ops_.render_gaussians_batched(m2, co, rgb, depths, radii, cl, view_start, settings[0],
                                                           {"stats_collector": collectors[0]})
            self._n_renders = 1
            gts = []
            for k, (y0, y1, _c0, _c1) in enumerate(rows4):
                if y1 == y0:
                    gts.append(None)
                elif resident:
                    gts.append(self._gt_strip(k, y0, y1, True))
                else:
                    gt, ev = gt_ready[k]
                    torch.cuda.current_stream().wait_event(ev)
                    gt.record_stream(torch.cuda.current_stream())
                    gts.append(gt)
            l1_ssim = ops_.fused_l1_ssim_batched(images, gts, rows4)
            # sum over the local strips of (1 - lambda) Ll1 + lambda (1 - ssim)
            loss_sum = torch.dot(l1_ssim.reshape(-1), coef) + const
            Vp = int(view_start[-1])
            Pl = sum((r[1] - r[0]) * self.W for r in rows4)
            strategies_loop = []
        else:
            strategies_loop = strategies
        for k, st in enumerate(strategies_loop):
            rows = st.local_rows()
            if rows is None:
                continue
            self._n_renders += 1
            m2, rgb, co, radii, depths = redistributed[k]
            ck = (tuple(st.gpu_ids), tuple(st.division_pos), st.rank)
            if ck not in self._mask_cache:
                self._mask_cache[ck] = st.get_compute_locally(self.tile_x, self.device)
            cl = self._mask_cache[ck]
            image, *_ = ops_.render_gaussians(m2, co, rgb, depths, radii, cl, settings[k],
                                              {"stats_collector": collectors[k]})
            y0, y1 = st.local_pixel_rows(self.H)
            if self.border_exchange and self.world > 1 and len(st.gpu_ids) > 1:
                from . import border
                image, (r0, r1), _ = border.add_remote_border_rows(image, st, self.H, self.group)
                loss = ops_.fused_loss(image, self.gts_dev[k][:, r0:r1, :].contiguous(), r0, r1, self.lambda_dssim, y0, y1)
            else:
                if resident:
                    gt = self._gt_strip(k, y0, y1, True)
                else:
                    gt, ev = gt_ready[k]
                    torch.cuda.current_stream().wait_event(ev)
                    gt.record_stream(torch.cuda.current_stream())
                loss = ops_.fused_loss(image, gt, y0, y1, self.lambda_dssim)
            loss_sum = loss if loss_sum is None else loss_sum + loss
            Vp += m2.shape[0]
            Pl += (y1 - y0) * self.W
        self._mark("r render+loss")
        loss_sum.backward()
        self._mark("b4 backward (rest)")
        self._collectors, self._strategies = collectors, strategies
        self._counts = dict(Vp=Vp, P_local=Pl)
        self.iteration += 1
        self._feed_back_times(strategies, collectors)
        self._mark("t time feedback")
        if resident:
            return None
        self._loss_host.copy_(loss_sum.detach().reshape(1), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return float(self._loss_host[0])

    def _times_of(self, strategies, collectors, n_renders):
        """This rank's gpu_camera_running_time row for one step: the render time of each camera it rendered a strip of."""
        from .division import running_time_of
        B = len(strategies)
        mine = [-1.0] * B
        rows = [(st.local_rows()[1] - st.local_rows()[0]) if st.local_rows() is not None else 0 for st in strategies]
        if n_renders == 1 and sum(1 for r in rows if r) > 1:
            # one batched render served all local strips: its time is apportioned by strip height (the reference times
            # every camera's render separately, render_final __init__.py:1217-1288)
            t = running_time_of(collectors[0])
            for k, r in enumerate(rows):
                if r:
                    mine[k] = t * r / sum(rows)
        else:
            for k, r in enumerate(rows):
                if r:
                    c = collectors[k] if "forward_render_time" in collectors[k] else collectors[0]
                    mine[k] = running_time_of(c)
        return mine

    def _feedback_before_exchange(self):
        """feedback_lag > 0: hand the render times of the step `feedback_lag` steps back (its events have completed: the
        host is never more than one step ahead of the device) to the exchange, which all-gathers them behind the sizes."""
        self._ex.PIGGYBACK_IN, self._sent_feedback = None, None
        if self.feedback_lag > 0 and len(self._pending_feedback) >= self.feedback_lag:
            entry = self._pending_feedback.pop(0)
            self._ex.PIGGYBACK_IN = self._times_of(entry[0], entry[1], entry[3])
            self._sent_feedback = entry

    def _feedback_after_exchange(self):
        if self._sent_feedback is None:
            return
        strategies, _collectors, iteration, _n = self._sent_feedback
        times = self._ex.PIGGYBACK_OUT
        self._ex.PIGGYBACK_IN, self._sent_feedback = None, None
        if times is not None:
            finish_strategy(self.history, strategies, times.tolist(), iteration, self.world, self.H, self.W,
                            self.heuristic_decay)

    def _feed_back_times(self, strategies, collectors):
        """finish_strategy_final (workload_division.py:944-998) + the time all-gather (utils/general_utils.py:249-269):
        every rank contributes the render time of each camera it rendered a strip of; the per-row cost heuristic is
        rebuilt from them and the strips of a later step move.  Only where the reference's gate enables it (more than
        one rank, and not when whole <= 1080p images can be handed out)."""
        import torch.distributed as dist
        B = len(strategies)
        if not (self.load_balance and self.world > 1 and
                heuristics_update_enabled(self.iteration, self.world, B, self.H, self.W)):
            self._pending_feedback.clear()
            return
        if self.feedback_lag > 0:   # fed back later, on the size all-gather of a coming exchange (_feedback_before_exchange)
            self._pending_feedback.append((strategies, collectors, self.iteration, self._n_renders))
            return
        mine = self._times_of(strategies, collectors, self._n_renders)
        loc = torch.tensor(mine, dtype=torch.float32, device=self.device)
        allt = torch.empty((self.world * B,), dtype=torch.float32, device=self.device)
        dist.all_gather_into_tensor(allt, loc, group=self.group)
        times = allt.reshape(self.world, B).cpu().tolist()       # gpu_camera_running_time[gpu][camera]
        finish_strategy(self.history, strategies, times, self.iteration, self.world, self.H, self.W, self.heuristic_decay)

    def evaluate(self, cams, gts, batch_size=None, protocol="report"):
        """Render held-out views with the current parameters and compare them with their ground truth (forward only; no
        effect on training state: division history, iteration, pending timing feedback, gradients, means2D / radii of
        the last step and last_info() stay as they were).
        cams: camera dicts (synthetic.make_camera) or DeviceCamera, all of one image size and background; gts: one uint8
        (3,H,W) tensor per camera, host or device (with distributed_dataset_storage only rank 0 holds them: pass None
        elsewhere).  Views go through in batches of batch_size (default: the training batch size), each split into
        uniform tile-row strips over the ranks.  Every rank must call it with the same cameras.
        protocol: "report" = training_report's numbers (train_internal.py:466-479: clamped image, PSNR averaged over
        channels); "saved" = render.py + metrics.py's (the image quantised to 8 bits as saved to PNG, one PSNR over the
        image).  -> {"per_view": [{"uid", "l1", "psnr", "ssim"}, ...], "l1", "psnr", "ssim"} (means over the views)."""
        from . import evaluate as _ev
        return _ev.run(self, cams, gts, batch_size, protocol)

    GROUP_OF = {"xyz": "_xyz", "f_dc": "_features_dc", "f_rest": "_features_rest", "opacity": "_opacity",
                "scaling": "_scaling", "rotation": "_rotation"}

    def optimizer_groups(self, lrs=None):
        """The reference's six single-tensor groups over this trainer's parameters (scene/gaussian_model.py:257-292)."""
        lrs = lrs or {"xyz": 0.00016, "f_dc": 0.0025, "f_rest": 0.0025 / 20, "opacity": 0.05, "scaling": 0.005,
                      "rotation": 0.001}            # arguments/__init__.py:110-119
        return [{"params": [getattr(self.params, attr)], "lr": lrs[name], "name": name} for name, attr in self.GROUP_OF.items()]

    def adopt_parameters(self, new):
        """After densification / redistribution replaced the optimizer's tensors: new = {group name: nn.Parameter}."""
        for name, attr in self.GROUP_OF.items():
            setattr(self.params, attr, new[name])
        self.n_local = int(new["xyz"].shape[0])

    def last_info(self):
        """Realised sizes of the last step on this rank: V visible, V' splats rendered, R instances."""
        V = int((self._radii_local > 0).sum())
        R = ops.LAST_R_TOTAL
        return dict(V=V, Vp=self._counts["Vp"], P_local=self._counts["P_local"], R=R)

    def io_bytes_per_step(self):
        """(host->device, device->host) bytes of the last resident=False step: GT strips in, loss out
        (+ the 8-byte instance count each render reads back)."""
        return int(self._h2d), 4 + 8 * self._n_renders
