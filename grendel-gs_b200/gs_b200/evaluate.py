"""Held-out evaluation of a pipeline.Trainer's model: render views it does not train on and compare them with their
ground truth -- the numbers of train_internal.py:356-493 (training_report) and of render.py:87-138 -> metrics.py.

The reference renders one camera at a time, all-reduces every full (3,H,W) image across ranks and computes L1 / PSNR /
SSIM with about 20 torch kernels per view.  Here a batch of views goes through the training path's forward stages
(batched preprocess, splat exchange, batched render without a backward workspace); each rank evaluates only its own
tile-row strip, widened by the 5 halo rows the 11x11 SSIM window needs from the neighbouring strips, with one
gs_metrics_batched launch per batch; only the (views, 3, 3) fp64 sums are all-reduced, and they are read back once.

Host helpers (pure, CPU-testable): plan_window / exchange_halo (the halo rows of a strip) and metrics_from_sums (the two
protocols' derivations).  run() is the device driver behind Trainer.evaluate.
"""
import math

import numpy as np
import torch

from .border import HALF_WINDOW, _exchange
from .division import StrategyHistory, start_strategy

PROTOCOLS = ("report", "saved")


# ---------------------------------------------------------------------------------------------------------
# strip windows: a rank's counted rows [y0, y1) and the window [r0, r1) its SSIM filter sees
# ---------------------------------------------------------------------------------------------------------
class Window:
    """Rows of one camera's strip on this rank.  up / down: global ranks of the neighbouring strips (None at the image
    edges); n_up / n_down: halo rows received from them.  Derived only from the shared division, so the sizes a rank
    sends agree with what its neighbours expect."""
    __slots__ = ("y0", "y1", "r0", "r1", "up", "down", "n_up", "n_down")

    def __init__(self, y0, y1, r0, r1, up, down):
        self.y0, self.y1, self.r0, self.r1, self.up, self.down = y0, y1, r0, r1, up, down
        self.n_up, self.n_down = y0 - r0, r1 - y1

    def rows4(self):
        return (self.r0, self.r1, self.y0, self.y1)


def _strip_rows(strategy, c, H, block_y=16):
    return strategy.division_pos[c] * block_y, min(strategy.division_pos[c + 1] * block_y, H)


def plan_window(strategy, image_height):
    """Window of this rank's strip of one camera (None if it renders none): the strip plus up to HALF_WINDOW rows above and
    below, clipped to the image.  A neighbour must own every halo row it is asked for: only the last strip of an image
    can be thinner than HALF_WINDOW rows (H mod 16 in 1..4), and it has no strip below it."""
    c = strategy.rank
    if c < 0:
        return None
    H = int(image_height)
    y0, y1 = _strip_rows(strategy, c, H)
    up = strategy.gpu_ids[c - 1] if c > 0 else None
    down = strategy.gpu_ids[c + 1] if c + 1 < len(strategy.gpu_ids) else None
    r0 = max(0, y0 - HALF_WINDOW) if up is not None else y0
    r1 = min(H, y1 + HALF_WINDOW) if down is not None else y1
    if up is not None:
        u0, u1 = _strip_rows(strategy, c - 1, H)
        if y0 - r0 > u1 - u0:
            raise ValueError(f"strip rows [{u0},{u1}) are fewer than the {y0 - r0} halo rows the strip below needs")
    if down is not None:
        d0, d1 = _strip_rows(strategy, c + 1, H)
        if r1 - y1 > d1 - d0:
            raise ValueError(f"strip rows [{d0},{d1}) are fewer than the {r1 - y1} halo rows the strip above needs")
    return Window(y0, y1, r0, r1, up, down)


def _rows_padded(image, a, b, at_end):
    """(3, HALF_WINDOW, W) message holding rows [a, b) of `image` (b - a <= HALF_WINDOW), zero-padded at the end (top rows
    going up) or at the front (bottom rows going down): every message of the exchange has the same shape."""
    out = torch.zeros((image.shape[0], HALF_WINDOW, image.shape[2]), dtype=image.dtype, device=image.device)
    n = b - a
    if n > 0:
        if at_end:
            out[:, :n] = image[:, a:b]
        else:
            out[:, HALF_WINDOW - n:] = image[:, a:b]
    return out


def exchange_halo(image, win, group=None):
    """Fill the halo rows of `win` in `image` (3,H,W) (this rank's strip rows [y0, y1) rendered) from the neighbouring
    strips, forward only, over border._exchange.  Every rank that renders a strip of the camera must call it."""
    if win is None or (win.up is None and win.down is None):
        return image
    h = HALF_WINDOW
    send_up = _rows_padded(image, win.y0, min(win.y0 + h, win.y1), at_end=True)
    send_down = _rows_padded(image, max(win.y1 - h, win.y0), win.y1, at_end=False)
    recv_up, recv_down = _exchange(send_up, send_down, win.up, win.down, group)
    if recv_up is not None and win.n_up:
        image[:, win.r0:win.y0] = recv_up[:, h - win.n_up:]
    if recv_down is not None and win.n_down:
        image[:, win.y1:win.r1] = recv_down[:, :win.n_down]
    return image


# ---------------------------------------------------------------------------------------------------------
# sums -> metrics
# ---------------------------------------------------------------------------------------------------------
def _psnr(sse, n):
    with np.errstate(divide="ignore"):
        return float(-10.0 * np.log10(sse / n)) if sse > 0 else math.inf


def metrics_from_sums(sums, image_height, image_width, protocol="report"):
    """sums (N,3,3): [v][0][c] = sum |x-y|, [v][1][c] = sum (x-y)^2, [v][2][c] = sum ssim_map over channel c of view v.
    -> list of N dicts {"l1", "psnr", "ssim"}.
      "report" (train_internal.py:466-479): psnr(image (3,H,W), gt) views the image as (3, -1), so the value is the mean
               over channels of the per-channel PSNR, mean_c(-10 log10(SSE_c / HW)).
      "saved"  (metrics.py:26-36 on (1,3,H,W) tensors): one PSNR over the whole image, -10 log10(sum SSE / 3HW).
    Both: l1 = sum SAD / 3HW, ssim = sum SSIM / 3HW."""
    if protocol not in PROTOCOLS:
        raise ValueError(f"protocol must be one of {PROTOCOLS}, got {protocol!r}")
    s = np.asarray(sums, dtype=np.float64).reshape(-1, 3, 3)
    hw = float(image_height) * float(image_width)
    out = []
    for v in s:
        if protocol == "report":
            psnr = float(np.mean([_psnr(v[1][c], hw) for c in range(3)]))
        else:
            psnr = _psnr(float(v[1].sum()), 3.0 * hw)
        out.append({"l1": float(v[0].sum() / (3.0 * hw)), "psnr": psnr, "ssim": float(v[2].sum() / (3.0 * hw))})
    return out


# ---------------------------------------------------------------------------------------------------------
# device driver (Trainer.evaluate)
# ---------------------------------------------------------------------------------------------------------
def _check_inputs(trainer, dcams, gts, batch_size):
    """Every rejection that can be decided from values all ranks share (camera list, sizes, batch size): raised before
    any collective, identically on every rank."""
    from . import exchange, ops
    if len(dcams) == 0:
        raise ValueError("evaluate needs at least one camera")
    H, W = dcams[0].image_height, dcams[0].image_width
    for c in dcams:
        if (c.image_height, c.image_width) != (H, W):
            raise ValueError("all views of one evaluate call must have the same image size")
        if c.bg_host != dcams[0].bg_host:
            raise ValueError("all views of one evaluate call must have the same background")
    limit = min(exchange.MAX_CAMERAS, ops.MAX_VIEWS) if trainer.world > 1 else ops.MAX_VIEWS
    if not 1 <= batch_size <= limit:
        raise ValueError(f"batch_size must be in [1, {limit}] ({trainer.world} ranks), got {batch_size}")
    if gts is not None and len(gts) != len(dcams):
        raise ValueError(f"{len(dcams)} cameras but {len(gts)} ground-truth images")
    return H, W


def _check_gts(gts, H, W):
    """Rank-local checks of the ground-truth images (a rank without them has nothing to check)."""
    if gts is None:
        return None
    for k, g in enumerate(gts):
        if not isinstance(g, torch.Tensor) or g.dtype != torch.uint8:
            return TypeError(f"ground truth {k} must be a uint8 tensor (3,H,W)")
        if tuple(g.shape) != (3, H, W):
            return ValueError(f"ground truth {k} must be (3,{H},{W}), got {tuple(g.shape)}")
    return None


def run(trainer, cams, gts, batch_size=None, protocol="report"):
    """Trainer.evaluate: see its docstring."""
    import torch.distributed as dist
    from . import ops
    from .pipeline import DeviceCamera
    if protocol not in PROTOCOLS:
        raise ValueError(f"protocol must be one of {PROTOCOLS}, got {protocol!r}")
    dev, world, rank, group = trainer.device, trainer.world, trainer.rank, trainer.group
    dcams = [c if isinstance(c, DeviceCamera) else DeviceCamera(c, dev) for c in cams]
    bsz = len(trainer.dcams) if batch_size is None else int(batch_size)
    H, W = _check_inputs(trainer, dcams, gts, bsz)
    distributed = trainer.distributed_dataset_storage
    if gts is None and not (distributed and rank != 0):
        raise ValueError("ground-truth images are required on this rank")
    err = _check_gts(gts, H, W)
    if distributed and world > 1:   # only rank 0 holds the images: every rank learns its verdict before going on
        flag = torch.tensor([0 if err is None else 1], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MAX, group=group)
        if err is None and int(flag.item()):
            err = ValueError("rank 0 rejected the ground-truth images")
    if err is not None:
        raise err
    N = len(dcams)
    p = trainer.params
    tile_y, tile_x = (H + 15) // 16, (W + 15) // 16
    saved = protocol == "saved"
    sums = torch.zeros((N, 3, 3), dtype=torch.float64, device=dev)
    ex = trainer._ex
    keep_state = (ops.LAST_R_TOTAL, ops.STEP_STREAM, ex.PIGGYBACK_IN, ex.PIGGYBACK_OUT)
    ops.STEP_STREAM = torch.cuda.current_stream().cuda_stream
    ex.PIGGYBACK_IN = None      # timing feedback of training steps rides only on training exchanges
    try:
        with torch.no_grad():
            for i0 in range(0, N, bsz):
                views = dcams[i0:i0 + bsz]
                B = len(views)
                settings = [c.settings(p.active_sh_degree) for c in views]
                uids = [c.uid for c in views]
                # uniform strips, as the reference builds a fresh DivisionStrategyHistoryFinal per evaluation
                strategies, tasks = start_strategy(uids, StrategyHistory(uids, tile_y, world), world, rank)
                batched = ops.preprocess_gaussians_batched(p._xyz, p._features_dc, p._features_rest, p._scaling,
                                                           p._rotation, p._opacity, ops.pack_cameras(settings), W, H,
                                                           p.active_sh_degree)
                if world > 1:
                    cat, view_start, _cnt = ex.exchange_cat(*batched, strategies, settings, world, rank, group,
                                                            trainer._peer)
                    cl = torch.zeros((B, tile_y, tile_x), dtype=torch.uint8, device=dev)
                    for k, st in enumerate(strategies):
                        r = st.local_rows()
                        if r is not None:
                            cl[k, r[0]:r[1]] = 1
                    cl = cl.reshape(B, -1)
                else:
                    Pn = batched[0].shape[1]
                    cat = (batched[0].reshape(-1, 2), batched[1].reshape(-1, 3), batched[2].reshape(-1, 4),
                           batched[3].reshape(-1), batched[4].reshape(-1))
                    view_start = [k * Pn for k in range(B + 1)]
                    cl = None
                m2, rgb, co, radii, depths = cat
                images, _stats = ops.render_gaussians_batched(m2, co, rgb, depths, radii, cl, view_start, settings[0])
                wins = [plan_window(st, H) for st in strategies]
                for k, win in enumerate(wins):
                    exchange_halo(images[k], win, group)
                gt_win = _gt_windows(trainer, gts[i0:i0 + B] if gts is not None else None, wins, tasks, tile_y, H, W)
                rows4 = [w.rows4() if w is not None else (0, 0, 0, 0) for w in wins]
                sums[i0:i0 + B] = ops.image_metrics_batched(images, gt_win, rows4, saved=saved)
        if world > 1:
            dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
        host = sums.cpu().numpy()     # the call's one read of the metrics
    finally:
        ops.LAST_R_TOTAL, ops.STEP_STREAM, ex.PIGGYBACK_IN, ex.PIGGYBACK_OUT = keep_state
    per = metrics_from_sums(host, H, W, protocol)
    per_view = [dict(uid=c.uid, **m) for c, m in zip(dcams, per)]
    mean = lambda key: float(np.mean([m[key] for m in per]))
    return {"per_view": per_view, "l1": mean("l1"), "psnr": mean("psnr"), "ssim": mean("ssim")}


def _gt_windows(trainer, gts, wins, tasks, tile_y, H, W):
    """The (3, r1-r0, W) uint8 ground truth of every window on this rank's device.  With distributed_dataset_storage the
    rows come from rank 0 (gt_scatter.scatter_gt_strips), asked for one tile row beyond each strip so that they cover
    its halo."""
    dev = trainer.device
    if trainer.distributed_dataset_storage:
        from . import gt_scatter
        wide = [[(k, max(0, l - 1), min(tile_y, r + 1)) for k, l, r in ts] for ts in tasks]
        strips, _h2d = gt_scatter.scatter_gt_strips(gts if trainer.rank == 0 else W, wide, H, dev, trainer.rank,
                                                    trainer.world, trainer.group)
        base = {k: gt_scatter.coverage(l, r, H)[0] for k, l, r in wide[trainer.rank]}
        return [None if w is None else strips[k][:, w.r0 - base[k]:w.r1 - base[k]].contiguous()
                for k, w in enumerate(wins)]
    return [None if w is None else gts[k][:, w.r0:w.r1].to(dev, non_blocking=True).contiguous()
            for k, w in enumerate(wins)]
