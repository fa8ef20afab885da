"""CPU tests of held-out evaluation: the metrics oracle against the reference's own L1 / PSNR / SSIM and PNG round trip
(tests/golden/metrics.npz), closed-form cases, strip windows with halo rows, and the halo exchange of gs_b200.evaluate
over a real gloo group."""
import os
import socket

import numpy as np
import pytest
import torch

from gs_b200 import division, evaluate
from oracle import metrics_oracle as mo

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "metrics.npz")


def _golden():
    """One dict per golden case: image, gt, saved_q, saved_gt_q and {report,saved}_{l1,psnr,ssim}_."""
    g = np.load(GOLDEN)
    keys = ["image", "gt", "saved_q", "saved_gt_q"] + [f"{p}_{m}_" for p in ("report", "saved") for m in ("l1", "psnr", "ssim")]
    return [{k: g[f"{k}{i}"] for k in keys} for i in range(int(g["n"]))]


@pytest.mark.parametrize("protocol", ["report", "saved"])
def test_oracle_reproduces_the_reference_metrics(protocol):
    for c in _golden():
        img, gt = c["image"], c["gt"]
        H, W = gt.shape[1:]
        m = mo.derive(mo.metric_sums(img, gt, saved=protocol == "saved"), H, W, protocol)
        assert abs(m["l1"] / float(c[f"{protocol}_l1_"]) - 1) <= 1e-6
        assert abs(m["psnr"] - float(c[f"{protocol}_psnr_"])) <= 1e-4
        assert abs(m["ssim"] - float(c[f"{protocol}_ssim_"])) <= 1e-5
        # the pure derivation of the product agrees with the oracle's
        e = evaluate.metrics_from_sums(mo.metric_sums(img, gt, saved=protocol == "saved")[None], H, W, protocol)[0]
        for key in ("l1", "psnr", "ssim"):
            assert abs(e[key] - m[key]) <= 1e-12 * max(1.0, abs(m[key]))


def test_quantisation_is_bit_identical_to_the_png_round_trip():
    for c in _golden():
        assert np.array_equal(mo.quantise_saved(mo.metric_input(c["image"])), c["saved_q"])
        assert np.array_equal(c["saved_gt_q"], c["gt"])       # the ground truth survives its own round trip


def test_closed_form_cases():
    rng = np.random.default_rng(3)
    gt = rng.integers(0, 256, (3, 21, 34), dtype=np.uint8)
    same = gt.astype(np.float32) / np.float32(255)
    for protocol in ("report", "saved"):
        m = evaluate.metrics_from_sums(mo.metric_sums(same, gt, saved=protocol == "saved")[None], 21, 34, protocol)[0]
        assert m["psnr"] == float("inf") and m["l1"] == 0.0 and abs(m["ssim"] - 1.0) <= 1e-12
    flat = np.full((3, 21, 34), 100, dtype=np.uint8)
    d = 0.0625                                               # exact in fp32: the offset survives the subtraction
    img = flat.astype(np.float32) / np.float32(255) + np.float32(d)
    s = mo.metric_sums(img, flat)
    for protocol in ("report", "saved"):
        m = evaluate.metrics_from_sums(s[None], 21, 34, protocol)[0]
        assert abs(m["psnr"] - (-20 * np.log10(d))) <= 1e-5
        assert abs(m["l1"] - d) <= 1e-7


def _strips(division_pos, H):
    return [(division_pos[c] * 16, min(division_pos[c + 1] * 16, H)) for c in range(len(division_pos) - 1)]


@pytest.mark.parametrize("H,division_pos", [(100, [0, 3, 7]), (100, [0, 2, 4, 7]), (1060, [0, 66, 67]),
                                            (1060, [0, 33, 66, 67]), (37, [0, 1, 2, 3])])
@pytest.mark.parametrize("saved", [False, True])
def test_strip_windows_sum_to_the_full_image(H, division_pos, saved):
    """A strip's window [r0, r1) plus counted rows [y0, y1) from plan_window: the strip sums add up to the whole image's,
    also when the last strip is thinner than the half window (H = 1060: 4 rows; H = 37: 5 rows)."""
    W = 19
    rng = np.random.default_rng(H + len(division_pos))
    img = rng.uniform(-0.1, 1.1, (3, H, W)).astype(np.float32)
    gt = rng.integers(0, 256, (3, H, W), dtype=np.uint8)
    full = mo.metric_sums(img, gt, saved)
    world = len(division_pos) - 1
    tot = np.zeros((3, 3))
    for me in range(world):
        st = division.DivisionStrategy(0, list(range(world)), division_pos, (H + 15) // 16, me)
        win = evaluate.plan_window(st, H)
        assert (win.y0, win.y1) == _strips(division_pos, H)[me]
        tot += mo.metric_sums(img, gt[:, win.r0:win.r1], saved, win.r0, win.r1, win.y0, win.y1)
    np.testing.assert_allclose(tot, full, rtol=1e-12, atol=0)


def test_plan_window_clips_the_halo_to_the_image():
    # the last strip holds 2 rows (H = 18): the window of the strip above stops at H, 2 rows below its strip
    st = division.DivisionStrategy(0, [0, 1], [0, 1, 2], 2, 0)
    assert evaluate.plan_window(st, 18).n_down == 2           # last strip has 2 rows: the window stops at H
    st = division.DivisionStrategy(0, [0, 1, 2], [0, 1, 2, 3], 3, 1)
    w = evaluate.plan_window(st, 34)
    assert (w.r0, w.y0, w.y1, w.r1) == (11, 16, 32, 34)


# ---------------------------------------------------------------------------------------------------
# halo exchange over gloo, world 2 and 3
# ---------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _halo_worker(rank, world, port, cases, q):
    import torch.distributed as dist
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    out = []
    for H, W, division_pos, saved in cases:
        rng = np.random.default_rng(H * 7 + W)
        img = rng.uniform(-0.1, 1.1, (3, H, W)).astype(np.float32)
        gt = rng.integers(0, 256, (3, H, W), dtype=np.uint8)
        tile_y = (H + 15) // 16
        if division_pos is None:     # uniform strips, as evaluate builds them
            st = division.start_strategy([0], division.StrategyHistory([0], tile_y, world), world, rank)[0][0]
        else:
            st = division.DivisionStrategy(0, list(range(world)), division_pos, tile_y, rank)
        win = evaluate.plan_window(st, H)
        mine = torch.zeros((3, H, W), dtype=torch.float32)   # rows outside the strip: not rendered here
        mine[:, win.y0:win.y1] = torch.from_numpy(img[:, win.y0:win.y1])
        evaluate.exchange_halo(mine, win)
        ok_rows = torch.equal(mine[:, win.r0:win.r1], torch.from_numpy(img[:, win.r0:win.r1]))
        s = torch.from_numpy(mo.metric_sums(mine.numpy(), gt[:, win.r0:win.r1], saved, win.r0, win.r1, win.y0, win.y1))
        dist.all_reduce(s, op=dist.ReduceOp.SUM)
        full = mo.metric_sums(img, gt, saved)
        out.append((bool(ok_rows), float(np.max(np.abs(s.numpy() - full) / np.abs(full))), st.division_pos))
    q.put((rank, out))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_halo_exchange_over_gloo_gives_full_image_metrics(world):
    """Each rank holds only its strip of the image, plans its window, exchanges the halo rows with its neighbours, runs
    the oracle on its window and SUM-all-reduces: the result is the full-image oracle.  Uniform strips, and a
    constructed division whose last strip is 4 rows (H = 1060), which uniform strips never produce."""
    import torch.multiprocessing as mp
    last = [0, 66, 67] if world == 2 else [0, 30, 66, 67]
    cases = [(100, 23, None, False), (1060, 9, None, True), (1060, 9, last, False), (1060, 9, last, True)]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_halo_worker, args=(r, world, port, cases, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=180) for _ in range(world)), key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
    for rank, out in res:
        for (ok_rows, rel, pos), case in zip(out, cases):
            assert ok_rows, (rank, case)
            assert rel <= 1e-12, (rank, case, rel)
    assert res[0][1][2][2] == last
