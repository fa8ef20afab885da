"""Round 3: issued-instruction prediction of the segment-parallel backward blend, round 2's kernel (k_blend_bwd_seg) against
round 3's (k_blend_bwd_seg3), on a 1/16-scale copy of c2 (125k Gaussians at 480x270, the scene of predict_seg_variants.py).

The walk is replayed exactly as the kernels do it: per (tile, 128-entry segment) unit, 32-entry staging passes; per
staged entry the 8x4-block mask of the forward's row-band cull (fp32 transcription from tests/test_band_cull.py), trimmed
to the blocks that still have a live pixel at that depth; per block in the mask the vote "some lane passes the exponent
test"; per entry whether any block passed (the reduction tail runs).  Costs per event are warp instructions counted in
the sm_100a SASS of the two kernels (profiles/r3_sass_blend_bwd.md).  Also reports the fraction of staged entries whose
trimmed mask is empty -- round 2 pays a loop head for each of them, round 3's compacted staging none.
Analysis tool: imports oracle/ and tests/, not product code.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "grendel-gs_b200"), os.path.join(ROOT, "tests")]
from gs_b200 import synthetic as syn  # noqa: E402
from oracle.oracle import Oracle      # noqa: E402
from test_band_cull import ellipse_bands, make_records  # noqa: E402

F = np.float32
SEG_K = 32 * 4
# warp instructions per event, read off the SASS (see profiles/r3_sass_blend_bwd.md); the per-unit set-up and per-pass
# staging costs are rough estimates (together under 1 instruction per instance)
COST = {
    "r2": dict(unit=120, pass_=40, empty=13, head=34, bit=2, block=11, body=31, tail=70, pair_extra=0),
    "r3": dict(unit=130, pass_=55, empty=0, head=27, bit=2, block=11, body=29, tail=45, pair_extra=46),
}


def main():
    W, H, n = 480, 270, 125_000
    cam = syn.make_camera(W, H)
    sc = syn.make_scene(n, W, H, seed=0)
    o = Oracle(np.float32, threads=max(1, (os.cpu_count() or 8) // 2))
    pre = o.preprocess_forward(sc["means3D"], sc["scales"], sc["rotations"], sc["shs"], sc["opacities"], cam)
    gx, gy = (W + 15) // 16, (H + 15) // 16
    fwd = o.render_forward(H, W, pre["means2D"], pre["conic_opacity"], pre["rgb"], pre["depths"], pre["radii"],
                           np.ones(gx * gy, np.uint8), (0, 0, 0))
    rec = make_records(pre["means2D"], pre["conic_opacity"])
    ids, ranges = fwd["ids"].astype(np.int64), fwd["ranges"].reshape(-1, 2)
    R = int(fwd["R"])
    yy, xx = np.meshgrid(np.arange(16), np.arange(16), indexing="ij")
    lx, ly = xx.reshape(-1), yy.reshape(-1)
    blk_of_pix = (ly // 4) * 2 + lx // 8            # 8x4 block b = 2 * band + column half
    ev = dict(units=0, passes=0, staged=0, empty=0, nonempty=0, blocks=0, passed=0, tails=0, pairs=0)
    for tile in range(gx * gy):
        beg, end = ranges[tile]
        X0, Y0 = (tile % gx) * 16, (tile // gx) * 16
        px, py = X0 + lx, Y0 + ly
        inside = (px < W) & (py < H)
        last = np.where(inside, fwd["n_contrib"][np.minimum(py, H - 1), np.minimum(px, W - 1)], 0).astype(np.int64)
        tl = int(last.max())
        if end <= beg or tl == 0:
            continue
        g = ids[beg:end][:tl]
        bands = ellipse_bands(rec, g, X0, Y0)
        mask = np.zeros((8, tl), bool)
        for q in range(4):
            bl, bh = bands[q]
            for half in range(2):
                mask[2 * q + half] = (bh >= 8 * half) & (bl <= 8 * half + 7)
        dx = rec["mx"][g][None, :] - px[:, None].astype(F)
        dy = rec["my"][g][None, :] - py[:, None].astype(F)
        power = dx * (rec["az"][g] * dx + rec["aw"][g] * dy) + rec["bx"][g] * dy * dy
        passes_px = (power >= rec["thr"][g]) & (power <= 0) & (np.arange(tl)[None, :] < last[:, None])
        for s in range((tl + SEG_K - 1) // SEG_K):
            sb = s * SEG_K
            cnt = min(SEG_K, tl - sb)
            live = np.clip(last - sb, 0, SEG_K)
            ev["units"] += 1
            ev["passes"] += (cnt + 31) // 32
            pend = False
            for i in range(cnt):
                e = sb + i
                m = np.array([mask[b, e] and i < live[blk_of_pix == b].max() for b in range(8)])
                ev["staged"] += 1
                if not m.any():
                    ev["empty"] += 1
                    continue
                ev["nonempty"] += 1
                ev["blocks"] += int(m.sum())
                full = False
                for b in np.nonzero(m)[0]:
                    if passes_px[blk_of_pix == b, e].any():
                        ev["passed"] += 1
                        full = True
                if full:
                    ev["tails"] += 1
                    ev["pairs"] += int(pend)
                    pend = not pend
    print(f"scene: {n} Gaussians @ {W}x{H}: R = {R} instances")
    print("events: " + ", ".join(f"{k} {v}" for k, v in ev.items()))
    print(f"staged entries with an empty trimmed mask: {ev['empty'] / ev['staged']:.3f} of {ev['staged']}")
    print(f"per instance: blocks in the mask {ev['blocks'] / R:.2f}, blocks past the vote {ev['passed'] / R:.2f}, "
          f"reduction tails {ev['tails'] / R:.2f}")
    for name, c in COST.items():
        tot = (c["unit"] * ev["units"] + c["pass_"] * ev["passes"] + c["empty"] * ev["empty"] +
               (c["head"] + 7 * c["bit"]) * ev["nonempty"] + c["block"] * ev["blocks"] + c["body"] * ev["passed"] +
               c["tail"] * ev["tails"] + c["pair_extra"] * ev["pairs"])
        print(f"{name}: {tot:.3e} warp instructions (x16 for c2: {16 * tot:.3e}), {tot / R:.1f} per instance")


if __name__ == "__main__":
    main()
