"""-m gpu: round 3's segment-parallel backward (k_blend_bwd_seg3, the default) against round 2's (k_blend_bwd_seg,
gs_debug_set(GS_DEBUG_BWD_SEG_R2)) and the oracle, on the parity cases of test_backward_kernels_agree.  Both kernels
compute the same nine sums per (splat, tile) bit for bit; round 3 reduces two splats' sums together, so the gradients
differ only by the order of fp32 additions (and the RED order already makes two runs of either kernel differ).  The
bar is that of the segment-vs-tile comparison; both kernels' distances to the oracle are printed side by side."""
import numpy as np
import pytest

import gpu_util as gu
from gs_b200 import synthetic as syn

pytestmark = pytest.mark.gpu

OUTLIER_FRAC = 2e-4


@pytest.fixture(scope="module")
def o32():
    import os
    from oracle.oracle import Oracle
    return Oracle(np.float32, threads=max(1, (os.cpu_count() or 8) // 2))


@pytest.mark.parametrize("n,W,H,rad,bg", [(20000, 320, 200, 7.0, (0.0, 0.0, 0.0)), (3000, 96, 64, 16.0, (0.3, 0.1, 0.7)),
                                          (30000, 200, 120, 9.0, (0.2, 0.5, 0.9)), (60000, 100, 70, 12.0, (0.1, 0.2, 0.3))])
def test_seg3_backward_agrees_with_seg2(o32, n, W, H, rad, bg):
    from gs_b200 import _lib
    cam = syn.make_camera(W, H, yaw_deg=3.0, sh_degree=3)
    sc = syn.make_scene(n, W, H, seed=3, radius_px=rad)
    ref = o32.preprocess_forward(sc["means3D"], sc["scales"], sc["rotations"], sc["shs"], sc["opacities"], cam)
    T = ((H + 15) // 16) * ((W + 15) // 16)
    cl = np.ones(T, np.uint8)
    rf = o32.render_forward(H, W, ref["means2D"], ref["conic_opacity"], ref["rgb"], ref["depths"], ref["radii"], cl, bg)
    f = gu.render_forward(H, W, gu.to_dev(ref["means2D"]), gu.to_dev(ref["conic_opacity"]), gu.to_dev(ref["rgb"]),
                          gu.to_dev(ref["depths"]), gu.to_dev(ref["radii"]), gu.to_dev(cl), bg)
    g = np.random.default_rng(2).normal(size=(3, H, W)).astype(np.float32)
    rb = o32.render_backward(H, W, ref["means2D"], ref["conic_opacity"], ref["rgb"], bg, rf, g)
    new = gu.render_backward(f, gu.to_dev(g))
    old_flags = _lib.debug_set(_lib.DEBUG_BWD_SEG_R2)
    try:
        old = gu.render_backward(f, gu.to_dev(g))
    finally:
        _lib.debug_set(old_flags)
    untouched = ~np.isin(np.arange(n), rf["ids"])
    for k in ("means2D", "conic_opacity", "rgb"):
        a, b = gu.npy(new[k]), gu.npy(old[k])
        assert np.isfinite(a).all()
        frac_new, worst_new = gu.rel_report(f"seg3.{k}", a, rb[k])
        frac_old, worst_old = gu.rel_report(f"seg2.{k}", b, rb[k])
        print(f"[seg3-vs-seg2] {k}: outside_tol {frac_new:.2e} (seg2 {frac_old:.2e})  worst_rel {worst_new:.3e} "
              f"(seg2 {worst_old:.3e})")
        assert frac_new <= 5 * OUTLIER_FRAC, k
        frac2, _ = gu.rel_report(f"seg3.vs_seg2.{k}", a, b)
        assert frac2 <= 5 * OUTLIER_FRAC, k
        assert (a[untouched] == 0).all()
