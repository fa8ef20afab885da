"""Compares three `bench.py --dump-outputs` directories: two runs of round 2's backward kernel (GS_B200_DEBUG_FLAGS=16)
and one of round 3's (the default).

    python profiles/r3_compare_outputs.py OLD_A OLD_B NEW

The loss does not depend on the backward, so it must be bit-identical.  Every gradient array differs between two runs of
the SAME kernel already (red.global order); the new kernel passes when its distance to the old one is at most twice that
run-to-run distance, per array, in max |diff| and in RMS diff.  Prints one line per array and exits 1 on a failure."""
import os
import sys

import numpy as np


def main(old_a, old_b, new):
    names = sorted(f[:-4] for f in os.listdir(old_a) if f.endswith(".npy"))
    ok = True
    for k in names:
        a, b, n = (np.load(os.path.join(d, k + ".npy")).astype(np.float64) for d in (old_a, old_b, new))
        if k in ("loss", "sample_rows", "radii"):
            same = np.array_equal(a, n) and np.array_equal(a, b)
            ok &= same
            print(f"{k:22s} bit-identical: {same}" + (f"   ({float(a):.9f})" if k == "loss" else ""))
            continue
        d_oo, d_no = np.abs(a - b), np.abs(n - a)
        r_oo, r_no = float(np.sqrt((d_oo ** 2).mean())), float(np.sqrt((d_no ** 2).mean()))
        m_oo, m_no = float(d_oo.max()), float(d_no.max())
        scale = float(np.sqrt((a ** 2).mean()))
        good = m_no <= 2 * m_oo and r_no <= 2 * r_oo
        ok &= good
        print(f"{k:22s} rms {scale:.3e}   old-vs-old max {m_oo:.3e} rms {r_oo:.3e}   new-vs-old max {m_no:.3e} "
              f"rms {r_no:.3e}   ratio max {m_no / max(m_oo, 1e-300):.2f} rms {r_no / max(r_oo, 1e-300):.2f}   "
              f"{'ok' if good else 'FAIL'}")
    print("all within 2x the run-to-run difference" if ok else "FAILED")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main(*sys.argv[1:4]))
