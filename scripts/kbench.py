"""Developer micro-benchmark of single stage kernels through the stage-level C ABI.
usage: python scripts/kbench.py <warp|median|iterate|outer|all> [size] [reps]"""
import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from fibsem_optflow_b200 import _native as N, synth

def timeit(fn, reps):
    fn(); N.check(N.lib().tvl1_dev_sync(0))
    t = time.perf_counter()
    for _ in range(reps): fn()
    N.check(N.lib().tvl1_dev_sync(0))
    return (time.perf_counter() - t) / reps

def main():
    which = sys.argv[1] if len(sys.argv) > 1 else "all"
    n = int(sys.argv[2]) if len(sys.argv) > 2 else 4096
    reps = int(sys.argv[3]) if len(sys.argv) > 3 else 10
    L = N.lib()
    I0, I1 = synth.make_pair(n, n, seed=7, shear=4.0 / n)
    rng = np.random.default_rng(0)
    f0 = N.Plane(n, n, 0, I0.astype(np.float32)); f1 = N.Plane(n, n, 0, I1.astype(np.float32))
    ut, vt = synth.true_flow(n, n, shear=4.0 / n)
    # a smooth perturbation of the true flow, like a solver state a few iterations before the stop
    yy, xx = np.mgrid[0:n, 0:n].astype(np.float32)
    du = (0.05 * np.sin(xx / 37.0) * np.cos(yy / 53.0)).astype(np.float32)
    u1 = N.Plane(n, n, 0, ut + du)
    u2 = N.Plane(n, n, 0, vt - du)
    del yy, xx, du
    outs = [N.Plane(n, n) for _ in range(4)]
    px = n * n
    # the warp always runs once: the iteration kernels must see real image gradients (with zero
    # planes the threshold never takes its division branch and they look ~9 % faster than they are)
    N.check(L.tvl1_k_warp(f0.ptr, f1.ptr, u1.ptr, u2.ptr, n, n, f0.pitch, None,
                          outs[0].ptr, outs[1].ptr, None, outs[2].ptr, None))
    if which in ("warp", "all"):
        dt = 1e9
        for _ in range(reps):
            N.check(L.tvl1_k_warp(f0.ptr, f1.ptr, u1.ptr, u2.ptr, n, n, f0.pitch, None,
                                  outs[0].ptr, outs[1].ptr, None, outs[2].ptr, None))
            dt = min(dt, N.k_last_ms() * 1e-3)
        print(f"k_warp    {n}^2: {dt*1e3:.3f} ms  {px/dt/1e9:.1f} Gpx/s  {40*px/dt/1e9:.0f} GB/s (40 B/px model)")
    if which in ("median", "all"):
        dt = 1e9
        for _ in range(reps):
            N.check(L.tvl1_k_median5(u1.ptr, n, n, u1.pitch, outs[0].ptr, None))
            dt = min(dt, N.k_last_ms() * 1e-3)
        print(f"k_median5 {n}^2 (1 plane): {dt*1e3:.3f} ms  {px/dt/1e9:.1f} Gpx/s  {8*px/dt/1e9:.0f} GB/s (8 B/px)")
    if which in ("iterate", "all"):
        p = [N.Plane(n, n) for _ in range(4)]
        best = 1e9
        for _ in range(3):
            N.check(L.tvl1_k_iterate(outs[0].ptr, outs[1].ptr, outs[0].ptr, outs[2].ptr, u1.ptr, u2.ptr, p[0].ptr, p[1].ptr,
                                     p[2].ptr, p[3].ptr, n, n, u1.pitch, 0.045, 0.3, 0.25 / 0.3, 40, None, None))
            best = min(best, N.k_last_ms() / 40)
        dt = best * 1e-3
        print(f"k_iterate {n}^2: {dt*1e6:.1f} us/iter  {64*px/dt/1e9:.0f} GB/s (64 B/px model)")
        best = 1e9
        for _ in range(3):
            N.check(L.tvl1_k_iterate_fused2(outs[0].ptr, outs[1].ptr, outs[0].ptr, outs[2].ptr, u1.ptr, u2.ptr, p[0].ptr, p[1].ptr,
                                            p[2].ptr, p[3].ptr, n, n, u1.pitch, 0.045, 0.3, 0.25 / 0.3, 40, None, None))
            best = min(best, N.k_last_ms() / 40)
        dt = best * 1e-3
        print(f"k_iterate2 {n}^2: {dt*1e6:.1f} us/iter  {64*px/dt/1e9:.0f} GB/s (64 B/px model)")
    if which in ("outer", "iterate", "all"):
        # the shipped kernel: NIT iterations in ONE cooperative k_outer launch
        NIT = int(os.environ.get("KB_OUTER_ITERS", 30))
        if which == "outer":
            p = [N.Plane(n, n) for _ in range(4)]
        best = 1e9
        for _ in range(reps if which == "outer" else 3):
            N.check(L.tvl1_k_outer(outs[0].ptr, outs[1].ptr, outs[0].ptr, outs[2].ptr, u1.ptr, u2.ptr, p[0].ptr, p[1].ptr,
                                   p[2].ptr, p[3].ptr, n, n, u1.pitch, 0.045, 0.3, 0.25 / 0.3, NIT, None, None))
            best = min(best, N.k_last_ms() / NIT)
        dt = best * 1e-3
        print(f"k_outer   {n}^2 ({NIT} iterations per launch): {dt*1e6:.1f} us/iter  {64*px/dt/1e9:.0f} GB/s (64 B/px model)")

if __name__ == "__main__":
    main()
