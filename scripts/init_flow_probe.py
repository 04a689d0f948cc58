"""Probe: what a warm start costs and saves on the configs[1] pair size (8192^2, 6 scales, 5 warps, lambda 0.15,
CPU-class semantics).  Two chained pairs of a synthetic stack (synth.make_stack): pair A = slices (0, 1), pair
B = slices (1, 2).  Pair B is solved three ways, frames resident on the device:

    u8     tvl1_calc_u8
    zero   tvl1_calc_ex with a zero initial flow
    warm   tvl1_calc_ex started from pair A's flow (the previous pair of a chained stack)

One warm-up solve per case, then `--steps` rounds that run the three cases in turn (CUDA events around each solve,
stats.ms_total), so that drift of the shared machine hits all three alike.

    python scripts/init_flow_probe.py [--size 8192] [--steps 5] [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

from fibsem_optflow_b200 import _native as N, synth  # noqa: E402


def card():
    try:
        q = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, limit = [x.strip() for x in q.splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": limit}
    except Exception as e:   # the numbers still stand; the card is then unnamed in the output
        return {"gpu": "unknown (%s)" % e, "power_limit": "unknown"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=8192)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out")
    a = ap.parse_args()
    N.require_device()
    n, seed = a.size, 11
    slices = synth.make_stack(2, n, n, seed=seed)
    shifts = np.random.default_rng(seed + 1).uniform(-1.5, 1.5, size=(2, 2))   # make_stack's per-slice offsets
    f = [N.DevBuf(n * n).upload(s) for s in slices]
    du, dv = N.DevBuf(n * n * 4), N.DevBuf(n * n * 4)          # solve output
    iu, iv = N.DevBuf(n * n * 4), N.DevBuf(n * n * 4)          # initial flow: zero, then pair A's flow
    p = N.default_params(lambda_=0.15, nscales=6, warps=5, inner_iterations=30, outer_iterations=10, median_filtering=5)
    s = N.Solver(p)
    st = s.stats
    # pair A's flow, the warm start of pair B
    s.calc_device(f[0].ptr, n, f[1].ptr, n, n, n, iu.ptr, iv.ptr, n * 4)
    flow_a = iu.download((n, n), np.float32), iv.download((n, n), np.float32)
    zu, zv = N.DevBuf(n * n * 4).zero(), N.DevBuf(n * n * 4).zero()

    def u8():
        s.calc_device(f[1].ptr, n, f[2].ptr, n, n, n, du.ptr, dv.ptr, n * 4)

    def zero():
        s.calc_ex_device(N.FRAME_U8, f[1].ptr, n, f[2].ptr, n, n, n, zu.ptr, zv.ptr, n * 4, du.ptr, dv.ptr, n * 4)

    def warm():
        s.calc_ex_device(N.FRAME_U8, f[1].ptr, n, f[2].ptr, n, n, n, iu.ptr, iv.ptr, n * 4, du.ptr, dv.ptr, n * 4)

    cases = {"u8": u8, "zero": zero, "warm": warm}
    res = {"workload": "configs[1] size: %dx%d chained synthetic stack (synth.make_stack seed %d), pair (1, 2); 6 scales, "
                       "5 warps, lambda 0.15, inner 30 x outer 10, median 5 (CPU-class semantics); warm = started "
                       "from pair (0, 1)'s flow" % (n, n, seed)}
    res.update(card())
    ms = {k: [] for k in cases}
    for k, fn in cases.items():   # warm-up
        fn()
    for _ in range(a.steps):
        for k, fn in cases.items():
            fn()
            ms[k].append(st.ms_total)
    tu, tv = -np.float32(shifts[1, 0]), -np.float32(shifts[1, 1])   # pair B's true flow (a uniform shift)
    flows = {}
    for k, fn in cases.items():
        fn()
        its = st.iters_array()
        u, v = du.download((n, n), np.float32), dv.download((n, n), np.float32)
        flows[k] = u, v
        res[k] = {"ms_per_pair": ms[k], "ms_median": float(np.median(ms[k])), "total_iterations": int(st.total_iterations),
                  "iterations_level0": its[0].tolist(), "iterations_per_level": its.sum(axis=1).tolist(),
                  "launches": int(st.launches),
                  "mean_epe_vs_truth_interior": float(np.hypot(u - tu, v - tv)[32:-32, 32:-32].mean())}
    res["zero_minus_u8_ms_median"] = res["zero"]["ms_median"] - res["u8"]["ms_median"]
    res["warm_minus_u8_ms_median"] = res["warm"]["ms_median"] - res["u8"]["ms_median"]
    res["zero_equals_u8_bitwise"] = bool(np.array_equal(flows["zero"][0], flows["u8"][0]) and
                                         np.array_equal(flows["zero"][1], flows["u8"][1]))
    res["pair_a_mean_flow"] = [float(flow_a[0].mean()), float(flow_a[1].mean())]
    s.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
