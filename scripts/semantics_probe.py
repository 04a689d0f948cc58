"""Probe: the configs[1] pair (8192^2, 6 scales, 5 warps, lambda 0.15) solved in both solver modes in one run --
TVL1_SEMANTICS_CPU (cv::DualTVL1OpticalFlow, inner 30 x outer 10) and TVL1_SEMANTICS_CUDA (cv::cuda's flat loop,
N = 300).  Frames resident on the device (tvl1_calc_u8); per mode one warm-up solve, then `--steps` timed solves
(CUDA events around each solve), then one solve with per-stage events for the stage split.

    python scripts/semantics_probe.py [--size 8192] [--steps 3] [--out FILE.json]
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
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out")
    a = ap.parse_args()
    N.require_device()
    n = a.size
    I0, I1 = synth.make_pair(n, n, seed=7, dx=1.3, dy=-0.7, shear=4.0 / n, margin=32)
    f0, f1 = N.DevBuf(n * n).upload(I0), N.DevBuf(n * n).upload(I1)
    du, dv = N.DevBuf(n * n * 4), N.DevBuf(n * n * 4)
    common = dict(lambda_=0.15, nscales=6, warps=5)
    modes = {"cpu": N.default_params(inner_iterations=30, outer_iterations=10, median_filtering=5, **common),
             "cuda": N.default_params(semantics="cuda", iterations=300, **common)}
    res = {"workload": "configs[1]: %dx%d synthetic pair (synth.make_pair seed 7, shift 1.3/-0.7 px, shear 4 px), "
                       "6 scales, 5 warps, lambda 0.15, epsilon 0.01" % (n, n)}
    res.update(card())
    flows = {}
    for name, p in modes.items():
        s = N.Solver(p)
        s.calc_device(f0.ptr, n, f1.ptr, n, n, n, du.ptr, dv.ptr, n * 4)          # warm-up
        ms = []
        for _ in range(a.steps):
            s.calc_device(f0.ptr, n, f1.ptr, n, n, n, du.ptr, dv.ptr, n * 4)
            ms.append(s.stats.ms_total)
        st = s.stats
        its = st.iters_array()
        out = {"ms_per_pair": ms, "ms_median": float(np.median(ms)), "total_iterations": int(st.total_iterations),
               "iterations_level0": its[0].tolist(), "launches": int(st.launches),
               "mpx_per_s": n * n / 1e6 / (float(np.median(ms)) / 1e3)}
        s.set_timing(True)
        s.calc_device(f0.ptr, n, f1.ptr, n, n, n, du.ptr, dv.ptr, n * 4)
        st = s.stats
        out["stages_ms"] = {"total": st.ms_total, "pyramid": st.ms_pyramid, "warp": st.ms_warp, "iterate": st.ms_iterate,
                            "median": st.ms_median, "other": st.ms_other}
        res[name] = out
        flows[name] = du.download((n, n), np.float32), dv.download((n, n), np.float32)
        s.close()
    ut, vt = synth.true_flow(n, n, shear=4.0 / n)
    for name, (u, v) in flows.items():
        res[name]["mean_epe_vs_truth_interior"] = float(np.hypot(u - ut, v - vt)[32:-32, 32:-32].mean())
    d = np.hypot(flows["cpu"][0] - flows["cuda"][0], flows["cpu"][1] - flows["cuda"][1])
    res["cpu_vs_cuda_flow_px"] = {"mean": float(d.mean()), "max": float(d.max())}
    res["warp_ms_cuda_over_cpu"] = res["cuda"]["stages_ms"]["warp"] / max(res["cpu"]["stages_ms"]["warp"], 1e-9)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
