"""Developer probe: tvl1_calc_batch_ex in the modes tvl1_calc_batch_u8 refuses, against the same pairs solved one by
one through tvl1_calc_u8 on a handle of the same parameters, in one run.

Modes: cv::cuda semantics ("semantics": "cuda", wrapper defaults otherwise: 300 iterations per (level, warp)) on the
ROI strips 100 x 4096 and 200 x 4096 (top / bottom ROI strips of gen_cross_file_list.py jobs) and a 2048^2 pair; and
the CPU class with gamma = 0.25 on 100 x 4096 strips.  n = 1, 8, 32, 128 pairs per batch; uint8 frames resident on
the device, zero initial flow.  The two ways alternate, ROUNDS rounds each, and the median round is reported.  The
first MAX_CHECK pairs of every case are checked bit for bit between the two ways.  Writes
profiles/batch_ex_probe.json (or the path given as argv[1]) with the card's name and power limit, read in the same
run.

    python scripts/batch_ex_probe.py [out.json]
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

from fibsem_optflow_b200 import _native as N, synth  # noqa: E402

MODES = (("cuda", dict(semantics=N.SEMANTICS_CUDA), ((100, 4096), (200, 4096), (2048, 2048))),
         ("gamma 0.25", dict(gamma=0.25), ((100, 4096),)))
COUNTS = (1, 8, 32, 128)
ROUNDS = 3
MAX_CHECK = 8


def card():
    out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                                  text=True).strip()
    name, limit = (x.strip() for x in out.split(","))
    return name, limit


def case(s, h, w, n):
    N.check(N.lib().tvl1_set_device(0))
    base = [synth.make_pair(h, w, seed=100 + k) for k in range(min(n, 8))]   # 8 distinct pairs, cycled
    pairs = [base[k % len(base)] for k in range(n)]
    plane = h * w
    frames = N.DevBuf(2 * n * plane, 0).upload(np.stack([p[0] for p in pairs] + [p[1] for p in pairs]))
    flows = [N.DevBuf(2 * n * plane * 4, 0) for _ in range(2)]   # [batch, one by one]
    f0 = [frames.ptr + k * plane for k in range(n)]
    f1 = [frames.ptr + (n + k) * plane for k in range(n)]
    du = [[fb.ptr + k * plane * 4 for k in range(n)] for fb in flows]
    dv = [[fb.ptr + (n + k) * plane * 4 for k in range(n)] for fb in flows]

    def batch():
        s.calc_batch_ex_device(N.FRAME_U8, f0, w, f1, w, w, h, None, None, 0, du[0], dv[0], w * 4)
        return s.batch_stats[0].launches, s.last_readbacks()

    def singles():
        launches = readbacks = 0
        for k in range(n):
            s.calc_device(f0[k], w, f1[k], w, w, h, du[1][k], dv[1][k], w * 4)
            launches += s.stats.launches
            readbacks += s.last_readbacks()
        return launches, readbacks

    batch(), singles()   # warm-up: arenas, tile searches, module loads
    tb, ts = [], []
    for _ in range(ROUNDS):
        for fn, acc in ((batch, tb), (singles, ts)):
            t = time.perf_counter()
            counts = fn()
            acc.append((time.perf_counter() - t) * 1e3)
            if fn is batch:
                cb = counts
            else:
                cs = counts
    m = min(n, MAX_CHECK)
    a = flows[0].download((2, n, h, w), np.float32)[:, :m]
    b = flows[1].download((2, n, h, w), np.float32)[:, :m]
    same = bool(np.array_equal(a, b))
    for x in [frames] + flows:
        x.free()
    mb, ms = float(np.median(tb)), float(np.median(ts))
    px = float(n) * h * w
    return {
        "h": h, "w": w, "n": n, "bit_equal_first_%d" % m: same,
        "batch": {"ms_per_batch": mb, "ms_per_pair": mb / n, "mpx_per_s": px / mb / 1e3,
                  "launches": cb[0], "readbacks": cb[1], "rounds_ms": tb},
        "one_by_one": {"ms_total": ms, "ms_per_pair": ms / n, "mpx_per_s": px / ms / 1e3,
                       "launches": cs[0], "readbacks": cs[1], "rounds_ms": ts},
        "speedup": ms / mb,
    }


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "batch_ex_probe.json")
    N.require_device()
    name, limit = card()
    rec = {"card": name, "power_limit": limit,
           "params": "wrapper defaults (lambda .05, 10 scales, 300 iterations) plus the mode's own",
           "timing": "host clock around calls that synchronise; median of %d alternated rounds" % ROUNDS, "cases": []}
    for mode, kw, shapes in MODES:
        s = N.Solver(N.default_params(**kw))
        for (h, w) in shapes:
            for n in COUNTS:
                r = dict(mode=mode, **case(s, h, w, n))
                rec["cases"].append(r)
                print("%-10s %5d x %-5d n %4d  batch %9.2f ms (%7.3f ms/pair, %7.1f Mpx/s, %6d launches, %5d read-backs)"
                      "  one by one %9.2f ms (%7.3f ms/pair, %6d launches, %5d read-backs)  x%.2f  equal %s"
                      % (mode, h, w, n, r["batch"]["ms_per_batch"], r["batch"]["ms_per_pair"], r["batch"]["mpx_per_s"],
                         r["batch"]["launches"], r["batch"]["readbacks"], r["one_by_one"]["ms_total"],
                         r["one_by_one"]["ms_per_pair"], r["one_by_one"]["launches"], r["one_by_one"]["readbacks"],
                         r["speedup"], [v for k, v in r.items() if k.startswith("bit_equal")][0]), flush=True)
        s.close()
    with open(out, "w") as f:
        json.dump(rec, f, indent=1)
    print("card %s, power limit %s -> %s" % (name, limit, out))


if __name__ == "__main__":
    main()
