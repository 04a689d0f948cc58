#!/usr/bin/env python
"""bench.py -- TV-L1 flow throughput on synthetic FIB-SEM-like slice pairs.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched under torchrun)
    python bench.py --impl reference --steps K --warmup W    (CPU restatement, host cores)

A "step" is one pass of the hot path (pyramid -> per-level warp / median / primal-dual
iterations -> flow) over one slice pair per GPU.  Workload = BASELINE.json configs[1]: one
8192x8192 8-bit pair, 6 scales, 5 warps, DualTVL1 CPU-class defaults otherwise.  Slice pairs
are independent, so N GPUs run N different pairs with no collective ("scaling": "weak").

One JSON line on stdout (rank 0):
  value     Mpx/s with the frames already resident in HBM (tvl1_calc_u8, CUDA events)
  e2e       Mpx/s through the host-buffer C-ABI call (tvl1_calc_u8_host): H2D of both frames
            from pinned memory and D2H of both flow planes inside the timed region
  roofline  the primal-dual iteration kernel k_outer (one cooperative launch per outer iteration: its
            two-iteration and single passes): 64 B/px/iteration (SURVEY.md 8(d)) x the px-iterations
            executed / its CUDA-event time inside the timed region (host read-backs of the stop flag
            included); `traffic` / `dram_frac` from the ncu capture of the same kernel (profiles/)
  parity    CUDA path vs the C oracle on configs[0] (2048^2 pair), outside the timed regions:
            mean / max endpoint error, iteration-count vector equality, bit-equality
  stack     configs[2]: 512 chained 4096^2 pairs, strong-scaled over the N GPUs (tvl1_stack_run)
  volume    configs[4]-style: chained 6144^2 slices per GPU, matches only (no flow download)
  cpu_baseline  the C oracle (oracle/, OpenMP) on a bounded crop of the same pair

--dump-outputs DIR writes what the timed path returned in its last timed step, so that two builds run
with the same arguments (hence the same seeded inputs) can be compared output for output:
  u.npy, v.npy      the flow planes (float32), whole when both fit in DUMP_BYTES, else the same fixed
                    seeded sample of pixels from each (flat row-major indices, see dump_index)
  iterations.npy    the iteration count of every (level, warp) (float64)
Only rank 0 writes.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from fibsem_optflow_b200 import synth  # noqa: E402

METRIC = "tvl1_flow_mpx_per_s"
UNIT = "Mpx/s"
CPU_CROP = 2048          # the CPU legs run a CPU_CROP^2 crop of the pair (bounded sample)
DUMP_BYTES = 64 << 20    # --dump-outputs: at most this much in all
DUMP_SAMPLE = 4 << 20    # pixels drawn per flow plane when the planes are larger than DUMP_BYTES


def dump_index(npx):
    """Flat pixel indices --dump-outputs keeps of an npx-pixel flow plane: None (all of them) when both
    float32 planes fit in DUMP_BYTES, else a fixed seeded draw, sorted and without repeats."""
    if 2 * 4 * npx <= DUMP_BYTES:
        return None
    return np.unique(np.random.default_rng(0).integers(0, npx, DUMP_SAMPLE))


def dump_outputs(d, u, v, iters):
    """Writes d/u.npy, d/v.npy (float32; u and v are NumPy arrays or torch tensors) and d/iterations.npy."""
    idx = dump_index(u.numel() if hasattr(u, "numel") else u.size)
    out = {}
    for name, a in (("u", u), ("v", v)):
        if idx is not None:
            a = a.reshape(-1)[idx]
        out[name] = np.asarray(a.cpu() if hasattr(a, "cpu") else a, dtype=np.float32)
    out["iterations"] = np.asarray(iters, dtype=np.float64)
    os.makedirs(d, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(d, name + ".npy"), a)


def workload(args):
    tag = {2048: "configs[0]", 8192: "configs[1]", 16384: "configs[3] (cross-section pair, large displacement)"}.get(
        args.size, "configs[1]-style")
    return {"workload": "%s: single %dx%d 8-bit slice pair, %d scales, %d warps" % (
                tag, args.size, args.size, args.scales, args.warps),
            "synthetic": {"shift_px": [args.dx, args.dy], "shear_px_over_height": args.shear_px, "seed": args.seed,
                          "texture_coarse": args.coarse},
            "width": args.size, "height": args.size, "nscales": args.scales, "warps": args.warps,
            "tau": 0.25, "lambda": 0.15, "theta": 0.3, "epsilon": 0.01, "scaleStep": 0.8,
            "innerIterations": 30, "outerIterations": 10, "medianFiltering": 5,
            "pairs_per_gpu_per_step": 1, "sharding": "by pair, no collective",
            "reference_arm_sample": "the CPU arm (--impl reference, cpu_baseline) solves the centre %dx%d crop of this "
                                    "pair per step (bounded sample; Mpx/s of the crop)" % (
                                        min(CPU_CROP, args.size), min(CPU_CROP, args.size)),
            "l2": "inputs larger than L2 (%.1f GB of planes per pair)" % (
                args.size * args.size * 4 * 24 / 1e9)}


def make_pair(args, rank):
    return synth.make_pair(args.size, args.size, seed=args.seed + rank, dx=args.dx, dy=args.dy,
                           shear=args.shear_px / args.size, margin=args.margin, coarse=args.coarse)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []      # (wall time, fields)
        self.proc = None
        self.t0 = self.t1 = None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def run(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append((time.time(), [c.strip() for c in line.split(",")]))
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        inwin = [r for (t, r) in self.rows
                 if self.t0 is None or (self.t0 - 0.05 <= t <= (self.t1 or t) + 0.25)]
        for r in (inwin or [r for (_, r) in self.rows[-3:]]):
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def cpu_leg(args, steps, warmup, crop=CPU_CROP):
    """The C oracle on the box's host cores, on a crop of the workload's pair."""
    from oracle import oracle as O
    I0, I1 = make_pair(args, 0)
    n = min(crop, args.size)
    o = (args.size - n) // 2
    c0 = np.ascontiguousarray(I0[o:o + n, o:o + n])
    c1 = np.ascontiguousarray(I1[o:o + n, o:o + n])
    cores = os.cpu_count() or 1
    p = O.default_params(nscales=args.scales, warps=args.warps, nthreads=cores)
    times = []
    u = v = iters = None
    for i in range(warmup + steps):
        t = time.perf_counter()
        u, v, iters, lev = O.tvl1_calc(c0, c1, params=p)
        dt = time.perf_counter() - t
        if i >= warmup:
            times.append(dt)
    total = sum(times)
    return {"value": n * n * len(times) / total / 1e6, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "center %dx%d crop of the %dx%d pair, same parameters, %d step(s), "
                      "%d total iterations" % (n, n, args.size, args.size, len(times),
                                               int(iters[iters >= 0].sum())),
            "ms_per_step": total / len(times) * 1e3, "outputs": (u, v, iters[:lev])}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    steps, warmup = args.steps, max(0, args.warmup)
    cb = cpu_leg(args, steps, min(warmup, 1))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *cb["outputs"])
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT,
            "n_gpus": args.gpus, "steps": steps, "warmup": min(warmup, 1),
            "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload(args), "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "CPU restatement of OpenCV DualTVL1 (oracle/tvl1_oracle.c, OpenMP); OpenCV's own "
                    "class is not installable here (BASELINE.md section 2)"}
    print(json.dumps(line), flush=True)
    return 0


def run_ours(args):
    import torch
    from fibsem_optflow_b200 import _native as N

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path "
                         "(use --impl reference for the CPU restatement)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        # slice pairs are independent: no collective touches the data path, so the only
        # cross-rank traffic is this control-plane barrier / MAX / SUM of three scalars (gloo)
        import torch.distributed as dist
        dist.init_process_group("gloo")

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allmin(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return float(t.item())

    def allsum(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    K, W = args.steps, max(3, args.warmup)
    S = args.size
    I0, I1 = make_pair(args, rank)
    solver = N.Solver(N.default_params(lambda_=0.15, nscales=args.scales, warps=args.warps,
                                       inner_iterations=30, outer_iterations=10), device=local)
    solver.set_timing(True)     # per-stage CUDA events: the roofline's kernel time comes from them
    # device-resident inputs / outputs (torch only allocates and hands out pointers)
    d0 = torch.from_numpy(I0).cuda()
    d1 = torch.from_numpy(I1).cuda()
    du = torch.empty((S, S), dtype=torch.float32, device="cuda")
    dv = torch.empty((S, S), dtype=torch.float32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def step_dev():
        solver.calc_device(d0.data_ptr(), S, d1.data_ptr(), S, S, S, du.data_ptr(), dv.data_ptr(),
                           S * 4, stream)

    # nvidia-smi wants the physical index: honour CUDA_VISIBLE_DEVICES if the launcher set it
    vis = [v for v in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if v.strip() != ""]
    phys = vis[local].strip() if local < len(vis) else str(local)
    sampler = ClockSampler(phys)
    sampler.start()
    for _ in range(W):
        step_dev()
    barrier()
    sampler.mark_begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    it_ms, it_px, launches, tot_iters = 0.0, 0, 0, 0
    lvl_ms = np.zeros(N.MAX_LEVELS)
    lvl_pxit = np.zeros(N.MAX_LEVELS)
    for _ in range(K):
        step_dev()
        st = solver.stats
        it_ms += st.ms_iterate
        it_px += st.px_iterations
        launches += st.launches
        tot_iters += st.total_iterations
        its = st.iters_array()
        for l in range(st.levels):
            lvl_ms[l] += st.ms_iterate_level[l]
            lvl_pxit[l] += float(st.width[l]) * st.height[l] * int(its[l].sum())
    e1.record()
    barrier()
    sampler.mark_end()
    ms_dev_own = e0.elapsed_time(e1)
    ms_dev = allmax(ms_dev_own)
    ms_dev_fastest = allmin(ms_dev_own)   # the spread over the ranks: a slow GPU (imbalance) or everybody (contention)?
    stats = solver.stats          # (overwritten by the later legs: keep what the line reports)
    levels = stats.level_sizes()
    iters_last = stats.iters_array().tolist()
    alg_bytes = stats.algorithmic_bytes
    stage_ms = {"total": stats.ms_total, "pyramid": stats.ms_pyramid, "warp": stats.ms_warp,
                "iterate": stats.ms_iterate, "median": stats.ms_median, "other": stats.ms_other}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, du, dv, iters_last)

    # this box's own copy bandwidth, measured the way MEASURED_PEAKS.json was (context only:
    # boxes of the pool differ by ~20 %; roofline.frac stays against the driver-written peak)
    copy_gbs = None
    try:
        ca = torch.empty(1 << 29, dtype=torch.bfloat16, device="cuda")
        cb = torch.empty_like(ca)
        best = 1e9
        for _ in range(6):
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            cb.copy_(ca)
            c1.record()
            torch.cuda.synchronize()
            best = min(best, c0.elapsed_time(c1))
        copy_gbs = 2.0 * ca.numel() * 2 / (best * 1e-3) / 1e9
        del ca, cb
    except Exception:
        pass

    # end to end: K pairs through the public pipelined call (tvl1_stack_run with an explicit pair list, the
    # "images" loop of a job): every step's two frames go up from pinned host memory and its two flow planes
    # come down inside the timed region; the runner overlaps pair k+1's upload and pair k-1's download with
    # pair k's solve.  The 2K host slices alternate between the same two pinned frames under DISTINCT slice
    # indices, so nothing is re-used on the device: every step pays its own H2D.
    h0 = torch.from_numpy(I0).pin_memory()
    h1 = torch.from_numpy(I1).pin_memory()
    hu = [torch.empty((S, S), dtype=torch.float32).pin_memory() for _ in range(2)]
    hv = [torch.empty((S, S), dtype=torch.float32).pin_memory() for _ in range(2)]

    def run_e2e(npairs):
        return solver.run_stack(slices=None, flows=True, apply_mask=False, npoints=-1,
                                out_u=[hu[k & 1].data_ptr() for k in range(npairs)],
                                out_v=[hv[k & 1].data_ptr() for k in range(npairs)],
                                slice_ptrs=[(h0, h1)[i & 1].data_ptr() for i in range(2 * npairs)], pitch=S,
                                shape=(S, S), pairs=[(2 * k, 2 * k + 1) for k in range(npairs)])

    solver.set_timing(False)
    run_e2e(2)
    barrier()
    t0 = time.perf_counter()
    run_e2e(K)
    barrier()
    ms_e2e = allmax((time.perf_counter() - t0) * 1e3)
    checksum = float(hu[(K - 1) & 1][::257, ::263].double().sum() + hv[(K - 1) & 1][::257, ::263].double().sum())

    # the same through the synchronous one-pair call (tvl1_calc_u8_host: H2D, solve, D2H back to back)
    def step_host():
        N.check(N.lib().tvl1_calc_u8_host(solver.handle, h0.data_ptr(), S, h1.data_ptr(), S, S, S,
                                          hu[0].data_ptr(), hv[0].data_ptr(), S * 4, C.byref(solver.stats)))

    step_host()
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        step_host()
    barrier()
    ms_e2e_sync = allmax((time.perf_counter() - t0) * 1e3)
    sampler.t1 = time.time()      # the clock window covers the timed regions
    clocks = sampler.stop()
    del hu, hv

    # ---- parity vs the oracle on configs[0] (outside every timed region; rank 0)
    parity = None
    if rank == 0 and not args.no_parity:
        from oracle import oracle as O
        P0, P1 = synth.make_pair(2048, 2048, seed=7)
        ps = N.Solver(N.default_params(lambda_=0.15, nscales=5, warps=5, inner_iterations=30,
                                       outer_iterations=10), device=local)
        gu, gv = ps.calc(P0, P1)
        ou, ov, oit, olev = O.tvl1_calc(P0, P1, **{"lambda": 0.15, "nscales": 5, "nthreads": os.cpu_count() or 1})
        epe = np.hypot(gu - ou, gv - ov)
        parity = {"config": "configs[0]: 2048x2048 pair, 5 scales, 5 warps, vs oracle/tvl1_oracle.c",
                  "mean_epe": float(epe.mean()), "max_epe": float(epe.max()),
                  "iters_equal": bool(ps.stats.levels == olev and np.array_equal(ps.stats.iters_array(), oit[:olev])),
                  "bit_equal": bool(np.array_equal(gu, ou) and np.array_equal(gv, ov)),
                  "bounds": {"mean_epe": 0.01, "max_epe": 0.1}}
        ps.close()
        del gu, gv, ou, ov, epe

    def chained(n_distinct, size, seed):
        """n_distinct+1 chained slices walked back and forth, so that ANY number of adjacent pairs can
        be formed from a few pinned buffers (slice k+1 is always a neighbour of slice k)."""
        sl = synth.make_stack(n_distinct, size, size, seed=seed)
        return [torch.from_numpy(a).pin_memory() for a in sl]

    def walk(n_slices, n_buf, start=0):
        period = 2 * (n_buf - 1)
        out = []
        for k in range(n_slices):
            r = (start + k) % period
            out.append(r if r < n_buf else period - r)
        return out

    # ---- configs[2]: a stack of 512 chained 4096^2 pairs, STRONG-scaled: rank r solves its contiguous
    # block of pairs through tvl1_stack_run (every slice uploaded once, uploads / flow downloads / match
    # sampling overlapped with the solves; flows land in a ring of pinned host planes)
    stack = None
    if args.stack_pairs > 0:
        SS = args.stack_size
        total = args.stack_pairs
        lo = rank * total // world
        hi = (rank + 1) * total // world
        mine = hi - lo
        hs = chained(8, SS, 100)
        ring = [torch.empty((SS, SS), dtype=torch.float32).pin_memory() for _ in range(8)]
        st_solver = N.Solver(N.default_params(lambda_=0.15, nscales=5, warps=5, inner_iterations=30,
                                              outer_iterations=10), device=local)

        def run(npairs, start):
            idx = walk(npairs + 1, len(hs), start)
            return st_solver.run_stack(slices=None, flows=True, apply_mask=True, npoints=25, scale=0.5, seed=1,
                                       out_u=[ring[(2 * k) % 8].data_ptr() for k in range(npairs)],
                                       out_v=[ring[(2 * k + 1) % 8].data_ptr() for k in range(npairs)],
                                       slice_ptrs=[hs[i].data_ptr() for i in idx], pitch=SS, shape=(SS, SS))
        run(3, 0)
        barrier()
        t0 = time.perf_counter()
        r = run(mine, lo) if mine > 0 else None
        ms_stack_own = (time.perf_counter() - t0) * 1e3     # this rank's own block, before it waits for the others
        solve_own = sum(x.ms_total for x in r["stats"]) / max(mine, 1) if r else 0.0
        barrier()
        ms_stack = allmax((time.perf_counter() - t0) * 1e3)
        ms_stack_fastest = allmin(ms_stack_own)
        solve_slowest, solve_fastest = allmax(solve_own), allmin(solve_own)
        stack = {"workload": "configs[2]: stack of %d chained %dx%d pairs sharded by contiguous block over %d GPU(s), "
                             "5 scales, 5 warps, mask + 25 matches + flow download per pair" % (total, SS, SS, world),
                 "value": float(SS) * SS * total / (ms_stack * 1e-3) / 1e6, "unit": UNIT, "scaling": "strong",
                 "pairs_total": total, "pairs_per_gpu": mine, "ms_per_pair_per_gpu": ms_stack / max(mine, 1),
                 "ms_per_pair_fastest_gpu": ms_stack_fastest / max(mine, 1),
                 "solve_ms_per_pair": {"slowest_gpu": solve_slowest, "fastest_gpu": solve_fastest},
                 "h2d_bytes_per_pair": SS * SS, "d2h_bytes_per_pair": 8 * SS * SS,
                 "api": "tvl1_stack_run (pinned host buffers, copy streams)",
                 "iterations_first_pairs": [int(x.total_iterations) for x in (r["stats"][:4] if r else [])]}
        st_solver.close()
        del hs, ring

    # ---- configs[4]-style: chained 6144^2 slices, matches only (flow never leaves the device)
    volume = None
    if args.volume_pairs > 0:
        VS = args.volume_size
        hs = chained(4, VS, 200)   # the same slices on every rank: weak scaling then measures the machine, not the content
        v_solver = N.Solver(N.default_params(lambda_=0.15, nscales=5, warps=5, inner_iterations=30,
                                             outer_iterations=10), device=local)

        def runv(npairs):
            idx = walk(npairs + 1, len(hs))
            return v_solver.run_stack(slices=None, flows=False, apply_mask=True, npoints=25, scale=0.5, seed=1,
                                      slice_ptrs=[hs[i].data_ptr() for i in idx], pitch=VS, shape=(VS, VS))
        runv(2)
        barrier()
        t0 = time.perf_counter()
        runv(args.volume_pairs)
        barrier()
        ms_vol = allmax((time.perf_counter() - t0) * 1e3)
        volume = {"workload": "configs[4]-style: %d chained %dx%d pairs per GPU, 5 scales, 5 warps, mask + 25 matches "
                              "per pair, no flow download (h_u = NULL)" % (args.volume_pairs, VS, VS),
                  "value": allsum(float(VS) * VS * args.volume_pairs) / (ms_vol * 1e-3) / 1e6, "unit": UNIT,
                  "scaling": "weak", "ms_per_pair": ms_vol / args.volume_pairs,
                  "h2d_bytes_per_pair": VS * VS, "d2h_bytes_per_pair": 25 * 5 * 8,
                  "api": "tvl1_stack_run (h_u = NULL)"}
        v_solver.close()
        del hs

    px_all = allsum(float(S) * S * K)
    total_launches = int(allsum(float(launches)))
    if rank == 0:
        peak, peak_src = peaks()
        ach = 64.0 * it_px / (it_ms * 1e-3) / 1e9 if it_ms > 0 else 0.0
        per_level = []
        for l, (w, h) in enumerate(levels):
            if lvl_ms[l] > 0:
                per_level.append({"level": l, "size": [w, h],
                                  "gbs": round(64.0 * lvl_pxit[l] / (lvl_ms[l] * 1e-3) / 1e9, 1),
                                  "ms": round(lvl_ms[l] / K, 3)})
        # DRAM traffic of the same kernel from its ncu --set full capture (profiles/k_outer_traffic.json:
        # one level-0 k_outer launch of a known iteration count): per launch, and per px-iteration so
        # that dram_frac can be formed from THIS run's kernel time
        traffic = traffic_kernel = dram_frac = bytes_px_it = None
        tp = os.path.join(ROOT, "profiles", "k_outer_traffic.json")
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                traffic = tj.get("dram_bytes_per_launch")
                traffic_kernel = tj.get("kernel")
                bytes_px_it = tj.get("dram_bytes_per_px_iteration")
                if bytes_px_it and it_ms > 0:
                    dram_frac = bytes_px_it * it_px / (it_ms * 1e-3) / 1e9 / peak
            except Exception:
                traffic = None
        line = {
            "metric": METRIC, "value": px_all / (ms_dev * 1e-3) / 1e6, "unit": UNIT,
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_dev / K,
            "ms_per_step_fastest_gpu": ms_dev_fastest / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload(args),
            "e2e": {"value": px_all / (ms_e2e * 1e-3) / 1e6, "unit": UNIT,
                    "h2d_bytes_per_step": 2 * S * S, "d2h_bytes_per_step": 8 * S * S,
                    "ms_per_step": ms_e2e / K,
                    "api": "tvl1_stack_run with a pair list (pinned host buffers; uploads / downloads overlap the solves)",
                    "checksum": checksum,
                    "sync_call": {"value": px_all / (ms_e2e_sync * 1e-3) / 1e6, "ms_per_step": ms_e2e_sync / K,
                                  "api": "tvl1_calc_u8_host (one pair per call: H2D, solve, D2H back to back)"}},
            "gpu_launches": total_launches,
            "roofline": {"bound": "hbm",
                         "kernel": "k_outer<4> (primal-dual iterations: its two-iteration and single passes, one "
                                   "cooperative launch per outer iteration, all levels, inside the timed region)",
                         "achieved": ach, "peak": peak, "unit": "GB/s",
                         "frac": ach / peak if peak else None, "traffic": traffic,
                         "dram_frac": dram_frac, "dram_bytes_per_px_iteration": bytes_px_it,
                         "peak_source": peak_src, "copy_gbs_this_box": copy_gbs,
                         "frac_of_this_box_copy": (ach / copy_gbs) if copy_gbs else None,
                         "bytes_per_px_iteration": 64,
                         "px_iterations_per_step": it_px / K, "kernel_ms_per_step": it_ms / K,
                         "traffic_kernel": traffic_kernel,
                         "note": "frac = 64 B/px/iteration model / measured copy peak: a two-iteration pass moves 60 B/px "
                                 "for TWO iterations (9 planes read + 6 written once), so frac > 1 is what temporal "
                                 "blocking is for; dram_frac = DRAM bytes ncu measured per px-iteration x this run's "
                                 "px-iterations / this run's kernel time / peak",
                         "per_level": per_level,
                         "pair_algorithmic_gbs": alg_bytes / (ms_dev / K * 1e-3) / 1e9},
            "clocks": clocks,
            "iterations_per_pair": int(tot_iters / K), "iters_last_pair": iters_last,
            "stage_ms_last_pair": stage_ms,
        }
        if parity is not None:
            line["parity"] = parity
        if stack is not None:
            line["stack"] = stack
        if volume is not None:
            line["volume"] = volume
        if world == 1 and not args.no_cpu:
            cb = cpu_leg(args, 1, 0)
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        print(json.dumps(line), flush=True)
    solver.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size", type=int, default=8192)
    ap.add_argument("--scales", type=int, default=6)
    ap.add_argument("--warps", type=int, default=5)
    ap.add_argument("--dx", type=float, default=1.3, help="synthetic shift of the pair (configs[3]: 8-20 px)")
    ap.add_argument("--dy", type=float, default=-0.7)
    ap.add_argument("--shear-px", type=float, default=4.0, help="shear over the frame height, px")
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--margin", type=int, default=32)
    ap.add_argument("--coarse", type=int, default=0, help="extra coarse texture component (configs[3]: 16)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-parity", action="store_true", help="skip the parity leg (configs[0] vs the oracle)")
    ap.add_argument("--stack-pairs", type=int, default=512, help="configs[2] leg: pairs of the whole stack, split over the GPUs (0 = off)")
    ap.add_argument("--stack-size", type=int, default=4096)
    ap.add_argument("--volume-pairs", type=int, default=16, help="configs[4] leg: pairs per GPU, matches only (0 = off)")
    ap.add_argument("--volume-size", type=int, default=6144)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
