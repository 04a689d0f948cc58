"""TVL1_SEMANTICS_CUDA on the GPU: its kernels (k_resize_cuda, k_warp_cuda) and whole solves bit for bit
against the CPU restatement (oracle/tvl1_oracle_cuda.c), under every schedule option, through handles switched
between modes, the stack runner and the job driver."""
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

from fibsem_optflow_b200 import synth
from oracle import oracle_cuda as OC

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def same(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


def cuda_params(gpu, **kw):
    return gpu.default_params(semantics=gpu.SEMANTICS_CUDA, **kw)


def oracle_kw(p):
    return dict(tau=p.tau, theta=p.theta, epsilon=p.epsilon, scale_step=p.scale_step, nscales=p.nscales,
                warps=p.warps, **{"lambda": p.lambda_})


def solve_both(gpu, I0, I1, p, options=()):
    s = gpu.Solver(p)
    for k, v in options:
        s.set_option(k, v)
    u, v = s.calc(I0, I1)
    it = s.stats.iters_array()
    st = s.stats
    ou, ov, oit, lev = OC.tvl1_calc_cuda(I0, I1, iterations=p.iterations, **oracle_kw(p))
    s.close()
    return (u, v, it, st), (ou, ov, oit[:lev], lev)


# ---- stages

@pytest.mark.parametrize("h,w,amp,shift,pitch", [
    (37, 61, 0.4, 0, None),       # odd size, smooth flow
    (64, 96, 3.0, 0, 128),        # rough flow, pitched planes
    (131, 77, 1.0, 35.0, None),   # large displacements: the global-memory fallback, windows outside the image
    (200, 300, 12.0, 0, 320),     # flow varying more than the staged window holds
    (16, 16, 0.0, 0, 64),         # integer (zero) flow on a tiny level
])
def test_k_warp_cuda_matches_oracle(gpu, h, w, amp, shift, pitch):
    rng = np.random.default_rng(h * w)
    I0 = (rng.random((h, w)) * 255).astype(np.float32)
    I1 = synth.texture(h, w, 3).astype(np.float32) * np.float32(255)
    u1 = (rng.standard_normal((h, w)) * amp).astype(np.float32)
    u2 = (rng.standard_normal((h, w)) * amp).astype(np.float32)
    if shift:
        u1[: h // 2] += np.float32(shift)
        u2[:, w // 3:] -= np.float32(shift)
    got = gpu.k_warp_cuda(I0, I1, u1, u2, pitch=pitch)
    want = OC.warp_cuda(I0, I1, u1, u2)
    for k, (g, x) in enumerate(zip(got, want)):
        assert same(g, x), k


@pytest.mark.parametrize("sh,sw,f,size,pitch", [
    (97, 131, 0.8, None, None), (97, 131, 0.5, None, 160), (64, 48, 0.8, None, None),
    (41, 33, 0.0, (52, 41), None), (78, 104, 0.0, (130, 97), 160), (17, 19, 0.0, (21, 24), None),
])
def test_k_resize_cuda_matches_oracle(gpu, sh, sw, f, size, pitch):
    rng = np.random.default_rng(sh + sw)
    src = (rng.standard_normal((sh, sw)) * 40).astype(np.float32)
    if size is None:
        got = gpu.k_resize_cuda(src, inv_scale=f, spitch=pitch, dpitch=pitch)
        want = OC.resize_cuda(src, inv_scale=f)
    else:
        got = gpu.k_resize_cuda(src, size[0], size[1], mul=1.25, spitch=pitch, dpitch=pitch)
        want = OC.resize_cuda(src, size[0], size[1]) * np.float32(1.25)
    assert same(got, want)


# ---- whole pairs

PAIRS = [
    (48, 64, 5, dict(lambda_=0.05, nscales=10, iterations=300)),            # the reference wrapper's defaults
    (192, 256, 7, dict(lambda_=0.05, nscales=10, iterations=300)),
    (150, 222, 9, dict(lambda_=0.15, nscales=5, iterations=41)),             # odd N
    (160, 208, 2, dict(lambda_=0.05, nscales=4, iterations=7)),              # N is hit before any stop
    (96, 130, 4, dict(lambda_=0.15, nscales=3, iterations=12, epsilon=0.0)),  # no error is ever evaluated
    (120, 144, 6, dict(lambda_=0.1, nscales=4, iterations=60, epsilon=0.2, scale_step=0.5)),
]


@pytest.mark.parametrize("h,w,seed,kw", PAIRS)
def test_calc_matches_oracle(gpu, h, w, seed, kw):
    I0, I1 = synth.make_pair(h, w, seed=seed)
    p = cuda_params(gpu, **kw)
    (u, v, it, st), (ou, ov, oit, lev) = solve_both(gpu, I0, I1, p)
    assert st.levels == lev and np.array_equal(it, oit)
    assert ((it == p.iterations) | (it % 2 == 0)).all()
    if p.epsilon == 0.0:
        assert (it == p.iterations).all()
    assert same(u, ou) and same(v, ov)
    assert not np.ctypeslib.as_array(st.outer).any()


def test_calc_large_matches_oracle(gpu):
    I0, I1 = synth.make_pair(2048, 2048, seed=12, shear=0.5 / 2048)
    p = cuda_params(gpu, lambda_=0.05, nscales=10, iterations=40, warps=2)
    (u, v, it, st), (ou, ov, oit, lev) = solve_both(gpu, I0, I1, p)
    assert st.levels == lev and np.array_equal(it, oit)
    assert same(u, ou) and same(v, ov)


SCHEDULES = [(("coop_outer", 0),), (("multi_iter", 0),), (("fused_min_px", 1e18),), (("fused_min_px", 1e18), ("multi_iter", 0)),
             (("coop_outer", 0), ("fused_min_px", 0))]


def test_every_schedule_gives_the_same_result(gpu):
    I0, I1 = synth.make_pair(200, 264, seed=8)
    p = cuda_params(gpu, lambda_=0.05, nscales=6, iterations=45)
    s = gpu.Solver(p)
    u0, v0 = s.calc(I0, I1)
    it0 = s.stats.iters_array()
    s.close()
    assert it0.max() > 2
    for opts in SCHEDULES:
        s = gpu.Solver(p)
        for k, v in opts:
            s.set_option(k, v)
        u, v = s.calc(I0, I1)
        assert np.array_equal(s.stats.iters_array(), it0), opts
        assert same(u, u0) and same(v, v0), opts
        s.close()


def test_stats_have_no_median(gpu):
    I0, I1 = synth.make_pair(128, 160, seed=1)
    s = gpu.Solver(cuda_params(gpu, lambda_=0.15, nscales=4, iterations=30))
    s.set_timing(True)
    s.calc(I0, I1)
    st = s.stats
    assert not np.ctypeslib.as_array(st.outer).any() and st.ms_median == 0.0
    its = st.iters_array()
    px = sum(w * h * int(its[l].sum()) for l, (w, h) in enumerate(st.level_sizes()))
    assert st.px_iterations == px and st.total_iterations == its.sum()
    base = 70.0 * 160 * 128 + sum(w * h * (12.0 + sum(40.0 + 64.0 * n for n in its[l]))
                                   for l, (w, h) in enumerate(st.level_sizes()))
    assert abs(st.algorithmic_bytes - base) <= 1e-6 * base      # no 16 B/px median term
    s.close()


def test_set_params_switches_modes(gpu):
    I0, I1 = synth.make_pair(96, 120, seed=13)
    pc = gpu.default_params(lambda_=0.15, nscales=4)
    pg = cuda_params(gpu, lambda_=0.15, nscales=4, iterations=50)
    fresh = {}
    for name, p in (("cpu", pc), ("cuda", pg)):
        s = gpu.Solver(p)
        fresh[name] = s.calc(I0, I1) + (s.stats.iters_array(),)
        s.close()
    s = gpu.Solver(pc)
    for name, p in (("cpu", pc), ("cuda", pg), ("cpu", pc), ("cuda", pg)):
        s.set_params(p)
        u, v = s.calc(I0, I1)
        assert same(u, fresh[name][0]) and same(v, fresh[name][1]) and np.array_equal(s.stats.iters_array(), fresh[name][2])
    s.close()
    assert not np.array_equal(fresh["cpu"][0], fresh["cuda"][0])


def test_stack_run_matches_calc(gpu):
    slices = synth.make_stack(3, 96, 128, seed=17)
    p = cuda_params(gpu, lambda_=0.1, nscales=4, iterations=40)
    s = gpu.Solver(p)
    res = s.run_stack(slices, flows=True)
    one = gpu.Solver(p)
    for k in range(3):
        u, v = one.calc(slices[k], slices[k + 1])
        assert same(res["u"][k], u) and same(res["v"][k], v)
        assert np.array_equal(res["stats"][k].iters_array(), one.stats.iters_array())
    s.close()
    one.close()


def test_flow_is_solved(gpu):
    """Sanity, not parity: the mode still finds the flow of a synthetic pair (mean EPE over the interior)."""
    for seed, (h, w) in ((3, (256, 256)), (21, (320, 384))):
        I0, I1 = synth.make_pair(h, w, seed=seed, shear=1.0 / h)
        ut, vt = synth.true_flow(h, w, shear=1.0 / h)
        s = gpu.Solver(cuda_params(gpu))
        u, v = s.calc(I0, I1)
        s.close()
        m = 32
        epe = np.hypot(u - ut, v - vt)[m:-m, m:-m]
        assert epe.mean() <= 0.05, (seed, epe.mean())


def test_rejected_params(gpu):
    h = C.c_void_p()
    p = cuda_params(gpu, gamma=0.1)
    assert gpu.lib().tvl1_create(C.byref(p), 0, C.byref(h)) == -3
    for kw in (dict(inner_iterations=30), dict(outer_iterations=2)):
        p = cuda_params(gpu, **kw)
        assert gpu.lib().tvl1_create(C.byref(p), 0, C.byref(h)) == -1
    p = gpu.default_params(semantics=2)
    assert gpu.lib().tvl1_create(C.byref(p), 0, C.byref(h)) == -1
    p = cuda_params(gpu, median_filtering=7)          # not read in this mode
    assert gpu.lib().tvl1_create(C.byref(p), 0, C.byref(h)) == 0
    gpu.lib().tvl1_destroy(h)


def test_job_driver_matches_api(gpu, tmp_path):
    import cv2
    from fibsem_optflow_b200 import api
    exe = os.path.join(ROOT, "fibsem_optflow_b200", "host", "optflow_b200")
    subprocess.check_call(["make", "-C", os.path.dirname(exe), "-s"])
    sl = synth.make_stack(2, 96, 128, seed=23)
    names = []
    for k, a in enumerate(sl):
        names.append(str(tmp_path / ("c%d.png" % k)))
        assert cv2.imwrite(names[-1], a)
    common = {"debug": True, "scale": 1.0, "lambda": 0.15, "nscales": 3, "iterations": 40, "npoints": 6,
              "semantics": "cuda", "output_dir": str(tmp_path), "rois": {"top": 48}}
    job = dict(common, images=[
        {"p": names[0], "q": names[1], "output_name": "a", "output_type": "map"},
        {"p": names[1], "q": names[2], "output_type": "random_points", "pId": "c1", "qId": "c2",
         "pGroupId": "1.0", "qGroupId": "2.0"}])
    jf = str(tmp_path / "job.json")
    json.dump(job, open(jf, "w"))
    subprocess.check_call([exe, jf], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    from PIL import Image
    args = {k: v for k, v in common.items() if k != "rois"}
    want = api.solve_rois(sl[0], sl[1], {"top": [0, 0, 128, 48]}, {"output_type": "map"}, args)["top"]
    assert same(np.array(Image.open(str(tmp_path / "a_1.00_top_x.tiff")), np.float32), want[0])
    assert same(np.array(Image.open(str(tmp_path / "a_1.00_top_y.tiff")), np.float32), want[1])
    im = {"output_type": "random_points", "pId": "c1", "qId": "c2", "pGroupId": "1.0", "qGroupId": "2.0"}
    api.solve_rois(sl[1], sl[2], {"top": [0, 0, 128, 48]}, im, args, seed=-1)
    got = json.load(open(str(tmp_path / "point_matches_000.json")))
    assert got == args["point_matches"]
    api.release_solvers()
    # a forbidden key is a pair error: the pair is skipped, nothing is written for it
    job = dict(common, medianFiltering=5, images=[{"p": names[0], "q": names[1], "output_name": "z", "output_type": "map"}])
    json.dump(job, open(jf, "w"))
    subprocess.call([exe, jf], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    assert not os.path.exists(str(tmp_path / "z_1.00_top_x.tiff"))
