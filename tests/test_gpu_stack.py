"""Stack of adjacent slices through tvl1_stack_run (pipelined uploads/downloads, slice re-use)
against per-pair oracle solves; debug-mode sampling continues one rand() stream across pairs."""
import numpy as np
import pytest

from fibsem_optflow_b200 import synth

pytestmark = pytest.mark.gpu


def test_stack_flows_and_matches(gpu, orc):
    slices = synth.make_stack(5, 96, 128, seed=11)        # 6 slices -> 5 pairs
    slices[2][:8, :] = 0                                  # a masked strip in one slice
    s = gpu.Solver(gpu.default_params(lambda_=0.15, nscales=4))
    res = s.run_stack(slices, flows=True, apply_mask=True, npoints=12, scale=0.5, seed=77)
    assert len(res["u"]) == 5
    for k in range(5):
        ou, ov, oit, lev = orc.tvl1_calc(slices[k], slices[k + 1], **{"lambda": 0.15, "nscales": 4})
        orc.mask_flow(slices[k + 1], ou, ov)
        assert np.array_equal(res["stats"][k].iters_array(), oit[:lev])
        assert np.array_equal(res["u"][k], ou) and np.array_equal(res["v"][k], ov)
        want = orc.random_points(slices[k], slices[k + 1], ou, ov, scale=0.5, npoints=12, seed=77)
        got = res["matches"][k]
        for j in range(5):
            assert np.array_equal(got[j], want[j])


def test_stack_debug_stream_continues(gpu, orc, tmp_path):
    """seed < 0: the reference's debug mode never calls srand, so pair k's shuffle starts where
    pair k-1's stopped.  The oracle reproduces that with real glibc rand() in a fresh process."""
    import json, os, subprocess, sys
    slices = synth.make_stack(3, 40, 56, seed=5)
    s = gpu.Solver(gpu.default_params(lambda_=0.15, nscales=2))
    res = s.run_stack(slices, flows=True, npoints=6, scale=1.0, seed=-1)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    npz = str(tmp_path / "stack_dbg.npz")
    np.savez(npz, slices=np.stack(slices), u=np.stack(res["u"]), v=np.stack(res["v"]))
    code = (
        "import sys, json; sys.path.insert(0, %r)\n"
        "import numpy as np\n"
        "from oracle import oracle as O\n"
        "d = np.load(%r); out = []\n"
        "for k in range(3):\n"
        "    r = O.random_points(d['slices'][k], d['slices'][k+1], d['u'][k], d['v'][k], scale=1.0, npoints=6, seed=-1)\n"
        "    out.append([a.tolist() for a in r[:5]])\n"
        "print(json.dumps(out))\n" % (root, npz))
    want = json.loads(subprocess.check_output([sys.executable, "-c", code]).decode())
    for k in range(3):
        for j in range(5):
            assert res["matches"][k][j].tolist() == want[k][j]


def test_stack_no_flow_download(gpu):
    slices = synth.make_stack(2, 64, 64, seed=3)
    s = gpu.Solver(gpu.default_params(lambda_=0.15, nscales=2))
    res = s.run_stack(slices, flows=False, npoints=25, seed=1)
    assert "u" not in res and len(res["matches"]) == 2 and len(res["matches"][0][0]) == 25
    with pytest.raises(gpu.Tvl1Error):
        s.run_stack(slices[:1])


@pytest.mark.parametrize("scale", [0.5, 0.4])
def test_stack_prescale_on_device(gpu, orc, scale):
    """Raw slices in, the loader's 8-bit cv::resize (src/optflow.cpp:111,124) applied on the device on
    the copy stream: flows and matches equal the oracle's on slices it shrank itself."""
    slices = synth.make_stack(3, 161, 230, seed=5)        # odd height: exercises the area path's border rule
    scf = float(np.float32(scale))
    small = [orc.prescale_u8(a, scf) for a in slices]
    s = gpu.Solver(gpu.default_params(lambda_=0.15, nscales=3))
    res = s.run_stack(slices, flows=True, apply_mask=True, npoints=9, scale=scale, seed=3, prescale=scf)
    for k in range(3):
        ou, ov, oit, lev = orc.tvl1_calc(small[k], small[k + 1], **{"lambda": 0.15, "nscales": 3})
        orc.mask_flow(small[k + 1], ou, ov)
        assert res["u"][k].shape == ou.shape
        assert np.array_equal(res["u"][k], ou) and np.array_equal(res["v"][k], ov)
        want = orc.random_points(small[k], small[k + 1], ou, ov, scale=scale, npoints=9, seed=3)
        for j in range(5):
            assert np.array_equal(res["matches"][k][j], want[j])
    s.close()


def test_stack_explicit_pairs(gpu, orc):
    """tvl1_stack_io.pair_p / pair_q: the "images" list of a job -- independent pairs, a repeated pair, a
    reversed pair and a chained one -- through the pipelined runner (4 slice slots, next pair's frames
    uploaded during the current solve): flows and matches equal per-pair oracle solves."""
    slices = synth.make_stack(5, 72, 100, seed=17)        # 6 slices
    pairs = [(0, 1), (2, 3), (4, 5), (5, 4), (4, 5), (1, 2), (2, 3), (0, 5)]
    s = gpu.Solver(gpu.default_params(lambda_=0.15, nscales=3))
    res = s.run_stack(slices, flows=True, apply_mask=True, npoints=10, scale=0.5, seed=9, pairs=pairs)
    assert len(res["u"]) == len(pairs)
    for k, (p, q) in enumerate(pairs):
        ou, ov, oit, lev = orc.tvl1_calc(slices[p], slices[q], **{"lambda": 0.15, "nscales": 3})
        orc.mask_flow(slices[q], ou, ov)
        assert np.array_equal(res["stats"][k].iters_array(), oit[:lev]), k
        assert np.array_equal(res["u"][k], ou) and np.array_equal(res["v"][k], ov), k
        want = orc.random_points(slices[p], slices[q], ou, ov, scale=0.5, npoints=10, seed=9)
        for j in range(5):
            assert np.array_equal(res["matches"][k][j], want[j]), (k, j)
    with pytest.raises(gpu.Tvl1Error):
        s.run_stack(slices, pairs=[(0, 6)])
    s.close()
