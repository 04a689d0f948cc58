"""tvl1_calc_batch_ex without a GPU: the symbol is exported with its argument types, and the Python wrappers refuse
malformed batches (mixed dtypes, mismatched initial flows, empty lists) before the library is called."""
import numpy as np
import pytest

from fibsem_optflow_b200 import _native as N, api


def test_batch_ex_symbol_exported(native):
    L = native.lib()
    assert hasattr(L, "tvl1_calc_batch_ex") and "tvl1_calc_batch_ex" in native.EXPORTS
    assert len(L.tvl1_calc_batch_ex.argtypes) == 17


def no_library_solver(monkeypatch):
    """a Solver that was never created, with every library call an error"""
    def refuse():
        raise AssertionError("the library was called")
    monkeypatch.setattr(N, "lib", refuse)
    s = object.__new__(N.Solver)
    s.handle, s.device = 1, 0
    return s


u8 = lambda h=4, w=5: np.zeros((h, w), np.uint8)
f32 = lambda h=4, w=5: np.zeros((h, w), np.float32)
flow = lambda h=4, w=5: (f32(h, w), f32(h, w))


@pytest.mark.parametrize("frames0, frames1, init, text", [
    ([], [], None, "non-empty"),
    ([u8()], [], None, "equally long"),
    ([u8()] * 2, [u8()], None, "equally long"),
    ([u8()], [f32()], None, "all be uint8 or all float32"),
    ([u8(), f32()], [u8(), u8()], None, "all be uint8 or all float32"),
    ([np.zeros((4, 5), np.float64)], [np.zeros((4, 5), np.float64)], None, "uint8 or float32"),
    ([np.zeros((4, 5, 3), np.uint8)], [np.zeros((4, 5, 3), np.uint8)], None, "2-D"),
    ([u8()], [u8(5, 4)], None, "one size"),
    ([u8(0, 5)], [u8(0, 5)], None, "empty"),
    ([u8()] * 2, [u8()] * 2, [flow()], "one \\(u0, v0\\) pair per pair"),
    ([u8()], [u8()], [flow(), flow()], "one \\(u0, v0\\) pair per pair"),
    ([u8()], [u8()], [], "one \\(u0, v0\\) pair per pair"),
    ([u8()], [u8()], [(f32(),)], "not a \\(u0, v0\\) pair"),
    ([u8()], [u8()], [(f32(), f32(), f32())], "not a \\(u0, v0\\) pair"),
    ([u8()], [u8()], [(f32(5, 4), f32())], "frames' size"),
    ([u8()], [u8()], [(f32(), f32(4, 6))], "frames' size"),
    ([u8()], [u8()], [(f32(), np.zeros((4, 5), np.float64))], "float32"),
])
def test_calc_batch_ex_rejects_malformed_input(monkeypatch, frames0, frames1, init, text):
    s = no_library_solver(monkeypatch)
    with pytest.raises(N.Tvl1Error, match=text):
        s.calc_batch_ex(frames0, frames1, init)


def test_calc_batch_ex_device_rejects_unequal_lists(monkeypatch):
    s = no_library_solver(monkeypatch)
    with pytest.raises(N.Tvl1Error, match="equally long"):
        s.calc_batch_ex_device(N.FRAME_U8, [1, 2], 8, [3, 4], 8, 8, 8, None, None, 0, [5], [6, 7], 32)
    with pytest.raises(N.Tvl1Error, match="non-empty"):
        s.calc_batch_ex_device(N.FRAME_U8, [], 8, [], 8, 8, 8, None, None, 0, [], [], 32)
    with pytest.raises(N.Tvl1Error, match="equally long"):   # one initial-flow list only, or one of another length
        s.calc_batch_ex_device(N.FRAME_U8, [1], 8, [3], 8, 8, 8, [9], None, 32, [5], [6], 32)
    with pytest.raises(N.Tvl1Error, match="equally long"):
        s.calc_batch_ex_device(N.FRAME_U8, [1], 8, [3], 8, 8, 8, [9, 9], [8], 32, [5], [6], 32)


def test_api_solve_batch_rejects_before_the_library(monkeypatch):
    s = no_library_solver(monkeypatch)
    monkeypatch.setattr(api, "_solver_for", lambda tv, device: s)
    tv = api.generate_TV_args({}, {"semantics": "cuda"})
    with pytest.raises(N.Tvl1Error, match="all be uint8 or all float32"):
        api.TVL1_solve_batch([u8()], [f32()], tv)
    with pytest.raises(N.Tvl1Error, match="per pair"):
        api.TVL1_solve_batch([u8()] * 2, [u8()] * 2, tv, init_flows=[flow()])


def test_stacks_and_init_are_lists():
    f0, f1, init = N.check_batch_ex(np.zeros((3, 4, 5), np.float32), np.ones((3, 4, 5), np.float32),
                                    [flow() for _ in range(3)])
    assert len(f0) == len(f1) == len(init) == 3 and f1[2][0, 0] == 1 and f0[0].dtype == np.float32
    assert all(u.flags.c_contiguous and v.shape == (4, 5) for u, v in init)
    assert N.check_batch_ex([u8()], [u8()])[2] is None
