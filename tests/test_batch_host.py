"""tvl1_calc_batch_u8 without a GPU: the symbol is exported, and the Python wrappers refuse malformed batches before
the library is called."""
import numpy as np
import pytest

from fibsem_optflow_b200 import _native as N


def test_batch_symbols_exported(native):
    for name in ("tvl1_calc_batch_u8", "tvl1_last_readbacks"):
        assert hasattr(native.lib(), name) and name in native.EXPORTS


def no_library_solver(monkeypatch):
    """a Solver that was never created, with every library call an error"""
    def refuse():
        raise AssertionError("the library was called")
    monkeypatch.setattr(N, "lib", refuse)
    s = object.__new__(N.Solver)
    s.handle, s.device = 1, 0
    return s


@pytest.mark.parametrize("frames0, frames1, text", [
    ([], [], "non-empty"),
    ([np.zeros((4, 5), np.uint8)], [], "equally long"),
    ([np.zeros((4, 5), np.uint8)] * 2, [np.zeros((4, 5), np.uint8)], "equally long"),
    ([np.zeros((4, 5), np.float32)], [np.zeros((4, 5), np.float32)], "uint8"),
    ([np.zeros((4, 5, 3), np.uint8)], [np.zeros((4, 5, 3), np.uint8)], "2-D"),
    ([np.zeros((4, 5), np.uint8)], [np.zeros((5, 4), np.uint8)], "one size"),
    ([np.zeros((4, 5), np.uint8), np.zeros((4, 6), np.uint8)], [np.zeros((4, 5), np.uint8)] * 2, "one size"),
    ([np.zeros((0, 5), np.uint8)], [np.zeros((0, 5), np.uint8)], "empty"),
])
def test_calc_batch_rejects_malformed_lists(monkeypatch, frames0, frames1, text):
    s = no_library_solver(monkeypatch)
    with pytest.raises(N.Tvl1Error, match=text):
        s.calc_batch(frames0, frames1)


def test_calc_batch_device_rejects_unequal_lists(monkeypatch):
    s = no_library_solver(monkeypatch)
    with pytest.raises(N.Tvl1Error, match="equally long"):
        s.calc_batch_device([1, 2], 8, [3, 4], 8, 8, 8, [5], [6, 7], 32)
    with pytest.raises(N.Tvl1Error, match="non-empty"):
        s.calc_batch_device([], 8, [], 8, 8, 8, [], [], 32)


def test_stack_is_a_list_of_frames():
    f0, f1 = N.check_batch_frames(np.zeros((3, 4, 5), np.uint8), np.ones((3, 4, 5), np.uint8))
    assert len(f0) == len(f1) == 3 and f0[0].shape == (4, 5) and f1[2][0, 0] == 1
