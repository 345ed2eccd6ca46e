"""The uint32 bindings (Bfv32, EvaluationKey32) check array shapes and key sizes before the library is reached: a
mis-shaped uint32 array is refused with HeError -1 instead of letting libhecuda read or write past the numpy buffer.
Needs neither a GPU nor the library."""
import numpy as np
import pytest

import hecuda


class StandInContext:
    L, degree, _h = 2, 16, None


@pytest.fixture(autouse=True)
def no_library(monkeypatch):
    def load_library(*args, **kwargs):
        pytest.fail("the library was reached with a mis-shaped array")

    monkeypatch.setattr(hecuda, "load_library", load_library)


def u32(*shape):
    return np.zeros(shape, dtype=np.uint32)


KEY = object()  # never dereferenced: the shape check comes first


CALLS = {
    "mulAssign": lambda g: hecuda.Bfv32.mulAssign(g, u32(1, 2, 2, 16), u32(1, 2, 2, 8)),
    "relinearize": lambda g: hecuda.Bfv32.relinearize(g, u32(1, 3, 2, 8), KEY),
    "modSwitchDown": lambda g: hecuda.Bfv32.modSwitchDown(g, u32(1, 2, 2, 8)),
    "mulRelinearize": lambda g: hecuda.Bfv32.mulRelinearize(g, u32(1, 2, 2, 16), u32(1, 2, 3, 16), KEY),
    "relinearizeModSwitchDown": lambda g: hecuda.Bfv32.relinearizeModSwitchDown(g, u32(1, 2, 2, 16), KEY),
    "applyGalois": lambda g: hecuda.Bfv32.applyGalois(g, u32(1, 3, 2, 16), 3, KEY),
    "innerProductCiphertexts": lambda g: hecuda.Bfv32.innerProductCiphertexts(g, u32(2, 2, 2, 2, 16), u32(2, 2, 2, 2, 8)),
    "forwardNtt": lambda g: hecuda.Bfv32.forwardNtt(g, u32(2, 2, 8)),
    "inverseNtt": lambda g: hecuda.Bfv32.inverseNtt(g, u32(2, 2, 8)),
    "liftQToQBsk": lambda g: hecuda.Bfv32.liftQToQBsk(g, u32(2, 3, 16)),
    "floorQBskToQ": lambda g: hecuda.Bfv32.floorQBskToQ(g, u32(2, 2, 16)),
}


@pytest.mark.parametrize("method", sorted(CALLS))
def test_bfv32_rejects_mis_shaped_arrays(method):
    with pytest.raises(hecuda.HeError) as ei:
        CALLS[method](StandInContext())
    assert ei.value.code == -1


def test_evaluation_key32_rejects_a_wrong_sized_relinearization_key():
    g = StandInContext()
    with pytest.raises(hecuda.HeError) as ei:
        hecuda.EvaluationKey32(g, u32(g.L, 2, g.L + 1, g.degree - 1))
    assert ei.value.code == -1


def test_evaluation_key32_rejects_a_wrong_sized_galois_key():
    g = StandInContext()
    key = hecuda.EvaluationKey32.__new__(hecuda.EvaluationKey32)  # a key without a library handle
    key.context, key._h, key.galoisElements = g, None, []
    with pytest.raises(hecuda.HeError) as ei:
        key.setGaloisKey(3, u32(g.L, 2, g.L, g.degree))
    assert ei.value.code == -1
