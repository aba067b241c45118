"""Argument checks of the device output allocator (qlnlp_device_alloc / _free / _alloc_info), which run before any
device work, and its refusal without a device."""
import ctypes as C

import pytest

import quadruped_landing_b200 as ql
from quadruped_landing_b200.evaluator import QLNLP_EINVAL, QLNLP_ENODEVICE, QLNLP_OK


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


@pytest.fixture(scope="module")
def nlp():
    return ql.HybridNLP.from_problem(ql.default_problem())


def test_alloc_argument_checks(nlp):
    L = ql.load_library()
    p = C.c_void_p(1234)
    assert L.qlnlp_device_alloc(None, 64, C.byref(p)) == QLNLP_EINVAL
    assert b"null handle" in L.qlnlp_last_error()
    assert L.qlnlp_device_alloc(nlp._h, 64, None) == QLNLP_EINVAL
    for bad in (0, -1, -(1 << 40)):
        p = C.c_void_p(1234)
        assert L.qlnlp_device_alloc(nlp._h, bad, C.byref(p)) == QLNLP_EINVAL
        assert b"bad allocation request" in L.qlnlp_last_error()


def test_free_and_info_refuse_foreign_pointers():
    L = ql.load_library()
    assert L.qlnlp_device_free(None) == QLNLP_OK                       # like free(NULL)
    foreign = C.create_string_buffer(64)
    assert L.qlnlp_device_free(C.cast(foreign, C.c_void_p)) == QLNLP_EINVAL
    assert b"was not returned by qlnlp_device_alloc" in L.qlnlp_last_error()
    info = (C.c_int64 * 3)()
    assert L.qlnlp_device_alloc_info(C.cast(foreign, C.c_void_p), info) == QLNLP_EINVAL
    assert L.qlnlp_device_alloc_info(None, info) == QLNLP_EINVAL
    assert L.qlnlp_device_alloc_info(C.cast(foreign, C.c_void_p), None) == QLNLP_EINVAL


def test_compressible_option_reaches_the_python_allocations(nlp):
    """The option the handle takes is the one the Python layer's output allocations follow."""
    assert nlp._compressible
    nlp.set_option("compressible", 0)
    assert not nlp._compressible
    nlp.set_option("compressible", 1)
    assert nlp._compressible
    with pytest.raises(ql.QlnlpError):
        nlp.set_option("compressibel", 0)


def test_alloc_outputs_refuses_a_foreign_device(nlp):
    """A single-device evaluator allocates its outputs on its own device only."""
    pytest.importorskip("torch")
    with pytest.raises(ValueError):
        nlp.alloc_outputs(4, device=nlp.device + 1)


def test_alloc_outputs_rejects_unknown_names(nlp):
    pytest.importorskip("torch")
    with pytest.raises(ValueError):
        nlp.alloc_outputs(4, want=("f", "hess"))


@pytest.mark.skipif(_has_gpu(), reason="checks the refusal without a device")
def test_alloc_without_a_device(nlp):
    L = ql.load_library()
    p = C.c_void_p(1234)
    assert L.qlnlp_device_alloc(nlp._h, 64, C.byref(p)) == QLNLP_ENODEVICE
    assert not p.value
    assert b"no CUDA device" in L.qlnlp_last_error()
