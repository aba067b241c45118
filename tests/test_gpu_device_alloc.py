"""Outputs the library allocates itself (a caching pool over qlnlp_device_alloc's blocks): compressible where the device
offers it, plain memory otherwise, bit-identical results either way, 16-byte aligned rows, reused instead of reallocated,
and a lifetime of their own."""
import ctypes as C
import gc

import numpy as np
import pytest

import quadruped_landing_b200 as ql
from conftest import perturbed_batch
from quadruped_landing_b200.evaluator import _device_empty, device_alloc_info, even_ld

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def _compression_supported(device=0):
    """CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED (107), asked of the driver directly rather than of the library"""
    attr = C.c_int(0)
    cuda = C.CDLL("libcuda.so.1")
    assert cuda.cuInit(0) == 0
    assert cuda.cuDeviceGetAttribute(C.byref(attr), 107, device) == 0
    return bool(attr.value)


def _batch(p, B, seed=0):
    Z = perturbed_batch(p, [ql.initial_guess(p)], B, 1e-2, seed)
    return torch.from_numpy(Z).cuda()


def _plain(nlp, B, want, width_of):
    out = {}
    for k in want:
        w = width_of[k]
        out[k] = (torch.empty(B, dtype=torch.float64, device="cuda") if w is None else
                  torch.empty((B, even_ld(w)), dtype=torch.float64, device="cuda")[:, :w])
    return out


def test_outputs_are_compressible_when_the_device_supports_it():
    supported = _compression_supported()
    nlp = ql.HybridNLP.from_problem(ql.default_problem())
    out = nlp.eval_batch(_batch(nlp.prob, 64))
    for k in ("f", "grad", "g", "jac"):
        info = device_alloc_info(out[k])
        assert info["compressible"] == int(supported), k
        assert info["device"] == 0
    torch.cuda.synchronize()


# five kernel instantiations: no Jacobian, SPARSE_BLOCK, SPARSE_TRUE, kinematic SPARSE_BLOCK, kinematic SPARSE_TRUE
CASES = [("block", False, ("f", "grad", "g")), ("block", False, ("f", "grad", "g", "jac")),
         ("true", False, ("f", "grad", "g", "jac")), ("block", True, ("f", "g", "jac")), ("true", True, ("g", "jac"))]


@pytest.mark.parametrize("B", [4096, 65536])
@pytest.mark.parametrize("pattern,kin,want", CASES)
def test_bit_identical_to_caller_buffers(B, pattern, kin, want):
    p = ql.default_problem()
    nlp = ql.HybridNLP.from_problem(p, pattern=pattern, kinematics=kin)
    Zb = _batch(p, 4096, seed=B)
    Z = Zb.repeat(B // 4096, 1)
    widths = {"f": None, "grad": nlp.n_nlp, "g": nlp.m_nlp, "jac": nlp.nnz_batch}
    mine = nlp.eval_batch(Z, want=want)
    theirs = nlp.eval_batch(Z, want=want, out=_plain(nlp, B, want, widths))
    torch.cuda.synchronize()
    for k in want:
        assert torch.equal(mine[k], theirs[k]), k
    del mine, theirs, Z
    torch.cuda.empty_cache()


def test_rows_are_16_byte_aligned_with_even_ld():
    nlp = ql.HybridNLP.from_problem(ql.default_problem(), pattern="true", hessian=True)
    for B in (1, 2, 37):
        out = nlp.alloc_outputs(B)
        for k, w in (("grad", nlp.n_nlp), ("g", nlp.m_nlp), ("jac", nlp.nnz_batch)):
            t = out[k]
            assert t.shape == (B, w) and t.stride() == (even_ld(w), 1), k
            assert t.data_ptr() % 256 == 0, k
        assert out["f"].data_ptr() % 256 == 0
        Z = _batch(nlp.prob, B)
        mu = torch.zeros((B, nlp.m_nlp), dtype=torch.float64, device="cuda")
        H = nlp.eval_hessian_batch(Z, mu)
        assert H.stride() == (even_ld(nlp.nnz_hess), 1) and H.data_ptr() % 16 == 0
        G = nlp.initial_guess_batch(torch.from_numpy(np.tile(nlp.prob.x0, (B, 1))).cuda())
        assert G.stride() == (even_ld(nlp.n_nlp), 1) and G.data_ptr() % 16 == 0
        device_alloc_info(H), device_alloc_info(G)
    torch.cuda.synchronize()


def test_tensors_outlive_the_handle():
    p = ql.default_problem()
    Z = _batch(p, 128)
    nlp = ql.HybridNLP.from_problem(p)
    out = nlp.eval_batch(Z)
    ref = {k: v.clone() for k, v in nlp.eval_batch(Z, out=_plain(nlp, 128, out, {"f": None, "grad": nlp.n_nlp,
                                                                                 "g": nlp.m_nlp, "jac": nlp.nnz_batch})).items()}
    torch.cuda.synchronize()
    del nlp
    gc.collect()
    for k in ref:                                   # still readable and unchanged after qlnlp_destroy
        assert torch.equal(out[k], ref[k]), k
    assert device_alloc_info(out["jac"])["device"] == 0


def test_dropped_outputs_are_reused():
    """A loop that lets each result go allocates nothing new: the pool hands the freed rows back in stream order."""
    p = ql.default_problem()
    nlp = ql.HybridNLP.from_problem(p)
    Z = _batch(p, 512)
    ptrs = set()
    for _ in range(5):
        out = nlp.eval_batch(Z)
        ptrs.add(out["jac"].data_ptr())
        del out
    assert len(ptrs) == 1
    torch.cuda.synchronize()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two devices")
def test_freed_on_its_own_device():
    p = ql.default_problem()
    nlp = ql.HybridNLP.from_problem(p, device=1)
    with torch.cuda.device(1):
        Z = torch.from_numpy(perturbed_batch(p, [ql.initial_guess(p)], 16, 1e-2, 0)).cuda()
    out = nlp.eval_batch(Z)
    assert out["jac"].device == torch.device("cuda", 1) and device_alloc_info(out["jac"])["device"] == 1
    del nlp
    torch.cuda.set_device(0)
    del out                                         # freed on device 1 while device 0 is current
    gc.collect()
    assert torch.cuda.current_device() == 0
    torch.cuda.synchronize(1)


def test_plain_memory_on_request():
    """With the "compressible" option off the outputs are ordinary torch memory (cudaIpcGetMemHandle works on it) and the
    bits are the same."""
    p = ql.default_problem()
    Z = _batch(p, 256)
    nlp = ql.HybridNLP.from_problem(p)
    comp = nlp.eval_batch(Z)
    nlp.set_option("compressible", 0)
    plain = nlp.eval_batch(Z)
    torch.cuda.synchronize()
    for k in comp:
        with pytest.raises(ql.QlnlpError):
            device_alloc_info(plain[k])
        assert torch.equal(comp[k], plain[k]), k
    nlp.set_option("compressible", 1)


class _Raw:
    """A qlnlp_device_alloc block seen by torch (``__cuda_array_interface__``); freed with the object."""

    def __init__(self, ptr, nbytes):
        self.ptr = ptr
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr.value, False), "version": 2}

    def __del__(self):
        ql.load_library().qlnlp_device_free(self.ptr)


def test_driver_refusal_is_served_with_plain_memory():
    """A compressible request the driver refuses (as it does when compressible backing runs out) is served with
    cudaMalloc memory, which the evaluator writes the same bits into."""
    p = ql.default_problem()
    nlp = ql.HybridNLP.from_problem(p)
    L = ql.load_library()
    B, ld = 64, even_ld(nlp.nnz_batch)
    ptr = C.c_void_p()
    assert L.qlnlp_debug_refuse_compressible(1) == 0
    assert L.qlnlp_device_alloc(nlp._h, B * ld * 8, C.byref(ptr)) == 0
    raw = torch.as_tensor(_Raw(ptr, B * ld * 8), device="cuda")
    assert ql.evaluator.device_alloc_info(raw)["compressible"] == 0
    jac = raw.view(torch.float64).view(B, ld)[:, :nlp.nnz_batch]
    Z = _batch(p, B)
    nlp.eval_batch(Z, want=("jac",), out={"jac": jac})
    ref = nlp.eval_batch(Z, want=("jac",))["jac"]
    torch.cuda.synchronize()
    assert device_alloc_info(ref)["compressible"] == int(_compression_supported())
    assert torch.equal(jac, ref)


def test_request_larger_than_the_device():
    """Refused as compressible and then by cudaMalloc: an out-of-memory error, and the next request is served."""
    nlp = ql.HybridNLP.from_problem(ql.default_problem())
    L = ql.load_library()
    p = C.c_void_p()
    total = torch.cuda.get_device_properties(0).total_memory
    assert L.qlnlp_device_alloc(nlp._h, 4 * total, C.byref(p)) == ql.evaluator.QLNLP_ENOMEM
    assert not p.value and b"cudaMalloc" in L.qlnlp_last_error()
    assert L.qlnlp_device_alloc(nlp._h, 1 << 20, C.byref(p)) == 0      # and the next request is served
    assert L.qlnlp_device_free(p) == 0


@pytest.mark.parametrize("N,kt,im", [(61, 21, 1), (2, 1, 1), (33, 33, 2)])
def test_no_write_outside_the_rows_on_library_memory(N, kt, im):
    """The canaries of test_gpu_parity.test_no_write_outside_the_rows, with the guarded buffers themselves taken from the
    library's output pool (compressible lines around the rows)."""
    p = ql.build_problem(N=N, k_trans=kt, init_mode=im)
    nlp = ql.HybridNLP.from_problem(p)
    B, guard, sentinel = 37, 3, -7.25
    Z = perturbed_batch(p, [ql.initial_guess(p) if kt > 1 else np.zeros(p.n_nlp)], B, 1e-2, 5)
    widths = {"grad": nlp.n_nlp, "g": nlp.m_nlp, "jac": nlp.nnz_block}
    for pad in (2, 3):                              # at least `pad` spare columns after every row
        ts = _device_empty(0, [(B + 2 * guard, w + pad, torch.float64) for w in widths.values()] +
                           [(B + 2 * guard, None, torch.float64)])
        big, views = {}, {}
        for (k, w), t in zip(widths.items(), ts):
            big[k] = t.fill_(sentinel)
            views[k] = big[k][guard:guard + B, :w]
        fbig = ts[-1].fill_(sentinel)
        views["f"] = fbig[guard:guard + B]
        assert all(device_alloc_info(t)["device"] == 0 for t in ts)
        out = nlp.eval_batch(torch.from_numpy(Z).cuda(), out=dict(views))
        torch.cuda.synchronize()
        for k, w in widths.items():
            assert bool((big[k][:guard] == sentinel).all()) and bool((big[k][guard + B:] == sentinel).all()), k
            assert bool((big[k][:, w:] == sentinel).all()), k
            assert not bool((out[k] == sentinel).any()), k
        assert bool((fbig[:guard] == sentinel).all()) and bool((fbig[guard + B:] == sentinel).all())
