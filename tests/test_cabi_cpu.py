"""The C-ABI shared library: loads, exports every symbol include/qlnlp.h declares, answers the host-only
queries, validates arguments, and refuses to evaluate without a GPU (no CPU fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import quadruped_landing_b200 as ql
from quadruped_landing_b200 import evaluator as ev

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def test_header_symbols_are_exported():
    hdr = open(os.path.join(ROOT, "include", "qlnlp.h")).read()
    declared = set(re.findall(r"\b(qlnlp_[a-z_]+)\s*\(", hdr))
    assert declared == set(ql.EXPORTED_SYMBOLS)
    L = ql.load_library()
    for name in declared:
        assert hasattr(L, name), name
    assert L.qlnlp_version() == 2


def test_host_queries_work_without_a_device():
    nlp = ql.HybridNLP.from_problem(ql.default_problem())
    assert (nlp.num_primals(), nlp.num_duals(), nlp.nnz_block) == (1215, 1093, 32161)
    assert nlp.features_available() == ["Grad", "Jac"] and nlp.initialize(["Grad"]) is None
    lb, ub = nlp.constraint_bounds()
    assert not lb.any() and not ub[:1032].any() and np.all(np.isinf(ub[1032:]))       # nlp.jl:66-69
    xl, xu = nlp.variable_bounds()
    # main.ipynb:222-223: 120 variables with only lower bounds, 121 with both
    only_lower = np.isfinite(xl) & ~np.isfinite(xu)
    both = np.isfinite(xl) & np.isfinite(xu)
    assert only_lower.sum() == 120 and both.sum() == 121
    assert [len(c) for c in nlp.cinds] == [15, 14, 900, 61, 41, 1, 61] and nlp.cinds[-1][-1] == 1093
    assert nlp.xinds[1][0] == 21 and nlp.uinds[0][0] == 16 and nlp.modes[19] == 1 and nlp.modes[20] == 3


def test_launch_geometry_arithmetic_for_the_b200():
    """Two integer rules of the launcher that went wrong silently once (profiles/r02_kernel_ab.md): the shared-memory
    carve-out is a percentage of the UNIFIED 256 KB (72..76 % selects the 196 KB configuration, 79 % and more 228 KB),
    and a SPARSE_BLOCK launch asks for so much shared memory that per_sm CTAs fit on an SM but per_sm + 1 never do."""
    import ctypes as C
    from quadruped_landing_b200.evaluator import load_library
    lib = load_library()
    per_sm_bytes, optin = 233472, 232448                      # sm_100: 228 KB per SM, 227 KB per block
    out = (C.c_int64 * 2)()
    for per_sm, smem in ((6, 27776), (5, 27776), (8, 27776), (4, 40000)):
        assert lib.qlnlp_debug_launch_geometry(per_sm_bytes, optin, per_sm, smem, out) == 0
        padded, pct = out[0], out[1]
        assert padded >= smem and padded % 128 == 0 and padded <= optin
        assert per_sm * (padded + 1024) <= per_sm_bytes                     # per_sm CTAs fit ...
        if padded > smem:
            assert (per_sm + 1) * (padded + 1024) > per_sm_bytes            # ... and one more never does
        need_kb = per_sm * (padded + 1024) / 1024
        cfg_kb = min(k for k in (0, 8, 16, 32, 64, 100, 132, 164, 196, 228) if k >= need_kb)
        # what the driver does with the percentage (measured on a B200): bytes = pct % of 256 KB, rounded UP to a configuration
        chosen = min(k for k in (0, 8, 16, 32, 64, 100, 132, 164, 196, 228) if k * 1024 >= pct * 262144 // 100)
        assert chosen == cfg_kb, (per_sm, smem, padded, pct, chosen, cfg_kb)
    assert lib.qlnlp_debug_launch_geometry(per_sm_bytes, optin, 6, 27776, out) == 0
    assert (out[0], out[1]) == (32384, 76)                                   # the default instance's headline launch


def test_reference_constructor_signature():
    p = ql.default_problem()
    xi, xt = ql.default_states()
    Xref, Uref = ql.reference_trajectory(p.model, 61, 21, xt, 1, 0.009)
    Q = np.diag([10.0] * 14 + [0.0])
    R = np.diag([1e-3, 1e-2, 1e-3, 1e-2, 0.0])
    obj = [ql.LQRCost(Q, R, Xref[k], Uref[k]) for k in range(60)] + [ql.LQRCost(Q, R * 0, Xref[60], Uref[0])]
    nlp = ql.HybridNLP(p.model, obj, 1, 21, 61, xi, xt)            # nlp.jl:33-36 argument order
    assert nlp.use_sparse_jacobian is False and nlp.nnz == 1093 * 1215   # reference default: dense structure
    assert np.array_equal(nlp.prob.q, p.q) and np.array_equal(nlp.prob.c, p.c)
    X, U = nlp.unpackZ(ql.initial_guess(p))
    assert np.array_equal(nlp.packZ(X, U), ql.initial_guess(p))


@pytest.mark.parametrize("kw", [dict(N=1), dict(k_trans=0), dict(k_trans=62), dict(init_mode=3)])
def test_create_rejects_bad_descriptors(kw):
    p = ql.default_problem()
    L = ql.load_library()
    d = ev._Desc()
    d.N, d.k_trans, d.init_mode = kw.get("N", 61), kw.get("k_trans", 21), kw.get("init_mode", 1)
    d.Q, d.R, d.q, d.r, d.c = (a.ctypes.data for a in (p.Q, p.R, p.q, p.r, p.c))
    h = C.c_void_p()
    assert L.qlnlp_create(C.byref(d), 0, 0, C.byref(h)) == ev.QLNLP_EINVAL
    assert h.value is None and len(L.qlnlp_last_error()) > 0


@pytest.mark.skipif(_has_gpu(), reason="checks the no-GPU behaviour")
def test_evaluation_fails_loudly_without_a_gpu():
    nlp = ql.HybridNLP.from_problem(ql.default_problem())
    with pytest.raises(ql.QlnlpError) as e:
        nlp.eval_objective(ql.initial_guess(nlp.prob))
    assert e.value.code == ev.QLNLP_ENODEVICE and "no CPU path" in str(e.value)
    with pytest.raises(ql.QlnlpError):
        nlp.eval_batch_host(np.zeros((2, 1215)))
    for devices in ([0], [0, 1]):                           # multi-device handles: the failing shard is named
        multi = ql.HybridNLP.from_problem(nlp.prob, devices=devices)
        with pytest.raises(ql.QlnlpError) as e:
            multi.eval_batch_host(np.zeros((2, 1215)))
        assert e.value.code == ev.QLNLP_ENODEVICE and f"error {ev.QLNLP_ENODEVICE}: device 0: no CUDA device" in str(e.value)


def test_allocation_failure_hook_reports_what_it_had_left():
    """qlnlp_debug_fail_alloc returns what the previous setting still had to go (-1: disarmed or used up), which is how
    the GPU sweep over allocation points tells an injected failure from one it never reached.  Arming allocates nothing."""
    L = ql.load_library()
    blocks = L.qlnlp_debug_owned_blocks()
    assert L.qlnlp_debug_fail_alloc(3) == -1
    assert L.qlnlp_debug_fail_alloc(0) == 3
    assert L.qlnlp_debug_fail_alloc(-7) == 0
    assert L.qlnlp_debug_fail_alloc(-1) == -1
    assert L.qlnlp_debug_owned_blocks() == blocks


@pytest.mark.parametrize("devices", [[0], [0, 1]])
def test_multi_device_handle_answers_like_a_plain_handle(devices):
    """qlnlp_create_multi needs no device until it evaluates: its host-side answers equal those of a plain handle, its
    devices split the host cores, and the entry points that take a single-device handle refuse it."""
    p = ql.default_problem()
    L = ql.load_library()
    one = ql.HybridNLP.from_problem(p)
    multi = ql.HybridNLP.from_problem(p, devices=devices)
    ids, n = (C.c_int * 4)(), C.c_int()
    assert L.qlnlp_devices(multi._h, ids, 4, C.byref(n)) == 0 and list(ids[:n.value]) == devices
    assert (multi.n_nlp, multi.m_nlp, multi.nnz, multi.nnz_block) == (one.n_nlp, one.m_nlp, one.nnz, one.nnz_block)
    for a, b in zip(multi.jacobian_structure_arrays(), one.jacobian_structure_arrays()):
        assert np.array_equal(a, b)
    assert np.array_equal(multi._debug_segments(), one._debug_segments())
    assert np.array_equal(multi._debug_vals_map(), one._debug_vals_map())
    jm, j1 = np.full((5, multi.nnz_batch), np.nan), np.full((5, one.nnz_batch), np.nan)
    multi.register_host_output(jm)
    one.register_host_output(j1)
    assert not np.isnan(jm).any() and np.array_equal(jm, j1)
    threads = one.host_path_info()["threads_per_device"]
    assert multi.host_path_info()["threads_per_device"] == max(1, threads // len(devices))
    with pytest.raises(ql.QlnlpError) as e:
        multi.set_option("bogus", 1)
    assert e.value.code == ev.QLNLP_EINVAL
    io, rg = ev._BatchIO(), ev._RaggedIO()
    refusals = [
        (lambda: L.qlnlp_eval_batch_device(multi._h, 1, C.byref(io), None),
         "multi-device handle: use qlnlp_eval_batch_device_multi"),
        (lambda: L.qlnlp_eval_ragged_device(multi._h, 1, C.byref(io), C.byref(rg), None),
         "multi-device handle: ragged launches take a single-device handle"),
        (lambda: L.qlnlp_eval_ragged_classes((C.c_void_p * 1)(multi._h.value), 1, 1, C.byref(io), C.byref(rg), None, None),
         "multi-device handle: ragged launches take single-device handles"),
        (lambda: L.qlnlp_eval_hessian_batch_device(multi._h, 1, None, 0, None, None, 0, None, 0, None),
         "multi-device handle: the Hessian takes a single-device handle"),
    ]
    for call, msg in refusals:
        assert call() == ev.QLNLP_EINVAL and L.qlnlp_last_error().decode() == msg


def test_batch_argument_checks_need_no_device():
    """The batched entry points on device pointers check their arguments before they bind the device, so an invalid
    call is refused the same way with or without a GPU."""
    prob = ql.build_problem(N=5, k_trans=3)
    L = ql.load_library()
    nlp = ql.HybridNLP.from_problem(prob, hessian=True)
    n, m, nnz, nh = nlp.n_nlp, nlp.m_nlp, nlp.nnz, nlp.nnz_hess
    Z, g, jac, lam, H = np.zeros(n + 1), np.zeros(m + 1), np.zeros(nnz + 1), np.zeros(m + 1), np.zeros(nh + 1)
    off = np.zeros(2, dtype=np.int64)

    def io(**kw):
        d = ev._BatchIO()
        d.Z, d.ldz = Z.ctypes.data, n
        for k, v in kw.items():
            setattr(d, k, v)
        return d

    def rg(**kw):
        r = ev._RaggedIO()
        r.z_off = off.ctypes.data
        for k, v in kw.items():
            setattr(r, k, v)
        return r

    def batch(B, d):
        return L.qlnlp_eval_batch_device(nlp._h, B, None if d is None else C.byref(d), None)

    def ragged(B, d, r):
        return L.qlnlp_eval_ragged_device(nlp._h, B, None if d is None else C.byref(d), C.byref(r), None)

    def classes(B, d, r):
        return L.qlnlp_eval_ragged_classes((C.c_void_p * 1)(nlp._h.value), 1, B, None if d is None else C.byref(d),
                                           C.byref(r), None, None)

    def hess(B, Zp=Z.ctypes.data, ldz=n, lp=lam.ctypes.data, ldl=m, hp=H.ctypes.data, ldh=nh):
        return L.qlnlp_eval_hessian_batch_device(nlp._h, B, Zp, ldz, None, lp, ldl, hp, ldh, None)

    invalid = [
        lambda: batch(-1, io()), lambda: batch(1, None), lambda: batch(1, io(Z=None)), lambda: batch(2, io(ldz=n - 1)),
        lambda: batch(2, io(g=g.ctypes.data, ldg=m - 1)), lambda: batch(2, io(jac=jac.ctypes.data, ldjac=nnz - 1)),
        lambda: batch(1, io(Z=Z.ctypes.data + 4)),
        lambda: ragged(-1, io(), rg()), lambda: ragged(1, None, rg()), lambda: ragged(1, io(), rg(z_off=None)),
        lambda: ragged(1, io(g=g.ctypes.data), rg()), lambda: ragged(1, io(jac=jac.ctypes.data), rg()),
        lambda: classes(-1, io(), rg()), lambda: classes(1, None, rg()), lambda: classes(1, io(), rg(z_off=None)),
        lambda: classes(1, io(jac=jac.ctypes.data), rg()),
        lambda: hess(-1), lambda: hess(1, Zp=None), lambda: hess(1, lp=None), lambda: hess(1, hp=None),
        lambda: hess(2, ldz=n - 1), lambda: hess(2, ldl=m - 1), lambda: hess(2, ldh=nh - 1),
    ]
    for i, call in enumerate(invalid):
        assert call() == ev.QLNLP_EINVAL, (i, L.qlnlp_last_error())
    assert batch(0, None) == ev.QLNLP_OK and hess(0, Zp=None, lp=None, hp=None) == ev.QLNLP_OK
    if not _has_gpu():                                     # valid arguments (host memory here) reach the device
        for call in (lambda: batch(1, io()), lambda: ragged(1, io(), rg()), lambda: classes(1, io(), rg()),
                     lambda: hess(1)):
            assert call() == ev.QLNLP_ENODEVICE


def _build_demo(tmp_path):
    import subprocess
    exe = str(tmp_path / "qlnlp_demo")
    ql.load_library()                                      # makes sure libqlnlp.so exists
    subprocess.run(["gcc", "-O2", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "qlnlp_demo.c"),
                    "-L" + os.path.join(ROOT, "quadruped_landing_b200"), "-lqlnlp", "-lm", "-o", exe], check=True)
    env = dict(os.environ, LD_LIBRARY_PATH=os.path.join(ROOT, "quadruped_landing_b200"))
    return subprocess.run([exe], capture_output=True, text=True, env=env, timeout=300)


@pytest.mark.skipif(_has_gpu(), reason="checks the no-GPU behaviour")
def test_plain_c_program_links_and_fails_loudly_without_a_gpu(tmp_path):
    """examples/qlnlp_demo.c uses nothing but include/qlnlp.h (Ipopt-shaped C callbacks): it must link against the
    shared library, answer the host-only queries and report the missing device instead of computing on the CPU."""
    r = _build_demo(tmp_path)
    assert "variables 1215  constraints 1093  jacobian nonzeros 32161" in r.stdout
    assert r.returncode == 2 and "no CPU path" in r.stderr


@pytest.mark.gpu
def test_plain_c_program_reproduces_iteration_zero(tmp_path):
    """Same program on a B200: the objective at Z0 and the primal infeasibility Ipopt prints at iteration 0
    (src/main.ipynb:232: inf_pr 3.13e-01)."""
    r = _build_demo(tmp_path)
    assert r.returncode == 0, r.stderr
    assert "objective(Z0) = 1.5438467869136" in r.stdout and "inf_pr(Z0) = 3.13" in r.stdout
    assert "first structure entries: (1,1) (2,1) ... last (929,1215); J[0] = 1" in r.stdout
