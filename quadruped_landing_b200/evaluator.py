"""Host-side mirror of the reference's evaluator interface over the C-ABI CUDA library.

``HybridNLP`` keeps the reference's names and argument meaning (src/nlp.jl:13-114 and the
``MOI.*`` methods of src/moi.jl:1-33): ``eval_objective``, ``eval_objective_gradient``,
``eval_constraint``, ``eval_constraint_jacobian``, ``jacobian_structure``,
``features_available``, ``initialize``, ``num_primals``, ``num_duals``, ``packZ``/``unpackZ``.
Every numeric call goes through ``libqlnlp.so`` (include/qlnlp.h) and runs on the GPU; there is
no CPU implementation in this package -- if the library or a B200 is missing the call raises.

Batched evaluation (many decision vectors per launch) has no counterpart in the reference; it
is exposed as ``eval_batch`` (device tensors, the timed path) and ``eval_batch_host``
(numpy / pinned host buffers, copies included).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np

from . import build as _build
from .problem import NX, NU, PlanarQuadruped, ProblemData, QuadraticCost, packZ as _packZ, unpackZ as _unpackZ

QLNLP_OK, QLNLP_EINVAL, QLNLP_ENODEVICE, QLNLP_ECUDA, QLNLP_ENOMEM = range(5)
JAC_SPARSE_BLOCK, JAC_DENSE, JAC_SPARSE_TRUE = 0, 1, 2
WITH_KINEMATICS = 0x100

# every symbol include/qlnlp.h declares
EXPORTED_SYMBOLS = (
    "qlnlp_version", "qlnlp_last_error", "qlnlp_create", "qlnlp_destroy", "qlnlp_dims",
    "qlnlp_jacobian_structure", "qlnlp_constraint_bounds", "qlnlp_variable_bounds",
    "qlnlp_eval_objective", "qlnlp_eval_objective_gradient", "qlnlp_eval_constraint",
    "qlnlp_eval_constraint_jacobian", "qlnlp_eval_batch_device", "qlnlp_eval_ragged_device", "qlnlp_eval_batch_host",
    "qlnlp_launch_info",
    "qlnlp_create_multi", "qlnlp_devices", "qlnlp_shard_bounds", "qlnlp_set_option", "qlnlp_eval_all",
    "qlnlp_eval_batch_device_multi", "qlnlp_synchronize", "qlnlp_host_output_register", "qlnlp_host_output_unregister",
    "qlnlp_host_pin", "qlnlp_host_unpin", "qlnlp_host_path_info", "qlnlp_host_alloc", "qlnlp_host_free",
    "qlnlp_eval_ragged_classes",
    "qlnlp_hessian_nnz", "qlnlp_hessian_structure", "qlnlp_eval_hessian_lagrangian", "qlnlp_eval_hessian_batch_device",
    "qlnlp_initial_guess_batch_device",
    "qlnlp_eval_jacobian_products_batch_device", "qlnlp_eval_hessian_product_batch_device",
    "qlnlp_eval_constraint_jacobian_product", "qlnlp_eval_constraint_jacobian_transpose_product",
    "qlnlp_eval_hessian_lagrangian_product",
    "qlnlp_kkt_solve_batch_device", "qlnlp_kkt_factor_size", "qlnlp_kkt_factor_batch_device",
    "qlnlp_kkt_solve_factored_batch_device", "qlnlp_kkt_residual_batch_device",
    "qlnlp_device_alloc", "qlnlp_device_free", "qlnlp_device_alloc_info",
)
_DEBUG_SYMBOLS = ("qlnlp_debug_segments", "qlnlp_debug_vals_map", "qlnlp_debug_build_rows", "qlnlp_debug_host_times",
                  "qlnlp_debug_launch_geometry", "qlnlp_debug_refuse_compressible", "qlnlp_debug_fail_alloc",
                  "qlnlp_debug_owned_blocks")


class QlnlpError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"qlnlp error {code}: {msg}")
        self.code = code


class _Model(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("g", "mb", "mf", "lb", "l1", "l2")]


class _Desc(C.Structure):
    _fields_ = [("N", C.c_int64), ("k_trans", C.c_int64), ("init_mode", C.c_int64),
                ("model", _Model), ("x0", C.c_double * 15), ("xf", C.c_double * 15),
                ("Q", C.c_void_p), ("R", C.c_void_p), ("q", C.c_void_p), ("r", C.c_void_p), ("c", C.c_void_p)]


class _BatchIO(C.Structure):
    _fields_ = [("Z", C.c_void_p), ("ldz", C.c_int64),
                ("x0", C.c_void_p), ("xf", C.c_void_p),
                ("f", C.c_void_p),
                ("grad", C.c_void_p), ("ldgrad", C.c_int64),
                ("g", C.c_void_p), ("ldg", C.c_int64),
                ("jac", C.c_void_p), ("ldjac", C.c_int64)]


class _ProductIO(C.Structure):
    _fields_ = [("w", C.c_void_p), ("ldw", C.c_int64), ("jw", C.c_void_p), ("ldjw", C.c_int64),
                ("y", C.c_void_p), ("ldy", C.c_int64), ("jty", C.c_void_p), ("ldjty", C.c_int64)]


class _KktIO(C.Structure):
    _fields_ = [("hess", C.c_void_p), ("ldhess", C.c_int64), ("jac", C.c_void_p), ("ldjac", C.c_int64),
                ("sx", C.c_void_p), ("ldsx", C.c_int64), ("dc", C.c_void_p), ("lddc", C.c_int64),
                ("r1", C.c_void_p), ("ldr1", C.c_int64), ("r2", C.c_void_p), ("ldr2", C.c_int64),
                ("px", C.c_void_p), ("ldpx", C.c_int64), ("pl", C.c_void_p), ("ldpl", C.c_int64),
                ("status", C.c_void_p)]


class _KktFactorIO(C.Structure):
    _fields_ = [("hess", C.c_void_p), ("ldhess", C.c_int64), ("jac", C.c_void_p), ("ldjac", C.c_int64),
                ("sx", C.c_void_p), ("ldsx", C.c_int64), ("dc", C.c_void_p), ("lddc", C.c_int64),
                ("factor", C.c_void_p), ("ldfactor", C.c_int64), ("status", C.c_void_p)]


class _KktRhsIO(C.Structure):
    _fields_ = [("factor", C.c_void_p), ("ldfactor", C.c_int64), ("nfactor", C.c_int64), ("index", C.c_void_p),
                ("r1", C.c_void_p), ("ldr1", C.c_int64), ("r2", C.c_void_p), ("ldr2", C.c_int64),
                ("px", C.c_void_p), ("ldpx", C.c_int64), ("pl", C.c_void_p), ("ldpl", C.c_int64),
                ("status", C.c_void_p)]


class _KktResidualIO(C.Structure):
    _fields_ = [("hess", C.c_void_p), ("ldhess", C.c_int64), ("jac", C.c_void_p), ("ldjac", C.c_int64),
                ("sx", C.c_void_p), ("ldsx", C.c_int64), ("dc", C.c_void_p), ("lddc", C.c_int64),
                ("r1", C.c_void_p), ("ldr1", C.c_int64), ("r2", C.c_void_p), ("ldr2", C.c_int64),
                ("px", C.c_void_p), ("ldpx", C.c_int64), ("pl", C.c_void_p), ("ldpl", C.c_int64),
                ("s1", C.c_void_p), ("lds1", C.c_int64), ("s2", C.c_void_p), ("lds2", C.c_int64)]


class _RaggedIO(C.Structure):
    _fields_ = [("index", C.c_void_p), ("z_off", C.c_void_p), ("g_off", C.c_void_p), ("jac_off", C.c_void_p),
                ("flags", C.c_int64)]


_lib = None
_lib_path = None


def load_library(rebuild_if_stale: bool = True):
    """dlopen libqlnlp.so (building it first if the sources are newer).  Raises if unavailable."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("QLNLP_LIB")          # experimental variants (tools/ab_bench.py)
    if not path:
        path = _build.LIB
        if rebuild_if_stale and _build.is_stale():
            path = _build.build()
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing: build it with `python -m quadruped_landing_b200.build` "
                           "(the evaluator has no CPU fallback)")
    L = C.CDLL(path)
    global _lib_path
    _lib_path = path
    vp, i64p = C.c_void_p, C.POINTER(C.c_int64)
    L.qlnlp_version.restype = C.c_int
    L.qlnlp_last_error.restype = C.c_char_p
    L.qlnlp_create.argtypes = [C.POINTER(_Desc), C.c_int, C.c_int, C.POINTER(vp)]
    L.qlnlp_destroy.argtypes = [vp]
    L.qlnlp_dims.argtypes = [vp, i64p, i64p, i64p, i64p]
    L.qlnlp_jacobian_structure.argtypes = [vp, vp, vp]
    L.qlnlp_constraint_bounds.argtypes = [vp, vp, vp]
    L.qlnlp_variable_bounds.argtypes = [vp, vp, vp]
    for name in ("qlnlp_eval_objective", "qlnlp_eval_objective_gradient", "qlnlp_eval_constraint",
                 "qlnlp_eval_constraint_jacobian"):
        getattr(L, name).argtypes = [vp, vp, vp]
    L.qlnlp_eval_batch_device.argtypes = [vp, C.c_int64, C.POINTER(_BatchIO), vp]
    L.qlnlp_eval_ragged_device.argtypes = [vp, C.c_int64, C.POINTER(_BatchIO), C.POINTER(_RaggedIO), vp]
    L.qlnlp_eval_batch_host.argtypes = [vp, C.c_int64, C.POINTER(_BatchIO)]
    L.qlnlp_eval_ragged_classes.argtypes = [C.POINTER(vp), C.c_int, C.c_int64, C.POINTER(_BatchIO), C.POINTER(_RaggedIO), vp, vp]
    L.qlnlp_launch_info.argtypes = [vp, i64p]
    L.qlnlp_debug_segments.argtypes = [vp, vp, C.c_int64, i64p]
    L.qlnlp_debug_vals_map.argtypes = [vp, vp, C.c_int64, i64p]
    L.qlnlp_debug_build_rows.argtypes = [vp, vp, C.c_int64, vp, C.c_int64, C.c_int64, C.c_int, C.c_int]
    L.qlnlp_debug_host_times.argtypes = [vp, C.POINTER(C.c_double)]
    L.qlnlp_debug_launch_geometry.argtypes = [C.c_int64, C.c_int64, C.c_int, C.c_int64, C.POINTER(C.c_int64)]
    L.qlnlp_create_multi.argtypes = [C.POINTER(_Desc), C.POINTER(C.c_int), C.c_int, C.c_int, C.POINTER(vp)]
    L.qlnlp_devices.argtypes = [vp, C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_int)]
    L.qlnlp_shard_bounds.argtypes = [C.c_int64, C.c_int, C.c_int, i64p, i64p]
    L.qlnlp_set_option.argtypes = [vp, C.c_char_p, C.c_int64]
    L.qlnlp_eval_all.argtypes = [vp, vp, vp, vp, vp, vp]
    L.qlnlp_eval_batch_device_multi.argtypes = [vp, i64p, C.POINTER(_BatchIO), C.POINTER(vp)]
    L.qlnlp_synchronize.argtypes = [vp]
    L.qlnlp_host_output_register.argtypes = [vp, vp, C.c_int64, C.c_int64]
    L.qlnlp_host_output_unregister.argtypes = [vp, vp]
    L.qlnlp_host_pin.argtypes = [vp, C.c_int64]
    L.qlnlp_host_unpin.argtypes = [vp]
    L.qlnlp_host_path_info.argtypes = [vp, i64p]
    L.qlnlp_hessian_nnz.argtypes = [vp, i64p]
    L.qlnlp_hessian_structure.argtypes = [vp, vp, vp]
    L.qlnlp_eval_hessian_lagrangian.argtypes = [vp, vp, C.c_double, vp, vp]
    L.qlnlp_eval_hessian_batch_device.argtypes = [vp, C.c_int64, vp, C.c_int64, vp, vp, C.c_int64, vp, C.c_int64, vp]
    L.qlnlp_initial_guess_batch_device.argtypes = [vp, C.c_int64, vp, vp, vp, C.c_int64, vp]
    L.qlnlp_eval_jacobian_products_batch_device.argtypes = [vp, C.c_int64, C.POINTER(_BatchIO), C.POINTER(_ProductIO), vp]
    L.qlnlp_eval_hessian_product_batch_device.argtypes = [vp, C.c_int64, vp, C.c_int64, vp, vp, C.c_int64, vp, C.c_int64,
                                                          vp, C.c_int64, vp]
    L.qlnlp_eval_constraint_jacobian_product.argtypes = [vp, vp, vp, vp]
    L.qlnlp_eval_constraint_jacobian_transpose_product.argtypes = [vp, vp, vp, vp]
    L.qlnlp_eval_hessian_lagrangian_product.argtypes = [vp, vp, vp, C.c_double, vp, vp]
    L.qlnlp_kkt_solve_batch_device.argtypes = [vp, C.c_int64, C.POINTER(_KktIO), vp]
    L.qlnlp_kkt_factor_size.argtypes = [vp, i64p]
    L.qlnlp_kkt_factor_batch_device.argtypes = [vp, C.c_int64, C.POINTER(_KktFactorIO), vp]
    L.qlnlp_kkt_solve_factored_batch_device.argtypes = [vp, C.c_int64, C.POINTER(_KktRhsIO), vp]
    L.qlnlp_kkt_residual_batch_device.argtypes = [vp, C.c_int64, C.POINTER(_KktResidualIO), vp]
    L.qlnlp_host_alloc.argtypes = [C.c_int64, C.POINTER(vp)]
    L.qlnlp_host_free.argtypes = [vp, C.c_int64]
    L.qlnlp_device_alloc.argtypes = [vp, C.c_int64, C.POINTER(vp)]
    L.qlnlp_device_free.argtypes = [vp]
    L.qlnlp_device_alloc_info.argtypes = [vp, i64p]
    L.qlnlp_debug_refuse_compressible.argtypes = [C.c_int]
    L.qlnlp_debug_fail_alloc.argtypes = [C.c_int]
    L.qlnlp_debug_owned_blocks.argtypes = []
    for name in [n for n in EXPORTED_SYMBOLS if n not in ("qlnlp_version", "qlnlp_last_error")] + list(_DEBUG_SYMBOLS):
        getattr(L, name).restype = C.c_int
    _lib = L
    return L


class _HostBlock:
    """Owner of a qlnlp_host_alloc block; numpy arrays made from it keep it alive through their ``base``."""

    def __init__(self, nbytes: int):
        self.nbytes = int(nbytes)
        self.ptr = C.c_void_p()
        rc = load_library().qlnlp_host_alloc(self.nbytes, C.byref(self.ptr))
        if rc != QLNLP_OK:
            raise QlnlpError(rc, load_library().qlnlp_last_error().decode())
        self.buf = (C.c_char * self.nbytes).from_address(self.ptr.value)

    def __del__(self):
        if getattr(self, "ptr", None) is not None and self.ptr.value and _lib is not None:
            _lib.qlnlp_host_free(self.ptr, self.nbytes)
            self.ptr = C.c_void_p()


def host_alloc(shape, dtype=np.float64) -> np.ndarray:
    """A zero-filled numpy array in page-locked host memory on 2 MB pages where the kernel grants them
    (``qlnlp_host_alloc``): the preferred home of the arrays handed to ``eval_batch_host``."""
    shape = (shape,) if isinstance(shape, int) else tuple(shape)
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    blk = _HostBlock(max(n, 1))
    a = np.frombuffer(blk.buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    a.flags.writeable = True
    _host_blocks[a.ctypes.data] = blk            # ctypes buffers do not keep python attributes: keep the owner here
    return a


_host_blocks = {}


def host_free(a: np.ndarray) -> None:
    """Release an array made by ``host_alloc`` (the array must not be used afterwards)."""
    _host_blocks.pop(a.ctypes.data, None)


def _check(rc: int):
    if rc != QLNLP_OK:
        raise QlnlpError(rc, load_library().qlnlp_last_error().decode())


def _check_sigma(sigma, B):
    """The C ABI reads sigma as B consecutive doubles: a strided view would hand it other rows' weights."""
    import torch
    if sigma is not None and not (sigma.is_cuda and sigma.dtype == torch.float64 and tuple(sigma.shape) == (B,)
                                  and (B <= 1 or sigma.stride(0) == 1)):
        raise ValueError(f"sigma must be a contiguous float64 CUDA tensor [{B}]")


def _np_ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def even_ld(n: int) -> int:
    """Leading dimension that keeps every row 16-byte aligned (what the TMA store path needs)."""
    return (n + 1) & ~1


_pools = {}                                           # device -> torch.cuda.MemPool over qlnlp_pool_alloc / _free


def _output_pool(device: int):
    """The caching pool the library's outputs come from on ``cuda:device``: torch's caching allocator over segments
    from ``qlnlp_pool_alloc`` (compressible where the device offers it).  Freed outputs return to the pool in stream
    order and are reused; nothing is synchronised and no driver allocation happens once the pool holds the sizes a caller
    uses.  The pools live for the process, so outputs outlive the handles that produced them."""
    import torch

    pool = _pools.get(device)
    if pool is None:
        load_library()
        alloc = torch.cuda.memory.CUDAPluggableAllocator(_lib_path, "qlnlp_pool_alloc", "qlnlp_pool_free")
        with torch.cuda.device(device):
            pool = _pools[device] = (torch.cuda.MemPool(alloc.allocator()), alloc)
    return pool[0]


def device_alloc_info(t) -> Dict[str, int]:
    """What ``qlnlp_device_alloc_info`` reports about the block holding tensor ``t`` (raises for other memory)."""
    info = (C.c_int64 * 3)()
    _check(load_library().qlnlp_device_alloc_info(C.c_void_p(t.data_ptr()), info))
    return dict(zip(("compressible", "device", "bytes"), list(info)))


def _device_empty(device: int, specs, compressible: bool = True) -> list:
    """Output tensors on ``cuda:device``.  ``specs``: ``(rows, width, dtype)``; ``width=None`` gives a 1-D tensor of
    ``rows`` entries, otherwise ``[rows, width]`` with rows padded to ``even_ld(width)`` (16-byte aligned rows).  They
    come from the compressible output pool unless ``compressible`` is false or the current stream is being captured
    into a CUDA graph (a capture keeps its allocations in its own pool, as torch.empty does)."""
    import torch

    def empty(rows, width, dtype):
        t = torch.empty(rows if width is None else (rows, even_ld(width)), dtype=dtype, device=torch.device("cuda", device))
        return t if width is None else t[:, :width]

    with torch.cuda.device(device):
        if not compressible or torch.cuda.is_current_stream_capturing():
            return [empty(*s) for s in specs]
        with torch.cuda.use_mem_pool(_output_pool(device), device):
            return [empty(*s) for s in specs]


def _check_rows(B: int, specs) -> None:
    """Each ``(tensor or None, width, name)`` is a float64 CUDA tensor ``[B, width]`` with unit inner stride."""
    import torch

    for t, wd, name in specs:
        if t is not None and not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float64
                                  and t.dim() == 2 and t.shape == (B, wd) and t.stride(1) == 1):
            raise ValueError(f"{name} must be a float64 CUDA tensor [{B}, {wd}] with unit inner stride")


def _check_status(t, B: int) -> None:
    import torch

    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.int32 and t.shape == (B,) and t.is_contiguous()):
        raise ValueError(f"out status must be a contiguous int32 CUDA tensor of shape ({B},)")


class HybridNLP:
    """GPU-backed stand-in for the reference's ``HybridNLP`` (src/nlp.jl:13-84).

    ``HybridNLP(model, obj, init_mode, k_trans, N, x0, xf; use_sparse_jacobian)`` -- same argument
    order as nlp.jl:33-36.  ``use_sparse_jacobian=False`` (the reference's default) reports the
    dense ``m_nlp x n_nlp`` column-major structure of moi.jl:31-33; ``True`` reports SPARSE_BLOCK,
    the column-major filter of the entries ``jac_c!`` assigns (the reference's own sparse branch,
    moi.jl:17-18, is not functional).  ``pattern="true"`` (with ``use_sparse_jacobian=True``) selects SPARSE_TRUE:
    only the structurally non-zero entries (identity blocks as diagonals, RK4 blocks as their mode pattern),
    4,840 values instead of 32,161 at the default instance, same column-major order.
    """

    def __init__(self, model: PlanarQuadruped, obj: Sequence[QuadraticCost], init_mode: int, k_trans: int,
                 N: int, x0, xf, integration: str = "RK4", *, use_sparse_jacobian: bool = False,
                 pattern: str = "block", device: int = 0, devices: Optional[Sequence[int]] = None,
                 hessian: bool = False, kinematics: bool = False, products: bool = False):
        if integration != "RK4":
            raise ValueError("only RK4 is implemented (as in the reference)")
        self._init(ProblemData.from_costs(model, obj, init_mode, k_trans, N, x0, xf), use_sparse_jacobian, device, pattern,
                   devices, kinematics)
        self.hessian = bool(hessian)
        self.products = bool(products)

    @classmethod
    def from_problem(cls, prob: ProblemData, *, use_sparse_jacobian: bool = True, pattern: str = "block",
                     device: int = 0, devices: Optional[Sequence[int]] = None, hessian: bool = False,
                     kinematics: bool = False, products: bool = False) -> "HybridNLP":
        """``devices=[0, 1, ...]`` builds a multi-device evaluator (``qlnlp_create_multi``): host-pointer batches are
        sharded over the listed GPUs by the library, ``eval_batch_multi`` launches one shard per device.
        ``hessian=True`` advertises ``"Hess"`` (the reference does not, src/moi.jl:26-28).  ``kinematics=True`` switches
        on the leg-length rows the reference keeps commented out (nlp.jl:60,70; constraints.jl:115-138,276-288).
        ``products=True`` advertises the matrix-free products: ``"JacVec"``, and ``"HessVec"`` with ``hessian=True``."""
        self = cls.__new__(cls)
        self._init(prob, use_sparse_jacobian, device, pattern, devices, kinematics)
        self.hessian = bool(hessian)
        self.products = bool(products)
        return self

    def _init(self, prob: ProblemData, use_sparse_jacobian: bool, device: int, pattern: str = "block",
              devices: Optional[Sequence[int]] = None, kinematics: bool = False):
        if pattern not in ("block", "true"):
            raise ValueError("pattern must be 'block' or 'true'")
        self.pattern = pattern
        L = load_library()
        self.prob = prob
        self.model = prob.model
        self.N, self.k_trans, self.init_mode = prob.N, prob.k_trans, prob.init_mode
        self.Nmodes = 2                                   # nlp.jl:45
        self.x0, self.xf = prob.x0, prob.xf
        self.modes = [prob.init_mode if k < prob.k_trans else 3 for k in range(1, prob.N + 1)]   # nlp.jl:42-44
        self.use_sparse_jacobian = bool(use_sparse_jacobian)
        self.devices = [int(x) for x in devices] if devices is not None else [int(device)]
        self.device = self.devices[0]
        d = _Desc()
        d.N, d.k_trans, d.init_mode = prob.N, prob.k_trans, prob.init_mode
        m = prob.model
        d.model = _Model(m.g, m.mb, m.mf, m.lb, m.l1, m.l2)
        for i in range(NX):
            d.x0[i] = float(prob.x0[i])
            d.xf[i] = float(prob.xf[i])
        d.Q, d.R, d.q, d.r, d.c = (a.ctypes.data for a in (prob.Q, prob.R, prob.q, prob.r, prob.c))
        self._h = C.c_void_p()
        mode = JAC_DENSE if not use_sparse_jacobian else (JAC_SPARSE_TRUE if pattern == "true" else JAC_SPARSE_BLOCK)
        self.kinematics = bool(kinematics)
        flags = mode | (WITH_KINEMATICS if kinematics else 0)
        if devices is None:
            _check(L.qlnlp_create(C.byref(d), self.device, flags, C.byref(self._h)))
        else:
            arr = (C.c_int * len(self.devices))(*self.devices)
            _check(L.qlnlp_create_multi(C.byref(d), arr, len(self.devices), flags, C.byref(self._h)))
        self._registered = {}
        self._compressible = True
        self.hessian = False
        self.products = False
        nh = C.c_int64()
        _check(L.qlnlp_hessian_nnz(self._h, C.byref(nh)))
        self.nnz_hess = nh.value
        n, mm, nnz, nnzb = (C.c_int64() for _ in range(4))
        _check(L.qlnlp_dims(self._h, C.byref(n), C.byref(mm), C.byref(nnz), C.byref(nnzb)))
        self.n_nlp, self.m_nlp, self.nnz, self.nnz_block = n.value, mm.value, nnz.value, nnzb.value
        # values per evaluation in BATCHED calls: the handle's sparse pattern (DENSE handles batch in SPARSE_BLOCK)
        self.nnz_batch = self.nnz if mode != JAC_DENSE else self.nnz_block
        # index maps, 1-based like nlp.jl:38-39,48-63
        self.xinds = [np.arange(1, NX + 1) + (k - 1) * (NX + NU) for k in range(1, self.N + 1)]
        self.uinds = [np.arange(NX + 1, NX + NU + 1) + (k - 1) * (NX + NU) for k in range(1, self.N)]
        N, kt = self.N, self.k_trans
        ends = np.cumsum([NX, NX - 1, (N - 1) * NX, N, N - kt + 1, 1, N])
        self.cinds = [range(int(e - w) + 1, int(e) + 1) for e, w in zip(ends, [NX, NX - 1, (N - 1) * NX, N, N - kt + 1, 1, N])]
        if kinematics:                                    # nlp.jl:60 (commented out upstream): cinds[8]
            self.cinds.append(range(int(ends[-1]) + 1, int(ends[-1]) + 2 * N + 1))
        self.lb, self.ub = self.constraint_bounds()
        self.zL = np.full(self.n_nlp, -np.inf)           # nlp.jl:73-74
        self.zU = np.full(self.n_nlp, np.inf)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value and _lib is not None:
            _lib.qlnlp_destroy(h)
            self._h = C.c_void_p()

    # ---- nlp.jl:85-114
    def size(self) -> Tuple[int, int, int]:
        return NX, NU, self.N

    def num_primals(self) -> int:
        return self.n_nlp

    def num_duals(self) -> int:
        return self.m_nlp

    def packZ(self, X, U) -> np.ndarray:
        return _packZ(self.N, X, U)

    def unpackZ(self, Z):
        return _unpackZ(self.N, Z)

    # ---- MOI surface, moi.jl:1-33
    def features_available(self) -> List[str]:
        feats = ["Grad", "Jac", "Hess"] if self.hessian else ["Grad", "Jac"]     # moi.jl:26-28 (+ opt-in :Hess)
        if self.products:                                                         # opt-in :JacVec / :HessVec
            feats += ["JacVec", "HessVec"] if self.hessian else ["JacVec"]
        return feats

    # ---- Lagrangian Hessian (MOI.hessian_lagrangian_structure / eval_hessian_lagrangian; not in the reference)
    def hessian_lagrangian_structure(self) -> List[Tuple[int, int]]:
        rows, cols = self.hessian_structure_arrays()
        return list(zip(rows.tolist(), cols.tolist()))

    def hessian_structure_arrays(self) -> Tuple[np.ndarray, np.ndarray]:
        rows = np.empty(self.nnz_hess, dtype=np.int64)
        cols = np.empty(self.nnz_hess, dtype=np.int64)
        _check(load_library().qlnlp_hessian_structure(self._h, _np_ptr(rows), _np_ptr(cols)))
        return rows, cols

    def eval_hessian_lagrangian(self, H: np.ndarray, x, sigma: float, mu) -> None:
        """``H[nnz_hess]`` <- sigma * Hess f(x) + sum_r mu_r Hess g_r(x) in ``hessian_lagrangian_structure`` order."""
        self._out(H, self.nnz_hess, "H")
        mu = self._x(mu, self.m_nlp)
        _check(load_library().qlnlp_eval_hessian_lagrangian(self._h, _np_ptr(self._x(x, self.n_nlp)), float(sigma),
                                                            _np_ptr(mu), _np_ptr(H)))

    def eval_hessian_batch(self, Z, mu, sigma=None, out=None, stream=None):
        """Device tensors: ``Z[B, n_nlp]``, ``mu[B, m_nlp]``, optional ``sigma[B]`` (default 1) -> ``H[B, nnz_hess]``."""
        import torch

        B = Z.shape[0]
        for t, w, name in ((Z, self.n_nlp, "Z"), (mu, self.m_nlp, "mu")):
            if not (t.is_cuda and t.dtype == torch.float64 and t.dim() == 2 and t.shape == (B, w) and t.stride(1) == 1):
                raise ValueError(f"{name} must be a float64 CUDA tensor [B, {w}]")
        _check_sigma(sigma, B)
        if out is None:
            out, = _device_empty(Z.device.index, [(B, self.nnz_hess, torch.float64)], self._compressible)
        s = torch.cuda.current_stream(Z.device) if stream is None else stream
        ld = lambda t, w: t.stride(0) if B > 1 else even_ld(w)
        _check(load_library().qlnlp_eval_hessian_batch_device(
            self._h, B, C.c_void_p(Z.data_ptr()), Z.stride(0) if B > 1 else self.n_nlp,
            None if sigma is None else C.c_void_p(sigma.data_ptr()), C.c_void_p(mu.data_ptr()),
            mu.stride(0) if B > 1 else self.m_nlp, C.c_void_p(out.data_ptr()), ld(out, self.nnz_hess), C.c_void_p(s.cuda_stream)))
        return out

    # ---- matrix-free products (MOI :JacVec / :HessVec; not in the reference).  The summation order is fixed
    # (include/qlnlp.h): each entry is the left fold of entry * vector over the structural non-zeros.
    def eval_constraint_jacobian_product(self, y: np.ndarray, x, w) -> None:
        """``y[m_nlp]`` <- J(x) w (MOI.eval_constraint_jacobian_product)."""
        self._out(y, self.m_nlp, "y")
        _check(load_library().qlnlp_eval_constraint_jacobian_product(
            self._h, _np_ptr(self._x(x, self.n_nlp)), _np_ptr(self._x(w, self.n_nlp)), _np_ptr(y)))

    def eval_constraint_jacobian_transpose_product(self, y: np.ndarray, x, w) -> None:
        """``y[n_nlp]`` <- J(x)' w (MOI.eval_constraint_jacobian_transpose_product; ``w`` has m_nlp entries)."""
        self._out(y, self.n_nlp, "y")
        _check(load_library().qlnlp_eval_constraint_jacobian_transpose_product(
            self._h, _np_ptr(self._x(x, self.n_nlp)), _np_ptr(self._x(w, self.m_nlp)), _np_ptr(y)))

    def eval_hessian_lagrangian_product(self, h: np.ndarray, x, v, sigma: float, mu) -> None:
        """``h[n_nlp]`` <- (sigma Hess f(x) + sum_r mu_r Hess g_r(x)) v (MOI.eval_hessian_lagrangian_product)."""
        self._out(h, self.n_nlp, "h")
        _check(load_library().qlnlp_eval_hessian_lagrangian_product(
            self._h, _np_ptr(self._x(x, self.n_nlp)), _np_ptr(self._x(v, self.n_nlp)), float(sigma),
            _np_ptr(self._x(mu, self.m_nlp)), _np_ptr(h)))

    def eval_products_batch(self, Z, *, w=None, y=None, want: Sequence[str] = (), x0=None, xf=None,
                            out: Optional[Dict[str, "object"]] = None, stream=None) -> Dict[str, "object"]:
        """One fused launch over ``Z[B, n_nlp]``: ``jw = J w`` (``w[B, n_nlp]``) and / or ``jty = J' y`` (``y[B, m_nlp]``),
        plus whichever of ``f``, ``grad``, ``g`` are in ``want`` (as ``eval_batch``).  Device tensors, rows padded to an
        even length; enqueued on the current torch stream and not synchronised."""
        import torch

        if w is None and y is None:
            raise ValueError("need w and / or y")
        B = Z.shape[0]
        for t, wd, name in ((Z, self.n_nlp, "Z"), (w, self.n_nlp, "w"), (y, self.m_nlp, "y")):
            if t is not None and not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float64
                                      and t.dim() == 2 and t.shape == (B, wd) and t.stride(1) == 1):
                raise ValueError(f"{name} must be a float64 CUDA tensor [B, {wd}] with unit inner stride")
        if Z.device.index != self.device:
            raise ValueError(f"Z lives on cuda:{Z.device.index}, the evaluator on cuda:{self.device}")
        out = {} if out is None else out
        dev = Z.device
        missing = [k for k in ("f", "grad", "g") if k in want and out.get(k) is None]
        missing += [k for k, v in (("jw", w), ("jty", y)) if v is not None and out.get(k) is None]
        if missing:                                     # the library's output pool, compressible where offered
            out.update(self.alloc_outputs(B, missing))

        def buf(name, width):
            t = out[name]
            if not (t.is_cuda and t.dtype == torch.float64 and t.shape == (B, width) and t.stride(1) == 1):
                raise ValueError(f"out[{name!r}] must be a float64 CUDA tensor of shape ({B}, {width})")
            return t

        ld = lambda t, width: t.stride(0) if B > 1 else width
        io = _BatchIO()
        io.Z, io.ldz = Z.data_ptr(), ld(Z, self.n_nlp)
        for name, arr in (("x0", x0), ("xf", xf)):
            if arr is not None:
                if not (arr.is_cuda and arr.dtype == torch.float64 and arr.shape == (B, NX) and arr.is_contiguous()):
                    raise ValueError(f"{name} must be a contiguous float64 CUDA tensor [B, 15]")
                setattr(io, name, arr.data_ptr())
        if "f" in want:
            io.f = out["f"].data_ptr()
        if "grad" in want:
            t = buf("grad", self.n_nlp)
            io.grad, io.ldgrad = t.data_ptr(), ld(t, even_ld(self.n_nlp))
        if "g" in want:
            t = buf("g", self.m_nlp)
            io.g, io.ldg = t.data_ptr(), ld(t, even_ld(self.m_nlp))
        pv = _ProductIO()
        if w is not None:
            t = buf("jw", self.m_nlp)
            pv.w, pv.ldw, pv.jw, pv.ldjw = w.data_ptr(), ld(w, self.n_nlp), t.data_ptr(), ld(t, even_ld(self.m_nlp))
        if y is not None:
            t = buf("jty", self.n_nlp)
            pv.y, pv.ldy, pv.jty, pv.ldjty = y.data_ptr(), ld(y, self.m_nlp), t.data_ptr(), ld(t, even_ld(self.n_nlp))
        s = torch.cuda.current_stream(dev) if stream is None else stream
        _check(load_library().qlnlp_eval_jacobian_products_batch_device(self._h, B, C.byref(io), C.byref(pv),
                                                                        C.c_void_p(s.cuda_stream)))
        return out

    def eval_hessian_product_batch(self, Z, mu, V, sigma=None, out=None, stream=None):
        """Device tensors: ``Z[B, n_nlp]``, ``mu[B, m_nlp]``, ``V[B, n_nlp]``, optional ``sigma[B]`` (default 1) ->
        ``HV[B, n_nlp]`` (rows padded to an even length)."""
        import torch

        B = Z.shape[0]
        for t, wd, name in ((Z, self.n_nlp, "Z"), (mu, self.m_nlp, "mu"), (V, self.n_nlp, "V")):
            if not (t.is_cuda and t.dtype == torch.float64 and t.dim() == 2 and t.shape == (B, wd) and t.stride(1) == 1):
                raise ValueError(f"{name} must be a float64 CUDA tensor [B, {wd}]")
        _check_sigma(sigma, B)
        if out is None:
            out, = _device_empty(Z.device.index, [(B, self.n_nlp, torch.float64)], self._compressible)
        s = torch.cuda.current_stream(Z.device) if stream is None else stream
        ld = lambda t, wd: t.stride(0) if B > 1 else wd
        _check(load_library().qlnlp_eval_hessian_product_batch_device(
            self._h, B, C.c_void_p(Z.data_ptr()), ld(Z, self.n_nlp), None if sigma is None else C.c_void_p(sigma.data_ptr()),
            C.c_void_p(mu.data_ptr()), ld(mu, self.m_nlp), C.c_void_p(V.data_ptr()), ld(V, self.n_nlp),
            C.c_void_p(out.data_ptr()), ld(out, even_ld(self.n_nlp)), C.c_void_p(s.cuda_stream)))
        return out

    # ---- batched Newton step (not in the reference): the regularised KKT system of each problem, include/qlnlp.h
    def kkt_solve_batch(self, hess, jac, dc, r1, r2, sx=None, out=None, stream=None):
        """Device tensors, one row per problem: ``hess[B, nnz_hess]`` (``eval_hessian_batch``), ``jac[B, nnz]``
        (SPARSE_TRUE values, ``eval_batch``), ``dc[B, m_nlp] > 0``, ``r1[B, n_nlp]``, ``r2[B, m_nlp]``, optional
        ``sx[B, n_nlp] >= 0`` (default 0) -> ``(px[B, n_nlp], pl[B, m_nlp], status[B] int32)``.  ``out`` may give the
        three outputs.  Enqueued on the current torch stream (or ``stream``), not synchronised."""
        import torch

        B = hess.shape[0]
        n, m = self.n_nlp, self.m_nlp
        for t, wd, name in ((hess, self.nnz_hess, "hess"), (jac, self.nnz, "jac"), (dc, m, "dc"), (r1, n, "r1"),
                            (r2, m, "r2"), (sx, n, "sx")):
            if t is not None and not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float64
                                      and t.dim() == 2 and t.shape == (B, wd) and t.stride(1) == 1):
                raise ValueError(f"{name} must be a float64 CUDA tensor [B, {wd}] with unit inner stride")
        dev = hess.device
        if out is None:
            out = tuple(_device_empty(dev.index, [(B, n, torch.float64), (B, m, torch.float64), (B, None, torch.int32)],
                                     self._compressible))
        px, pl, status = out
        for t, wd, name in ((px, n, "px"), (pl, m, "pl")):
            if not (t.is_cuda and t.dtype == torch.float64 and t.shape == (B, wd) and t.stride(1) == 1):
                raise ValueError(f"out {name} must be a float64 CUDA tensor of shape ({B}, {wd})")
        if not (status.is_cuda and status.dtype == torch.int32 and status.shape == (B,) and status.is_contiguous()):
            raise ValueError(f"out status must be a contiguous int32 CUDA tensor of shape ({B},)")
        ld = lambda t, wd: t.stride(0) if B > 1 else wd
        io = _KktIO()
        io.hess, io.ldhess = hess.data_ptr(), ld(hess, self.nnz_hess)
        io.jac, io.ldjac = jac.data_ptr(), ld(jac, self.nnz)
        if sx is not None:
            io.sx, io.ldsx = sx.data_ptr(), ld(sx, n)
        io.dc, io.lddc = dc.data_ptr(), ld(dc, m)
        io.r1, io.ldr1 = r1.data_ptr(), ld(r1, n)
        io.r2, io.ldr2 = r2.data_ptr(), ld(r2, m)
        io.px, io.ldpx = px.data_ptr(), ld(px, n)
        io.pl, io.ldpl = pl.data_ptr(), ld(pl, m)
        io.status = status.data_ptr()
        s = torch.cuda.current_stream(dev) if stream is None else stream
        _check(load_library().qlnlp_kkt_solve_batch_device(self._h, B, C.byref(io), C.c_void_p(s.cuda_stream)))
        return px, pl, status

    # The same solve split in two: factorise once, solve many right-hand sides (include/qlnlp.h).  A factor followed by
    # a factored solve gives the bits of kkt_solve_batch.
    @property
    def kkt_factor_size(self) -> int:
        """Doubles in one problem's factor row (``qlnlp_kkt_factor_size``)."""
        v = C.c_int64()
        _check(load_library().qlnlp_kkt_factor_size(self._h, C.byref(v)))
        return v.value

    def kkt_factor_batch(self, hess, jac, dc, sx=None, out=None, stream=None):
        """Device tensors as ``kkt_solve_batch`` -> ``(factor[B, kkt_factor_size], status[B] int32)``.  The factor holds
        everything a later solve reads: overwriting the inputs afterwards changes no solve.  ``out`` may give both
        outputs.  Enqueued on the current torch stream (or ``stream``), not synchronised."""
        import torch

        B = hess.shape[0]
        size = self.kkt_factor_size
        _check_rows(B, ((hess, self.nnz_hess, "hess"), (jac, self.nnz, "jac"), (dc, self.m_nlp, "dc"),
                        (sx, self.n_nlp, "sx")))
        dev = hess.device
        if out is None:
            out = tuple(_device_empty(dev.index, [(B, size, torch.float64), (B, None, torch.int32)], self._compressible))
        factor, status = out
        _check_rows(B, ((factor, size, "out factor"),))
        _check_status(status, B)
        ld = lambda t, wd: t.stride(0) if B > 1 else wd
        io = _KktFactorIO()
        io.hess, io.ldhess = hess.data_ptr(), ld(hess, self.nnz_hess)
        io.jac, io.ldjac = jac.data_ptr(), ld(jac, self.nnz)
        if sx is not None:
            io.sx, io.ldsx = sx.data_ptr(), ld(sx, self.n_nlp)
        io.dc, io.lddc = dc.data_ptr(), ld(dc, self.m_nlp)
        io.factor, io.ldfactor = factor.data_ptr(), ld(factor, size)
        io.status = status.data_ptr()
        s = torch.cuda.current_stream(dev) if stream is None else stream
        _check(load_library().qlnlp_kkt_factor_batch_device(self._h, B, C.byref(io), C.c_void_p(s.cuda_stream)))
        return factor, status

    def kkt_solve_factored_batch(self, factor, r1, r2, index=None, out=None, stream=None):
        """``factor[F, kkt_factor_size]`` (``kkt_factor_batch``), ``r1[R, n_nlp]``, ``r2[R, m_nlp]``, optional
        ``index[R]`` int64 (the factor row of each right-hand side; default: row i uses factor i) -> ``(px[R, n_nlp],
        pl[R, m_nlp], status[R] int32)``.  status: 0, the factor's own non-zero status, -2 for an index outside
        ``[0, F)``, -3 for a factor of another class.  Enqueued on the current torch stream (or ``stream``)."""
        import torch

        R, F = r1.shape[0], factor.shape[0]
        n, m, size = self.n_nlp, self.m_nlp, self.kkt_factor_size
        _check_rows(F, ((factor, size, "factor"),))
        _check_rows(R, ((r1, n, "r1"), (r2, m, "r2")))
        if index is not None and not (isinstance(index, torch.Tensor) and index.is_cuda and index.dtype == torch.int64
                                      and index.shape == (R,) and index.is_contiguous()):
            raise ValueError(f"index must be a contiguous int64 CUDA tensor of shape ({R},)")
        dev = r1.device
        if out is None:
            out = tuple(_device_empty(dev.index, [(R, n, torch.float64), (R, m, torch.float64), (R, None, torch.int32)],
                                      self._compressible))
        px, pl, status = out
        _check_rows(R, ((px, n, "out px"), (pl, m, "out pl")))
        _check_status(status, R)
        io = _KktRhsIO()
        io.factor, io.ldfactor, io.nfactor = factor.data_ptr(), factor.stride(0) if F > 1 else size, F
        if index is not None:
            io.index = index.data_ptr()
        ld = lambda t, wd: t.stride(0) if R > 1 else wd
        io.r1, io.ldr1 = r1.data_ptr(), ld(r1, n)
        io.r2, io.ldr2 = r2.data_ptr(), ld(r2, m)
        io.px, io.ldpx = px.data_ptr(), ld(px, n)
        io.pl, io.ldpl = pl.data_ptr(), ld(pl, m)
        io.status = status.data_ptr()
        s = torch.cuda.current_stream(dev) if stream is None else stream
        _check(load_library().qlnlp_kkt_solve_factored_batch_device(self._h, R, C.byref(io), C.c_void_p(s.cuda_stream)))
        return px, pl, status

    def kkt_residual_batch(self, hess, jac, dc, px, pl, r1, r2, sx=None, out=None, stream=None):
        """Device tensors as ``kkt_solve_batch``, with a step ``px[B, n_nlp]``, ``pl[B, m_nlp]`` -> ``(s1[B, n_nlp],
        s2[B, m_nlp])``, the residual ``s1 = r1 - (W + diag(sx)) px - J' pl``, ``s2 = r2 - J px + dc * pl`` in the fixed
        summation order of include/qlnlp.h.  ``out`` may give both outputs.  Enqueued on the current torch stream (or
        ``stream``), not synchronised."""
        import torch

        B = hess.shape[0]
        n, m = self.n_nlp, self.m_nlp
        _check_rows(B, ((hess, self.nnz_hess, "hess"), (jac, self.nnz, "jac"), (dc, m, "dc"), (px, n, "px"),
                        (pl, m, "pl"), (r1, n, "r1"), (r2, m, "r2"), (sx, n, "sx")))
        dev = hess.device
        if out is None:
            out = tuple(_device_empty(dev.index, [(B, n, torch.float64), (B, m, torch.float64)], self._compressible))
        s1, s2 = out
        _check_rows(B, ((s1, n, "out s1"), (s2, m, "out s2")))
        ld = lambda t, wd: t.stride(0) if B > 1 else wd
        io = _KktResidualIO()
        io.hess, io.ldhess = hess.data_ptr(), ld(hess, self.nnz_hess)
        io.jac, io.ldjac = jac.data_ptr(), ld(jac, self.nnz)
        if sx is not None:
            io.sx, io.ldsx = sx.data_ptr(), ld(sx, n)
        io.dc, io.lddc = dc.data_ptr(), ld(dc, m)
        io.r1, io.ldr1 = r1.data_ptr(), ld(r1, n)
        io.r2, io.ldr2 = r2.data_ptr(), ld(r2, m)
        io.px, io.ldpx = px.data_ptr(), ld(px, n)
        io.pl, io.ldpl = pl.data_ptr(), ld(pl, m)
        io.s1, io.lds1 = s1.data_ptr(), ld(s1, n)
        io.s2, io.lds2 = s2.data_ptr(), ld(s2, m)
        s = torch.cuda.current_stream(dev) if stream is None else stream
        _check(load_library().qlnlp_kkt_residual_batch_device(self._h, B, C.byref(io), C.c_void_p(s.cuda_stream)))
        return s1, s2

    def kkt_solve_refined_batch(self, hess, jac, dc, r1, r2, sx=None, steps=3, out=None, stream=None):
        """The step of ``kkt_solve_batch`` followed by ``steps`` rounds of iterative refinement against the kept factor:
        factored solve of the residual of K (``kkt_residual_batch``), ``px + dpx``, ``pl + dpl``.  The condensed solve
        loses digits of px when dc is small (include/qlnlp.h, "Accuracy"); refinement restores them where the factor is
        close enough to K.  Where it is not, refinement can diverge, so each row keeps its new iterate only when that
        iterate's componentwise backward error max_i |r - K z|_i / (|r| + |K| |z|)_i is at most half the kept one's (a
        rejected row then repeats the same step; near convergence only steps at rounding level are refused): the
        result's is never larger than the unrefined step's.  The
        denominator comes from the residual kernel on absolute values, one more launch per step, and takes copies of
        |hess| and |jac| for the call.  With ``steps = 0`` the result has the bits
        of ``kkt_solve_batch``.  Same arguments and outputs as ``kkt_solve_batch``; status is the factor's, and rows with
        a non-zero status stay NaN.  Everything is enqueued on the current torch stream (or ``stream``) with no host
        synchronisation, so the chain can be captured in a graph."""
        import torch

        if steps < 0:
            raise ValueError("steps must be >= 0")
        B = hess.shape[0]
        n, m = self.n_nlp, self.m_nlp
        dev = hess.device
        s = torch.cuda.current_stream(dev) if stream is None else stream
        with torch.cuda.stream(s):
            factor, _ = self.kkt_factor_batch(hess, jac, dc, sx=sx, stream=s)
            px, pl, status = self.kkt_solve_factored_batch(factor, r1, r2, out=out, stream=s)
            if steps:
                s1, s2, dpx, dpl, qx, ql, t1, t2, a1, a2 = (torch.empty((B, w), dtype=torch.float64, device=dev)
                                                            for w in (n, m, n, m, n, m, n, m, n, m))
                dst = torch.empty((B,), dtype=torch.int32, device=dev)
                # |r| + |K| |z| by the same kernel: with |W|, |J|, -dc, -|px|, -|pl|, |r1|, |r2| every term of its fold
                # is non-negative (the diagonal is RN(|W_ii| + sx_i) >= |W_ii + sx_i|)
                ah, aj, ndc, ar1, ar2 = hess.abs(), jac.abs(), -dc, r1.abs(), r2.abs()

                def omega(x, y, u, v):
                    """componentwise backward error max_i |s_i| / (|r| + |K| |z|)_i of z = [x; y] with residual [u; v]"""
                    self.kkt_residual_batch(ah, aj, ndc, -x.abs(), -y.abs(), ar1, ar2, sx=sx, out=(a1, a2), stream=s)
                    return torch.maximum((u.abs() / a1.clamp_min(1e-300)).amax(dim=1),
                                         (v.abs() / a2.clamp_min(1e-300)).amax(dim=1))

                self.kkt_residual_batch(hess, jac, dc, px, pl, r1, r2, sx=sx, out=(s1, s2), stream=s)
                kept = omega(px, pl, s1, s2)
                for _ in range(steps):
                    self.kkt_solve_factored_batch(factor, s1, s2, out=(dpx, dpl, dst), stream=s)
                    torch.add(px, dpx, out=qx)
                    torch.add(pl, dpl, out=ql)
                    self.kkt_residual_batch(hess, jac, dc, qx, ql, r1, r2, sx=sx, out=(t1, t2), stream=s)
                    new = omega(qx, ql, t1, t2)
                    take = new < 0.5 * kept             # False for NaN rows: a failed factor's rows stay NaN
                    for old, cand in ((px, qx), (pl, ql), (s1, t1), (s2, t2)):
                        old.copy_(torch.where(take[:, None], cand, old))
                    kept = torch.where(take, new, kept)
        return px, pl, status

    def initialize(self, features: Iterable[str] = ()) -> None:
        return None                                       # moi.jl:30

    def jacobian_structure(self) -> List[Tuple[int, int]]:
        rows, cols = self.jacobian_structure_arrays()
        return list(zip(rows.tolist(), cols.tolist()))

    def jacobian_structure_arrays(self) -> Tuple[np.ndarray, np.ndarray]:
        rows = np.empty(self.nnz, dtype=np.int64)
        cols = np.empty(self.nnz, dtype=np.int64)
        _check(load_library().qlnlp_jacobian_structure(self._h, _np_ptr(rows), _np_ptr(cols)))
        return rows, cols

    def constraint_bounds(self) -> Tuple[np.ndarray, np.ndarray]:
        lb, ub = np.empty(self.m_nlp), np.empty(self.m_nlp)
        _check(load_library().qlnlp_constraint_bounds(self._h, _np_ptr(lb), _np_ptr(ub)))
        return lb, ub

    def variable_bounds(self) -> Tuple[np.ndarray, np.ndarray]:
        xl, xu = np.empty(self.n_nlp), np.empty(self.n_nlp)
        _check(load_library().qlnlp_variable_bounds(self._h, _np_ptr(xl), _np_ptr(xu)))
        return xl, xu

    @staticmethod
    def _x(x, n) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.float64)
        if x.shape != (n,):
            raise ValueError(f"x must have {n} entries")
        return x

    @staticmethod
    def _out(a, n, name) -> np.ndarray:
        if not (isinstance(a, np.ndarray) and a.dtype == np.float64 and a.flags.c_contiguous and a.size == n):
            raise ValueError(f"{name} must be a contiguous float64 array with {n} entries (written in place)")
        return a

    def eval_objective(self, x) -> float:
        f = np.empty(1)
        _check(load_library().qlnlp_eval_objective(self._h, _np_ptr(self._x(x, self.n_nlp)), _np_ptr(f)))
        return float(f[0])

    def eval_objective_gradient(self, grad_f: np.ndarray, x) -> None:
        self._out(grad_f, self.n_nlp, "grad_f")
        _check(load_library().qlnlp_eval_objective_gradient(self._h, _np_ptr(self._x(x, self.n_nlp)), _np_ptr(grad_f)))

    def eval_constraint(self, g: np.ndarray, x) -> None:
        self._out(g, self.m_nlp, "g")
        _check(load_library().qlnlp_eval_constraint(self._h, _np_ptr(self._x(x, self.n_nlp)), _np_ptr(g)))

    def eval_constraint_jacobian(self, vec: np.ndarray, x) -> None:
        self._out(vec, self.nnz, "vec")
        _check(load_library().qlnlp_eval_constraint_jacobian(self._h, _np_ptr(self._x(x, self.n_nlp)), _np_ptr(vec)))

    def eval_all(self, x, f: Optional[np.ndarray] = None, grad_f: Optional[np.ndarray] = None,
                 g: Optional[np.ndarray] = None, vec: Optional[np.ndarray] = None) -> None:
        """All four callbacks of one iterate with one launch (``qlnlp_eval_all``); any output may be omitted.
        ``f`` is a 1-element array."""
        if f is not None:
            self._out(f, 1, "f")
        if grad_f is not None:
            self._out(grad_f, self.n_nlp, "grad_f")
        if g is not None:
            self._out(g, self.m_nlp, "g")
        if vec is not None:
            self._out(vec, self.nnz, "vec")
        _check(load_library().qlnlp_eval_all(self._h, _np_ptr(self._x(x, self.n_nlp)), _np_ptr(f), _np_ptr(grad_f),
                                             _np_ptr(g), _np_ptr(vec)))

    def set_option(self, name: str, value: int) -> None:
        _check(load_library().qlnlp_set_option(self._h, name.encode(), int(value)))
        if name == "compressible":                      # the outputs this object allocates follow the handle's option
            self._compressible = bool(value)

    # ---- host-pointer path helpers
    def register_host_output(self, jac: np.ndarray) -> None:
        """``qlnlp_host_output_register``: write the constant image of the pattern into ``jac[B, nnz_batch]`` once;
        later ``eval_batch_host(..., out={"jac": jac or a row-slice of it})`` rewrites only the lines that change."""
        if not (isinstance(jac, np.ndarray) and jac.dtype == np.float64 and jac.ndim == 2 and jac.flags.c_contiguous
                and jac.shape[1] == self.nnz_batch):
            raise ValueError(f"jac must be a contiguous float64 array [B, {self.nnz_batch}]")
        _check(load_library().qlnlp_host_output_register(self._h, jac.ctypes.data, jac.shape[1], jac.shape[0]))
        self._registered[jac.ctypes.data] = jac          # keep it alive while it is registered

    def unregister_host_output(self, jac: np.ndarray) -> None:
        _check(load_library().qlnlp_host_output_unregister(self._h, jac.ctypes.data))
        self._registered.pop(jac.ctypes.data, None)

    def host_path_info(self) -> Dict[str, int]:
        info = (C.c_int64 * 8)()
        _check(load_library().qlnlp_host_path_info(self._h, info))
        return dict(zip(("threads_per_device", "pcie_jac_doubles_per_eval", "row_doubles", "touched_lines_per_row",
                         "lines_per_row", "avx512", "rows_built", "lines_written"), list(info)))

    # ---- batched evaluation
    def alloc_outputs(self, B: int, want: Sequence[str] = ("f", "grad", "g", "jac"), device: Optional[int] = None
                      ) -> Dict[str, "object"]:
        """The output arrays ``eval_batch`` (and ``eval_products_batch``: ``jw``, ``jty``) would allocate for a batch of
        ``B`` on ``cuda:device`` (default: the evaluator's device, which is the only one a single-device evaluator
        accepts), from the library's caching output pool: compressible where the device offers it, which cuts the DRAM
        traffic of the zero-rich Jacobian rows.  Rows are padded to an even length (16-byte aligned).  Pass the dict as
        ``out=`` to reuse it."""
        import torch

        widths = {"f": None, "grad": self.n_nlp, "g": self.m_nlp, "jac": self.nnz_batch, "jw": self.m_nlp,
                  "jty": self.n_nlp}
        names = [k for k in widths if k in want]
        if any(k not in widths for k in want):
            raise ValueError(f"want may name {sorted(widths)}, got {list(want)}")
        dev = self.device if device is None else int(device)
        if dev not in self.devices:
            raise ValueError(f"device {dev} is not one of the evaluator's devices {self.devices}")
        ts = _device_empty(dev, [(int(B), widths[k], torch.float64) for k in names], self._compressible)
        return dict(zip(names, ts))

    def eval_batch(self, Z, *, x0=None, xf=None, want: Sequence[str] = ("f", "grad", "g", "jac"),
                   out: Optional[Dict[str, "object"]] = None, stream=None) -> Dict[str, "object"]:
        """Evaluate ``B`` decision vectors held in a CUDA tensor ``Z[B, ldz>=n_nlp]`` (fp64, row-major).

        Returns device tensors ``f[B]``, ``grad[B, n_nlp]``, ``g[B, m_nlp]``, ``jac[B, nnz_batch]`` (views of
        buffers whose rows are padded to an even length so every row is 16-byte aligned).  The launch is
        enqueued on the current torch stream and NOT synchronised.
        """
        import torch

        if not (isinstance(Z, torch.Tensor) and Z.is_cuda and Z.dtype == torch.float64 and Z.dim() == 2):
            raise ValueError("Z must be a 2-D float64 CUDA tensor")
        if Z.stride(1) != 1 or Z.shape[1] != self.n_nlp:
            raise ValueError(f"Z must be [B, {self.n_nlp}] with unit inner stride")
        if Z.device.index != self.device:
            raise ValueError(f"Z lives on cuda:{Z.device.index}, the evaluator on cuda:{self.device}")
        B = Z.shape[0]
        out = {} if out is None else out
        dev = Z.device
        missing = [k for k in ("f", "grad", "g", "jac") if k in want and out.get(k) is None]
        if missing:                                     # the library's output pool, compressible where offered
            out.update(self.alloc_outputs(B, missing))

        def buf(name, width):
            t = out[name]
            if not (t.is_cuda and t.dtype == torch.float64 and t.shape == (B, width) and t.stride(1) == 1):
                raise ValueError(f"out[{name!r}] must be a float64 CUDA tensor of shape ({B}, {width})")
            return t

        io = _BatchIO()
        io.Z, io.ldz = Z.data_ptr(), Z.stride(0) if B > 1 else self.n_nlp
        for name, arr in (("x0", x0), ("xf", xf)):
            if arr is not None:
                if not (arr.is_cuda and arr.dtype == torch.float64 and arr.shape == (B, NX) and arr.is_contiguous()):
                    raise ValueError(f"{name} must be a contiguous float64 CUDA tensor [B, 15]")
                setattr(io, name, arr.data_ptr())
        if "f" in want:
            io.f = out["f"].data_ptr()
        if "grad" in want:
            t = buf("grad", self.n_nlp)
            io.grad, io.ldgrad = t.data_ptr(), t.stride(0) if B > 1 else self.n_nlp
        if "g" in want:
            t = buf("g", self.m_nlp)
            io.g, io.ldg = t.data_ptr(), t.stride(0) if B > 1 else self.m_nlp
        if "jac" in want:
            t = buf("jac", self.nnz_batch)
            io.jac, io.ldjac = t.data_ptr(), t.stride(0) if B > 1 else even_ld(self.nnz_batch)
        s = torch.cuda.current_stream(dev) if stream is None else stream
        _check(load_library().qlnlp_eval_batch_device(self._h, B, C.byref(io), C.c_void_p(s.cuda_stream)))
        return out

    def eval_batch_multi(self, Zs: Sequence["object"], *, want: Sequence[str] = ("f", "grad", "g", "jac"),
                         outs: Optional[List[Dict[str, "object"]]] = None) -> List[Dict[str, "object"]]:
        """One shard per device of a multi-device evaluator: ``Zs[i]`` is a float64 CUDA tensor ``[B_i, n_nlp]`` on
        ``cuda:devices[i]``.  One ``qlnlp_eval_batch_device_multi`` call enqueues a fused launch on every device's
        current torch stream; nothing is synchronised (``synchronize()`` waits for all devices)."""
        import torch

        nd = len(self.devices)
        if len(Zs) != nd:
            raise ValueError(f"need one Z per device ({nd})")
        outs = [{} for _ in range(nd)] if outs is None else outs
        ios = (_BatchIO * nd)()
        Bs = (C.c_int64 * nd)()
        streams = (C.c_void_p * nd)()
        for i, (Z, out) in enumerate(zip(Zs, outs)):
            if not (Z.is_cuda and Z.dtype == torch.float64 and Z.dim() == 2 and Z.shape[1] == self.n_nlp and Z.stride(1) == 1):
                raise ValueError(f"Zs[{i}] must be a float64 CUDA tensor [B, {self.n_nlp}]")
            if Z.device.index != self.devices[i]:
                raise ValueError(f"Zs[{i}] lives on cuda:{Z.device.index}, shard {i} runs on cuda:{self.devices[i]}")
            B = Z.shape[0]
            Bs[i] = B
            io = ios[i]
            io.Z, io.ldz = Z.data_ptr(), Z.stride(0) if B > 1 else self.n_nlp
            widths = {"grad": self.n_nlp, "g": self.m_nlp, "jac": self.nnz_batch}
            missing = [k for k in ("f", "grad", "g", "jac") if k in want and out.get(k) is None]
            if missing:
                out.update(self.alloc_outputs(B, missing, device=Z.device.index))
            if "f" in want:
                io.f = out["f"].data_ptr()
            for name, w in widths.items():
                if name not in want:
                    continue
                t = out[name]
                setattr(io, name, t.data_ptr())
                setattr(io, "ld" + name, t.stride(0) if B > 1 else even_ld(w))
            streams[i] = torch.cuda.current_stream(Z.device).cuda_stream
        _check(load_library().qlnlp_eval_batch_device_multi(self._h, Bs, ios, streams))
        return outs

    def synchronize(self) -> None:
        _check(load_library().qlnlp_synchronize(self._h))

    def initial_guess_batch(self, x0, dt: float = 0.009, out=None, stream=None):
        """Cell-7 guesses (src/main.ipynb:181-196) for a sweep, built by a CUDA kernel: ``x0`` is a float64 CUDA tensor
        ``[B, 15]`` of initial states; returns ``Z[B, n_nlp]`` (rows padded to an even length).  Same values, bit for bit,
        as ``problem.initial_guess_batch`` on the host."""
        import torch
        from .problem import initial_guess

        if not (x0.is_cuda and x0.dtype == torch.float64 and x0.dim() == 2 and x0.shape[1] == NX and x0.is_contiguous()):
            raise ValueError("x0 must be a contiguous float64 CUDA tensor [B, 15]")
        B = x0.shape[0]
        key = ("guess_base", float(dt), x0.device.index)
        base = self._registered.get(key)
        if base is None:
            base = torch.from_numpy(initial_guess(self.prob, dt)).to(x0.device)
            self._registered[key] = base
        if out is None:
            out, = _device_empty(x0.device.index, [(B, self.n_nlp, torch.float64)], self._compressible)
        s = torch.cuda.current_stream(x0.device) if stream is None else stream
        _check(load_library().qlnlp_initial_guess_batch_device(self._h, B, C.c_void_p(base.data_ptr()), C.c_void_p(x0.data_ptr()),
                                                               C.c_void_p(out.data_ptr()), out.stride(0) if B > 1 else even_ld(self.n_nlp),
                                                               C.c_void_p(s.cuda_stream)))
        return out

    def eval_ragged(self, index, flat: Dict[str, "object"], offsets: Dict[str, "object"], *, x0=None, xf=None,
                    stream=None, z_padded: bool = False) -> None:
        """Evaluate the problems ``index`` (int64 CUDA tensor of problem numbers) of a flat, mixed-size batch.

        ``flat`` holds the flat float64 CUDA tensors ``Z`` and any of ``f`` (indexed by problem number), ``grad``,
        ``g``, ``jac``; ``offsets`` the int64 CUDA tensors ``z_off``, ``g_off``, ``j_off`` (start of every problem's
        rows, in doubles).  Outputs are written in place; nothing is copied or gathered.  Not synchronised."""
        import torch

        B = int(index.shape[0])
        io = _BatchIO()
        io.Z = flat["Z"].data_ptr()
        for name in ("f", "grad", "g", "jac"):
            if flat.get(name) is not None:
                setattr(io, name, flat[name].data_ptr())
        if x0 is not None:
            io.x0 = x0.data_ptr()
        if xf is not None:
            io.xf = xf.data_ptr()
        rg = _RaggedIO(index.data_ptr(), offsets["z_off"].data_ptr(),
                       offsets["g_off"].data_ptr() if flat.get("g") is not None else None,
                       offsets["j_off"].data_ptr() if flat.get("jac") is not None else None,
                       1 if z_padded else 0)
        dev = flat["Z"].device
        s = torch.cuda.current_stream(dev) if stream is None else stream
        _check(load_library().qlnlp_eval_ragged_device(self._h, B, C.byref(io), C.byref(rg), C.c_void_p(s.cuda_stream)))

    @staticmethod
    def eval_ragged_classes(nlps: Sequence["HybridNLP"], index, class_of, flat: Dict[str, "object"],
                            offsets: Dict[str, "object"], *, x0=None, xf=None, stream=None, z_padded: bool = False) -> None:
        """The whole mixed batch in ONE launch (``qlnlp_eval_ragged_classes``): problem ``i`` belongs to
        ``nlps[class_of[i]]`` (``class_of``: int32 CUDA tensor over all problems); the launch evaluates the problems
        ``index`` (int64 CUDA tensor; order it by class).  Other arguments as in ``eval_ragged``."""
        import torch

        B = int(index.shape[0])
        io = _BatchIO()
        io.Z = flat["Z"].data_ptr()
        for name in ("f", "grad", "g", "jac"):
            if flat.get(name) is not None:
                setattr(io, name, flat[name].data_ptr())
        if x0 is not None:
            io.x0 = x0.data_ptr()
        if xf is not None:
            io.xf = xf.data_ptr()
        rg = _RaggedIO(index.data_ptr(), offsets["z_off"].data_ptr(),
                       offsets["g_off"].data_ptr() if flat.get("g") is not None else None,
                       offsets["j_off"].data_ptr() if flat.get("jac") is not None else None,
                       1 if z_padded else 0)
        hs = (C.c_void_p * len(nlps))(*[n._h.value for n in nlps])
        dev = flat["Z"].device
        s = torch.cuda.current_stream(dev) if stream is None else stream
        if class_of.dtype != torch.int32:
            raise ValueError("class_of must be an int32 CUDA tensor")
        _check(load_library().qlnlp_eval_ragged_classes(hs, len(nlps), B, C.byref(io), C.byref(rg),
                                                        C.c_void_p(class_of.data_ptr()), C.c_void_p(s.cuda_stream)))

    def eval_batch_host(self, Z: np.ndarray, *, x0: Optional[np.ndarray] = None, xf: Optional[np.ndarray] = None,
                        want: Sequence[str] = ("f", "grad", "g", "jac"),
                        out: Optional[Dict[str, np.ndarray]] = None) -> Dict[str, np.ndarray]:
        """Same evaluation on HOST arrays: H2D copy of Z, one fused launch per chunk, D2H copy of the outputs.

        ``Z`` is ``[B, n_nlp]`` float64 (numpy; pinned memory makes the copies asynchronous).  Returns
        numpy arrays; pass ``out`` to reuse (pinned) buffers.
        """
        Z = np.ascontiguousarray(Z, dtype=np.float64)
        if Z.ndim != 2 or Z.shape[1] != self.n_nlp:
            raise ValueError(f"Z must be [B, {self.n_nlp}]")
        B = Z.shape[0]
        out = {} if out is None else out
        io = _BatchIO()
        io.Z, io.ldz = Z.ctypes.data, self.n_nlp
        keep = [Z]
        for name, arr in (("x0", x0), ("xf", xf)):
            if arr is not None:
                arr = np.ascontiguousarray(arr, dtype=np.float64)
                if arr.shape != (B, NX):
                    raise ValueError(f"{name} must be [B, 15]")
                keep.append(arr)
                setattr(io, name, arr.ctypes.data)
        widths = {"f": None, "grad": self.n_nlp, "g": self.m_nlp, "jac": self.nnz_batch}
        for name in want:
            w = widths[name]
            shape = (B,) if w is None else (B, w)
            a = out.get(name)
            if a is None:
                a = np.empty(shape)
                out[name] = a
            if not (a.dtype == np.float64 and a.shape == shape and a.flags.c_contiguous):
                raise ValueError(f"out[{name!r}] must be contiguous float64 of shape {shape}")
            setattr(io, name, a.ctypes.data)
            if w is not None:
                setattr(io, "ld" + name, w)
        _check(load_library().qlnlp_eval_batch_host(self._h, B, C.byref(io)))
        return out

    def launch_info(self) -> Dict[str, int]:
        info = (C.c_int64 * 5)()
        _check(load_library().qlnlp_launch_info(self._h, info))
        return dict(zip(("blocks", "threads_per_block", "smem_bytes", "blocks_per_sm", "sm_count"), list(info)))

    def _debug_host_times(self) -> Dict[str, float]:
        t = (C.c_double * 4)()
        _check(load_library().qlnlp_debug_host_times(self._h, t))
        return dict(zip(("total", "enqueue", "wait", "build"), list(t)))

    def _debug_vals_map(self) -> np.ndarray:
        n = C.c_int64()
        L = load_library()
        _check(L.qlnlp_debug_vals_map(self._h, None, 0, C.byref(n)))
        pos = np.empty(n.value, dtype=np.int32)
        _check(L.qlnlp_debug_vals_map(self._h, _np_ptr(pos), n.value, C.byref(n)))
        return pos

    def _debug_build_rows(self, vals: np.ndarray, jac: np.ndarray, touched_only: bool, threads: int = 1) -> None:
        """The host row builder alone (CPU tests): rows of the batch pattern from VALS rows."""
        assert vals.flags.c_contiguous and jac.dtype == np.float64 and jac.strides[-1] == 8
        _check(load_library().qlnlp_debug_build_rows(self._h, _np_ptr(vals), vals.shape[1], jac.ctypes.data,
                                                     jac.strides[0] // 8, jac.shape[0], int(touched_only), threads))

    def _debug_segments(self) -> np.ndarray:
        n = C.c_int64()
        L = load_library()
        _check(L.qlnlp_debug_segments(self._h, None, 0, C.byref(n)))
        segs = np.empty((n.value, 6), dtype=np.int64)
        _check(L.qlnlp_debug_segments(self._h, _np_ptr(segs), n.value, C.byref(n)))
        return segs
