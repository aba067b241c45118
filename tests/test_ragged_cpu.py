"""Ragged launches without a device: the refusals that run before a device is bound, and the flat-layout builder the
GPU tests (tests/test_gpu_ragged.py) lay their batches out with, checked here so that a mistake in the test itself
costs no GPU time."""
import ctypes as C

import numpy as np
import pytest

import quadruped_landing_b200 as ql
from quadruped_landing_b200 import evaluator as ev

# Fills every output double the launch must not write: a signalling-NaN payload that no evaluation produces
SENTINEL = 0x7FF4_0BAD_CAFE_F00D
LAYOUTS = ("padded", "packed", "gapped")
TAIL = 3                      # doubles after the last row


def flat_layout(widths, kind, seed=0):
    """Row starts (in doubles) of rows of the given widths laid out in one flat array; entry -1 is the length to
    allocate, which leaves TAIL doubles after the last row.
      padded: every row padded to an even length, so every start is even (16-byte aligned rows, the TMA paths);
      packed: rows back to back, so the starts take both parities when widths are odd;
      gapped: 1 to 3 unused doubles after every row (the tests also start these arrays 8 bytes past a 16-byte
              boundary, so no row is aligned)."""
    w = np.asarray(widths, dtype=np.int64)
    if kind == "padded":
        step = (w + 1) & ~1
    elif kind == "packed":
        step = w
    elif kind == "gapped":
        step = w + np.random.default_rng(seed).integers(1, 4, size=w.size)
    else:
        raise ValueError(kind)
    off = np.concatenate([[0], np.cumsum(step)])
    off[-1] += TAIL
    return off


def covered(off, widths, rows):
    """Mask of the flat array: True on the doubles of the given rows (problem numbers)."""
    mask = np.zeros(int(off[-1]), dtype=bool)
    for i in rows:
        mask[off[i]:off[i] + widths[i]] = True
    return mask


@pytest.mark.parametrize("kind", LAYOUTS)
def test_flat_layout_gives_each_layout_what_it_promises(kind):
    rng = np.random.default_rng(4)
    widths = rng.integers(1, 40, size=200)                 # odd and even widths
    widths[:4] = [1215, 1093, 32161, 969]                  # odd ones the evaluator has (n, m, nnz of the default class)
    off = flat_layout(widths, kind, seed=9)
    starts, gaps = off[:-1], off[1:-1] - (off[:-2] + widths[:-1])
    assert off.dtype == np.int64 and off.shape == (widths.size + 1,) and off[0] == 0
    assert off[-1] - (starts[-1] + widths[-1]) >= TAIL
    assert (gaps >= 0).all()                                # rows do not overlap
    if kind == "padded":
        assert (starts % 2 == 0).all() and (gaps == widths[:-1] % 2).all()
    elif kind == "packed":
        assert (gaps == 0).all() and set(starts % 2) == {0, 1}
    else:
        assert gaps.min() == 1 and gaps.max() == 3 and set(starts % 2) == {0, 1}
        assert np.array_equal(off, flat_layout(widths, kind, seed=9))      # seeded: one layout per seed
    # the sentinel mask: exactly the doubles outside the chosen rows
    rows = np.arange(1, widths.size, 2)
    mask = covered(off, widths, rows)
    assert mask.sum() == widths[rows].sum()
    for i in (1, 3, widths.size - 1):
        assert mask[off[i]:off[i] + widths[i]].all()
    for i in (0, 2):
        assert not mask[off[i]:off[i] + widths[i]].any()
    assert not mask[off[-2] + widths[-1]:].any()
    assert not mask[np.concatenate([np.arange(off[i] + widths[i], off[i + 1]) for i in range(widths.size)])].any()


def test_ragged_launches_refuse_mixed_patterns_and_kinematic_rows():
    """Both ragged entry points refuse, with QLNLP_EINVAL and the library's message, a launch whose classes mix
    SPARSE_BLOCK and SPARSE_TRUE handles and any kinematic handle.  The checks run before a device is bound, so the
    answer is the same with or without a GPU (no QLNLP_ENODEVICE)."""
    from test_cabi_cpu import _has_gpu

    L = ql.load_library()
    p, q = ql.build_problem(N=5, k_trans=3, init_mode=1), ql.build_problem(N=2, k_trans=1, init_mode=2)
    block, true = ql.HybridNLP.from_problem(p), ql.HybridNLP.from_problem(q, pattern="true")
    kin_block = ql.HybridNLP.from_problem(q, kinematics=True)
    kin_true = ql.HybridNLP.from_problem(p, pattern="true", kinematics=True)
    Z, off = np.zeros(2 * p.n_nlp + 2), np.zeros(2, dtype=np.int64)
    cls = np.zeros(2, dtype=np.int32)
    io, rg = ev._BatchIO(), ev._RaggedIO(None, off.ctypes.data, None, None, 0)
    # valid host pointers would reach a kernel on a GPU machine if a refusal were missing: there, Z stays NULL (and
    # the message below tells the two refusals apart)
    io.Z = None if _has_gpu() else Z.ctypes.data

    def classes(*nlps):
        hs = (C.c_void_p * len(nlps))(*[n._h.value for n in nlps])
        return L.qlnlp_eval_ragged_classes(hs, len(nlps), 1, C.byref(io), C.byref(rg), C.c_void_p(cls.ctypes.data), None)

    pattern, kin = "the classes of a ragged launch must share one Jacobian pattern", "ragged launches do not carry the kinematic rows"
    refusals = [
        (lambda: classes(block, true), pattern), (lambda: classes(true, block), pattern),
        (lambda: classes(true, true, block), pattern),
        (lambda: classes(kin_block), kin), (lambda: classes(block, kin_block), kin), (lambda: classes(true, kin_true), kin),
        (lambda: L.qlnlp_eval_ragged_device(kin_block._h, 1, C.byref(io), C.byref(rg), None), kin),
        (lambda: L.qlnlp_eval_ragged_device(kin_true._h, 1, C.byref(io), C.byref(rg), None), kin),
    ]
    for i, (call, msg) in enumerate(refusals):
        assert call() == ev.QLNLP_EINVAL and L.qlnlp_last_error().decode() == msg, (i, L.qlnlp_last_error())
    # B = 0 is no excuse: the classes are checked first
    hs = (C.c_void_p * 2)(block._h.value, true._h.value)
    assert L.qlnlp_eval_ragged_classes(hs, 2, 0, C.byref(io), C.byref(rg), C.c_void_p(cls.ctypes.data), None) == ev.QLNLP_EINVAL
    assert L.qlnlp_last_error().decode() == pattern
    assert L.qlnlp_eval_ragged_device(kin_block._h, 0, C.byref(io), C.byref(rg), None) == ev.QLNLP_EINVAL
    assert L.qlnlp_last_error().decode() == kin
