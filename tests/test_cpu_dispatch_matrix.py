"""CPU: every row of the dispatch matrix (tests/dispatch_cases.py) still reaches the kernel family and cluster size it was written for,
through the shape-only ABI queries gpode_forward_kernel and gpode_cluster_size -- no CUDA call.  When a launch heuristic is retuned,
this names the row whose GPU parity test (tests/test_gpu_dispatch_matrix.py) no longer exercises its kernel."""
import ctypes

import pytest

from dispatch_cases import ROWS, problem_fields, row_id


def _problem(row):
    from gpode_b200 import _lib
    variant, Lm, N, D_in, D_out, M, S, flags = problem_fields(row)
    p = _lib.GpodeProblem()
    p.variant, p.L, p.N, p.D_in, p.D_out, p.M, p.S, p.flags = _lib.VARIANTS[variant], Lm, N, D_in, D_out, M, S, flags
    return p


@pytest.mark.parametrize("row", ROWS, ids=row_id)
def test_row_reaches_its_family(row):
    from gpode_b200 import _lib
    lib = _lib.load()
    p = _problem(row)
    assert lib.gpode_forward_kernel(ctypes.byref(p)) == row.fwd_kernel, row.family
    assert lib.gpode_cluster_size(ctypes.byref(p)) == row.cluster, row.family
    small = row.family.split()[0].endswith("_small")
    assert (row.cluster > 1) <= small
    # the family name and the fields agree: small rows have 32-state CTAs, tensor rows D > 8 and a chip-filling batch
    if small:
        assert row.N * row.L <= 148 * 32 and row.fwd_per == row.bwd_per == 32
    if row.fwd_kernel:
        assert row.D_in > 8 and row.N * row.L >= 32768


def test_rows_are_distinct():
    ids = [row_id(r) for r in ROWS]
    assert len(set(ids)) == len(ids)
