"""Row-slab partition of the Bratu grid over the GPUs of one box (SURVEY 8e).

Pure integer host logic (no torch, no CUDA) so that it is testable everywhere.  The m grid rows
(slow index i) are split into ``world`` contiguous slabs whose sizes differ by at most one; slab
boundaries always fall on whole grid rows, so a halo is exactly ``depth`` rows of m doubles.
"""
from __future__ import annotations

HALO = 2  # stored halo depth (rows): depth 2 lets F be evaluated on one halo row without an exchange


def slab_bounds(m: int, world: int, rank: int):
    """Rows [i0, i1) owned by ``rank``; the first m % world ranks get one extra row."""
    if world < 1 or not (0 <= rank < world):
        raise ValueError("bad rank/world")
    base, extra = divmod(m, world)
    i0 = rank * base + min(rank, extra)
    i1 = i0 + base + (1 if rank < extra else 0)
    return i0, i1


def all_counts(m: int, world: int):
    """Owned unknowns per rank (rows * m), rank order."""
    return [(b - a) * m for a, b in (slab_bounds(m, world, r) for r in range(world))]


LS_TENSOR_MIN_ROWS = 16384  # smallest slab the tensor-pipe least squares accepts (csrc/tsqr.cu: gnk_tsqr_ls)


def tensor_ls_on_every_rank(m: int, world: int) -> bool:
    """True if every rank's slab qualifies for the tensor-pipe least squares (>= 16384 owned unknowns, even count).
    The library picks its path per call from the local slab; the tensor-pipe path and the Householder TSQR issue
    different collectives, so with slabs on both sides of the line the host must pin one path for all ranks."""
    return all(cn >= LS_TENSOR_MIN_ROWS and cn % 2 == 0 for cn in all_counts(m, world))


def trial_project_fused(m: int, world: int) -> bool:
    """True if gauss_newton_krylow forms its speculative Armijo trial and the first Gram-Schmidt inner products in one
    pass over the basis (gnk_bratu_trial_project): an even row length and slabs of >= 16384 owned unknowns -- the grids
    the pass is built for; smaller ones, where launches rather than the basis traffic dominate, and the numpy mock of the
    C ABI keep the separate kernels.  One rank only: the fused pass takes the Gram-Schmidt dots' place in the sequence
    of collectives, and several ranks keep today's sequence until that has run on more than one GPU.  Decided from m
    and world alone, so every rank decides alike."""
    return world == 1 and m % 2 == 0 and all(cn >= LS_TENSOR_MIN_ROWS for cn in all_counts(m, world))


def round_up(x: int, q: int) -> int:
    return (x + q - 1) // q * q


def stencil_layout_fields(m: int, world: int, rank: int):
    """Fields of gnk_layout for this rank's slab (see include/gnk_b200.h)."""
    i0, i1 = slab_bounds(m, world, rank)
    rows = i1 - i0
    if world > 1 and rows < HALO:
        raise ValueError(f"slab of {rows} grid rows is thinner than the halo ({HALO}); use fewer ranks")
    return dict(n_own=rows * m, off=HALO * m, ld=round_up((rows + 2 * HALO) * m, 16), m=m, rows=rows, halo=HALO,
                has_lo=int(rank > 0), has_hi=int(rank < world - 1), i0=i0, i1=i1)


def flat_layout_fields(n: int):
    return dict(n_own=n, off=0, ld=round_up(max(n, 1), 16), m=0, rows=0, halo=0, has_lo=0, has_hi=0, i0=0, i1=0)


def stored_column_from_global(x_global, fields, out):
    """Copy the rows [i0-HALO, i1+HALO) of a global vector into a stored column (numpy arrays);
    rows outside the domain stay zero (Dirichlet)."""
    m, i0, i1 = fields["m"], fields["i0"], fields["i1"]
    M = x_global.shape[0] // m
    lo = max(i0 - HALO, 0)
    hi = min(i1 + HALO, M)
    dst0 = (lo - (i0 - HALO)) * m
    out[:] = 0.0
    out[dst0:dst0 + (hi - lo) * m] = x_global[lo * m:hi * m]
    return out
