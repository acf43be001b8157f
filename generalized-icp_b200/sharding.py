"""How the path shards over the ranks of one box (SURVEY.md 8e).  Pure host logic.

* independent scan pairs (BASELINE config 4): rank r registers the pairs of
  :func:`pair_range`; no collective on the data path;
* one large pair (config 5): every rank holds both clouds, rank r computes the
  target covariances of :func:`equal_slice` (all-gathered once inside the library)
  and runs the per-iteration reduction on the source points of
  :func:`source_slice`; the ranks' partial reduced forms are summed by one
  all-reduce of 80 doubles per outer iteration (ncclAllReduce inside
  libgicp_b200.so; the gloo stand-in below is what the CPU tests use).
"""
from __future__ import annotations


def pair_range(n_pairs: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous block of pairs of rank `rank`: sizes differ by at most one."""
    return n_pairs * rank // world, n_pairs * (rank + 1) // world


def source_slice(n_points: int, rank: int, world: int) -> tuple[int, int]:
    """Slice of the (Morton-sorted) source handled by `rank`: the slice plan_loop (csrc/plan.h) gives the
    registration loop (checked in tests/test_plan_host.py)."""
    return n_points * rank // world, n_points * (rank + 1) // world


def equal_slice(n_points: int, rank: int, world: int) -> tuple[int, int]:
    """Equal-length slices (the all-gather needs them); the tail slice is clipped.  The slice plan_setup (csrc/plan.h)
    gives the covariance estimation (checked in tests/test_plan_host.py)."""
    per = (n_points + world - 1) // world
    return min(n_points, per * rank), min(n_points, per * (rank + 1))


def allreduce_reduced_form(partial, group=None):
    """Sum the ranks' partial reduced forms (torch.distributed, any backend)."""
    import torch
    import torch.distributed as dist

    t = torch.as_tensor(partial, dtype=torch.float64).clone()
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t
