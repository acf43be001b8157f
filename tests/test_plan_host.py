"""CPU-only checks of the host-side plans (generalized-icp_b200/csrc/plan.h, compiled for the host by
tests/host_harness/plan_host.cu): every path decision of a set-up, a registration and gicpSetPair against a
restatement of the expressions gicp_b200.cu used before the plans existed (commit 780211f; the line numbers below are
that file's), on batch shapes the GPU suite cannot afford and on both sides of every threshold."""
import ctypes as C
import itertools
import os
import shutil
import subprocess

import numpy as np
import pytest

SMALL_GRID_MAX, KNN_BRUTE_MAX = 2048, 128                      # grid.cuh, knn_cov.cuh
OBJ_THREADS, OBJ_MAX_PPT, PRESUM_SPAN = 128, 16, 64             # objective.cuh, solve.cuh
LIST_CAP = {True: 8192 // (32 * 8), False: 8192 // (32 * 12)}   # knn_list_cap<float> = 32, <double> = 21
ZERO, IDENTITY, KNN = 0, 1, 2                                   # CovSource
BRUTE, GENERAL, HIST_GENERAL = 0, 1, 2                          # KnnPath
SOURCE, TARGET = 0, 1


class Switches(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("no_skip", "track_max_cells", "shell_search", "centre_first", "corr_split",
                                       "active_list", "fused_loop", "small_grid", "knn_brute")] + \
               [("pair_overlap_max", C.c_longlong)]


DEFAULT_SW = dict(no_skip=0, track_max_cells=1 << 30, shell_search=1, centre_first=1, corr_split=2, active_list=1,
                  fused_loop=1, small_grid=1, knn_brute=1, pair_overlap_max=1 << 20)


class Setup(C.Structure):
    _fields_ = [("error", C.c_int), ("n_clouds", C.c_int), ("max_n", C.c_int), ("n_total", C.c_longlong),
                ("knn_cell", C.c_double), ("nn_cell", C.c_double), ("shared", C.c_int), ("budget", C.c_longlong)] + \
               [(n, C.c_int) for n in ("single_block", "inline_n", "cov", "knn", "knn_whole", "kc", "sharded",
                                       "slice_begin", "slice_end")] + [("slice_len", C.c_longlong)]


class Loop(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("slice_begin", "slice_end", "acc_ppt", "bpp", "search_ppt", "search_bpp",
                                       "fused", "self_init", "fused_ppt", "presum", "bpp2", "active_list", "sharded",
                                       "poll_every")]


def as_dict(s):
    return {f: getattr(s, f) for f, _ in s._fields_}


@pytest.fixture(scope="module")
def plan(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    out = str(tmp_path_factory.mktemp("plan_host") / "plan_host.so")
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_harness", "plan_host.cu")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O2", "-Xcompiler", "-fPIC",
                    "-shared", "-o", out, src], check=True)
    lib = C.CDLL(out)
    from generalized_icp_b200._lib import GicpParams
    P, S, I64 = C.POINTER(GicpParams), C.POINTER(Switches), C.POINTER(C.c_int64)
    lib.gicp_test_plan_setup.argtypes = [P, S, I64] + [C.c_int] * 6 + [C.POINTER(Setup)]
    lib.gicp_test_plan_loop.argtypes = [P, S, I64] + [C.c_int] * 7 + [C.POINTER(Loop)]
    lib.gicp_test_pair_overlap.argtypes = [S, C.c_int, C.c_int, C.c_longlong, C.c_longlong]
    lib.gicp_test_read_switches.argtypes = [S]
    lib.gicp_test_plan_loop_kernel.argtypes = [P, S, I64, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int)]

    def params(**kw):
        p = GicpParams(k=6, max_iterations=100, tolerance=1e-6, max_distance_correspondence=150.0,
                       max_distance_nearest_neighbors=50.0, lambda_tangent=100.0, lambda_normal=10.0,
                       inner_max_iterations=50)
        for k, v in kw.items():
            setattr(p, k, v)
        return p

    def setup(prm, sw, off, which=TARGET, f32=True, comm=0, n_ranks=1, rank=0):
        off = np.ascontiguousarray(off, dtype=np.int64)
        out = Setup()
        lib.gicp_test_plan_setup(C.byref(params(**prm)), C.byref(Switches(**{**DEFAULT_SW, **sw})),
                                 off.ctypes.data_as(I64), len(off) - 1, which, int(f32), comm, n_ranks, rank,
                                 C.byref(out))
        return as_dict(out)

    def loop(prm, sw, off, comm=0, n_ranks=1, rank=0, sliced=1, prof_on=0, has_T0=0):
        off = np.ascontiguousarray(off, dtype=np.int64)
        out = Loop()
        lib.gicp_test_plan_loop(C.byref(params(**prm)), C.byref(Switches(**{**DEFAULT_SW, **sw})),
                                off.ctypes.data_as(I64), len(off) - 1, comm, n_ranks, rank, sliced, prof_on, has_T0,
                                C.byref(out))
        return as_dict(out)

    def overlap(sw, comm, prof_on, n_t, n_s):
        return lib.gicp_test_pair_overlap(C.byref(Switches(**{**DEFAULT_SW, **sw})), comm, prof_on, n_t, n_s)

    def loop_kernel(prm, sw, off, robust, adaptive):
        off = np.ascontiguousarray(off, dtype=np.int64)
        out = (C.c_int * 4)()
        lib.gicp_test_plan_loop_kernel(C.byref(params(**prm)), C.byref(Switches(**{**DEFAULT_SW, **sw})),
                                       off.ctypes.data_as(I64), len(off) - 1, int(robust), int(adaptive), out)
        return dict(zip(("fused", "robust", "adaptive", "presum"), out))

    lib.setup, lib.loop, lib.overlap, lib.loop_kernel = setup, loop, overlap, loop_kernel
    return lib


# ------------------------------------------------------------------------------------------------
# the parent's expressions
# ------------------------------------------------------------------------------------------------
def _prm(prm):
    p = dict(k=6, max_distance_correspondence=150.0, max_distance_nearest_neighbors=50.0, covariance_model=0,
             knn_cell=0.0, nn_cell=0.0, max_cells_per_cloud=0)
    p.update(prm)
    return p


def parent_setup(prm, sw, off, which=TARGET, f32=True, comm=0, n_ranks=1, rank=0):
    p, sw = _prm(prm), {**DEFAULT_SW, **sw}
    off = np.asarray(off, dtype=np.int64)
    nc = len(off) - 1
    n_total, max_n = int(off[-1]), int(np.diff(off).max())
    r, d_max = p["max_distance_nearest_neighbors"], p["max_distance_correspondence"]
    # auto_knn_cell / auto_nn_cell, l. 477-488 (without the removed environment overrides)
    h_knn = max(p["knn_cell"], r / 8.0) if p["knn_cell"] > 0 else 0.25 * r
    h_nn = max(p["nn_cell"], d_max / 8.0) if p["nn_cell"] > 0 else 0.5 * d_max
    shared = h_knn <= 2.0 * h_nn and h_knn >= d_max / 8.0                        # l. 541-542
    mcpc = p["max_cells_per_cloud"]                                              # build_grid, l. 228-244
    budget = mcpc
    if budget <= 0:
        budget = 4096
        while budget < 8 * max_n:
            budget <<= 1
    if mcpc <= 0:
        while budget * nc > (1 << 30) and budget > 4096 and budget // 2 >= max_n:
            budget >>= 1
    if budget * nc > (1 << 30):
        budget = (1 << 30) // nc
    single = max_n <= SMALL_GRID_MAX and budget <= (1 << 20) and n_total > 0 and sw["small_grid"] != 0   # l. 264-265
    # latency_path, l. 492-501, and inline_n, l. 530
    latency_path = sw["small_grid"] != 0 and mcpc <= (1 << 20) and max_n <= SMALL_GRID_MAX and 0 < n_total <= 65536
    inline_n = n_total if nc == 1 and latency_path else -1
    model = p["covariance_model"]                                                # l. 561-564
    if model == 1 or (model == 2 and which == SOURCE):
        cov = IDENTITY if model == 1 and which == TARGET else ZERO
    else:
        cov = KNN
    sharded = bool(comm) and nc == 1                                             # l. 549-557
    slice_b = slice_e = -1
    per = 0
    if sharded:
        per = (n_total + n_ranks - 1) // n_ranks
        slice_b, slice_e = min(n_total, per * rank), min(n_total, per * (rank + 1))

    def knn(sb):                                                                 # launch_knn, l. 417-435, 440-465
        latency_mode = max_n <= SMALL_GRID_MAX and n_total <= 65536 and sw["small_grid"] != 0
        fast = p["k"] + 8 <= LIST_CAP[f32] and not latency_mode
        if latency_mode and max_n <= KNN_BRUTE_MAX and sb < 0 and sw["knn_brute"] != 0:
            return BRUTE
        return HIST_GENERAL if fast else GENERAL

    kc = 6 if p["k"] <= 6 else 20 if p["k"] <= 20 else 32
    return dict(error=0, n_clouds=nc, max_n=max_n, n_total=n_total, knn_cell=h_knn, nn_cell=h_nn, shared=int(shared),
                budget=budget, single_block=int(single), inline_n=inline_n, cov=cov, knn=knn(slice_b),
                knn_whole=knn(-1), kc=kc, sharded=int(sharded), slice_begin=slice_b, slice_end=slice_e,
                slice_len=per)


def parent_loop(prm, sw, off, comm=0, n_ranks=1, rank=0, sliced=1, prof_on=0, has_T0=0):
    sw = {**DEFAULT_SW, **sw}
    off = np.asarray(off, dtype=np.int64)
    np_ = len(off) - 1
    n_total, max_n = int(off[-1]), int(np.diff(off).max())
    span, sb, se = max_n, -1, -1                                                 # objective_args, l. 634-639
    if sliced and comm and np_ == 1:
        sb, se = n_total * rank // n_ranks, n_total * (rank + 1) // n_ranks
        span = se - sb
    total_pts = max(span, 1) * np_                                               # l. 641-649
    ppt = max(1, min(2 * OBJ_MAX_PPT, total_pts // (148 * 8 * OBJ_THREADS)))
    bpp = max(1, (span + OBJ_THREADS * ppt - 1) // (OBJ_THREADS * ppt))
    sharded = bool(comm) and np_ == 1                                            # do_register, l. 759
    fused = not sharded and not prof_on and max_n <= OBJ_THREADS * OBJ_MAX_PPT and sw["fused_loop"] != 0  # l. 693-694
    split = sw["corr_split"]                                                     # l. 752-757
    while int(ppt / split) > OBJ_MAX_PPT // 2:                                   # C integer division (split > 0 here)
        split *= 2
    while split > 1 and ppt % split:
        split -= 1
    oc_ppt = ppt // max(split, 1)
    return dict(slice_begin=sb, slice_end=se, acc_ppt=ppt, bpp=bpp, search_ppt=oc_ppt, search_bpp=bpp * (ppt // oc_ppt),
                fused=int(fused), self_init=int(fused and not has_T0),          # l. 696
                fused_ppt=max(1, (max_n + OBJ_THREADS - 1) // OBJ_THREADS),      # l. 726
                presum=int(bpp > 2 * PRESUM_SPAN), bpp2=(bpp + PRESUM_SPAN - 1) // PRESUM_SPAN,   # l. 741-742
                active_list=int(not sharded and np_ >= 64 and sw["active_list"] != 0),           # l. 772
                sharded=int(sharded), poll_every=2 if sharded else 1)            # l. 786, 832


def parent_overlap(sw, comm, prof_on, n_t, n_s):                                 # gicpSetPair, l. 1208-1210
    m = {**DEFAULT_SW, **sw}["pair_overlap_max"]
    return int(not comm and not prof_on and n_t <= m and n_s <= m)


# ------------------------------------------------------------------------------------------------
# shapes
# ------------------------------------------------------------------------------------------------
def _offs(sizes):
    return np.concatenate([[0], np.cumsum(np.asarray(sizes, dtype=np.int64))])


def _batches():
    """(name, offsets): both sides of max_n 128 / 2048, n_total 65536, np 64, bpp 2 * PRESUM_SPAN, 1 to 65535 clouds,
    the bench shape (4096 x 32768) and the config-5 pair (2^24 points), empty clouds."""
    b = {}
    for n in (1, 127, 128, 129, 2047, 2048, 2049, 16384, 16385, 100_000, 1 << 24):
        b[f"1x{n}"] = _offs([n])
    b["1x0"] = _offs([0])
    for nc, n in ((32, 2048), (512, 128), (29, 360), (1152, 700), (63, 500), (64, 500), (4096, 32768),
                  (65535, 1), (65535, 300), (16384, 2049), (2, 128)):
        b[f"{nc}x{n}"] = _offs([n] * nc)
    b["n_total 65537, max_n 2048"] = _offs([2048] * 32 + [1])
    b["n_total 65537, max_n 128"] = _offs([128] * 512 + [1])
    b["n_total 65536, max_n 129"] = _offs([128] * 511 + [129, 127])
    b["empty in the middle"] = _offs([300, 0, 217, 360])
    b["mixed 1..4000"] = _offs(np.random.default_rng(3).integers(0, 4000, 777))
    return b


BATCHES = _batches()
SWITCH_SETS = [{}, {"small_grid": 0}, {"knn_brute": 0}, {"fused_loop": 0}, {"active_list": 0}, {"no_skip": 1},
               {"corr_split": 1}, {"corr_split": 3}, {"corr_split": 4}, {"small_grid": 0, "fused_loop": 0, "knn_brute": 0}]
PARAM_SETS = [{}, {"k": 20, "max_distance_nearest_neighbors": 5.0, "max_distance_correspondence": 2.0},
              {"k": 24}, {"k": 25}, {"k": 13}, {"k": 14}, {"k": 32}, {"k": 7},
              {"max_distance_nearest_neighbors": 2.0, "max_distance_correspondence": 150.0},     # second grid
              {"knn_cell": 0.1, "nn_cell": 3.0, "max_distance_correspondence": 4.0},
              {"knn_cell": 9.0, "max_distance_nearest_neighbors": 5.0, "max_distance_correspondence": 2.0},
              {"max_cells_per_cloud": 1000}, {"max_cells_per_cloud": 1 << 20}, {"max_cells_per_cloud": (1 << 20) + 1},
              {"max_cells_per_cloud": 1 << 31},
              {"covariance_model": 1}, {"covariance_model": 2}]


def _check_setup(plan, prm, sw, off, **kw):
    got, want = plan.setup(prm, sw, off, **kw), parent_setup(prm, sw, off, **kw)
    assert got == want, (prm, sw, kw, {k: (got[k], want[k]) for k in got if got[k] != want[k]})
    # the offsets are never uploaded for an inline cloud: only the single-block build reads them from the argument
    assert got["inline_n"] < 0 or got["single_block"] == 1
    return got


@pytest.mark.parametrize("batch", list(BATCHES))
def test_setup_plan_matches_the_parent(plan, batch):
    off = BATCHES[batch]
    for prm in PARAM_SETS:
        for f32 in (True, False):
            _check_setup(plan, prm, {}, off, f32=f32, which=TARGET)
            _check_setup(plan, prm, {}, off, f32=f32, which=SOURCE)
    for sw in SWITCH_SETS:
        for prm in PARAM_SETS[:2]:
            _check_setup(plan, prm, sw, off)
    for prm, (n_ranks, rank) in itertools.product(PARAM_SETS[:2] + [{"covariance_model": 1}],
                                                  [(1, 0), (2, 0), (2, 1), (3, 2), (8, 0), (8, 7)]):
        _check_setup(plan, prm, {}, off, comm=1, n_ranks=n_ranks, rank=rank)


@pytest.mark.parametrize("batch", list(BATCHES))
def test_loop_plan_matches_the_parent(plan, batch):
    off = BATCHES[batch]
    for sw in SWITCH_SETS + [{"corr_split": -2}]:
        for prof_on, has_T0, sliced in itertools.product((0, 1), (0, 1), (0, 1)):
            got = plan.loop({}, sw, off, sliced=sliced, prof_on=prof_on, has_T0=has_T0)
            assert got == parent_loop({}, sw, off, sliced=sliced, prof_on=prof_on, has_T0=has_T0), (sw, prof_on, has_T0)
    for n_ranks, rank in [(1, 0), (2, 0), (2, 1), (8, 3), (8, 7)]:
        for sliced in (0, 1):
            got = plan.loop({}, {}, off, comm=1, n_ranks=n_ranks, rank=rank, sliced=sliced)
            assert got == parent_loop({}, {}, off, comm=1, n_ranks=n_ranks, rank=rank, sliced=sliced)


def test_search_split_for_every_ppt(plan):
    """Every accumulation ppt from 1 to 32 through the search split, including the ones without a small divisor
    (17, 19, 23, ...) that leave the search block unsplit - kept as measured."""
    seen = {}
    for ppt in range(1, 2 * OBJ_MAX_PPT + 1):
        off = _offs([ppt * 148 * 8 * OBJ_THREADS])
        for split in (1, 2, 3, 4, 8):
            got = plan.loop({}, {"corr_split": split}, off)
            assert got == parent_loop({}, {"corr_split": split}, off), (ppt, split)
            assert got["acc_ppt"] == ppt
            if split == 2:
                seen[ppt] = got["search_ppt"]
    assert seen[16] == 8 and seen[32] == 8 and seen[12] == 6
    assert seen[17] == 17 and seen[19] == 19 and seen[23] == 23 and seen[31] == 31   # the unsplit quirk


def test_sharding_slices_match_the_plans(plan):
    """sharding.equal_slice / source_slice are the slices the library's set-up and loop take."""
    from generalized_icp_b200 import sharding
    for n in (0, 1, 7, 1000, 100_001, 1 << 24):
        off = _offs([n])
        for world in (1, 2, 3, 8):
            for rank in range(world):
                s = plan.setup({}, {}, off, comm=1, n_ranks=world, rank=rank)
                assert (s["slice_begin"], s["slice_end"]) == sharding.equal_slice(n, rank, world)
                lp = plan.loop({}, {}, off, comm=1, n_ranks=world, rank=rank)
                assert (lp["slice_begin"], lp["slice_end"]) == sharding.source_slice(n, rank, world)


def test_pair_overlap_matches_the_parent(plan):
    for sw in ({}, {"pair_overlap_max": 0}, {"pair_overlap_max": 100_000}):
        for comm, prof_on in itertools.product((0, 1), (0, 1)):
            for n_t, n_s in itertools.product((0, 90, 100_000, 100_001, 1 << 20, (1 << 20) + 1), repeat=2):
                assert plan.overlap(sw, comm, prof_on, n_t, n_s) == parent_overlap(sw, comm, prof_on, n_t, n_s)


def test_invalid_offsets_are_refused(plan):
    for off in ([5, 10], [0, 10, 9], [0, (1 << 31) - 1024], [0, 1, (1 << 31)]):
        assert plan.setup({}, {}, off)["error"] == 1, off
    assert plan.setup({}, {}, [0] * 65537)["error"] == 1           # 65536 clouds
    assert plan.setup({}, {}, [0] * 65536)["error"] == 0


def test_read_switches(plan, monkeypatch):
    """Unset switches give the defaults; a set switch is parsed as the library parsed it (atoi / atoll)."""
    names = {"no_skip": "GICP_NO_SKIP", "track_max_cells": "GICP_TRACK_CELLS", "shell_search": "GICP_SHELL_SEARCH",
             "centre_first": "GICP_CENTRE_FIRST", "corr_split": "GICP_CORR_SPLIT", "active_list": "GICP_ACTIVE_LIST",
             "fused_loop": "GICP_FUSED_LOOP", "small_grid": "GICP_SMALL_GRID", "knn_brute": "GICP_KNN_BRUTE",
             "pair_overlap_max": "GICP_PAIR_OVERLAP_MAX"}
    for v in names.values():
        monkeypatch.delenv(v, raising=False)

    def read():
        s = Switches()
        plan.gicp_test_read_switches(C.byref(s))
        return as_dict(s)

    assert read() == DEFAULT_SW
    flags = ("no_skip", "active_list", "fused_loop", "small_grid", "knn_brute")
    for value, want in (("0", 0), ("1", 1), ("8", 8), ("", 0)):
        for k, v in names.items():
            monkeypatch.setenv(v, value)
        got = read()
        for k in names:
            assert got[k] == (int(want != 0) if k in flags else want), (k, value)


def test_param_table_reaches_its_plans(plan):
    """The fixed tables of tests/test_gpu_params.py reach the plans they are meant to: every cell row its cell edges,
    shared or unshared grid, budget and grid build on each input of part D; every K2 row of part A its k-NN path."""
    from test_gpu_params import CELL_DMAX, CELL_R, CELL_ROWS, CELL_SIZES, K2_PATHS, K2_RADIUS
    for case, (ns, nt) in CELL_SIZES.items():
        f32 = case == "3d_f32"
        k = 6 if case == "2d_f64" else 20
        for name, knobs, h_knn, h_nn, shared, budget, single_small in CELL_ROWS:
            prm = dict(k=k, max_distance_nearest_neighbors=CELL_R, max_distance_correspondence=CELL_DMAX, **knobs)
            for which, sizes in ((SOURCE, ns), (TARGET, nt)):
                got = _check_setup(plan, prm, {}, _offs(sizes), which=which, f32=f32)
                assert (got["knn_cell"], got["nn_cell"], got["shared"]) == (h_knn, h_nn, shared), (case, name)
                if budget is not None:
                    assert got["budget"] == budget, (case, name)
                assert got["single_block"] == int(single_small and max(sizes) <= SMALL_GRID_MAX), (case, name)
    for name, n, ks, storages in K2_PATHS:
        for dim, k in ks.items():
            for storage in storages:
                prm = dict(k=k, max_distance_nearest_neighbors=K2_RADIUS[dim], max_distance_correspondence=3.0)
                got = _check_setup(plan, prm, {}, _offs([n]), f32=storage == "f32")
                want = {"brute": BRUTE, "general_latency": GENERAL, "hist": HIST_GENERAL}.get(name, GENERAL)
                assert got["knn"] == want, (name, dim, storage, got["knn"])


def test_inner_minimum_rows_reach_their_loops(plan):
    """Every row of tests/test_gpu_inner_minimum.py reaches the loop it names: fused or multi-launch, plain, robust or
    adaptive, so the GPU table runs every instantiation of register_loop_kernel, accumulate_kernel, scale_select_kernel
    and solve_kernel it claims.  The 20 k-point row also folds its block partials first (presum_kernel)."""
    from test_gpu_inner_minimum import INPUTS, ROWS
    seen = set()
    for name, inp, storage, loop, kernel, model in ROWS:
        dim, n, params = INPUTS[inp]
        prm = {k: v for k, v in params.items() if k != "max_iterations"}
        sw = {"fused_loop": int(loop == "fused")} if n <= 2048 else {}
        got = plan.loop_kernel(dict(prm, covariance_model=model), sw, _offs([n]), kernel is not None,
                               kernel is not None and kernel[0] == "adaptive")
        want_kind = "plain" if kernel is None else kernel[0]
        assert got["fused"] == int(loop == "fused"), name
        assert got["robust"] == int(kernel is not None) and got["adaptive"] == int(want_kind == "adaptive"), name
        if inp == "big":
            assert got["presum"] == 1, name
        seen.add((dim, storage, loop, want_kind))
        seen.add((dim, storage, model))
    for dim, storage in itertools.product((2, 3), ("f32", "f64")):
        for kind in ("plain", "fixed", "adaptive"):                       # register_loop_kernel<D, Real, robust, adaptive>
            assert (dim, storage, "fused", kind) in seen, (dim, storage, kind)
        for kind in ("plain", "adaptive"):                                # accumulate_kernel, scale_select_kernel
            assert (dim, storage, "multi", kind) in seen, (dim, storage, kind)
        for model in (0, 1, 2):
            assert (dim, storage, model) in seen, (dim, storage, model)
    for dim, model in itertools.product((2, 3), (1, 2)):                  # models 1 and 2 in both loops
        for loop in ("fused", "multi"):
            assert any(INPUTS[r[1]][0] == dim and r[3] == loop and r[5] == model for r in ROWS), (dim, model, loop)
