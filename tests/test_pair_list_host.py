"""CPU-only checks of plan_pairs (generalized-icp_b200/csrc/plan.h, compiled for the host by
tests/host_harness/pair_plan_host.cu): every refusal of gicpSetPairList's contract, the pair offsets, and the loop plan
of a pair list against that of the one-to-one batch it stands for (the batch whose p-th source is the pair's source
cloud), on shapes on both sides of the fused-loop, active-list, presum and acc_ppt > 16 thresholds."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

SOURCE, TARGET = 0, 1
FUSED_MAX = 128 * 16                 # OBJ_THREADS * OBJ_MAX_PPT
ACC_PPT_17 = 17 * 148 * 8 * 128      # total source points from which acc_ppt exceeds 16


class Loop(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("slice_begin", "slice_end", "acc_ppt", "bpp", "search_ppt", "search_bpp",
                                       "fused", "self_init", "fused_ppt", "presum", "bpp2", "active_list", "sharded",
                                       "poll_every", "robust", "adaptive")]


def as_dict(s):
    return {f: getattr(s, f) for f, _ in s._fields_}


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    out = str(tmp_path_factory.mktemp("pair_plan_host") / "pair_plan_host.so")
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_harness", "pair_plan_host.cu")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O2", "-Xcompiler", "-fPIC",
                    "-shared", "-o", out, src], check=True)
    lib = C.CDLL(out)
    I32, I64 = C.POINTER(C.c_int32), C.POINTER(C.c_int64)
    from generalized_icp_b200._lib import GicpParams
    lib.gicp_test_plan_pairs.argtypes = [C.c_int, I32, I32, C.c_int, I64, C.c_int, I64, C.c_int] + [C.c_int] * 4 + \
        [I64, C.POINTER(C.c_longlong), C.POINTER(Loop), C.c_char_p, C.c_int]
    lib.gicp_test_plan_loop_batch.argtypes = [C.POINTER(GicpParams), I64, C.c_int] + [C.c_int] * 4 + [C.POINTER(Loop)]
    prm = GicpParams(k=6, max_iterations=100, tolerance=1e-6, max_distance_correspondence=150.0,
                     max_distance_nearest_neighbors=50.0, lambda_tangent=100.0, lambda_normal=10.0,
                     inner_max_iterations=50)

    def plan_pairs(src, tgt, source_set, src_sizes, tgt_sizes, comm=0, has_T0=0, robust=0, adaptive=0, n_pairs=None):
        s = np.ascontiguousarray(src, dtype=np.int32)
        t = np.ascontiguousarray(tgt, dtype=np.int32)
        n_pairs = len(s) if n_pairs is None else n_pairs

        def offs(sizes):
            if sizes is None:
                return None, 0
            o = np.zeros(len(sizes) + 1, dtype=np.int64)
            o[1:] = np.cumsum(np.asarray(sizes, dtype=np.int64))
            return o, len(sizes)
        so, ns = offs(src_sizes)
        to, nt = offs(tgt_sizes)
        out_off = np.zeros(max(n_pairs, 0) + 1, dtype=np.int64)
        view = (C.c_longlong * 3)()
        loop = Loop()
        err = C.create_string_buffer(256)
        rc = lib.gicp_test_plan_pairs(n_pairs, s.ctypes.data_as(I32), t.ctypes.data_as(I32), source_set,
                                      so.ctypes.data_as(I64) if so is not None else None, ns,
                                      to.ctypes.data_as(I64) if to is not None else None, nt, comm, has_T0, robust,
                                      adaptive, out_off.ctypes.data_as(I64), view, C.byref(loop), err, 256)
        if rc:
            return err.value.decode()
        return out_off, tuple(view), as_dict(loop)

    def batch_loop(sizes, has_T0=0, robust=0, adaptive=0):
        o = np.zeros(len(sizes) + 1, dtype=np.int64)
        o[1:] = np.cumsum(np.asarray(sizes, dtype=np.int64))
        loop = Loop()
        lib.gicp_test_plan_loop_batch(C.byref(prm), o.ctypes.data_as(I64), len(sizes), 1, has_T0, robust, adaptive,
                                      C.byref(loop))
        return as_dict(loop)

    return plan_pairs, batch_loop


SIZES = [0, 1, 128, 129, 2048, 2049, 5000]


@pytest.mark.parametrize("source_set", [SOURCE, TARGET])
def test_offsets_and_view(lib, source_set):
    plan_pairs, _ = lib
    set_sizes = SIZES
    other = [7, 3]   # the target set when the sources come from the source set
    src = [6, 0, 1, 1, 4, 6, 2]
    tgt = [0, 1, 0, 1, 1, 0, 1] if source_set == SOURCE else [6, 6, 0, 1, 4, 2, 3]
    if source_set == SOURCE:
        r = plan_pairs(src, tgt, source_set, set_sizes, other)
    else:
        r = plan_pairs(src, tgt, source_set, None, set_sizes)
    off, view, _ = r
    sizes = [set_sizes[i] for i in src]
    assert off.tolist() == [0] + np.cumsum(sizes).tolist()
    assert view == (len(src), max(sizes), sum(sizes))


def test_refusals(lib):
    plan_pairs, _ = lib
    sz = [10, 20, 30]
    ok = plan_pairs([0, 2], [1, 2], SOURCE, sz, sz)
    assert not isinstance(ok, str)
    assert "communicator" in plan_pairs([0], [0], SOURCE, sz, sz, comm=1)
    for n in (0, -1, 65536):
        assert "n_pairs" in plan_pairs([0], [0], SOURCE, sz, sz, n_pairs=n)
    assert not isinstance(plan_pairs([0] * 65535, [0] * 65535, SOURCE, sz, sz), str)
    for bad in (-1, 2, 7):
        assert "source_set" in plan_pairs([0], [0], bad, sz, sz)
    assert "set source and target first" == plan_pairs([0], [0], SOURCE, None, sz)
    assert "set source and target first" == plan_pairs([0], [0], SOURCE, sz, None)
    assert "set the target first" == plan_pairs([0], [0], TARGET, sz, None)
    assert not isinstance(plan_pairs([0], [0], TARGET, None, sz), str)     # no source set needed
    for s, t in (([-1], [0]), ([3], [0]), ([0], [-1]), ([0], [3]), ([0, 1, 3], [0, 0, 0])):
        assert "out of range" in plan_pairs(s, t, SOURCE, sz, sz)
    # the source index range is the set it refers to
    assert "out of range" in plan_pairs([2], [0], SOURCE, [5, 5], [5, 5, 5])
    assert not isinstance(plan_pairs([2], [0], TARGET, [5, 5], [5, 5, 5]), str)
    assert "out of range" in plan_pairs([0], [2], TARGET, [5, 5, 5], [5, 5])
    # 2^31 - 1024 points summed over the pairs' sources, however few the clouds are
    lim = (1 << 31) - 1024
    big = [lim - 1, 1 << 29]
    assert not isinstance(plan_pairs([0], [0], SOURCE, big, big), str)
    assert "2^31" in plan_pairs([0, 0], [0, 0], SOURCE, big, big)
    assert "2^31" in plan_pairs([1, 1, 1, 1], [0] * 4, TARGET, None, big)
    assert not isinstance(plan_pairs([1, 1, 1], [0] * 3, TARGET, None, big), str)
    assert "2^31" in plan_pairs([0, 1], [0, 0], TARGET, None, [lim - 5, 5])
    assert not isinstance(plan_pairs([0, 1], [0, 0], TARGET, None, [lim - 5, 4]), str)


# (set sizes, pair sources): each row reaches its paths from either side of a threshold
ROWS = [
    ("fused", [100, 2048, 7], [0, 1, 1, 2]),
    ("fused_edge", [2049, 2048], [1, 1, 1]),
    ("multi", [2049, 2048], [1, 0]),
    ("empty", [0, 0, 1], [0, 1, 0]),
    ("active_63", [300, 4000], [0] * 62 + [1]),
    ("active_64", [300, 4000], [0] * 63 + [1]),
    ("active_64_fused", [300, 40], [1] * 64),
    ("presum_no", [16384, 10], [0]),
    ("presum_yes", [16385, 10], [0]),
    ("presum_large", [2_200_000], [0]),
    ("acc_ppt_16", [32768], [0] * (ACC_PPT_17 // 32768 - 1)),
    ("acc_ppt_17", [32768], [0] * (ACC_PPT_17 // 32768 + 1)),
    ("acc_ppt_32", [32768, 500], [0, 1] * 90),
]


@pytest.mark.parametrize("name,set_sizes,src", ROWS, ids=[r[0] for r in ROWS])
@pytest.mark.parametrize("source_set", [SOURCE, TARGET])
def test_loop_plan_equals_one_to_one(lib, name, set_sizes, src, source_set):
    plan_pairs, batch_loop = lib
    tgt = [i % 2 for i in range(len(src))]
    tsizes = [100, 200]
    sizes = [set_sizes[i] for i in src]
    seen = set()
    for has_T0 in (0, 1):
        for robust, adaptive in ((0, 0), (1, 0), (1, 1)):
            if source_set == SOURCE:
                r = plan_pairs(src, tgt, SOURCE, set_sizes, tsizes, has_T0=has_T0, robust=robust, adaptive=adaptive)
            else:
                r = plan_pairs(src, [s % len(set_sizes) for s in tgt], TARGET, None, set_sizes, has_T0=has_T0,
                               robust=robust, adaptive=adaptive)
            assert not isinstance(r, str), r
            _, _, loop = r
            assert loop == batch_loop(sizes, has_T0, robust, adaptive)
            seen.add((loop["fused"], loop["active_list"], loop["presum"], loop["acc_ppt"] > 16))
    fused, active, presum, ppt17 = seen.pop()
    expect = {"fused": (1, 0, 0, 0), "fused_edge": (1, 0, 0, 0), "multi": (0, 0, 0, 0), "empty": (1, 0, 0, 0),
              "active_63": (0, 0, 0, 0), "active_64": (0, 1, 0, 0), "active_64_fused": (1, 1, 0, 0),
              "presum_no": (0, 0, 0, 0), "presum_yes": (0, 0, 1, 0), "presum_large": (0, 0, 1, 0),
              "acc_ppt_16": (0, 1, 0, 0), "acc_ppt_17": (0, 1, 0, 1), "acc_ppt_32": (0, 1, 0, 1)}[name]
    assert (fused, active, presum, ppt17) == expect
