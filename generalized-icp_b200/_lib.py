"""ctypes binding of libgicp_b200.so (include/gicp_b200.h).  There is no CPU
fallback: if the shared library is missing this raises."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# GICP_B200_LIB: another build of the same library (A/B timing of kernel variants)
LIB_PATH = os.environ.get("GICP_B200_LIB") or os.path.join(_HERE, "libgicp_b200.so")

# every symbol include/gicp_b200.h declares
SYMBOLS = [
    "gicpCreate", "gicpDestroy", "gicpGetLastError", "gicpVersion", "gicpDefaultParams", "gicpSetParams",
    "gicpSetTarget", "gicpSetSource", "gicpSetPair", "gicpPromoteTargetToSource", "gicpRegister", "gicpKnn", "gicpCovariances", "gicpCorrespond",
    "gicpNormalEquations", "gicpSourceCovariancesAt", "gicpCommGetUniqueId", "gicpCommInit", "gicpCommDestroy",
    "gicpLaunchCount", "gicpProfile", "gicpProfileRead", "gicpRayCast", "gicpVoxelDownsample",
]


class GicpParams(C.Structure):
    """Mirror of ``struct gicpParams``."""
    _fields_ = [
        ("k", C.c_int32),
        ("max_iterations", C.c_int32),
        ("tolerance", C.c_double),
        ("max_distance_correspondence", C.c_double),
        ("max_distance_nearest_neighbors", C.c_double),
        ("lambda_tangent", C.c_double),
        ("lambda_normal", C.c_double),
        ("inner_max_iterations", C.c_int32),
        ("covariance_model", C.c_int32),
        ("knn_cell", C.c_double),
        ("nn_cell", C.c_double),
        ("max_cells_per_cloud", C.c_int64),
    ]


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  This engine has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, dp = C.c_void_p, C.c_int32, C.c_int64, C.POINTER(C.c_double)
    lib.gicpGetLastError.restype = C.c_char_p
    lib.gicpCreate.argtypes = [C.POINTER(vp), C.c_int, C.c_int, C.c_int]
    lib.gicpDestroy.argtypes = [vp]
    lib.gicpDefaultParams.argtypes = [C.POINTER(GicpParams)]
    lib.gicpSetParams.argtypes = [vp, C.POINTER(GicpParams)]
    for f in (lib.gicpSetTarget, lib.gicpSetSource):
        f.argtypes = [vp, vp, C.POINTER(i64), i32, vp]
    lib.gicpSetPair.argtypes = [vp, vp, C.POINTER(i64), vp, C.POINTER(i64), i32, vp]
    lib.gicpPromoteTargetToSource.argtypes = [vp]
    lib.gicpRegister.argtypes = [vp, dp, vp, vp, vp, vp, vp, vp, vp]
    lib.gicpKnn.argtypes = [vp, C.c_int, vp, vp, vp]
    lib.gicpCovariances.argtypes = [vp, C.c_int, vp, vp]
    lib.gicpCorrespond.argtypes = [vp, dp, vp, vp, vp, vp]
    lib.gicpNormalEquations.argtypes = [vp, dp, dp, vp]
    lib.gicpSourceCovariancesAt.argtypes = [vp, dp, i32, vp, vp]
    lib.gicpCommGetUniqueId.argtypes = [C.c_char_p]
    lib.gicpCommInit.argtypes = [vp, i32, i32, C.c_char_p]
    lib.gicpCommDestroy.argtypes = [vp]
    lib.gicpLaunchCount.argtypes = [vp]
    lib.gicpLaunchCount.restype = i64
    lib.gicpRayCast.argtypes = [C.c_int, vp, i32, i32, vp, i32, vp, i32, C.c_double, vp, vp, vp, vp]
    lib.gicpVoxelDownsample.argtypes = [vp, vp, C.POINTER(i64), i32, C.c_double, i32, vp, C.POINTER(i64), vp, vp, vp]
    lib.gicpProfile.argtypes = [vp, C.c_int]
    lib.gicpProfileRead.argtypes = [vp, dp, C.POINTER(i64)]
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise RuntimeError("libgicp_b200: " + load().gicpGetLastError().decode("utf-8", "replace"))
