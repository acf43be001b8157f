"""Host side of the engine: a thin object over the C ABI (include/gicp_b200.h).

PyTorch is used for device memory and streams only; every computation happens
in libgicp_b200.so.  Method names mirror the stages of the reference's
``gicp()`` (python-implementation/gicp.py:78-174)."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from ._lib import GicpParams  # noqa: F401

SOURCE, TARGET = 0, 1
# robust kernels on the correspondence distance (GICP_ROBUST_*, include/gicp_b200.h)
ROBUST_KINDS = {None: 0, "huber": 1, "cauchy": 2, "tukey": 3}
_STORAGE = {"f32": (0, torch.float32), "f64": (1, torch.float64)}


@dataclass
class RegistrationResult:
    """Device-resident outputs of :meth:`GicpEngine.register` (one row per pair)."""
    T: torch.Tensor            # (P, d+1, d+1) f64   final transform (gicp.py:174 [0])
    n_outer: torch.Tensor      # (P,) i32            outer iterations executed
    converged_at: torch.Tensor  # (P,) i32           "Converged at iteration k" (gicp.py:161) or -1
    loss_hist: torch.Tensor | None   # (P, max_it) f64 min_loss per iteration (gicp.py:154)
    T_hist: torch.Tensor | None      # (P, max_it+1, d+1, d+1) all_transformations (gicp.py:108,167)
    inliers: torch.Tensor | None     # (P, max_it) i32


@dataclass
class RegistrationQuality:
    """Device-resident outputs of :meth:`GicpEngine.evaluate` at given transforms T (one row per pair; definitions in
    include/gicp_b200.h, gicpEvaluate).  xi = (rotation, translation), left perturbation T(xi) = Exp(xi) T."""
    n_inliers: torch.Tensor     # (P,) i32    gated-in correspondences at T
    fitness: torch.Tensor       # (P,) f64    n_inliers / source size (0 for an empty source)
    inlier_rmse: torch.Tensor   # (P,) f64    sqrt(mean d_i^2) over the inliers, Euclidean (0 without inliers)
    loss: torch.Tensor          # (P,) f64    sum w_i e_i^T W_i e_i (gicpNormalEquations' loss slot)
    H: torch.Tensor             # (P, 6, 6) / (P, 3, 3) f64  sum J^T w W J: information matrix, rotation first
    b: torch.Tensor             # (P, 6) / (P, 3) f64        sum J^T w W e: GN step H^-1 b, gradient -2 b


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class GicpEngine:
    """One engine = one C handle, bound to one device, one dimension and one storage type."""

    def __init__(self, dim: int, storage: str = "f32", device: int | None = None):
        if not torch.cuda.is_available():
            raise RuntimeError("GicpEngine needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        self.dim = int(dim)
        self.storage = storage
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", self.device_index)
        self._storage_code, self.dtype = _STORAGE[storage]
        self._h = C.c_void_p()
        _lib.check(self.lib.gicpCreate(C.byref(self._h), self.device_index, self.dim, self._storage_code))
        self.params = GicpParams()
        _lib.check(self.lib.gicpDefaultParams(C.byref(self.params)))
        self._keep = {}
        self._n = {SOURCE: (0, 0), TARGET: (0, 0)}

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.gicpDestroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- parameters (names of gicp.py:78 plus the engine's own) ----
    def set_params(self, **kw):
        """Set the named fields (include/gicp_b200.h, gicpParams).  A rejected set leaves the engine's parameters and
        set-up clouds as they were."""
        p = GicpParams.from_buffer_copy(self.params)
        for k, v in kw.items():
            if not hasattr(p, k):
                raise TypeError(f"unknown parameter {k!r}")
            setattr(p, k, v)
        _lib.check(self.lib.gicpSetParams(self._h, C.byref(p)))
        self.params = p

    def set_robust_kernel(self, kind, scale=None, *, adaptive=None, min_scale=None):
        """Weight every gated-in correspondence by a robust kernel of its distance d (IRLS, weights frozen at T_k):
        ``kind`` None (no weighting, the default), "huber", "cauchy" or "tukey"; ``scale`` c > 0 in the units of the
        points, like max_distance_correspondence.  Or, instead of ``scale``, ``adaptive`` = kappa with ``min_scale``:
        every pair's scale is set at every outer iteration to max(min_scale, kappa * median of its gated-in
        distances).  Semantics in include/gicp_b200.h.  Applies to every later register / correspond /
        normal_equations / robust_scales; the set-up clouds are kept."""
        if kind not in ROBUST_KINDS:
            raise ValueError(f"unknown robust kernel {kind!r}; expected one of None, 'huber', 'cauchy', 'tukey'")
        if kind is None:
            if adaptive is not None or min_scale is not None:
                raise ValueError("adaptive / min_scale need a kernel")
            _lib.check(self.lib.gicpSetRobustKernel(self._h, 0, 0.0))
            return
        if (scale is None) == (adaptive is None):
            raise ValueError(f"the {kind} kernel needs exactly one of a scale and adaptive=kappa")
        if adaptive is None:
            if min_scale is not None:
                raise ValueError("min_scale goes with adaptive=kappa")
            _lib.check(self.lib.gicpSetRobustKernel(self._h, ROBUST_KINDS[kind], float(scale)))
            return
        if min_scale is None:
            raise ValueError("an adaptive scale needs min_scale")
        _lib.check(self.lib.gicpSetRobustKernelAdaptive(self._h, ROBUST_KINDS[kind], float(adaptive), float(min_scale)))

    def robust_scales(self, T):
        """(P,) float64 numpy: every pair's robust scale at the transforms T (P, d+1, d+1) - the adaptive scale at the
        correspondences of T, a fixed scale as set, 0 without a kernel."""
        n_pairs = self._n[SOURCE][1]
        T, tp = self._T_arg(T)
        out = np.zeros((n_pairs,), dtype=np.float64)
        _lib.check(self.lib.gicpRobustScales(self._h, tp, out.ctypes.data_as(C.POINTER(C.c_double)), self._stream()))
        return out

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _prep(self, points, offsets):
        if not isinstance(points, torch.Tensor):
            points = torch.as_tensor(np.ascontiguousarray(np.asarray(points)), device=self.device)
        points = points.to(device=self.device, dtype=self.dtype).contiguous()
        if points.ndim != 2 or points.shape[1] != self.dim:
            raise ValueError(f"expected (N, {self.dim}) points, got {tuple(points.shape)}")
        if offsets is None:
            offsets = [0, points.shape[0]]
        off = np.ascontiguousarray(np.asarray(offsets, dtype=np.int64))
        if off[-1] != points.shape[0]:
            raise ValueError("offsets[-1] must equal the number of points")
        return points, off

    def _set(self, which, points, offsets):
        points, off = self._prep(points, offsets)
        self._keep[which] = points  # the library reads the caller's array later (covariance stage)
        self._n[which] = (points.shape[0], len(off) - 1)
        fn = self.lib.gicpSetTarget if which == TARGET else self.lib.gicpSetSource
        _lib.check(fn(self._h, _ptr(points), off.ctypes.data_as(C.POINTER(C.c_int64)), len(off) - 1, self._stream()))

    def set_target(self, points, offsets=None):
        """Grid build + covariances of the target(s): KDTree + compute_covariance_matrix, gicp.py:104."""
        self._set(TARGET, points, offsets)

    def set_source(self, points, offsets=None):
        """Grid build + covariances of the source(s): gicp.py:111."""
        self._set(SOURCE, points, offsets)

    def set_pair(self, target, source, target_offsets=None, source_offsets=None):
        """Both sides of one gicp() call (gicp.py:104 and :111) through gicpSetPair: same result as set_target +
        set_source; the set-up kernels of small clouds run concurrently on the device."""
        tp, toff = self._prep(target, target_offsets)
        sp, soff = self._prep(source, source_offsets)
        if len(toff) != len(soff):
            raise ValueError("source and target need the same number of clouds")
        self._keep[TARGET], self._keep[SOURCE] = tp, sp
        self._n[TARGET], self._n[SOURCE] = (tp.shape[0], len(toff) - 1), (sp.shape[0], len(soff) - 1)
        i64p = C.POINTER(C.c_int64)
        _lib.check(self.lib.gicpSetPair(self._h, _ptr(tp), toff.ctypes.data_as(i64p), _ptr(sp), soff.ctypes.data_as(i64p),
                                        len(toff) - 1, self._stream()))

    def promote_target_to_source(self):
        """Scan sequences: the current target (grids + covariances) becomes the source of the next pair
        (robot-visualization.py:250-251) without being rebuilt."""
        _lib.check(self.lib.gicpPromoteTargetToSource(self._h))
        self._keep[SOURCE] = self._keep.pop(TARGET, None)
        self._n[SOURCE] = self._n[TARGET]
        self._n[TARGET] = (0, 0)

    # ---- the loop ----
    def register(self, T0=None, history=True) -> RegistrationResult:
        n_pairs = self._n[SOURCE][1]
        d1 = self.dim + 1
        mi = int(self.params.max_iterations)
        dev = self.device
        T = torch.empty((n_pairs, d1, d1), dtype=torch.float64, device=dev)
        n_outer = torch.empty((n_pairs,), dtype=torch.int32, device=dev)
        conv = torch.empty((n_pairs,), dtype=torch.int32, device=dev)
        loss = torch.full((n_pairs, mi), float("nan"), dtype=torch.float64, device=dev) if history else None
        T_hist = torch.full((n_pairs, mi + 1, d1, d1), float("nan"), dtype=torch.float64, device=dev) if history else None
        inl = torch.zeros((n_pairs, mi), dtype=torch.int32, device=dev) if history else None
        t0p = None
        if T0 is not None:
            T0 = np.ascontiguousarray(np.asarray(T0, dtype=np.float64).reshape(n_pairs, d1, d1))
            t0p = T0.ctypes.data_as(C.POINTER(C.c_double))
        _lib.check(self.lib.gicpRegister(self._h, t0p, _ptr(T), _ptr(n_outer), _ptr(conv), _ptr(loss), _ptr(T_hist),
                                         _ptr(inl), self._stream()))
        return RegistrationResult(T, n_outer, conv, loss, T_hist, inl)

    def evaluate(self, T) -> RegistrationQuality:
        """Quality of every pair at the transforms T (P, d+1, d+1) through gicpEvaluate: inlier count, fitness, inlier
        RMSE, loss, information matrix H and vector b, as device tensors.  Stream-ordered, no synchronisation: a
        contiguous float64 T on the engine's device (e.g. ``register().T``) is read in place, anything else is copied
        there first."""
        n_pairs = self._n[SOURCE][1]
        d1, npar = self.dim + 1, 6 if self.dim == 3 else 3
        if not (isinstance(T, torch.Tensor) and T.device == self.device and T.dtype == torch.float64
                and T.is_contiguous()):
            T = torch.as_tensor(np.asarray(T, dtype=np.float64) if not isinstance(T, torch.Tensor) else T)
            T = T.to(device=self.device, dtype=torch.float64).contiguous()
        T = T.reshape(n_pairs, d1, d1)
        q = torch.empty((n_pairs, 4), dtype=torch.float64, device=self.device)
        H = torch.empty((n_pairs, npar, npar), dtype=torch.float64, device=self.device)
        b = torch.empty((n_pairs, npar), dtype=torch.float64, device=self.device)
        _lib.check(self.lib.gicpEvaluate(self._h, _ptr(T), _ptr(q), _ptr(H), _ptr(b), self._stream()))
        return RegistrationQuality(q[:, 0].to(torch.int32), q[:, 1], q[:, 2], q[:, 3], H, b)

    def register_pair_host(self, src, tgt):
        """One pair given as HOST arrays, everything the reference's 7-tuple needs back as host numpy arrays, with
        the fewest host<->device round trips: both clouds travel in ONE staged copy (pinned, cached), every output
        of gicpRegister + gicpCovariances lands in one cached device buffer that comes back in one copy.
        (`set_target` + `set_source` + `register` + `covariances` issue 9 small copies / synchronisations for the
        same result, which is most of the wall time of a 360-point registration.)  Returns a dict: T, T_hist, loss_hist,
        inliers, n_outer, converged_at, src_cov0, tgt_cov."""
        d, d1 = self.dim, self.dim + 1
        mi = int(self.params.max_iterations)
        np_dt = np.float64 if self.storage == "f64" else np.float32
        src = np.ascontiguousarray(src, dtype=np_dt)
        tgt = np.ascontiguousarray(tgt, dtype=np_dt)
        if src.ndim != 2 or tgt.ndim != 2 or src.shape[1] != d or tgt.shape[1] != d:
            raise ValueError(f"expected (N, {d}) points, got {src.shape} and {tgt.shape}")
        n_s, n_t = src.shape[0], tgt.shape[0]
        pad_s = (n_s + 3) & ~3                                  # keeps the target rows 16-byte aligned
        rows = pad_s + n_t
        if getattr(self, "_pp_rows", -1) < rows:
            cap = max(rows, 1024)
            self._pp_host = torch.empty((cap, d), dtype=self.dtype, pin_memory=True)
            self._pp_dev = torch.empty((cap, d), dtype=self.dtype, device=self.device)
            self._pp_rows = cap
        hv = self._pp_host.numpy()
        hv[:n_s] = src
        hv[pad_s:rows] = tgt
        self._pp_dev[:rows].copy_(self._pp_host[:rows], non_blocking=True)
        # both clouds through gicpSetPair, straight from the staging buffer (no per-call tensor views or checks: the
        # host's submission time is on the critical path of a 90-point registration)
        vp = C.c_void_p
        st = self._stream()
        base, row_bytes = self._pp_dev.data_ptr(), d * self._pp_dev.element_size()
        self._keep[TARGET] = self._keep[SOURCE] = self._pp_dev
        self._n[TARGET], self._n[SOURCE] = (n_t, 1), (n_s, 1)
        _lib.check(self.lib.gicpSetPair(self._h, vp(base + pad_s * row_bytes), (C.c_int64 * 2)(0, n_t), vp(base),
                                        (C.c_int64 * 2)(0, n_s), 1, st))
        # outputs: [T | loss_hist | T_hist | src_cov | tgt_cov] (f64) followed by [n_outer | converged | inliers] (i32)
        # in ONE cached device buffer with a pinned host mirror: one device->host copy, no fill kernels (the rows the
        # loop did not reach are set to NaN on the host copy)
        sizes = [d1 * d1, mi, (mi + 1) * d1 * d1, n_s * d * d, n_t * d * d]
        offs = [0]
        for z in sizes:
            offs.append(offs[-1] + z)
        nd = offs[-1]
        tot = nd + (2 + mi + 1) // 2
        if getattr(self, "_po_len", -1) < tot:
            cap = max(tot, 4096)
            self._po_dev = torch.empty((cap,), dtype=torch.float64, device=self.device)
            self._po_host = torch.empty((cap,), dtype=torch.float64, pin_memory=True)
            self._po_len = cap
        dp = self._po_dev.data_ptr()
        ip = dp + 8 * nd
        _lib.check(self.lib.gicpRegister(self._h, None, vp(dp), vp(ip), vp(ip + 4), vp(dp + 8 * offs[1]),
                                         vp(dp + 8 * offs[2]), vp(ip + 8), st))
        if n_s:
            _lib.check(self.lib.gicpCovariances(self._h, SOURCE, vp(dp + 8 * offs[3]), st))
        if n_t:
            _lib.check(self.lib.gicpCovariances(self._h, TARGET, vp(dp + 8 * offs[4]), st))
        self._po_host[:tot].copy_(self._po_dev[:tot], non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        hd = self._po_host.numpy()[:tot].copy()     # the pinned mirror is reused by the next call
        hi = hd[nd:].view(np.int32)
        n_outer, conv = int(hi[0]), int(hi[1])
        T_hist = hd[offs[2]:offs[3]].reshape(mi + 1, d1, d1)
        T_hist[(n_outer if conv >= 0 else n_outer + 1):] = np.nan   # rows the loop wrote: SURVEY appendix A rule 12
        return dict(T=hd[:offs[1]].reshape(d1, d1), loss_hist=hd[offs[1]:offs[2]][:n_outer], T_hist=T_hist,
                    src_cov0=hd[offs[3]:offs[4]].reshape(n_s, d, d), tgt_cov=hd[offs[4]:offs[5]].reshape(n_t, d, d),
                    n_outer=n_outer, converged_at=conv, inliers=hi[2:2 + mi][:n_outer])

    def register_next_scan_host(self, scan, have_previous, evaluate=False):
        """Scan sequences with HOST scans (robot-visualization.py:246-252): the previous target is promoted to the
        source (grids + covariances reused), `scan` becomes the target, the pair is registered.  One staged upload, one
        read-back (T, n_outer, converged_at), no per-call allocations; the first scan of a sequence
        (`have_previous=False`) is only set up.  Returns None or dict(T, n_outer, converged_at).  With ``evaluate``
        gicpEvaluate runs on the device T before the read-back and the dict also holds ``quality``: dict(n_inliers,
        fitness, inlier_rmse, loss, H, b) at T, brought back by the same copy."""
        d, d1 = self.dim, self.dim + 1
        np_dt = np.float64 if self.storage == "f64" else np.float32
        scan = np.ascontiguousarray(scan, dtype=np_dt)
        if scan.ndim != 2 or scan.shape[1] != d:
            raise ValueError(f"expected (N, {d}) points, got {scan.shape}")
        n = scan.shape[0]
        if getattr(self, "_sc_rows", -1) < n:
            cap = max(n, 1024)
            # two slots: the promoted source still refers to the previous scan's device array
            self._sc_host = [torch.empty((cap, d), dtype=self.dtype, pin_memory=True) for _ in range(2)]
            self._sc_dev = [torch.empty((cap, d), dtype=self.dtype, device=self.device) for _ in range(2)]
            self._sc_out_dev = torch.empty((d1 * d1 + 1,), dtype=torch.float64, device=self.device)
            self._sc_out_host = torch.empty((d1 * d1 + 1,), dtype=torch.float64, pin_memory=True)
            self._sc_rows, self._sc_slot = cap, 0
        slot = self._sc_slot = self._sc_slot ^ 1
        self._sc_host[slot].numpy()[:n] = scan
        self._sc_dev[slot][:n].copy_(self._sc_host[slot][:n], non_blocking=True)
        vp = C.c_void_p
        st = self._stream()
        if have_previous:
            self.promote_target_to_source()
        self._keep[TARGET] = self._sc_dev[slot]
        self._n[TARGET] = (n, 1)
        _lib.check(self.lib.gicpSetTarget(self._h, vp(self._sc_dev[slot].data_ptr()), (C.c_int64 * 2)(0, n), 1, st))
        if not have_previous:
            return None
        # outputs: [T | n_outer, converged_at (i32)] and, with evaluate, [quality (4) | H | b] behind them
        npar = 6 if d == 3 else 3
        if evaluate and getattr(self, "_sc_q_dev", None) is None:
            n_q = d1 * d1 + 1 + 4 + npar * npar + npar
            self._sc_q_dev = torch.empty((n_q,), dtype=torch.float64, device=self.device)
            self._sc_q_host = torch.empty((n_q,), dtype=torch.float64, pin_memory=True)
        out_dev, out_host = (self._sc_q_dev, self._sc_q_host) if evaluate else (self._sc_out_dev, self._sc_out_host)
        dp = out_dev.data_ptr()
        ip = dp + 8 * d1 * d1
        _lib.check(self.lib.gicpRegister(self._h, None, vp(dp), vp(ip), vp(ip + 4), None, None, None, st))
        if evaluate:
            qp = ip + 8
            _lib.check(self.lib.gicpEvaluate(self._h, vp(dp), vp(qp), vp(qp + 32), vp(qp + 32 + 8 * npar * npar), st))
        out_host.copy_(out_dev, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        hd = out_host.numpy().copy()
        hi = hd[d1 * d1:d1 * d1 + 1].view(np.int32)
        r = dict(T=hd[:d1 * d1].reshape(d1, d1), n_outer=int(hi[0]), converged_at=int(hi[1]))
        if evaluate:
            q = hd[d1 * d1 + 1:]
            r["quality"] = dict(n_inliers=int(q[0]), fitness=float(q[1]), inlier_rmse=float(q[2]), loss=float(q[3]),
                                H=q[4:4 + npar * npar].reshape(npar, npar), b=q[4 + npar * npar:])
        return r

    def register_host_batch(self, h_src, h_tgt, offsets, chunk_pairs=1024, history=False):
        """Batches that live in (pinned) HOST memory: pairs are registered in chunks, and the host->device
        copy of chunk i+1 runs on a second stream while chunk i is being registered, so the PCIe transfer
        hides behind the compute (the first chunk is 1/8 of the others: its upload is exposed).  h_src / h_tgt: (n_total, dim) CPU tensors (pin them for real overlap),
        offsets: (n_pairs + 1,) row offsets shared by both sides.  Returns (T (P, d+1, d+1), n_outer (P,),
        converged_at (P,)) as pinned host tensors."""
        off = np.asarray(offsets, dtype=np.int64)
        n_pairs = len(off) - 1
        d1 = self.dim + 1
        T_out = torch.empty((n_pairs, d1, d1), dtype=torch.float64, pin_memory=True)
        n_out = torch.empty((n_pairs,), dtype=torch.int32, pin_memory=True)
        c_out = torch.empty((n_pairs,), dtype=torch.int32, pin_memory=True)
        # the first chunk's upload is the only one nothing hides behind: keep it small (1/8 of a chunk; a chunk's
        # upload takes ~1/8 of its registration on the bench workload, so the second upload is still hidden).
        # Doubling the chunk size from there was measured too: 95.7 % instead of 96.4 % of the device-resident rate
        # (every extra chunk adds a convergence tail).
        first = min(n_pairs, max(1, chunk_pairs // 8)) if n_pairs > chunk_pairs else n_pairs
        chunks = [(0, first)] + [(a, min(a + chunk_pairs, n_pairs)) for a in range(first, n_pairs, chunk_pairs)]
        rows = max(int(off[b] - off[a]) for a, b in chunks)
        if getattr(self, "_hb_rows", 0) < rows:
            self._hb = [(torch.empty((rows, self.dim), dtype=self.dtype, device=self.device),
                         torch.empty((rows, self.dim), dtype=self.dtype, device=self.device)) for _ in range(2)]
            self._hb_rows = rows
            self._copy_stream = torch.cuda.Stream(device=self.device)
        main = torch.cuda.current_stream(self.device)

        def upload(i):
            a, b = chunks[i]
            r0, r1 = int(off[a]), int(off[b])
            ds, dt = self._hb[i % 2]
            self._copy_stream.wait_stream(main)       # the buffer's previous user (chunk i-2) is done
            with torch.cuda.stream(self._copy_stream):
                ds[:r1 - r0].copy_(h_src[r0:r1], non_blocking=True)
                dt[:r1 - r0].copy_(h_tgt[r0:r1], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self._copy_stream)
            return ev

        ev = upload(0)
        for i, (a, b) in enumerate(chunks):
            r0, r1 = int(off[a]), int(off[b])
            ds, dt = self._hb[i % 2]
            main.wait_event(ev)
            if i + 1 < len(chunks):
                ev = upload(i + 1)                    # in flight while this chunk is registered
            loc = off[a:b + 1] - off[a]
            self.set_target(dt[:r1 - r0], loc)
            self.set_source(ds[:r1 - r0], loc)
            r = self.register(history=history)
            T_out[a:b].copy_(r.T, non_blocking=True)
            n_out[a:b].copy_(r.n_outer, non_blocking=True)
            c_out[a:b].copy_(r.converged_at, non_blocking=True)
        torch.cuda.synchronize(self.device)
        return T_out, n_out, c_out

    # ---- voxel-grid downsampling ----
    def voxel_downsample(self, points, offsets=None, *, voxel_size, min_points=1, with_index=False):
        """Voxel-grid filter of a batch on the device (gicpVoxelDownsample; semantics in include/gicp_b200.h): every
        voxel of edge ``voxel_size`` with >= ``min_points`` finite points becomes their centroid, in the order of each
        voxel's lowest input row.  Returns ``(pts, out_offsets)`` - pts (M, d) on the engine's device in its dtype, a
        tensor of its own (safe to pass to set_source / set_target: no later call writes it), out_offsets (P+1,)
        int64 numpy, usable as the offsets of set_*.  With ``with_index`` also ``(voxel_of (N,) i32, counts (M,) i32)``:
        each input row's cloud-local output row (-1 when dropped) and the points behind each output row.  Leaves the
        engine's source and target as they are."""
        points, off = self._prep(points, offsets)
        n, nc = points.shape[0], len(off) - 1
        out = torch.empty((n, self.dim), dtype=self.dtype, device=self.device)
        out_off = np.zeros(nc + 1, dtype=np.int64)
        vox = torch.empty((n,), dtype=torch.int32, device=self.device) if with_index else None
        cnt = torch.empty((n,), dtype=torch.int32, device=self.device) if with_index else None
        i64p = C.POINTER(C.c_int64)
        _lib.check(self.lib.gicpVoxelDownsample(self._h, _ptr(points), off.ctypes.data_as(i64p), nc, float(voxel_size),
                                                int(min_points), _ptr(out), out_off.ctypes.data_as(i64p), _ptr(vox),
                                                _ptr(cnt), self._stream()))
        m = int(out_off[-1])
        pts = out[:m].clone() if m < n else out
        if with_index:
            return pts, out_off, vox, cnt[:m].clone()
        return pts, out_off

    # ---- stage entry points ----
    def knn(self, which, with_dist=True):
        n = self._n[which][0]
        k = int(self.params.k)
        idx = torch.empty((n, k), dtype=torch.int32, device=self.device)
        dist = torch.empty((n, k), dtype=torch.float64, device=self.device) if with_dist else None
        _lib.check(self.lib.gicpKnn(self._h, which, _ptr(idx), _ptr(dist), self._stream()))
        return idx, dist

    def covariances(self, which):
        n = self._n[which][0]
        out = torch.empty((n, self.dim, self.dim), dtype=torch.float64, device=self.device)
        _lib.check(self.lib.gicpCovariances(self._h, which, _ptr(out), self._stream()))
        return out

    def _T_arg(self, T, lead=()):
        n_pairs = self._n[SOURCE][1]
        d1 = self.dim + 1
        T = np.ascontiguousarray(np.asarray(T, dtype=np.float64).reshape(*lead, n_pairs, d1, d1))
        return T, T.ctypes.data_as(C.POINTER(C.c_double))

    def correspond(self, T, with_W=True):
        n = self._n[SOURCE][0]
        T, tp = self._T_arg(T)
        idx = torch.empty((n,), dtype=torch.int32, device=self.device)
        dist = torch.empty((n,), dtype=torch.float64, device=self.device)
        W = torch.empty((n, self.dim, self.dim), dtype=torch.float64, device=self.device) if with_W else None
        _lib.check(self.lib.gicpCorrespond(self._h, tp, _ptr(idx), _ptr(dist), _ptr(W), self._stream()))
        return idx, dist, W

    def normal_equations(self, T):
        n_pairs = self._n[SOURCE][1]
        T, tp = self._T_arg(T)
        nred = 80 if self.dim == 3 else 32
        out = np.zeros((n_pairs, nred), dtype=np.float64)
        _lib.check(self.lib.gicpNormalEquations(self._h, tp, out.ctypes.data_as(C.POINTER(C.c_double)), self._stream()))
        return out

    def source_covariances_at(self, Ts):
        Ts = np.asarray(Ts, dtype=np.float64)
        n_T = Ts.shape[0]
        T, tp = self._T_arg(Ts, lead=(n_T,))
        n = self._n[SOURCE][0]
        out = torch.empty((n_T, n, self.dim, self.dim), dtype=torch.float64, device=self.device)
        _lib.check(self.lib.gicpSourceCovariancesAt(self._h, tp, n_T, _ptr(out), self._stream()))
        return out

    # ---- multi-GPU (sharded source, config 5) ----
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        _lib.check(_lib.load().gicpCommGetUniqueId(buf))
        return buf.raw

    def comm_init(self, n_ranks, rank, unique_id: bytes):
        _lib.check(self.lib.gicpCommInit(self._h, n_ranks, rank, C.create_string_buffer(unique_id, 128)))

    def comm_destroy(self):
        _lib.check(self.lib.gicpCommDestroy(self._h))

    STAGES = ("grid_build", "knn_cov", "correspond", "accumulate", "solve")

    def profile(self, enable=True):
        _lib.check(self.lib.gicpProfile(self._h, int(bool(enable))))

    def profile_read(self, scale_select=False):
        """{stage: (milliseconds, timed sections)} since the last read (device-synchronising).  With
        ``scale_select`` also "scale_select": the adaptive robust scale's select of the multi-launch loop."""
        names = self.STAGES + (("scale_select",) if scale_select else ())
        ms = (C.c_double * len(names))()
        cnt = (C.c_int64 * len(names))()
        _lib.check(self.lib.gicpProfileReadStages(self._h, len(names), ms, cnt))
        return {s: (float(ms[i]), int(cnt[i])) for i, s in enumerate(names)}

    @property
    def launch_count(self):
        return int(self.lib.gicpLaunchCount(self._h))


def reduced_form_loss(red, dim, T_lin, T_eval):
    """f(Z) = c - 2<G,Z> + <Z,HZ> with Z = [dt | dR - I] for the transform T_eval expressed
    relative to the linearisation transform T_lin (layout: include/gicp_b200.h)."""
    d = dim
    NP, NS = d + 1, d * (d + 1) // 2
    NAB = NP * (NP + 1) // 2
    NH = NAB * NS
    Hq = red[:NH].reshape(NAB, NS)
    G = red[NH:NH + d * NP].reshape(d, NP)
    c = red[NH + d * NP]
    mu = red[NH + d * NP + 2:NH + d * NP + 2 + d]
    dR = T_eval[:d, :d] @ np.linalg.inv(T_lin[:d, :d])
    dt = T_eval[:d, d] - dR @ T_lin[:d, d]
    dtc = dt + (dR - np.eye(d)) @ mu
    Z = np.concatenate([dtc[:, None], dR - np.eye(d)], axis=1)          # (d, NP)

    def sym(n, a, b):
        a, b = min(a, b), max(a, b)
        return a * n - a * (a - 1) // 2 + (b - a)

    quad = 0.0
    for a in range(NP):
        for b in range(NP):
            for cc in range(d):
                for dd in range(d):
                    quad += Z[cc, a] * Z[dd, b] * Hq[sym(NP, a, b), sym(d, cc, dd)]
    return float(c - 2.0 * np.sum(G * Z) + quad)


def reduced_form_grad2d(red, T_lin, x):
    """Gradient of the frozen inner objective with respect to the reference's parameters (tx, ty, theta)
    (what grad_loss returns, gicp.py:60-76), derived from the reduced form K3 accumulates:
    f(Z) = c - 2<G,Z> + <Z,HZ>, Z(x) = [dt_c | dR - I], dR = R(theta) R_lin^-1, dt_c = t - dR t_lin + (dR - I) mu,
    so df/dx = <2 (H Z - G), dZ/dx>."""
    d, NP, NS = 2, 3, 3
    NAB = NP * (NP + 1) // 2
    NH = NAB * NS
    Hq = red[:NH].reshape(NAB, NS)
    G = red[NH:NH + d * NP].reshape(d, NP)
    mu = red[NH + d * NP + 2:NH + d * NP + 2 + d]
    th = float(x[2])
    R = np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]])
    dRdth = np.array([[-np.sin(th), -np.cos(th)], [np.cos(th), -np.sin(th)]])
    Rl_inv = np.linalg.inv(T_lin[:d, :d])
    dR = R @ Rl_inv
    dtc = np.asarray(x[:2], dtype=np.float64) - dR @ T_lin[:d, d] + (dR - np.eye(d)) @ mu
    Z = np.concatenate([dtc[:, None], dR - np.eye(d)], axis=1)

    def sym(n, a, b):
        a, b = min(a, b), max(a, b)
        return a * n - a * (a - 1) // 2 + (b - a)

    HZ = np.zeros_like(Z)
    for cc in range(d):
        for a in range(NP):
            HZ[cc, a] = sum(Hq[sym(NP, a, b), sym(d, cc, dd)] * Z[dd, b] for dd in range(d) for b in range(NP))
    Gam = 2.0 * (HZ - G)
    grad = np.zeros(3)
    for c in range(d):                                   # d/dt_c: dZ = e_c in column 0
        grad[c] = Gam[c, 0]
    dRp = dRdth @ Rl_inv                                 # d/dtheta
    dZ = np.concatenate([(-dRp @ T_lin[:d, d] + dRp @ mu)[:, None], dRp], axis=1)
    grad[2] = float(np.sum(Gam * dZ))
    return grad


def ray_cast(poses, num_rays=90, obstacles=None, max_range=400.0, noise=None, device=None):
    """Batched LiDAR scans on the device (robot-visualization.py:42-120, 222-237).
    poses: (n, 3) x, y, yaw_deg.  obstacles: list of (x, y, w, h) rectangles and (cx, cy, r) circles - default
    = the demo's world (robot-visualization.py:35-40).  noise: optional (n, num_rays) additive range noise.
    Returns (rel_xy (n, num_rays, 2) f64, hit (n, num_rays) bool) as device tensors."""
    lib = _lib.load()
    dev = torch.device("cuda", torch.cuda.current_device() if device is None else int(device))
    if obstacles is None:
        obstacles = [(100, 250, 200, 50), (400, 450, 50, 200), (600, 300, 50), (200, 550, 75)]
    segs, circs = [], []
    for ob in obstacles:
        if len(ob) == 4:
            x, y, w, h = ob
            tl, tr, bl, br = (x, y), (x + w, y), (x, y + h), (x + w, y + h)
            for p3, p4 in ((tl, tr), (tr, br), (br, bl), (bl, tl)):          # robot-visualization.py:52-57
                segs.append([*p3, *p4])
        else:
            circs.append(list(ob))
    poses_t = torch.as_tensor(np.asarray(poses, dtype=np.float64), device=dev).contiguous()
    n = poses_t.shape[0]
    seg_t = torch.as_tensor(np.asarray(segs, dtype=np.float64).reshape(-1, 4), device=dev)
    circ_t = torch.as_tensor(np.asarray(circs, dtype=np.float64).reshape(-1, 3), device=dev)
    noise_t = None if noise is None else torch.as_tensor(np.asarray(noise, dtype=np.float64), device=dev).contiguous()
    rel = torch.empty((n, num_rays, 2), dtype=torch.float64, device=dev)
    hit = torch.empty((n, num_rays), dtype=torch.int32, device=dev)
    _lib.check(lib.gicpRayCast(dev.index, _ptr(poses_t), n, num_rays, _ptr(seg_t), seg_t.shape[0], _ptr(circ_t),
                               circ_t.shape[0], float(max_range), _ptr(noise_t), _ptr(rel), _ptr(hit),
                               C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return rel, hit.bool()
