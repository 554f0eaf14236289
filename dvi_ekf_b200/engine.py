"""Batched VI-ESKF engine: thin Python wrapper over the C ABI.

``BatchFilter(N)`` owns N independent filters on one GPU.  Arrays may be numpy
arrays (host memory: copied by the library inside the call) or torch CUDA
tensors (device memory: used in place); all FP64, C-contiguous.  The verbs
mirror the reference's ``Filter`` (dvi_ekf/filter/Filter.py): ``propagate``,
``update``, ``run``, ``reset`` (= ``set_state``), ``update_noise_matrices``
(= ``set_noise``).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import numpy as np

from . import _lib
from ._lib import MEM_DEVICE, MEM_HOST, NCARRY, NCONS, NDOFSUM, NSTAT, EskfModel, EskfStreams, check


def _is_torch(a) -> bool:
    return type(a).__module__.startswith("torch")


class _Arg:
    """pointer + leading dimension + memory kind of one array argument"""

    def __init__(self, a, width: Optional[int], dtype=np.float64, name="array"):
        self.keep = None
        if a is None:
            self.ptr, self.rows, self.mem = None, 0, None
            return
        if _is_torch(a):
            import torch

            want = torch.float64 if dtype == np.float64 else torch.int32
            if not a.is_cuda:
                a = a.numpy()
            else:
                if a.dtype != want or not a.is_contiguous():
                    raise TypeError(f"{name}: CUDA tensors must be contiguous {want}")
                self.keep = a
                self.ptr = C.c_void_p(a.data_ptr())
                self.mem = MEM_DEVICE
                n = a.numel()
                self.rows = n // width if width else n
                if width and n % width:
                    raise ValueError(f"{name}: size {n} is not a multiple of {width}")
                return
        a = np.ascontiguousarray(a, dtype=dtype)
        self.keep = a
        self.ptr = a.ctypes.data_as(C.c_void_p)
        self.mem = MEM_HOST
        n = a.size
        self.rows = n // width if width else n
        if width and n % width:
            raise ValueError(f"{name}: size {n} is not a multiple of {width}")


def _common_mem(args: Sequence[_Arg]) -> int:
    mems = {a.mem for a in args if a.mem is not None}
    if len(mems) > 1:
        raise TypeError("all arrays of one call must live in the same memory space (all numpy or all CUDA tensors)")
    return mems.pop() if mems else MEM_HOST


def check_run_geometry(n_filters: int, n_traj: int, filters_per_traj: int, filter_id0: int, n_steps: int, n_epochs: int,
                       n_prop=None, epochs=None) -> None:
    """The argument checks of ``eskf_run`` / ``eskf_run_epochs`` (csrc/eskf_api.cu), mirrored on the host so that a bad shard
    plan or epoch range fails with a clear ``ValueError`` before anything is launched: the kernels pick a filter's trajectory
    from its GLOBAL id, ``(filter_id0 + f) // filters_per_traj``, and the sample stream by the running sum of ``n_prop``;
    ``epochs = (e0, e1)`` must satisfy 0 <= e0 <= e1 <= n_epochs."""
    if n_filters <= 0 or n_traj < 1 or n_steps < 0 or n_epochs < 0:
        raise ValueError("n_filters, n_traj must be positive and n_steps, n_epochs non-negative")
    if epochs is not None:
        e0, e1 = (int(v) for v in epochs)
        if not 0 <= e0 <= e1 <= n_epochs:
            raise ValueError(f"epoch range [{e0}, {e1}) is not within [0, n_epochs = {n_epochs}]")
    if filter_id0 < 0:
        raise ValueError("filter_id0 must be non-negative")
    if n_traj > 1:
        if filters_per_traj <= 0:
            raise ValueError("filters_per_traj must be positive when several trajectories are stacked")
        if filter_id0 % filters_per_traj:
            raise ValueError("filter_id0 must be a multiple of filters_per_traj (a shard starts at a trajectory boundary)")
        if filter_id0 + n_filters > n_traj * filters_per_traj:
            raise ValueError(f"filter_id0 + n_filters = {filter_id0 + n_filters} exceeds n_traj * filters_per_traj = "
                             f"{n_traj * filters_per_traj} (the streams of {n_traj} trajectories were passed)")
    if isinstance(n_prop, np.ndarray):
        npr = np.asarray(n_prop).reshape(n_traj, -1)
        if (npr < 0).any():
            raise ValueError("negative n_prop entry")
        tot = npr.sum(axis=1)
        if (tot > n_steps).any():
            raise ValueError(f"sum(n_prop) = {int(tot.max())} exceeds n_steps = {n_steps}")


def drop_prob_array(prob, n_traj: int, n_epochs: int, name: str = "drop_prob") -> np.ndarray:
    """The drop probabilities of ``BatchFilter.run(drop_prob=...)`` as the C-contiguous float64 [n_traj, n_epochs] array
    eskf_set_meas_dropout takes: ``prob`` is a scalar, [n_epochs] (every trajectory) or [n_traj, n_epochs], every entry
    finite and in [0, 1].  Raises ``ValueError`` otherwise.  (The outlier probabilities of eskf_set_meas_outliers are
    checked the same way; ``name`` names the argument in the message.)"""
    p = np.asarray(prob, dtype=np.float64)
    if p.ndim > 2 or (p.ndim >= 1 and p.shape[-1] != n_epochs) or (p.ndim == 2 and p.shape[0] != n_traj):
        raise ValueError(f"{name} must be a scalar, [{n_epochs}] or [{n_traj}, {n_epochs}] (n_traj, n_epochs of the streams), "
                         f"not of shape {p.shape}")
    if not np.isfinite(p).all():
        raise ValueError(f"{name} must be finite (NaN or infinite entry)")
    if (p < 0).any() or (p > 1).any():
        raise ValueError(f"{name} entries are probabilities in [0, 1], not {float(p.min())} .. {float(p.max())}")
    return np.ascontiguousarray(np.broadcast_to(p, (n_traj, n_epochs)))


def mask_from_uniforms(u, p, noise_free) -> np.ndarray:
    """The dropout rule of eskf_set_meas_dropout (include/eskf.h) on given uniforms: ``u`` and ``p`` [n, E] (the filters'
    uniforms and drop probabilities), ``noise_free`` [n] (noise-free reference filters, which lose only the epochs with
    p == 1).  Returns bool [n, E]: dropped iff u < p."""
    u, p = np.asarray(u, dtype=np.float64), np.asarray(p, dtype=np.float64)
    m = u < p
    nf = np.asarray(noise_free, dtype=bool)
    m[nf] = p[nf] == 1.0
    return m


def outlier_std_array(std) -> np.ndarray:
    """The offset standard deviations of eskf_set_meas_outliers: 7 finite values >= 0 (position 3, small body rotation 3,
    notch 1, in the units of cam_noise_std) as a float64 array.  Raises ``ValueError`` otherwise."""
    if std is None:
        raise ValueError("outlier_std (7 values) is required with outlier probabilities")
    s = np.asarray(std, dtype=np.float64)
    if s.shape != (7,):
        raise ValueError(f"outlier_std must have 7 entries (position 3, rotation 3, notch 1), not shape {s.shape}")
    if not (np.isfinite(s).all() and (s >= 0).all()):
        raise ValueError(f"outlier_std entries must be finite and >= 0, not {s.tolist()}")
    return np.ascontiguousarray(s)


def nis_gate_array(thr, n: int) -> np.ndarray:
    """The thresholds of eskf_set_innovation_gate: a scalar (every filter) or [n] (one per filter), each >= 0 and not NaN
    (+inf: never gated), as a C-contiguous float64 array of 1 or n entries.  Raises ``ValueError`` otherwise."""
    t = np.asarray(thr, dtype=np.float64)
    if t.ndim > 1 or (t.ndim == 1 and t.shape[0] not in (1, n)):
        raise ValueError(f"nis_gate must be a scalar or [{n}] (one threshold per filter), not of shape {t.shape}")
    if np.isnan(t).any() or (t < 0).any():
        raise ValueError("nis_gate thresholds must be >= 0 and not NaN (+inf switches a filter's gate off)")
    return np.ascontiguousarray(t.reshape(-1))


def segment_steps(n_prop, n_steps: int, e0: int, e1: int):
    """(k0, k1), each [n_traj]: the global steps at which every trajectory's epochs e0 and e1 start, as the kernels count
    them -- the running sum of n_prop with every epoch clamped to what is left of the n_steps-long stream (a negative entry
    counts 0).  A segment ``run(..., epochs=(e0, e1))`` executes steps [k0[t], k1[t]) of trajectory t and writes those
    trace rows.  ``n_prop`` is [E] or [n_traj, E]."""
    npr = np.atleast_2d(np.asarray(n_prop, dtype=np.int64))
    c = np.minimum(np.cumsum(np.maximum(npr, 0), axis=1), n_steps)  # the clamped running sum saturates at n_steps
    c = np.hstack((np.zeros((len(npr), 1), dtype=np.int64), c))
    return c[:, e0].copy(), c[:, e1].copy()


class BatchFilter:
    """N independent VI-ESKF instances resident on one GPU."""

    NX, NE, NM, NQ = 26, 24, 7, 13

    def __init__(self, n_filters: int, scope_length: float = 50.0, cam_angle_rad: float = np.deg2rad(30.0),
                 frozen_dofs: Sequence[int] = (1, 1, 1, 1, 1, 1), zero_frozen_dofs: bool = True, device: int = 0,
                 stream: int = 0, variant: Optional[int] = None):
        self._lib = _lib.load()
        self.n = int(n_filters)
        self.device = int(device)
        mask = 0
        for i, f in enumerate(frozen_dofs):
            if f:
                mask |= 1 << i
        m = EskfModel(float(scope_length), float(cam_angle_rad), mask, _lib.FLAG_ZERO_FROZEN if zero_frozen_dofs else 0)
        h = C.c_void_p()
        check(self._lib.eskf_create(C.byref(m), self.n, self.device, C.c_void_p(stream), C.byref(h)), "eskf_create")
        self._h = h
        self.last_carry = None  # carry returned by the last run(..., epochs=...)
        if variant is None:
            variant = int(os.environ.get("ESKF_B200_VARIANT", "0"))
        if variant:
            self.set_variant(variant)

    # -- lifetime -----------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._lib.eskf_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- state ------------------------------------------------------------------
    def set_state(self, x=None, P=None, u_old=None, R_old=None):
        """``Filter.__init__`` / ``Filter.reset`` (Filter.py:44-45,78-80,95-108).  Each array has leading
        dimension N or 1 (broadcast); ``R_old=None`` sets it to rot(q)."""
        ax, aP, au, aR = _Arg(x, 26, name="x"), _Arg(P, 576, name="P"), _Arg(u_old, 6, name="u_old"), _Arg(R_old, 9, name="R_old")
        mem = _common_mem([ax, aP, au, aR])
        check(self._lib.eskf_set_state(self._h, ax.ptr, ax.rows, aP.ptr, aP.rows, au.ptr, au.rows, aR.ptr, aR.rows, mem),
              "eskf_set_state")

    def set_noise(self, Qdiag=None, Rdiag=None, sigma_om=None):
        """``Filter.update_noise_matrices`` (Filter.py:110-117): diagonals of Q (13) and R (7), plus the
        gyro noise std the reference plugs into its Jacobians (Filter.py:330-331)."""
        aq, ar, as_ = _Arg(Qdiag, 13, name="Qdiag"), _Arg(Rdiag, 7, name="Rdiag"), _Arg(sigma_om, 3, name="sigma_om")
        mem = _common_mem([aq, ar, as_])
        check(self._lib.eskf_set_noise(self._h, aq.ptr, aq.rows, ar.ptr, ar.rows, as_.ptr, as_.rows, mem), "eskf_set_noise")

    def get_state(self, device: bool = False):
        """Returns (x [N,26], P [N,24,24], u_old [N,6], R_old [N,9], status [N])."""
        n = self.n
        if device:
            import torch

            dev = torch.device("cuda", self.device)
            x = torch.empty((n, 26), dtype=torch.float64, device=dev)
            P = torch.empty((n, 24, 24), dtype=torch.float64, device=dev)
            u = torch.empty((n, 6), dtype=torch.float64, device=dev)
            R = torch.empty((n, 9), dtype=torch.float64, device=dev)
            st = torch.empty((n,), dtype=torch.int32, device=dev)
            ptr = lambda t: C.c_void_p(t.data_ptr())
            check(self._lib.eskf_get_state(self._h, ptr(x), ptr(P), ptr(u), ptr(R), ptr(st), MEM_DEVICE), "eskf_get_state")
            return x, P, u, R, st
        x = np.empty((n, 26))
        P = np.empty((n, 24, 24))
        u = np.empty((n, 6))
        R = np.empty((n, 9))
        st = np.empty((n,), dtype=np.int32)
        ptr = lambda a: a.ctypes.data_as(C.c_void_p)
        check(self._lib.eskf_get_state(self._h, ptr(x), ptr(P), ptr(u), ptr(R), ptr(st), MEM_HOST), "eskf_get_state")
        return x, P, u, R, st

    # -- verbs -------------------------------------------------------------------
    def propagate(self, dt, om_acc):
        """T x ``Filter.propagate`` (Filter.py:219-230).  ``dt`` [T]; ``om_acc`` [T,6] shared by all
        filters or [N,T,6] per filter."""
        adt = _Arg(dt, None, name="dt")
        T = adt.rows
        aoa = _Arg(om_acc, 6 * T if T else None, name="om_acc")
        if T == 0:
            return
        if aoa.rows not in (1, self.n):
            raise ValueError("om_acc must be [T,6] or [N,T,6]")
        per = 1 if (aoa.rows == self.n and self.n > 1) else 0
        mem = _common_mem([adt, aoa])
        check(self._lib.eskf_propagate(self._h, adt.ptr, aoa.ptr, T, per, mem), "eskf_propagate")

    def update(self, cam, notch, want_gain: bool = False):
        """``Filter.update`` (Filter.py:351-395).  ``cam`` [7] / [N,7] = position + raw quaternion xyzw,
        ``notch`` scalar / [N].  Returns K [N,24,7] if ``want_gain``."""
        ac = _Arg(cam, 7, name="cam")
        an = _Arg(np.atleast_1d(notch) if not _is_torch(notch) else notch, 1, name="notch")
        if ac.rows != an.rows or ac.rows not in (1, self.n):
            raise ValueError("cam must be [7] or [N,7] with matching notch")
        per = 1 if (ac.rows == self.n and self.n > 1) else 0
        mem = _common_mem([ac, an])
        K = None
        kp = None
        if want_gain:
            if mem == MEM_DEVICE:
                import torch

                K = torch.empty((self.n, 24, 7), dtype=torch.float64, device=torch.device("cuda", self.device))
                kp = C.c_void_p(K.data_ptr())
            else:
                K = np.empty((self.n, 24, 7))
                kp = K.ctypes.data_as(C.c_void_p)
        check(self._lib.eskf_update(self._h, ac.ptr, an.ptr, per, kp, mem), "eskf_update")
        return K

    def run(self, dt, om_acc, n_prop, cam, notch, cam_ref=None, imu_ref=None, gt_dofs=(0, 0, 0, 0, 0, 20.0),
            n_traj: int = 1, filters_per_traj: Optional[int] = None, seed: int = 0, filter_id0: int = 0,
            imu_noise_std=None, cam_noise_std=None, noise_free_filter0: bool = True, want_stats: bool = True,
            stats_on_device: bool = False, trace=None, noise_id_modulus: int = 0, epochs=None, carry=None, drop_prob=None,
            nis_gate=None, outlier_prob=None, outlier_std=None):
        """``Filter.run`` (Filter.py:144-185) for every filter, in one persistent kernel.
        Returns (stats [N,16], stats_sum [16]) (see include/eskf.h) or None.
        ``trace``: optional [N,T,26] float64 array (numpy for host streams, CUDA tensor for device streams) that
        receives the nominal state after every IMU step, updated state at the update instants (FilterTraj rows).
        ``noise_id_modulus`` r > 0: the noise of global filter g is that of id g % r (common random numbers for
        groups of r filters that differ only by their parameters).
        ``epochs = (e0, e1)``: only epochs [e0, e1) of the trajectory passed (the whole one, not a slice), continuing from the
        current state (eskf_run_epochs, include/eskf.h); returns (stats, stats_sum, carry), stats over epochs [0, e1), None
        without ``want_stats`` and for an empty range (which runs nothing).  ``carry`` [N,4] (the running update-MSE sums, applied updates and status word) comes
        from the previous segment's return value, None to start fresh; it and the returned one live where the statistics
        do (numpy, or CUDA tensors with ``stats_on_device``), and the returned one is also kept as ``last_carry``.  Segments
        run back to back give bit for bit what one run gives; a checkpoint is ``get_state()``, the carry and e1.
        ``drop_prob``: simulated frame loss (``set_meas_dropout``): a scalar, [E] or [n_traj, E] (numpy, or a CUDA tensor) of
        per-epoch probabilities that a filter loses the camera measurement; None runs without dropout.
        ``nis_gate``: the innovation gate (``set_innovation_gate``): a scalar or [N] NIS threshold; an update whose NIS exceeds
        it is rejected.  ``outlier_prob`` / ``outlier_std``: simulated outlier frames (``set_meas_outliers``): a scalar, [E] or
        [n_traj, E] of per-epoch probabilities and the 7 offset standard deviations.  None runs without either."""
        adt = _Arg(dt, None, name="dt")
        anp = _Arg(n_prop, None, dtype=np.int32, name="n_prop")
        T = adt.rows // n_traj
        E = anp.rows // n_traj
        aoa, acm, ano = _Arg(om_acc, 6, name="om_acc"), _Arg(cam, 7, name="cam"), _Arg(notch, 1, name="notch")
        acr, air = _Arg(cam_ref, 6, name="cam_ref"), _Arg(imu_ref, 6, name="imu_ref")
        if aoa.rows != n_traj * T or acm.rows != n_traj * E or ano.rows != n_traj * E:
            raise ValueError("stream shapes do not match (n_traj, T, E)")
        mem = _common_mem([adt, anp, aoa, acm, ano, acr, air])
        check_run_geometry(self.n, n_traj, int(filters_per_traj if filters_per_traj else self.n), int(filter_id0), T, E,
                           n_prop if isinstance(n_prop, np.ndarray) else None, epochs)
        s = EskfStreams()
        s.n_steps, s.n_epochs, s.n_traj, s.mem = T, E, n_traj, mem
        s.filters_per_traj = int(filters_per_traj if filters_per_traj else self.n)
        s.dt, s.om_acc, s.n_prop, s.cam, s.notch = adt.ptr, aoa.ptr, anp.ptr, acm.ptr, ano.ptr
        s.cam_ref, s.imu_ref = acr.ptr, air.ptr
        s.gt_dofs = (C.c_double * 6)(*[float(v) for v in gt_dofs])
        s.seed, s.filter_id0 = int(seed), int(filter_id0)
        s.imu_noise_std = (C.c_double * 6)(*([0.0] * 6 if imu_noise_std is None else [float(v) for v in imu_noise_std]))
        s.cam_noise_std = (C.c_double * 7)(*([0.0] * 7 if cam_noise_std is None else [float(v) for v in cam_noise_std]))
        s.noise_free_filter0 = 1 if noise_free_filter0 else 0
        s.noise_id_modulus = int(noise_id_modulus)
        if trace is not None:
            if tuple(trace.shape) != (self.n, T, 26):
                raise ValueError(f"trace must have shape {(self.n, T, 26)}")
            if isinstance(trace, np.ndarray) and not (trace.flags.c_contiguous and trace.dtype == np.float64):
                raise TypeError("trace must be a C-contiguous float64 array (it is written in place)")
            atr = _Arg(trace.reshape(self.n * T, 26), 26, name="trace")
            if atr.mem != mem:
                raise ValueError("trace must live where the streams live (host numpy / CUDA tensor)")
            s.trace_x = atr.ptr
        self.set_meas_dropout(drop_prob, n_traj, E)
        self.set_innovation_gate(nis_gate)
        self.set_meas_outliers(outlier_prob, outlier_std, n_traj, E)
        if epochs is not None:
            return self._run_epochs(s, int(epochs[0]), int(epochs[1]), carry, want_stats, stats_on_device)
        if not want_stats:
            check(self._lib.eskf_run(self._h, C.byref(s), None, None, MEM_HOST), "eskf_run")
            return None
        if stats_on_device:
            import torch

            dev = torch.device("cuda", self.device)
            st = torch.empty((self.n, NSTAT), dtype=torch.float64, device=dev)
            sm = torch.empty((NSTAT,), dtype=torch.float64, device=dev)
            check(self._lib.eskf_run(self._h, C.byref(s), C.c_void_p(st.data_ptr()), C.c_void_p(sm.data_ptr()), MEM_DEVICE),
                  "eskf_run")
            return st, sm
        st = np.empty((self.n, NSTAT))
        sm = np.empty((NSTAT,))
        check(self._lib.eskf_run(self._h, C.byref(s), st.ctypes.data_as(C.c_void_p), sm.ctypes.data_as(C.c_void_p), MEM_HOST),
              "eskf_run")
        return st, sm

    def _run_epochs(self, s, e0: int, e1: int, carry, want_stats: bool, on_device: bool):
        """eskf_run_epochs with the streams ``s``: (stats, stats_sum, carry) in host or device memory"""
        if on_device:
            import torch

            dev = torch.device("cuda", self.device)
            new = lambda shape: torch.empty(shape, dtype=torch.float64, device=dev)
            ptr = lambda a: C.c_void_p(a.data_ptr())
            mem = MEM_DEVICE
            if carry is not None:
                carry = torch.as_tensor(carry, dtype=torch.float64, device=dev).contiguous()
        else:
            new, ptr, mem = np.empty, (lambda a: a.ctypes.data_as(C.c_void_p)), MEM_HOST
            if carry is not None:
                carry = np.ascontiguousarray(carry.cpu().numpy() if _is_torch(carry) else carry, dtype=np.float64)
        if carry is not None and tuple(carry.shape) != (self.n, NCARRY):
            raise ValueError(f"carry must have shape {(self.n, NCARRY)}")
        st, sm = (new((self.n, NSTAT)), new((NSTAT,))) if want_stats and e1 > e0 else (None, None)  # (empty: not written)
        out = new((self.n, NCARRY))
        arg = lambda a: None if a is None else ptr(a)
        check(self._lib.eskf_run_epochs(self._h, C.byref(s), e0, e1, arg(carry), ptr(out), arg(st), arg(sm), mem), "eskf_run_epochs")
        self.last_carry = out
        return st, sm, out

    def run_segments(self, dt, om_acc, n_prop, cam, notch, boundaries, carry=None, **kw):
        """Generator: the trajectory in segments [boundaries[i], boundaries[i + 1]) (``run`` with ``epochs``), yielding
        (e0, e1, stats, stats_sum) after each one, the carry threaded from one to the next (``last_carry`` holds the latest:
        with ``get_state()`` and e1 it is the checkpoint to continue from).  The caller may inspect the state, checkpoint or
        stop between segments; a generator that is not resumed runs nothing more, so the handle keeps the state of the last
        finished segment.  ``kw`` are the keyword arguments of ``run``."""
        b = [int(v) for v in boundaries]
        if len(b) < 2 or any(x > y for x, y in zip(b, b[1:])):
            raise ValueError("boundaries must be at least two non-decreasing epoch indices")
        for e0, e1 in zip(b, b[1:]):
            st, sm, carry = self.run(dt, om_acc, n_prop, cam, notch, epochs=(e0, e1), carry=carry, **kw)
            yield e0, e1, st, sm

    def set_meas_dropout(self, prob, n_traj: int = 1, n_epochs: Optional[int] = None):
        """Simulated frame loss of every later ``run`` (eskf_set_meas_dropout, include/eskf.h): filter g loses the camera
        measurement of epoch e with probability prob[trajectory, e], decided on the device from the run's seed and the
        filter's noise id (``dropout_mask`` gives the mask).  ``prob``: a scalar, [n_epochs] or [n_traj, n_epochs] (numpy, or a
        CUDA tensor), broadcast to [n_traj, n_epochs] (the streams' shape, which a run checks); None switches it off."""
        if prob is None:
            check(self._lib.eskf_set_meas_dropout(self._h, None, 0, 0, MEM_HOST), "eskf_set_meas_dropout")
            return
        if n_epochs is None:
            if np.ndim(prob) == 0:
                raise ValueError("n_epochs is needed for a scalar probability")
            n_epochs = int(prob.shape[-1]) if _is_torch(prob) else np.shape(prob)[-1]
        if _is_torch(prob) and prob.is_cuda:
            import torch

            drop_prob_array(prob.detach().cpu().numpy(), n_traj, n_epochs)  # (the shape and value checks, on a host copy)
            t = torch.broadcast_to(prob.to(torch.float64), (n_traj, n_epochs)).contiguous()
            check(self._lib.eskf_set_meas_dropout(self._h, C.c_void_p(t.data_ptr()), n_traj, n_epochs, MEM_DEVICE),
                  "eskf_set_meas_dropout")
            return
        p = drop_prob_array(prob.numpy() if _is_torch(prob) else prob, n_traj, n_epochs)
        check(self._lib.eskf_set_meas_dropout(self._h, p.ctypes.data_as(C.c_void_p), n_traj, n_epochs, MEM_HOST),
              "eskf_set_meas_dropout")

    def set_innovation_gate(self, thr):
        """Innovation gate of every later ``run`` (eskf_set_innovation_gate, include/eskf.h): an update whose residual is
        valid and whose NIS r^T inv(S) r exceeds the filter's threshold is rejected (state and covariance stay at the
        prior, no status bit).  ``thr``: a scalar or [N] (numpy, or a CUDA tensor), each >= 0 and not NaN, +inf never
        gates; None switches the gate off."""
        if thr is None:
            check(self._lib.eskf_set_innovation_gate(self._h, None, 0, MEM_HOST), "eskf_set_innovation_gate")
            return
        if _is_torch(thr) and thr.is_cuda:
            import torch

            nis_gate_array(thr.detach().cpu().numpy(), self.n)  # (the shape and value checks, on a host copy)
            t = thr.to(torch.float64).reshape(-1).contiguous()
            check(self._lib.eskf_set_innovation_gate(self._h, C.c_void_p(t.data_ptr()), int(t.numel()), MEM_DEVICE),
                  "eskf_set_innovation_gate")
            return
        t = nis_gate_array(thr.numpy() if _is_torch(thr) else thr, self.n)
        check(self._lib.eskf_set_innovation_gate(self._h, t.ctypes.data_as(C.c_void_p), int(t.size), MEM_HOST),
              "eskf_set_innovation_gate")

    def set_meas_outliers(self, prob, std=None, n_traj: int = 1, n_epochs: Optional[int] = None):
        """Simulated outlier frames of every later ``run`` (eskf_set_meas_outliers, include/eskf.h): filter g's camera
        measurement of epoch e is offset with probability prob[trajectory, e] by std * z (z standard normals drawn on the
        device from the run's seed and the filter's noise id; ``outlier_mask`` gives the mask).  ``prob`` as for
        ``set_meas_dropout``; ``std`` 7 values >= 0 (position 3, small body rotation 3, notch 1); None switches it off."""
        if prob is None:
            check(self._lib.eskf_set_meas_outliers(self._h, None, 0, 0, None, MEM_HOST), "eskf_set_meas_outliers")
            return
        sd = outlier_std_array(std)
        if n_epochs is None:
            if np.ndim(prob) == 0:
                raise ValueError("n_epochs is needed for a scalar probability")
            n_epochs = int(prob.shape[-1]) if _is_torch(prob) else np.shape(prob)[-1]
        sdp = sd.ctypes.data_as(C.c_void_p)
        if _is_torch(prob) and prob.is_cuda:
            import torch

            drop_prob_array(prob.detach().cpu().numpy(), n_traj, n_epochs, "outlier_prob")  # (the checks, on a host copy)
            t = torch.broadcast_to(prob.to(torch.float64), (n_traj, n_epochs)).contiguous()
            check(self._lib.eskf_set_meas_outliers(self._h, C.c_void_p(t.data_ptr()), n_traj, n_epochs, sdp, MEM_DEVICE),
                  "eskf_set_meas_outliers")
            return
        p = drop_prob_array(prob.numpy() if _is_torch(prob) else prob, n_traj, n_epochs, "outlier_prob")
        check(self._lib.eskf_set_meas_outliers(self._h, p.ctypes.data_as(C.c_void_p), n_traj, n_epochs, sdp, MEM_HOST),
              "eskf_set_meas_outliers")

    def sync(self):
        check(self._lib.eskf_sync(self._h), "eskf_sync")

    @property
    def launch_count(self) -> int:
        return int(self._lib.eskf_launch_count(self._h))

    def set_tuning(self, filters_per_cta: int = 0):
        check(self._lib.eskf_set_tuning(self._h, int(filters_per_cta)), "eskf_set_tuning")

    def keep_jacobians(self, on: bool = True):
        """The kernels file the Jacobian record of the last IMU step of every ``propagate`` / ``run`` (eskf_keep_jacobians)."""
        check(self._lib.eskf_keep_jacobians(self._h, 1 if on else 0), "eskf_keep_jacobians")

    def get_jacobians(self):
        """``Filter.Fx`` [N,24,24] and ``Filter.Fi`` [N,24,13] of the last IMU step (Filter.py:249-342), dense, as numpy
        arrays; needs ``keep_jacobians()`` before the propagation."""
        Fx, Fi = np.empty((self.n, 24, 24)), np.empty((self.n, 24, 13))
        check(self._lib.eskf_get_jacobians(self._h, Fx.ctypes.data_as(C.c_void_p), Fi.ctypes.data_as(C.c_void_p), MEM_HOST),
              "eskf_get_jacobians")
        return Fx, Fi

    def keep_consistency(self, on: bool = True):
        """Every later ``run`` files the NIS of each filter's updates and the NEES of its estimated DOFs after them
        (eskf_keep_consistency, include/eskf.h); read them with ``get_consistency``.  Runs the export instantiation of the
        persistent kernel and needs N * E * 368 bytes of device memory; default kernel only."""
        check(self._lib.eskf_keep_consistency(self._h, 1 if on else 0), "eskf_keep_consistency")

    def get_consistency(self, device: bool = False):
        """(nis [N,E], nees [N,E], epoch_sum [E,8]) of the last ``run`` since ``keep_consistency()``: NaN where the update was
        not applied or the value is not finite; epoch_sum holds per epoch the count, sum and sum of squares of the finite NIS
        ([0:3]) and NEES ([3:6]) and the number of filters with a NaN ([6]).  numpy arrays, or CUDA tensors with ``device``."""
        E = C.c_int64()
        check(self._lib.eskf_get_consistency(self._h, None, None, None, C.byref(E), MEM_HOST), "eskf_get_consistency")
        E = int(E.value)
        if device:
            import torch

            dev = torch.device("cuda", self.device)
            out = [torch.empty(shape, dtype=torch.float64, device=dev) for shape in ((self.n, E), (self.n, E), (E, NCONS))]
            ptrs, mem = [C.c_void_p(t.data_ptr()) for t in out], MEM_DEVICE
        else:
            out = [np.empty(shape) for shape in ((self.n, E), (self.n, E), (E, NCONS))]
            ptrs, mem = [a.ctypes.data_as(C.c_void_p) for a in out], MEM_HOST
        check(self._lib.eskf_get_consistency(self._h, *ptrs, None, mem), "eskf_get_consistency")
        if device:
            self.sync()  # (the copies ran on the handle's stream)
        return tuple(out)

    def _cons_outputs(self, fn, name, shapes, device):
        """arrays of ``shapes(E)`` filled by the consistency getter ``fn(h, *ptrs, n_epochs, mem)`` (E queried first)"""
        E = C.c_int64()
        check(fn(self._h, *([None] * len(shapes(0))), C.byref(E), MEM_HOST), name)
        E = int(E.value)
        if device:
            import torch

            dev = torch.device("cuda", self.device)
            out = [torch.empty(shape, dtype=torch.float64, device=dev) for shape in shapes(E)]
            ptrs, mem = [C.c_void_p(t.data_ptr()) for t in out], MEM_DEVICE
        else:
            out = [np.empty(shape) for shape in shapes(E)]
            ptrs, mem = [a.ctypes.data_as(C.c_void_p) for a in out], MEM_HOST
        check(fn(self._h, *ptrs, None, mem), name)
        if device:
            self.sync()  # (the kernels and copies ran on the handle's stream)
        return out

    def get_dof_history(self, device: bool = False):
        """(dofs [N,E,6], var [N,E,6]) of the last ``run`` since ``keep_consistency()`` (eskf_get_dof_history,
        include/eskf.h): every filter's calibration DOFs x[10:16] after each epoch's update, as the consistency records hold
        them (before it where the update was not applied: nis NaN), and the diagonal of the DOF covariance block at the same
        instant.  numpy arrays, or CUDA tensors with ``device``."""
        return tuple(self._cons_outputs(self._lib.eskf_get_dof_history, "eskf_get_dof_history",
                                        lambda E: ((self.n, E, 6), (self.n, E, 6)), device))

    def get_dof_envelope(self, device: bool = False):
        """dof_sum [E, 80] of the last ``run`` since ``keep_consistency()`` (eskf_get_dof_envelope, include/eskf.h): per
        epoch, sums over this handle's contributing filters of the DOF errors, their squares, the filter variances, the
        normalised squared errors, the 1 / 2 / 3 sigma coverage counts and the pair products, for
        ``consistency.summarise_dofs``.  Computed from the records on every call; shards add their sums.  numpy array, or
        CUDA tensor with ``device``."""
        return self._cons_outputs(self._lib.eskf_get_dof_envelope, "eskf_get_dof_envelope", lambda E: ((E, NDOFSUM),), device)[0]

    def set_groups(self, group_size: int):
        """Filter groups of the next ``run`` (eskf_set_groups, include/eskf.h): filter f of a handle whose run has
        ``filter_id0 = id0`` belongs to global group ``(id0 + f) // group_size``; ``group_size = filters_per_traj`` gives one
        group per trajectory, ``noise_id_modulus`` one per tuning candidate; 0 (the default) is one group, the whole
        handle.  A run with groups also reduces its statistics rows per group (``get_group_sums``)."""
        if isinstance(group_size, bool) or int(group_size) != group_size:
            raise TypeError(f"group_size must be an integer, not {group_size!r}")
        if group_size < 0:
            raise ValueError(f"group_size must be 0 (no groups) or positive, not {group_size}")
        check(self._lib.eskf_set_groups(self._h, int(group_size)), "eskf_set_groups")

    def get_group_sums(self, stats: bool = True, consistency: bool = False, dof_envelope: bool = False, device: bool = False):
        """(group0, stats_sum [G,16], epoch_sum [G,E,8], dof_sum [G,E,80]) of the last ``run`` (eskf_get_group_sums,
        include/eskf.h): row k is global group ``group0 + k``, with the layout and meaning of ``run``'s ``stats_sum``,
        ``get_consistency``'s ``epoch_sum`` and ``get_dof_envelope``'s ``dof_sum``.  Each array is None unless asked for;
        ``stats`` needs a run with statistics and groups, ``consistency`` / ``dof_envelope`` the records of a run since
        ``keep_consistency()``.  numpy arrays, or CUDA tensors with ``device``.  A shard's rows go into the job's with
        ``sharding.place_group_rows``."""
        g0, G, E = C.c_int64(), C.c_int64(), C.c_int64()
        fn = self._lib.eskf_get_group_sums
        check(fn(self._h, None, None, None, C.byref(g0), C.byref(G), C.byref(E), MEM_HOST), "eskf_get_group_sums")
        G, E = int(G.value), int(E.value)
        shapes = ((G, NSTAT) if stats else None, (G, E, NCONS) if consistency else None,
                  (G, E, NDOFSUM) if dof_envelope else None)
        if device:
            import torch

            dev = torch.device("cuda", self.device)
            out = [None if s is None else torch.empty(s, dtype=torch.float64, device=dev) for s in shapes]
            ptrs, mem = [None if t is None else C.c_void_p(t.data_ptr()) for t in out], MEM_DEVICE
        else:
            out = [None if s is None else np.empty(s) for s in shapes]
            ptrs, mem = [None if a is None else a.ctypes.data_as(C.c_void_p) for a in out], MEM_HOST
        check(fn(self._h, *ptrs, None, None, None, mem), "eskf_get_group_sums")
        if device:
            self.sync()  # (the kernels and copies ran on the handle's stream)
        return (int(g0.value), *out)

    def set_prepass_budget(self, n_bytes: int):
        """Memory ``run`` may use to keep the Monte-Carlo generator and the update-MSE statistics out of the persistent kernel
        (include/eskf.h, eskf_set_prepass_budget); 0 = everything inside the kernel.  Both ways give the same bits."""
        check(self._lib.eskf_set_prepass_budget(self._h, int(n_bytes)), "eskf_set_prepass_budget")

    def set_variant(self, variant: int = 0):
        """0 = default kernel (warp-specialised eskf_kernel3), 1 = first kernel (eskf_kernel), 3 = eskf_kernel3."""
        check(self._lib.eskf_set_variant(self._h, int(variant)), "eskf_set_variant")


NOISE_IMU, NOISE_CAM, NOISE_DROP, NOISE_OUTLIER = 1, 2, 3, 4


def noise_samples(seed: int, filter_id0: int, n_filters: int, step0: int, n_steps: int, kind: int, device: int = 0):
    """The standard normals ``eskf_run`` draws (see include/eskf.h, eskf_noise_dump): array [n_filters, n_steps, 8]."""
    lib = _lib.load()
    out = np.empty((n_filters, n_steps, 8))
    check(lib.eskf_noise_dump(int(device), None, int(seed), int(filter_id0), int(n_filters), int(step0), int(n_steps), int(kind),
                              out.ctypes.data_as(C.c_void_p), MEM_HOST), "eskf_noise_dump")
    return out


def dropout_mask(prob, seed: int, filter_id0: int, n_filters: int, epochs, n_traj: int = 1, filters_per_traj: Optional[int] = None,
                 noise_id_modulus: int = 0, noise_free_filter0: bool = True, device: int = 0) -> np.ndarray:
    """bool [n_filters, e1 - e0]: which of global epochs ``epochs = (e0, e1)`` filters ``filter_id0 ..`` lose in a run with
    ``drop_prob = prob`` (a scalar, [E] or [n_traj, E]) and these run arguments, from the uniforms the device draws
    (``eskf_noise_dump`` with ESKF_NOISE_DROP: the definition of the draw)."""
    e0, e1 = (int(v) for v in epochs)
    E = int(np.shape(prob)[-1]) if np.ndim(prob) else e1
    p = drop_prob_array(prob, n_traj, E)
    if not 0 <= e0 <= e1 <= E:
        raise ValueError(f"epochs [{e0}, {e1}) is not within [0, {E}]")
    g = int(filter_id0) + np.arange(int(n_filters))
    traj = g // int(filters_per_traj or n_filters) if n_traj > 1 else np.zeros_like(g)
    gid = g % noise_id_modulus if noise_id_modulus > 0 else g
    if e1 == e0:
        return np.zeros((len(g), 0), dtype=bool)
    lo = int(gid.min())
    u = noise_samples(seed, lo, int(gid.max()) - lo + 1, e0, e1 - e0, NOISE_DROP, device)[:, :, 0]
    return mask_from_uniforms(u[gid - lo], p[traj, e0:e1], (gid == 0) & bool(noise_free_filter0))


def outlier_mask(prob, seed: int, filter_id0: int, n_filters: int, epochs, n_traj: int = 1, filters_per_traj: Optional[int] = None,
                 noise_id_modulus: int = 0, noise_free_filter0: bool = True, device: int = 0):
    """(mask bool [n_filters, e1 - e0], offsets [n_filters, e1 - e0, 7]): which of global epochs ``epochs = (e0, e1)`` of
    filters ``filter_id0 ..`` are outliers in a run with ``outlier_prob = prob`` (a scalar, [E] or [n_traj, E]) and these run
    arguments, and the standard normals of their offsets (scale them by ``outlier_std``), from the draws of the device
    (``eskf_noise_dump`` with ESKF_NOISE_OUTLIER: the definition).  The noise-free reference filter is never corrupted."""
    e0, e1 = (int(v) for v in epochs)
    E = int(np.shape(prob)[-1]) if np.ndim(prob) else e1
    p = drop_prob_array(prob, n_traj, E, "outlier_prob")
    if not 0 <= e0 <= e1 <= E:
        raise ValueError(f"epochs [{e0}, {e1}) is not within [0, {E}]")
    g = int(filter_id0) + np.arange(int(n_filters))
    traj = g // int(filters_per_traj or n_filters) if n_traj > 1 else np.zeros_like(g)
    gid = g % noise_id_modulus if noise_id_modulus > 0 else g
    if e1 == e0:
        return np.zeros((len(g), 0), dtype=bool), np.zeros((len(g), 0, 7))
    lo = int(gid.min())
    d = noise_samples(seed, lo, int(gid.max()) - lo + 1, e0, e1 - e0, NOISE_OUTLIER, device)[gid - lo]
    nf = (gid == 0) & bool(noise_free_filter0)
    m = mask_from_uniforms(d[:, :, 0], p[traj, e0:e1], np.zeros(len(g), dtype=bool))
    m[nf] = False  # (unlike a dropout, the noise-free reference filter is never corrupted, even at p = 1)
    return m, d[:, :, 1:8]


def fp64_peak_tflops(device: int = 0, repeats: int = 5) -> float:
    """Measured FP64 FMA throughput of the device (TFLOP/s): the roofline denominator of bench.py."""
    lib = _lib.load()
    out, ms = C.c_double(), C.c_double()
    check(lib.eskf_fp64_peak(int(device), None, int(repeats), C.byref(out), C.byref(ms)), "eskf_fp64_peak")
    return float(out.value)
