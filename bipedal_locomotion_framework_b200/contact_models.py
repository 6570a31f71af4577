"""Python mirror of the reference's interface for this path, computing ONLY through the C ABI.

Names and argument meaning follow the reference so the parity tests read like its own:
  StdImplementation           src/ParametersHandler/.../StdImplementation.h:27-236 (scalar subset)
  ContinuousContactModel      src/ContactModels/.../ContactModel.h:33-146 +
                              ContinuousContactModel.h:41-143 (per-instance facade, lazy getters)
  ContinuousContactModelBatch the batched entry point this build adds (SURVEY.md section 3.4)

The C++17 classes under cpp/ are the host layer a reference user links; this module exists for the
pytest / bench harness.  torch supplies device memory and streams (plumbing only).
"""
from __future__ import annotations

import ctypes as C
import os
import sys

import numpy as np

from . import _capi
from ._capi import AUTODYN, CTRL, FULL, REGRESSOR, WRENCH  # noqa: F401


# --------------------------------------------------------------------------------------------------
# parameters handler (host logic)
# --------------------------------------------------------------------------------------------------

class StdImplementation:
    """Key -> value store with the strict typing of std::any_cast
    (StdImplementation.tpp:21-42): a value set as int cannot be read as double."""

    def __init__(self):
        self._map: dict = {}

    def setParameter(self, name: str, value) -> None:
        self._map[name] = value

    def getParameter(self, name: str, kind: type):
        """Returns (ok, value).  Mirrors `bool getParameter(const std::string&, T&)`."""
        if name not in self._map:
            print(f"[StdImplementation::getParameterPrivate] Parameter named {name} not found.",
                  file=sys.stderr)
            return False, None
        v = self._map[name]
        if type(v) is not kind:
            print(f"[StdImplementation::getParameterPrivate] The type of the parameter named {name} "
                  "is different from the one expected", file=sys.stderr)
            return False, None
        return True, v

    def setGroup(self, name: str, group: "StdImplementation") -> bool:
        if not isinstance(group, StdImplementation):
            print("[StdImplementation::setGroup] Unable to downcast the pointer to "
                  "StdImplementation.", file=sys.stderr)
            return False
        self._map[name] = group
        return True

    def getGroup(self, name: str) -> "StdImplementation":
        g = self._map.get(name)
        return g if isinstance(g, StdImplementation) else StdImplementation()

    def set(self, obj: dict) -> None:
        self._map = dict(obj)

    def toString(self) -> str:
        return "".join(k + " " for k in self._map)

    def isEmpty(self) -> bool:
        return len(self._map) == 0

    def clear(self) -> None:
        self._map.clear()


_PARAM_KEYS = ("length", "width", "spring_coeff", "damper_coeff")


def _read_params(handler, who: str):
    """ContinuousContactModel.cpp:24-65: four required double keys, in this order."""
    if handler is None:
        print(f"[{who}::initialize] The parameter handler is corrupted. Please make sure that the "
              "handler exists.", file=sys.stderr)
        return None
    vals = []
    for key in _PARAM_KEYS:
        ok, v = handler.getParameter(key, float)
        if not ok:
            print(f"[{who}::initialize] Unable to get the variable named {key}.", file=sys.stderr)
            return None
        vals.append(v)
    return vals


# --------------------------------------------------------------------------------------------------
# handle
# --------------------------------------------------------------------------------------------------

class _Handle:
    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        _capi.check(_capi.lib().blf_ccm_create(int(device), C.byref(self._h)))
        self.device = int(device)

    def close(self):
        if self._h:
            _capi.lib().blf_ccm_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def ptr(self):
        return self._h

    def set_uniform_params(self, length, width, spring, damper):
        _capi.check(_capi.lib().blf_ccm_set_uniform_params(self._h, length, width, spring, damper))

    @property
    def launch_count(self) -> int:
        return int(_capi.lib().blf_ccm_launch_count(self._h))

    @property
    def last_path(self) -> int:
        return int(_capi.lib().blf_ccm_last_path(self._h))

    @property
    def sm_count(self) -> int:
        return int(_capi.lib().blf_ccm_sm_count(self._h))


class _CompressibleBuffer:
    """Owner of one blf_ccm_device_alloc_compressible allocation of float64s, exposed through
    __cuda_array_interface__.  A tensor made from it with torch.as_tensor holds a reference to it,
    and so does every view or slice of that tensor: the memory is freed (after a device
    synchronise, see blf_ccm_device_free) when the last of them goes away."""

    def __init__(self, handle: _Handle, shape):
        self._handle = handle            # the handle must outlive the allocation
        self.ptr = 0
        p, granted = C.c_void_p(), C.c_int()
        _capi.check(_capi.lib().blf_ccm_device_alloc_compressible(
            handle.ptr, 8 * int(np.prod(shape)), C.byref(p), C.byref(granted)))
        self.ptr = p.value or 0
        self.granted = bool(granted.value)
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<f8", "data": (self.ptr, False),
                                         "strides": None, "version": 3}

    def __del__(self):
        if self.ptr:
            try:
                _capi.lib().blf_ccm_device_free(self._handle.ptr, self.ptr)
            except Exception:
                pass
            self.ptr = 0


def _np_ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _ptr_array(ptrs):
    arr = (C.c_void_p * len(ptrs))(*[C.c_void_p(p) if p else None for p in ptrs])
    return arr


# --------------------------------------------------------------------------------------------------
# per-instance facade
# --------------------------------------------------------------------------------------------------

class ContinuousContactModel:
    """Per-instance facade with the reference's lazy-evaluation protocol; every compute* goes to
    the GPU through blf_ccm_eval_batch_host with n = 1."""

    def __init__(self, device: int = 0):
        self._handle = None
        self._device = device
        self._flags = {WRENCH: False, AUTODYN: False, CTRL: False, REGRESSOR: False}
        # ContinuousContactModel.cpp:16-22 and header defaults (:44-57)
        self._wrench = np.zeros(6)
        self._autodyn = np.zeros(6)
        self._ctrl = np.zeros(36)
        self._regressor = np.zeros(12)
        ident = np.concatenate([np.zeros(3), np.eye(3).reshape(9)])
        self._frame = ident.copy()
        self._null = ident.copy()
        self._twist = np.zeros(6)
        self._params = [0.0, 0.0, 0.0, 0.0]  # length, width, spring, damper
        self._params_dirty = True
        # one launch per state: all four outputs of the current state, tagged with the parameters
        # they were computed with (see cpp/.../ContinuousContactModel.h, m_all)
        self._all = {WRENCH: np.zeros(6), AUTODYN: np.zeros(6), CTRL: np.zeros(36),
                     REGRESSOR: np.zeros(12)}
        self._all_params = None

    def _invalidate(self):
        for k in self._flags:
            self._flags[k] = False
        self._all_params = None

    def initialize(self, handler) -> bool:
        self._invalidate()  # ContactModel.cpp:15-18: flags cleared before initializePrivate
        vals = _read_params(handler, "ContinuousContactModel")
        if vals is None:
            return False
        try:
            if self._handle is None:
                self._handle = _Handle(self._device)
        except (_capi.BlfCcmError, ImportError) as e:
            print(f"[ContinuousContactModel::initialize] CUDA backend unavailable: {e}",
                  file=sys.stderr)
            return False
        self._params = list(vals)
        self._params_dirty = True
        return True

    def setState(self, twist, transform) -> None:
        self._invalidate()
        self._twist = np.ascontiguousarray(twist, dtype=np.float64).reshape(6).copy()
        self._frame = np.ascontiguousarray(transform, dtype=np.float64).reshape(12).copy()

    def setNullForceTransform(self, transform) -> None:
        self._invalidate()
        self._null = np.ascontiguousarray(transform, dtype=np.float64).reshape(12).copy()

    def _compute(self, bit: int):
        if self._handle is None:
            raise RuntimeError("[ContinuousContactModel] initialize() must succeed before any getter "
                               "(there is no CPU path)")
        out = {WRENCH: self._wrench, AUTODYN: self._autodyn, CTRL: self._ctrl,
               REGRESSOR: self._regressor}
        if self._all_params != tuple(self._params):
            # first getter of this state (or the coefficients were written since): ONE evaluation
            # of all four outputs with the live parameters
            if self._params_dirty:
                self._handle.set_uniform_params(*self._params)
                self._params_dirty = False
            al = self._all
            _capi.check(_capi.lib().blf_ccm_eval_batch_host(
                self._handle.ptr, 1, _np_ptr(self._twist), _np_ptr(self._frame), _np_ptr(self._null),
                None, WRENCH | AUTODYN | CTRL | REGRESSOR, _np_ptr(al[WRENCH]), _np_ptr(al[AUTODYN]),
                _np_ptr(al[CTRL]), _np_ptr(al[REGRESSOR])))
            self._all_params = tuple(self._params)
        out[bit][:] = self._all[bit]
        self._flags[bit] = True

    def getContactWrench(self):
        if not self._flags[WRENCH]:
            self._compute(WRENCH)
        return self._wrench

    def getAutonomousDynamics(self):
        if not self._flags[AUTODYN]:
            self._compute(AUTODYN)
        return self._autodyn

    def getControlMatrix(self):
        if not self._flags[CTRL]:
            self._compute(CTRL)
        return self._ctrl.reshape(6, 6)

    def getRegressor(self):
        if not self._flags[REGRESSOR]:
            self._compute(REGRESSOR)
        return self._regressor.reshape(6, 2)

    def _points(self, xs, ys):
        import torch
        if self._handle is None:
            raise RuntimeError("[ContinuousContactModel] initialize() must succeed first")
        if self._params_dirty:
            self._handle.set_uniform_params(*self._params)
            self._params_dirty = False
        dev = torch.device("cuda", self._device)
        xy = torch.tensor(np.stack([np.atleast_1d(xs), np.atleast_1d(ys)], axis=1),
                          dtype=torch.float64, device=dev).contiguous()
        m = xy.shape[0]
        f = torch.empty((m, 3), dtype=torch.float64, device=dev)
        t = torch.empty((m, 3), dtype=torch.float64, device=dev)
        st = torch.cuda.current_stream(dev).cuda_stream
        _capi.check(_capi.lib().blf_ccm_eval_surface_points(
            self._handle.ptr, _np_ptr(self._twist), _np_ptr(self._frame), _np_ptr(self._null), m,
            xy.data_ptr(), f.data_ptr(), t.data_ptr(), st))
        return f.cpu().numpy(), t.cpu().numpy()

    def getForceAtPoint(self, x, y):
        return self._points(x, y)[0][0]

    def getTorqueGeneratedAtPoint(self, x, y):
        return self._points(x, y)[1][0]

    def surfacePointWrenches(self, xs, ys):
        """Batched form of the two calls above: (m,3) forces and torques in one launch."""
        return self._points(xs, ys)

    # ContinuousContactModel.cpp:256-274 -- mutable access that does NOT clear the lazy flags
    @property
    def springCoeff(self):
        return self._params[2]

    @springCoeff.setter
    def springCoeff(self, v):
        self._params[2] = float(v)
        self._params_dirty = True

    @property
    def damperCoeff(self):
        return self._params[3]

    @damperCoeff.setter
    def damperCoeff(self, v):
        self._params[3] = float(v)
        self._params_dirty = True


# --------------------------------------------------------------------------------------------------
# batched entry point
# --------------------------------------------------------------------------------------------------

class ContinuousContactModelBatch:
    """Batched evaluation on one GPU.  Inputs/outputs are torch CUDA tensors (float64) or, for
    evaluate_host, numpy arrays; all arithmetic happens in libblf_ccm.so."""

    def __init__(self, device: int = 0):
        import torch
        self._torch = torch
        self.device = torch.device("cuda", device)
        self._handle = _Handle(device)

    @property
    def handle(self) -> _Handle:
        return self._handle

    def initialize(self, handler) -> bool:
        vals = _read_params(handler, "ContinuousContactModelBatch")
        if vals is None:
            return False
        self._handle.set_uniform_params(*vals)
        return True

    def set_uniform_params(self, length, width, spring, damper):
        self._handle.set_uniform_params(float(length), float(width), float(spring), float(damper))

    def load_parameter_table(self, handler):
        """Per-contact parameter table (four equally long float lists, e.g. a group of a `.ini`
        file read with ini.load_ini_file) -> (4, n) device planes for `param_planes`; None (and a
        message) when a key is missing, mistyped or of a different length."""
        from .ini import parameter_table
        t = parameter_table(handler)
        return None if t is None else self._torch.from_numpy(t).to(self.device)

    def _stream(self):
        return self._torch.cuda.current_stream(self.device).cuda_stream

    def alloc_ctrl(self, n: int):
        """(n, 36) float64 device tensor for the dense control matrix, in compressible memory where
        the device supports it (blf_ccm_device_alloc_compressible): 24 of the 36 entries are
        structural +0.0, so the hardware moves fewer bytes to and from HBM; the values are the
        ones written.  BLF_CCM_TUNE_NO_COMPRESS=1 gives a plain torch.empty tensor."""
        t = self._torch
        if n == 0 or os.environ.get("BLF_CCM_TUNE_NO_COMPRESS", "0") not in ("", "0"):
            return t.empty((n, 36), dtype=t.float64, device=self.device)
        return t.as_tensor(_CompressibleBuffer(self._handle, (n, 36)), device=self.device)

    def is_compressible(self, tensor) -> bool:
        """True when the tensor's memory lies in a compressible allocation of this batch's handle."""
        out = C.c_int()
        _capi.check(_capi.lib().blf_ccm_pointer_is_compressible(self._handle.ptr, tensor.data_ptr(),
                                                                C.byref(out)))
        return bool(out.value)

    def alloc_soa_outputs(self, n: int, mask: int) -> dict:
        t = self._torch
        mk = lambda *s: t.empty(s, dtype=t.float64, device=self.device)
        return {
            "wrench": mk(6, n) if mask & WRENCH else None,
            "autodyn": mk(6, n) if mask & AUTODYN else None,
            "ctrl": self.alloc_ctrl(n) if mask & CTRL else None,
            "regressor": mk(12, n) if mask & REGRESSOR else None,
        }

    def alloc_aos_outputs(self, n: int, mask: int) -> dict:
        t = self._torch
        mk = lambda *s: t.empty(s, dtype=t.float64, device=self.device)
        return {
            "wrench": mk(n, 6) if mask & WRENCH else None,
            "autodyn": mk(n, 6) if mask & AUTODYN else None,
            "ctrl": self.alloc_ctrl(n) if mask & CTRL else None,
            "regressor": mk(n, 12) if mask & REGRESSOR else None,
        }

    @staticmethod
    def _plane_ptrs(t, count):
        """2-D (count, n) tensor with unit inner stride, or a list of 1-D tensors / None."""
        if t is None:
            return None
        if isinstance(t, (list, tuple)):
            assert len(t) == count
            return _ptr_array([None if p is None else p.data_ptr() for p in t])
        assert t.shape[0] == count and (t.shape[1] <= 1 or t.stride(1) == 1)
        return _ptr_array([t[i].data_ptr() for i in range(count)])

    @staticmethod
    def _num_contacts(planes):
        if isinstance(planes, (list, tuple)):
            return next(p for p in planes if p is not None).shape[0]
        return planes.shape[1]

    def evaluate_soa(self, planes, param_planes=None, mask: int = FULL, out: dict | None = None):
        """planes: (30, n) float64 CUDA tensor (rows may be views with their own alignment), or a
        list of 30 1-D tensors where dead planes may be None."""
        n = self._num_contacts(planes)
        out = out if out is not None else self.alloc_soa_outputs(n, mask)
        inp = self._plane_ptrs(planes, 30)
        prm = self._plane_ptrs(param_planes, 4)
        _capi.check(_capi.lib().blf_ccm_eval_batch_soa(
            self._handle.ptr, n, inp, prm, mask,
            self._plane_ptrs(out["wrench"], 6), self._plane_ptrs(out["autodyn"], 6),
            out["ctrl"].data_ptr() if out["ctrl"] is not None else None,
            self._plane_ptrs(out["regressor"], 12), self._stream()))
        return out

    def prepare_soa(self, planes, param_planes=None, mask: int = FULL, out: dict | None = None):
        """Bind every argument of blf_ccm_eval_batch_soa once; the returned callable is a single
        foreign call (a few microseconds of host time), for launch-rate-sensitive loops.
        Returns (call, out)."""
        n = self._num_contacts(planes)
        out = out if out is not None else self.alloc_soa_outputs(n, mask)
        args = (self._handle.ptr, n, self._plane_ptrs(planes, 30), self._plane_ptrs(param_planes, 4),
                mask, self._plane_ptrs(out["wrench"], 6), self._plane_ptrs(out["autodyn"], 6),
                out["ctrl"].data_ptr() if out["ctrl"] is not None else None,
                self._plane_ptrs(out["regressor"], 12), self._stream())
        fn = _capi.lib().blf_ccm_eval_batch_soa
        keep = (planes, param_planes, out)

        def call(_keep=keep):
            rc = fn(*args)
            if rc:
                _capi.check(rc)
        return call, out

    def prepare_aos(self, twists, poses, null_poses, params=None, mask: int = FULL,
                    out: dict | None = None):
        n = poses.shape[0]
        out = out if out is not None else self.alloc_aos_outputs(n, mask)
        dp = lambda t: t.data_ptr() if t is not None else None
        args = (self._handle.ptr, n, dp(twists), dp(poses), dp(null_poses), dp(params), mask,
                dp(out["wrench"]), dp(out["autodyn"]), dp(out["ctrl"]), dp(out["regressor"]),
                self._stream())
        fn = _capi.lib().blf_ccm_eval_batch_aos
        keep = (twists, poses, null_poses, params, out)

        def call(_keep=keep):
            rc = fn(*args)
            if rc:
                _capi.check(rc)
        return call, out

    def prepare_rollout(self, planes, rollout_len: int, wrench_ref, weights, param_planes=None,
                        mask: int = 0, index_base: int = 0, out: dict | None = None,
                        want_cost: bool = True):
        """Prepared form of rollout_cost_argmin.  Returns (call, out, cost, best)."""
        t = self._torch
        n = self._num_contacts(planes)
        assert n % rollout_len == 0
        n_rollouts = n // rollout_len
        out = out if out is not None else self.alloc_soa_outputs(n, mask)
        cost = t.empty(n_rollouts, dtype=t.float64, device=self.device) if want_cost else None
        best = t.empty(2, dtype=t.int64, device=self.device)
        ref = np.ascontiguousarray(wrench_ref, dtype=np.float64)
        wts = np.ascontiguousarray(weights, dtype=np.float64)
        args = (self._handle.ptr, n_rollouts, rollout_len, self._plane_ptrs(planes, 30),
                self._plane_ptrs(param_planes, 4), mask, self._plane_ptrs(out["wrench"], 6),
                self._plane_ptrs(out["autodyn"], 6),
                out["ctrl"].data_ptr() if out["ctrl"] is not None else None,
                _np_ptr(ref), _np_ptr(wts), int(index_base),
                cost.data_ptr() if cost is not None else None, best.data_ptr(), self._stream())
        fn = _capi.lib().blf_ccm_rollout_cost_argmin_soa
        keep = (planes, param_planes, out, ref, wts, cost, best)

        def call(_keep=keep):
            rc = fn(*args)
            if rc:
                _capi.check(rc)
        return call, out, cost, best

    def evaluate_aos(self, twists, poses, null_poses, params=None, mask: int = FULL,
                     out: dict | None = None):
        n = poses.shape[0]
        out = out if out is not None else self.alloc_aos_outputs(n, mask)
        dp = lambda t: t.data_ptr() if t is not None else None
        _capi.check(_capi.lib().blf_ccm_eval_batch_aos(
            self._handle.ptr, n, dp(twists), dp(poses), dp(null_poses), dp(params), mask,
            dp(out["wrench"]), dp(out["autodyn"]), dp(out["ctrl"]), dp(out["regressor"]),
            self._stream()))
        return out

    def evaluate_host(self, twists, poses, null_poses, params=None, mask: int = FULL,
                      out: dict | None = None):
        """numpy (or pinned torch CPU) arrays in, numpy/pinned arrays out; returns when done."""
        n = poses.shape[0]
        if out is None:
            out = {
                "wrench": np.empty((n, 6)) if mask & WRENCH else None,
                "autodyn": np.empty((n, 6)) if mask & AUTODYN else None,
                "ctrl": np.empty((n, 36)) if mask & CTRL else None,
                "regressor": np.empty((n, 12)) if mask & REGRESSOR else None,
            }

        def hp(a):
            if a is None:
                return None
            if isinstance(a, np.ndarray):
                return a.ctypes.data_as(C.c_void_p)
            return C.c_void_p(a.data_ptr())

        _capi.check(_capi.lib().blf_ccm_eval_batch_host(
            self._handle.ptr, n, hp(twists), hp(poses), hp(null_poses), hp(params), mask,
            hp(out["wrench"]), hp(out["autodyn"]), hp(out["ctrl"]), hp(out["regressor"])))
        return out

    def set_host_chunk(self, contacts: int):
        _capi.check(_capi.lib().blf_ccm_set_host_chunk(self._handle.ptr, int(contacts)))

    def set_host_threads(self, threads: int):
        """Worker threads that expand the compact control-matrix download of evaluate_host
        (-1 automatic, 0 = dense download)."""
        _capi.check(_capi.lib().blf_ccm_set_host_threads(self._handle.ptr, int(threads)))

    def rollout_cost_argmin(self, planes, rollout_len: int, wrench_ref, weights,
                            param_planes=None, mask: int = 0, index_base: int = 0,
                            out: dict | None = None, want_cost: bool = True):
        """Evaluate a rollout-major batch, reduce the per-rollout cost and arg-min, one launch.
        Returns (out, cost tensor or None, best) with best a (2,) int64-viewable tensor:
        best.view(float64)[0] = cost, best[1] = index."""
        t = self._torch
        n = self._num_contacts(planes)
        assert n % rollout_len == 0
        n_rollouts = n // rollout_len
        out = out if out is not None else self.alloc_soa_outputs(n, mask)
        cost = t.empty(n_rollouts, dtype=t.float64, device=self.device) if want_cost else None
        best = t.empty(2, dtype=t.int64, device=self.device)
        ref = np.ascontiguousarray(wrench_ref, dtype=np.float64)
        wts = np.ascontiguousarray(weights, dtype=np.float64)
        _capi.check(_capi.lib().blf_ccm_rollout_cost_argmin_soa(
            self._handle.ptr, n_rollouts, rollout_len, self._plane_ptrs(planes, 30),
            self._plane_ptrs(param_planes, 4), mask, self._plane_ptrs(out["wrench"], 6),
            self._plane_ptrs(out["autodyn"], 6),
            out["ctrl"].data_ptr() if out["ctrl"] is not None else None,
            _np_ptr(ref), _np_ptr(wts), int(index_base),
            cost.data_ptr() if cost is not None else None, best.data_ptr(), self._stream()))
        return out, cost, best

    def argmin_pairs(self, pairs):
        """pairs: (k, 2) int64 tensor of (cost bits, index) -> (2,) best."""
        t = self._torch
        best = t.empty(2, dtype=t.int64, device=self.device)
        _capi.check(_capi.lib().blf_ccm_argmin_pairs(self._handle.ptr, pairs.shape[0],
                                                     pairs.data_ptr(), best.data_ptr(),
                                                     self._stream()))
        return best

    @staticmethod
    def decode_best(best):
        import torch
        b = best.cpu()
        return float(b.view(torch.float64)[0]), int(b[1])
