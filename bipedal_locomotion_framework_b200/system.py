"""Python mirror of the reference's System pieces either side of the contact model, computing ONLY
through the C ABI (SURVEY.md section 8(f) rows 2 and 3).

  FloatingBaseSystemKinematics   src/System/include/BipedalLocomotion/System/
                                 FloatingBaseSystemKinematics.h + src/.../FloatingBaseSystemKinematics.cpp
  ForwardEuler                   ForwardEuler.h / .tpp on top of FixedStepIntegrator.tpp:19-76
  KinematicsBatch                one ForwardEuler step for n systems on device planes
  RolloutBatch                   fused integrate -> contact model -> cost rollouts
  GeneralizedForceBatch          out = base + sum J^T wrench (FloatingBaseSystemDynamics.cpp:199-226)

The C++17 classes under cpp/ are what a reference user links; this module is the pytest / bench
harness.  torch supplies device memory and streams (plumbing only).
"""
from __future__ import annotations

import ctypes as C
import math
import sys

import numpy as np

from . import _capi
from .contact_models import (ContinuousContactModelBatch, _Handle, _np_ptr, _ptr_array)


class FloatingBaseSystemKinematics:
    """State = (position(3), rotation(3,3), joint positions); control = (twist(6), joint
    velocities); `initalize` [sic, the reference's spelling] reads the Baumgarte key "rho"."""

    def __init__(self, device: int = 0):
        self._device = device
        self._handle = None
        self._rho = 0.0
        self._state = (np.zeros(3), np.eye(3), np.zeros(0))
        self._input = (np.zeros(6), np.zeros(0))

    def _h(self):
        if self._handle is None:
            self._handle = _Handle(self._device)   # raises without a device: no CPU path
        return self._handle

    def initalize(self, handler) -> bool:
        if handler is None:
            print("[FloatingBaseSystemKinematics::initalize] The parameter handler is expired. "
                  "Please call the function passing a pointer pointing an already allocated memory.",
                  file=sys.stderr)
            return False
        ok, rho = handler.getParameter("rho", float)
        if not ok:
            print("[FloatingBaseSystemKinematics::initalize] Unable to load the Baumgarte "
                  "stabilization parameter.", file=sys.stderr)
            return False
        self._rho = rho
        return True

    def setState(self, state) -> bool:
        p, R, s = state
        self._state = (np.array(p, dtype=np.float64).reshape(3), np.array(R, dtype=np.float64).reshape(3, 3),
                       np.array(s, dtype=np.float64).reshape(-1))
        return True

    def getState(self):
        return self._state

    def setControlInput(self, control) -> bool:
        tw, sdot = control
        self._input = (np.array(tw, dtype=np.float64).reshape(6),
                       np.array(sdot, dtype=np.float64).reshape(-1))
        return True

    def dynamics(self, time: float = 0.0):
        """Returns (ok, (pos_dot, rot_dot, joint_velocity)); FloatingBaseSystemKinematics.cpp:36-73."""
        tw, sdot = self._input
        p, R, s = self._state
        if sdot.size != s.size:
            print("[FloatingBaseSystemKinematics::dynamics] Wrong size of the vectors.", file=sys.stderr)
            return False, None
        pd, rd = np.empty(3), np.empty(9)
        Rc = np.ascontiguousarray(R).reshape(9)
        _capi.check(_capi.lib().blf_sys_kinematics_dynamics_host(
            self._h().ptr, 1, self._rho, _np_ptr(tw), _np_ptr(Rc), _np_ptr(pd), _np_ptr(rd)))
        return True, (pd, rd.reshape(3, 3), sdot.copy())

    def _euler_steps(self, step_dT: float, last_dT: float, steps: int) -> bool:
        tw, sdot = self._input
        p, R, s = self._state
        if sdot.size != s.size:
            print("[FloatingBaseSystemKinematics::dynamics] Wrong size of the vectors.", file=sys.stderr)
            return False
        p = p.copy()
        Rc = np.ascontiguousarray(R).reshape(9).copy()
        s = s.copy()
        _capi.check(_capi.lib().blf_sys_kinematics_integrate_host(
            self._h().ptr, 1, self._rho, step_dT, last_dT, steps, _np_ptr(tw), _np_ptr(p), _np_ptr(Rc),
            s.size, _np_ptr(sdot) if s.size else None, _np_ptr(s) if s.size else None))
        self._state = (p, Rc.reshape(3, 3), s)
        return True


class ForwardEuler:
    """ForwardEuler<FloatingBaseSystemKinematics>: integrate(t0, tf) with FixedStepIntegrator's
    step schedule (FixedStepIntegrator.tpp:48-64, including its doubled last step), every step on
    the device."""

    def __init__(self, dT: float):
        self._dT = float(dT)
        self._system = None

    def setDynamicalSystem(self, system) -> bool:
        if self._system is not None:
            print("[Integrator::setDynamicalSystem] The dynamical system has been already set.",
                  file=sys.stderr)
            return False
        self._system = system
        return True

    def dynamicalSystem(self):
        return self._system

    def getSolution(self):
        return self._system.getState()

    def integrate(self, initialTime: float, finalTime: float) -> bool:
        if self._system is None:
            print("[FixedStepIntegrator::integrate] Please set the dynamical system before call "
                  "this function.", file=sys.stderr)
            return False
        if initialTime > finalTime:
            print("[FixedStepIntegrator::integrate] The final time has to be greater than the "
                  "initial one.", file=sys.stderr)
            return False
        if self._dT <= 0:
            print("[FixedStepIntegrator::integrate] The sampling time must be a strictly positive "
                  "number.", file=sys.stderr)
            return False
        iterations = int(math.ceil((finalTime - initialTime) / self._dT))
        if iterations < 1:
            # the reference's loop bound underflows here (size_t i < int(-1)) and never terminates
            print("[FixedStepIntegrator::integrate] finalTime == initialTime is not integrable.",
                  file=sys.stderr)
            return False
        current = initialTime
        for i in range(iterations - 1):
            current = initialTime + self._dT * i
        return self._system._euler_steps(self._dT, finalTime - current, iterations)


class KinematicsBatch:
    """One ForwardEuler step of FloatingBaseSystemKinematics for n systems (device planes)."""

    def __init__(self, device: int = 0, handle: _Handle | None = None):
        import torch
        self._torch = torch
        self.device = torch.device("cuda", device)
        self._handle = handle or _Handle(device)

    def euler_step(self, rho: float, dT: float, twist_planes, pos_planes, rot_planes):
        """(6,n), (3,n), (9,n) float64 CUDA tensors; pos/rot updated in place."""
        n = twist_planes.shape[1]
        pp = ContinuousContactModelBatch._plane_ptrs
        st = self._torch.cuda.current_stream(self.device).cuda_stream
        _capi.check(_capi.lib().blf_sys_kinematics_euler_step_soa(
            self._handle.ptr, n, float(rho), float(dT), pp(twist_planes, 6), pp(pos_planes, 3),
            pp(rot_planes, 9), st))

    def prepare_euler_step(self, rho, dT, twist_planes, pos_planes, rot_planes):
        n = twist_planes.shape[1]
        pp = ContinuousContactModelBatch._plane_ptrs
        st = self._torch.cuda.current_stream(self.device).cuda_stream
        args = (self._handle.ptr, n, float(rho), float(dT), pp(twist_planes, 6), pp(pos_planes, 3),
                pp(rot_planes, 9), st)
        fn = _capi.lib().blf_sys_kinematics_euler_step_soa
        keep = (twist_planes, pos_planes, rot_planes)

        def call(_keep=keep):
            rc = fn(*args)
            if rc:
                _capi.check(rc)
        return call


# gradient groups of blf_ccm_rollout_cost_vjp and the output planes of each
ROLLOUT_VJP_GROUPS = {"twist": ("twist",), "pose": ("pos", "rot"), "null": ("null",), "params": ("params",)}

_ROLLOUT_COST_FN = None


def _rollout_cost_function():
    """torch.autograd.Function of RolloutBatch.rollout_cost (built on first use, so importing this
    module does not import torch)."""
    global _ROLLOUT_COST_FN
    if _ROLLOUT_COST_FN is not None:
        return _ROLLOUT_COST_FN
    import torch
    from torch.autograd.function import once_differentiable

    class RolloutCost(torch.autograd.Function):
        @staticmethod
        def forward(ctx, rb, cfg, twist, pos, rot, null, params):
            ctx.rb, ctx.cfg = rb, cfg
            ctx.save_for_backward(twist, pos, rot, null, params)
            return rb.run(*cfg[:5], twist, pos, rot, null, *cfg[5:], param_planes=params)["cost"]

        @staticmethod
        @once_differentiable
        def backward(ctx, grad_cost):
            twist, pos, rot, null, params = ctx.saved_tensors
            need = dict(zip(("twist", "pos", "rot", "null", "params"), ctx.needs_input_grad[2:]))
            groups = {g for g, keys in ROLLOUT_VJP_GROUPS.items() if any(need[k] for k in keys)}
            if not groups:
                return (None,) * 7
            g = ctx.rb.cost_vjp(*ctx.cfg[:5], twist, pos, rot, null, *ctx.cfg[5:], grad_cost.contiguous(),
                                param_planes=params, inputs=groups)
            return (None, None) + tuple(g.get(k) if need[k] else None
                                        for k in ("twist", "pos", "rot", "null", "params"))

    _ROLLOUT_COST_FN = RolloutCost
    return RolloutCost


class RolloutBatch:
    """Fused sampling-MPC rollouts (blf_ccm_rollout_integrate_cost) on one GPU."""

    def __init__(self, batch: ContinuousContactModelBatch):
        self._b = batch
        self._torch = batch._torch
        self.device = batch.device

    def prepare(self, n_rollouts, feet, horizon, dT, rho, twist_planes, pos_planes, rot_planes,
                null_planes, wrench_ref, weights, param_planes=None, mask: int = 0,
                index_base: int = 0, want_final: bool = False, want_cost: bool = True):
        """twist_planes (6, horizon*chains) time-major; pos (3,chains), rot (9,chains),
        null (12,chains) or list with None for the dead third-column planes.
        Returns (call, out) with out: wrench/autodyn (6,n) / ctrl (n,36) trajectories, final_pos,
        final_rot, cost, best."""
        t = self._torch
        chains = n_rollouts * feet
        n = horizon * chains
        mk = lambda *s: t.empty(s, dtype=t.float64, device=self.device)
        out = {
            "wrench": mk(6, n) if mask & 1 else None,
            "autodyn": mk(6, n) if mask & 2 else None,
            "ctrl": mk(n, 36) if mask & 4 else None,
            "final_pos": mk(3, chains) if want_final else None,
            "final_rot": mk(9, chains) if want_final else None,
            "cost": mk(n_rollouts) if want_cost else None,
            "best": t.empty(2, dtype=t.int64, device=self.device),
        }
        ref = np.ascontiguousarray(wrench_ref, dtype=np.float64)
        wts = np.ascontiguousarray(weights, dtype=np.float64)
        pp = ContinuousContactModelBatch._plane_ptrs
        dp = lambda x: x.data_ptr() if x is not None else None
        args = (self._b.handle.ptr, int(n_rollouts), int(feet), int(horizon), float(dT), float(rho),
                pp(twist_planes, 6), pp(pos_planes, 3), pp(rot_planes, 9), pp(null_planes, 12),
                pp(param_planes, 4), int(mask), pp(out["wrench"], 6), pp(out["autodyn"], 6),
                dp(out["ctrl"]), pp(out["final_pos"], 3), pp(out["final_rot"], 9), _np_ptr(ref),
                _np_ptr(wts), int(index_base), dp(out["cost"]), dp(out["best"]), self._b._stream())
        fn = _capi.lib().blf_ccm_rollout_integrate_cost
        keep = (twist_planes, pos_planes, rot_planes, null_planes, param_planes, out, ref, wts)

        def call(_keep=keep):
            rc = fn(*args)
            if rc:
                _capi.check(rc)
        return call, out

    def run(self, *args, **kw):
        call, out = self.prepare(*args, **kw)
        call()
        return out

    def _vjp_args(self, n_rollouts, feet, horizon, dT, rho, twist_planes, pos_planes, rot_planes,
                  null_planes, wrench_ref, weights, grad_cost, param_planes, inputs, out):
        """Arguments of blf_ccm_rollout_cost_vjp and the output dict (see cost_vjp)."""
        t = self._torch
        chains = n_rollouts * feet
        groups = set(ROLLOUT_VJP_GROUPS) if inputs is True else set(inputs or ())
        assert groups <= set(ROLLOUT_VJP_GROUPS), f"unknown gradient groups {groups - set(ROLLOUT_VJP_GROUPS)}"
        if out is None:
            mk = lambda *s: t.empty(s, dtype=t.float64, device=self.device)
            shapes = {"twist": (6, horizon * chains), "pos": (3, chains), "rot": (9, chains),
                      "null": (12, chains), "params": (4, chains)}
            out = {k: mk(*shapes[k]) for g in groups for k in ROLLOUT_VJP_GROUPS[g]}
        ref = np.ascontiguousarray(wrench_ref, dtype=np.float64)
        wts = np.ascontiguousarray(weights, dtype=np.float64)
        pp = ContinuousContactModelBatch._plane_ptrs
        args = (self._b.handle.ptr, int(n_rollouts), int(feet), int(horizon), float(dT), float(rho),
                pp(twist_planes, 6), pp(pos_planes, 3), pp(rot_planes, 9), pp(null_planes, 12),
                pp(param_planes, 4), _np_ptr(ref), _np_ptr(wts), grad_cost.data_ptr(),
                pp(out.get("twist"), 6), pp(out.get("pos"), 3), pp(out.get("rot"), 9),
                pp(out.get("null"), 12), pp(out.get("params"), 4), self._b._stream())
        keep = (twist_planes, pos_planes, rot_planes, null_planes, param_planes, grad_cost, out, ref, wts)
        return args, out, keep

    def cost_vjp(self, n_rollouts, feet, horizon, dT, rho, twist_planes, pos_planes, rot_planes,
                 null_planes, wrench_ref, weights, grad_cost, param_planes=None, inputs=True,
                 out: dict | None = None) -> dict:
        """Reverse mode of the rollouts' cost (blf_ccm_rollout_cost_vjp): for the (n_rollouts,)
        cotangent `grad_cost` of the cost `run` computes from the same arguments, returns
        grad_cost^T dcost/d(input) for the requested groups only.  `inputs`: True for every group or
        a subset of "twist", "pose", "null", "params"; the dict holds "twist" (6, horizon*chains),
        "pos" (3, chains) and "rot" (9, chains) for "pose", "null" (12, chains) and "params"
        (4, chains: each chain's contribution; with uniform parameters the sum is their gradient)."""
        args, out, _ = self._vjp_args(n_rollouts, feet, horizon, dT, rho, twist_planes, pos_planes,
                                      rot_planes, null_planes, wrench_ref, weights, grad_cost,
                                      param_planes, inputs, out)
        _capi.check(_capi.lib().blf_ccm_rollout_cost_vjp(*args))
        return out

    def prepare_cost_vjp(self, n_rollouts, feet, horizon, dT, rho, twist_planes, pos_planes,
                         rot_planes, null_planes, wrench_ref, weights, grad_cost, param_planes=None,
                         inputs=True, out: dict | None = None):
        """Prepared form of cost_vjp (every argument bound once).  Returns (call, out)."""
        args, out, keep = self._vjp_args(n_rollouts, feet, horizon, dT, rho, twist_planes, pos_planes,
                                         rot_planes, null_planes, wrench_ref, weights, grad_cost,
                                         param_planes, inputs, out)
        fn = _capi.lib().blf_ccm_rollout_cost_vjp

        def call(_keep=keep):
            rc = fn(*args)
            if rc:
                _capi.check(rc)
        return call, out

    def rollout_cost(self, n_rollouts, feet, horizon, dT, rho, twist_planes, pos_planes, rot_planes,
                     null_planes, wrench_ref, weights, param_planes=None):
        """(n_rollouts,) cost of `run` through torch.autograd: gradients reach the twist (6,
        horizon*chains), pos (3, chains), rot (9, chains), null (12, chains) and param (4, chains)
        tensors that require them.  The backward is blf_ccm_rollout_cost_vjp, asked only for the
        groups that need a gradient; it is not itself differentiable."""
        cfg = (int(n_rollouts), int(feet), int(horizon), float(dT), float(rho),
               np.array(wrench_ref, dtype=np.float64), np.array(weights, dtype=np.float64))
        return _rollout_cost_function().apply(self, cfg, twist_planes, pos_planes, rot_planes,
                                              null_planes, param_planes)

    def run_host(self, n_rollouts, feet, horizon, dT, rho, twist_planes, pos_planes, rot_planes,
                 null_planes, wrench_ref, weights, param_planes=None, want_cost: bool = True):
        """Host arrays in ((6, horizon*chains) etc.; numpy or pinned torch CPU tensors), pair out:
        blf_ccm_rollout_integrate_cost_host.  Returns (best_cost, best_index, cost or None)."""
        def rows(t, count):
            if t is None:
                return None
            if isinstance(t, np.ndarray):
                assert t.shape[0] == count and t.dtype == np.float64 and t.strides[1] == 8
                return _ptr_array([t[i].ctypes.data for i in range(count)])
            assert t.shape[0] == count and t.stride(1) == 1
            return _ptr_array([t[i].data_ptr() for i in range(count)])
        ref = np.ascontiguousarray(wrench_ref, dtype=np.float64)
        wts = np.ascontiguousarray(weights, dtype=np.float64)
        cost = np.empty(n_rollouts) if want_cost else None
        bc, bi = C.c_double(), C.c_int64()
        _capi.check(_capi.lib().blf_ccm_rollout_integrate_cost_host(
            self._b.handle.ptr, int(n_rollouts), int(feet), int(horizon), float(dT), float(rho),
            rows(twist_planes, 6), rows(pos_planes, 3), rows(rot_planes, 9), rows(null_planes, 12),
            rows(param_planes, 4), _np_ptr(ref), _np_ptr(wts), _np_ptr(cost), C.byref(bc), C.byref(bi)))
        return bc.value, bi.value, cost


class GeneralizedForceBatch:
    """out[s] = base[s] + sum_c J_c^T wrench_c on one GPU (blf_ccm_generalized_force_soa)."""

    def __init__(self, batch: ContinuousContactModelBatch):
        self._b = batch
        self._torch = batch._torch
        self.device = batch.device

    def prepare(self, contacts_per_system, ncols, planes, jacobians, base=None, param_planes=None,
                out=None, want_wrench: bool = False):
        """planes (30,n) or list; jacobians (n,6,ncols) CUDA tensor; base/out (n_systems,ncols)."""
        t = self._torch
        n = self._b._num_contacts(planes)
        assert n % contacts_per_system == 0
        ns = n // contacts_per_system
        out = out if out is not None else t.empty((ns, ncols), dtype=t.float64, device=self.device)
        wrench = t.empty((6, n), dtype=t.float64, device=self.device) if want_wrench else None
        pp = ContinuousContactModelBatch._plane_ptrs
        dp = lambda x: x.data_ptr() if x is not None else None
        args = (self._b.handle.ptr, ns, int(contacts_per_system), int(ncols), pp(planes, 30),
                pp(param_planes, 4), dp(jacobians), dp(base), dp(out), pp(wrench, 6),
                self._b._stream())
        fn = _capi.lib().blf_ccm_generalized_force_soa
        keep = (planes, jacobians, base, param_planes, out, wrench)

        def call(_keep=keep):
            rc = fn(*args)
            if rc:
                _capi.check(rc)
        return call, out, wrench

    def run(self, *args, **kw):
        call, out, wrench = self.prepare(*args, **kw)
        call()
        return (out, wrench) if wrench is not None else out


class FloatingBaseDynamicsBatch:
    """FloatingBaseDynamicalSystem::dynamics from the bias forces on, batched on one GPU
    (reference: src/System/src/FloatingBaseSystemDynamics.cpp:188-248); the rigid-body quantities
    (mass matrices, bias forces, frame Jacobians) are the caller's.

    solve():         acc = (mass + regularization).llt().solve(known [+ joint torques])
                     (blf_sys_mass_matrix_solve)
    acceleration():  known = -bias + sum_c J_c^T wrench_c, then the same solve
                     (blf_sys_floating_base_acceleration)
    """

    def __init__(self, batch: ContinuousContactModelBatch):
        self._b = batch
        self._torch = batch._torch
        self.device = batch.device

    def prepare_solve(self, mass, known, joint_torques=None, regularization=None, out=None):
        """mass (n,nc,nc), known (n,nc), joint_torques (n,nc-6) or None, regularization (nc,nc)
        or None: CUDA float64 tensors.  out may be `known` itself (in place)."""
        t = self._torch
        ns, nc = int(known.shape[0]), int(known.shape[1])
        assert tuple(mass.shape) == (ns, nc, nc) and mass.is_contiguous() and known.is_contiguous()
        out = out if out is not None else t.empty((ns, nc), dtype=t.float64, device=self.device)
        dp = lambda x: x.data_ptr() if x is not None else None
        args = (self._b.handle.ptr, ns, nc, dp(mass), dp(regularization), dp(known), dp(joint_torques),
                dp(out), self._b._stream())
        fn = _capi.lib().blf_sys_mass_matrix_solve
        keep = (mass, known, joint_torques, regularization, out)

        def call(_keep=keep):
            rc = fn(*args)
            if rc:
                _capi.check(rc)
        return call, out

    def solve(self, *args, **kw):
        call, out = self.prepare_solve(*args, **kw)
        call()
        return out

    def prepare_acceleration(self, contacts_per_system, planes, jacobians, bias, mass,
                             joint_torques=None, regularization=None, param_planes=None, out=None,
                             want_wrench: bool = False):
        """planes (30,n) contact states; jacobians (n,6,nc); bias (n_systems,nc) = generalized bias
        forces [base wrench; joint torques]; mass (n_systems,nc,nc)."""
        t = self._torch
        n = self._b._num_contacts(planes)
        assert n % contacts_per_system == 0
        ns, nc = n // contacts_per_system, int(bias.shape[1])
        assert tuple(mass.shape) == (ns, nc, nc) and int(bias.shape[0]) == ns
        out = out if out is not None else t.empty((ns, nc), dtype=t.float64, device=self.device)
        wrench = t.empty((6, n), dtype=t.float64, device=self.device) if want_wrench else None
        pp = ContinuousContactModelBatch._plane_ptrs
        dp = lambda x: x.data_ptr() if x is not None else None
        args = (self._b.handle.ptr, ns, int(contacts_per_system), nc, pp(planes, 30), pp(param_planes, 4),
                dp(jacobians), dp(bias), dp(joint_torques), dp(mass), dp(regularization), dp(out),
                pp(wrench, 6), self._b._stream())
        fn = _capi.lib().blf_sys_floating_base_acceleration
        keep = (planes, jacobians, bias, mass, joint_torques, regularization, param_planes, out, wrench)

        def call(_keep=keep):
            rc = fn(*args)
            if rc:
                _capi.check(rc)
        return call, out, wrench

    def acceleration(self, *args, **kw):
        call, out, wrench = self.prepare_acceleration(*args, **kw)
        call()
        return (out, wrench) if wrench is not None else out

    def prepare_euler_step(self, rho, dT, acc, nu, joint_pos, base_pos, base_rot):
        """One ForwardEuler step of FloatingBaseDynamicalSystem in place (blf_sys_floating_base_euler_step):
        acc, nu (n,nc); joint_pos (n,nc-6) or None; base_pos (n,3); base_rot (n,3,3) or (n,9)."""
        ns, nc = int(nu.shape[0]), int(nu.shape[1])
        for x in (acc, nu, joint_pos, base_pos, base_rot):
            assert x is None or x.is_contiguous()
        dp = lambda x: x.data_ptr() if x is not None else None
        args = (self._b.handle.ptr, ns, nc, float(rho), float(dT), dp(acc), dp(nu), dp(joint_pos), dp(base_pos),
                dp(base_rot), self._b._stream())
        fn = _capi.lib().blf_sys_floating_base_euler_step
        keep = (acc, nu, joint_pos, base_pos, base_rot)

        def call(_keep=keep):
            rc = fn(*args)
            if rc:
                _capi.check(rc)
        return call

    def euler_step(self, *args, **kw):
        self.prepare_euler_step(*args, **kw)()
