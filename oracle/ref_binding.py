"""ctypes view of oracle/_ref/libblf_reference.so = the REFERENCE'S OWN SOURCES compiled in place.

TEST INFRASTRUCTURE ONLY -- importable from tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs, never from the product package.

What the library is (oracle/refbuild/README.md): the unmodified translation units
src/ContactModels/src/{ContactModel,ContinuousContactModel}.cpp,
src/ParametersHandler/src/StdImplementation.cpp, src/Estimators/src/RecursiveLeastSquare.cpp,
src/System/src/FloatingBaseSystemKinematics.cpp (+ the header-only ForwardEuler / FixedStepIntegrator)
compiled from the original project's tree named by BLF_REFERENCE_ROOT against stand-in Eigen /
iDynTree headers, plus oracle/refbuild/ref_driver.cpp, which only calls their public interface.  It
can be (re)built only where that tree is given; tests/reference_samples.py stands in for it elsewhere.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(_HERE, "_ref")
LIB_PATH = os.path.join(REF_DIR, "libblf_reference.so")
REFBUILD_DIR = os.path.join(_HERE, "refbuild")
REFERENCE_ROOT = os.environ.get("BLF_REFERENCE_ROOT", "")   # the original project's source tree, when given
REFERENCE_TESTS = ("ContinuousContactModelReferenceTests", "IntegratorReferenceTests",
                   "ParametersHandlerReferenceTests")
FACADE_TEST = "ContinuousContactModelReferenceTests_on_b200_facade"  # needs a CUDA device to run
FACADE_INTEGRATOR_TEST = "IntegratorReferenceTests_on_b200_facade"    # second section needs a CUDA device
FACADE_HANDLER_TEST = "ParametersHandlerReferenceTests_on_b200_facade"  # host only

WRENCH, AUTODYN, CTRL, REGRESSOR = 1, 2, 4, 8


def reference_sources_present() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isfile(
        os.path.join(REFERENCE_ROOT, "src", "ContactModels", "src", "ContinuousContactModel.cpp"))


def build(force: bool = False) -> str | None:
    """make -C oracle/refbuild: the stand-in self-test and the facade driver always, the reference
    build where the reference tree is given.  Returns the reference library's path, or None when the
    reference tree is absent and nothing was prebuilt."""
    facade = os.path.exists(os.path.join(os.path.dirname(_HERE), "bipedal_locomotion_framework_b200", "lib",
                                         "libblf_contact.so"))
    targets = ["selftest"] + (["facade_driver"] if facade else [])
    if reference_sources_present():
        # + the reference's unmodified tests linked to the product facade
        targets = ["all"] + (["facade"] if facade else [])
    cmd = ["make", "-C", REFBUILD_DIR, f"REF={REFERENCE_ROOT}", *targets] + (["-B"] if force else [])
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("building oracle/_ref failed:\n" + r.stdout)
    return LIB_PATH if os.path.exists(LIB_PATH) else None


def available() -> bool:
    return os.path.exists(LIB_PATH) or (reference_sources_present() and build() is not None)


def usable() -> bool:
    """available() AND the library actually loads here (a prebuilt .so can be present but unloadable on
    a box with another toolchain); callers that only want a baseline fall back to the C port then."""
    if not available():
        return False
    try:
        lib()
        return True
    except OSError:
        return False


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH) and build() is None:
            raise RuntimeError("oracle/_ref/libblf_reference.so is absent and BLF_REFERENCE_ROOT names no "
                               "reference tree to build it from")
        L = C.CDLL(LIB_PATH)
        vp, d, i, sz = C.c_void_p, C.c_double, C.c_int, C.c_size_t
        L.blf_ref_description.restype = C.c_char_p
        L.blf_ref_now.restype = d
        L.blf_ref_ccm_eval_batch_aos.argtypes = [sz] + [vp] * 5 + [C.c_uint] + [vp] * 4 + [i]
        L.blf_ref_ccm_surface_points.argtypes = [vp] * 4 + [sz] + [vp] * 3
        L.blf_ref_ccm_stale_cache_probe.argtypes = [vp] * 4 + [d, vp]
        L.blf_ref_ccm_initialize_probe.argtypes = [i]
        L.blf_ref_rls_run.argtypes = [i, i, vp, d, vp, vp, i, vp, vp, vp, vp]
        L.blf_ref_kin_dynamics.argtypes = [d, vp, vp, vp, vp]
        L.blf_ref_kin_integrate.argtypes = [d, d, d, d, vp, vp, vp, i, vp, vp]
        L.blf_ref_rollout.argtypes = [sz, i, d, d, vp, vp, vp, vp, vp, C.c_uint, vp, vp, vp, i]
        L.blf_ref_generalized_force.argtypes = [sz, i, i] + [vp] * 9 + [i]
        L.blf_ref_floating_base_dynamics.argtypes = [sz, i, i] + [vp] * 12 + [i]
        L.blf_ref_floating_base_euler_step.argtypes = [sz, i, i] + [vp] * 10 + [d, d] + [vp] * 9 + [i]
        _lib = L
    return _lib


ALT_LIB_PATH = os.path.join(REF_DIR, "libblf_reference_alt.so")


def eval_batch_states_alt(states: dict, mask=WRENCH | AUTODYN | CTRL | REGRESSOR, nthreads=1) -> dict:
    """The same reference sources built with the OTHER choices a real-Eigen build could make
    (tree-shaped inner sums, FMA contraction): oracle/_ref/libblf_reference_alt.so.  Only used to
    bound how far such choices move the results."""
    if not os.path.exists(ALT_LIB_PATH):
        build()
    L = C.CDLL(ALT_LIB_PATH)
    L.blf_ref_ccm_eval_batch_aos.argtypes = [C.c_size_t] + [C.c_void_p] * 5 + [C.c_uint] + [C.c_void_p] * 4 + [C.c_int]
    n = states["twists"].shape[0]
    tw, po, nu = _f64(states["twists"]), _f64(states["poses"]), _f64(states["null_poses"])
    pr = None if states.get("params") is None else _f64(states["params"])
    uni = np.asarray(states.get("uniform") if states.get("uniform") is not None else (0, 0, 0, 0), dtype=np.float64)
    out = {"wrench": np.empty((n, 6)) if mask & WRENCH else None,
           "autodyn": np.empty((n, 6)) if mask & AUTODYN else None,
           "ctrl": np.empty((n, 36)) if mask & CTRL else None,
           "regressor": np.empty((n, 12)) if mask & REGRESSOR else None}
    rc = L.blf_ref_ccm_eval_batch_aos(n, _ptr(tw), _ptr(po), _ptr(nu), _ptr(pr), _ptr(uni), mask,
                                      _ptr(out["wrench"]), _ptr(out["autodyn"]), _ptr(out["ctrl"]),
                                      _ptr(out["regressor"]), int(nthreads))
    if rc != 0:
        raise RuntimeError(f"reference initialize() refused (rc={rc})")
    return out


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a if shape is None else a.reshape(shape)


def description() -> str:
    return lib().blf_ref_description().decode()


def now() -> float:
    return lib().blf_ref_now()


def eval_batch_aos(twists, poses, null_poses, params=None, uniform=None,
                   mask=WRENCH | AUTODYN | CTRL, nthreads=1) -> dict:
    """Same signature and result layout as oracle.ccm_oracle.eval_batch_aos, computed by the
    reference's ContinuousContactModel objects (one per thread)."""
    n = twists.shape[0]
    twists, poses, null_poses = _f64(twists), _f64(poses), _f64(null_poses)
    if params is not None:
        params = _f64(params)
    uni = np.asarray(uniform if uniform is not None else (0, 0, 0, 0), dtype=np.float64)
    out = {
        "wrench": np.empty((n, 6)) if mask & WRENCH else None,
        "autodyn": np.empty((n, 6)) if mask & AUTODYN else None,
        "ctrl": np.empty((n, 36)) if mask & CTRL else None,
        "regressor": np.empty((n, 12)) if mask & REGRESSOR else None,
    }
    rc = lib().blf_ref_ccm_eval_batch_aos(n, _ptr(twists), _ptr(poses), _ptr(null_poses),
                                          _ptr(params), _ptr(uni), mask, _ptr(out["wrench"]),
                                          _ptr(out["autodyn"]), _ptr(out["ctrl"]),
                                          _ptr(out["regressor"]), int(nthreads))
    if rc != 0:
        raise RuntimeError(f"reference initialize() refused (rc={rc})")
    return out


def eval_batch_states(states: dict, mask=WRENCH | AUTODYN | CTRL, nthreads=1) -> dict:
    return eval_batch_aos(states["twists"], states["poses"], states["null_poses"],
                          states.get("params"), states.get("uniform"), mask, nthreads)


def surface_points(twist, pose, null_pose, par, xy):
    """getForceAtPoint / getTorqueGeneratedAtPoint of one model state at the points xy (k, 2)."""
    xy = _f64(xy).reshape(-1, 2)
    k = xy.shape[0]
    force, torque = np.empty((k, 3)), np.empty((k, 3))
    rc = lib().blf_ref_ccm_surface_points(_ptr(_f64(twist, 6)), _ptr(_f64(pose, 12)),
                                          _ptr(_f64(null_pose, 12)), _ptr(_f64(par, 4)), k,
                                          _ptr(xy), _ptr(force), _ptr(torque))
    if rc != 0:
        raise RuntimeError("reference initialize() refused")
    return force, torque


def stale_cache_probe(twist, pose, null_pose, par, new_spring):
    out = np.empty(18)
    rc = lib().blf_ref_ccm_stale_cache_probe(_ptr(_f64(twist, 6)), _ptr(_f64(pose, 12)),
                                             _ptr(_f64(null_pose, 12)), _ptr(_f64(par, 4)),
                                             float(new_spring), _ptr(out))
    if rc != 0:
        raise RuntimeError("reference initialize() refused")
    return out[0:6], out[6:12], out[12:18]


def initialize_probe(which: int) -> bool:
    return bool(lib().blf_ref_ccm_initialize_probe(int(which)))


def rls_run(measurement_cov, lam, state0, state_cov_diag, Y, z):
    """nsteps x (setMeasurements + advance) on ONE reference RecursiveLeastSquare.
    Y (nsteps, m, p), z (nsteps, m) -> theta (nsteps, p), P (nsteps, p, p) after every step."""
    Y = _f64(Y)
    nsteps, m, p = Y.shape
    z = _f64(z).reshape(nsteps, m)
    theta, P = np.empty((nsteps, p)), np.empty((nsteps, p, p))
    rc = lib().blf_ref_rls_run(p, m, _ptr(_f64(measurement_cov, m)), float(lam), _ptr(_f64(state0, p)),
                               _ptr(_f64(state_cov_diag, p)), nsteps, _ptr(Y), _ptr(z), _ptr(theta),
                               _ptr(P))
    if rc != 0:
        raise RuntimeError(f"reference RecursiveLeastSquare failed (rc={rc})")
    return theta, P


def kin_dynamics(rho, twist, rot):
    pd, rd = np.empty(3), np.empty(9)
    rc = lib().blf_ref_kin_dynamics(float(rho), _ptr(_f64(twist, 6)), _ptr(_f64(rot, 9)), _ptr(pd),
                                    _ptr(rd))
    if rc != 0:
        raise RuntimeError(f"reference FloatingBaseSystemKinematics failed (rc={rc})")
    return pd, rd.reshape(3, 3)


def kin_integrate(rho, step_dT, t0, tf, twist, pos, rot, joint_vel=None, joint_pos=None):
    """ForwardEuler<FloatingBaseSystemKinematics>(step_dT).integrate(t0, tf); returns
    (ok, pos, rot[, joint_pos])."""
    pos = np.array(pos, dtype=np.float64).reshape(3).copy()
    rot = np.array(rot, dtype=np.float64).reshape(9).copy()
    nj = 0 if joint_vel is None else len(joint_vel)
    jv = None if nj == 0 else _f64(joint_vel, nj)
    jp = None if nj == 0 else np.array(joint_pos, dtype=np.float64).reshape(nj).copy()
    rc = lib().blf_ref_kin_integrate(float(rho), float(step_dT), float(t0), float(tf),
                                     _ptr(_f64(twist, 6)), _ptr(pos), _ptr(rot), nj, _ptr(jv), _ptr(jp))
    if rc == -1:
        raise RuntimeError("reference kinematics set-up failed")
    return rc == 0, pos, rot.reshape(3, 3), jp


def rollout(twists, poses, null_poses, dT, rho, params=None, uniform=None,
            mask=WRENCH, nthreads=1) -> dict:
    """integrate -> contact model over a horizon with the reference's objects.
    twists (horizon, chains, 6); poses (chains, 12) initial; returns time-major outputs
    (horizon*chains, ...) and the final poses."""
    twists = _f64(twists)
    horizon, chains, _ = twists.shape
    poses = np.array(poses, dtype=np.float64).reshape(chains, 12).copy()
    null_poses = _f64(null_poses).reshape(chains, 12)
    if params is not None:
        params = _f64(params).reshape(chains, 4)
    uni = np.asarray(uniform if uniform is not None else (0, 0, 0, 0), dtype=np.float64)
    n = horizon * chains
    out = {
        "wrench": np.empty((n, 6)) if mask & WRENCH else None,
        "autodyn": np.empty((n, 6)) if mask & AUTODYN else None,
        "ctrl": np.empty((n, 36)) if mask & CTRL else None,
    }
    rc = lib().blf_ref_rollout(chains, horizon, float(dT), float(rho), _ptr(twists), _ptr(poses),
                               _ptr(null_poses), _ptr(params), _ptr(uni), mask, _ptr(out["wrench"]),
                               _ptr(out["autodyn"]), _ptr(out["ctrl"]), int(nthreads))
    if rc != 0:
        raise RuntimeError(f"reference rollout failed (rc={rc})")
    out["final_poses"] = poses
    return out


def generalized_force(contacts_per_system, ncols, twists, poses, null_poses, jacobians, base=None,
                      params=None, uniform=None, want_wrench=False, nthreads=1):
    """FloatingBaseDynamicalSystem::dynamics run from the reference's own source over the
    KinDynComputations test double (identity mass matrix, injected Jacobians and bias forces):
    out[s] = base[s] + sum_c J_c^T wrench_c.  AoS states (n = n_systems * contacts_per_system),
    jacobians (n, 6, ncols), base (n_systems, ncols) or None."""
    twists, poses, null_poses = _f64(twists), _f64(poses), _f64(null_poses)
    n = twists.shape[0]
    assert n % contacts_per_system == 0
    ns = n // contacts_per_system
    J = _f64(jacobians)
    assert J.size == n * 6 * ncols
    b = None if base is None else _f64(base).reshape(ns, ncols)
    pr = None if params is None else _f64(params).reshape(n, 4)
    uni = np.asarray(uniform if uniform is not None else (0, 0, 0, 0), dtype=np.float64)
    out = np.empty((ns, ncols))
    wr = np.empty((n, 6)) if want_wrench else None
    rc = lib().blf_ref_generalized_force(ns, int(contacts_per_system), int(ncols), _ptr(twists), _ptr(poses),
                                         _ptr(null_poses), _ptr(pr), _ptr(uni), _ptr(J), _ptr(b), _ptr(out),
                                         _ptr(wr), int(nthreads))
    if rc != 0:
        raise RuntimeError(f"reference FloatingBaseDynamicalSystem failed (rc={rc})")
    return (out, wr) if want_wrench else out


def floating_base_dynamics(contacts_per_system, twists, poses, null_poses, jacobians, bias, mass,
                           joint_torques=None, reg=None, params=None, uniform=None, want_wrench=False,
                           nthreads=1):
    """The whole of FloatingBaseDynamicalSystem::dynamics from the bias forces on, run from the
    reference's own source over the KinDynComputations test double loaded with the given mass
    matrices (n_systems, nc, nc), bias forces (n_systems, nc) and contact frames; reg (nc, nc)
    goes through setMassMatrixRegularization.  Returns [base acc; joint acc] (n_systems, nc)."""
    twists, poses, null_poses = _f64(twists), _f64(poses), _f64(null_poses)
    n = twists.shape[0]
    assert n % contacts_per_system == 0
    ns = n // contacts_per_system
    b = _f64(bias)
    ncols = b.shape[1]
    assert b.shape[0] == ns
    J = _f64(jacobians)
    assert J.size == n * 6 * ncols
    M = _f64(mass)
    assert M.shape == (ns, ncols, ncols)
    tau = None if joint_torques is None else _f64(joint_torques).reshape(ns, ncols - 6)
    rg = None if reg is None else _f64(reg).reshape(ncols, ncols)
    pr = None if params is None else _f64(params).reshape(n, 4)
    uni = np.asarray(uniform if uniform is not None else (0, 0, 0, 0), dtype=np.float64)
    out = np.empty((ns, ncols))
    wr = np.empty((n, 6)) if want_wrench else None
    rc = lib().blf_ref_floating_base_dynamics(ns, int(contacts_per_system), int(ncols), _ptr(twists),
                                              _ptr(poses), _ptr(null_poses), _ptr(pr), _ptr(uni), _ptr(J),
                                              _ptr(b), _ptr(tau), _ptr(M), _ptr(rg), _ptr(out), _ptr(wr),
                                              int(nthreads))
    if rc != 0:
        raise RuntimeError(f"reference FloatingBaseDynamicalSystem failed (rc={rc})")
    return (out, wr) if want_wrench else out


def floating_base_euler_step(contacts_per_system, twists, poses, null_poses, jacobians, bias, mass, rho, dT, nu,
                             joint_pos, base_pos, base_rot, joint_torques=None, reg=None, params=None,
                             uniform=None, nthreads=1):
    """ForwardEuler<FloatingBaseDynamicalSystem>(dT).integrate(0, dT) per system from the reference's own
    sources over the KinDynComputations test double.  Returns (acc, nu, joint_pos, base_pos, base_rot)."""
    twists, poses, null_poses = _f64(twists), _f64(poses), _f64(null_poses)
    n = twists.shape[0]
    ns = n // contacts_per_system
    b = _f64(bias)
    ncols = b.shape[1]
    J, M = _f64(jacobians), _f64(mass)
    tau = None if joint_torques is None else _f64(joint_torques).reshape(ns, ncols - 6)
    rg = None if reg is None else _f64(reg).reshape(ncols, ncols)
    pr = None if params is None else _f64(params).reshape(n, 4)
    uni = np.asarray(uniform if uniform is not None else (0, 0, 0, 0), dtype=np.float64)
    v, p, r = _f64(nu).reshape(ns, ncols), _f64(base_pos).reshape(ns, 3), _f64(base_rot).reshape(ns, 9)
    jp = np.zeros((ns, max(ncols - 6, 0))) if joint_pos is None else _f64(joint_pos).reshape(ns, ncols - 6)
    acc, vo, jo = np.empty((ns, ncols)), np.empty((ns, ncols)), np.empty((ns, max(ncols - 6, 0)))
    po, ro = np.empty((ns, 3)), np.empty((ns, 9))
    rc = lib().blf_ref_floating_base_euler_step(ns, int(contacts_per_system), int(ncols), _ptr(twists), _ptr(poses),
                                                _ptr(null_poses), _ptr(pr), _ptr(uni), _ptr(J), _ptr(b), _ptr(tau),
                                                _ptr(M), _ptr(rg), float(rho), float(dT), _ptr(v), _ptr(jp), _ptr(p),
                                                _ptr(r), _ptr(acc), _ptr(vo), _ptr(jo), _ptr(po), _ptr(ro),
                                                int(nthreads))
    if rc != 0:
        raise RuntimeError(f"reference ForwardEuler<FloatingBaseDynamicalSystem> failed (rc={rc})")
    return acc, vo, jo, po, ro.reshape(ns, 3, 3)


FACADE_FBD_DRIVER = "libblf_facade_fbd_driver.so"   # facade_glue/facade_fbd_driver.cpp; needs a CUDA device to run
_facade_fbd = None


def facade_floating_base_euler_step(contacts_per_system, twists, poses, null_poses, jacobians, bias, mass, rho, dT,
                                    nu, joint_pos, base_pos, base_rot, joint_torques=None, reg=None, params=None,
                                    uniform=None):
    """The same call as floating_base_euler_step, answered by the PRODUCT's C++ facade classes
    (System::FloatingBaseDynamicalSystem + ForwardEuler on the GPU) through facade_fbd_driver.cpp."""
    global _facade_fbd
    if _facade_fbd is None:
        path = os.path.join(REF_DIR, FACADE_FBD_DRIVER)
        if not os.path.exists(path):
            build()
        _facade_fbd = C.CDLL(path)
        vp, dbl = C.c_void_p, C.c_double
        _facade_fbd.blf_facade_floating_base_euler_step.argtypes = [C.c_size_t, C.c_int, C.c_int] + [vp] * 10 + \
            [dbl, dbl] + [vp] * 9
        _facade_fbd.blf_facade_floating_base_euler_step.restype = C.c_int
    twists, poses, null_poses = _f64(twists), _f64(poses), _f64(null_poses)
    n = twists.shape[0]
    ns = n // contacts_per_system
    b = _f64(bias)
    ncols = b.shape[1]
    J, M = _f64(jacobians), _f64(mass)
    tau = None if joint_torques is None else _f64(joint_torques).reshape(ns, ncols - 6)
    rg = None if reg is None else _f64(reg).reshape(ncols, ncols)
    pr = None if params is None else _f64(params).reshape(n, 4)
    uni = np.asarray(uniform if uniform is not None else (0, 0, 0, 0), dtype=np.float64)
    v, p, r = _f64(nu).reshape(ns, ncols), _f64(base_pos).reshape(ns, 3), _f64(base_rot).reshape(ns, 9)
    jp = np.zeros((ns, max(ncols - 6, 0))) if joint_pos is None else _f64(joint_pos).reshape(ns, ncols - 6)
    acc, vo, jo = np.empty((ns, ncols)), np.empty((ns, ncols)), np.empty((ns, max(ncols - 6, 0)))
    po, ro = np.empty((ns, 3)), np.empty((ns, 9))
    rc = _facade_fbd.blf_facade_floating_base_euler_step(
        ns, int(contacts_per_system), int(ncols), _ptr(twists), _ptr(poses), _ptr(null_poses), _ptr(pr), _ptr(uni),
        _ptr(J), _ptr(b), _ptr(tau), _ptr(M), _ptr(rg), float(rho), float(dT), _ptr(v), _ptr(jp), _ptr(p), _ptr(r),
        _ptr(acc), _ptr(vo), _ptr(jo), _ptr(po), _ptr(ro))
    if rc != 0:
        raise RuntimeError(f"facade ForwardEuler<FloatingBaseDynamicalSystem> failed (rc={rc})")
    return acc, vo, jo, po, ro.reshape(ns, 3, 3)


def run_reference_test(name: str, timeout: float = 600.0) -> subprocess.CompletedProcess:
    """Run one of the reference's own (unmodified) Catch2 test executables built into oracle/_ref."""
    exe = os.path.join(REF_DIR, name)
    if not os.path.exists(exe):
        build()
    return subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                          timeout=timeout)
