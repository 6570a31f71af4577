"""What the reference build (oracle/_ref: the original project's sources compiled against the stand-in
headers of oracle/refbuild/) answers in the GPU tests, without the original project's source tree.

Every function has the signature and result layout of its namesake in oracle/ref_binding.py.  The
answer comes from the C restatement (oracle/*.c), which tests/test_reference_build.py holds bit for bit
to the reference build wherever that tree is given.  Each answer is then pinned: a fixed, seeded sample
of at most SAMPLE_ROWS rows of every output, chosen from a hash of the call's inputs, must equal what
tests/golden/reference_samples.npz stores for those inputs.  A change to the restatement therefore
cannot move the GPU tests' yardstick unnoticed.

With BLF_RECORD_REFERENCE_SAMPLES=<file.npz> set, calls are recorded into that file (written at exit)
instead of checked; that is how the stored samples were made, from the GPU tests that use this module.
"""
from __future__ import annotations

import atexit
import hashlib
import os

import numpy as np

from bipedal_locomotion_framework_b200 import synthetic as syn

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_samples.npz")
SAMPLE_ROWS = 16
WRENCH, AUTODYN, CTRL, REGRESSOR = 1, 2, 4, 8

_record_path = os.environ.get("BLF_RECORD_REFERENCE_SAMPLES")
_recorded: dict[str, np.ndarray] = {}
_stored = None


def _feed(h, x):
    if isinstance(x, dict):
        for k in sorted(x):
            h.update(k.encode())
            _feed(h, x[k])
    elif x is None:
        h.update(b"None")
    elif isinstance(x, (int, float, np.integer, np.floating)) and not isinstance(x, bool):
        h.update(np.float64(x).tobytes())
    else:
        a = np.ascontiguousarray(x, dtype=np.float64)
        h.update(str(a.shape).encode())
        h.update(a.tobytes())


def _pin(name: str, inputs, outputs):
    """Check (or record) a seeded sample of rows of every output array of one call."""
    h = hashlib.sha1(name.encode())
    for x in inputs:
        _feed(h, x)
    key = f"{name}:{h.hexdigest()}"
    rng = np.random.default_rng(int(h.hexdigest()[:15], 16))
    parts = []
    for out in outputs:
        if out is None:
            continue
        a = np.asarray(out, dtype=np.float64)
        a = a.reshape(a.shape[0], -1) if a.ndim else a.reshape(1, 1)
        rows = np.sort(rng.choice(a.shape[0], min(a.shape[0], SAMPLE_ROWS), replace=False))
        parts.append(a[rows].ravel())
    got = np.concatenate(parts) if parts else np.zeros(0)
    if _record_path:
        _recorded[key] = got
        return
    global _stored
    if _stored is None:
        with np.load(GOLDEN) as z:
            keys, offsets, values = z["keys"].astype(str), z["offsets"], z["values"]
        _stored = {str(k): values[offsets[i]:offsets[i + 1]] for i, k in enumerate(keys)}
    want = _stored.get(key)
    assert want is not None, f"{name}: no stored reference sample for these inputs ({GOLDEN})"
    assert np.array_equal(got, want, equal_nan=True), \
        f"{name}: the C restatement no longer reproduces the stored reference sample"


@atexit.register
def _write_recorded():
    if _record_path and _recorded:
        keys = sorted(_recorded)
        offsets = np.cumsum([0] + [_recorded[k].size for k in keys])
        np.savez_compressed(_record_path, keys=np.array(keys, dtype="S"), offsets=offsets,
                            values=np.concatenate([_recorded[k] for k in keys]))


def _oracles():
    from oracle import ccm_oracle, sys_oracle
    ccm_oracle.build()
    return ccm_oracle, sys_oracle


def eval_batch_aos(twists, poses, null_poses, params=None, uniform=None, mask=WRENCH | AUTODYN | CTRL, nthreads=1):
    co, _ = _oracles()
    out = co.eval_batch_aos(twists, poses, null_poses, params, uniform, mask, nthreads)
    _pin("eval_batch_aos", (twists, poses, null_poses, params, uniform, mask),
         [out[k] for k in ("wrench", "autodyn", "ctrl", "regressor")])
    return out


def eval_batch_states(states: dict, mask=WRENCH | AUTODYN | CTRL, nthreads=1) -> dict:
    return eval_batch_aos(states["twists"], states["poses"], states["null_poses"], states.get("params"),
                          states.get("uniform"), mask, nthreads)


def surface_points(twist, pose, null_pose, par, xy):
    co, _ = _oracles()
    m = co.ContinuousContactModel()
    L, W, k, b = (float(v) for v in par)
    assert m.initialize({"length": L, "width": W, "spring_coeff": k, "damper_coeff": b})
    m.setState(twist, pose)
    m.setNullForceTransform(null_pose)
    xy = np.asarray(xy, dtype=np.float64).reshape(-1, 2)
    force = np.array([m.getForceAtPoint(x, y) for x, y in xy]).reshape(-1, 3)
    torque = np.array([m.getTorqueGeneratedAtPoint(x, y) for x, y in xy]).reshape(-1, 3)
    _pin("surface_points", (twist, pose, null_pose, par, xy), [force, torque])
    return force, torque


def rls_run(measurement_cov, lam, state0, state_cov_diag, Y, z):
    co, _ = _oracles()
    Y = np.asarray(Y, dtype=np.float64)
    nsteps, m, p = Y.shape
    z = np.asarray(z, dtype=np.float64).reshape(nsteps, m)
    th = np.asarray(state0, dtype=np.float64).reshape(1, p).copy()
    P = np.diag(np.asarray(state_cov_diag, dtype=np.float64).reshape(p))[None].copy()
    theta, Ps = np.empty((nsteps, p)), np.empty((nsteps, p, p))
    for s in range(nsteps):
        th, P = co.rls_advance_batch(Y[s][None], z[s][None], measurement_cov, lam, th, P)
        theta[s], Ps[s] = th[0], P[0]
    _pin("rls_run", (measurement_cov, lam, state0, state_cov_diag, Y, z), [theta, Ps])
    return theta, Ps


def kin_integrate(rho, step_dT, t0, tf, twist, pos, rot, joint_vel=None, joint_pos=None):
    _, so = _oracles()
    if joint_vel is None:
        steps, p, r = so.integrate(rho, step_dT, t0, tf, twist, pos, rot)
        jp = None
    else:
        steps, p, r, jp = so.integrate(rho, step_dT, t0, tf, twist, pos, rot, joint_vel, joint_pos)
    _pin("kin_integrate", (rho, step_dT, t0, tf, twist, pos, rot, joint_vel, joint_pos), [[steps], p, r, jp])
    return steps >= 0, p, r, jp


def rollout(twists, poses, null_poses, dT, rho, params=None, uniform=None, mask=WRENCH, nthreads=1) -> dict:
    _, so = _oracles()
    tw = np.asarray(twists, dtype=np.float64)
    horizon, chains, _ = tw.shape
    poses = np.asarray(poses, dtype=np.float64).reshape(chains, 12)
    o = so.rollout(chains, 1, horizon, dT, rho, np.ascontiguousarray(tw.reshape(horizon * chains, 6).T),
                   np.ascontiguousarray(poses[:, :3].T), np.ascontiguousarray(poses[:, 3:].T),
                   np.ascontiguousarray(np.asarray(null_poses, dtype=np.float64).reshape(chains, 12).T),
                   param_planes=None if params is None else np.ascontiguousarray(np.asarray(params).reshape(chains, 4).T),
                   uniform=uniform, mask=mask, wrench_ref=np.zeros(6), weights=np.ones(2), nthreads=nthreads)
    out = {"wrench": None if o["wrench"] is None else o["wrench"].T.copy(),
           "autodyn": None if o["autodyn"] is None else o["autodyn"].T.copy(),
           "ctrl": o["ctrl"], "final_poses": np.concatenate([o["pos"].T, o["rot"].T], axis=1)}
    _pin("rollout", (tw, poses, null_poses, dT, rho, params, uniform, mask),
         [out[k] for k in ("wrench", "autodyn", "ctrl", "final_poses")])
    return out


def _planes_and_params(twists, poses, null_poses, params, n):
    planes = syn.aos_to_planes(np.asarray(twists, dtype=np.float64), np.asarray(poses, dtype=np.float64),
                               np.asarray(null_poses, dtype=np.float64))
    pp = None if params is None else np.ascontiguousarray(np.asarray(params, dtype=np.float64).reshape(n, 4).T)
    return planes, pp


def generalized_force(contacts_per_system, ncols, twists, poses, null_poses, jacobians, base=None,
                      params=None, uniform=None, want_wrench=False, nthreads=1):
    _, so = _oracles()
    n = np.asarray(twists).shape[0]
    planes, pp = _planes_and_params(twists, poses, null_poses, params, n)
    out, wr = so.generalized_force(contacts_per_system, ncols, planes, jacobians, base, param_planes=pp,
                                   uniform=uniform, want_wrench=True, nthreads=nthreads)
    wr = wr.T.copy()
    _pin("generalized_force", (contacts_per_system, ncols, twists, poses, null_poses, jacobians, base, params,
                               uniform), [out, wr])
    return (out, wr) if want_wrench else out


def floating_base_dynamics(contacts_per_system, twists, poses, null_poses, jacobians, bias, mass,
                           joint_torques=None, reg=None, params=None, uniform=None, want_wrench=False,
                           nthreads=1):
    _, so = _oracles()
    n = np.asarray(twists).shape[0]
    planes, pp = _planes_and_params(twists, poses, null_poses, params, n)
    acc, wr = so.floating_base_acceleration(contacts_per_system, planes, jacobians, bias, mass, joint_torques, reg,
                                            param_planes=pp, uniform=uniform, want_wrench=True, nthreads=nthreads)
    wr = wr.T.copy()
    _pin("floating_base_dynamics", (contacts_per_system, twists, poses, null_poses, jacobians, bias, mass,
                                    joint_torques, reg, params, uniform), [acc, wr])
    return (acc, wr) if want_wrench else acc


def floating_base_euler_step(contacts_per_system, twists, poses, null_poses, jacobians, bias, mass, rho, dT, nu,
                             joint_pos, base_pos, base_rot, joint_torques=None, reg=None, params=None,
                             uniform=None, nthreads=1):
    _, so = _oracles()
    n = np.asarray(twists).shape[0]
    planes, pp = _planes_and_params(twists, poses, null_poses, params, n)
    acc = so.floating_base_acceleration(contacts_per_system, planes, jacobians, bias, mass, joint_torques, reg,
                                        param_planes=pp, uniform=uniform, nthreads=nthreads)
    v, q, p, R = so.floating_base_euler_step(rho, dT, acc, nu, joint_pos, base_pos, base_rot, nthreads=nthreads)
    _pin("floating_base_euler_step", (contacts_per_system, twists, poses, null_poses, jacobians, bias, mass, rho,
                                      dT, nu, joint_pos, base_pos, base_rot, joint_torques, reg, params, uniform),
         [acc, v, q, p, R])
    return acc, v, q, p, R


def facade_floating_base_euler_step(*args, **kw):
    """The product's C++ facade classes, through oracle/refbuild/facade_glue (built without the original tree)."""
    from oracle import ref_binding
    return ref_binding.facade_floating_base_euler_step(*args, **kw)
