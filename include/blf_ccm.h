/*
 * blf_ccm.h -- C ABI of the B200 (sm_100a) backend for ContactModels::ContinuousContactModel.
 *
 * This is the drop-in boundary: host code (the C++17 facade in
 * bipedal_locomotion_framework_b200/cpp, or any FFI) reaches CUDA only through these functions.
 * Plain pointers and sizes, no C++/torch types.  There is NO CPU fallback behind any of them: with
 * no CUDA device blf_ccm_create() fails and every other call returns BLF_CCM_ERR_INVALID_HANDLE.
 *
 * What each entry point replaces in the reference (paths relative to the reference tree):
 *   blf_ccm_set_uniform_params   ContinuousContactModel::initializePrivate, the four doubles read
 *                                from the handler  src/ContactModels/src/ContinuousContactModel.cpp:24-65
 *   blf_ccm_eval_batch_*         per state: ContactModel::setState (src/ContactModels/src/ContactModel.cpp:35-48),
 *                                setNullForceTransform (:23-33), getContactWrench (:50-59 ->
 *                                ContinuousContactModel.cpp:79-108), getAutonomousDynamics (:61-70 ->
 *                                :110-146), getControlMatrix (:72-81 -> :148-171), getRegressor
 *                                (:83-92 -> :223-254); the loop over contacts is the caller's, e.g.
 *                                src/System/src/FloatingBaseSystemDynamics.cpp:199-226
 *   blf_ccm_eval_surface_points  ContinuousContactModel::getForceAtPoint / getTorqueGeneratedAtPoint
 *                                ContinuousContactModel.cpp:173-221
 *   blf_ccm_rollout_*            no reference equivalent (sampling-MPC cost + arg-min; DESIGN.md)
 *
 * Data layouts (all FP64; identical to iDynTree's so arrays of iDynTree objects can be passed):
 *   twist      6  doubles: linear xyz, angular xyz (mixed representation)  iDynTree::Twist
 *   pose       12 doubles: position xyz, rotation 3x3 ROW-major           iDynTree::Transform
 *   wrench     6  doubles: force xyz, torque xyz                           iDynTree::Wrench
 *   autodyn    6  doubles                                                  iDynTree::Vector6
 *   ctrl       36 doubles, dense ROW-major 6x6, structural zeros = +0.0    iDynTree::Matrix6x6
 *   regressor  12 doubles, ROW-major 6x2                                   iDynTree::MatrixDynSize
 *   SoA input planes, each n doubles, index = BLF_CCM_PLANE_*:
 *     0-2 v | 3-5 omega | 6-8 p | 9-17 R row-major | 18-20 p0 | 21-29 R0 row-major
 *     Planes that cannot affect the requested outputs may be NULL: R0's third column (23,26,29)
 *     always; R02,R12 (11,14) unless AUTODYN is requested.
 *
 * Pointers are DEVICE pointers unless the function name says host.  The arrays-of-pointers
 * themselves (in_planes etc.) are HOST arrays of device pointers.  Alignment: 8 bytes is always
 * accepted.  SoA planes are read/written with coalesced 64-bit accesses and need no more.  Buffers
 * that are staged through shared memory with bulk async copies (the dense ctrl array, and every
 * array of the AoS entry points) take that path when 16-byte aligned; otherwise a direct 64-bit
 * path is dispatched -- same results, and blf_ccm_last_path reports which (checked, not silent).
 *
 * Threading: a handle is used from one host thread at a time; distinct handles are independent.
 * Launches are asynchronous on the caller's stream (void* = cudaStream_t, NULL = default stream).
 * Every call makes the handle's device current for its own duration and restores the caller's
 * current device before it returns.
 * Streams: the evaluation entry points (blf_ccm_eval_batch_soa/_aos, blf_rls_*, blf_sys_*_soa,
 * blf_ccm_generalized_force_soa) keep no state between calls and may be in flight on any number of
 * streams at once.  The rollout entry points (blf_ccm_rollout_cost_argmin_soa,
 * blf_ccm_rollout_integrate_cost and its _host form) share ONE set of reduction scratch per handle:
 * a rollout call issued on another stream than the previous one is ordered after it by the library
 * (event wait), i.e. rollout calls of one handle are serialised, never corrupted; use one handle
 * per stream for concurrent rollouts.
 * Errors: 0 = ok, negative = blf_ccm_status; text via blf_ccm_last_error(); nothing throws.
 */
#ifndef BLF_CCM_H
#define BLF_CCM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define BLF_CCM_API
#else
#define BLF_CCM_API __attribute__((visibility("default")))
#endif

typedef struct blf_ccm_handle blf_ccm_handle;

typedef enum {
    BLF_CCM_OK = 0,
    BLF_CCM_ERR_INVALID_ARG = -1,
    BLF_CCM_ERR_INVALID_HANDLE = -2,
    BLF_CCM_ERR_CUDA = -3,
    BLF_CCM_ERR_NO_DEVICE = -4,
    BLF_CCM_ERR_NOT_INITIALIZED = -5,
    BLF_CCM_ERR_NCCL = -6
} blf_ccm_status;

/* out_mask bits */
enum {
    BLF_CCM_WRENCH = 1,    /* getContactWrench      */
    BLF_CCM_AUTODYN = 2,   /* getAutonomousDynamics */
    BLF_CCM_CTRL = 4,      /* getControlMatrix      */
    BLF_CCM_REGRESSOR = 8  /* getRegressor          */
};

enum { BLF_CCM_NUM_IN_PLANES = 30, BLF_CCM_NUM_PARAM_PLANES = 4 };

/* per-contact parameters for the AoS entry points (keys of initializePrivate, same order as
 * blf_ccm_set_uniform_params) */
typedef struct {
    double length;
    double width;
    double spring_coeff;
    double damper_coeff;
} blf_ccm_params;

/* code path taken by the last evaluation on a handle */
enum {
    BLF_CCM_PATH_NONE = 0,
    BLF_CCM_PATH_BULK = 1,    /* bulk-copy (TMA) staging in use: every staged buffer 16-byte aligned */
    BLF_CCM_PATH_DIRECT64 = 2,/* a staged buffer is only 8-byte aligned: direct 64-bit accesses     */
    BLF_CCM_PATH_LLT_WARP = 3,/* mass-matrix solve: warp-level kernel (ncols <= 64)                 */
    BLF_CCM_PATH_LLT_BLOCK = 4/* mass-matrix solve: block-level kernel (ncols 65..128)              */
};

BLF_CCM_API const char* blf_ccm_version(void);
BLF_CCM_API const char* blf_ccm_last_error(void);

/* Create a handle bound to CUDA device `device`.  Fails with BLF_CCM_ERR_NO_DEVICE when there is
 * no usable device (there is no CPU path). */
BLF_CCM_API int blf_ccm_create(int device, blf_ccm_handle** out);
BLF_CCM_API int blf_ccm_destroy(blf_ccm_handle* h);

/* length, width, spring_coeff, damper_coeff for every contact of subsequent evaluations that pass
 * no per-contact parameters.  No range validation, as in the reference. */
BLF_CCM_API int blf_ccm_set_uniform_params(blf_ccm_handle* h, double length, double width,
                                           double spring_coeff, double damper_coeff);

/* Structure-of-arrays evaluation.  wrench_planes[6], autodyn_planes[6], regressor_planes[12] are
 * host arrays of device plane pointers (NULL when the bit is not in out_mask); ctrl is one dense
 * n*36 array.  param_planes = NULL -> uniform parameters, else 4 planes length,width,spring,damper. */
BLF_CCM_API int blf_ccm_eval_batch_soa(blf_ccm_handle* h, int64_t n,
                                       const double* const* in_planes,
                                       const double* const* param_planes, unsigned out_mask,
                                       double* const* wrench_planes,
                                       double* const* autodyn_planes, double* ctrl,
                                       double* const* regressor_planes, void* stream);

/* Array-of-structures evaluation: arrays of iDynTree-layout objects in, arrays of
 * iDynTree-layout objects out.  twists n*6, poses n*12, null_poses n*12, params NULL or n structs;
 * wrench n*6, autodyn n*6, ctrl n*36, regressor n*12 (NULL when not in out_mask). */
BLF_CCM_API int blf_ccm_eval_batch_aos(blf_ccm_handle* h, int64_t n, const double* twists,
                                       const double* poses, const double* null_poses,
                                       const blf_ccm_params* params, unsigned out_mask,
                                       double* wrench, double* autodyn, double* ctrl,
                                       double* regressor, void* stream);

/* Same as blf_ccm_eval_batch_aos but every pointer is a HOST pointer (pinned memory gives full
 * PCIe speed; pageable works).  Chunks the batch, and overlaps host->device copies, the kernel and
 * device->host copies on the handle's own streams; returns after the results are in host memory. */
BLF_CCM_API int blf_ccm_eval_batch_host(blf_ccm_handle* h, int64_t n, const double* twists,
                                        const double* poses, const double* null_poses,
                                        const blf_ccm_params* params, unsigned out_mask,
                                        double* wrench, double* autodyn, double* ctrl,
                                        double* regressor);

/* Largest chunk (contacts) of the blf_ccm_eval_batch_host pipeline (default 131072, measured best on B200 + PCIe Gen5;
 * the schedule ramps chunk/4, chunk/2, chunk ... chunk, chunk/2, chunk/4; tuning knob). */
BLF_CCM_API int blf_ccm_set_host_chunk(blf_ccm_handle* h, int64_t contacts);

/* blf_ccm_eval_batch_host moves the control matrix over PCIe in compact form (its 7 distinct values,
 * 64 instead of 288 bytes per contact) and `threads` host worker threads of the library expand it
 * into the caller's dense Matrix6x6 array, structural zeros +0.0, bit-identical to the device
 * layout.  -1 (default) = min(4, cores/2) (cores divided by LOCAL_WORLD_SIZE when a launcher sets
 * it); 0 = download the dense array instead (no host threads).  Environment override at create:
 * BLF_CCM_HOST_THREADS. */
BLF_CCM_API int blf_ccm_set_host_threads(blf_ccm_handle* h, int threads);

/* Surface-point forces of ONE contact state held in host memory (twist[6], pose[12],
 * null_pose[12]), for m points xy (device, m*2): force_out / torque_out device m*3 (either may be
 * NULL).  Zero outside |x| <= length/2, |y| <= width/2.  Uses the uniform parameters. */
BLF_CCM_API int blf_ccm_eval_surface_points(blf_ccm_handle* h, const double* host_twist,
                                            const double* host_pose, const double* host_null_pose,
                                            int64_t m, const double* xy, double* force_out,
                                            double* torque_out, void* stream);

/*
 * Sampling-MPC epilogue.  The batch is n_rollouts * rollout_len contact states, rollout-major
 * (all evaluations of a rollout are contiguous).  The evaluation kernel (outputs per out_mask
 * exactly as blf_ccm_eval_batch_soa; out_mask may be 0 to keep only the cost) also reduces the
 * cost per (rollout, tile) in its epilogue, so the wrench is never re-read; a second tiny launch
 * sums each rollout's few partials, i.e.
 *   cost[r] = sum_e  weights[0]*|force_e - wrench_ref[0:3]|^2 + weights[1]*|torque_e - wrench_ref[3:6]|^2
 * per rollout in a fixed order (deterministic), and arg-mins over the local rollouts with
 * lowest-index tie-break.  cost (device, n_rollouts) may be NULL.  best (device, 2 x 8 bytes):
 * best[0] = min cost as double, best[1] = rollout index as int64, offset by index_base (the first
 * global rollout index owned by this rank).
 */
BLF_CCM_API int blf_ccm_rollout_cost_argmin_soa(blf_ccm_handle* h, int64_t n_rollouts,
                                                int64_t rollout_len,
                                                const double* const* in_planes,
                                                const double* const* param_planes,
                                                unsigned out_mask, double* const* wrench_planes,
                                                double* const* autodyn_planes, double* ctrl,
                                                const double* host_wrench_ref,
                                                const double* host_weights, int64_t index_base,
                                                double* cost, void* best, void* stream);

/* Combine per-rank (cost, index) pairs (device, n_pairs x 16 bytes, e.g. the all-gather of every
 * rank's `best`) into the global arg-min with lowest-index tie-break; result to best (device, 16 B). */
BLF_CCM_API int blf_ccm_argmin_pairs(blf_ccm_handle* h, int n_pairs, const void* pairs,
                                     void* best, void* stream);

/* Optional NCCL exchange of the 16-byte (cost,index) pair, for C/C++ hosts that own an
 * ncclComm_t (void* comm).  libnccl is dlopen()ed on first use; BLF_CCM_ERR_NCCL if absent.
 * In-place all-gather of `best` into gathered (device, nranks*16 B) then blf_ccm_argmin_pairs. */
BLF_CCM_API int blf_ccm_argmin_allgather_nccl(blf_ccm_handle* h, void* comm, int nranks,
                                              const void* best, void* gathered, void* global_best,
                                              void* stream);

/*
 * Peer-memory arg-min exchange (NVLink / NVSwitch P2P, one process per GPU on one node): replaces
 * the NCCL all-gather of the 16-byte pair.  Every rank creates a mailbox in its own device memory
 * and gets a CUDA IPC handle for it (BLF_CCM_IPC_HANDLE_BYTES bytes); the ranks exchange the
 * handles by any means (e.g. torch.distributed.all_gather) and connect.  After that ONE single-warp
 * kernel per rank and per exchange stores the rank's pair into every peer's mailbox over NVLink,
 * waits for the peers' pairs in its own mailbox and reduces them with the lowest-index tie-break
 * -- no host round trip, no collective library.  Every rank must call the exchange the same number
 * of times (it is a collective); a peer that never arrives makes the kernel give up after ~2 s and
 * report index -2.  best / global_best: device, 16 bytes {double cost, int64 index}.
 */
enum { BLF_CCM_IPC_HANDLE_BYTES = 64 };
BLF_CCM_API int blf_ccm_p2p_mailbox_create(blf_ccm_handle* h, int nranks, int rank,
                                           void* ipc_handle_out);
BLF_CCM_API int blf_ccm_p2p_mailbox_connect(blf_ccm_handle* h, const void* all_ipc_handles);
BLF_CCM_API int blf_ccm_argmin_exchange_p2p(blf_ccm_handle* h, const void* best,
                                            void* global_best, void* stream);
/* Fuse the exchange into the rollout entry points: with global_best != NULL (device, 16 bytes,
 * 16-byte aligned) every later blf_ccm_rollout_cost_argmin_soa / blf_ccm_rollout_integrate_cost call
 * ALSO runs the peer exchange -- inside the last block of its own cost-reduction kernel, i.e.
 * reduction + collective in one launch -- and writes the global arg-min to global_best (`best`
 * still receives the local one).  NULL switches it off.  Collective semantics as above. */
BLF_CCM_API int blf_ccm_rollout_set_exchange(blf_ccm_handle* h, void* global_best);
BLF_CCM_API int blf_ccm_p2p_mailbox_destroy(blf_ccm_handle* h);

/*
 * Batched Estimators::RecursiveLeastSquare::advance (reference:
 * src/Estimators/src/RecursiveLeastSquare.cpp:96-133), n independent estimators, one step each:
 *   K = P Y^T (lambda R + Y P Y^T)^-1 ; theta += K (z - Y theta) ; P = (P - K Y P) / lambda
 * p parameters, m measurements (1..512 each, as the reference takes any size).  SoA device planes
 * of n doubles: regressor_planes[m*p] (row-major m x p index), measurement_planes[m],
 * state_planes[p] (in/out), cov_planes[p*p] (row-major, in/out).  host_measurement_cov[m] is the
 * diagonal of R (the reference assumes uncorrelated measurements, RecursiveLeastSquare.cpp:38-50).
 * Two code paths, chosen per call: p <= 4, m <= 6 and lambda * R > 0 (S symmetric positive
 * definite) run in registers with an LDL^T factorisation at the HBM roofline; any other size, or a
 * zero / negative lambda * R entry, runs the reference's own algorithm -- inverse of S by LU with
 * partial pivoting -- in a general kernel with global scratch (a singular S gives inf/NaN, as the
 * reference).
 */
BLF_CCM_API int blf_rls_advance_batch(blf_ccm_handle* h, int64_t n, int p, int m,
                                      const double* const* regressor_planes,
                                      const double* const* measurement_planes,
                                      const double* host_measurement_cov, double lambda,
                                      double* const* state_planes, double* const* cov_planes,
                                      void* stream);

/* Same update for n estimators held in HOST arrays (array-of-structures: Y n*(m*p) row-major per
 * estimator, z n*m, theta n*p in/out, P n*(p*p) in/out); what the per-instance
 * RecursiveLeastSquare facade calls with n = 1.  Synchronous. */
BLF_CCM_API int blf_rls_advance_host(blf_ccm_handle* h, int64_t n, int p, int m, const double* Y,
                                     const double* z, const double* host_measurement_cov,
                                     double lambda, double* theta, double* P);

/*
 * Fused identification step for the contact model: per contact, the 6x2 regressor
 * (ContinuousContactModel.cpp:223-254) is computed from the contact state in registers and used at
 * once for one RLS step on theta = [spring_coeff; damper_coeff] with the measured wrench -- the
 * regressor never goes to HBM.  in_planes as in blf_ccm_eval_batch_soa (the 25 planes live for the
 * regressor); geometry_planes = {length, width} planes or NULL for the handle's uniform geometry;
 * measured_wrench_planes[6]; state_planes[2] = spring, damper estimates (in/out); cov_planes[4].
 */
BLF_CCM_API int blf_ccm_rls_advance_contacts(blf_ccm_handle* h, int64_t n,
                                             const double* const* in_planes,
                                             const double* const* geometry_planes,
                                             const double* const* measured_wrench_planes,
                                             const double* host_measurement_cov, double lambda,
                                             double* const* state_planes,
                                             double* const* cov_planes, void* stream);

/*
 * ---- System component: the steps either side of the contact model ------------------------------
 *
 * blf_sys_kinematics_*: System::FloatingBaseSystemKinematics::dynamics (base position + rotation;
 * src/System/src/FloatingBaseSystemKinematics.cpp:36-73)
 *   pos_dot = twist.head<3>();  rot_dot = -R.colwise().cross(w) + rho/2 ((R R^T)^-1 - I) R
 * advanced by System::ForwardEuler (x += dx*dT, src/System/include/BipedalLocomotion/System/
 * ForwardEuler.h:45-53, ForwardEuler.tpp:19-49).  rho is the Baumgarte parameter ("rho" key of
 * FloatingBaseSystemKinematics::initalize, :13-34).  With rho == 0 the inverse is skipped (the
 * reference would turn a singular R into NaN there; this backend leaves it finite).
 */

/* One ForwardEuler step for n independent systems, SoA device planes of n doubles:
 * twist_planes[6] (linear xyz, angular xyz), pos_planes[3] and rot_planes[9] (row-major index)
 * updated in place. */
BLF_CCM_API int blf_sys_kinematics_euler_step_soa(blf_ccm_handle* h, int64_t n, double rho,
                                                  double dT, const double* const* twist_planes,
                                                  double* const* pos_planes,
                                                  double* const* rot_planes, void* stream);

/* dynamics() for n systems held in HOST arrays (what the per-instance facade calls with n = 1):
 * twists n*6, rotations n*9 row-major -> pos_dot n*3, rot_dot n*9.  Synchronous. */
BLF_CCM_API int blf_sys_kinematics_dynamics_host(blf_ccm_handle* h, int64_t n, double rho,
                                                 const double* twists, const double* rotations,
                                                 double* pos_dot, double* rot_dot);

/* The same for arrays already on the device (n*6, n*9 -> n*3, n*9), asynchronous on `stream`: what
 * FloatingBaseDynamicalSystem::dynamics needs beside the acceleration
 * (src/System/src/FloatingBaseSystemDynamics.cpp:134-140, the same formula). */
BLF_CCM_API int blf_sys_kinematics_dynamics(blf_ccm_handle* h, int64_t n, double rho,
                                            const double* twists, const double* rotations,
                                            double* pos_dot, double* rot_dot, void* stream);

/* FixedStepIntegrator::integrate on HOST arrays with a constant control input: n_steps Euler
 * steps, the first n_steps-1 of size step_dT and the last of size last_dT (the caller computes
 * the reference's schedule, FixedStepIntegrator.tpp:48-64).  positions n*3, rotations n*9 in/out;
 * joint_pos (n_joint_values doubles, any layout) += joint_vel * dT per step, NULL/0 for none. */
BLF_CCM_API int blf_sys_kinematics_integrate_host(blf_ccm_handle* h, int64_t n, double rho,
                                                  double step_dT, double last_dT, int n_steps,
                                                  const double* twists, double* positions,
                                                  double* rotations, int64_t n_joint_values,
                                                  const double* joint_vel, double* joint_pos);

/*
 * Fused sampling-MPC rollout: integrate -> contact model -> cost, the pose never leaves registers.
 * chains = n_rollouts * feet, chain c = rollout*feet + foot.  For t = 0..horizon-1 and every chain:
 * the contact model is evaluated at (twist[t][c], pose_c) exactly as blf_ccm_eval_batch_soa would
 * (outputs per out_mask at index t*chains + c: TIME-major), the cost term is accumulated, then
 * pose_c advances by one ForwardEuler step of FloatingBaseSystemKinematics with that twist -- the
 * order in which FloatingBaseDynamicalSystem::dynamics + ForwardEuler visit them.
 *   twist_planes[6]            each horizon*chains doubles, index t*chains + c
 *   pos_planes[3], rot_planes[9]   initial pose per chain (chains doubles each), not modified
 *   null_planes[12]            null-force pose per chain: pos 0-2, rot row-major 3-11; the third
 *                              rotation column (5, 8, 11) may be NULL
 *   param_planes[4]            per-chain length,width,spring,damper, or NULL -> uniform parameters
 *   out_mask                   subset of WRENCH|AUTODYN|CTRL to write as trajectories (0 = none);
 *                              wrench_planes[6], autodyn_planes[6]: horizon*chains; ctrl dense
 *                              horizon*chains*36
 *   final_pos_planes[3], final_rot_planes[9]   pose after the last step, or both NULL
 *   cost[r] = sum_foot ( sum_t  w0|F-Fref|^2 + w1|T-Tref|^2 )  (t inner, in order; then feet in
 *   order: deterministic); cost may be NULL.  best as in blf_ccm_rollout_cost_argmin_soa.
 * Per step only the 48-byte twist (and the requested outputs) cross HBM.
 */
BLF_CCM_API int blf_ccm_rollout_integrate_cost(
    blf_ccm_handle* h, int64_t n_rollouts, int feet, int horizon, double dT, double rho,
    const double* const* twist_planes, const double* const* pos_planes,
    const double* const* rot_planes, const double* const* null_planes,
    const double* const* param_planes, unsigned out_mask, double* const* wrench_planes,
    double* const* autodyn_planes, double* ctrl, double* const* final_pos_planes,
    double* const* final_rot_planes, const double* host_wrench_ref, const double* host_weights,
    int64_t index_base, double* cost, void* best, void* stream);

/* Same rollouts with every plane in HOST memory (pinned gives full PCIe speed), cost only: the
 * horizon is cut into time chunks (contiguous in the time-major planes, so every upload is a plain
 * 1-D copy), pipelined through four slots -- the upload of the next chunk overlaps the kernel of
 * the current one, poses and costs carry over on the device; per evaluation only the 48-byte
 * twist crosses PCIe, one pair comes back.  cost (host, n_rollouts) may be NULL.  Returns when best_cost / best_index are written
 * (index -1 when there is nothing to compare).  Not part of a peer exchange (local arg-min). */
BLF_CCM_API int blf_ccm_rollout_integrate_cost_host(
    blf_ccm_handle* h, int64_t n_rollouts, int feet, int horizon, double dT, double rho,
    const double* const* twist_planes, const double* const* pos_planes,
    const double* const* rot_planes, const double* const* null_planes,
    const double* const* param_planes, const double* host_wrench_ref, const double* host_weights,
    double* cost, double* best_cost, int64_t* best_index);

/*
 * Contact part of FloatingBaseDynamicalSystem::dynamics
 * (src/System/src/FloatingBaseSystemDynamics.cpp:199-226): per system s
 *   out[s] = base[s] + sum_{c < contacts_per_system, in order}  J_c^T * wrench_c
 * wrench_c = getContactWrench() of contact s*contacts_per_system + c, evaluated from the SoA state
 * planes in registers (in_planes / param_planes as blf_ccm_eval_batch_soa with out_mask WRENCH);
 * J_c = 6 x ncols row-major frame Jacobian (iDynTree::MatrixDynSize), jacobians =
 * n_systems*contacts_per_system*6*ncols doubles; base (NULL = zeros; the reference starts from the
 * negated bias forces, :191-196) and out are n_systems*ncols; base may alias out.
 * wrench_planes[6] optional (NULL): also write the wrenches.  contacts_per_system 1..32,
 * ncols 1..128.  jacobians 16-byte aligned -> TMA ring, else direct loads (blf_ccm_last_path).
 */
BLF_CCM_API int blf_ccm_generalized_force_soa(blf_ccm_handle* h, int64_t n_systems,
                                              int contacts_per_system, int ncols,
                                              const double* const* in_planes,
                                              const double* const* param_planes,
                                              const double* jacobians, const double* base,
                                              double* out, double* const* wrench_planes,
                                              void* stream);

/*
 * Last step of FloatingBaseDynamicalSystem::dynamics
 * (src/System/src/FloatingBaseSystemDynamics.cpp:226-248), n_systems independent systems of
 * ncols = 6 + actuated DoFs unknowns:
 *   rhs[s] = known[s];  rhs[s][6 ..] += joint_torques[s]                               (:226-227)
 *   acc[s] = (mass[s] + regularization).llt().solve(rhs[s])                            (:235-243)
 * mass: n_systems*ncols*ncols doubles, row-major per system (iDynTree::MatrixDynSize as
 * getFreeFloatingMassMatrix fills it); like Eigen's LLT only the LOWER triangle is read.
 * regularization: ncols*ncols row-major DEVICE array shared by all systems (what
 * setMassMatrixRegularization stores, :72-95) or NULL.  known, acc: n_systems*ncols (acc may alias
 * known); joint_torques: n_systems*(ncols-6) or NULL.  ncols 1..128: up to 64 a warp-level kernel
 * (rows in registers), above a block-level one (blf_ccm_last_path tells which).  A matrix that is
 * not positive definite yields NaN for that system (the reference's Eigen stops factorising and
 * solves with the partial factor: meaningless numbers, no error there either).
 */
BLF_CCM_API int blf_sys_mass_matrix_solve(blf_ccm_handle* h, int64_t n_systems, int ncols,
                                          const double* mass, const double* regularization,
                                          const double* known, const double* joint_torques,
                                          double* acc, void* stream);

/*
 * FloatingBaseDynamicalSystem::dynamics from the bias forces on (:188-248), the rigid-body
 * quantities (mass matrix, bias forces, frame Jacobians, frame poses/twists: iDynTree
 * KinDynComputations in the reference) supplied by the caller:
 *   known = -bias_forces + sum_c J_c^T wrench_c ;  known[6 ..] += joint_torques ;
 *   acc   = (mass + regularization).llt().solve(known)         = [base acc (6); joint acc]
 * Arguments as blf_ccm_generalized_force_soa (in_planes, param_planes, jacobians, wrench_planes)
 * and blf_sys_mass_matrix_solve (mass, regularization, joint_torques); bias_forces =
 * n_systems*ncols, [base wrench (6); joint torques] of generalizedBiasForces; ncols >= 6.
 * Two launches on `stream` (J^T wrench accumulation into acc, then the solve in place).
 */
BLF_CCM_API int blf_sys_floating_base_acceleration(
    blf_ccm_handle* h, int64_t n_systems, int contacts_per_system, int ncols,
    const double* const* in_planes, const double* const* param_planes, const double* jacobians,
    const double* bias_forces, const double* joint_torques, const double* mass,
    const double* regularization, double* acc, double* const* wrench_planes, void* stream);

/*
 * One ForwardEuler step of FloatingBaseDynamicalSystem
 * (src/System/include/BipedalLocomotion/System/ForwardEuler.tpp:19-49, x = x0 + dx * dT over the state
 * tuple of FloatingBaseSystemDynamics.h:33-52), every derivative taken at the state BEFORE the step:
 *   base_pos += nu[0..2] * dT;  base_rot += (rotation rate of FloatingBaseSystemDynamics.cpp:139-145,
 *   rho = the Baumgarte parameter of initalize, :17-37) * dT;  joint_pos += nu[6..] * dT;  nu += acc * dT
 * acc = what blf_sys_floating_base_acceleration returned for that state.  Per-system arrays as the
 * reference holds them: acc, nu n_systems*ncols ([base (6); joints]); joint_pos n_systems*(ncols-6)
 * (NULL when ncols == 6); base_pos n_systems*3; base_rot n_systems*9 row-major; all but acc updated
 * in place.  ncols 6..128.  With rho == 0 the Baumgarte term is skipped (as blf_sys_kinematics_*).
 * 8-byte alignment is enough; when all five arrays are 16-byte aligned (any cudaMalloc'ed array is) the
 * tiles move by bulk copies, the fast route.  acc must not alias nu.  One launch on `stream`.
 */
BLF_CCM_API int blf_sys_floating_base_euler_step(blf_ccm_handle* h, int64_t n_systems, int ncols,
                                                 double rho, double dT, const double* acc, double* nu,
                                                 double* joint_pos, double* base_pos, double* base_rot,
                                                 void* stream);

/*
 * Device / pinned-host memory and stream helpers, so that host code above this ABI (the C++17
 * facade, the device-side SoA container) needs no CUDA headers.  Device allocations are 256-byte
 * aligned.  Copies are asynchronous on `stream` when the host side is pinned.
 */
BLF_CCM_API int blf_ccm_device_alloc(blf_ccm_handle* h, uint64_t bytes, void** out);
/* Frees memory from blf_ccm_device_alloc or blf_ccm_device_alloc_compressible.  A compressible
 * allocation is released after a device synchronise (the driver's unmap, unlike cudaFree, does not
 * wait for kernels still using it). */
BLF_CCM_API int blf_ccm_device_free(blf_ccm_handle* h, void* ptr);
/*
 * Device memory with Compute Data Compression requested (cuMemCreate, CU_MEM_ALLOCATION_COMP_GENERIC),
 * meant for the dense n x 36 control-matrix array: 24 of its 36 entries are structural +0.0, and the
 * memory system can keep such data compressed between L2 and HBM.  Compression is invisible to every
 * reader (kernels, copies): the values are the ones written.  *granted (may be NULL) is 1 when the
 * driver granted compression; when the device has no compression or the driver does not grant it,
 * the memory comes from cudaMalloc and *granted is 0.  The size is rounded up to the allocation
 * granularity; the base is at least 256-byte aligned.  Free with blf_ccm_device_free.
 */
BLF_CCM_API int blf_ccm_device_alloc_compressible(blf_ccm_handle* h, uint64_t bytes, void** out,
                                                  int* granted);
/* *out = 1 when ptr lies inside a live compressible allocation of this handle, else 0. */
BLF_CCM_API int blf_ccm_pointer_is_compressible(blf_ccm_handle* h, const void* ptr, int* out);
BLF_CCM_API int blf_ccm_host_alloc(blf_ccm_handle* h, uint64_t bytes, void** out); /* pinned */
BLF_CCM_API int blf_ccm_host_free(blf_ccm_handle* h, void* ptr);
BLF_CCM_API int blf_ccm_copy_h2d(blf_ccm_handle* h, void* dst_device, const void* src_host,
                                 uint64_t bytes, void* stream);
BLF_CCM_API int blf_ccm_copy_d2h(blf_ccm_handle* h, void* dst_host, const void* src_device,
                                 uint64_t bytes, void* stream);
BLF_CCM_API int blf_ccm_stream_synchronize(blf_ccm_handle* h, void* stream);

/* Introspection */
BLF_CCM_API int blf_ccm_last_path(const blf_ccm_handle* h);
BLF_CCM_API int64_t blf_ccm_launch_count(const blf_ccm_handle* h); /* kernels launched so far */
BLF_CCM_API int blf_ccm_device(const blf_ccm_handle* h);
BLF_CCM_API int blf_ccm_sm_count(const blf_ccm_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* BLF_CCM_H */
