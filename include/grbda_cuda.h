/* grbda_cuda — C ABI of the B200-native batched ClusterTreeModel dynamics path.
 *
 * The reference (ROAM-Lab-ND/generalized_rbda) has no FFI: its boundary is the C++ class
 * grbda::ClusterTreeModel. Every entry point below names the reference interface it replaces
 * (paths relative to the reference repository). A maintainer binds the reference to this library
 * by walking an existing ClusterTreeModel into a grbda_schedule_t (INTEGRATION.md shows the code)
 * and calling the batched functions instead of looping over setState()/inverseDynamics().
 *
 * Conventions
 *   - every function returns a grbda_status (0 = ok); no exception crosses the boundary; the
 *     message of the last error of the calling thread is grbda_cuda_last_error_string()
 *     (the reference throws std::runtime_error, e.g. src/Dynamics/ClusterJoints/ClusterJoint.cpp:41-48);
 *   - batched arrays hold one state per column, contiguous per state: element i of state b of an
 *     array with n entries per state is x[b * n + i];
 *   - q uses the layout of ClusterTreeModel::setState (src/Dynamics/ClusterTreeModel.cpp:256-308):
 *     concatenation over clusters of num_positions_ entries — [p(3); quat w,x,y,z] for a free
 *     base, independent angles for explicit clusters, ALL spanning angles for clusters with an
 *     implicit loop constraint (they must satisfy phi(q) = 0, GenericJoint.cpp:246-249);
 *     yd / ydd / tau are the independent velocities / accelerations / generalized forces;
 *   - `_f64` / `_f32` entry points take DEVICE pointers and are asynchronous on `stream`
 *     (a cudaStream_t passed as void*, NULL = default stream); `_host` entry points take HOST
 *     pointers and return when the results are in the host buffers: page-locked buffers are used in
 *     place (copies and kernels of consecutive chunks overlap), pageable buffers are staged chunk by
 *     chunk through pinned memory the handle owns;
 *   - a batched call enqueues two kernels on `stream` (the straight-line kernel and a normally empty
 *     pass that recomputes 128-state tiles holding a joint angle beyond 1e12 rad with the library
 *     sin/cos) and uses a small scratch buffer that the model handle keeps per stream: calls on
 *     different streams may overlap, calls can be captured in CUDA graphs after one warm-up call;
 *   - there is no CPU implementation behind this API: without a CUDA device calls fail with
 *     GRBDA_ERR_NO_DEVICE; a model without ahead-of-time kernels is compiled at run time (below),
 *     and fails with GRBDA_ERR_NOT_COMPILED if that is disabled or impossible.
 */
#ifndef GRBDA_CUDA_H
#define GRBDA_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef int grbda_status;
enum
{
    GRBDA_OK = 0,
    GRBDA_ERR_INVALID_ARGUMENT = 1,
    GRBDA_ERR_INVALID_MODEL = 2,  /* model description violates a ClusterTreeModel rule          */
    GRBDA_ERR_NOT_COMPILED = 3,   /* no sm_100a kernels were built for this model                */
    GRBDA_ERR_NO_DEVICE = 4,
    GRBDA_ERR_CUDA = 5,
    GRBDA_ERR_IO = 6,
    GRBDA_ERR_INTERNAL = 7
};

/* cluster_type values (what the reference's ClusterJoints classes reduce to for the kernels) */
enum
{
    GRBDA_CLUSTER_FREE_QUATERNION = 0, /* ClusterJoints::Free<.., ori_representation::Quaternion>  */
    GRBDA_CLUSTER_FREE_RPY = 1,        /* ClusterJoints::Free<.., ori_representation::RollPitchYaw> */
    GRBDA_CLUSTER_EXPLICIT = 2,        /* Revolute, RevoluteWithRotor, RevolutePair(WithRotor),
                                          RevoluteTripleWithRotor, Generic + LoopConstraint::Static */
    GRBDA_CLUSTER_IMPLICIT = 3         /* Generic + LoopConstraint::GenericImplicit / FourBar       */
};

/* One op of the straight-line program of an implicit constraint phi(q_spanning).
 * op: 0 const(val) 1 input(b = spanning coordinate) 2 add 3 sub 4 mul 5 div 6 neg 7 sin 8 cos;
 * a, b index earlier ops of the same cluster's program. Replaces the casadi::SX lambda handed to
 * LoopConstraint::GenericImplicit (include/grbda/Dynamics/ClusterJoints/GenericJoint.h). */
typedef struct grbda_phi_op
{
    int32_t op, a, b;
    double val;
} grbda_phi_op;

/* Flattened structure-of-arrays topology schedule of one ClusterTreeModel.
 * Replaces: Body (include/grbda/Dynamics/Body.h:12-43), ClusterTreeNode / TreeNode
 * (Nodes/ClusterTreeNode.h:12-55, Nodes/TreeNode.h:16-75) and the per-type ClusterJoints data.
 * Bodies are listed in registration order (= body index); the bodies of a cluster are contiguous.
 * All arrays are caller-owned and copied by grbda_cuda_model_create. */
typedef struct grbda_schedule
{
    int32_t num_bodies;
    int32_t num_clusters;
    double gravity[3];                  /* TreeModel::setGravity, TreeModel.h:56                  */

    /* per body */
    const int32_t *body_parent;         /* Body::parent_index_, -1 = ground                       */
    const int32_t *body_joint_axis;     /* 0/1/2 = ori::CoordinateAxis X/Y/Z (ignored for free)   */
    const double *body_xtree_E;         /* 9 per body, row-major rotation of Body::Xtree_         */
    const double *body_xtree_r;         /* 3 per body, translation of Body::Xtree_                */
    const double *body_inertia;         /* 36 per body, row-major SpatialInertia::getMatrix()     */
    const uint8_t *body_independent;    /* implicit clusters: 1 = independent spanning coordinate */

    /* per cluster */
    const int32_t *cluster_type;        /* GRBDA_CLUSTER_*                                        */
    const int32_t *cluster_num_bodies;
    const int32_t *cluster_num_independent; /* ClusterJoints::Base::numVelocities()               */
    const int32_t *cluster_G_offset;    /* explicit: offset into G_values of the row-major
                                           (num_bodies x num_independent) LoopConstraint G        */
    const double *G_values;
    const int32_t *cluster_phi_offset;  /* implicit: first op of the cluster's phi program        */
    const int32_t *cluster_phi_count;   /* implicit: number of ops                                */
    const int32_t *cluster_phi_out_offset; /* implicit: offset into phi_outputs                   */
    const int32_t *cluster_num_constraints;
    const grbda_phi_op *phi_ops;
    const int32_t *phi_outputs;         /* op index (within the cluster program) of each phi row  */
} grbda_schedule;

typedef struct grbda_model grbda_model; /* opaque; immutable after creation; one per device       */

const char *grbda_cuda_last_error_string(void);
const char *grbda_cuda_version(void);

/* ---- model creation ------------------------------------------------------------------------ */
/* From a schedule. Replaces the registerBody / appendRegisteredBodiesAsCluster construction
 * sequence, src/Dynamics/ClusterTreeModel.cpp:9-67. device < 0: host-only handle (introspection). */
grbda_status grbda_cuda_model_create(const grbda_schedule *schedule, int device, grbda_model **out);
/* From a URDF+ file. Replaces ClusterTreeModel(const std::string &urdf_filename),
 * include/grbda/Dynamics/ClusterTreeModel.h:33-46 + src/Dynamics/ClusterTreeParsing.cpp. */
grbda_status grbda_cuda_model_create_from_urdf(const char *urdf_path, int device, grbda_model **out);
/* From several URDF+ files that together describe one robot (every file names the links it attaches to as empty
 * <link/> stubs). Replaces buildModelFromURDF(const std::vector<std::string> &urdf_filenames),
 * include/grbda/Dynamics/ClusterTreeModel.h:48-53 (UnitTests/testUrdfParser.cpp:398-445). */
grbda_status grbda_cuda_model_create_from_urdfs(const char *const *urdf_paths, int num_paths, int device,
                                                grbda_model **out);
/* The front end's reading of the file(s) as JSON text: link order, parent / children / loop links / supporting chain
 * of every link, clusters with parent and child clusters - the quantities UnitTests/testUrdfParser.cpp:39-396 checks
 * of the parser. Call with json = NULL to get the size in *needed. No GPU involved. */
grbda_status grbda_cuda_describe_urdf(const char *const *urdf_paths, int num_paths, char *json, int64_t capacity,
                                      int64_t *needed);
/* From one of the reference's robot classes (include/grbda/Robots): "tello", "tello_with_arms",
 * "mini_cheetah", "mit_humanoid", "revolute_chain_with_rotor_<N>",
 * "revolute_pair_chain_with_rotor_<N>", or a URDF name from robot-models ("four_bar", ...). */
grbda_status grbda_cuda_model_create_from_robot(const char *name, int device, grbda_model **out);
grbda_status grbda_cuda_model_destroy(grbda_model *model);

/* ---- introspection (TreeModel.h:25-28, ClusterTreeModel.h:97,151-153) ---------------------- */
int grbda_cuda_num_positions(const grbda_model *m);          /* getNumPositions()                 */
int grbda_cuda_num_degrees_of_freedom(const grbda_model *m); /* getNumDegreesOfFreedom()          */
int grbda_cuda_num_bodies(const grbda_model *m);             /* getNumBodies()                    */
int grbda_cuda_num_clusters(const grbda_model *m);           /* clusters().size()                 */
uint64_t grbda_cuda_model_hash(const grbda_model *m);
/* cluster: info[8] = {parent, num_bodies, num_positions, num_velocities, position_index,
 * velocity_index, cluster_type, first_body}; type_name64: ClusterJoints class name. */
grbda_status grbda_cuda_cluster_info(const grbda_model *m, int cluster, int32_t *info8, char *type_name64);
/* body: info[4] = {parent, cluster, sub_index_within_cluster, joint_axis} */
grbda_status grbda_cuda_body_info(const grbda_model *m, int body, char *name64, int32_t *info4,
                                  double *xtree_E9, double *xtree_r3, double *inertia36);
grbda_status grbda_cuda_model_gravity(const grbda_model *m, double *gravity3);
/* implicit cluster: its phi program and independence flags. Pass ops = NULL to query the sizes:
 * sizes2 = {number of ops, number of phi rows}. */
grbda_status grbda_cuda_cluster_phi(const grbda_model *m, int cluster, grbda_phi_op *ops, int32_t *outputs,
                                    uint8_t *independent, int32_t *sizes2);
/* explicit cluster: G (num_bodies x num_independent, row-major) */
grbda_status grbda_cuda_cluster_G(const grbda_model *m, int cluster, double *G);
/* Emitted program of one algorithm (0 ID, 1 FD (articulated-body sweep), 2 FK, 3 H, 4 phi/Kd,
 * 5 / 6 tau_in +/- J^T f_ext, 7 FD as H^-1 (tau - C): cluster CRBA + RNEA bias + branch-sparse L^T D L,
 * 8-11 operational space, 12 / 13 ID / FD Jacobians, 14 / 15 ID / FD vector-Jacobian products, 16 / 17 the
 * vector-Jacobian products of programs 5 / 6 (in: q, f_ext, w; out: q_bar, f_bar), 18 the one of contact kinematics
 * (in: q, yd, [p_bar; v_bar]; out: q_bar, yd_bar)) written as a binary tape to
 * `path` (format: csrc/compiler/compile.h); counts[8] = {nodes, add, mul, div, sqrt, sin, cos,
 * fusable mul+add pairs} of the straight-line program each thread executes. */
grbda_status grbda_cuda_dump_program(const grbda_model *m, int algo, const char *path, int64_t *counts8);

/* The CUDA source the model compiler emits for one program (0 ID, 1 FD, 2 FK, 3 H, 4 phi, 5/6 external-force programs, 7 FD/LTDL):
 * constant table + `struct Body` (sizes, generated range check, run<real, FAST>()), exactly what
 * build.py feeds to nvcc, written to `path`. park != 0: the variant that parks long-lived values in the
 * thread's shared-memory tile row; park = 1 + n: with a park area of n more slots per thread behind the tiles
 * (kernels/shapes.h shapeParkBytes). Used by the emitter self test, which compiles this text for the
 * host with the kernel-side helpers stubbed (tests/host_body_prelude.h) and compares with the oracle. */
grbda_status grbda_cuda_emit_source(const grbda_model *m, int program, int park, const char *path);

/* Operation counts (same 8 fields) of the program the DEFAULT compiled kernel of entry point `algo`
 * (0 ID, 1 FD, 2 FK, 3 H, 4 phi, 5 gfa, 6 gfs) executes per state. It can differ from dump_program(algo): the default
 * forward-dynamics kernel of a model may run program 7 (CRBA + bias + sparse L^T D L) instead of the
 * articulated-body sweep (program 1); both are ClusterTreeModel::forwardDynamics
 * (ClusterTreeDynamics.cpp:10-19 / :59-155) up to rounding. */
grbda_status grbda_cuda_kernel_counts(const grbda_model *m, int algo, int64_t *counts8);

/* ---- kernel provenance / run-time compilation ------------------------------------------------- */
/* A model that build.py did not compile ahead of time gets its kernels from the same model compiler
 * at run time: NVRTC builds the emitted program for sm_100a when an entry point is first used and
 * the cubin is cached on disk (GRBDA_CACHE_DIR, default ~/.cache/grbda_cuda). This is what lets
 * grbda_cuda_model_create / _from_urdf accept ANY ClusterTreeModel, as the reference's constructors
 * do (include/grbda/Dynamics/ClusterTreeModel.h:27-53). GRBDA_JIT=0 turns it off (create then fails
 * with GRBDA_ERR_NOT_COMPILED), GRBDA_JIT=force ignores the ahead-of-time kernels.
 * prepare: compile / load the kernels of one entry point now (algo 0 ID, 1 FD, 2 FK, 3 H, 4 phi,
 * 5 gfa, 6 gfs, 19 contact forward dynamics, 20 contact impulse (FP64, for the current contact set),
 * GRBDA_PROGRAM_INTEGRATE_VJP) instead of on first use, e.g. before capturing a CUDA graph. */
grbda_status grbda_cuda_model_prepare(const grbda_model *m, int algo, int f32);
/* Program id of the reverse integration step (grbda_cuda_integrate_vjp_f64) for grbda_cuda_model_prepare and
 * grbda_cuda_jit_compile; it is compiled at run time for every model, also for those built ahead of time. */
#define GRBDA_PROGRAM_INTEGRATE_VJP (-2)
/* info8 = {source (0 ahead of time, 1 run-time compiled), CTA size, CTAs per SM, dynamic shared
 * memory, program, flags (1 parked, 2 bulk-copy staged, 4 direct I/O, 8 loaded from the disk cache),
 * NVRTC milliseconds, ready}; fields 1-6 are reported for run-time compiled kernels only. */
grbda_status grbda_cuda_kernel_info(const grbda_model *m, int algo, int f32, int64_t *info8);
/* The run-time compiler without a device: writes the CUDA text of one entry point (algo -1: the
 * state generator, GRBDA_PROGRAM_INTEGRATE_VJP: the reverse integration step) to source_path and / or the sm_100a
 * cubin NVRTC makes of it to cubin_path. */
grbda_status grbda_cuda_jit_compile(const grbda_model *m, int algo, int f32, const char *source_path,
                                    const char *cubin_path);

/* ---- batched hot path, device pointers ----------------------------------------------------- */
/* tau = ID(q, yd, ydd). Replaces setState + ClusterTreeModel::inverseDynamics(ydd),
 * src/Dynamics/ClusterTreeDynamics.cpp:79-83 -> TreeModel.cpp:174-212. */
grbda_status grbda_cuda_inverse_dynamics_f64(const grbda_model *m, const double *q, const double *yd,
                                             const double *ydd, double *tau, int64_t batch, void *stream);
grbda_status grbda_cuda_inverse_dynamics_f32(const grbda_model *m, const float *q, const float *yd,
                                             const float *ydd, float *tau, int64_t batch, void *stream);
/* External forces (TreeModel::setExternalForces, src/Dynamics/TreeModel.cpp:215-239; applied at
 * TreeModel.cpp:189-193 and ClusterTreeDynamics.cpp:100-105). By default on the model's terminal links
 * (leaf bodies that are not motor rotors: feet, hands, chain tips), or on the set chosen with
 * grbda_cuda_set_external_force_bodies: body_indices receives the body indices in the order the
 * f_ext arrays use; pass body_indices = NULL to query the count.
 * f_ext[batch][count][6] = one spatial force [n; f] per listed body, in WORLD coordinates as the
 * reference takes them. f_ext = NULL means no external forces. */
grbda_status grbda_cuda_external_force_bodies(const grbda_model *m, int32_t *body_indices, int32_t *count);
/* Choose the bodies that take external forces: ANY distinct bodies of the model (the reference's test
 * puts a force on every body, UnitTests/testRigidBodyDynamicsAlgos.cpp:201-236); count = 0 restores
 * the default (terminal links). The force programs are specialised for the set and compiled at run
 * time when it is first used. Not to be called while launches on this handle are in flight (it is the
 * one mutating call of an otherwise immutable handle; it synchronises the device). */
grbda_status grbda_cuda_set_external_force_bodies(grbda_model *m, const int32_t *body_indices, int32_t count);
grbda_status grbda_cuda_inverse_dynamics_ext_f64(const grbda_model *m, const double *q, const double *yd,
                                                 const double *ydd, const double *f_ext, double *tau,
                                                 int64_t batch, void *stream);
grbda_status grbda_cuda_forward_dynamics_ext_f64(const grbda_model *m, const double *q, const double *yd,
                                                 const double *tau, const double *f_ext, double *ydd,
                                                 int64_t batch, void *stream);
/* ---- operational space: contact points, Jacobians, apply-test-force, inverse OSIM ------------------ */
/* Contact points of the model (TreeModel::appendContactPoint / appendEndEffector,
 * src/Dynamics/ClusterTreeModel.cpp:129-190): body index, offset in the body frame, end-effector flag
 * (NULL: none is). Replaces any earlier set; the programs below are specialised for it and compiled at
 * run time when first used. Like grbda_cuda_set_external_force_bodies it mutates the handle. */
grbda_status grbda_cuda_set_contact_points(grbda_model *m, int32_t count, const int32_t *body_indices,
                                           const double *local_offsets, const uint8_t *is_end_effector);
int grbda_cuda_num_contact_points(const grbda_model *m);
int grbda_cuda_num_end_effectors(const grbda_model *m);
/* p[batch][n_cp][3] world position, v[batch][n_cp][3] world linear velocity of every contact point.
 * Replaces setState + contactPointForwardKinematics, src/Dynamics/TreeModel.cpp:60-78. */
grbda_status grbda_cuda_contact_kinematics_f64(const grbda_model *m, const double *q, const double *yd, double *p,
                                               double *v, int64_t batch, void *stream);
/* J[batch][n_cp][6][nv]: world-frame contact Jacobians, rows [angular; linear]. Replaces
 * contactJacobianWorldFrame, src/Dynamics/ClusterTreeDynamics.cpp:10-45. */
grbda_status grbda_cuda_contact_jacobians_f64(const grbda_model *m, const double *q, double *J, int64_t batch,
                                              void *stream);
/* For a world-frame force[batch][n_cp][3] on each contact point (one at a time): dstate[batch][n_cp][nv]
 * = H^-1 J_lin^T f and lambda_inv[batch][n_cp] = f^T J_lin H^-1 J_lin^T f. Replaces applyTestForce,
 * src/Dynamics/ClusterTreeDynamics.cpp:193-290. */
grbda_status grbda_cuda_apply_test_force_f64(const grbda_model *m, const double *q, const double *force,
                                             double *dstate, double *lambda_inv, int64_t batch, void *stream);
/* lambda_inv[batch][6 n_ee][6 n_ee] = J H^-1 J^T over the end-effectors (6-row Jacobians in the
 * orientation of their body, at the contact point). Replaces inverseOperationalSpaceInertiaMatrix
 * (the extended force propagator algorithm), src/Dynamics/ClusterTreeDynamics.cpp:292-435. */
grbda_status grbda_cuda_inverse_osim_f64(const grbda_model *m, const double *q, double *lambda_inv, int64_t batch,
                                         void *stream);
/* ---- rigid point contacts: contact-constrained forward dynamics and contact impulses --------------------------- */
/* The contact points are those of grbda_cuda_set_contact_points, n_c of them, m = 3 n_c. J (m x nv) stacks the LINEAR
 * rows (3..5) of each contact's world-frame Jacobian, as applyTestForce uses them. active[batch][n_c] is a per-state
 * activity mask s (nonzero = active; active = NULL: all active), S = diag(s (x) 1_3); damping eps >= 0 is one value per
 * call. c = Jdot yd is the classical world-frame acceleration of every contact point at ydd = 0, WITHOUT gravity: with
 * (w, v_o) the spatial velocity and (wdot, a_o) the spatial acceleration of the body (body coordinates, ydd = 0, zero
 * gravity), d the offset and E the body's rotation (world -> body),
 *   c_k = E^T (a_o + w x v_o + wdot x d + w x (w x d)).
 * Both entry points share
 *   Y = H^-1 J^T (m solves with one factorisation),   A = S (J Y) S + (I - S) + eps I,
 * and solve A x = b with an unrolled LDL^T of the m x m matrix.
 * Contact-constrained forward dynamics: tau[batch][nv] in, ydd[batch][nv] and lambda[batch][n_c][3] out:
 *   ydd0 = H^-1 (tau - C) (what grbda_cuda_forward_dynamics_f64 returns),  b = -S (J ydd0 + c),
 *   lambda = A^-1 b,  ydd = ydd0 + Y lambda.
 * lambda is the world-frame force applied to the robot at each contact point. The result satisfies H ydd + C =
 * tau + J^T lambda; J_a ydd + c_a = -eps lambda_a for the active contacts; lambda = 0 exactly for the inactive ones
 * (their rows and columns of A and their entries of b are exact zeros, which the factorisation keeps while the values
 * are finite).
 * Contact impulse: yd[batch][nv] is the velocity before the impact, yd_plus[batch][nv] the velocity after it and
 * impulse[batch][n_c][3] the world-frame impulse at each contact point; restitution e in [0, 1]:
 *   b = -(1 + e) S J yd,  impulse = A^-1 b,  yd_plus = yd + Y impulse,
 * so that J_a yd_plus = -e J_a yd - eps impulse_a and impulse = 0 for the inactive contacts.
 * The factorisation has no pivoting (the program is straight-line): with eps = 0 the active rows of J must be linearly
 * independent. Two or more points on one rigid body (toe and heel of one foot: 6 rows of rank 5) are not, and need
 * eps > 0; the equations above then hold with that eps.
 * FP64 only. The programs are specialised for the contact set and compiled at run time when first used (GRBDA_JIT=0:
 * GRBDA_ERR_NOT_COMPILED). One hand-written kernel packs [tau; s; eps] (contact dynamics) or [s; e; eps] (impulse) per
 * state into the per-stream scratch buffer of the VJP entry points on `stream`, then the program runs on `stream`; that
 * buffer belongs to the (handle, stream) pair, with the same concurrency caveat. Refused with
 * GRBDA_ERR_INVALID_ARGUMENT: a model without contact points, batch < 0, a NULL pointer other than `active`, eps < 0
 * or not finite, e outside [0, 1]; GRBDA_ERR_NO_DEVICE for a host-only handle. batch = 0 returns GRBDA_OK without
 * launching anything. */
grbda_status grbda_cuda_contact_forward_dynamics_f64(const grbda_model *m, const double *q, const double *yd,
                                                     const double *tau, const uint8_t *active, double damping,
                                                     double *ydd, double *lambda, int64_t batch, void *stream);
grbda_status grbda_cuda_contact_impulse_f64(const grbda_model *m, const double *q, const double *yd,
                                            const uint8_t *active, double restitution, double damping, double *yd_plus,
                                            double *impulse, int64_t batch, void *stream);

/* Derivatives of the dynamics (SURVEY 8 f4). The reference has no closed-form derivative algorithm: it takes
 * CasADi's jacobian() of its symbolic model with respect to a tangent-space perturbation dq of the positions, the
 * velocities and the third argument (UnitTests/testRigidBodyDynamicsAlgosDerivatives.cpp:126-155, 339-383;
 * q (+) dq = UnitTests/testHelpers.hpp:50-112: q + dq per one-dof coordinate, floating base
 * [p + R^T dp; quat + 1/2 quat (x) (0, dw)] with dq = [dw; dp]; clusters with an implicit loop constraint move along
 * the constraint manifold, dq_span = G dy). These entry points evaluate the same Jacobians, generated by
 * differentiating the model's compiled program; all matrices are nv x nv, COLUMN-major as Eigen / CasADi store
 * them: element [j * nv + i] = d out_i / d x_j (one contiguous column per perturbed coordinate).
 * The programs are compiled at run time when first used.
 *   inverse dynamics: dtau_dq, dtau_dyd  (d tau / d ydd is grbda_cuda_mass_matrix_f64)
 *   forward dynamics: dydd_dq, dydd_dyd, dydd_dtau (= H^-1) */
grbda_status grbda_cuda_inverse_dynamics_derivatives_f64(const grbda_model *m, const double *q, const double *yd,
                                                         const double *ydd, double *dtau_dq, double *dtau_dyd,
                                                         int64_t batch, void *stream);
grbda_status grbda_cuda_forward_dynamics_derivatives_f64(const grbda_model *m, const double *q, const double *yd,
                                                         const double *tau, double *dydd_dq, double *dydd_dyd,
                                                         double *dydd_dtau, int64_t batch, void *stream);

/* Reverse mode: vector-Jacobian products of the dynamics, what the gradient of a scalar loss of tau or ydd needs
 * (the torch.autograd functions of the Python package call them). For a cotangent w[batch][nv] of the output:
 *   inverse dynamics: q_bar = w^T d tau / d q, yd_bar = w^T d tau / d yd, ydd_bar = H w
 *   forward dynamics: q_bar = w^T d ydd / d q, yd_bar = w^T d ydd / d yd, tau_bar = H^-1 w
 * One reverse sweep of the model's compiled program per state; the outputs are nq + 2 nv values per state instead
 * of the 2-3 nv x nv matrices of the Jacobian entry points. q_bar[batch][nq] is the gradient with respect to the
 * STORED position entries, q_bar[k] = sum_i w_i d out_i / d q[k]:
 *   inverse dynamics: the exact derivative of the inverse-dynamics program for every entry;
 *   forward dynamics: contracted with any direction that keeps quaternions unit and implicit clusters on phi = 0,
 *     it equals w^T times the tangent Jacobian of grbda_cuda_forward_dynamics_derivatives_f64; its component
 *     normal to that set is the one of -H^-1 d ID / d q (implicit function theorem), not the derivative of one
 *     particular forward-dynamics kernel off the set.
 * FP64 only; the programs are compiled at run time when first used. The two per-state input arrays of the third
 * argument are packed into [batch][2 nv] in a per-stream scratch buffer of the handle with two device-to-device
 * copies on `stream`, then the kernel runs on `stream`. batch = 0 returns GRBDA_OK without launching anything.
 * That buffer belongs to the (handle, stream) pair, as the intermediate buffer of the *_ext entry points does: calls
 * on ONE stream of one handle from several host threads at once are not supported (their copies and kernels may
 * interleave); give each thread its own stream. */
grbda_status grbda_cuda_inverse_dynamics_vjp_f64(const grbda_model *m, const double *q, const double *yd,
                                                 const double *ydd, const double *tau_bar, double *q_bar,
                                                 double *yd_bar, double *ydd_bar, int64_t batch, void *stream);
grbda_status grbda_cuda_forward_dynamics_vjp_f64(const grbda_model *m, const double *q, const double *yd,
                                                 const double *tau, const double *ydd_bar, double *q_bar,
                                                 double *yd_bar, double *tau_bar, int64_t batch, void *stream);
/* The same with external forces f_ext[batch][nf][6] on grbda_cuda_external_force_bodies (as the *_ext entry points
 * take them); f_bar[batch][nf][6] receives their cotangent. f_ext = NULL means no external forces: the call is then
 * exactly the VJP above and f_bar is not written (it may be NULL).
 *   inverse dynamics, tau = ID(q, yd, ydd) - J^T f: q_bar, yd_bar, ydd_bar = H tau_bar as above, f_bar = -J tau_bar.
 *     Launches: the ID VJP (two copies + one kernel), the program of -J^T f reversed (q contribution to a per-stream
 *     scratch buffer of nq doubles per state), one elementwise kernel that adds it to q_bar.
 *   forward dynamics, ydd = FD(q, yd, tau + J^T f): tau_bar = H^-1 ydd_bar, f_bar = J tau_bar. Launches: tau + J^T f
 *     into a scratch buffer (what grbda_cuda_forward_dynamics_ext_f64 runs), the FD VJP at that torque (two copies +
 *     one kernel), the program of J^T f reversed with tau_bar, one elementwise kernel that adds its q contribution.
 * q_bar: the external-force part is the exact derivative of the program J(q)^T f for every stored position entry;
 * the dynamics part means what it means above (exact for ID; for FD the manifold convention above, at tau + J^T f).
 * The scratch buffers and the concurrency caveat are those of the VJP entry points above. */
grbda_status grbda_cuda_inverse_dynamics_ext_vjp_f64(const grbda_model *m, const double *q, const double *yd,
                                                     const double *ydd, const double *f_ext, const double *tau_bar,
                                                     double *q_bar, double *yd_bar, double *ydd_bar, double *f_bar,
                                                     int64_t batch, void *stream);
grbda_status grbda_cuda_forward_dynamics_ext_vjp_f64(const grbda_model *m, const double *q, const double *yd,
                                                     const double *tau, const double *f_ext, const double *ydd_bar,
                                                     double *q_bar, double *yd_bar, double *tau_bar, double *f_bar,
                                                     int64_t batch, void *stream);
/* Reverse mode of grbda_cuda_contact_kinematics_f64: for cotangents p_bar[batch][n_cp][3] and v_bar[batch][n_cp][3]
 * of the contact positions and velocities, yd_bar[batch][nv] = J_lin^T v_bar (J_lin: the linear rows of the contact
 * Jacobians) and q_bar[batch][nq], the exact derivative of the contact-kinematics program for every stored position
 * entry (as for the inverse dynamics). p_bar and v_bar are packed into [batch][6 n_cp] in the per-stream scratch
 * buffer of the VJP entry points (two copies), then one kernel runs; same concurrency caveat. The program is
 * specialised for the contact set and compiled at run time when first used; a model without contact points is
 * refused as by grbda_cuda_contact_kinematics_f64. */
grbda_status grbda_cuda_contact_kinematics_vjp_f64(const grbda_model *m, const double *q, const double *yd,
                                                   const double *p_bar, const double *v_bar, double *q_bar,
                                                   double *yd_bar, int64_t batch, void *stream);

/* Integration step (semi-implicit Euler): yd_out = yd + dt ydd, q_out = q advanced with yd_out -
 * revolute coordinates q + dt yd; free base p + dt R v_body and ori::integrateQuat(quat, R omega_body,
 * dt) (include/grbda/Utils/OrientationTools.h:387-413); clusters with an implicit loop constraint
 * advance their independent coordinates and are projected back onto phi(q) = 0 (Newton on the
 * dependent coordinates, the iteration of GenericJoint.cpp:290-385). flags (optional, int32 per
 * state): 1 where the projection did not converge. A roll-pitch-yaw free base (GRBDA_CLUSTER_FREE_RPY) has no
 * integration rule and is refused per state: flags = 1 for every state, its six positions are copied unchanged to
 * q_out, the other clusters advance as above, and yd_out still holds yd + dt ydd. q_out / yd_out may alias q / yd. */
grbda_status grbda_cuda_integrate_f64(const grbda_model *m, const double *q, const double *yd, const double *ydd,
                                      double dt, double *q_out, double *yd_out, int32_t *flags, int64_t batch,
                                      void *stream);
/* One simulation step: forwardDynamics (with external forces when f_ext != NULL) followed by the
 * integration step above; the accelerations live in a per-stream scratch buffer of the handle. */
grbda_status grbda_cuda_step_f64(const grbda_model *m, const double *q, const double *yd, const double *tau,
                                 const double *f_ext, double dt, double *q_out, double *yd_out, int32_t *flags,
                                 int64_t batch, void *stream);
/* Reverse mode of the integration step, what the gradient of a loss over a rollout needs. For cotangents
 * q_out_bar[batch][nq] and yd_out_bar[batch][nv] of (q_out, yd_out) = integrate(q, yd, ydd, dt):
 *   v_bar = yd_out_bar + (d q_out / d yd')^T q_out_bar  (yd' = yd + dt ydd),  yd_bar = v_bar,  ydd_bar = dt v_bar,
 *   q_bar = (d q_out / d q)^T q_out_bar,
 * q_bar being the exact derivative of what the step computes for every stored position entry:
 *   one-dof / explicit clusters: q_bar = q_out_bar, and dt q_out_bar enters v_bar;
 *   quaternion base: the derivative of p + dt R(quat) v_body and of the renormalised product, R being the polynomial
 *     of the raw stored entries (also off the unit sphere); finite and continuous at omega = 0 (Taylor series of the
 *     rotation increment there);
 *   implicit clusters: the converged projection differentiated by the implicit function theorem at the projected
 *     point q': K_dep^T lambda = q_out_bar_dep, q_ind_bar = q_out_bar_ind - K_ind^T lambda (= G^T q_out_bar), and
 *     dt q_ind_bar enters v_bar. The old dependent coordinates are only Newton's starting point: their q_bar is 0;
 *   roll-pitch-yaw base: the step copies its positions, so q_bar = q_out_bar there, and the state is flagged.
 * Each state's step is re-run (Newton included) by the kernel; there is no saved q_out to pass. flags (optional)
 * receives the flags grbda_cuda_integrate_f64 writes; the values of a flagged state are the formula at the point
 * where Newton stopped and are meaningless: mask them with the flags. One kernel launch, elementwise, compiled at
 * run time (GRBDA_PROGRAM_INTEGRATE_VJP) for every model; GRBDA_JIT=0 gives GRBDA_ERR_NOT_COMPILED. batch = 0
 * returns GRBDA_OK without launching anything. FP64 only. */
grbda_status grbda_cuda_integrate_vjp_f64(const grbda_model *m, const double *q, const double *yd, const double *ydd,
                                          double dt, const double *q_out_bar, const double *yd_out_bar,
                                          double *q_bar, double *yd_bar, double *ydd_bar, int32_t *flags,
                                          int64_t batch, void *stream);
/* Reverse mode of grbda_cuda_step_f64 for the same cotangents: q_bar[batch][nq], yd_bar[batch][nv],
 * tau_bar[batch][nv] and, when f_ext != NULL, f_bar[batch][nf][6] (f_ext = NULL: f_bar is not written and may be
 * NULL). Launches, in order:
 *   1. the forward dynamics ydd = FD(q, yd, tau [+ J^T f]) into the per-stream acceleration buffer, exactly as
 *      grbda_cuda_step_f64 (the launches of grbda_cuda_forward_dynamics_ext_f64);
 *   2. grbda_cuda_integrate_vjp_f64 at that ydd, its q_bar / yd_bar parts and ydd_bar to a per-stream scratch
 *      buffer of the handle (one launch);
 *   3. grbda_cuda_forward_dynamics_ext_vjp_f64 with that ydd_bar (its launches; without forces that is
 *      grbda_cuda_forward_dynamics_vjp_f64);
 *   4. one elementwise kernel that adds the integration parts to q_bar and yd_bar.
 * q_bar: the integration part is exact as above; the dynamics part keeps the manifold convention of the
 * forward-dynamics VJP. flags as for grbda_cuda_integrate_vjp_f64. The scratch buffers belong to the (handle,
 * stream) pair, with the concurrency caveat of the VJP entry points above. FP64 only. */
grbda_status grbda_cuda_step_vjp_f64(const grbda_model *m, const double *q, const double *yd, const double *tau,
                                     const double *f_ext, double dt, const double *q_out_bar, const double *yd_out_bar,
                                     double *q_bar, double *yd_bar, double *tau_bar, double *f_bar, int32_t *flags,
                                     int64_t batch, void *stream);
/* ydd = FD(q, yd, tau). Replaces setState + ClusterTreeModel::forwardDynamics(tau),
 * src/Dynamics/ClusterTreeDynamics.cpp:85-191. */
grbda_status grbda_cuda_forward_dynamics_f64(const grbda_model *m, const double *q, const double *yd,
                                             const double *tau, double *ydd, int64_t batch, void *stream);
grbda_status grbda_cuda_forward_dynamics_f32(const grbda_model *m, const float *q, const float *yd,
                                             const float *tau, float *ydd, int64_t batch, void *stream);
/* H (nv x nv per state, symmetric). Replaces setState + getMassMatrix(),
 * src/Dynamics/ClusterTreeModel.cpp:98-103 -> TreeModel.cpp:116-160. */
grbda_status grbda_cuda_mass_matrix_f64(const grbda_model *m, const double *q, double *H, int64_t batch,
                                        void *stream);
grbda_status grbda_cuda_mass_matrix_f32(const grbda_model *m, const float *q, float *H, int64_t batch,
                                        void *stream);
/* Per state and body: p[3] world position of the body origin (getPosition), R[9] row-major
 * body-to-world rotation (getOrientation), v[6] = [world angular velocity; world linear velocity of
 * the origin] (getAngularVelocity, getLinearVelocity). Replaces setState + forwardKinematics() +
 * getters, TreeModel.cpp:7-32, ClusterTreeModel.cpp:319-373. */
grbda_status grbda_cuda_forward_kinematics_f64(const grbda_model *m, const double *q, const double *yd,
                                               double *p, double *R, double *v, int64_t batch, void *stream);
grbda_status grbda_cuda_forward_kinematics_f32(const grbda_model *m, const float *q, const float *yd,
                                               float *p, float *R, float *v, int64_t batch, void *stream);

/* ---- batched hot path, host pointers (H2D, kernel, D2H pipelined over pinned staging) -------- */
/* algo: 0 ID (in3 = ydd, out = tau), 1 FD (in3 = tau, out = ydd) */
grbda_status grbda_cuda_dynamics_host_f64(const grbda_model *m, int algo, const double *q, const double *yd,
                                          const double *in3, double *out, int64_t batch);

/* One benchmark step on host buffers: ydd = FD(q, yd, tau) followed by tau_back = ID(q, yd, ydd); q, yd
 * and tau cross PCIe once, both results come back. */
grbda_status grbda_cuda_forward_inverse_host_f64(const grbda_model *m, const double *q, const double *yd,
                                                 const double *tau, double *ydd, double *tau_back,
                                                 int64_t batch);

/* Place the calling thread (and what it allocates from now on, e.g. the pinned buffers handed to the
 * _host entry points) on the NUMA node of `device`'s PCIe root: CPU affinity to the node's cores that
 * the process may use, memory policy "prefer that node". One process per GPU calls it once before
 * allocating. info4 (optional) = {numa node or -1, cpus bound, memory policy set, cpus allowed before}. */
grbda_status grbda_cuda_bind_host_to_device(int device, int32_t *info4);

/* ---- synthetic states, checks, measurement --------------------------------------------------- */
/* Random valid states for global state indices [first_index, first_index + count): counter based
 * (Philox4x32-10), so a shard is reproducible whatever the GPU count. Ranges follow
 * ClusterJoints::Base::randomJointState (ClusterJoint.cpp:74-81), Free (FreeJoint.cpp:49-60) and
 * Generic (GenericJoint.cpp:290-385: Newton solve of phi for the dependent coordinates).
 * aux receives nv uniform [-1,1) values (ydd or tau). flags (optional, int32 per state) is set to
 * 1 for states whose implicit clusters could not be solved. */
grbda_status grbda_cuda_generate_states(const grbda_model *m, uint64_t seed, int64_t first_index,
                                        int64_t count, double *q, double *yd, double *aux,
                                        int32_t *flags, void *stream);
/* max |phi| over the implicit clusters of each state (isValidSpanningPosition, LoopConstraint.cpp:15-20) */
grbda_status grbda_cuda_constraint_violation_f64(const grbda_model *m, const double *q, double *max_abs_phi,
                                                 int64_t batch, void *stream);
/* out[0] = sum x_i, out[1] = sum |x_i| in double (device pointer x, host pointer out; synchronises) */
grbda_status grbda_cuda_checksum_f64(const double *x, int64_t n, double *out2, void *stream);
/* Achieved FP64 FMA throughput (FLOP/s, FMA = 2) and FP32 of the device with a dependent-free
 * FMA loop over all SMs; the roofline denominator for ID / FD. */
grbda_status grbda_cuda_measure_fma_peak(int device, int fp32, double seconds, double *flops_per_s);
/* Kernel launches issued by this library since load (bench.py's gpu_launches). */
int64_t grbda_cuda_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* GRBDA_CUDA_H */
