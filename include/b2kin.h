/*
 * b2kin.h -- C ABI of libb2kin.so: batched serial-chain kinematics / dynamics on B200 (sm_100a).
 *
 * This is the drop-in boundary for the reference's native fast path
 * (petercorke/robotics-toolbox-python, src/roboticstoolbox/core/).  Each entry point names
 * the reference interface it replaces (file:line relative to the reference repo).  The
 * reference boundary is two CPython extension modules taking PyObject tuples and PyCapsule
 * handles (fknm.cpp:23-93, frne.c:42-62); this one is plain C: POD arguments, opaque handles,
 * no Python.h, no torch types.  INTEGRATION.md shows the ctypes binding a reference maintainer
 * would add.
 *
 * Conventions
 *   - every batched array is a DEVICE pointer, contiguous, row-major:
 *       q (N, ldq)   T (N,4,4)   J (N,6,n)   tau (N,n)   Tep (N,4,4)
 *     i.e. the values of numpy.asarray(reference_result) for row i of the batch
 *     (reference batch FK layout: fknm.cpp:1005,1048-1051; single-q results are F-ordered
 *     there, fknm.cpp:993,813 -- same values, different strides).
 *   - small per-call constants (base, tool, gravity, fext, mask) are HOST pointers, fp64,
 *     4x4 matrices row-major; NULL means "not given" exactly like None in the reference.
 *   - dtype selects the arithmetic type of the device arrays: B2K_F32 or B2K_F64.
 *   - stream is a cudaStream_t passed as void* (NULL = legacy default stream).  All compute
 *     entry points are asynchronous on that stream.
 *   - every function returns 0 on success, a negative b2k_status otherwise; the message for
 *     the calling thread is available from b2k_last_error().
 *   - handles are immutable after creation: safe to use from many host threads / streams
 *     (the reference's frne capsule is mutated per call, frne.c:142-153,193-207).
 */
#ifndef B2KIN_H
#define B2KIN_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2K_VERSION 100 /* 0.1.0 */

#define B2K_F32 0
#define B2K_F64 1

/* largest number of joints a chain / DH robot may have (kernels are unrolled per n) */
#define B2K_MAX_JOINTS 10
/* largest q row width (max jindex + 1); reference: q may be wider than n, methods.cpp:338 */
#define B2K_MAX_QWIDTH 16

/* elementary-transform axis codes, as reference ET.py:244-266 */
#define B2K_RX 0
#define B2K_RY 1
#define B2K_RZ 2
#define B2K_TX 3
#define B2K_TY 4
#define B2K_TZ 5

/* LM damping rule, reference ik.cpp:157-209 / IK.py:997-1005 */
#define B2K_LM_CHAN 0     /* Wn = lambda * E * I   */
#define B2K_LM_WAMPLER 1  /* Wn = lambda * I       */
#define B2K_LM_SUGIHARA 2 /* Wn = (E + lambda) * I */
/* the other two solvers of the fknm module ride the same loop and entry point (method argument of b2k_ik_lm) */
#define B2K_IK_NR 3 /* Newton-Raphson, dq = pinv_d(J) e, lambda = pinv_damping: fknm.IK_NR_c, ik.cpp:121-155 */
#define B2K_IK_GN 4 /* Gauss-Newton, min-norm solution of (J^T We J) dq = J^T We e: fknm.IK_GN_c, ik.cpp:79-119 */

/* which of the reference's two LM loops to reproduce */
#define B2K_IK_SEM_CPP 0    /* fknm.IK_LM_c -> _IK_loop, ik.cpp:19-75 (ETS.ik_LM)       */
#define B2K_IK_SEM_PYTHON 1 /* IKSolver._solve + IK_LM.step, IK.py:297-367,994-1017 (ETS.ikine_LM) */

typedef enum {
    B2K_OK = 0,
    B2K_ERR_INVALID = -1, /* bad argument (shape, dtype, NULL, n too large, ...) */
    B2K_ERR_CUDA = -2,    /* a CUDA runtime call failed; message carries cudaGetErrorString */
    B2K_ERR_ALLOC = -3
} b2k_status;

typedef struct b2k_chain_s *b2k_chain_t; /* replaces the "ETS" PyCapsule, structs.h:25-56 */
typedef struct b2k_rne_s *b2k_rne_t;     /* replaces the "Robot" PyCapsule, frne.h            */
typedef struct b2k_tree_s *b2k_tree_t;   /* a rigid-body tree as Robot.rne walks it, Robot.py:1704-1903 */

const char *b2k_last_error(void);
int b2k_version(void);

/* ---------------------------------------------------------------- chain description
 * Replaces fknm.ET_init + fknm.ETS_init (fknm.cpp:1182-1239, 1066-1114; Python side
 * ET.py:100-125, ETS.py:62-69).  m elementary transforms, in chain order:
 *   isjoint[i]  1 = variable joint, 0 = constant
 *   axis[i]     B2K_RX..B2K_TZ (joints only)
 *   flip[i]     1 = joint moves in the opposite direction (eta = -q)
 *   jindex[i]   column of q this joint reads (joints only)
 *   T[i*16..]   constant 4x4, row-major (constants only; ignored for joints)
 *   qlim[i*2..] joint limits low/high (joints only; the caller applies the reference defaults
 *               [-pi,pi] / [0,1], ET.py:109-115)
 * All constants are copied (the reference keeps a borrowed pointer, fknm.cpp:1207).
 * Runs of constants are folded into one SE(3) constant per joint on the host -- the
 * reference's own ETS.compile() rule, ETS.py:857-906.
 */
int b2k_chain_create(int m, const int32_t *isjoint, const int32_t *axis, const int32_t *flip,
                     const int32_t *jindex, const double *T, const double *qlim,
                     b2k_chain_t *out);
int b2k_chain_destroy(b2k_chain_t chain);
/* n = joints, m = elementary transforms, q_width = max jindex + 1 */
int b2k_chain_info(b2k_chain_t chain, int *n, int *m, int *q_width);

/* ---------------------------------------------------------------- forward kinematics
 * Replaces fknm.ETS_fkine (fknm.cpp:923-1064 -> _ETS_fkine methods.cpp:318-352):
 *   T[i] = base * prod_k ET_k(q[i, jindex_k]) * tool
 * ldq = row stride of q in elements (>= q_width).
 * Output alignment, here and in b2k_jacob0 / b2k_jacobe / b2k_fkine_jacob0 / b2k_fkine_jacobe (a misaligned
 * output is refused with B2K_ERR_INVALID; every cudaMalloc / torch allocation qualifies):
 *   T (N,4,4): 32-byte aligned;
 *   J (N,6,n): 16-byte aligned for B2K_F64 and for B2K_F32 with even n, 8-byte aligned for B2K_F32 with odd n.
 * q needs only the alignment of its element type.
 */
int b2k_fkine(b2k_chain_t chain, int dtype, const void *q, int64_t N, int64_t ldq,
              const double *base, const double *tool, void *T, void *stream);

/* The poses of several frames along one chain from a single walk: the device side of fkine_all (reference
 * Robot.fkine_all, Robot.py:638-700, and DHRobot.fkine_all, DHRobot.py:1018-1064: Python loops over the links).
 * Frame k is  base * A_0 J_0(q) ... J_after[k](q) * tails[k]  -- the pose right after joint after[k] (0-based position
 * of the joint along the chain) times a constant 4x4 (row-major, host) -- or, for after[k] = -1, the constant tails[k]
 * itself (the base frame, links that depend on no joint; the caller multiplies the base in).  after[] ascending.
 * out is (N, nslots, 4, 4) row-major, 32-byte aligned; frame k goes to slot[k] of every row; slots not named are left
 * untouched (a branched robot takes one call per branch into the same array).  The chain's tool constant and the
 * transforms behind its last joint do not enter. */
int b2k_fkine_frames(b2k_chain_t chain, int dtype, const void *q, int64_t N, int64_t ldq, const double *base,
                     int nframes, const int32_t *after, const int32_t *slot, const double *tails, void *out,
                     int64_t nslots, void *stream);

/* Replaces fknm.ETS_jacob0 (fknm.cpp:785-850 -> _ETS_jacob0 methods.cpp:112-216), batched:
 * J[i] = geometric Jacobian in the chain's start frame, (6,n) row-major per row; no base
 * (reference RobotKinematics.py:158), tool included.  J aligned as for b2k_fkine above. */
int b2k_jacob0(b2k_chain_t chain, int dtype, const void *q, int64_t N, int64_t ldq,
               const double *tool, void *J, void *stream);

/* Replaces fknm.ETS_jacobe (fknm.cpp:852-921 -> _ETS_jacobe methods.cpp:219-316), batched:
 * Jacobian in the end-effector frame.  J aligned as for b2k_fkine above. */
int b2k_jacobe(b2k_chain_t chain, int dtype, const void *q, int64_t N, int64_t ldq,
               const double *tool, void *J, void *stream);

/* Fused pose + base-frame Jacobian in one pass over q (the BASELINE headline op):
 * T as b2k_fkine (base and tool applied), J as b2k_jacob0 (tool applied, no base).  T 32-byte aligned, J as for
 * b2k_fkine above. */
int b2k_fkine_jacob0(b2k_chain_t chain, int dtype, const void *q, int64_t N, int64_t ldq,
                     const double *base, const double *tool, void *T, void *J, void *stream);

/* Fused pose + end-effector-frame Jacobian.  T 32-byte aligned, J as for b2k_fkine above. */
int b2k_fkine_jacobe(b2k_chain_t chain, int dtype, const void *q, int64_t N, int64_t ldq,
                     const double *base, const double *tool, void *T, void *J, void *stream);

/* ---------------------------------------------------------------- inverse kinematics
 * Replaces fknm.IK_LM_c (fknm.cpp:394-525 -> _IK_LM_Chan/_Wampler/_Sugihara ik.cpp:157-209
 * -> _IK_loop ik.cpp:19-75) for N targets at once, and -- with semantics =
 * B2K_IK_SEM_PYTHON -- the Python solver behind ETS.ikine_LM (IK.py:297-367, 994-1017).
 *   Tep      (N,4,4) device, row-major
 *   q0       (N,n) device initial guesses or NULL (then drawn inside the joint limits)
 *   we       host 6-vector of Cartesian weights or NULL (= ones); We = diag(we)
 *   reject_jl  reject converged solutions outside the joint limits and restart
 *   seed     seed of the counter-based restart generator (the reference uses unseeded libc
 *            rand(), ik.cpp:293, or numpy default_rng, IK.py:166)
 *   rng_per_row  1: restart draws keyed by (seed,row,search); 0: shared by all rows
 *            (IKSolver.solve reuses one set of restarts for a whole trajectory, IK.py:222-272)
 * Outputs (device): q_out (N,n), success/iterations/searches int32 (N), residual (N) in dtype
 * -- the tuple IK_LM_c returns (fknm.cpp:516), one entry per target.
 * q0 and q_out hold the chain's n joints in chain order, i.e. q[ets.jindices] -- exactly what the reference's Python
 * solver hands back for an ETS whose jindices are not 0..n-1 (it pads q to max_jindex + 1 internally, IK.py:216-240,
 * and returns q[ets.jindices], IK.py:346), so sub-chains of a larger robot are served as they are (the reference's
 * C++ loop assumes dense jindices, ik.cpp:34-35).  Two joints sharing one jindex are rejected.
 * method = B2K_IK_NR / B2K_IK_GN select fknm.IK_NR_c / IK_GN_c (fknm.cpp:164-392) and, with the
 * Python semantics, IK_NR.step / IK_GN.step (IK.py:714-762, 1154-1219; both take pinv(J) e there).
 * The pseudo-inverse step is evaluated as Jw^T (Jw Jw^T + d^2)^-1 ew (6x6 Cholesky); pinv = False
 * on a square chain (J.inverse() e) is the same vector and is not a separate code path.
 */
int b2k_ik_lm(b2k_chain_t chain, int dtype, const void *Tep, int64_t N, const void *q0,
              int ilimit, int slimit, double tol, int reject_jl, const double *we, double lambda,
              int method, uint64_t seed, int semantics, int rng_per_row, void *q_out,
              int32_t *success, int32_t *iterations, int32_t *searches, void *residual,
              void *stream);

/* ---------------------------------------------------------------- inverse dynamics (DH RNE)
 * b2k_rne_create replaces frne.init (frne.c:233-299): n links, mdh = 0 standard / 1 modified
 * DH, L = 24 doubles per link packed as reference DHRobot.py:1340-1358
 *   [alpha, a, theta, d, sigma, offset, m, r(3), I(9 row-major), Jm, G, B, Tc+, Tc-].
 * b2k_rne replaces the per-row frne.frne loop (frne.c:106-230 -> newton_euler ne.c:62-492):
 *   tau[i] = RNE(q[i], qd[i], qdd[i]) for i < N, arrays (N,n).
 *   grav : host 3-vector handed to the recursion as the base acceleration, i.e. MINUS the
 *          robot's gravity exactly as DHRobot.rne passes it (DHRobot.py:1449); must not be NULL
 *   fext : host 6-vector wrench at the tip or NULL (= zeros)
 */
int b2k_rne_create(int n, int mdh, const double *L, b2k_rne_t *out);
int b2k_rne_destroy(b2k_rne_t rne);
int b2k_rne(b2k_rne_t rne, int dtype, const void *q, const void *qd, const void *qdd, int64_t N,
            const double *grav, const double *fext, void *tau, void *stream);

/* Robot-specialised kernels.  For all-revolute arms b2k_rne (and the dynamics entry points below) run a kernel that is
 * generated for THIS robot's link table and compiled for sm_100a at first use (NVRTC): terms whose link parameter is zero
 * are never emitted, alpha = k pi/2 turns rotations into permutations, constants are folded (csrc/b2k_rne_gen.cpp,
 * b2k_rne_spec.cu).  Results equal the generic kernel's to rounding.  Environment: B2K_RNE_SPEC=0 disables it, =2 makes a
 * failure to specialise an error; B2K_NVRTC_PATH names libnvrtc.so.12 when it is not on the loader path.
 *   b2k_rne_spec_info  writes a one-line description of the kernel that serves (mode, dtype, grav pattern, has_fext) for
 *                      this robot into buf -- mode: 0 rne, 1 inertia, 2 gravload, 3 itorque, 4 coriolis, 5 accel.
 *   b2k_rne_codegen    returns the generated row function (plain C in terms of `real`; also valid host C++) and its
 *                      constant bank, so the generator can be checked against the oracle without a GPU;
 *                      counts[3] = multiplications, fused multiply-adds, additions per row. */
int b2k_rne_spec_info(b2k_rne_t rne, int mode, int dtype, const double *grav, int has_fext, char *buf, int64_t cap);
int b2k_rne_codegen(b2k_rne_t rne, int mode, int grav_mask, int has_fext, char *src, int64_t src_cap, double *consts,
                    int32_t consts_cap, int32_t *n_consts, int32_t *counts);

/* ---------------------------------------------------------------- inverse dynamics of ETS / URDF robots (rigid-body trees)
 * Replaces the pure-Python Robot.rne (Robot.py:1704-1903: Featherstone's recursion over spatial vectors, one Python loop
 * iteration per trajectory row).  The tree is described the way that function walks it: n joint groups in link order;
 * group j hangs off group parent[j] (-1 = the base) through the constant transform C[j] (3x4 row-major: the static links
 * of the group and the constant part of the joint link, folded) followed by ONE joint of kind axis[j] (B2K_RX..B2K_TZ,
 * flip[j]) that reads q[jindex[j]]; I6[j] (6x6 row-major, [linear; angular] order as spatialmath's SpatialInertia) is the
 * inertia of the group in the joint link's frame.  b2k_tree_rne: tau (N,n) = rne(q, qd, qdd) rows, arrays (N,n) device,
 * 16-byte aligned; grav = MINUS the robot's gravity (Robot.rne's a_grav), host 3-vector.  Reference quirks kept: the
 * joint motion subspace ignores `flip` (ET.s, ET.py:592-608), torques are listed in group order.  The kernel is generated
 * for the tree at hand and compiled with NVRTC at first use (there is no pre-compiled kernel for an arbitrary tree). */
int b2k_tree_create(int n, const int32_t *parent, const int32_t *axis, const int32_t *flip, const int32_t *jindex,
                    const double *C, const double *I6, b2k_tree_t *out);
int b2k_tree_destroy(b2k_tree_t tree);
int b2k_tree_rne(b2k_tree_t tree, int dtype, const void *q, const void *qd, const void *qdd, int64_t N, const double *grav,
                 void *tau, void *stream);
/* The operations DynamicsMixin derives from rne (Dynamics.py: inertia 752-758, gravload 912-915, itorque 1456-1459,
 * coriolis 825-857, accel 490-503) for a tree robot -- in the reference n to n(n+1)/2 + 1 Python rne loops per row, here
 * one generated kernel per operation (the same recursion over symbolic unit / zero inputs, like the DH entry points below).
 *   op B2K_DYN_INERTIA  in0 = q                      out (N,n,n)  row i = rne(q, 0, e_i, gravity 0)
 *      B2K_DYN_GRAVLOAD in0 = q                      out (N,n)    rne(q, 0, 0)                          uses grav
 *      B2K_DYN_ITORQUE  in0 = q, in1 = qdd           out (N,n)    rne(q, 0, qdd, gravity 0)
 *      B2K_DYN_CORIOLIS in0 = q, in1 = qd            out (N,n,n)  the reference's combination rule
 *      B2K_DYN_ACCEL    in0 = q, in1 = qd, in2 = tau out (N,n)    M(q)^-1 (tau - rne(q, qd, 0))         uses grav
 * (B2K_DYN_RNE = b2k_tree_rne).  e_i and the input columns are in q order, the torque columns in group order, exactly as
 * the reference's calls produce them.  b2k_tree_codegen / b2k_tree_info take the same op codes. */
#define B2K_DYN_RNE 0
#define B2K_DYN_INERTIA 1
#define B2K_DYN_GRAVLOAD 2
#define B2K_DYN_ITORQUE 3
#define B2K_DYN_CORIOLIS 4
#define B2K_DYN_ACCEL 5
int b2k_tree_dyn(b2k_tree_t tree, int op, int dtype, const void *in0, const void *in1, const void *in2, int64_t N,
                 const double *grav, void *out, void *stream);
int b2k_tree_codegen(b2k_tree_t tree, int op, int grav_mask, char *src, int64_t src_cap, double *consts, int32_t consts_cap,
                     int32_t *n_consts, int32_t *counts);
int b2k_tree_info(b2k_tree_t tree, int op, int dtype, const double *grav, char *buf, int64_t cap);

/* ---------------------------------------------------------------- dynamics built on the recursion
 * The reference's DynamicsMixin (robot/Dynamics.py) obtains these by looping frne calls in
 * Python; here each is ONE kernel in which a lane performs all the recursions of its row
 * (SURVEY 8f-1).  q, qd, qdd, torque are (N,n) device arrays; gravity conventions as b2k_rne
 * (grav = MINUS the robot's gravity, host 3-vector).
 *   b2k_rne_inertia   M (N,n,n): row i of M[k] = rne(q_k, 0, e_i, g=0)          Dynamics.py:704-763
 *   b2k_rne_gravload  taug (N,n) = rne(q, 0, 0, g)                              Dynamics.py:863-921
 *   b2k_rne_itorque   taui (N,n) = rne(q, 0, qdd, g=0)                          Dynamics.py:1407-1465
 *   b2k_rne_coriolis  C (N,n,n), on a friction-free copy of the robot           Dynamics.py:765-861
 *   b2k_rne_accel     qdd (N,n) = M^-1 (torque - rne(q, qd, 0, g)), friction kept  Dynamics.py:424-510
 */
int b2k_rne_inertia(b2k_rne_t rne, int dtype, const void *q, int64_t N, void *M, void *stream);
int b2k_rne_gravload(b2k_rne_t rne, int dtype, const void *q, int64_t N, const double *grav, void *taug, void *stream);
int b2k_rne_itorque(b2k_rne_t rne, int dtype, const void *q, const void *qdd, int64_t N, void *taui, void *stream);
int b2k_rne_coriolis(b2k_rne_t rne, int dtype, const void *q, const void *qd, int64_t N, void *C, void *stream);
int b2k_rne_accel(b2k_rne_t rne, int dtype, const void *q, const void *qd, const void *torque, int64_t N,
                  const double *grav, void *qdd, void *stream);

/* b2k_rne_fdyn integrates the forward dynamics of an ENSEMBLE of initial states (DynamicsMixin.fdyn, Dynamics.py:185-422,
 * integrates one): one lane per trajectory, Dormand-Prince 5(4) with scipy RK45's step control (rtol, atol, max_step,
 * first_step <= 0: automatic), every stage's acceleration from the robot-specialised recursion.  q0, qd0 (ntraj,n) device
 * (qd0 may be NULL = at rest).  Torque: torque_mode 0 none, 1 constant tau (host n), 2 tau_rows (ntraj,n) device,
 * 3 PD kp (qstar - q) - kd qd (host n-vectors).  Output, M slots per trajectory: grid = 0 the accepted steps (t, q, qd as
 * scipy's integrator visits them), grid = 1 the uniform grid k dt by linear interpolation (the reference's interp1d);
 * out_t (ntraj,M), out_q / out_qd (ntraj,M,n), out_count (samples produced; > M means the capacity was too small),
 * out_status (bit 0: step size underflow, bit 1: capacity exceeded).  All-revolute robots; needs NVRTC. */
int b2k_rne_fdyn(b2k_rne_t rne, int dtype, const void *q0, const void *qd0, int64_t ntraj, double T, const double *grav,
                 int torque_mode, const double *tau, const void *tau_rows, const double *kp, const double *kd, const double *qstar,
                 double rtol, double atol, double max_step, double first_step, double dt, int grid, int M, void *out_t,
                 void *out_q, void *out_qd, int32_t *out_count, int32_t *out_status, void *stream);
/* the same integrator around the accel recursion of a rigid-body tree (Robot.fdyn); grav = MINUS the robot's gravity */
int b2k_tree_fdyn(b2k_tree_t tree, int dtype, const void *q0, const void *qd0, int64_t ntraj, double T, const double *grav,
                 int torque_mode, const double *tau, const void *tau_rows, const double *kp, const double *kd, const double *qstar,
                 double rtol, double atol, double max_step, double first_step, double dt, int grid, int M, void *out_t,
                 void *out_q, void *out_qd, int32_t *out_count, int32_t *out_status, void *stream);

/* ---------------------------------------------------------------- pure functions of the Jacobian
 * b2k_hessian replaces fknm.ETS_hessian0 / ETS_hessiane (fknm.cpp:583-783 -> _ETS_hessian
 * methods.cpp:16-32): H (N,n,6,n) from J (N,6,n); pass jacob0 for hessian0, jacobe for hessiane.
 * b2k_manipulability is the Yoshikawa measure of ETS.manipulability (ETS.py:1780-1787):
 * m = sqrt|det(Ja Ja^T)| over the Cartesian rows selected by axes_mask (bit k = row k of J;
 * 63 = all, 7 = translational, 56 = rotational); |det Ja| when Ja is square. */
int b2k_hessian(int dtype, int n, const void *J, int64_t N, void *H, void *stream);
int b2k_manipulability(int dtype, int n, const void *J, int64_t N, uint32_t axes_mask, void *m, void *stream);
/* The singular-value measures of ETS.manipulability (ETS.py:1789-1796) over the Cartesian rows in axes_mask:
 * kind 0 "minsingular" = numpy svd(Ja)[-1] (the smallest of min(rows, n) singular values), kind 1 "invcondition" =
 * 1 / numpy.linalg.cond(Ja) = s_min / s_max.  One-sided Jacobi SVD per row, in registers / local memory. */
int b2k_manipulability_svd(int dtype, int n, const void *J, int64_t N, uint32_t axes_mask, int kind, void *m, void *stream);
/* b2k_jacob_dot: Jd (N,6,n) = sum_i H[i] qd[i], the Jacobian time derivative of Robot.jacob0_dot
 * (Robot.py:964-1099, representation None: np.tensordot(hessian0, qd, (0,0))), from J (N,6,n) and qd (N,n)
 * without materialising the Hessian.
 * b2k_jacobm: the manipulability Jacobian dm/dq (N,n) of ETS.jacobm (ETS.py:1628-1685) / Robot.jacobm
 * (Robot.py:1124-1232) over the Cartesian rows in axes_mask: Jm[i] = m * vec(Ja Ha_i^T) . vec(inv(Ja Ja^T)). */
int b2k_jacob_dot(int dtype, int n, const void *J, const void *qd, int64_t N, void *Jd, void *stream);
int b2k_jacobm(int dtype, int n, const void *J, int64_t N, uint32_t axes_mask, void *Jm, void *stream);

/* ---------------------------------------------------------------- pose error, position-based servo
 * b2k_angle_axis replaces fknm.Angle_Axis (fknm.cpp:112-162 -> _angle_axis ik.cpp:241-286), batched:
 * e (N,6) = [translation error; angle-axis rotation error] between Te (N,4,4) and Tep.
 * tep_stride = 16: one target per row, Tep (N,4,4); tep_stride = 0: a single (4,4) target for every row.
 * b2k_p_servo is tools/p_servo.py:46-106 with method="angle-axis": v (N,6) = gain .* e (gain: host
 * 6-vector or NULL = ones), arrived (N) int32 = sum|e| < threshold. */
int b2k_angle_axis(int dtype, const void *Te, const void *Tep, int64_t N, int64_t tep_stride, void *e, void *stream);
int b2k_p_servo(int dtype, const void *Te, const void *Tep, int64_t N, int64_t tep_stride, const double *gain,
                double threshold, void *v, int32_t *arrived, void *stream);

/* b2k_p_servo_rpy is tools/p_servo.py:46-106 with the reference's default method="rpy": the error is taken in the
 * end-effector frame, e = [t(Te^-1 Tep); tr2rpy(Te^-1 Tep, order="zyx")]; arguments as b2k_p_servo.
 * b2k_jacob0_analytical is ETS.jacob0_analytical (ETS.py:1570-1626): Ja (N,6,n) = blkdiag(I, A^-1(Gamma(R))) J0 from
 * the poses T (N,4,4) and base-frame Jacobians J (N,6,n); representation 0 "rpy/xyz", 1 "rpy/zyx", 2 "eul", 3 "exp".
 * tr2rpy / tr2eul / rotvelxform belong to spatialmath-python (not under the reference tree): their documented
 * conventions are restated in csrc/b2k_pose.cu and pinned by derivative identities in tests/, not by the package. */
int b2k_p_servo_rpy(int dtype, const void *Te, const void *Tep, int64_t N, int64_t tep_stride, const double *gain,
                    double threshold, void *v, int32_t *arrived, void *stream);
int b2k_jacob0_analytical(int dtype, int n, const void *T, const void *J, int64_t N, int representation, void *Ja,
                          void *stream);

/* ---------------------------------------------------------------- trajectory producer
 * b2k_jtraj replaces tools.trajectory.jtraj (tools/trajectory.py:686-780): quintic joint-space blend
 * from q0 to qf (host n-vectors; qd0 / qd1 boundary velocities or NULL = 0) sampled at N points,
 * written straight into device buffers q, qd, qdd (N,n) (qd / qdd may be NULL) so the batch can feed
 * b2k_fkine / b2k_rne without touching the host.
 *   t == NULL: N samples of normalised time np.linspace(0, 1, N), tscal must be 1 (the `t: int` form);
 *   t != NULL: device vector of N sample times (dtype), tscal = max(t) (the time-vector form). */
int b2k_jtraj(int dtype, int n, const double *q0, const double *qf, const double *qd0, const double *qd1,
              int64_t N, const void *t, double tscal, void *q, void *qd, void *qdd, void *stream);

/* b2k_mtraj replaces tools.trajectory.quintic (trajectory.py:271-416), trapezoidal (429-615) and their
 * multi-axis form mtraj (617-684): n axes, each following a quintic (kind 0; boundary velocities qd0 / qdf
 * or NULL = 0) or trapezoidal (kind 1; V = per-axis velocity of the linear segment, NULL or NaN = the
 * reference's default 1.5 (qf - q0) / tf) profile from q0[j] to qf[j]; outputs s, sd, sdd (N,n) device
 * (sd / sdd may be NULL).  t == NULL: sample times 0, 1, ..., N-1 (the `t: int` form, tf must be N-1);
 * t != NULL: device vector of N sample times, tf = max(t).  tblend (host, n doubles or NULL) receives the
 * blend times of the trapezoidal profile.  "V too small" / "V too big" (trajectory.py:555-558) -> B2K_ERR_INVALID. */
int b2k_mtraj(int dtype, int kind, int n, const double *q0, const double *qf, const double *qd0, const double *qdf,
              const double *V, int64_t N, const void *t, double tf, void *s, void *sd, void *sdd, double *tblend,
              void *stream);

/* b2k_ctraj replaces tools.trajectory.ctraj (trajectory.py:782-841 -> SE3.interp): N poses between T0 and T1 (host,
 * 4x4 row-major) at the path fractions s (device, N values in [0,1], clipped): translation interpolated linearly,
 * orientation by unit-quaternion slerp along the shorter arc; T (N,4,4) device.
 * b2k_mstraj evaluates the sample table of tools.trajectory.mstraj (trajectory.py:852-1152): the caller plans the
 * segments on the host exactly as the reference does and passes the pieces in row order -- kind 0: quintic blend
 * (jtraj coefficients A B C E F per axis in coef[piece][axis][0..4], sampled at t = (k+1) dt over a blend of length
 * tscal), kind 1: linear segment (coef = q_prev, q_next; s = (t0 + k dt) / tscal) -- and q (N,n) is written on the device. */
int b2k_ctraj(int dtype, const double *T0, const double *T1, const void *s, int64_t N, void *T, void *stream);
int b2k_mstraj(int dtype, int n, int npieces, const int64_t *row0, const int64_t *rows, const int32_t *kind,
               const double *tscal, const double *t0, const double *dt, const double *coef, int64_t N, void *q, void *stream);

/* ---------------------------------------------------------------- host-buffer front ends
 * The same operations for callers that hold HOST arrays (what the reference's API takes):
 * the library streams row chunks host->device, runs the kernel and streams results back on
 * several CUDA streams so copies overlap compute.  Pinned host memory (b2k_host_alloc, or
 * memory the caller registered) gets full PCIe/C2C bandwidth; pageable memory works too.
 * Synchronous: results are complete in the host arrays on return.  device = CUDA ordinal.
 */
int b2k_host_alloc(void **ptr, int64_t bytes);
int b2k_host_free(void *ptr);
int b2k_fkine_jacob0_host(b2k_chain_t chain, int dtype, const void *q_host, int64_t N,
                          int64_t ldq, const double *base, const double *tool, void *T_host,
                          void *J_host, int device);
int b2k_fkine_host(b2k_chain_t chain, int dtype, const void *q_host, int64_t N, int64_t ldq,
                   const double *base, const double *tool, void *T_host, int device);
int b2k_rne_host(b2k_rne_t rne, int dtype, const void *q_host, const void *qd_host,
                 const void *qdd_host, int64_t N, const double *grav, const double *fext,
                 void *tau_host, int device);

/* number of kernel launches this library has issued in the calling process (all threads);
 * bench.py reports the delta over its timed region as "gpu_launches". */
int64_t b2k_launch_count(void);

/* Test hook: evaluates the kernels' in-house sincos (csrc/b2k_trig.cuh) on n device values so
 * its accuracy can be checked in isolation: s[i], c[i] = sin(x[i]), cos(x[i]). */
int b2k_selftest_sincos(int dtype, const void *x, int64_t n, void *s, void *c, void *stream);

/* kernel variant switch for measurements: 0 = default (lane-per-configuration, warp-tiled
 * I/O), 1 = literal warp-per-configuration walk (one joint configuration per warp),
 * 2 = memory skeleton (default kernel without the chain walk: outputs are NOT valid),
 * 3 = arithmetic skeleton (default kernel without the output stores),
 * 4 = persistent grid-stride scheduling instead of the default one-tile-per-warp grid.
 * Affects b2k_fkine / b2k_jacob0 / b2k_fkine_jacob0 only; never set it in production. */
int b2k_set_variant(int variant);

#ifdef __cplusplus
}
#endif
#endif /* B2KIN_H */
