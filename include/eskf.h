/* C ABI of the B200 batched VI-ESKF engine (libeskf_b200.so).
 *
 * The reference (salehahr/dvi-ekf) is pure Python and has no FFI; the seam this
 * library sits behind is the Python class dvi_ekf/filter/Filter.py:28 (`Filter`)
 * and its driver dvi_ekf/filter/Simulator.py:24.  Each entry point below names the
 * reference method it replaces.  Plain pointers and sizes only; every function
 * returns 0 on success or a negative ESKF_E* code and never throws.  A handle is
 * bound to one device + stream, is not thread-safe, and all calls are ordered on
 * that stream (asynchronous w.r.t. the host unless a host buffer has to be read
 * back, in which case the call synchronises the stream before returning).
 *
 * Layouts (row-major FP64):
 *   x      [N,26]  p(3) v(3) q_xyzw(4) dofs(6) notch,notch_d,notch_dd(3) p_cam(3) q_cam_xyzw(4)
 *                  (dvi_ekf/filter/state.py:11-29)
 *   P      [N,24,24] error covariance, error-state order dp dv dth ddofs(6) dnotch(3) dpc dthc
 *                  (state.py:105-115)
 *   u_old  [N,6]   previous IMU sample om(3), acc(3)      (Filter.py:78-79,225-226)
 *   R_old  [N,9]   rot(q) at the end of the last propagate (Filter.py:80,227; NOT refreshed by update)
 *   Qdiag  [N|1,13], Rdiag [N|1,7], sigma_om [N|1,3]      (Filter.py:68-75,330-331)
 */
#ifndef ESKF_B200_H
#define ESKF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct eskf_handle eskf_t;

enum { ESKF_MEM_HOST = 0, ESKF_MEM_DEVICE = 1 };

enum {
  ESKF_OK = 0,
  ESKF_EINVAL = -1,  /* bad argument */
  ESKF_ECUDA = -2,   /* CUDA runtime error (see eskf_last_error) */
  ESKF_ENOMEM = -3
};

/* model flags */
enum { ESKF_FLAG_ZERO_FROZEN = 1 /* HEAD behaviour, Filter.py:243-245 */ };

/* per-filter status bits (eskf_get_state) */
enum {
  ESKF_STATUS_UPDATE_SKIPPED = 1, /* singular / non-finite S: the LinAlgError branch, Filter.py:356-361 */
  ESKF_STATUS_ASIN_DOMAIN = 2     /* |v| > 1 in Quaternion.angle (math.asin would raise) */
};

typedef struct {
  double scope_length;   /* config.yaml model.length              (Probe.py:162) */
  double cam_angle_rad;  /* config.yaml model.angle, in radians    (config.py:130-132) */
  int32_t frozen_mask;   /* bit i set: DOF i frozen                (Filter.py:56) */
  int32_t flags;         /* ESKF_FLAG_* */
} eskf_model_t;

/* Trajectory streams for eskf_run == Filter.run (Filter.py:144-185).
 * All arrays live in `mem` space.  n_traj trajectories are stacked; filter i uses
 * trajectory (filter_id0 + i) / filters_per_traj  (n_traj = 1: every filter shares one). */
typedef struct {
  int64_t n_steps;          /* T: IMU samples per trajectory */
  int64_t n_epochs;         /* E: camera frames after the initial one */
  int32_t n_traj;
  int32_t mem;              /* ESKF_MEM_* */
  int64_t filters_per_traj;
  const double* dt;         /* [n_traj,T]   per-step dt (Filter.py:214; quirk Q14: never assumed uniform) */
  const double* om_acc;     /* [n_traj,T,6] IMU samples (Imu.eval_expr_single, Imu.py:141-196) */
  const int32_t* n_prop;    /* [n_traj,E]   IMU samples in each epoch (Camera.py:320-347) */
  const double* cam;        /* [n_traj,E,7] camera position + RAW quaternion xyzw (VisualTrajectory.py:120-134) */
  const double* notch;      /* [n_traj,E]   measured notch angle (Camera.get_notch_vec_at) */
  /* references for the error statistics (nullable: statistics then only hold the DOF error) */
  const double* cam_ref;    /* [n_traj,E,6] camera x y z rx ry rz(deg)      (Filter.py:401-406) */
  const double* imu_ref;    /* [n_traj,E,6] IMU ref vx vy vz rx ry rz(deg)  (Filter.py:408-413) */
  double gt_dofs[6];        /* config.gt_imu_dofs (Filter.py:452-455) */
  /* Monte-Carlo extension (the reference is noise free): zero-mean Gaussian noise drawn
   * in-kernel from Philox4x32-10(key = seed, counter = (step, kind, filter id)), single-precision
   * Box-Muller on the SFU; the samples of a run can be read back with eskf_noise_dump() */
  uint64_t seed;
  int64_t filter_id0;       /* global id of this handle's first filter (multi-GPU sharding) */
  double imu_noise_std[6];  /* added to om(3), acc(3) of every IMU sample */
  double cam_noise_std[7];  /* added to camera position(3), as small rotation(3), notch(1) */
  int32_t noise_free_filter0; /* global filter 0 stays noise free (= the oracle run) */
  int32_t noise_id_modulus;   /* r > 0: filter g draws the noise of id g % r (common random numbers across parameter
                               * candidates that each own r consecutive filters); 0: every filter its own noise */
  /* trace mode (nullable, in `mem` space): [N,T,26] nominal state after every IMU step, the row of the last step
   * of an epoch holding the UPDATED state -- the rows FilterTraj keeps (FilterTraj.py:34-69, Filter.py:229,382).
   * 208 B per filter-step: a diagnostic / export mode, HBM bound, not the production path. */
  double* trace_x;
} eskf_streams_t;

#define ESKF_NSTAT 16
/* per-filter statistics row written by eskf_run: [0:6] (dofs - gt)^2, [6] dof metric (Filter.py:452-455),
 * [7] update_mse of the last epoch (Filter.py:397-418), [8] sum of update_mse over epochs,
 * [9] number of applied updates, [10] status word, [11] 1, [12:16] reserved.
 * stats_sum (the vector a multi-GPU launcher all-reduces) is reduced from the rows after the launch, deterministically
 * (fixed tree, no atomics) and MASKED: [0:10] sum the rows of the HEALTHY filters only (all of [0:10] finite and status
 * word 0), [10] = number of filters with a non-zero status word, [11] = number of healthy filters (the divisor of every
 * mean), [12] = number of filters with a non-finite row, [13:16] reserved (0).  A diverged filter therefore shows up in
 * the counts and never turns the reduced vector into NaN. */

/* Simulator.__init__ / Filter.__init__ (Simulator.py:30-68, Filter.py:34-93) */
int eskf_create(const eskf_model_t* model, int64_t n_filters, int device, void* cuda_stream, eskf_t** out);
int eskf_destroy(eskf_t* h);

/* Filter.__init__ / Filter.reset (Filter.py:44-45,78-80,95-108).  nx, nP, nu, nR are the leading
 * dimensions of the arrays passed: N, or 1 to broadcast one row to every filter.
 * R_old may be NULL: it is then set to rot(q) (Filter.py:80). */
int eskf_set_state(eskf_t* h, const double* x, int64_t nx, const double* P, int64_t nP, const double* u_old,
                   int64_t nu, const double* R_old, int64_t nR, int mem);

/* Filter.__init__ noise setup / update_noise_matrices (Filter.py:68-75,110-117) */
int eskf_set_noise(eskf_t* h, const double* Qdiag, int64_t nq, const double* Rdiag, int64_t nr,
                   const double* sigma_om, int64_t ns, int mem);

/* T calls of Filter.propagate(t, om, acc) (Filter.py:219-230) on every filter.
 * om_acc is [T,6] (per_filter = 0) or [N,T,6] (per_filter = 1); dt is [T]. */
int eskf_propagate(eskf_t* h, const double* dt, const double* om_acc, int64_t T, int per_filter, int mem);

/* Filter.update(t, camera, ang_notch) -> K (Filter.py:351-395).  cam is [1,7] / [N,7]
 * (position + raw quaternion xyzw), notch [1] / [N].  K_out is NULL or [N,24,7]. */
int eskf_update(eskf_t* h, const double* cam, const double* notch, int per_filter, double* K_out, int mem);

/* Filter.run (Filter.py:144-185): the whole trajectory in ONE persistent kernel, covariance resident
 * on-chip.  stats_out is NULL or [N,ESKF_NSTAT]; stats_sum is NULL or [ESKF_NSTAT] (sum over this
 * handle's filters, the vector a multi-GPU launcher all-reduces). */
int eskf_run(eskf_t* h, const eskf_streams_t* streams, double* stats_out, double* stats_sum, int mem);

#define ESKF_NCARRY 4
/* Epochs [epoch_begin, epoch_end) of the trajectory in `streams` (no reference counterpart), continuing from the handle's state:
 * a run in segments, with control between them, bit-identical to one eskf_run.  `streams` is the WHOLE trajectory eskf_run
 * takes, not a slice: trajectory t starts at step k0[t] = sum over e < epoch_begin of n_prop[t, e] (clamped to n_steps as the
 * kernels clamp every epoch), the Monte-Carlo noise is drawn by global step and epoch, and the references, the trace rows and
 * the per-epoch streams are read at their global rows.
 *   carry_in / carry_out: NULL or [N,ESKF_NCARRY] in `mem` space (they may be the same array), the per-filter accumulators the
 *     statistics row cannot hold without loss: [0] and [1] the two running squared-error sums of Filter.calculate_update_mse
 *     (row [8] is (sum0 + sum1) / 12), [2] the applied updates, [3] the status word.  carry_in = NULL continues with zero
 *     sums from the handle's status word, as eskf_run does; otherwise the sums start from it and the status word is set from
 *     [3], so that its sticky bits survive eskf_set_state on a new handle.  The checkpoint of a run is eskf_get_state +
 *     carry_out + epoch_end: enough to continue in another process, on another handle or on another GPU.
 *   stats_out / stats_sum: as for eskf_run, accumulated over epochs [0, epoch_end); row [7] is the update MSE of epoch
 *     epoch_end - 1.  After the last segment every column is bit-identical to the one-launch run.
 *   trace_x: the rows of the segment's steps are written at their global step rows of [N,T,26] (and, where the segment
 *     begins with epochs of 0 steps, the row before them, which their updates overwrite as in one launch); the other rows
 *     keep the caller's content.  A host trace is staged whole (N * T * 208 bytes of device memory), as for eskf_run.
 *   Jacobian record (eskf_keep_jacobians): the last step the segment executes.
 *   Consistency (eskf_keep_consistency) and the per-DOF getters cover the segment: *n_epochs = epoch_end - epoch_begin, row k
 *     is global epoch epoch_begin + k, bit-identical to that row of the whole run; the records and the ESKF_ENOMEM check are
 *     sized by the segment (N * (epoch_end - epoch_begin) * 352 bytes).
 *   Pre-pass budget (eskf_set_prepass_budget): sized by the segment's steps and epochs, so a segment can take the pre-pass
 *     path where the whole run would not.  With device-resident streams the segment's step counts are read back to size it
 *     (a small copy that makes the call synchronous); only when noise is on and a pre-pass is possible.
 * Rules: 0 <= epoch_begin <= epoch_end <= n_epochs, otherwise ESKF_EINVAL; variant 1 (eskf_kernel): ESKF_EINVAL.  An empty
 * range (epoch_begin == epoch_end) launches nothing and changes nothing on the handle except that the consistency getters
 * then report zero epochs (with eskf_keep_consistency on) and eskf_get_group_sums reports its groups and no statistics; it copies carry_in to carry_out (zeros without carry_in) and does
 * NOT write stats_out / stats_sum.  A refused call leaves the handle unchanged.  eskf_run(h, s, ...) with n_epochs > 0 is
 * eskf_run_epochs(h, s, 0, n_epochs, NULL, NULL, ...). */
int eskf_run_epochs(eskf_t* h, const eskf_streams_t* streams, int64_t epoch_begin, int64_t epoch_end, const double* carry_in,
                    double* carry_out, double* stats_out, double* stats_sum, int mem);

/* Filter._states / _P / buffers read-back.  Any pointer may be NULL. */
int eskf_get_state(eskf_t* h, double* x, double* P, double* u_old, double* R_old, int32_t* status, int mem);

/* Filter.Fx / Filter.Fi (Filter.py:249-268; the reference sets both on every propagate): after eskf_keep_jacobians(h, 1)
 * the kernels file the Jacobian record of the LAST IMU step of every eskf_propagate / eskf_run launch (720 B per filter;
 * with stacked trajectories, the last step of the filter's own trajectory: sum(n_prop) may be less than n_steps),
 * and eskf_get_jacobians expands it into the dense matrices the reference holds: Fx [N,24,24], Fi [N,24,13]; either
 * pointer may be NULL.  Default kernel only. */
int eskf_keep_jacobians(eskf_t* h, int on);
int eskf_get_jacobians(eskf_t* h, double* Fx, double* Fi, int mem);

#define ESKF_NCONS 8
/* Filter consistency of eskf_run (no reference counterpart): after eskf_keep_consistency(h, 1) every eskf_run files, per
 * filter i and epoch e (every epoch has one update, n_prop[e] = 0 included):
 *   nis[i,e]  = r^T inv(S) r, r the 7-dim residual of the update (Filter.py:363-375), S = H P- H^T + R the innovation
 *               covariance it inverts; 7 in expectation for a consistent filter;
 *   nees[i,e] = eps^T inv(B) eps over the ESTIMATED DOFs (bit k of frozen_mask clear, d = 6 - popcount(frozen_mask & 63)
 *               of them): eps = dofs+ - gt_dofs after the update (rad / cm, the units of x[10:16]), B the block of error-state
 *               rows / columns 9..14 of the covariance after the update (Joseph form and reset), solved by LU with partial
 *               pivoting; d in expectation; NaN when d = 0.
 * Both are NaN where the update was not applied (ESKF_STATUS_* cases) and where the value is not finite.  Where the
 * measurement was dropped (eskf_set_meas_dropout) nis is NaN and nees is that of the PRIOR DOFs and DOF block (no update).
 * epoch_sum[e, 0:8] sums over the handle's filters, FINITE values only (a diverged filter is counted, never propagates):
 *   [0] number of finite NIS, [1] sum of NIS, [2] sum of NIS^2, [3] number of finite NEES, [4] sum, [5] sum of squares,
 *   [6] filters whose NIS is NaN although their measurement was not dropped, or whose NEES is NaN (d > 0), at e,
 *   [7] filters whose measurement was dropped at e (0 without dropout).
 * Fixed reduction tree, no atomics: the same inputs give the same bits; plain sums, so shards combine by all-reduce.
 * eskf_get_consistency returns those of the LAST such run: nis, nees [N,E]; epoch_sum [E,ESKF_NCONS]; *n_epochs = E.
 * Any pointer may be NULL (query E first).  The run files the records through the export instantiation of the persistent
 * kernel and needs N * E * 352 bytes of device memory for them (plus N * E * 16 for the results): eskf_run returns
 * ESKF_ENOMEM, before anything is launched and with the handle unchanged, when they do not fit.  eskf_propagate /
 * eskf_update neither file nor clear them; eskf_get_consistency before any such run is ESKF_EINVAL.  Default kernel only
 * (variant 1: ESKF_EINVAL). */
int eskf_keep_consistency(eskf_t* h, int on);
int eskf_get_consistency(eskf_t* h, double* nis, double* nees, double* epoch_sum, int64_t* n_epochs, int mem);

#define ESKF_NDOFSUM 80
/* Per-DOF view of the same records (no reference counterpart), for the calibration DOFs x[10:16] (three rotations in rad,
 * three translations in cm).  Both calls read the records of the LAST eskf_run since eskf_keep_consistency(h, 1), as
 * eskf_get_consistency does, with its rules: ESKF_EINVAL before any such run, after eskf_keep_consistency(h, 0) and with
 * variant 1; any pointer may be NULL; *n_epochs = E (E = 0 gives empty outputs); mem is ESKF_MEM_HOST (the call
 * synchronises) or ESKF_MEM_DEVICE (asynchronous on the handle's stream).  Neither changes anything eskf_run returned, and
 * eskf_run does no work for them.
 *
 * eskf_get_dof_history: dofs [N,E,6], the DOFs as the record holds them (after the update; before it where it was not
 * applied, which a NaN nis marks), and var [N,E,6], the diagonal of the DOF covariance block at the same instant.  A host
 * destination is filled through a device staging buffer of at most 64 MiB, filter rows at a time: the two arrays take
 * N * E * 96 bytes and need not fit in device memory.
 *
 * eskf_get_dof_envelope: dof_sum [E,ESKF_NDOFSUM], per epoch sums over the handle's filters, computed by the call from the
 * records.  With eps_i = dofs_i - gt_dofs[i] (the gt_dofs of that run) and B the 6x6 DOF block of the record, filter f
 * CONTRIBUTES at epoch e when its nis is finite or its measurement was dropped (its prior then) and, for every estimated DOF i (bit i of frozen_mask clear), eps_i and B_ii
 * are finite and B_ii > 0 and, for every pair of estimated DOFs, B_ij and B_ji are finite.  Row e:
 *   [0]  M, the contributing filters;  [1]  N - M, the excluded ones;
 *   [2 + 7 i .. 2 + 7 i + 6] for DOF i = 0..5: sum eps_i, sum eps_i^2, sum B_ii, sum eps_i^2 / B_ii, and the number of
 *        filters with eps_i^2 <= B_ii, eps_i^2 <= 4 B_ii, eps_i^2 <= 9 B_ii (compared as written: no square root);
 *   [44 .. 58] sum eps_i eps_j over the 15 pairs i < j, row-major (0,1), (0,2), ..., (4,5);
 *   [59 .. 73] sum (B_ij + B_ji) / 2 over the same pairs;   [74] filters whose measurement was dropped (eskf_set_meas_dropout);
 *   [75 .. 79] reserved (0).
 * Sums over contributing filters only; entries of frozen DOFs, and of pairs that involve one, are 0.  Fixed reduction tree,
 * no atomics: the same records give the same bits.  Plain sums: shards combine them by all-reduce.  The run reserves the
 * row and its partial sums with the records (ESKF_ENOMEM before launch covers them). */
int eskf_get_dof_history(eskf_t* h, double* dofs, double* var, int64_t* n_epochs, int mem);
int eskf_get_dof_envelope(eskf_t* h, double* dof_sum, int64_t* n_epochs, int mem);

/* Filter groups (no reference counterpart): the sums of eskf_run (stats_sum), eskf_get_consistency (epoch_sum) and
 * eskf_get_dof_envelope (dof_sum) per group of filters instead of over the whole handle, for batches whose filters are not
 * exchangeable: stacked trajectories, tuning candidates.
 *
 * eskf_set_groups: group size g of the NEXT eskf_run / eskf_run_epochs; 0 (the default) is no grouping, a negative value
 * ESKF_EINVAL.  Filter f of a handle whose run had filter_id0 = id0 belongs to GLOBAL group (id0 + f) / g, the rule of the
 * trajectories and of noise_id_modulus: g = filters_per_traj gives one group per trajectory, g = noise_id_modulus one per
 * candidate.  The handle's filters cover groups group0 = id0 / g .. (id0 + N - 1) / g; the first and the last may be
 * partial.  A run records its g and filter_id0 with its results: eskf_set_groups between a run and a getter changes nothing
 * the getter returns.  With g > 0, a run that produces statistics rows (stats_out or stats_sum non-NULL) also reduces them
 * per group into the handle (two more small launches; none without groups), masked as stats_sum; a segment's are
 * accumulated over epochs [0, epoch_end) like its stats_sum.  Everything else a run returns is the same with or without
 * groups.
 *
 * eskf_get_group_sums: stats_sum [G,ESKF_NSTAT], epoch_sum [G,E,ESKF_NCONS], dof_sum [G,E,ESKF_NDOFSUM] of the last run;
 * row k is global group *group0 + k and has the layout and meaning of the ungrouped vector.  G = 1 and *group0 = 0 for a run
 * without groups.  Any pointer may be NULL (query G and E first).  epoch_sum and dof_sum follow the rules of
 * eskf_get_consistency / eskf_get_dof_envelope: the records of the last run since eskf_keep_consistency(h, 1), ESKF_EINVAL
 * otherwise and with variant 1, a segment's epochs only; they are computed by the call from the records, which it does not
 * change, nor anything else a run returned.  A non-NULL stats_sum is ESKF_EINVAL when the last run produced no statistics
 * rows or ran without groups (an empty eskf_run_epochs range produces none).  *n_epochs = E (0 without records).
 * ESKF_EINVAL when E x blocks, the grid of the consistency or envelope reduction, exceeds 2^31 - 1 (tiny groups over many
 * epochs): take larger groups or shorter segments.  The call allocates its partial sums (E * blocks * 88
 * doubles, blocks = G + N / 4096 at most, plus the outputs for a host destination); ESKF_ENOMEM when they do not fit,
 * leaving every result readable.  mem: as for eskf_get_dof_envelope.
 * Reduction: every group is cut into blocks of at most 4096 filters from its first one, each block summed over a fixed
 * tree, the blocks of a group added in order: the same records give the same bits, and a group's row is bit-identical to the
 * ungrouped sum of a handle holding exactly that group's filters.  Shards: a group cut by a shard boundary appears as a
 * partial row in both shards; adding the rows gives the group's sums (dvi_ekf_b200.sharding.place_group_rows puts a shard's
 * rows at their global groups for the all-reduce). */
int eskf_set_groups(eskf_t* h, int64_t group_size);
int eskf_get_group_sums(eskf_t* h, double* stats_sum, double* epoch_sum, double* dof_sum, int64_t* group0, int64_t* n_groups,
                        int64_t* n_epochs, int mem);

/* Simulated frame loss (no reference counterpart): per-filter, per-epoch measurement dropout of eskf_run / eskf_run_epochs, drawn
 * on the device.  prob [n_traj, n_epochs] in `mem` space (the whole trajectory's epochs, as the streams) is copied into the
 * handle and applies to every later run until it is changed; NULL switches dropout off (the default).  Every entry must be
 * finite and in [0, 1], else ESKF_EINVAL and the handle is unchanged; a device array is read back to check it (the call is
 * synchronous).  A run returns ESKF_EINVAL, before anything is launched and with the handle unchanged, when (n_traj, n_epochs)
 * differ from its streams' or with variant 1.  eskf_propagate / eskf_update ignore the setting.
 * Rule: filter g (global id) with noise id gid (g % noise_id_modulus when the modulus is > 0, else g) loses the measurement of
 * global epoch e iff u < prob[trajectory of g, e], u = (x + 1/2) 2^-32 in (0, 1) and x word 0 of Philox4x32-10(key = seed,
 * counter = (e lo, 3 * 16 + (e hi << 8), gid lo, gid hi)) -- the layout of the noise draws with kind ESKF_NOISE_DROP
 * (eskf_noise_dump reads u back).  prob = 0 never drops, prob = 1 always drops; with noise_free_filter0, noise id 0 makes no
 * random drop and loses exactly the epochs with prob = 1.  Within one noise id the masks nest: prob1 <= prob2 drops a subset
 * of the epochs prob2 drops.  The draw depends on neither noise std, and no other draw moves: segments, shards and
 * noise_id_modulus see the masks of one whole run.
 * A dropped measurement: the update is not applied (state and covariance stay at the prior; the trace row of the epoch's last
 * step keeps the propagated state), no status bit is set and the residual is not evaluated; statistics row [9] does not count
 * it; the update MSE of the epoch is evaluated as always, from the state at the frame instant.  Consistency: see
 * eskf_get_consistency and eskf_get_dof_envelope (nis NaN, nees of the prior, epoch_sum[7] and dof_sum[74] the dropped count).
 * A run with dropout runs the export instantiation of the persistent kernel. */
int eskf_set_meas_dropout(eskf_t* h, const double* prob, int64_t n_traj, int64_t n_epochs, int mem);

/* blocks until everything queued on the handle's stream has finished */
int eskf_sync(eskf_t* h);

/* number of kernels this library has launched on the handle so far */
int64_t eskf_launch_count(const eskf_t* h);
/* filters per CTA used for the kernels (tunable; 0 = automatic) */
int eskf_set_tuning(eskf_t* h, int filters_per_cta);
/* eskf_run keeps the Monte-Carlo generator and the update-MSE statistics OUT of the persistent kernel when their buffers
 * fit this budget: a pre-pass kernel writes the noisy per-filter sample streams ([T,N,6] + [E,N,8] doubles), the
 * persistent kernel leaves a 14-double snapshot per filter and update ([E,N,14]) and a post-pass evaluates the Euler
 * angles of Filter.calculate_update_mse (Filter.py:397-418) from them.  Same generator, same operations: bit-identical to
 * the in-kernel path (bytes = 0), which serves the sizes that do not fit.  Default: 32 GiB or ESKF_B200_PP_MAX_BYTES. */
int eskf_set_prepass_budget(eskf_t* h, int64_t bytes);
/* kernel variant: 0 = default (the warp-specialised eskf_kernel3), 1 = eskf_kernel (first version, kept for
 * A/B measurements), 3 = eskf_kernel3 */
int eskf_set_variant(eskf_t* h, int variant);

/* Monte-Carlo noise read-back (no reference counterpart): the standard normals the kernels draw for
 * filters filter_id0 .. filter_id0 + n_filters - 1 and steps step0 .. step0 + n_steps - 1 of one stream,
 * out[n_filters][n_steps][8].  kind = ESKF_NOISE_IMU: z[0..5] scale om(3), acc(3) of IMU sample `step`;
 * kind = ESKF_NOISE_CAM: z[0..2] camera position, z[3..5] small body rotation of the measured quaternion,
 * z[6] notch angle of camera epoch `step`.  The generator uses the device's SFU approximations, so THIS is
 * the definition of the noise a run saw: parity tests feed these samples to the oracle.  kind = ESKF_NOISE_DROP: z[0] is the
 * dropout uniform u of filter id `filter_id0 + f` and epoch `step` (eskf_set_meas_dropout), z[1..7] are 0. */
enum { ESKF_NOISE_IMU = 1, ESKF_NOISE_CAM = 2, ESKF_NOISE_DROP = 3 };
int eskf_noise_dump(int device, void* cuda_stream, uint64_t seed, int64_t filter_id0, int64_t n_filters, int64_t step0,
                    int64_t n_steps, int kind, double* out, int mem);

/* GPU pre-pass == Simulator.__init__ / Camera / Interpolator / Imu.eval_expr_single (Simulator.py:30-68,
 * Camera.py:84-118,158-170,299-347, Interpolator.py:25-88, Imu.py:141-226, tools/utils.py:54-75): from one camera
 * trajectory to the streams eskf_run consumes.  Inputs are HOST arrays, outputs DEVICE buffers owned by the caller with
 * capacity T_max = (n_frames - 1) * interframe_vals steps and E = n_frames - 1 epochs; the number of IMU steps actually
 * produced (epoch membership is decided by t_interp <= t_frame, quirk Q14) is returned in *n_steps_out. */
typedef struct {
  int64_t n_frames;
  int32_t interframe_vals;  /* config.yaml imu.interframe_vals */
  int32_t euler_mode;       /* 0: extrinsic xyz (HEAD); 1: zyx reversed (the revision that wrote the golden files) */
  double scale;             /* camera.scale (VisualTrajectory.py:99-108) */
  double gt_dofs[6];        /* config.gt_imu_dofs: probe used to synthesise the IMU */
  double ic_dofs[6];        /* config.ic_imu_dofs: DOFs of the initial state */
  const double* t;          /* [n]   frame stamps */
  const double* xyz;        /* [n,3] unscaled positions */
  const double* q_xyzw;     /* [n,4] raw quaternions */
  const double* notch3;     /* [n,3] notch angle, rate, acceleration, or NULL (with_notch: false).  When given, the IMU
                               samples, x0 and cam_ref come from the ROTATED camera (Camera.gen_rotated, Camera.py:172-208)
                               and `cam` keeps the raw quaternions of the un-rotated one, as Filter.run sees them */
} eskf_prepass_in_t;
typedef struct {
  double* x0;               /* [26]       initial nominal state */
  double* u0;               /* [6]        first IMU sample (Filter.py:63,78-79) */
  double* dt;               /* [T_max] */
  double* om_acc;           /* [T_max,6] */
  double* t_imu;            /* [T_max]    nullable */
  int32_t* n_prop;          /* [E] */
  double* cam;              /* [E,7] */
  double* notch;            /* [E] */
  double* cam_ref;          /* [E,6] */
  double* imu_ref;          /* [E,6] */
  double* imu_ref_rows;     /* [T_max,14] ImuRefTraj rows (ImuRefTraj.py:18-55), nullable */
} eskf_prepass_out_t;
int eskf_prepass(int device, void* cuda_stream, const eskf_model_t* model, const eskf_prepass_in_t* in,
                 const eskf_prepass_out_t* out, int64_t* n_steps_out);
const char* eskf_prepass_last_error(void);

/* Measurement aid (no reference counterpart): sustained FP64 FMA throughput of the device in
 * TFLOP/s (best of `repeats` launches of a pure DFMA kernel) -- the roofline denominator. */
int eskf_fp64_peak(int device, void* cuda_stream, int repeats, double* tflops_out, double* ms_out);

const char* eskf_last_error(void);
const char* eskf_version(void);

#ifdef __cplusplus
}
#endif
#endif /* ESKF_B200_H */
