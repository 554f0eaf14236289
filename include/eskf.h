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

/* Filter._states / _P / buffers read-back.  Any pointer may be NULL. */
int eskf_get_state(eskf_t* h, double* x, double* P, double* u_old, double* R_old, int32_t* status, int mem);

/* Filter.Fx / Filter.Fi (Filter.py:249-268; the reference sets both on every propagate): after eskf_keep_jacobians(h, 1)
 * the kernels file the Jacobian record of the LAST IMU step of every eskf_propagate / eskf_run launch (720 B per filter;
 * with stacked trajectories, the last step of the filter's own trajectory: sum(n_prop) may be less than n_steps),
 * and eskf_get_jacobians expands it into the dense matrices the reference holds: Fx [N,24,24], Fi [N,24,13]; either
 * pointer may be NULL.  Default kernel only. */
int eskf_keep_jacobians(eskf_t* h, int on);
int eskf_get_jacobians(eskf_t* h, double* Fx, double* Fi, int mem);

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
 * the definition of the noise a run saw: parity tests feed these samples to the oracle. */
enum { ESKF_NOISE_IMU = 1, ESKF_NOISE_CAM = 2 };
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
