/*
 * cpi_b200.h -- C ABI of libcpi_b200.so: batched closed-form IMU preintegration (CPI) on B200 (sm_100a).
 *
 * This is the drop-in boundary for the ONE hot path of rpng/cpi (reference tree paths are relative to
 * /root/reference/cpi_compare/src):
 *
 *   cpi_preintegrate_batch*    replaces the per-sample loop  CpiV1::feed_IMU  (cpi/CpiV1.h:62-361) and
 *                              CpiV2::feed_IMU (cpi/CpiV2.h:84-467) as driven, once per factor, by
 *                              GraphSolver::createimufactor_cpi_v1/_v2 (solvers/GraphSolver_IMU.cpp:43-75, 97-130),
 *                              for MANY windows at once.  Its per-window output record is exactly the set of public
 *                              CpiBase fields the caller reads afterwards (cpi/CpiBase.h:99-124, cpi/CpiV2.h:62-63).
 *   cpi_imu_factor_eval_batch* replaces ImuFactorCPIv1::evaluateError (gtsam/ImuFactorCPIv1.cpp:37-208) and
 *                              ImuFactorCPIv2::evaluateError (gtsam/ImuFactorCPIv2.cpp:38-212): unwhitened 15-d
 *                              residual and the two 15x15 Jacobians, for many factors at once.
 *   cpi_imu_factor_hessian_batch  the step GTSAM performs next: information-form blocks H^T P^-1 H, -H^T P^-1 e per factor.
 *   cpi_predict_state_batch*   replaces GraphSolver::getpredictedstate_v1/_v2 (solvers/GraphSolver_IMU.cpp:263-307).
 *   cpi_retract_batch*         replaces JPLNavState::retract (gtsam/JPLNavState.cpp:37-71).
 *
 * Conventions (all identical to the reference):  fp64; matrices COLUMN-major (Eigen default); JPL quaternion
 * [x y z w]; 15-d error-state order [dtheta(0:3), b_g(3:6), v/beta(6:9), b_a(9:12), p/alpha(12:15)]
 * (cpi/CpiV1.h:277-281, gtsam/ImuFactorCPIv1.cpp:80-88).
 *
 * Functions without the _host suffix take DEVICE pointers and enqueue on `stream` (a cudaStream_t passed as
 * void*; NULL = legacy default stream) without synchronising.  *_host variants take HOST pointers (pinned or pageable),
 * copy through device buffers owned by the library -- big batches in a 4-deep H2D / kernel / D2H pipeline -- and return
 * after the results are in the caller's buffers.
 * Every function returns CPI_OK (0) or a negative CPI_E* code; cpi_last_error() gives the message of the last
 * failure on the calling thread.  (The reference has no error convention for this path: feed_IMU returns void and
 * never checks its inputs -- CpiBase.h:86.)  No function falls back to a CPU implementation.
 */
#ifndef CPI_B200_H
#define CPI_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- layouts -------------------------------------------------------------------------------------------------- */

/* One IMU entry: [wx wy wz ax ay az dt] ; dt = t_{i+1} - t_i (seconds) is the length of the step that STARTS at this
 * entry, i.e. feed_IMU(t_i, t_i + dt, w_i, a_i, w_{i+1}, a_{i+1}).  The reference's line format "wx wy wz ax ay az
 * <unused> t_ms" (sim/SimParser.h:148-175) maps to this after differencing the time stamps. */
#define CPI_SAMPLE_DOUBLES 7
/* Per-window linearisation point = arguments of CpiBase::setLinearizationPoints (cpi/CpiBase.h:73-80):
 * [b_w_lin(3) b_a_lin(3) q_k_lin(4, JPL xyzw) grav(3)].  Model 1 ignores q_k_lin for preintegration; grav is only
 * carried to the factor (GraphSolver_IMU.cpp:74). */
#define CPI_LIN_DOUBLES 13
/* JPLNavState value (gtsam/JPLNavState.h:62-66): [q_GtoI(4) b_g(3) v_IinG(3) b_a(3) p_IinG(3)] */
#define CPI_STATE_DOUBLES 16

/* Per-window result record, doubles.  Field order = order the factor constructors consume them
 * (gtsam/ImuFactorCPIv1.h:78-81, gtsam/ImuFactorCPIv2.h:82-85). */
#define CPI_REC_Q      0    /* q_k2tau  [4]  rot_2_quat(R_k2tau)            CpiBase.h:102 */
#define CPI_REC_R      4    /* R_k2tau  [9]  col-major                      CpiBase.h:103 */
#define CPI_REC_ALPHA  13   /* alpha_tau[3]                                 CpiBase.h:100 */
#define CPI_REC_BETA   16   /* beta_tau [3]                                 CpiBase.h:101 */
#define CPI_REC_DT     19   /* DT                                           CpiBase.h:99  */
#define CPI_REC_JQ     20   /* J_q [9]  d(theta)/d(b_w)                     CpiBase.h:106 */
#define CPI_REC_JA     29   /* J_a [9]  d(alpha)/d(b_w)                     CpiBase.h:107 */
#define CPI_REC_JB     38   /* J_b [9]  d(beta)/d(b_w)                      CpiBase.h:108 */
#define CPI_REC_HA     47   /* H_a [9]  d(alpha)/d(b_a)                     CpiBase.h:109 */
#define CPI_REC_HB     56   /* H_b [9]  d(beta)/d(b_a)                      CpiBase.h:110 */
#define CPI_REC_P      65   /* P_meas [225] col-major 15x15                 CpiBase.h:124 */
#define CPI_REC_V1_DOUBLES 290
#define CPI_REC_OA     290  /* O_a [9]  d(alpha)/d(theta_k_lin)  (model 2)  CpiV2.h:62 */
#define CPI_REC_OB     299  /* O_b [9]  d(beta)/d(theta_k_lin)   (model 2)  CpiV2.h:63 */
#define CPI_REC_V2_DOUBLES 308

/* flags */
#define CPI_FLAG_IMU_AVG             1  /* CpiBase::imu_avg = true (CpiBase.h:95); each window then carries ONE extra
                                           trailing entry whose (w,a) are the "_1" arguments of the last step */
#define CPI_FLAG_ANALYTIC_JACOBIANS  2  /* model 2 only: state_transition_jacobians = false (CpiV2.h:58); default
                                           (flag clear) is the reference's default/true path (GraphSolver_IMU.cpp:100) */

/* error codes */
#define CPI_OK          0
#define CPI_EINVAL     -1   /* bad argument (NULL pointer, unknown model/dtype, negative count) */
#define CPI_ECUDA      -2   /* a CUDA runtime call failed; see cpi_last_error() */
#define CPI_ENODEVICE  -3   /* no CUDA device / not an sm_100 device */
#define CPI_ENOMEM     -4

/* ---- preintegration ---------------------------------------------------------------------------------------------- */

/*
 * Preintegrate n_windows independent windows.
 *   model          1 (CpiV1) or 2 (CpiV2)
 *   dtype          64 (fp64; samples/lin/records are double) or 32 (fp32 storage: float samples/lin/records,
 *                  see DESIGN.md for the mixed-precision rule)
 *   sample_offsets device int64[n_windows+1], entry index (not bytes) of each window's first entry in `samples`;
 *                  or NULL for uniform windows of `ns_uniform` steps laid out back to back.
 *                  Window w has  steps = offsets[w+1]-offsets[w]  (minus 1 if CPI_FLAG_IMU_AVG).  Device-resident offsets cannot
 *                  be validated by this entry point: a decreasing pair yields a zero-step window (the _host variant checks
 *                  its host copy and returns CPI_EINVAL instead).
 *   samples        device, CPI_SAMPLE_DOUBLES per entry.  The kernels stage every window's stream with 128-byte TMA bulk reads that
 *                  start at the 16-byte boundary at or below the window's first entry: `samples` must be 16-byte aligned (any
 *                  cudaMalloc / torch allocation is), so that no read begins before the buffer; reads never extend past the
 *                  last entry of the buffer (the tail of every window is read with plain loads).
 *   lin            device, CPI_LIN_DOUBLES per window
 *   sigmas         HOST double[4] = {sigma_w, sigma_wb, sigma_a, sigma_ab}  (CpiBase ctor, CpiBase.h:52-57)
 *   out_records    device, CPI_REC_V1_DOUBLES (model 1) or CPI_REC_V2_DOUBLES (model 2) per window
 * A window with zero steps yields the reference's freshly constructed object: R = I, everything else 0
 * (q_k2tau is uninitialised in the reference, CpiBase.h:102; this library writes [0 0 0 1]).
 */
int cpi_preintegrate_batch(int model, int dtype, int64_t n_windows,
                           const int64_t* sample_offsets, int64_t ns_uniform,
                           const void* samples, const void* lin, const double* sigmas, int flags,
                           void* out_records, void* stream);

/*
 * Continue n_windows preintegrations with MORE samples: `records` (device) holds, per window, the record left by an earlier
 * cpi_preintegrate_batch / _continue call and is updated in place -- the batched form of calling feed_IMU again on existing CpiV1 /
 * CpiV2 objects (feed_IMU accumulates into the object's fields, CpiBase.h:86, 99-124; every one of them is in the record).
 * `samples` / `sample_offsets` / `ns_uniform` describe the NEW samples only; lin, sigmas, flags must be those of the first call.
 * fp64: agrees with the one-shot call to rounding (~1e-15 relative; P_pp is re-split symmetrically).  dtype 32 continues from the
 * float-rounded record (the one-shot call carries the covariance state in fp64).  Default modes only (no CPI_FLAG_IMU_AVG, model 2
 * without CPI_FLAG_ANALYTIC_JACOBIANS): CPI_EINVAL otherwise.
 */
int cpi_preintegrate_batch_continue(int model, int dtype, int64_t n_windows,
                                    const int64_t* sample_offsets, int64_t ns_uniform,
                                    const void* samples, const void* lin, const double* sigmas, int flags,
                                    void* records, void* stream);

/* Same with HOST buffers: H2D + kernel + D2H, synchronous, through device buffers owned by the library; batches above 16 MB are
 * pipelined in up to 16 whole-window chunks (copy-in of chunk k+1 under the kernel of chunk k, copy-out under the next kernel); with a
 * uniform layout in the default fp64 modes the LAST windows of the batch (as many as take about one sample chain to transfer) travel
 * sample-major instead -- four strided segment copies, each followed by a continuation kernel over those windows -- so that their
 * chains of dependent samples run while the samples are still arriving and only a quarter of one chain is left behind the last byte
 * (results agree with the device entry point to rounding, ~1e-15; CPI_B200_HOST_WAVE="groups,segments[,head %]" overrides).  sample_offsets
 * is a HOST array.  The copies are cudaMemcpyAsync straight from / to the caller's buffers: PINNED buffers (cudaHostAlloc, or
 * cpi_host_register below) overlap with the kernels; pageable buffers are legal but the CUDA driver stages them synchronously, so
 * the pipeline degrades to copy-then-compute.  Calls from several host threads serialise on the library's scratch buffers. */
int cpi_preintegrate_batch_host(int model, int dtype, int64_t n_windows,
                                const int64_t* sample_offsets, int64_t ns_uniform,
                                const void* samples, const void* lin, const double* sigmas, int flags,
                                void* out_records);

/* Diagnostics of the last cpi_preintegrate_batch_host call of this process: host time until everything was enqueued, and until the
 * streams were drained (milliseconds).  Either pointer may be NULL. */
int cpi_host_last_timing(double* submit_ms, double* total_ms);

/* Pin / unpin a caller-owned host buffer for the *_host entry points (cudaHostRegister / cudaHostUnregister), for C callers that do
 * not link the CUDA runtime themselves.  Registering is expensive (~ms per 100 MB): do it once per buffer, not per call. */
int cpi_host_register(void* ptr, size_t bytes);
int cpi_host_unregister(void* ptr);

/* ---- factor evaluation ------------------------------------------------------------------------------------------- */

/*
 * Evaluate n IMU factors.  Factor f links states[idx_i[f]] -> states[idx_j[f]] (idx arrays may be NULL: then
 * idx_i[f] = f, idx_j[f] = f+1, the reference's chain X(k),X(k+1) -- GraphSolver_IMU.cpp:74) and uses
 * records[f] / lin[f] (the window's record and linearisation point, i.e. the factor's constructor arguments).
 *   e   device double[n*15]            residual  [2*q_r(0:3); bg_j-bg_i; betahat-beta; ba_j-ba_i; alphahat-alpha]
 *   H1  device double[n*225] col-major d e / d x_i   (may be NULL)
 *   H2  device double[n*225] col-major d e / d x_j   (may be NULL)
 * Unwhitened, exactly what evaluateError returns; the Gaussian::Covariance(P_meas) whitening lives in GTSAM.
 */
int cpi_imu_factor_eval_batch(int model, int64_t n_factors,
                              const double* states, const int64_t* idx_i, const int64_t* idx_j,
                              const double* records, const double* lin,
                              double* e, double* H1, double* H2, void* stream);

int cpi_imu_factor_eval_batch_host(int model, int64_t n_factors, int64_t n_states,
                                   const double* states, const int64_t* idx_i, const int64_t* idx_j,
                                   const double* records, const double* lin,
                                   double* e, double* H1, double* H2);

/*
 * Information-form linearisation of n factors (device pointers), the step GTSAM performs right after evaluateError with
 * the factor's noise model noiseModel::Gaussian::Covariance(P_meas) (gtsam/ImuFactorCPIv1.h:82, ImuFactorCPIv2.h:86):
 *     G11 = H1^T P^-1 H1, G12 = H1^T P^-1 H2, G22 = H2^T P^-1 H2  (15x15 column-major each),
 *     g1 = -H1^T P^-1 e, g2 = -H2^T P^-1 e  (15 each),  f = e^T P^-1 e      [HessianFactor convention: G, g = A^T b, f = b^T b]
 * P = records[f].P_meas; e / H1 / H2 as produced by cpi_imu_factor_eval_batch.  A factor whose covariance is not positive
 * definite (e.g. a zero-step window) gets NaN outputs (GTSAM throws there).  GTSAM itself is not in the reference tree
 * (bitbucket gtborg/gtsam @ c21186c), so this entry point is validated against a dense CPU solve only: PARITY UNPINNED.
 */
int cpi_imu_factor_hessian_batch(int model, int64_t n_factors, const double* records,
                                 const double* e, const double* H1, const double* H2,
                                 double* G11, double* G12, double* G22, double* g1, double* g2, double* f, void* stream);

/*
 * The explicitly whitened Jacobian form GTSAM's NoiseModelFactor::linearize produces with Gaussian::Covariance(P_meas):
 *     A1 = R_w H1,  A2 = R_w H2  (15x15 column-major each),  b = -R_w e  (15),   R_w = upper Cholesky factor of P_meas^-1.
 * PARITY UNPINNED (GTSAM is not in the reference tree); validated against numpy: A^T A = H^T P^-1 H, R_w upper triangular.
 */
int cpi_imu_factor_whiten_batch(int model, int64_t n_factors, const double* records,
                                const double* e, const double* H1, const double* H2,
                                double* A1, double* A2, double* b, void* stream);

/*
 * IMU-only chain x_0 - x_1 - ... - x_n (factor f links states f and f+1): what the smoother assembles and solves after the
 * linearisation (solvers/GraphSolver.cpp:202-203), on the device.
 *   cpi_imu_chain_assemble   scatter-add of the blocks of cpi_imu_factor_hessian_batch into the block-tridiagonal normal equations:
 *       D[k] (n+1 blocks 15x15) = G22[k-1] + G11[k] (+ prior_info0 on x_0) + damping,  E[k] (n blocks, block (k,k+1)) = G12[k],
 *       rhs[k] (15) = g2[k-1] + g1[k] (+ prior_rhs0).  prior_* may be NULL.  Damping as in GTSAM's LevenbergMarquardtParams:
 *       lambda I (diagonal_damping = 0, GTSAM's default) or lambda * clamp(diag D[k], 1e-6, 1e32) (diagonal_damping = 1, Marquardt).
 *       NOTE: an IMU-only chain anchored by one prior is numerically singular in fp64 beyond a few hundred keyframes with
 *       undamped / lambda-I normal equations (the drift modes carry ~1e-16 of the largest eigenvalue) -- for ANY elimination order;
 *       diagonal damping (or the camera factors of the real graph) restores a well-posed system (DESIGN.md section 5).
 *   cpi_imu_chain_solve      x = (that SPD block-tridiagonal matrix)^-1 rhs by block cyclic reduction (Cholesky on the 15x15 pivots):
 *       ~2 log2(n) + 1 kernel launches instead of an n-step sequential block recurrence.  `workspace`: device buffer of
 *       cpi_imu_chain_solve_workspace(n_states) bytes.  The step is then applied with cpi_retract_batch.
 * All pointers are DEVICE pointers.  PARITY UNPINNED; validated against banded / dense CPU solves of the same system.
 */
int cpi_imu_chain_assemble(int64_t n_factors, const double* G11, const double* G12, const double* G22,
                           const double* g1, const double* g2, double lambda, int diagonal_damping,
                           const double* prior_info0, const double* prior_rhs0,
                           double* D, double* E, double* rhs, void* stream);
int64_t cpi_imu_chain_solve_workspace(int64_t n_states);
int cpi_imu_chain_solve(int64_t n_states, const double* D, const double* E, const double* rhs,
                        double* x, void* workspace, void* stream);

/*
 * Marginal covariances of the chain: the diagonal and first off-diagonal 15x15 blocks of Sigma = A^-1 for the SPD block-tridiagonal
 * A = tridiag(E^T, D, E) of cpi_imu_chain_assemble -- what GTSAM's Marginals::marginalCovariance(x_k) and the (x_k, x_k+1) block of
 * jointMarginalCovariance return at the linearisation point (assemble with lambda = 0 for that).  Selected inversion by block cyclic
 * reduction: the forward sweep of cpi_imu_chain_solve without right-hand side, then one pass per level from the root down, 3 ceil(log2 n) + 1
 * kernel launches; no dense inverse is formed.
 *   S_diag  device double[n_states * 225]      block k = Sigma_kk, column-major, exactly symmetric
 *   S_off   device double[(n_states-1) * 225]  block k = Sigma_k,k+1 (column-major), or NULL when only the diagonal blocks are wanted
 *   workspace  device buffer of cpi_imu_chain_marginals_workspace(n_states) bytes
 * All pointers are DEVICE pointers; enqueued on `stream` without synchronising; n_states = 0 is a no-op.  A matrix that is not positive
 * definite gives NaN outputs.  The NOTE above applies unchanged: an undamped IMU-only chain anchored by one prior is numerically singular in
 * fp64 beyond a few hundred keyframes, and so are its covariances; the other factors of the real graph (or a prior per keyframe) make it
 * well posed.  PARITY UNPINNED (GTSAM is not in the reference tree); validated against dense inverses, against the covariance the filter's
 * forward propagation gives for a chain anchored at x_0 only, and against refined banded CPU solves.
 */
int64_t cpi_imu_chain_marginals_workspace(int64_t n_states);
int cpi_imu_chain_marginals(int64_t n_states, const double* D, const double* E,
                            double* S_diag, double* S_off, void* workspace, void* stream);

/* ---- callers either side of the factor ("next" rows) ----------------------------------------------------------------- */

/* x_{k+1} prediction from x_k and a record: getpredictedstate_v1/_v2 (GraphSolver_IMU.cpp:263-307).
 * states_k / states_k1: device, CPI_STATE_DOUBLES per window. */
int cpi_predict_state_batch(int model, int64_t n, const double* states_k, const double* records, const double* lin,
                            double* states_k1, void* stream);

/* JPLNavState::retract (JPLNavState.cpp:37-71): states_out[i] = states[i] (+) xi[i], xi = 15 doubles each. */
int cpi_retract_batch(int64_t n, const double* states, const double* xi, double* states_out, void* stream);

/* ---- window builder (host) ------------------------------------------------------------------------------------------------------ */

/*
 * Cut one IMU stream into the windows the reference preintegrates, one per update (camera) time: the loop of
 * GraphSolver::createimufactor_cpi_v1/_v2 (solvers/GraphSolver_IMU.cpp:50-69, 105-124) incl. the partial tail step and the
 * rewrite of the front stamp, fed as SimulationLoader::execute_publishing delivers the messages (sim/SimulationLoader.cpp:214-290:
 * the IMU reading first at equal stamps) and initialised as GraphSolver::trytoinitalize does (solvers/GraphSolver.cpp:264, 357: the
 * first update that finds >= imu_wait queued readings emits no window and keeps only the newest reading; imu_wait = 0: no such phase).
 *   t[n_imu] seconds (non-decreasing), w / a [n_imu * 3], update_times[n_updates] (non-decreasing) -- all HOST arrays
 *   samples   HOST, capacity cap_entries entries of CPI_SAMPLE_DOUBLES (may be NULL to count only)
 *   offsets   HOST int64[n_updates + 1]; window k is entries offsets[k] .. offsets[k+1]-1 (CSR layout of cpi_preintegrate_batch)
 * Returns the number of windows (<= n_updates) or a negative CPI_E* code; *n_entries receives the number of entries.
 */
int64_t cpi_cut_windows(int64_t n_imu, const double* t, const double* w, const double* a,
                        int64_t n_updates, const double* update_times, int64_t imu_wait,
                        int64_t cap_entries, double* samples, int64_t* offsets, int64_t* n_entries);

/* ---- multi-GPU: one process per GPU, window batches sharded over the ranks ------------------------------------------------ */

/*
 * Windows share nothing but the four sigmas (the reference constructs a fresh preintegrator per factor,
 * solvers/GraphSolver_IMU.cpp:43), so a batch shards contiguously: rank r preintegrates its n_local windows and the only
 * exchange is ONE in-place all-gather of the fixed-size records (NCCL, or copy-engine peer copies for registered buffers), after which every rank -- in particular rank 0, where
 * the solver lives -- holds all world * n_local records in window order.  NCCL is bound at run time (dlopen libnccl.so.2).
 *
 *   cpi_comm_unique_id   rank 0: 128-byte NCCL id to hand to the other ranks (any out-of-band channel)
 *   cpi_comm_create      collective over all ranks, on the CURRENT device of each process
 *   cpi_preintegrate_batch_sharded
 *        enqueues the kernel for this rank's n_local windows on `stream`, writing records straight into slice `rank` of
 *        gather_records (device, world * n_local records: no pack kernel), then the all-gather on the communicator's own
 *        stream behind an event.  Returns without synchronising: the next batch's kernel (into ANOTHER gather buffer)
 *        overlaps the collective.  Re-using a gather buffer orders the new kernel behind that buffer's previous all-gather.
 *        n_local must be the same on every rank (pad a short last shard with zero-step windows).
 *   cpi_comm_register    collective, optional, once per gather buffer (same buffers in the same order on every rank): exports the buffer
 *        with CUDA IPC and maps the peers' buffers, after which cpi_preintegrate_batch_sharded exchanges the records by COPY-ENGINE
 *        copies of every rank's slice into the peers' buffers over NVLink instead of an ncclAllGather kernel, bracketed by two barriers
 *        that are SM-free as well (4-byte copy-engine writes into the peers' flag words + cuStreamWaitValue32; one-element NCCL
 *        all-reduces where stream memory operations are unavailable): nothing is taken from, or has to wait for, the preintegration
 *        kernel that runs beside the exchange.  *peer_copies (may be NULL)
 *        tells whether that path is active; it is not when any rank could not export / import (e.g. memory from a VMM / async pool) --
 *        the buffer then simply keeps the NCCL path.
 *   cpi_comm_unregister  drops the registration of one buffer (NULL: of all) and closes the peer mappings nothing refers to any more.
 *        EVERY rank must have unregistered a buffer before ANY rank frees it (freeing memory a peer still has mapped is undefined in
 *        CUDA IPC): unregister, synchronise the ranks, then free.
 *   cpi_comm_wait        makes `stream` wait for the most recently enqueued exchange (call before consuming the records)
 * The usual NCCL rule applies: collectives of ANOTHER communicator on the same devices (e.g. an MPI / torch.distributed NCCL group)
 * must not be in flight at the same time as this communicator's all-gathers -- synchronise the device between the two.
 */
#define CPI_COMM_ID_BYTES 128
typedef struct cpi_comm cpi_comm;
int cpi_comm_unique_id(void* id_out);
int cpi_comm_create(const void* id, int rank, int world, cpi_comm** out);
int cpi_comm_destroy(cpi_comm* comm);
int cpi_comm_rank(const cpi_comm* comm);
int cpi_comm_world(const cpi_comm* comm);
int cpi_comm_sm_free_barriers(const cpi_comm* comm);   /* 1: the peer-copy exchange synchronises with copy-engine flag writes + stream wait-value ops; 0: with NCCL all-reduces */
int cpi_comm_register(cpi_comm* comm, void* gather_records, size_t bytes, int* peer_copies);
int cpi_comm_unregister(cpi_comm* comm, void* gather_records);
int cpi_preintegrate_batch_sharded(cpi_comm* comm, int model, int dtype, int64_t n_local,
                                   const int64_t* sample_offsets, int64_t ns_uniform,
                                   const void* samples, const void* lin, const double* sigmas, int flags,
                                   void* gather_records, void* stream);
int cpi_comm_wait(cpi_comm* comm, void* stream);

/* ---- misc ----------------------------------------------------------------------------------------------------------- */

const char* cpi_last_error(void);
const char* cpi_version(void);
int cpi_record_doubles(int model);          /* 290 or 308; CPI_EINVAL otherwise */
int cpi_device_count(void);                 /* number of usable sm_100 devices, or negative error */
/* number of kernel launches issued by this library on the calling process since load (for bench.py's gpu_launches) */
int64_t cpi_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* CPI_B200_H */
