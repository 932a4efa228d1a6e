/*
 * spp_b200.h -- C ABI of libspp_b200.so: the B200-native (sm_100a, FP64) implementation of the
 * nonlinear-least-squares hot path of SLAM++ (linearise -> landmark Schur complement -> FP64
 * Cholesky of the reduced camera / pose system -> landmark back-substitution).
 *
 * This is the drop-in boundary. Plain pointers and sizes only; every host pointer is BORROWED for
 * the duration of the call and never retained; the context owns all device memory. One caller
 * thread per context (the reference's solvers are single-caller, parallelism is internal); one
 * context drives one GPU (one process per GPU; the multi-GPU reduction is plugged in through
 * spp_set_allreduce()). There is NO CPU fallback: every entry point fails with SPP_ERR_CUDA when
 * no sm_100 device is usable.
 *
 * Each entry point cites the reference interface it replaces (paths relative to the SLAM++ tree).
 * Return codes: 0 ok, SPP_NOT_POSDEF (1) = the factorisation met a non-positive pivot (the
 * reference's solvers return false in that case), < 0 = error, text via spp_last_error().
 */
#ifndef SPP_B200_H
#define SPP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPP_OK 0
#define SPP_NOT_POSDEF 1
#define SPP_ERR_INVALID (-1)   /* bad argument / call order / unsupported structure */
#define SPP_ERR_CUDA (-2)      /* CUDA runtime error or no usable device */
#define SPP_ERR_NOMEM (-3)     /* host or device allocation failed (adapters throw std::bad_alloc) */
#define SPP_ERR_COMM (-4)      /* the all-reduce hook failed */

typedef struct spp_ctx *spp_ctx_t; /* opaque; models optimizer_t of include/ba_interface_example/BAOptimizer.h:120 */

/* Jacobian evaluation of the BA / SE(3) edges */
#define SPP_JAC_FD_REFERENCE 0 /* forward differences, delta = 1e-9, same operation order as the reference
                                  (include/slam/BASolverBase.h:579-619, include/slam/3DSolverBase.h:1336-1370) */
#define SPP_JAC_ANALYTIC 1     /* closed-form derivatives (agrees with the FD variant at the FD noise floor) */

/* report of one spp_*_optimize() call; mirrors what CNonlinearSolver_Lambda_LM::Optimize() prints / keeps
 * (include/slam/NonlinearSolver_Lambda_LM.h:796-1116) */
#define SPP_MAX_TRACE 64
typedef struct {
	int32_t n_iterations;       /* linear solves performed (incl. rejected LM steps) */
	int32_t n_accepted;         /* accepted steps */
	int32_t n_rejected;         /* rejected steps ("warning: chi2 rising") */
	int32_t status;             /* 0 ok, SPP_NOT_POSDEF if a factorisation failed (the loop stops, as the reference) */
	double chi2_initial;        /* f_Chi_Squared_Error_Denorm() before the first step */
	double chi2_final;          /* after the last accepted step */
	double alpha_initial;       /* LM: tau * max per-edge Hessian diagonal (LM.h:151-199); 0 for Gauss-Newton */
	double alpha_final;
	double last_dx_norm;        /* "residual norm" of the last increment */
	/* per-solve trace, first min(n_iterations, SPP_MAX_TRACE) entries */
	double trace_alpha[SPP_MAX_TRACE];    /* damping used by the solve */
	double trace_chi2[SPP_MAX_TRACE];     /* chi2 after applying the step (before accept/reject) */
	double trace_dx_norm[SPP_MAX_TRACE];
	uint8_t trace_accepted[SPP_MAX_TRACE];
	/* device time of the phases, milliseconds, summed over the call (CUDA events); phase names follow the
	 * reference's Dump() (LM.h:547-..): lambda, rhs/schur, linsolve, update, chi2 */
	double ms_linearise, ms_schur, ms_factor, ms_backsubst, ms_update, ms_chi2, ms_total;
	/* part of ms_factor: the launches of the dense factorisation kernel alone (k_chol_dataflow; 0 when the reduced system
	 * is factored block-sparse) -- the launch duration the roofline of that kernel is computed from */
	double ms_factor_kernel;
} spp_report_t;

/* ---- context ---------------------------------------------------------------------------------------- */

/* replaces New_Optimizer() / Free_Optimizer() (include/ba_interface_example/BAOptimizer.h:122-123) */
int spp_create(int device, spp_ctx_t *p_ctx);
void spp_destroy(spp_ctx_t ctx);
/* last error text of this context (valid until the next call); ctx may be NULL for creation errors */
const char *spp_last_error(spp_ctx_t ctx);
/* library / device identification: writes a short text such as "spp_b200 0.1 sm_100 NVIDIA B200" */
int spp_describe(spp_ctx_t ctx, char *p_buffer, size_t n_buffer_size);
/* number of kernel launches issued by this context since creation (bench.py reports it) */
uint64_t spp_kernel_launches(spp_ctx_t ctx);
/* the CUDA stream (cudaStream_t) all kernels of this context are launched on; for event timing by the caller */
void *spp_stream(spp_ctx_t ctx);
int spp_synchronize(spp_ctx_t ctx);

/* Multi-GPU hook. When set, the partial reduced camera system [S_upper | b] (and the scalar partial sums of
 * chi2, |dx|^2, ...) of this rank are summed over ranks by calling fn(user, device_pointer, n_doubles) -- the
 * caller implements it with torch.distributed / ncclAllReduce(sum, double) on the stream returned by
 * spp_stream() or any stream ordered after a spp_synchronize(). fn returns 0 on success.
 * rank / world select this rank's landmark slice (contiguous, balanced by sum k_p^2; SURVEY 8(e)).
 * The reference has no counterpart (single process, OpenMP). */
typedef int (*spp_allreduce_fn)(void *p_user, void *p_device_doubles, size_t n_doubles);
int spp_set_allreduce(spp_ctx_t ctx, spp_allreduce_fn fn, void *p_user, int rank, int world);

/* The library's own NCCL path (what a C++ host uses; the hook above remains for host-side tests over gloo). One process
 * per GPU: rank 0 calls spp_nccl_get_unique_id() and hands the SPP_NCCL_UNIQUE_ID_BYTES bytes to every rank by any means
 * (a file, MPI, torch.distributed); every rank then calls spp_set_nccl() -- collectively, it runs ncclCommInitRank. From
 * then on the partial reduced camera systems and the scalar partial sums are summed with ncclAllReduce(double, sum) on
 * the context's stream, inside the library, without host synchronisation. libnccl.so.2 is opened at run time (dlopen):
 * a process that already holds an NCCL, e.g. torch's, gets that one. world == 1 drops the communicator.
 * rank / world select the landmark slice as for spp_set_allreduce(); call before spp_ba_set_graph(). */
#define SPP_NCCL_UNIQUE_ID_BYTES 128
int spp_nccl_get_unique_id(void *p_unique_id);
int spp_set_nccl(spp_ctx_t ctx, const void *p_unique_id, int rank, int world);

/* Pure host helper (no context, no GPU): the landmark slices used by the multi-GPU path. p_track_length[p] = number
 * of observations of landmark p; p_bounds[world + 1] receives the slice boundaries (rank r owns landmarks
 * p_bounds[r] .. p_bounds[r + 1]), contiguous and balanced by the Schur-product work k (k + 1) / 2 + k. */
int spp_partition_landmarks(size_t n_points, const uint32_t *p_track_length, int world, uint64_t *p_bounds);

/* Pure host helper (no context, no GPU): the upper block list of the reduced camera system of a whole BA graph --
 * cameras i <= j share a block when some landmark is seen by both (the structure of schur_compl,
 * include/slam/LinearSolver_Schur.h:1757-1767): the C diagonal blocks first, then the off-diagonal blocks in row-major
 * order. This is the list under which several ranks sum their partial reduced camera systems. p_obs_camera /
 * p_obs_point: camera / point index (not vertex id) of every observation. Call with NULL arrays for the count;
 * *p_n_blocks is the capacity on input, the count on output. */
int spp_rcs_block_pattern(size_t n_cameras, size_t n_points, size_t n_observations, const uint32_t *p_obs_camera,
	const uint32_t *p_obs_point, uint64_t *p_n_blocks, uint32_t *p_block_row, uint32_t *p_block_col);

/* The landmark slice [*p_begin, *p_end) (indices into the point array given to spp_ba_set_graph) owned by this
 * context; the whole range when world == 1. spp_ba_get_states / spp_ba_set_states touch only this slice. */
int spp_ba_get_partition(spp_ctx_t ctx, uint64_t *p_begin, uint64_t *p_end);

/* ---- slot 3: bundle adjustment system resident on the device --------------------------------------- */

/* Replaces Add_CamVertex / Add_XYZVertex / Add_P2C3DEdge called in a loop (BAOptimizer.h:130-133;
 * src/ba_interface_example/BAOptimizer.cpp:214-230 -> CFlatSystem::r_Get_Vertex / r_Add_Edge) plus the one-time
 * structure build of lambda_utils::CLambdaOps2::Extend_Lambda (include/slam/NonlinearSolver_Lambda_Base.h:1634,
 * 1853-1931) and CLinearSolver_Schur::SymbolicDecomposition_Blocky (include/slam/LinearSolver_Schur.h:1566-1606).
 *   p_vertex_type[n_vertices]  0 = camera (6 DoF), 1 = point (3 DoF); vertex ids are shared, as in CFlatSystem
 *   p_cam_params[11 * C]       per camera in id order: t(3), axis-angle(3), fx, fy, cx, cy, d   (CVertexCam, BA_Types.h:54-75)
 *   p_points[3 * P]            per point in id order                                          (CVertexXYZ, BA_Types.h:355)
 *   p_obs_point / p_obs_camera vertex ids of each observation, in edge insertion order       (CEdgeP2C3D, BA_Types.h:403)
 *   p_z[2 * O], p_info[4 * O]  measurement and 2x2 information matrix per observation
 * The first vertex (id 0) receives the reference's automatic unary factor (identity information,
 * FlatSystem.h:337,432-473; Lambda_Base.h:1903-1923).
 * Restriction: a landmark observed twice by the SAME camera (a duplicate edge) is refused with SPP_ERR_INVALID; the
 * reference accepts such graphs and sums the two contributions (Lambda_Base.h:682-738). Pose graphs (spp_pose_set_graph)
 * do accept duplicate edges.
 * Host pointers are borrowed for the duration of the call, on every exit path. */
int spp_ba_set_graph(spp_ctx_t ctx, size_t n_vertices, const uint8_t *p_vertex_type,
	const double *p_cam_params, const double *p_points, size_t n_observations,
	const uint64_t *p_obs_point, const uint64_t *p_obs_camera, const double *p_z, const double *p_info);

/* Appends vertices and observations to the graph on the device: incremental bundle adjustment, where cameras and their
 * landmarks arrive in batches between two Optimize() calls (SURVEY 8(f) rank 2; the reference's system is append-only as
 * well, CFlatSystem::r_Get_Vertex / r_Add_Edge, FlatSystem.h:578-745, and its solver extends lambda for the new vertices
 * and edges only, NonlinearSolver_Lambda_Base.h:1665-1684). Arrays as for spp_ba_set_graph, holding the NEW vertices and
 * observations only; vertex ids continue the numbering (the first new vertex has id = vertices so far), observations may
 * reference old and new vertices. The states of the vertices already there stay as they are on the device (the result
 * of the last optimisation, or what spp_ba_set_states put there). The result is the same, bit for bit, as
 * spp_ba_set_graph of the concatenated arrays followed by spp_ba_set_states of the old vertices' current states -- but
 * only the new data cross the link; the structure is rebuilt on the device from the staged copies. Single-GPU contexts
 * whose graph was set by spp_ba_set_graph (device-side analysis); SPP_ERR_INVALID otherwise, the caller then falls
 * back to spp_ba_set_graph. */
int spp_ba_append_graph(spp_ctx_t ctx, size_t n_new_vertices, const uint8_t *p_vertex_type,
	const double *p_cam_params, const double *p_points, size_t n_new_observations,
	const uint64_t *p_obs_point, const uint64_t *p_obs_camera, const double *p_z, const double *p_info);

/* Overwrite / read the vertex states (CBAOptimizer::r_Vertex_State, BAOptimizer.cpp:196-204).
 * p_cam_states[6 * C] (t, axis-angle), p_points[3 * P]; either pointer may be NULL. */
int spp_ba_set_states(spp_ctx_t ctx, const double *p_cam_states, const double *p_points);
int spp_ba_get_states(spp_ctx_t ctx, double *p_cam_states, double *p_points);

/* Several ranks: the states of ALL vertices on every rank -- the cameras are replicated, the landmark slices are summed
 * into one array with one all-reduce on the device (a collective: every rank calls it). On one rank the same as
 * spp_ba_get_states. p_cam_states[6 * C], p_points[3 * P] of the whole graph; either may be NULL (on several ranks all
 * of them must then pass NULL for the points, or none). The reference has no counterpart (single process); the slot-3
 * adapter writes these states back into the caller's system, so that an application whose ranks all hold the whole
 * CFlatSystem sees the same optimised system everywhere. */
int spp_ba_gather_states(spp_ctx_t ctx, double *p_cam_states, double *p_points);

/* Restores the vertex states uploaded by the last spp_ba_set_graph() from a device-side snapshot (no host
 * traffic); lets a benchmark repeat Optimize() on the same resident problem. No reference counterpart. */
int spp_ba_restore_initial(spp_ctx_t ctx);

int spp_ba_set_jacobian_mode(spp_ctx_t ctx, int mode); /* SPP_JAC_* ; default SPP_JAC_FD_REFERENCE */

/* Robust loss of the BA observations (g2o-style IRLS; the reference's kernels: RobustUtils.h:368-586). With s2 = r^T
 * Omega r the squared Mahalanobis error of an observation (r = z - h; s is in pixels when Omega = I) and k the scale:
 *   SPP_LOSS_NONE    rho = s2                                      w = 1
 *   SPP_LOSS_HUBER   rho = s2 if s2 <= k^2, else 2 k sqrt(s2) - k^2 w = 1 if s2 <= k^2, else k / sqrt(s2)
 *   SPP_LOSS_CAUCHY  rho = k^2 log1p(s2 / k^2)                      w = 1 / (1 + s2 / k^2)
 * The linearisation replaces Omega by w Omega before any other use, so U, g_c, W, V, g_p and the initial damping are
 * those of the weighted problem -- and so are spp_ba_get_lambda, spp_ba_get_blocks, spp_ba_solve_step and every
 * marginal / covariance entry point (the convention of Ceres and g2o for the covariance of a robust problem). Both
 * vertices of an observation see the same weight: this is NOT the reference's robust binary edge, which weights vertex
 * 0's gradient by w^2 and vertex 1's by w (BaseTypes_Binary.h:820-843). spp_ba_chi2, chi2_initial / chi2_final /
 * trace_chi2 of spp_report_t and the LM acceptance test then hold sum rho; the predicted decrease stays
 * dx^T (alpha dx + eta) (the IRLS model). An observation with w = 1 contributes exactly what it does without a loss. */
#define SPP_LOSS_NONE 0   /* default */
#define SPP_LOSS_HUBER 1
#define SPP_LOSS_CAUCHY 2

/* Context state, like the Jacobian mode: kept across spp_ba_set_graph, spp_ba_append_graph and spp_ba_restore_initial;
 * marks the linearisation stale. scale (k, in units of s) must be finite and > 0 for HUBER and CAUCHY and is ignored for
 * NONE. An unknown kind or a bad scale returns SPP_ERR_INVALID and keeps the previous setting. No reference counterpart
 * for BA (the reference sets a robust kernel per edge type at compile time). */
int spp_ba_set_robust_loss(spp_ctx_t ctx, int kind, double scale);

/* s2 (p_sq_error[O]) and the weight w = rho'(s2) (p_weight[O]) of every observation at the current states, in EDGE
 * INSERTION order (as W of spp_ba_get_blocks). The residual is computed as the linearisation in the current Jacobian mode
 * computes it, so w is bit for bit the weight a linearisation at these states uses. Either pointer may be NULL. Lets a
 * caller find and drop outliers between two optimisations. Refused on a landmark-partitioned (multi-GPU) context. No
 * reference counterpart. */
int spp_ba_get_observation_errors(spp_ctx_t ctx, double *p_sq_error, double *p_weight);

/* Replaces CLambdaOps2::Refresh_Lambda + Collect_RightHandSide_Vector (Lambda_Base.h:1659-1706):
 * per-edge Jacobians (CEdgeP2C3D::Calculate_Jacobians_Expectation_Error, BA_Types.h:494-505), Hessian blocks
 * (CBaseEdgeImpl::Calculate_Hessians_v2, BaseTypes_Binary.h:759-848) and their reduction into lambda / eta. */
int spp_ba_linearise(spp_ctx_t ctx);

/* Export of the linearised system in the reference's own layout (upper block-triangular, vertex id order,
 * column-major blocks; CUberBlockMatrix accessors BlockMatrix.h:343-430,470-485), WITHOUT damping.
 * Call first with p_values == NULL to obtain the sizes. Used by the parity tests (SURVEY 8(c) P2). */
int spp_ba_get_lambda(spp_ctx_t ctx, uint64_t *p_n_block_cols, uint64_t *p_n_blocks, uint64_t *p_n_values,
	uint64_t *p_col_dims, uint64_t *p_col_ptr, uint64_t *p_row_idx, double *p_values, double *p_eta);

/* The same linearised system as raw block arrays, for full-size checks where the column-ordered export above is
 * unwieldy: p_U[36 * C] / p_V[9 * P] diagonal blocks in camera / point id order, p_W[18 * O] the camera x point
 * block J_c^T Sigma^-1 J_p (6 x 3, column-major) of every observation in EDGE INSERTION order, p_eta_c[6 * C],
 * p_eta_p[3 * P]. Undamped; any pointer may be NULL. (CUberBlockMatrix::t_Block_AtColumn, BlockMatrix.h:470-485) */
int spp_ba_get_blocks(spp_ctx_t ctx, double *p_U, double *p_V, double *p_W, double *p_eta_c, double *p_eta_p);

/* Replaces CNonlinearSolver_Lambda_LM::f_Chi_Squared_Error_Denorm (NonlinearSolver_Base.h:278-297 ->
 * CEdgeP2C3D::f_Chi_Squared_Error, BA_Types.h:511-531). Under a robust loss (spp_ba_set_robust_loss): sum rho(s2). */
int spp_ba_chi2(spp_ctx_t ctx, double *p_chi2);

/* One damped Newton step on the current linearisation: solves (lambda + alpha I) dx = eta through the landmark
 * Schur complement and returns dx in vertex id order (6 per camera, 3 per point). Does not move the vertices.
 * = Apply_Damping + LinearSolve of LM.h:942-967,1512-1568. */
int spp_ba_solve_step(spp_ctx_t ctx, double alpha, double *p_dx);

/* Replaces CNonlinearSolver_Lambda_LM::Optimize(max_iter, min_dx_norm) (LM.h:796-1116), control flow included
 * (initial damping, rho test, rollback, <= 10 extra iterations on rejected steps). */
int spp_ba_optimize(spp_ctx_t ctx, size_t n_max_iterations, double f_min_dx_norm, spp_report_t *p_report);

/* Block diagonal of the covariance (lambda + alpha I)^-1 at the current vertex states, recovered from the
 * Schur-complemented system. Replaces the marginals step at the end of CNonlinearSolver_Lambda_LM::Optimize()
 * (NonlinearSolver_Lambda_LM.h:1118-1350, policy mpart_Diagonal) -> CSchurComplement_Marginals::Schur_Marginals
 * (include/slam/BAMarginals.h:579-760); the reference uses alpha = 0.
 *   p_cam_cov[36 * n_cameras]  6x6 blocks, cameras in vertex id order (symmetric: row- or column-major)
 *   p_pt_cov[9 * n_points]     3x3 blocks, points in vertex id order
 * Either output may be null. Needs the dense reduced camera system (6 * n_cameras <= 16384 or
 * spp_schur_set_rcs_solver(SPP_RCS_DENSE)) and 16 * ld^2 bytes of device memory, ld = 6 * n_cameras rounded up to 128.
 * Returns SPP_OK / SPP_NOT_POSDEF. Note: a monocular BA system with one fixed camera has an unobservable scale; its
 * variance (1 / the smallest eigenvalue of lambda, finite-difference noise) dominates every block at alpha = 0. */
int spp_ba_marginals(spp_ctx_t ctx, double alpha, double *p_cam_cov, double *p_pt_cov);

/* ---- slot 1: linear solver on a lambda given by the caller ------------------------------------------ */

/* Replaces CLinearSolver_Schur::SymbolicDecomposition_Blocky(lambda) (LinearSolver_Schur.h:1566-1606): takes the
 * block structure of an upper block-triangular lambda (block columns with dims in {3, 6}; guided ordering =
 * 6-wide vertices first, then 3-wide, original order kept within each group, Schur.cpp:771-838).
 *   p_col_dims[n]      width of each block column
 *   p_col_ptr[n + 1]   block column pointers
 *   p_row_idx[nnzb]    block row of every block (ascending within a column; the diagonal block is the last)
 * Optional outputs: p_order[n] receives the ordering (new position -> original block column), *p_cut = #6-wide. */
int spp_schur_symbolic(spp_ctx_t ctx, size_t n_block_cols, const uint64_t *p_col_dims, const uint64_t *p_col_ptr,
	const uint64_t *p_row_idx, uint64_t *p_order, uint64_t *p_cut);

/* Replaces CLinearSolver_Schur::Solve_PosDef_Blocky(lambda, eta) (LinearSolver_Schur.h:1623-1935): p_values are
 * the blocks of lambda in the order of the structure given to spp_schur_symbolic (column-major blocks);
 * p_eta_dx[n_scalars] is the right-hand side on input and the solution on output.
 * Returns SPP_NOT_POSDEF where the reference returns false. */
int spp_schur_solve(spp_ctx_t ctx, const double *p_values, double *p_eta_dx);

/* Schur_Marginals (include/slam/BAMarginals.h:579-760) on the lambda of the last spp_schur_solve: block diagonal of
 * (lambda + alpha I)^-1, 6-wide block columns in p_cam_cov[36 * cut], 3-wide ones in p_pt_cov[9 * (n - cut)], each
 * group in the order of the block columns. Same requirements and return values as spp_ba_marginals. */
int spp_schur_marginals(spp_ctx_t ctx, double alpha, double *p_cam_cov, double *p_pt_cov);

/* Block diagonal of (lambda + alpha I)^-1 like spp_ba_marginals, recovered from the block-sparse (supernodal)
 * factorisation of the reduced camera system by selected inversion: no dense S^-1, any number of cameras. Uses the
 * supernodal path whatever spp_schur_set_rcs_solver says. Same output layout and return values as spp_ba_marginals. */
int spp_ba_marginals_sparse(spp_ctx_t ctx, double alpha, double *p_cam_cov, double *p_pt_cov);
/* the same on the lambda of the last spp_schur_solve (slot 1), output as spp_schur_marginals */
int spp_schur_marginals_sparse(spp_ctx_t ctx, double alpha, double *p_cam_cov, double *p_pt_cov);

/* Selected blocks of (lambda + alpha I)^-1 in one factorisation + inversion, on the dense or supernodal reduced camera
 * system as spp_schur_set_rcs_solver selects. Cameras by index (id order among cameras), observations by edge insertion
 * index. p_pair_cov[36 n_pairs]: Cov(cam_a[k], cam_b[k]), 6x6 column-major; the pair must share a landmark or be equal.
 * p_obs_cov[18 n_obs]: Cov(camera, point) of observation p_obs[k], 6x3 column-major (the layout of W in
 * spp_ba_get_blocks). p_cam_cov / p_pt_cov: the block diagonal, bit-identical to spp_ba_marginals(_sparse) on that path.
 * Any output may be NULL (with its count 0). SPP_OK / SPP_NOT_POSDEF / SPP_ERR_INVALID.
 * Extends the marginals of CSchurComplement_Marginals::Schur_Marginals (include/slam/BAMarginals.h:579-760), which
 * computes the block diagonal only. On the supernodal path the state rules of spp_ba_marginals_sparse apply. */
int spp_ba_covariance_blocks(spp_ctx_t ctx, double alpha,
	size_t n_pairs, const uint64_t *p_cam_a, const uint64_t *p_cam_b, double *p_pair_cov,
	size_t n_obs, const uint64_t *p_obs, double *p_obs_cov,
	double *p_cam_cov, double *p_pt_cov);

/* Slot 1: (lambda + alpha I)^-1 restricted to the block pattern of the lambda of the last spp_schur_solve, written in the
 * layout of that call's p_values (n_values doubles): diagonal blocks and every camera-landmark block. Extends
 * Schur_Marginals (include/slam/BAMarginals.h:579-760), which computes the block diagonal only. Path as
 * spp_ba_covariance_blocks. SPP_OK / SPP_NOT_POSDEF / SPP_ERR_INVALID. */
int spp_schur_covariance_pattern(spp_ctx_t ctx, double alpha, double *p_cov_values);

/* Joint marginal covariance of sets of vertices: for set k (vertex ids p_vertices[p_set_ptr[k] .. p_set_ptr[k+1]]),
 * the D_k x D_k matrix Sigma_KK of (lambda + alpha I)^-1, D_k = sum of the vertices' dims (6 camera, 3 point),
 * column-major, vertices in the order given; sets one after another in p_cov (offset sum_{j<k} D_j^2).
 * Any vertex pair may appear, on the block pattern of the reduced camera system or off it (cameras that share no
 * landmark, landmark-landmark blocks). Forward solves with the factor of S: Sigma_uv = [u = v landmark] C_v^-1 +
 * F_u^T F_v, F_v = R^-T P b_v; the blocks of the reference's computeMarginals(blockIndices) style queries, which
 * Schur_Marginals (include/slam/BAMarginals.h:579-760) does not provide. Path as spp_ba_covariance_blocks; on the
 * supernodal path the state rules of spp_ba_marginals_sparse apply. A set's result does not depend on the other sets of
 * the call. SPP_OK / SPP_NOT_POSDEF / SPP_ERR_INVALID (vertex id out of range, empty set, set wider than 16 384
 * columns, several ranks). */
int spp_ba_joint_marginals(spp_ctx_t ctx, double alpha, size_t n_sets, const uint64_t *p_set_ptr,
	const uint64_t *p_vertices, double *p_cov);
/* the same on the lambda of the last spp_schur_solve; sets of block columns in the numbering given to spp_schur_symbolic */
int spp_schur_joint_marginals(spp_ctx_t ctx, double alpha, size_t n_sets, const uint64_t *p_set_ptr,
	const uint64_t *p_block_cols, double *p_cov);

/* Stage outputs of the last Schur solve, for the parity tests (SURVEY 8(c) P1): the reduced camera system as a
 * dense column-major (6C x 6C) matrix (upper triangle valid), its right-hand side, and the pattern of non-zero
 * 6x6 blocks of the upper triangle (row-major bitmap, C*C bytes). Any pointer may be NULL. */
int spp_schur_get_reduced_system(spp_ctx_t ctx, uint64_t *p_n, double *p_S, double *p_rhs, uint8_t *p_block_pattern);

/* ---- solver of the reduced camera system (RCS) ------------------------------------------------------------ */

/* Replaces the reference's choice between CLinearSolver_DenseEigen and, when the dense matrix cannot be allocated
 * (std::bad_alloc), CLinearSolver_UberBlock on the block-sparse Schur complement (include/slam/LinearSolver_Schur.h:
 * 1427-1435, 1836-1847). SPP_RCS_AUTO: dense up to 16 384 unknowns, supernodal block-sparse above. Applies to the
 * spp_ba_* and spp_schur_* entry points of this context. */
#define SPP_RCS_AUTO 0
#define SPP_RCS_DENSE 1
#define SPP_RCS_SPARSE 2
int spp_schur_set_rcs_solver(spp_ctx_t ctx, int mode);

/* The fill-reducing ordering of the cameras used by the block-sparse RCS solver: p_order[new position] = camera index
 * (position among the 6-wide vertices in id order). The reference-side adapter passes the reference's own AMD
 * permutation (CMatrixOrdering::p_BlockOrdering on the Schur complement, src/slam/OrderingMagic.cpp:701-1033, called
 * from LinearSolver_UberBlock.h:272-296) so that the elimination order is the reference's bit for bit; with NULL (the
 * default) the library computes an approximate-minimum-degree ordering itself (spp_block_ordering). */
int spp_schur_set_rcs_ordering(spp_ctx_t ctx, size_t n_cameras, const uint64_t *p_order);

/* After a solve on the block-sparse path: the ordering in use (p_order[C], may be NULL) and p_stats[8] = cameras,
 * non-zero 6x6 blocks of the upper RCS, supernodes, blocks of the exact factor, blocks of the factor as stored
 * (amalgamation zeros included), flops of one numeric factorisation, bytes of factor storage, supernode updates. */
int spp_schur_get_rcs_info(spp_ctx_t ctx, uint64_t *p_order, double *p_stats);

/* Several ranks: who factors which supernode of the block-sparse reduced camera system. p_owner[supernodes] (the count
 * is p_stats[2] of spp_schur_get_rcs_info): the rank that owns the supernode's subtree, or -1 for the supernodes at the
 * top of the elimination tree that every rank factors after the contributions to their panels have been summed
 * (all -1 on one rank, or when sharing the work out would not pay). The reference has no counterpart. */
int spp_schur_get_rcs_owners(spp_ctx_t ctx, int32_t *p_owner);

/* After a successful solve on the block-sparse path: || S dx_cam - b || / || b || of the reduced camera system, evaluated
 * on the device from the block list of S (which survives the factorisation) -- the size-independent check of stage 3
 * at sizes where no dense copy of S can be taken (BAL-13682 shape). The reference has no counterpart. */
int spp_schur_get_rcs_residual(spp_ctx_t ctx, double *p_relative_residual);

/* Pure host helpers (no context, no GPU). spp_block_ordering: the fill-reducing ordering (approximate minimum degree on
 * the block graph of A + A^T) of a block structure in block CSC (upper, lower or both triangles; diagonal present or
 * not) -- what CMatrixOrdering::p_BlockOrdering / SuiteSparse amd_l2 does in the reference (src/slam/OrderingMagic.cpp:
 * 701-1033), and the same permutation entry for entry (csrc/amd_exact.cpp). spp_block_symbolic_stats: symbolic Cholesky under an
 * ordering (NULL = natural): p_col_count[n] blocks per column of the factor, p_parent[n] elimination tree
 * (UINT64_MAX = root), p_stats[3] = blocks of the factor, sum of count^2, maximal supernodes. Any output may be NULL.
 * (CUberBlockMatrix::Build_EliminationTree, src/slam/BlockMatrix.cpp:9403.) */
int spp_block_ordering(size_t n_block_cols, const uint64_t *p_col_ptr, const uint64_t *p_row_idx, uint64_t *p_order);
int spp_block_symbolic_stats(size_t n_block_cols, const uint64_t *p_col_ptr, const uint64_t *p_row_idx,
	const uint64_t *p_order, uint64_t *p_col_count, uint64_t *p_parent, double *p_stats);
/* Several ranks: the plan that shares the block-sparse factorisation of a reduced camera system out over n_world ranks
 * (pure host helper; the solver computes the same plan internally, spp_schur_get_rcs_owners reports it). Under the
 * ordering p_order (NULL = natural) and the solver's supernode amalgamation: p_owner[n_block_cols] = for every PERMUTED
 * block column the rank that factors its supernode, -1 = every rank (the top of the elimination tree); p_stats[3] =
 * predicted time as a fraction of the replicated factorisation (1 = no plan saves f_min_saving), supernodes, shared
 * supernodes. The reference has no counterpart (single process). */
int spp_block_subtree_owners(size_t n_block_cols, const uint64_t *p_col_ptr, const uint64_t *p_row_idx,
	const uint64_t *p_order, int n_world, double f_min_saving, int32_t *p_owner, double *p_stats);

/* ---- dense FP64 Cholesky (the reduced camera system solver) ----------------------------------------- */

/* Replaces CLinearSolver_DenseEigen::Solve_PosDef (src/slam/LinearSolver_Schur.cpp:2314-2333): Eigen::LLT<MatrixXd,
 * Upper> of a dense column-major n x n matrix of which only the upper triangle is read, then two triangular
 * solves; p_rhs_x is the right-hand side on input, the solution on output. Host pointers. */
int spp_dense_posdef_solve(spp_ctx_t ctx, size_t n, const double *p_A, double *p_rhs_x);
/* The dense front primitive underneath both Cholesky paths (the dense reduced camera system is one front with its
 * right-hand side, a supernode of the block-sparse factorisation a front with its row structure): p_panel is column-major
 * with n_rows rows (a multiple of 128) and n_cols >= n_rows columns (a multiple of 128); on return its leading n_rows x
 * n_rows upper triangle holds R11 (R11^T R11 = A11; the strictly lower triangle is unspecified) and the remaining columns
 * R11^-T A12. Returns SPP_NOT_POSDEF at a non-positive pivot. Exposed for tests and for callers that bring their own
 * frontal scheme; the reference has no counterpart (its dense step is Eigen's LLT, src/slam/LinearSolver_Schur.cpp:
 * 2314-2333, its sparse one the block-column CholeskyOf_FBS, include/slam/BlockMatrixFBS.inl:2341-2513). */
int spp_dense_panel_factor(spp_ctx_t ctx, size_t n_rows, size_t n_cols, double *p_panel);

/* ---- block-sparse FP64 Cholesky (pose graphs; sparse reduced camera systems) ------------------------------ */

/* Replaces CLinearSolver_UberBlock::SymbolicDecomposition_Blocky (include/slam/LinearSolver_UberBlock.h:272-296):
 * takes the block structure of an upper block-triangular matrix whose block columns are all block_size wide (2, 3
 * or 6; the reference's fbs_ut lists) and prepares the factorisation: ordering, elimination tree, factor pattern.
 *   p_col_ptr[n + 1], p_row_idx[nnzb]   block CSC, rows ascending, diagonal block present
 *   p_order_in[n] or NULL   the fill-reducing block ordering to use (new position -> original block column). The
 *                           reference-side adapter passes the reference's own AMD ordering
 *                           (CMatrixOrdering::p_BlockOrdering, src/slam/OrderingMagic.cpp:701-1033) so that the
 *                           elimination order is the reference's, bit for bit; with NULL the approximate-minimum-degree ordering of spp_block_ordering is
 *                           computed by the library.
 *   p_order_out[n] or NULL  receives the ordering in use. */
int spp_chol_symbolic(spp_ctx_t ctx, size_t n_block_cols, size_t block_size, const uint64_t *p_col_ptr,
	const uint64_t *p_row_idx, const uint64_t *p_order_in, uint64_t *p_order_out);

/* Replaces CLinearSolver_UberBlock::Solve_PosDef_Blocky (LinearSolver_UberBlock.h:312-426): permutation, block
 * Cholesky (CUberBlockMatrix::CholeskyOf_FBS, include/slam/BlockMatrixFBS.inl:2341-2513) and the two triangular
 * solves (:2136-2275). p_values: the blocks in the order of the structure (column-major blocks; of the diagonal
 * blocks the full symmetric block is read); p_eta_dx: right-hand side in, solution out.
 * Returns SPP_NOT_POSDEF where the reference returns false.
 * The slot and the pose-graph solves (spp_pose_solve_step, spp_pose_optimize) share one analysis per context. A pose
 * solve replaces the slot's analysis with its own, and the slot does not keep its structure: spp_chol_solve after a pose
 * solve returns SPP_ERR_INVALID until spp_chol_symbolic is called again. A pose solve after spp_chol_symbolic repeats
 * the pose graph's analysis by itself. */
int spp_chol_solve(spp_ctx_t ctx, const double *p_values, double *p_eta_dx);

/* The factor of the last spp_chol_solve / spp_pose_* solve in the reference's form, the upper factor R with
 * R^T R = P lambda P^T (block CSC in the permuted order, rows ascending, diagonal last; column-major blocks), for the
 * parity tests: with the reference's ordering the block pattern of R must be the reference's, bit for bit.
 * After a pose solve this is the pose graph's factor: n_poses block columns of dim x dim blocks.
 * Call with NULL arrays to obtain the block count. */
int spp_chol_get_factor(spp_ctx_t ctx, uint64_t *p_n_blocks, uint64_t *p_col_ptr, uint64_t *p_row_idx, double *p_values);

/* ---- pose graphs resident on the device (SE(2) and SE(3); Gauss-Newton) ---------------------------------------- */

/* Replaces r_Get_Vertex<CVertexPose2D> / r_Add_Edge(CEdgePose2D(...)) called in a loop (src/slam_simple_example/
 * Main.cpp; include/slam/SE2_Types.h:178-260) plus the structure build of CLambdaOps2::Extend_Lambda
 * (include/slam/NonlinearSolver_Lambda_Base.h:1634, 1853-1931).
 *   dim            3 = SE(2) poses [x, y, theta] (CVertexPose2D / CEdgePose2D, analytic Jacobians);
 *                  6 = SE(3) poses [t, axis-angle] (CVertexPose3D / CEdgePose3D, include/slam/SE3_Types.h:45-48, 128-129,
 *                  265-288: forward-difference Jacobians with delta = 1e-9 in the reference's operation order, Huber
 *                  weight on |r| / 0.3 applied exactly as the reference's robust Calculate_Hessians_v2 does)
 *   p_states[dim * n_poses], p_from / p_to[n_edges] vertex ids (any order; duplicates allowed)
 *   p_z[dim * n_edges] relative pose measurements, p_info[dim * dim * n_edges] information matrices (symmetric)
 * Vertex 0 receives the reference's automatic unary factor (identity). */
int spp_pose_set_graph(spp_ctx_t ctx, int dim, size_t n_poses, const double *p_states, size_t n_edges,
	const uint64_t *p_from, const uint64_t *p_to, const double *p_z, const double *p_info);
/* optional: the block ordering for the factorisation (see spp_chol_symbolic); NULL = computed by the library */
int spp_pose_set_ordering(spp_ctx_t ctx, const uint64_t *p_order);
int spp_pose_set_states(spp_ctx_t ctx, const double *p_states);
int spp_pose_get_states(spp_ctx_t ctx, double *p_states);
int spp_pose_restore_initial(spp_ctx_t ctx);
/* CLambdaOps2::Refresh_Lambda + Collect_RightHandSide_Vector for CEdgePose2D (SE2_Types.h:308-319; analytic
 * Jacobians include/slam/2DSolverBase.h:373-430; BaseTypes_Binary.h:759-848) */
int spp_pose_linearise(spp_ctx_t ctx);
/* lambda / eta of the last linearisation in the reference's layout (upper block CSC in vertex order, rows ascending,
 * diagonal last, column-major blocks). Call with NULL arrays for the sizes. */
int spp_pose_get_lambda(spp_ctx_t ctx, uint64_t *p_n_block_cols, uint64_t *p_n_blocks, uint64_t *p_col_ptr,
	uint64_t *p_row_idx, double *p_values, double *p_eta);
/* f_Chi_Squared_Error_Denorm (NonlinearSolver_Base.h:278-297 -> CEdgePose2D::f_Chi_Squared_Error, SE2_Types.h:325-335) */
int spp_pose_chi2(spp_ctx_t ctx, double *p_chi2);
/* one Gauss-Newton increment on the current linearisation: lambda dx = eta; does not move the vertices */
int spp_pose_solve_step(spp_ctx_t ctx, double *p_dx);
/* Block diagonal of lambda^-1 at the current states: replaces the marginals step at the end of
 * CNonlinearSolver_Lambda::Optimize() (NonlinearSolver_Lambda.h:669-767 -> CMarginals::
 * Calculate_DenseMarginals_Recurrent_FBS, policy mpart_Diagonal). p_cov[n_poses * dim * dim], poses in id order. Through a
 * dense inverse on the FP64 tensor pipe: at most 16384 unknowns. Returns SPP_OK / SPP_NOT_POSDEF. */
int spp_pose_marginals(spp_ctx_t ctx, double *p_cov);
/* Replaces CNonlinearSolver_Lambda::Optimize(max_iter, min_dx_norm) (include/slam/NonlinearSolver_Lambda.h:476-667) */
int spp_pose_optimize(spp_ctx_t ctx, size_t n_max_iterations, double f_min_dx_norm, spp_report_t *p_report);

#ifdef __cplusplus
}
#endif

#endif /* SPP_B200_H */
