// spp_api.cu -- the C ABI of libspp_b200.so (include/spp_b200.h) and the host control flow of the
// nonlinear solvers (LM loop), mirroring CNonlinearSolver_Lambda_LM::Optimize
// (include/slam/NonlinearSolver_Lambda_LM.h:796-1116) with the system resident on the device.

#include "spp_ctx.h"
#include <nccl.h>  // types only: the library is opened with dlopen (see nccl_api())
#include <dlfcn.h>
#include <string.h>
#include <math.h>
#include <algorithm>
#include <stdlib.h>

namespace spp {

// kernels / stages implemented in the other translation units
void build_schur_structure(spp_ctx *ctx, size_t C, size_t P, const std::vector<uint32_t> &h_cam,
	const std::vector<uint32_t> &h_pt, std::vector<uint32_t> &obs_orig, std::vector<uint32_t> &t_cam,
	std::vector<uint32_t> &t_pt);
bool schur_structure_device_supported(size_t C);
void ba_upload_and_analyse_device(spp_ctx *ctx, size_t C, size_t P, size_t O, const uint64_t *p_obs_point,
	const uint64_t *p_obs_camera, const double *p_z, const double *p_info);
void ba_append_and_analyse_device(spp_ctx *ctx, size_t C, size_t P, size_t O_old, size_t O_new, const uint64_t *p_obs_point,
	const uint64_t *p_obs_camera, const double *p_z, const double *p_info);
void ba_upload_and_analyse_device_sliced(spp_ctx *ctx, size_t C, size_t P, size_t O, const uint64_t *p_obs_point,
	const uint64_t *p_obs_camera, const double *p_z, const double *p_info);
void ba_fetch_host_maps(spp_ctx *ctx);
void schur_fetch_host_pattern(spp_ctx *ctx);
void build_global_rcs_pattern(size_t C, size_t P, const std::vector<uint32_t> &h_cam, const std::vector<uint32_t> &h_pt,
	std::vector<uint32_t> &g_row, std::vector<uint32_t> &g_col);
void map_blocks_to_global(size_t C, const std::vector<uint32_t> &l_row, const std::vector<uint32_t> &l_col,
	const std::vector<uint32_t> &g_row, const std::vector<uint32_t> &g_col, std::vector<uint32_t> &slot);
void ba_linearise(spp_ctx *ctx, bool b_want_maxdiag);
void ba_chi2_device(spp_ctx *ctx, double *d_out);
void ba_obs_errors_device(spp_ctx *ctx, double *d_sq_err, double *d_weight);
void ba_step_dots_device(spp_ctx *ctx, double alpha, double *d_out);
void ba_apply_update(spp_ctx *ctx);
void schur_form_reduced_system(spp_ctx *ctx, double alpha, double alpha_diag, bool sparse_rcs);
void snode_symbolic(spp_ctx *ctx, size_t n, const std::vector<uint32_t> &blk_row, const std::vector<uint32_t> &blk_col);
int snode_factor_solve(spp_ctx *ctx, const double *d_Sblk, const double *d_b, double *d_dx);
void schur_backsubstitute(spp_ctx *ctx);
size_t dense_chol_ld(size_t n);
size_t dense_chol_storage(size_t n);
int dense_chol_solve_device(spp_ctx *ctx, double *A, size_t n, double *d_rhs_x);
void dense_chol_factor_panel(spp_ctx *ctx, double *A, size_t ld, size_t n_cols, double *Rinv, int *info, bool identity_tail);
void dense_chol_factor_dataflow(spp_ctx *ctx, double *A, size_t ld, size_t n_cols, double *Rinv, int *info);
bool dense_chol_dataflow_enabled();
int schur_marginals_current(spp_ctx *ctx, double alpha, double *d_cam_cov, double *d_pt_cov);
int schur_marginals_sparse_current(spp_ctx *ctx, double alpha, double *d_cam_cov, double *d_pt_cov, float *ms_phases);
int schur_covariance_blocks_current(spp_ctx *ctx, double alpha, bool sparse, double *d_cam_cov, double *d_pt_cov, size_t n_pairs,
	const uint32_t *d_cam_a, const uint32_t *d_cam_b, double *d_pair_cov, size_t n_obs, const uint32_t *d_obs, double *d_obs_cov,
	float *ms_phases);
int slot_covariance_pattern(spp_ctx *ctx, double alpha, bool sparse, double *d_vals, float *ms_phases);
int joint_marginals_to_host(spp_ctx *ctx, double alpha, bool sparse, const std::vector<uint64_t> &set_ptr,
	const std::vector<uint32_t> &verts, double *p_cov, bool timing);
int pose_marginals(spp_ctx *ctx, double *d_cov);
void slot_symbolic(spp_ctx *ctx, size_t n, const uint64_t *col_dims, const uint64_t *col_ptr, const uint64_t *row_idx,
	uint64_t *p_order, uint64_t *p_cut);
int slot_solve(spp_ctx *ctx, const double *p_values, double *p_eta_dx);

void sparse_chol_symbolic(spp_ctx *ctx, int owner, size_t n, size_t B, const uint64_t *col_ptr, const uint64_t *row_idx,
	const uint64_t *p_order_in);
int sparse_chol_solve_device(spp_ctx *ctx, const double *d_A, const double *d_rhs, double *d_x);
void pose_set_graph(spp_ctx *ctx, int dim, size_t N, const double *p_states, size_t E, const uint64_t *p_from,
	const uint64_t *p_to, const double *p_z, const double *p_info);
void pose_linearise(spp_ctx *ctx);
double pose_chi2(spp_ctx *ctx);
int pose_solve(spp_ctx *ctx);
int pose_optimize(spp_ctx *ctx, size_t n_max_iteration_num, double f_min_dx_norm, spp_report_t *rep);

static thread_local std::string g_create_error;

struct comm_error : std::runtime_error {
	explicit comm_error(const std::string &t) : std::runtime_error(t) {}
};

// ---- NCCL, bound at run time ----------------------------------------------------------------------------
// The library calls NCCL itself (ncclAllReduce on the context's stream: no host round trip, no Python in the data
// plane). libnccl.so.2 is opened with dlopen when spp_set_nccl / spp_nccl_get_unique_id is first called: a process that
// already holds an NCCL (torch's bundled one) gets that very library, a plain C++ host the system's. Single-GPU users
// never load it.
struct NcclApi {
	void *handle;
	ncclResult_t (*GetUniqueId)(ncclUniqueId*);
	ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int);
	ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t);
	ncclResult_t (*CommAbort)(ncclComm_t); // teardown without a rendezvous: the peers may already be gone
	const char *(*GetErrorString)(ncclResult_t);
	NcclApi() : handle(0), GetUniqueId(0), CommInitRank(0), AllReduce(0), CommAbort(0), GetErrorString(0) {}
};

static NcclApi &nccl_api()
{
	static NcclApi api;
	if(!api.handle) {
		void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
		if(!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
		if(!h)
			throw comm_error(std::string("cannot load libnccl.so.2: ") + dlerror());
		api.GetUniqueId = (ncclResult_t (*)(ncclUniqueId*))dlsym(h, "ncclGetUniqueId");
		api.CommInitRank = (ncclResult_t (*)(ncclComm_t*, int, ncclUniqueId, int))dlsym(h, "ncclCommInitRank");
		api.AllReduce = (ncclResult_t (*)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t))dlsym(h, "ncclAllReduce");
		api.CommAbort = (ncclResult_t (*)(ncclComm_t))dlsym(h, "ncclCommAbort");
		api.GetErrorString = (const char *(*)(ncclResult_t))dlsym(h, "ncclGetErrorString");
		if(!api.GetUniqueId || !api.CommInitRank || !api.AllReduce || !api.CommAbort || !api.GetErrorString)
			throw comm_error("libnccl.so.2 lacks one of ncclGetUniqueId / ncclCommInitRank / ncclAllReduce / ncclCommAbort");
		api.handle = h;
	}
	return api;
}

#define SPP_NCCL(call) do { ncclResult_t r_ = (call); if(r_ != ncclSuccess) \
	throw comm_error(std::string(#call ": ") + nccl_api().GetErrorString(r_)); } while(0)

// sums n doubles at d_ptr over the ranks (no-op on one rank): ncclAllReduce on the context's stream when the context owns
// a communicator (spp_set_nccl), else through the hook installed by spp_set_allreduce (host-side tests over gloo; the
// hook orders itself on the context's stream).
void allreduce_device(spp_ctx *ctx, double *d_ptr, size_t n)
{
	if(ctx->world <= 1 || !n)
		return;
	if(ctx->nccl_comm) {
		SPP_NCCL(nccl_api().AllReduce(d_ptr, d_ptr, n, ncclDouble, ncclSum, (ncclComm_t)ctx->nccl_comm, ctx->stream));
		return;
	}
	if(!ctx->allreduce)
		throw invalid_error("world > 1 but neither a communicator (spp_set_nccl) nor an all-reduce hook (spp_set_allreduce)");
	if(ctx->allreduce(ctx->allreduce_user, d_ptr, n) != 0)
		throw comm_error("the all-reduce hook failed");
}

struct EventTimer {
	spp_ctx *ctx;
	cudaEvent_t a, b;
	EventTimer(spp_ctx *c) : ctx(c), a(c->ev[0]), b(c->ev[1]) {}
	void start() { cudaEventRecord(a, ctx->stream); }
	double stop_ms()
	{
		cudaEventRecord(b, ctx->stream);
		cudaEventSynchronize(b);
		float ms = 0;
		cudaEventElapsedTime(&ms, a, b);
		return ms;
	}
};

// r += S x for the symmetric matrix given by its upper block list (diagnostics: atomics are fine here)
__global__ void k_blocks_symv(size_t n_vals, const double *__restrict__ Sblk, const uint32_t *__restrict__ blk_row,
	const uint32_t *__restrict__ blk_col, const double *__restrict__ x, double *__restrict__ r)
{
	const size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(e >= n_vals) return;
	const size_t b = e / 36;
	const unsigned q = (unsigned)(e - b * 36), c = q / 6, rr = q - c * 6;
	const size_t i = (size_t)blk_row[b] * 6 + rr, j = (size_t)blk_col[b] * 6 + c;
	const double v = Sblk[e];
	if(blk_row[b] != blk_col[b]) {
		atomicAdd(r + i, v * x[j]);
		atomicAdd(r + j, v * x[i]);
	} else if(rr <= c) { // the diagonal blocks hold both triangles: take the upper one
		atomicAdd(r + i, v * x[j]);
		if(rr != c) atomicAdd(r + j, v * x[i]);
	}
}

__global__ void k_residual_norms(size_t n, const double *__restrict__ r, const double *__restrict__ b, double *__restrict__ out)
{
	__shared__ double s0[256], s1[256];
	double a0 = 0, a1 = 0;
	for(size_t i = threadIdx.x; i < n; i += 256) {
		const double d = r[i] - b[i];
		a0 += d * d;
		a1 += b[i] * b[i];
	}
	s0[threadIdx.x] = a0; s1[threadIdx.x] = a1;
	__syncthreads();
	for(int w = 128; w > 0; w >>= 1) {
		if((int)threadIdx.x < w) { s0[threadIdx.x] += s0[threadIdx.x + w]; s1[threadIdx.x] += s1[threadIdx.x + w]; }
		__syncthreads();
	}
	if(threadIdx.x == 0) { out[0] = s0[0]; out[1] = s1[0]; }
}

// scatters the compact block list of S into a dense column-major n x n matrix (upper blocks; diagnostics only)
__global__ void k_blocks_to_dense(size_t n_vals, const double *__restrict__ Sblk, const uint32_t *__restrict__ blk_row,
	const uint32_t *__restrict__ blk_col, size_t ld, double *__restrict__ S)
{
	const size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(e >= n_vals) return;
	const size_t b = e / 36;
	const unsigned q = (unsigned)(e - b * 36), c = q / 6, r = q - c * 6;
	S[((size_t)blk_col[b] * 6 + c) * ld + (size_t)blk_row[b] * 6 + r] = Sblk[e];
}

// The reference tries the dense solver on the reduced camera system first and falls back to the block-sparse one when
// the dense matrix cannot be allocated (LinearSolver_Schur.h:1836-1847). Here the choice is explicit: SPP_RCS_AUTO takes
// the dense path up to 16 384 unknowns (2 GiB of FP64, n^3 / 3 = 1.5e12 flop) and the supernodal one above.
static bool rcs_is_sparse(spp_ctx *ctx, size_t C)
{
	const int mode = ctx->snode.mode;
	if(mode == SPP_RCS_DENSE) return false;
	if(mode == SPP_RCS_SPARSE) return true;
	return C * 6 > 16384;
}

static const size_t g_phase_field[PH_COUNT] = {offsetof(spp_report_t, ms_linearise), offsetof(spp_report_t, ms_schur),
	offsetof(spp_report_t, ms_factor), offsetof(spp_report_t, ms_backsubst), offsetof(spp_report_t, ms_update),
	offsetof(spp_report_t, ms_chi2), offsetof(spp_report_t, ms_factor_kernel)};

static void phase_begin(spp_ctx *ctx, int ph)
{
	if(!ctx->phase_ev[ph][0]) {
		SPP_CUDA(cudaEventCreate(&ctx->phase_ev[ph][0]));
		SPP_CUDA(cudaEventCreate(&ctx->phase_ev[ph][1]));
	}
	SPP_CUDA(cudaEventRecord(ctx->phase_ev[ph][0], ctx->stream));
}

static void phase_add(spp_ctx *ctx, int ph, spp_report_t *rep)
{
	float ms = 0;
	cudaEventElapsedTime(&ms, ctx->phase_ev[ph][0], ctx->phase_ev[ph][1]);
	if(rep) *reinterpret_cast<double*>(reinterpret_cast<char*>(rep) + g_phase_field[ph]) += ms;
}

// synchronous mode: waits for the phase and adds its time to the report; asynchronous mode: only records the event
static void phase_end(spp_ctx *ctx, int ph, spp_report_t *rep)
{
	SPP_CUDA(cudaEventRecord(ctx->phase_ev[ph][1], ctx->stream));
	if(ctx->async_mode) {
		ctx->phase_used[ph] = true;
		return;
	}
	SPP_CUDA(cudaEventSynchronize(ctx->phase_ev[ph][1]));
	phase_add(ctx, ph, rep);
}

// after the synchronisation of an asynchronous iteration
static void phase_collect(spp_ctx *ctx, spp_report_t *rep)
{
	for(int ph = 0; ph < PH_COUNT; ++ ph) {
		if(ctx->phase_used[ph]) phase_add(ctx, ph, rep);
		ctx->phase_used[ph] = false;
	}
}

// Solves the damped Schur system on the current (U, V, W, gc, gp): dxc, dxp. Returns SPP_OK / SPP_NOT_POSDEF (in
// asynchronous mode always SPP_OK: the status arrives in ctx->async_info with the next synchronisation).
int schur_solve_current(spp_ctx *ctx, double alpha, spp_report_t *rep)
{
	SchurSystem &s = ctx->sys;
	const size_t n = s.C * 6;
	const bool sparse = rcs_is_sparse(ctx, s.C);
	if(ctx->world > 1 && !s.n_blocks_global)
		throw invalid_error("several ranks: the global block list of the reduced camera system is missing (spp_ba_set_graph builds it)");
	const bool compact = sparse || ctx->world > 1; // S as a compact block list (then scattered into the dense matrix if !sparse)
	if(sparse && !ctx->snode.valid) { // one-time symbolic analysis of the structure (host)
		if(ctx->world > 1) // the block list of the whole graph: every rank derives the same ordering and supernodes
			snode_symbolic(ctx, s.C, s.h_gblk_row, s.h_gblk_col);
		else {
			schur_fetch_host_pattern(ctx);
			snode_symbolic(ctx, s.C, s.h_blk_row, s.h_blk_col);
		}
	}
	phase_begin(ctx, PH_SCHUR);
	schur_form_reduced_system(ctx, alpha, (ctx->rank == 0)? alpha : 0.0, compact); // dense: S lives in the padded storage of the dense solver
	if(ctx->world > 1) { // sum the partial reduced camera systems and right-hand sides over the ranks
		allreduce_device(ctx, s.Sblk.p(), s.n_blocks_global * 36);
		allreduce_device(ctx, s.b.p(), n);
		if(!sparse) { // scatter the summed block list into the dense solver's storage
			const size_t ld = dense_chol_ld(n);
			s.S.resize(dense_chol_storage(n));
			s.S.zero(ctx->stream);
			k_blocks_to_dense<<<n_blocks(s.n_blocks_global * 36, 256), 256, 0, ctx->stream>>>(s.n_blocks_global * 36, s.Sblk.p(),
				s.gblk_row.p(), s.gblk_col.p(), ld, s.S.p());
			++ ctx->n_launches;
			SPP_CUDA(cudaGetLastError());
		}
	}
	if(s.keep_reduced && sparse && (s.n_blocks_global || n > 32768))
		s.S_copy.resize(0); // no dense copy of a block-sparse system this large / on several ranks: the query will say so
	else if(s.keep_reduced) {
		s.b_copy.resize(n);
		if(sparse) {
			const size_t ld = dense_chol_ld(n);
			s.S_copy.resize(dense_chol_storage(n));
			s.S_copy.zero(ctx->stream);
			k_blocks_to_dense<<<n_blocks(s.n_blocks * 36, 256), 256, 0, ctx->stream>>>(s.n_blocks * 36, s.Sblk.p(), s.blk_row.p(),
				s.blk_col.p(), ld, s.S_copy.p());
			++ ctx->n_launches;
			SPP_CUDA(cudaGetLastError());
		} else {
			s.S_copy.resize(s.S.size());
			SPP_CUDA(cudaMemcpyAsync(s.S_copy.p(), s.S.p(), s.S.size() * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
		}
		SPP_CUDA(cudaMemcpyAsync(s.b_copy.p(), s.b.p(), n * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
	}
	phase_end(ctx, PH_SCHUR, rep);
	phase_begin(ctx, PH_FACTOR);
	if(sparse) { // the block list survives the factorisation: with a copy of b the residual can be checked afterwards
		s.b_copy.resize(n);
		SPP_CUDA(cudaMemcpyAsync(s.b_copy.p(), s.b.p(), n * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
	}
	int rc = sparse? snode_factor_solve(ctx, s.Sblk.p(), s.b.p(), s.b.p()) : dense_chol_solve_device(ctx, s.S.p(), n, s.b.p());
	s.sparse_solved = sparse && rc == SPP_OK;
	phase_end(ctx, PH_FACTOR, rep);
	if(rc != SPP_OK)
		return rc;
	phase_begin(ctx, PH_BACKSUBST);
	s.dxc.resize(n);
	SPP_CUDA(cudaMemcpyAsync(s.dxc.p(), s.b.p(), n * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
	schur_backsubstitute(ctx);
	phase_end(ctx, PH_BACKSUBST, rep);
	return SPP_OK;
}

static double read_scalar(spp_ctx *ctx, const double *d_ptr, int n, double *out)
{
	ctx->h_scalars.resize(16);
	SPP_CUDA(cudaMemcpyAsync(ctx->h_scalars.p(), d_ptr, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
	SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	for(int i = 0; i < n; ++ i)
		out[i] = ctx->h_scalars[i];
	return out[0];
}

static double ba_chi2_host(spp_ctx *ctx)
{
	BAProblem &ba = ctx->ba;
	ba.partial.resize(4 * 1024);
	double *d_out = ba.partial.p() + 2048;
	ba_chi2_device(ctx, d_out);
	allreduce_device(ctx, d_out, 1);
	double v;
	read_scalar(ctx, d_out, 1, &v);
	return v;
}

static void ba_save_state(spp_ctx *ctx)
{
	BAProblem &ba = ctx->ba;
	ba.cam_state_saved.resize(ba.cam_state.size());
	ba.pts_saved.resize(ba.pts.size());
	SPP_CUDA(cudaMemcpyAsync(ba.cam_state_saved.p(), ba.cam_state.p(), ba.cam_state.size() * 8, cudaMemcpyDeviceToDevice, ctx->stream));
	SPP_CUDA(cudaMemcpyAsync(ba.pts_saved.p(), ba.pts.p(), ba.pts.size() * 8, cudaMemcpyDeviceToDevice, ctx->stream));
}

static void ba_load_state(spp_ctx *ctx)
{
	BAProblem &ba = ctx->ba;
	SPP_CUDA(cudaMemcpyAsync(ba.cam_state.p(), ba.cam_state_saved.p(), ba.cam_state.size() * 8, cudaMemcpyDeviceToDevice, ctx->stream));
	SPP_CUDA(cudaMemcpyAsync(ba.pts.p(), ba.pts_saved.p(), ba.pts.size() * 8, cudaMemcpyDeviceToDevice, ctx->stream));
}

// CNonlinearSolver_Lambda_LM::Optimize, LM.h:796-1116 (batch use: the system is "dirty" on entry)
static int ba_optimize(spp_ctx *ctx, size_t n_max_iteration_num, double f_min_dx_norm, spp_report_t *rep)
{
	BAProblem &ba = ctx->ba;
	SchurSystem &s = ctx->sys;
	memset(rep, 0, sizeof(*rep));
	if(!s.O)
		return SPP_OK; // "the system contains no edges at all: nothing to optimize"
	EventTimer total(ctx);
	cudaEvent_t t0 = ctx->ev[2], t1 = ctx->ev[3];
	SPP_CUDA(cudaEventRecord(t0, ctx->stream));
	EventTimer tm(ctx);

	tm.start();
	ba_linearise(ctx, true); // Refresh_Lambda, LM.h:828-831
	rep->ms_linearise += tm.stop_ms();
	// f_InitialDamping: tau * max over edges of the per-edge vertex Hessian diagonals, LM.h:151-199
	unsigned long long bits = 0;
	SPP_CUDA(cudaMemcpyAsync(&bits, ba.maxdiag.p(), 8, cudaMemcpyDeviceToHost, ctx->stream));
	SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	double f_max_diag;
	memcpy(&f_max_diag, &bits, 8);
	if(ctx->world > 1) { // max over ranks through the sum hook: every rank fills its own slot
		std::vector<double> slots(ctx->world, 0.0);
		slots[ctx->rank] = f_max_diag;
		ba.partial.resize(4 * 1024);
		double *d_slots = ba.partial.p() + 3072;
		SPP_CUDA(cudaMemcpyAsync(d_slots, slots.data(), ctx->world * 8, cudaMemcpyHostToDevice, ctx->stream));
		allreduce_device(ctx, d_slots, ctx->world);
		SPP_CUDA(cudaMemcpyAsync(slots.data(), d_slots, ctx->world * 8, cudaMemcpyDeviceToHost, ctx->stream));
		SPP_CUDA(cudaStreamSynchronize(ctx->stream));
		f_max_diag = *std::max_element(slots.begin(), slots.end());
	}
	double f_alpha = f_max_diag * 1e-3;
	double f_nu = 2.0;
	rep->alpha_initial = f_alpha;

	tm.start();
	double f_last_error = ba_chi2_host(ctx); // LM.h:899
	rep->ms_chi2 += tm.stop_ms();
	rep->chi2_initial = f_last_error;
	rep->chi2_final = f_last_error;

	bool b_system_dirty = false; // lambda matches the current linearisation point
	int fail = 10;
	// One host synchronisation per iteration: solve, step norms, update and chi2 are enqueued back to back, then the
	// factorisation status, the two dot products and chi2 are read together. The reference tests the step norm BEFORE it
	// applies the update (LM.h:1054) and stops at a failed factorisation (LM.h:972-974): both cases are undone here by
	// restoring the saved state, which leaves the same system behind.
	ctx->h_scalars.resize(16);
	double *h_vals = ctx->h_scalars.p();                    // [0..1] dots, [2] chi2
	int *h_info = reinterpret_cast<int*>(ctx->h_scalars.p() + 8);
	struct AsyncGuard { // the stages fall back to synchronous behaviour however this function is left
		spp_ctx *c;
		AsyncGuard(spp_ctx *ctx, int *info) : c(ctx) { c->async_mode = true; c->async_info = info; }
		~AsyncGuard() { c->async_mode = false; c->async_info = 0; for(int i = 0; i < PH_COUNT; ++ i) c->phase_used[i] = false; }
	} guard(ctx, h_info);
	for(size_t n_iteration = 0; n_iteration < n_max_iteration_num; ++ n_iteration) {
		if(n_iteration && b_system_dirty) {
			phase_begin(ctx, PH_LINEARISE);
			ba_linearise(ctx, false); // LM.h:942-949; a rejected step only re-damps (alpha is applied on the fly)
			phase_end(ctx, PH_LINEARISE, rep);
		}
		b_system_dirty = false;

		*h_info = 0;
		schur_solve_current(ctx, f_alpha, rep); // LinearSolve, LM.h:1512-1568 (status deferred)
		const int it = rep->n_iterations;
		++ rep->n_iterations;
		if(it < SPP_MAX_TRACE)
			rep->trace_alpha[it] = f_alpha;

		ba.partial.resize(4 * 1024);
		ba_step_dots_device(ctx, f_alpha, ba.partial.p() + 2048);
		allreduce_device(ctx, ba.partial.p() + 2048, 2);
		SPP_CUDA(cudaMemcpyAsync(h_vals, ba.partial.p() + 2048, 2 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));

		phase_begin(ctx, PH_UPDATE);
		ba_save_state(ctx);       // LM.h:1062
		ba_apply_update(ctx);     // PushValuesInGraphSystem, LM.h:1066
		phase_end(ctx, PH_UPDATE, rep);

		phase_begin(ctx, PH_CHI2);
		{
			double *d_chi2 = ba.partial.p() + 2048 + 8; // LM.h:1078
			ba_chi2_device(ctx, d_chi2);
			allreduce_device(ctx, d_chi2, 1);
			SPP_CUDA(cudaMemcpyAsync(h_vals + 2, d_chi2, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
		}
		phase_end(ctx, PH_CHI2, rep);

		SPP_CUDA(cudaStreamSynchronize(ctx->stream)); // the one synchronisation of the iteration
		phase_collect(ctx, rep);
		if(*h_info != 0) {
			ba_load_state(ctx);
			s.sparse_solved = false;
			rep->status = SPP_NOT_POSDEF;
			break; // "in case cholesky failed, quit", LM.h:972-974
		}
		const double dots[2] = {h_vals[0], h_vals[1]};
		const double f_residual_norm = sqrt(dots[0]);
		rep->last_dx_norm = f_residual_norm;
		if(it < SPP_MAX_TRACE)
			rep->trace_dx_norm[it] = f_residual_norm;
		if(f_residual_norm <= f_min_dx_norm) {
			ba_load_state(ctx); // the reference leaves before applying this step
			break; // LM.h:1054
		}
		const double f_error = h_vals[2];
		if(it < SPP_MAX_TRACE)
			rep->trace_chi2[it] = f_error;

		// CLevenbergMarquardt_Baseline::Aftermath, LM.h:204-223
		const double rho = (f_last_error - f_error) / dots[1];
		if(rho > 0) {
			f_alpha *= std::max(1 / 3.0, 1.0 - pow((2 * rho - 1), 3));
			f_nu = 2;
			f_last_error = f_error;
			rep->chi2_final = f_error;
			++ rep->n_accepted;
			if(it < SPP_MAX_TRACE)
				rep->trace_accepted[it] = 1;
			b_system_dirty = true;
		} else {
			f_alpha *= f_nu;
			f_nu *= 2;
			++ rep->n_rejected;
			ba_load_state(ctx); // "warning: chi2 rising", LM.h:1096-1106
			if(fail > 0) {
				-- fail;
				++ n_max_iteration_num;
			}
		}
	}
	rep->alpha_final = f_alpha;
	ba.linearised = !b_system_dirty;
	SPP_CUDA(cudaEventRecord(t1, ctx->stream));
	SPP_CUDA(cudaEventSynchronize(t1));
	float ms = 0;
	cudaEventElapsedTime(&ms, t0, t1);
	rep->ms_total = ms;
	return SPP_OK;
}

} // namespace spp

using namespace spp;

// ---------------------------------------------------------------------------------------------------

#define API_BEGIN(ctx) if(!(ctx)) return SPP_ERR_INVALID; try { SPP_CUDA(cudaSetDevice((ctx)->device));
#define API_END(ctx) } catch(const std::bad_alloc&) { (ctx)->last_error = "out of memory"; return SPP_ERR_NOMEM; } \
	catch(const spp::invalid_error &e) { (ctx)->last_error = e.what(); return SPP_ERR_INVALID; } \
	catch(const spp::comm_error &e) { (ctx)->last_error = e.what(); return SPP_ERR_COMM; } \
	catch(const std::exception &e) { (ctx)->last_error = e.what(); return SPP_ERR_CUDA; } return SPP_OK;

extern "C" {

int spp_create(int device, spp_ctx_t *p_ctx)
{
	if(!p_ctx)
		return SPP_ERR_INVALID;
	*p_ctx = 0;
	int n_dev = 0;
	cudaError_t e = cudaGetDeviceCount(&n_dev);
	if(e != cudaSuccess || n_dev == 0) {
		g_create_error = std::string("no CUDA device: ") + cudaGetErrorString(e) + " (libspp_b200 has no CPU fallback)";
		return SPP_ERR_CUDA;
	}
	if(device < 0 || device >= n_dev) {
		g_create_error = "device index out of range";
		return SPP_ERR_INVALID;
	}
	cudaDeviceProp prop;
	if(cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major != 10) {
		g_create_error = "libspp_b200 is built for sm_100a (B200) only";
		return SPP_ERR_CUDA;
	}
	spp_ctx *ctx = new(std::nothrow) spp_ctx();
	if(!ctx)
		return SPP_ERR_NOMEM;
	ctx->device = device;
	ctx->n_launches = 0;
	ctx->allreduce = 0;
	ctx->allreduce_user = 0;
	ctx->nccl_comm = 0;
	ctx->rank = 0;
	ctx->world = 1;
	ctx->async_mode = false;
	ctx->async_info = 0;
	for(int i = 0; i < PH_COUNT; ++ i) { ctx->phase_ev[i][0] = ctx->phase_ev[i][1] = 0; ctx->phase_used[i] = false; }
	ctx->stream = 0;
	ctx->copy_stream = 0;
	ctx->copy_done = 0;
	for(int i = 0; i < 16; ++ i) ctx->ev[i] = 0;
	try {
		SPP_CUDA(cudaSetDevice(device));
		int prio_lo = 0, prio_hi = 0;
		SPP_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
		SPP_CUDA(cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, prio_hi));
		for(int i = 0; i < 16; ++ i)
			SPP_CUDA(cudaEventCreate(&ctx->ev[i]));
		ctx->h_scalars.resize(16);
	} catch(const std::exception &ex) {
		g_create_error = ex.what();
		delete ctx;
		return SPP_ERR_CUDA;
	}
	char buf[256];
	if(spp::dbuf_use_pool()) { // freed device buffers stay in the pool (see dbuf_malloc); spp_destroy trims it
		cudaMemPool_t pool;
		if(cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
			uint64_t n_threshold = UINT64_MAX;
			cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &n_threshold);
		}
		(void)cudaGetLastError();
	}
	snprintf(buf, sizeof(buf), "spp_b200 0.1 sm_%d%d %s (%d SMs)", prop.major, prop.minor, prop.name, prop.multiProcessorCount);
	ctx->description = buf;
	*p_ctx = ctx;
	return SPP_OK;
}

void spp_destroy(spp_ctx_t ctx)
{
	if(!ctx)
		return;
	cudaSetDevice(ctx->device);
	if(ctx->stream)
		cudaStreamSynchronize(ctx->stream);
	if(getenv("SPP_ALLOC_STATS")) {
		const spp::DBufStats &as = spp::DBufStats::get();
		fprintf(stderr, "[spp alloc] %zu cudaMalloc (%.1f MB), %zu cudaFree, %.1f ms in both\n", as.n_malloc, as.bytes * 1e-6, as.n_free, as.ms);
	}
	if(ctx->nccl_comm) {
		// the stream is idle: ncclCommAbort frees the communicator without waiting for the other ranks (ncclCommDestroy
		// finalises collectively and hangs when a peer has already left)
		try { spp::nccl_api().CommAbort((ncclComm_t)ctx->nccl_comm); } catch(...) { }
		ctx->nccl_comm = 0;
	}
	if(ctx->stream)
		cudaStreamDestroy(ctx->stream);
	for(int i = 0; i < 16; ++ i)
		if(ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
	for(int i = 0; i < PH_COUNT; ++ i) {
		if(ctx->phase_ev[i][0]) { cudaEventDestroy(ctx->phase_ev[i][0]); cudaEventDestroy(ctx->phase_ev[i][1]); }
	}
	if(ctx->copy_stream) {
		cudaStreamDestroy(ctx->copy_stream);
		cudaEventDestroy(ctx->copy_done);
	}
	// side streams and events of the two Cholesky drivers
	spp::DenseChol &ch = ctx->chol;
	if(ch.bulk_stream) {
		cudaStreamDestroy(ch.bulk_stream);
		cudaStreamDestroy(ch.row_stream);
		for(int i = 0; i < 2; ++ i) {
			cudaEventDestroy(ch.ev_potrf[i]); cudaEventDestroy(ch.ev_first[i]); cudaEventDestroy(ch.ev_panel[i]);
			cudaEventDestroy(ch.ev_bulk[i]); cudaEventDestroy(ch.ev_row[i]);
		}
	}
	spp::SupernodalChol &sc = ctx->snode;
	for(int i = 0; i < spp::SupernodalChol::N_STREAMS; ++ i)
		if(sc.side[i]) cudaStreamDestroy(sc.side[i]);
	for(size_t i = 0; i < sc.ev_factor.size(); ++ i) {
		cudaEventDestroy(sc.ev_factor[i]); cudaEventDestroy(sc.ev_target[i]); cudaEventDestroy(sc.ev_x[i]);
	}
	const int n_device = ctx->device;
	delete ctx;
	if(spp::dbuf_use_pool()) { // what the context's buffers held goes back to the driver
		cudaMemPool_t pool;
		cudaDeviceSynchronize();
		if(cudaDeviceGetDefaultMemPool(&pool, n_device) == cudaSuccess)
			cudaMemPoolTrimTo(pool, 0);
		(void)cudaGetLastError();
	}
}

const char *spp_last_error(spp_ctx_t ctx)
{
	return ctx? ctx->last_error.c_str() : g_create_error.c_str();
}

int spp_describe(spp_ctx_t ctx, char *p_buffer, size_t n_buffer_size)
{
	if(!ctx || !p_buffer || !n_buffer_size)
		return SPP_ERR_INVALID;
	snprintf(p_buffer, n_buffer_size, "%s", ctx->description.c_str());
	return SPP_OK;
}

uint64_t spp_kernel_launches(spp_ctx_t ctx)
{
	return ctx? ctx->n_launches : 0;
}

void *spp_stream(spp_ctx_t ctx)
{
	return ctx? (void*)ctx->stream : 0;
}

int spp_synchronize(spp_ctx_t ctx)
{
	API_BEGIN(ctx)
	SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	API_END(ctx)
}

int spp_set_allreduce(spp_ctx_t ctx, spp_allreduce_fn fn, void *p_user, int rank, int world)
{
	if(!ctx || world < 1 || rank < 0 || rank >= world)
		return SPP_ERR_INVALID;
	if(rank != ctx->rank || world != ctx->world) {
		// the landmark partition and the global block list of a resident graph belong to the old (rank, world): a graph
		// must be set again before anything is solved
		ctx->ba.valid = false;
		ctx->snode.valid = false;
		ctx->slot.valid = false;
		ctx->sys.n_blocks_global = 0;
	}
	ctx->allreduce = fn;
	ctx->allreduce_user = p_user;
	ctx->rank = rank;
	ctx->world = world;
	return SPP_OK;
}

int spp_nccl_get_unique_id(void *p_id)
{
	if(!p_id)
		return SPP_ERR_INVALID;
	try {
		static_assert(sizeof(ncclUniqueId) == SPP_NCCL_UNIQUE_ID_BYTES, "ncclUniqueId size");
		ncclUniqueId id;
		SPP_NCCL(nccl_api().GetUniqueId(&id));
		memcpy(p_id, &id, sizeof(id));
	} catch(const std::exception &e) {
		g_create_error = e.what();
		return SPP_ERR_COMM;
	}
	return SPP_OK;
}

int spp_set_nccl(spp_ctx_t ctx, const void *p_id, int rank, int world)
{
	API_BEGIN(ctx)
	if(world < 1 || rank < 0 || rank >= world || (world > 1 && !p_id)) throw invalid_error("bad rank / world / id");
	if(ctx->nccl_comm) {
		SPP_CUDA(cudaStreamSynchronize(ctx->stream)); // nothing of ours is in flight: ncclCommAbort only frees
		nccl_api().CommAbort((ncclComm_t)ctx->nccl_comm);
		ctx->nccl_comm = 0;
	}
	if(rank != ctx->rank || world != ctx->world) { // as spp_set_allreduce: the resident graph belongs to the old (rank, world)
		ctx->ba.valid = false;
		ctx->snode.valid = false;
		ctx->slot.valid = false;
		ctx->sys.n_blocks_global = 0;
	}
	ctx->rank = rank;
	ctx->world = world;
	if(world > 1) {
		ncclUniqueId id;
		memcpy(&id, p_id, sizeof(id));
		ncclComm_t comm;
		SPP_NCCL(nccl_api().CommInitRank(&comm, world, id, rank));
		ctx->nccl_comm = comm;
	}
	API_END(ctx)
}

int spp_ba_set_graph(spp_ctx_t ctx, size_t n_vertices, const uint8_t *p_vertex_type,
	const double *p_cam_params, const double *p_points, size_t n_observations,
	const uint64_t *p_obs_point, const uint64_t *p_obs_camera, const double *p_z, const double *p_info)
{
	API_BEGIN(ctx)
	// host pointers are borrowed for the duration of the call: whichever way it is left (an invalid_error thrown by the
	// analysis included), no copy from the caller's buffers may still be in flight on the side stream
	struct CopyGuard {
		spp_ctx *c;
		~CopyGuard() { if(c->copy_stream) cudaStreamSynchronize(c->copy_stream); }
	} copy_guard = {ctx};
	BAProblem &ba = ctx->ba;
	ba.valid = false;
	ba.raw_on_device = false;
	ctx->slot.valid = false;
	ctx->slot.filled = false;
	ctx->snode.valid = false;
	ctx->sys.n_blocks_global = 0;
	if(!p_vertex_type || (n_observations && (!p_obs_point || !p_obs_camera || !p_z || !p_info)))
		throw invalid_error("null argument");
	ba.n_vertices = n_vertices;
	ba.vtype.assign(p_vertex_type, p_vertex_type + n_vertices);
	ba.vertex_local.resize(n_vertices);
	{ // local index of every vertex within its type, and the two inverse lists (half a million vertices: no push_back)
		size_t n_cam = 0;
		for(size_t v = 0; v < n_vertices; ++ v) {
			if(p_vertex_type[v] > 1)
				throw invalid_error("vertex type must be 0 (camera) or 1 (point)");
			n_cam += p_vertex_type[v] == 0;
		}
		ba.cam_vertex.resize(n_cam);
		ba.pt_vertex.resize(n_vertices - n_cam);
		uint32_t ic = 0, ip = 0;
		uint32_t *p_local = n_vertices? &ba.vertex_local[0] : 0, *p_cv = n_cam? &ba.cam_vertex[0] : 0,
			*p_pv = (n_vertices - n_cam)? &ba.pt_vertex[0] : 0;
		for(size_t v = 0; v < n_vertices; ++ v) {
			if(p_vertex_type[v] == 0) {
				p_local[v] = ic;
				p_cv[ic ++] = (uint32_t)v;
			} else {
				p_local[v] = ip;
				p_pv[ip ++] = (uint32_t)v;
			}
		}
	}
	const size_t C = ba.cam_vertex.size(), P = ba.pt_vertex.size(), O = n_observations;
	if((C && !p_cam_params) || (P && !p_points))
		throw invalid_error("null vertex data");
	ba.uf_is_cam = n_vertices? (p_vertex_type[0] == 0) : 1;
	ba.uf_index = n_vertices? 0 : -1; // vertex id 0 is local index 0 of its type

	cudaStream_t st = ctx->stream;
	std::vector<double> cs(C * 6), ci(C * 5);
	for(size_t c = 0; c < C; ++ c) {
		for(int k = 0; k < 6; ++ k) cs[c * 6 + k] = p_cam_params[c * 11 + k];
		for(int k = 0; k < 5; ++ k) ci[c * 5 + k] = p_cam_params[c * 11 + 6 + k];
	}
	ba.P_global = P;
	ba.pt_begin = 0;
	ba.pt_end = P;
	if(ctx->world == 1 && schur_structure_device_supported(C) && !getenv("SPP_HOST_SYMBOLIC")) {
		// single GPU: the observation arrays go to the device as they are; local indices, tracks, camera lists, the
		// block and pair lists of the reduced camera system and the track-ordered measurements are built there
		ba_upload_and_analyse_device(ctx, C, P, O, p_obs_point, p_obs_camera, p_z, p_info);
		ba.pts.upload(p_points, P * 3, st);
		ba.pts0.upload(p_points, P * 3, st);
		ba.raw_on_device = true;
		ba.n_obs_raw = O;
	} else if(ctx->world > 1 && schur_structure_device_supported(C) && !getenv("SPP_HOST_SYMBOLIC")) {
		// several ranks: the same analysis on the device, for the whole graph (global block list, track lengths) and
		// then for this rank's landmark slice
		ba_upload_and_analyse_device_sliced(ctx, C, P, O, p_obs_point, p_obs_camera, p_z, p_info);
		const size_t P_local = ba.pt_end - ba.pt_begin;
		ba.pts.upload(p_points + ba.pt_begin * 3, P_local * 3, st);
		ba.pts0.upload(p_points + ba.pt_begin * 3, P_local * 3, st);
	} else {
		std::vector<uint32_t> h_cam(O), h_pt(O);
		for(size_t e = 0; e < O; ++ e) {
			uint64_t vp = p_obs_point[e], vc = p_obs_camera[e];
			if(vp >= n_vertices || vc >= n_vertices || p_vertex_type[vp] != 1 || p_vertex_type[vc] != 0)
				throw invalid_error("observation references a vertex of the wrong type or out of range");
			h_cam[e] = ba.vertex_local[vc];
			h_pt[e] = ba.vertex_local[vp];
		}
		// multi-GPU: this rank keeps a contiguous slice of the landmarks with all their observations; cameras are
		// replicated (SURVEY 8(e)). The slice bounds balance the Schur-product work sum k_p (k_p + 1) / 2 + k_p.
		ctx->sys.n_blocks_global = 0;
		std::vector<uint32_t> g_row, g_col;
		// several ranks: the partial reduced camera systems are summed as compact block lists under the block pattern of
		// the whole graph (Venice: 33 MB instead of the 220 MB dense matrix), for the dense and the block-sparse solver alike
		const bool b_global_pattern = ctx->world > 1;
		if(b_global_pattern)
			build_global_rcs_pattern(C, P, h_cam, h_pt, g_row, g_col);
		if(ctx->world > 1) {
			std::vector<uint32_t> track_len(P, 0);
			for(size_t e = 0; e < O; ++ e)
				++ track_len[h_pt[e]];
			std::vector<uint64_t> bounds(ctx->world + 1);
			spp_partition_landmarks(P, P? &track_len[0] : 0, ctx->world, &bounds[0]);
			ba.pt_begin = bounds[ctx->rank];
			ba.pt_end = bounds[ctx->rank + 1];
			std::vector<uint32_t> l_cam, l_pt, kept;
			for(size_t e = 0; e < O; ++ e) {
				if(h_pt[e] >= ba.pt_begin && h_pt[e] < ba.pt_end) {
					l_cam.push_back(h_cam[e]);
					l_pt.push_back(uint32_t(h_pt[e] - ba.pt_begin));
					kept.push_back((uint32_t)e);
				}
			}
			h_cam.swap(l_cam);
			h_pt.swap(l_pt);
			build_schur_structure(ctx, C, ba.pt_end - ba.pt_begin, h_cam, h_pt, ba.obs_orig, ba.h_obs_cam, ba.h_obs_pt);
			for(size_t k = 0; k < ba.obs_orig.size(); ++ k)
				ba.obs_orig[k] = kept[ba.obs_orig[k]]; // local track position -> original (global) edge index
			if(b_global_pattern) {
				std::vector<uint32_t> slot;
				map_blocks_to_global(C, ctx->sys.h_blk_row, ctx->sys.h_blk_col, g_row, g_col, slot);
				ctx->sys.blk_slot.upload(slot, st);
				ctx->sys.gblk_row.upload(g_row, st);
				ctx->sys.gblk_col.upload(g_col, st);
				ctx->sys.n_blocks_global = g_row.size();
				ctx->sys.h_gblk_row.swap(g_row);
				ctx->sys.h_gblk_col.swap(g_col);
				SPP_CUDA(cudaStreamSynchronize(st));
			}
		} else
			build_schur_structure(ctx, C, P, h_cam, h_pt, ba.obs_orig, ba.h_obs_cam, ba.h_obs_pt);
		ba.host_maps_valid = true;
		ba.d_obs_orig.upload(ba.obs_orig, st);
		const size_t P_local = ba.pt_end - ba.pt_begin, O_local = ba.obs_orig.size();
		ba.pts.upload(p_points + ba.pt_begin * 3, P_local * 3, st);
		ba.pts0.upload(p_points + ba.pt_begin * 3, P_local * 3, st);
		std::vector<double> tz(O_local * 2), ti(O_local * 4);
		for(size_t k = 0; k < O_local; ++ k) {
			size_t e = ba.obs_orig[k];
			tz[k * 2] = p_z[e * 2]; tz[k * 2 + 1] = p_z[e * 2 + 1];
			for(int q = 0; q < 4; ++ q) ti[k * 4 + q] = p_info[e * 4 + q];
		}
		ba.z.upload(tz, st);
		ba.info.upload(ti, st);
		SPP_CUDA(cudaStreamSynchronize(st)); // the host vectors go out of scope
	}
	{
		const size_t P_local = ba.pt_end - ba.pt_begin;
		if(!ba.uf_is_cam && n_vertices) // the unary factor sits on landmark 0: only its owner adds it
			ba.uf_index = (ba.pt_begin == 0 && P_local)? 0 : -1;
		else if(ctx->rank != 0)
			ba.uf_index = -1; // camera 0: added once, by rank 0
	}
	ba.cam_state.upload(cs, st);
	ba.cam_intr.upload(ci, st);
	ba.cam_state0.upload(cs, st);
	ba.camRt.resize(C * 84);
	ba.camK.resize(C * 5);
	ba.partial.resize(4 * 1024);
	ba.maxdiag.resize(1);
	SPP_CUDA(cudaStreamSynchronize(st));
	ba.linearised = false;
	ba.valid = true;
	API_END(ctx)
}

int spp_ba_append_graph(spp_ctx_t ctx, size_t n_new_vertices, const uint8_t *p_vertex_type,
	const double *p_cam_params, const double *p_points, size_t n_new_observations,
	const uint64_t *p_obs_point, const uint64_t *p_obs_camera, const double *p_z, const double *p_info)
{
	API_BEGIN(ctx)
	struct CopyGuard {
		spp_ctx *c;
		~CopyGuard() { if(c->copy_stream) cudaStreamSynchronize(c->copy_stream); cudaStreamSynchronize(c->stream); }
	} copy_guard = {ctx};
	BAProblem &ba = ctx->ba;
	if(!ba.valid || !ba.raw_on_device || ctx->world != 1)
		throw invalid_error("spp_ba_append_graph: needs a graph set by spp_ba_set_graph on a single-GPU context (device-side analysis)");
	if((n_new_vertices && !p_vertex_type) || (n_new_observations && (!p_obs_point || !p_obs_camera || !p_z || !p_info)))
		throw invalid_error("null argument");
	size_t n_new_cams = 0;
	for(size_t v = 0; v < n_new_vertices; ++ v) {
		if(p_vertex_type[v] > 1)
			throw invalid_error("vertex type must be 0 (camera) or 1 (point)");
		n_new_cams += p_vertex_type[v] == 0;
	}
	const size_t n_new_pts = n_new_vertices - n_new_cams;
	if((n_new_cams && !p_cam_params) || (n_new_pts && !p_points))
		throw invalid_error("null vertex data");
	const size_t V0 = ba.n_vertices, C0 = ba.cam_vertex.size(), P0 = ba.pt_vertex.size(), O0 = ba.n_obs_raw;
	const size_t C = C0 + n_new_cams, P = P0 + n_new_pts;
	if(!schur_structure_device_supported(C))
		throw invalid_error("spp_ba_append_graph: too many cameras for the device-side analysis");
	// from here on the context holds no valid graph until the analysis went through
	ba.valid = false;
	ctx->slot.valid = false;
	ctx->slot.filled = false;
	ctx->snode.valid = false;
	ctx->sys.n_blocks_global = 0;
	ba.raw_on_device = false;
	ba.vtype.insert(ba.vtype.end(), p_vertex_type, p_vertex_type + n_new_vertices);
	ba.vertex_local.resize(V0 + n_new_vertices);
	for(size_t v = 0; v < n_new_vertices; ++ v) {
		if(p_vertex_type[v] == 0) {
			ba.vertex_local[V0 + v] = (uint32_t)ba.cam_vertex.size();
			ba.cam_vertex.push_back(uint32_t(V0 + v));
		} else {
			ba.vertex_local[V0 + v] = (uint32_t)ba.pt_vertex.size();
			ba.pt_vertex.push_back(uint32_t(V0 + v));
		}
	}
	ba.n_vertices = V0 + n_new_vertices;
	if(!V0 && n_new_vertices) { // (an empty graph was set before: vertex id 0 arrives now)
		ba.uf_is_cam = p_vertex_type[0] == 0;
		ba.uf_index = 0;
	}
	cudaStream_t st = ctx->stream;
	// the vertices already there keep their current (and their initial) states; the new ones go behind them
	std::vector<double> cs(n_new_cams * 6), ci(n_new_cams * 5);
	for(size_t c = 0; c < n_new_cams; ++ c) {
		for(int k = 0; k < 6; ++ k) cs[c * 6 + k] = p_cam_params[c * 11 + k];
		for(int k = 0; k < 5; ++ k) ci[c * 5 + k] = p_cam_params[c * 11 + 6 + k];
	}
	ba.cam_state.grow_keep(C * 6, st);
	ba.cam_state0.grow_keep(C * 6, st);
	ba.cam_intr.grow_keep(C * 5, st);
	ba.pts.grow_keep(P * 3, st);
	ba.pts0.grow_keep(P * 3, st);
	if(n_new_cams) {
		SPP_CUDA(cudaMemcpyAsync(ba.cam_state.p() + C0 * 6, cs.data(), cs.size() * sizeof(double), cudaMemcpyHostToDevice, st));
		SPP_CUDA(cudaMemcpyAsync(ba.cam_state0.p() + C0 * 6, cs.data(), cs.size() * sizeof(double), cudaMemcpyHostToDevice, st));
		SPP_CUDA(cudaMemcpyAsync(ba.cam_intr.p() + C0 * 5, ci.data(), ci.size() * sizeof(double), cudaMemcpyHostToDevice, st));
	}
	if(n_new_pts) {
		SPP_CUDA(cudaMemcpyAsync(ba.pts.p() + P0 * 3, p_points, n_new_pts * 3 * sizeof(double), cudaMemcpyHostToDevice, st));
		SPP_CUDA(cudaMemcpyAsync(ba.pts0.p() + P0 * 3, p_points, n_new_pts * 3 * sizeof(double), cudaMemcpyHostToDevice, st));
	}
	ba.P_global = P;
	ba.pt_begin = 0;
	ba.pt_end = P;
	ba_append_and_analyse_device(ctx, C, P, O0, n_new_observations, p_obs_point, p_obs_camera, p_z, p_info);
	ba.camRt.resize(C * 84);
	ba.camK.resize(C * 5);
	SPP_CUDA(cudaStreamSynchronize(st)); // the host vectors go out of scope
	ba.n_obs_raw = O0 + n_new_observations;
	ba.raw_on_device = true;
	ba.linearised = false;
	ba.valid = true;
	API_END(ctx)
}

int spp_ba_set_states(spp_ctx_t ctx, const double *p_cam_states, const double *p_points)
{
	API_BEGIN(ctx)
	if(!ctx->ba.valid) throw invalid_error("no BA graph");
	if(p_cam_states)
		SPP_CUDA(cudaMemcpyAsync(ctx->ba.cam_state.p(), p_cam_states, ctx->sys.C * 6 * 8, cudaMemcpyHostToDevice, ctx->stream));
	if(p_points) // p_points is the full point array; this context holds the slice [pt_begin, pt_end)
		SPP_CUDA(cudaMemcpyAsync(ctx->ba.pts.p(), p_points + ctx->ba.pt_begin * 3, ctx->sys.P * 3 * 8, cudaMemcpyHostToDevice, ctx->stream));
	SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	ctx->ba.linearised = false;
	API_END(ctx)
}

int spp_ba_get_partition(spp_ctx_t ctx, uint64_t *p_begin, uint64_t *p_end)
{
	if(!ctx || !ctx->ba.valid)
		return SPP_ERR_INVALID;
	if(p_begin) *p_begin = ctx->ba.pt_begin;
	if(p_end) *p_end = ctx->ba.pt_end;
	return SPP_OK;
}

int spp_ba_get_states(spp_ctx_t ctx, double *p_cam_states, double *p_points)
{
	API_BEGIN(ctx)
	if(!ctx->ba.valid) throw invalid_error("no BA graph");
	if(p_cam_states)
		ctx->ba.cam_state.download(p_cam_states, ctx->sys.C * 6, ctx->stream);
	if(p_points) // only this context's slice of the full point array is written
		ctx->ba.pts.download(p_points + ctx->ba.pt_begin * 3, ctx->sys.P * 3, ctx->stream);
	SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	API_END(ctx)
}

int spp_ba_gather_states(spp_ctx_t ctx, double *p_cam_states, double *p_points)
{
	API_BEGIN(ctx)
	BAProblem &ba = ctx->ba;
	if(!ba.valid) throw invalid_error("no BA graph");
	if(p_cam_states) // the cameras are replicated: every rank holds the same states
		ba.cam_state.download(p_cam_states, ctx->sys.C * 6, ctx->stream);
	if(p_points) {
		if(ctx->world > 1) { // every rank contributes its landmark slice to a zeroed array of all landmarks; one sum
			DBuf<double> &all = ctx->sys.cov_pt; // (scratch of the marginals, which a partitioned context does not provide)
			all.resize(ba.P_global * 3);
			all.zero(ctx->stream);
			SPP_CUDA(cudaMemcpyAsync(all.p() + ba.pt_begin * 3, ba.pts.p(), ctx->sys.P * 3 * sizeof(double), cudaMemcpyDeviceToDevice,
				ctx->stream));
			allreduce_device(ctx, all.p(), ba.P_global * 3);
			all.download(p_points, ba.P_global * 3, ctx->stream);
		} else
			ba.pts.download(p_points, ctx->sys.P * 3, ctx->stream);
	}
	SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	API_END(ctx)
}

int spp_ba_restore_initial(spp_ctx_t ctx)
{
	API_BEGIN(ctx)
	BAProblem &ba = ctx->ba;
	if(!ba.valid) throw invalid_error("no BA graph");
	SPP_CUDA(cudaMemcpyAsync(ba.cam_state.p(), ba.cam_state0.p(), ba.cam_state.size() * 8, cudaMemcpyDeviceToDevice, ctx->stream));
	SPP_CUDA(cudaMemcpyAsync(ba.pts.p(), ba.pts0.p(), ba.pts.size() * 8, cudaMemcpyDeviceToDevice, ctx->stream));
	ba.linearised = false;
	API_END(ctx)
}

int spp_ba_set_jacobian_mode(spp_ctx_t ctx, int mode)
{
	if(!ctx || (mode != SPP_JAC_FD_REFERENCE && mode != SPP_JAC_ANALYTIC))
		return SPP_ERR_INVALID;
	ctx->ba.jac_mode = mode;
	ctx->ba.linearised = false;
	return SPP_OK;
}

int spp_ba_set_robust_loss(spp_ctx_t ctx, int kind, double scale)
{
	if(!ctx || (kind != SPP_LOSS_NONE && kind != SPP_LOSS_HUBER && kind != SPP_LOSS_CAUCHY))
		return SPP_ERR_INVALID;
	if(kind != SPP_LOSS_NONE && !(std::isfinite(scale) && scale > 0))
		return SPP_ERR_INVALID;
	ctx->ba.loss_kind = kind;
	ctx->ba.loss_scale = kind == SPP_LOSS_NONE? 1.0 : scale;
	ctx->ba.linearised = false;
	return SPP_OK;
}

int spp_ba_get_observation_errors(spp_ctx_t ctx, double *p_sq_error, double *p_weight)
{
	API_BEGIN(ctx)
	BAProblem &ba = ctx->ba;
	SchurSystem &s = ctx->sys;
	if(!ba.valid) throw invalid_error("no BA graph");
	if(ctx->world > 1) throw invalid_error("not available on a landmark-partitioned (multi-GPU) context");
	ba.obs_err.resize(2 * s.O + 2);
	ba_obs_errors_device(ctx, ba.obs_err.p(), ba.obs_err.p() + s.O);
	if(p_sq_error) ba.obs_err.download(p_sq_error, s.O, ctx->stream);
	if(p_weight && s.O) SPP_CUDA(cudaMemcpyAsync(p_weight, ba.obs_err.p() + s.O, s.O * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
	SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	API_END(ctx)
}

int spp_ba_linearise(spp_ctx_t ctx)
{
	API_BEGIN(ctx)
	if(!ctx->ba.valid) throw invalid_error("no BA graph");
	ba_linearise(ctx, true);
	SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	API_END(ctx)
}

int spp_ba_get_lambda(spp_ctx_t ctx, uint64_t *p_n_block_cols, uint64_t *p_n_blocks, uint64_t *p_n_values,
	uint64_t *p_col_dims, uint64_t *p_col_ptr, uint64_t *p_row_idx, double *p_values, double *p_eta)
{
	API_BEGIN(ctx)
	BAProblem &ba = ctx->ba;
	SchurSystem &s = ctx->sys;
	if(!ba.valid) throw invalid_error("no BA graph");
	if(ctx->world > 1) throw invalid_error("not available on a landmark-partitioned (multi-GPU) context");
	const size_t NV = ba.n_vertices, O = s.O;
	ba_fetch_host_maps(ctx);
	// structure in vertex id order: column v holds the off-diagonal blocks (row u < v) and the diagonal block last
	std::vector<std::vector<std::pair<uint32_t, uint32_t> > > cols(NV); // (row vertex, track position)
	for(size_t k = 0; k < O; ++ k) {
		uint32_t vc = ba.cam_vertex[ba.h_obs_cam[k]], vp = ba.pt_vertex[ba.h_obs_pt[k]];
		uint32_t r = std::min(vc, vp), c = std::max(vc, vp);
		cols[c].push_back(std::make_pair(r, (uint32_t)k));
	}
	size_t n_blocks_total = 0, n_values = 0;
	for(size_t v = 0; v < NV; ++ v) {
		std::sort(cols[v].begin(), cols[v].end());
		n_blocks_total += cols[v].size() + 1;
		size_t d = ba.vtype[v] == 0? 6 : 3;
		n_values += cols[v].size() * 18 + d * d;
	}
	if(p_n_block_cols) *p_n_block_cols = NV;
	if(p_n_blocks) *p_n_blocks = n_blocks_total;
	if(p_n_values) *p_n_values = n_values;
	if(p_col_dims)
		for(size_t v = 0; v < NV; ++ v) p_col_dims[v] = ba.vtype[v] == 0? 6 : 3;
	if(p_col_ptr || p_row_idx || p_values) {
		if(p_values && !ba.linearised) throw invalid_error("spp_ba_linearise() has not been called");
		std::vector<double> hU, hV, hW;
		if(p_values) {
			hU.resize(s.C * 36); hV.resize(s.P * 9); hW.resize(O * 18);
			s.U.download(hU.data(), hU.size(), ctx->stream);
			s.V.download(hV.data(), hV.size(), ctx->stream);
			s.W.download(hW.data(), hW.size(), ctx->stream);
			SPP_CUDA(cudaStreamSynchronize(ctx->stream));
		}
		size_t nb = 0, nv = 0;
		for(size_t v = 0; v < NV; ++ v) {
			if(p_col_ptr) p_col_ptr[v] = nb;
			const bool v_is_cam = ba.vtype[v] == 0;
			for(size_t q = 0; q < cols[v].size(); ++ q, ++ nb) {
				if(p_row_idx) p_row_idx[nb] = cols[v][q].first;
				if(p_values) {
					const double *w = &hW[(size_t)cols[v][q].second * 18]; // 6x3 column-major
					if(!v_is_cam) { // row = camera, column = point: block is W (6x3)
						for(int i = 0; i < 18; ++ i) p_values[nv + i] = w[i];
					} else { // row = point, column = camera: block is W^T (3x6)
						for(int c = 0; c < 6; ++ c)
							for(int r = 0; r < 3; ++ r)
								p_values[nv + c * 3 + r] = w[r * 6 + c];
					}
				}
				nv += 18;
			}
			if(p_row_idx) p_row_idx[nb] = v;
			++ nb;
			const size_t d = v_is_cam? 6 : 3;
			if(p_values) {
				const double *src = v_is_cam? &hU[(size_t)ba.vertex_local[v] * 36] : &hV[(size_t)ba.vertex_local[v] * 9];
				for(size_t i = 0; i < d * d; ++ i) p_values[nv + i] = src[i];
			}
			nv += d * d;
		}
		if(p_col_ptr) p_col_ptr[NV] = nb;
	}
	if(p_eta) {
		if(!ba.linearised) throw invalid_error("spp_ba_linearise() has not been called");
		std::vector<double> hgc(s.C * 6), hgp(s.P * 3);
		s.gc.download(hgc.data(), hgc.size(), ctx->stream);
		s.gp.download(hgp.data(), hgp.size(), ctx->stream);
		SPP_CUDA(cudaStreamSynchronize(ctx->stream));
		size_t off = 0;
		for(size_t v = 0; v < NV; ++ v) {
			if(ba.vtype[v] == 0) {
				for(int i = 0; i < 6; ++ i) p_eta[off + i] = hgc[(size_t)ba.vertex_local[v] * 6 + i];
				off += 6;
			} else {
				for(int i = 0; i < 3; ++ i) p_eta[off + i] = hgp[(size_t)ba.vertex_local[v] * 3 + i];
				off += 3;
			}
		}
	}
	API_END(ctx)
}

int spp_ba_get_blocks(spp_ctx_t ctx, double *p_U, double *p_V, double *p_W, double *p_eta_c, double *p_eta_p)
{
	API_BEGIN(ctx)
	BAProblem &ba = ctx->ba;
	SchurSystem &s = ctx->sys;
	if(!ba.valid) throw invalid_error("no BA graph");
	if(ctx->world > 1) throw invalid_error("not available on a landmark-partitioned (multi-GPU) context");
	if(!ba.linearised) throw invalid_error("spp_ba_linearise() has not been called");
	if(p_U) s.U.download(p_U, s.C * 36, ctx->stream);
	if(p_V) s.V.download(p_V, s.P * 9, ctx->stream);
	if(p_eta_c) s.gc.download(p_eta_c, s.C * 6, ctx->stream);
	if(p_eta_p) s.gp.download(p_eta_p, s.P * 3, ctx->stream);
	std::vector<double> hW;
	if(p_W) {
		hW.resize(s.O * 18);
		s.W.download(hW.data(), hW.size(), ctx->stream);
	}
	SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	if(p_W)
		ba_fetch_host_maps(ctx);
	if(p_W) { // track order -> edge insertion order
		for(size_t k = 0; k < s.O; ++ k)
			memcpy(p_W + (size_t)ba.obs_orig[k] * 18, &hW[k * 18], 18 * sizeof(double));
	}
	API_END(ctx)
}

int spp_ba_chi2(spp_ctx_t ctx, double *p_chi2)
{
	API_BEGIN(ctx)
	if(!ctx->ba.valid || !p_chi2) throw invalid_error("no BA graph");
	*p_chi2 = ba_chi2_host(ctx);
	API_END(ctx)
}

static void ba_download_dx(spp_ctx *ctx, double *p_dx)
{
	BAProblem &ba = ctx->ba;
	SchurSystem &s = ctx->sys;
	std::vector<double> hc(s.C * 6), hp(s.P * 3);
	s.dxc.download(hc.data(), hc.size(), ctx->stream);
	s.dxp.download(hp.data(), hp.size(), ctx->stream);
	SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	size_t off = 0;
	for(size_t v = 0; v < ba.n_vertices; ++ v) {
		if(ba.vtype[v] == 0) {
			for(int i = 0; i < 6; ++ i) p_dx[off + i] = hc[(size_t)ba.vertex_local[v] * 6 + i];
			off += 6;
		} else {
			for(int i = 0; i < 3; ++ i) p_dx[off + i] = hp[(size_t)ba.vertex_local[v] * 3 + i];
			off += 3;
		}
	}
}

int spp_ba_solve_step(spp_ctx_t ctx, double alpha, double *p_dx)
{
	int rc = SPP_OK;
	API_BEGIN(ctx)
	if(!ctx->ba.valid) throw invalid_error("no BA graph");
	if(ctx->world > 1) throw invalid_error("not available on a landmark-partitioned (multi-GPU) context");
	if(!ctx->ba.linearised) ba_linearise(ctx, true);
	rc = schur_solve_current(ctx, alpha, 0);
	if(rc == SPP_OK && p_dx)
		ba_download_dx(ctx, p_dx);
	if(rc != SPP_OK) return rc;
	API_END(ctx)
}

// marginals of the system held as (U, V, W) to host arrays (local camera / point order)
static int marginals_to_host(spp_ctx *ctx, double alpha, double *p_cam_cov, double *p_pt_cov)
{
	SchurSystem &s = ctx->sys;
	if(ctx->world > 1) throw invalid_error("marginals are not available on a landmark-partitioned (multi-GPU) context");
	if(!s.C) throw invalid_error("no cameras");
	if(rcs_is_sparse(ctx, s.C))
		throw invalid_error("marginals need the dense reduced camera system (6 C <= 16384, or spp_schur_set_rcs_solver(SPP_RCS_DENSE))");
	DBuf<double> &d_cam = s.cov_cam, &d_pt = s.cov_pt;
	if(p_cam_cov) d_cam.resize(s.C * 36);
	if(p_pt_cov) d_pt.resize(s.P * 9);
	int rc = schur_marginals_current(ctx, alpha, p_cam_cov? d_cam.p() : 0, p_pt_cov? d_pt.p() : 0);
	if(rc != SPP_OK)
		return rc;
	if(p_cam_cov) d_cam.download(p_cam_cov, s.C * 36, ctx->stream);
	if(p_pt_cov) d_pt.download(p_pt_cov, s.P * 9, ctx->stream);
	SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	return SPP_OK;
}

int spp_ba_marginals(spp_ctx_t ctx, double alpha, double *p_cam_cov, double *p_pt_cov)
{
	int rc = SPP_OK;
	API_BEGIN(ctx)
	if(!ctx->ba.valid) throw invalid_error("no BA graph");
	if(!ctx->ba.linearised) ba_linearise(ctx, true);
	rc = marginals_to_host(ctx, alpha, p_cam_cov, p_pt_cov);
	if(rc != SPP_OK) return rc;
	API_END(ctx)
}

int spp_schur_marginals(spp_ctx_t ctx, double alpha, double *p_cam_cov, double *p_pt_cov)
{
	int rc = SPP_OK;
	API_BEGIN(ctx)
	if(!ctx->slot.valid || !ctx->slot.filled) throw invalid_error("no system: spp_schur_symbolic and spp_schur_solve first");
	rc = marginals_to_host(ctx, alpha, p_cam_cov, p_pt_cov);
	if(rc != SPP_OK) return rc;
	API_END(ctx)
}

// the same through the block-sparse (supernodal) factorisation and its selected inversion, whatever the solver mode
static int marginals_sparse_to_host(spp_ctx *ctx, double alpha, double *p_cam_cov, double *p_pt_cov)
{
	SchurSystem &s = ctx->sys;
	if(ctx->world > 1) throw invalid_error("marginals are not available on a landmark-partitioned (multi-GPU) context");
	if(!s.C) throw invalid_error("no cameras");
	DBuf<double> &d_cam = s.cov_cam, &d_pt = s.cov_pt;
	if(p_cam_cov) d_cam.resize(s.C * 36);
	if(p_pt_cov) d_pt.resize(s.P * 9);
	// SPP_MARGINALS_TIMING: the phases of the call to stderr
	static const bool timing = getenv("SPP_MARGINALS_TIMING") != 0;
	float ms[5] = {0, 0, 0, 0, 0};
	int rc = schur_marginals_sparse_current(ctx, alpha, p_cam_cov? d_cam.p() : 0, p_pt_cov? d_pt.p() : 0, timing? ms : 0);
	if(rc != SPP_OK)
		return rc;
	if(timing) {
		const SupernodalChol &sc = ctx->snode;
		fprintf(stderr, "[spp marginals sparse] schur %.3f ms, factor %.3f ms, selected inversion %.3f ms (%.3e flops, %.2f TFLOP/s), "
			"cameras %.3f ms, points %.3f ms; scratch %.3f GB (main) + %d x %.3f GB (lanes), panels %.3f GB\n", ms[0], ms[1], ms[2],
			sc.selinv_flops, sc.selinv_flops / ms[2] * 1e-9, ms[3], ms[4], sc.selinv_main_doubles * 8e-9, (int)SupernodalChol::N_STREAMS,
			sc.selinv_lane_doubles * 8e-9, sc.d_L.size() * 8e-9);
	}
	if(p_cam_cov) d_cam.download(p_cam_cov, s.C * 36, ctx->stream);
	if(p_pt_cov) d_pt.download(p_pt_cov, s.P * 9, ctx->stream);
	SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	return SPP_OK;
}

int spp_ba_marginals_sparse(spp_ctx_t ctx, double alpha, double *p_cam_cov, double *p_pt_cov)
{
	int rc = SPP_OK;
	API_BEGIN(ctx)
	if(!ctx->ba.valid) throw invalid_error("no BA graph");
	if(!ctx->ba.linearised) ba_linearise(ctx, true);
	rc = marginals_sparse_to_host(ctx, alpha, p_cam_cov, p_pt_cov);
	if(rc != SPP_OK) return rc;
	API_END(ctx)
}

int spp_schur_marginals_sparse(spp_ctx_t ctx, double alpha, double *p_cam_cov, double *p_pt_cov)
{
	int rc = SPP_OK;
	API_BEGIN(ctx)
	if(!ctx->slot.valid || !ctx->slot.filled) throw invalid_error("no system: spp_schur_symbolic and spp_schur_solve first");
	rc = marginals_sparse_to_host(ctx, alpha, p_cam_cov, p_pt_cov);
	if(rc != SPP_OK) return rc;
	API_END(ctx)
}

// SPP_MARGINALS_TIMING: the phases of a covariance-blocks call to stderr (ms[8] as schur_covariance_blocks_current fills it)
static void print_covariance_timing(bool sparse, const float *ms, size_t n_pairs, size_t n_obs, double ms_check, double ms_copy,
	double copy_gb)
{
	if(sparse)
		fprintf(stderr, "[spp covariance blocks] supernodal path %.3f ms: schur %.3f ms, factor %.3f ms, selected inversion %.3f ms, "
			"cameras %.3f ms, points %.3f ms;", ms[7], ms[0], ms[1], ms[2], ms[3], ms[4]);
	else
		fprintf(stderr, "[spp covariance blocks] dense path %.3f ms (schur, inverse, block diagonal);", ms[7]);
	fprintf(stderr, " pairs %.3f ms (%zu), observations %.3f ms (%zu); pattern check %.3f ms, copy to host %.3f ms (%.3f GB)\n",
		ms[5], n_pairs, ms[6], n_obs, ms_check, ms_copy, copy_gb);
}

// selected blocks of the covariance of the system held as (U, V, W) to host arrays; the path as the solver mode selects
static int covariance_blocks_to_host(spp_ctx *ctx, double alpha, size_t n_pairs, const uint64_t *p_cam_a, const uint64_t *p_cam_b,
	double *p_pair_cov, size_t n_obs, const uint64_t *p_obs, double *p_obs_cov, double *p_cam_cov, double *p_pt_cov)
{
	SchurSystem &s = ctx->sys;
	if(ctx->world > 1) throw invalid_error("covariance blocks are not available on a landmark-partitioned (multi-GPU) context");
	if(!s.C) throw invalid_error("no cameras");
	if(n_pairs && (!p_cam_a || !p_cam_b || !p_pair_cov)) throw invalid_error("camera pairs requested without their arrays");
	if(n_obs && (!p_obs || !p_obs_cov)) throw invalid_error("observations requested without their arrays");
	static const bool timing = getenv("SPP_MARGINALS_TIMING") != 0;
	auto t0 = std::chrono::steady_clock::now();
	// the sparse accessor finds a block by a binary search in the pattern of S: only covisible or equal pairs are valid
	std::vector<uint32_t> cam_a(n_pairs), cam_b(n_pairs), obs(n_obs);
	std::vector<uint64_t> want; // off-diagonal pairs as lo * C + hi, sorted, unique
	for(size_t k = 0; k < n_pairs; ++ k) {
		if(p_cam_a[k] >= s.C || p_cam_b[k] >= s.C) throw invalid_error("camera index out of range");
		cam_a[k] = (uint32_t)p_cam_a[k];
		cam_b[k] = (uint32_t)p_cam_b[k];
		if(cam_a[k] != cam_b[k])
			want.push_back((uint64_t)std::min(cam_a[k], cam_b[k]) * s.C + std::max(cam_a[k], cam_b[k]));
	}
	for(size_t k = 0; k < n_obs; ++ k) {
		if(p_obs[k] >= s.O) throw invalid_error("observation index out of range");
		obs[k] = (uint32_t)p_obs[k];
	}
	if(!want.empty()) {
		std::sort(want.begin(), want.end());
		want.erase(std::unique(want.begin(), want.end()), want.end());
		schur_fetch_host_pattern(ctx);
		std::vector<char> found(want.size(), 0);
		for(size_t b = 0; b < s.n_blocks; ++ b) {
			const uint64_t key = (uint64_t)s.h_blk_row[b] * s.C + s.h_blk_col[b]; // upper blocks: row <= col
			auto it = std::lower_bound(want.begin(), want.end(), key);
			if(it != want.end() && *it == key) found[it - want.begin()] = 1;
		}
		for(size_t i = 0; i < want.size(); ++ i)
			if(!found[i])
				throw invalid_error("camera pair (" + std::to_string(want[i] / s.C) + ", " + std::to_string(want[i] % s.C) +
					") shares no landmark: its covariance block is not on the pattern of the reduced camera system");
	}
	const double ms_check = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
	cudaStream_t st = ctx->stream;
	s.cov_cam_a.upload(cam_a, st);
	s.cov_cam_b.upload(cam_b, st);
	s.cov_obs_idx.upload(obs, st);
	if(p_cam_cov) s.cov_cam.resize(s.C * 36);
	if(p_pt_cov) s.cov_pt.resize(s.P * 9);
	s.cov_pair.resize(n_pairs * 36);
	s.cov_obs.resize(n_obs * 18);
	const bool sparse = rcs_is_sparse(ctx, s.C);
	float ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};
	int rc = schur_covariance_blocks_current(ctx, alpha, sparse, p_cam_cov? s.cov_cam.p() : 0, p_pt_cov? s.cov_pt.p() : 0, n_pairs,
		s.cov_cam_a.p(), s.cov_cam_b.p(), s.cov_pair.p(), n_obs, s.cov_obs_idx.p(), s.cov_obs.p(), timing? ms : 0);
	if(rc != SPP_OK)
		return rc;
	t0 = std::chrono::steady_clock::now();
	if(p_cam_cov) s.cov_cam.download(p_cam_cov, s.C * 36, st);
	if(p_pt_cov) s.cov_pt.download(p_pt_cov, s.P * 9, st);
	s.cov_pair.download(p_pair_cov, n_pairs * 36, st);
	s.cov_obs.download(p_obs_cov, n_obs * 18, st);
	SPP_CUDA(cudaStreamSynchronize(st));
	if(timing)
		print_covariance_timing(sparse, ms, n_pairs, n_obs, ms_check,
			std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(),
			8e-9 * ((p_cam_cov? s.C * 36 : 0) + (p_pt_cov? s.P * 9 : 0) + n_pairs * 36 + n_obs * 18));
	return SPP_OK;
}

int spp_ba_covariance_blocks(spp_ctx_t ctx, double alpha, size_t n_pairs, const uint64_t *p_cam_a, const uint64_t *p_cam_b,
	double *p_pair_cov, size_t n_obs, const uint64_t *p_obs, double *p_obs_cov, double *p_cam_cov, double *p_pt_cov)
{
	int rc = SPP_OK;
	API_BEGIN(ctx)
	if(!ctx->ba.valid) throw invalid_error("no BA graph");
	if(!ctx->ba.linearised) ba_linearise(ctx, true);
	rc = covariance_blocks_to_host(ctx, alpha, n_pairs, p_cam_a, p_cam_b, p_pair_cov, n_obs, p_obs, p_obs_cov, p_cam_cov, p_pt_cov);
	if(rc != SPP_OK) return rc;
	API_END(ctx)
}

int spp_schur_covariance_pattern(spp_ctx_t ctx, double alpha, double *p_cov_values)
{
	int rc = SPP_OK;
	API_BEGIN(ctx)
	SchurSlot &sl = ctx->slot;
	SchurSystem &s = ctx->sys;
	if(!sl.valid || !sl.filled) throw invalid_error("no system: spp_schur_symbolic and spp_schur_solve first");
	if(!p_cov_values) throw invalid_error("null argument");
	if(ctx->world > 1) throw invalid_error("covariance blocks are not available on a landmark-partitioned (multi-GPU) context");
	static const bool timing = getenv("SPP_MARGINALS_TIMING") != 0;
	const bool sparse = rcs_is_sparse(ctx, s.C);
	float ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};
	rc = slot_covariance_pattern(ctx, alpha, sparse, sl.vals.p(), timing? ms : 0); // the staged lambda is not needed again
	if(rc != SPP_OK) return rc;
	const auto t0 = std::chrono::steady_clock::now();
	SPP_CUDA(cudaMemcpyAsync(p_cov_values, sl.vals.p(), sl.n_values * 8, cudaMemcpyDeviceToHost, ctx->stream));
	SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	if(timing)
		print_covariance_timing(sparse, ms, 0, s.O, 0, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(),
			sl.n_values * 8e-9);
	API_END(ctx)
}

// joint marginals: sets of vertices, each already mapped to (landmark ? 1 << 31 : 0) | local index << 3; checks the sets
// and runs on the path the solver mode selects
static int joint_marginals_checked(spp_ctx *ctx, double alpha, size_t n_sets, const uint64_t *p_set_ptr,
	const std::vector<uint32_t> &verts, double *p_cov)
{
	SchurSystem &s = ctx->sys;
	if(ctx->world > 1) throw invalid_error("joint marginals are not available on a landmark-partitioned (multi-GPU) context");
	if(!s.C) throw invalid_error("no cameras");
	std::vector<uint64_t> set_ptr(p_set_ptr, p_set_ptr + n_sets + 1);
	for(size_t k = 0; k < n_sets; ++ k) {
		if(set_ptr[k + 1] <= set_ptr[k]) throw invalid_error("joint marginals: set " + std::to_string(k) + " is empty");
		uint64_t D = 0;
		for(uint64_t q = set_ptr[k]; q < set_ptr[k + 1]; ++ q) D += (verts[q] & 0x80000000u)? 3 : 6;
		if(D > 16384) throw invalid_error("joint marginals: set " + std::to_string(k) + " is wider than 16384 columns");
	}
	if(!n_sets) return SPP_OK;
	static const bool timing = getenv("SPP_MARGINALS_TIMING") != 0;
	return joint_marginals_to_host(ctx, alpha, rcs_is_sparse(ctx, s.C), set_ptr, verts, p_cov, timing);
}

static void joint_check_args(size_t n_sets, const uint64_t *p_set_ptr, const uint64_t *p_ids, double *p_cov)
{
	if(n_sets && (!p_set_ptr || !p_ids || !p_cov)) throw invalid_error("null argument");
	if(p_set_ptr && p_set_ptr[0] != 0) throw invalid_error("joint marginals: p_set_ptr[0] must be 0");
	for(size_t k = 0; k < n_sets; ++ k)
		if(p_set_ptr[k + 1] < p_set_ptr[k]) throw invalid_error("joint marginals: p_set_ptr must not decrease");
}

int spp_ba_joint_marginals(spp_ctx_t ctx, double alpha, size_t n_sets, const uint64_t *p_set_ptr, const uint64_t *p_vertices,
	double *p_cov)
{
	int rc = SPP_OK;
	API_BEGIN(ctx)
	BAProblem &ba = ctx->ba;
	if(!ba.valid) throw invalid_error("no BA graph");
	joint_check_args(n_sets, p_set_ptr, p_vertices, p_cov);
	const size_t n_ids = n_sets? p_set_ptr[n_sets] : 0;
	std::vector<uint32_t> verts(n_ids);
	for(size_t q = 0; q < n_ids; ++ q) {
		const uint64_t v = p_vertices[q];
		if(v >= ba.n_vertices) throw invalid_error("joint marginals: vertex id " + std::to_string(v) + " out of range");
		verts[q] = ((ba.vtype[v] == 0)? 0u : 0x80000000u) | (ba.vertex_local[v] << 3);
	}
	if(ctx->world > 1) throw invalid_error("joint marginals are not available on a landmark-partitioned (multi-GPU) context");
	if(!ba.linearised) ba_linearise(ctx, true);
	rc = joint_marginals_checked(ctx, alpha, n_sets, p_set_ptr, verts, p_cov);
	if(rc != SPP_OK) return rc;
	API_END(ctx)
}

int spp_schur_joint_marginals(spp_ctx_t ctx, double alpha, size_t n_sets, const uint64_t *p_set_ptr, const uint64_t *p_block_cols,
	double *p_cov)
{
	int rc = SPP_OK;
	API_BEGIN(ctx)
	SchurSlot &sl = ctx->slot;
	if(!sl.valid || !sl.filled) throw invalid_error("no system: spp_schur_symbolic and spp_schur_solve first");
	joint_check_args(n_sets, p_set_ptr, p_block_cols, p_cov);
	std::vector<uint32_t> new_pos(sl.n_bcols);
	for(size_t i = 0; i < sl.n_bcols; ++ i) new_pos[sl.order[i]] = (uint32_t)i;
	const size_t n_ids = n_sets? p_set_ptr[n_sets] : 0;
	std::vector<uint32_t> verts(n_ids);
	for(size_t q = 0; q < n_ids; ++ q) {
		const uint64_t b = p_block_cols[q];
		if(b >= sl.n_bcols) throw invalid_error("joint marginals: block column " + std::to_string(b) + " out of range");
		const uint32_t p = new_pos[b];
		verts[q] = (p < sl.cut)? (p << 3) : (0x80000000u | ((uint32_t)(p - sl.cut) << 3));
	}
	rc = joint_marginals_checked(ctx, alpha, n_sets, p_set_ptr, verts, p_cov);
	if(rc != SPP_OK) return rc;
	API_END(ctx)
}

int spp_ba_optimize(spp_ctx_t ctx, size_t n_max_iterations, double f_min_dx_norm, spp_report_t *p_report)
{
	API_BEGIN(ctx)
	if(!ctx->ba.valid) throw invalid_error("no BA graph");
	spp_report_t local;
	ba_optimize(ctx, n_max_iterations, f_min_dx_norm, p_report? p_report : &local);
	API_END(ctx)
}

int spp_schur_symbolic(spp_ctx_t ctx, size_t n_block_cols, const uint64_t *p_col_dims, const uint64_t *p_col_ptr,
	const uint64_t *p_row_idx, uint64_t *p_order, uint64_t *p_cut)
{
	API_BEGIN(ctx)
	if(!n_block_cols || !p_col_dims || !p_col_ptr || !p_row_idx) throw invalid_error("null argument");
	ctx->snode.valid = false;
	ctx->sys.n_blocks_global = 0;
	slot_symbolic(ctx, n_block_cols, p_col_dims, p_col_ptr, p_row_idx, p_order, p_cut);
	API_END(ctx)
}

int spp_schur_solve(spp_ctx_t ctx, const double *p_values, double *p_eta_dx)
{
	int rc = SPP_OK;
	API_BEGIN(ctx)
	if(!p_values || !p_eta_dx) throw invalid_error("null argument");
	rc = slot_solve(ctx, p_values, p_eta_dx);
	if(rc != SPP_OK) return rc;
	API_END(ctx)
}

int spp_schur_get_reduced_system(spp_ctx_t ctx, uint64_t *p_n, double *p_S, double *p_rhs, uint8_t *p_block_pattern)
{
	API_BEGIN(ctx)
	SchurSystem &s = ctx->sys;
	const size_t n = s.C * 6;
	if(p_n) *p_n = n;
	if(p_S || p_rhs) {
		if(!s.keep_reduced || s.S_copy.size() == 0)
			throw invalid_error("no reduced system kept: solve first (the context keeps a copy after the first query; no dense "
				"copy is taken of a block-sparse system with more than 32768 unknowns or on several ranks)");
		const size_t ld = dense_chol_ld(n);
		if(p_S)
			SPP_CUDA(cudaMemcpy2DAsync(p_S, n * 8, s.S_copy.p(), ld * 8, n * 8, n, cudaMemcpyDeviceToHost, ctx->stream));
		if(p_rhs)
			s.b_copy.download(p_rhs, n, ctx->stream);
		SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	}
	if(p_block_pattern) {
		schur_fetch_host_pattern(ctx);
		memset(p_block_pattern, 0, s.C * s.C);
		for(size_t i = 0; i < s.h_blk_row.size(); ++ i)
			p_block_pattern[(size_t)s.h_blk_row[i] * s.C + s.h_blk_col[i]] = 1;
	}
	if(p_S || p_rhs || !p_block_pattern)
		s.keep_reduced = true; // a pattern-only query does not make the following solves keep a dense copy
	API_END(ctx)
}

int spp_schur_set_rcs_solver(spp_ctx_t ctx, int mode)
{
	API_BEGIN(ctx)
	if(mode != SPP_RCS_AUTO && mode != SPP_RCS_DENSE && mode != SPP_RCS_SPARSE) throw invalid_error("unknown reduced-camera-system solver");
	ctx->snode.mode = mode;
	API_END(ctx)
}

int spp_schur_set_rcs_ordering(spp_ctx_t ctx, size_t n_cameras, const uint64_t *p_order)
{
	API_BEGIN(ctx)
	SupernodalChol &sc = ctx->snode;
	sc.valid = false;
	sc.user_order.clear();
	if(p_order) {
		std::vector<char> seen(n_cameras, 0);
		for(size_t i = 0; i < n_cameras; ++ i) {
			if(p_order[i] >= n_cameras || seen[p_order[i]]) throw invalid_error("the ordering is not a permutation");
			seen[p_order[i]] = 1;
		}
		sc.user_order.assign(p_order, p_order + n_cameras);
	}
	API_END(ctx)
}

int spp_schur_get_rcs_info(spp_ctx_t ctx, uint64_t *p_order, double *p_stats)
{
	API_BEGIN(ctx)
	SupernodalChol &sc = ctx->snode;
	if(!sc.valid) throw invalid_error("no block-sparse factorisation of a reduced camera system yet");
	if(p_order)
		for(size_t i = 0; i < sc.n; ++ i) p_order[i] = sc.h_order[i];
	if(p_stats) {
		p_stats[0] = (double)sc.n;
		p_stats[1] = (double)sc.n_s_blocks;
		p_stats[2] = (double)sc.sn.n_super();
		p_stats[3] = (double)sc.sn.nnzb_exact;
		p_stats[4] = (double)sc.sn.nnzb_factor;
		p_stats[5] = sc.factor_flops;
		p_stats[6] = (double)sc.d_L.size() * 8.0;
		p_stats[7] = (double)sc.updates.size();
	}
	API_END(ctx)
}

int spp_schur_get_rcs_owners(spp_ctx_t ctx, int32_t *p_owner)
{
	API_BEGIN(ctx)
	SupernodalChol &sc = ctx->snode;
	if(!sc.valid) throw invalid_error("no block-sparse factorisation of a reduced camera system yet");
	if(!p_owner) throw invalid_error("null argument");
	for(size_t s = 0, ns = sc.sn.n_super(); s < ns; ++ s)
		p_owner[s] = (s < sc.owner.size())? sc.owner[s] : -1;
	API_END(ctx)
}

int spp_schur_get_rcs_residual(spp_ctx_t ctx, double *p_relative_residual)
{
	API_BEGIN(ctx)
	SchurSystem &s = ctx->sys;
	if(!p_relative_residual) throw invalid_error("null argument");
	if(!s.sparse_solved) throw invalid_error("no successful solve on the block-sparse path to check");
	const size_t n = s.C * 6, nb = s.n_blocks_global? s.n_blocks_global : s.n_blocks;
	const uint32_t *rows = s.n_blocks_global? s.gblk_row.p() : s.blk_row.p(), *cols = s.n_blocks_global? s.gblk_col.p() : s.blk_col.p();
	DBuf<double> r, out;
	r.resize(n);
	out.resize(2);
	r.zero(ctx->stream);
	k_blocks_symv<<<n_blocks(nb * 36, 256), 256, 0, ctx->stream>>>(nb * 36, s.Sblk.p(), rows, cols, s.dxc.p(), r.p());
	k_residual_norms<<<1, 256, 0, ctx->stream>>>(n, r.p(), s.b_copy.p(), out.p());
	ctx->n_launches += 2;
	SPP_CUDA(cudaGetLastError());
	double h[2];
	out.download(h, 2, ctx->stream);
	SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	*p_relative_residual = (h[1] > 0)? sqrt(h[0] / h[1]) : sqrt(h[0]);
	API_END(ctx)
}

int spp_dense_panel_factor(spp_ctx_t ctx, size_t n_rows, size_t n_cols, double *p_panel)
{
	int rc = SPP_OK;
	API_BEGIN(ctx)
	if(!n_rows || n_rows % 128 || n_cols % 128 || n_cols < n_rows || !p_panel) throw invalid_error("bad panel shape");
	DBuf<double> A, Rinv;
	DBuf<int> info;
	A.upload(p_panel, n_rows * n_cols, ctx->stream);
	Rinv.resize((n_rows / 128) * 128 * 128);
	Rinv.zero(ctx->stream);
	info.resize(1);
	info.zero(ctx->stream);
	if(dense_chol_dataflow_enabled())
		dense_chol_factor_dataflow(ctx, A.p(), n_rows, n_cols, Rinv.p(), info.p());
	else
		dense_chol_factor_panel(ctx, A.p(), n_rows, n_cols, Rinv.p(), info.p(), false);
	int h_info = 0;
	SPP_CUDA(cudaMemcpyAsync(&h_info, info.p(), sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
	A.download(p_panel, n_rows * n_cols, ctx->stream);
	SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	if(h_info < 0) throw cuda_error("dense panel factorisation: the dataflow kernel's watchdog fired");
	rc = h_info? SPP_NOT_POSDEF : SPP_OK;
	if(rc != SPP_OK) return rc;
	API_END(ctx)
}

int spp_dense_posdef_solve(spp_ctx_t ctx, size_t n, const double *p_A, double *p_rhs_x)
{
	int rc = SPP_OK;
	API_BEGIN(ctx)
	if(!n || !p_A || !p_rhs_x) throw invalid_error("null argument");
	const size_t ld = dense_chol_ld(n);
	DBuf<double> A, b;
	A.resize(dense_chol_storage(n));
	A.zero(ctx->stream);
	b.upload(p_rhs_x, n, ctx->stream);
	SPP_CUDA(cudaMemcpy2DAsync(A.p(), ld * 8, p_A, n * 8, n * 8, n, cudaMemcpyHostToDevice, ctx->stream));
	rc = dense_chol_solve_device(ctx, A.p(), n, b.p());
	b.download(p_rhs_x, n, ctx->stream);
	SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	if(rc != SPP_OK) return rc;
	API_END(ctx)
}

// ---- block-sparse Cholesky slot ---------------------------------------------------------------------

int spp_chol_symbolic(spp_ctx_t ctx, size_t n_block_cols, size_t block_size, const uint64_t *p_col_ptr,
	const uint64_t *p_row_idx, const uint64_t *p_order_in, uint64_t *p_order_out)
{
	API_BEGIN(ctx)
	if(!n_block_cols || !p_col_ptr || !p_row_idx) throw invalid_error("null argument");
	if(block_size != 2 && block_size != 3 && block_size != 6) throw invalid_error("block size must be 2, 3 or 6");
	sparse_chol_symbolic(ctx, SC_OWNER_SLOT, n_block_cols, block_size, p_col_ptr, p_row_idx, p_order_in);
	if(p_order_out)
		for(size_t i = 0; i < n_block_cols; ++ i) p_order_out[i] = ctx->schol.h_order[i];
	API_END(ctx)
}

int spp_chol_solve(spp_ctx_t ctx, const double *p_values, double *p_eta_dx)
{
	int rc = SPP_OK;
	API_BEGIN(ctx)
	SparseChol &sc = ctx->schol;
	if(!sc.valid) throw invalid_error("spp_chol_symbolic() has not been called");
	// the slot does not keep its structure: after a pose solve, the analysis in memory is the pose graph's
	if(sc.owner != SC_OWNER_SLOT) throw invalid_error("the block-sparse analysis in use is the pose graph's: call spp_chol_symbolic again");
	if(!p_values || !p_eta_dx) throw invalid_error("null argument");
	const size_t nv = sc.n_a_blocks * sc.B * sc.B, ns = sc.n * sc.B;
	sc.slot_vals.upload(p_values, nv, ctx->stream);
	sc.slot_rhs.upload(p_eta_dx, ns, ctx->stream);
	sc.slot_x.resize(ns);
	rc = sparse_chol_solve_device(ctx, sc.slot_vals.p(), sc.slot_rhs.p(), sc.slot_x.p());
	sc.slot_x.download(p_eta_dx, ns, ctx->stream);
	SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	if(rc != SPP_OK) return rc;
	API_END(ctx)
}

int spp_chol_get_factor(spp_ctx_t ctx, uint64_t *p_n_blocks, uint64_t *p_col_ptr, uint64_t *p_row_idx, double *p_values)
{
	API_BEGIN(ctx)
	SparseChol &sc = ctx->schol;
	if(!sc.valid) throw invalid_error("no block-sparse factorisation");
	const size_t n = sc.n, BB = sc.B * sc.B, B = sc.B, nb = sc.n_l_blocks;
	if(p_n_blocks) *p_n_blocks = nb;
	if(p_col_ptr || p_row_idx || p_values) {
		// L is stored by columns (rows >= column); R = L^T by columns = L by rows
		std::vector<uint64_t> cnt(n + 1, 0);
		for(size_t j = 0; j < n; ++ j)
			for(uint64_t b = sc.h_lptr[j]; b < sc.h_lptr[j + 1]; ++ b)
				++ cnt[sc.h_lrow[b] + 1];
		for(size_t j = 0; j < n; ++ j) cnt[j + 1] += cnt[j];
		if(p_col_ptr) std::copy(cnt.begin(), cnt.end(), p_col_ptr);
		std::vector<double> hL;
		if(p_values) {
			hL.resize(nb * BB);
			sc.d_L.download(hL.data(), nb * BB, ctx->stream);
			SPP_CUDA(cudaStreamSynchronize(ctx->stream));
			if(sc.n_root) { // the blocks of the dense root front live in the dense factor (upper, column-major)
				const size_t nd = sc.n_root * B, ld = dense_chol_ld(nd);
				std::vector<double> hS(ld * nd);
				sc.d_root_S.download(hS.data(), ld * nd, ctx->stream);
				SPP_CUDA(cudaStreamSynchronize(ctx->stream));
				for(size_t j = 0; j < n; ++ j) {
					if(sc.h_ridx[j] == 0xffffffffu)
						continue;
					const size_t rj = sc.h_ridx[j];
					for(uint64_t b = sc.h_lptr[j]; b < sc.h_lptr[j + 1]; ++ b) {
						const size_t i = sc.h_lrow[b], ri = sc.h_ridx[i];
						for(size_t c = 0; c < B; ++ c)
							for(size_t r = 0; r < B; ++ r) // L(i, j)(r, c) = R(rj B + c, ri B + r)
								hL[b * BB + c * B + r] = (i > j || r >= c)? hS[(ri * B + r) * ld + rj * B + c] : 0.0;
					}
				}
			}
		}
		std::vector<uint64_t> fill(cnt.begin(), cnt.end() - 1);
		for(size_t j = 0; j < n; ++ j) { // ascending j = ascending row of R inside every column
			for(uint64_t b = sc.h_lptr[j]; b < sc.h_lptr[j + 1]; ++ b) {
				const uint64_t dst = fill[sc.h_lrow[b]] ++;
				if(p_row_idx) p_row_idx[dst] = j;
				if(p_values)
					for(size_t c = 0; c < B; ++ c)
						for(size_t r = 0; r < B; ++ r)
							p_values[dst * BB + c * B + r] = hL[b * BB + r * B + c]; // R(j, i) = L(i, j)^T
			}
		}
	}
	API_END(ctx)
}

// ---- pose graphs ---------------------------------------------------------------------------------------

int spp_pose_set_graph(spp_ctx_t ctx, int dim, size_t n_poses, const double *p_states, size_t n_edges,
	const uint64_t *p_from, const uint64_t *p_to, const double *p_z, const double *p_info)
{
	API_BEGIN(ctx)
	if((n_poses && !p_states) || (n_edges && (!p_from || !p_to || !p_z || !p_info))) throw invalid_error("null argument");
	ctx->pose.h_order_in.clear();
	pose_set_graph(ctx, dim, n_poses, p_states, n_edges, p_from, p_to, p_z, p_info);
	API_END(ctx)
}

int spp_pose_set_ordering(spp_ctx_t ctx, const uint64_t *p_order)
{
	API_BEGIN(ctx)
	PoseProblem &pp = ctx->pose;
	if(!pp.valid) throw invalid_error("no pose graph");
	if(p_order) pp.h_order_in.assign(p_order, p_order + pp.N);
	else pp.h_order_in.clear();
	pp.symbolic_done = false;
	API_END(ctx)
}

int spp_pose_set_states(spp_ctx_t ctx, const double *p_states)
{
	API_BEGIN(ctx)
	PoseProblem &pp = ctx->pose;
	if(!pp.valid || !p_states) throw invalid_error("no pose graph");
	SPP_CUDA(cudaMemcpyAsync(pp.states.p(), p_states, pp.N * pp.dim * 8, cudaMemcpyHostToDevice, ctx->stream));
	SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	pp.linearised = false;
	API_END(ctx)
}

int spp_pose_get_states(spp_ctx_t ctx, double *p_states)
{
	API_BEGIN(ctx)
	PoseProblem &pp = ctx->pose;
	if(!pp.valid || !p_states) throw invalid_error("no pose graph");
	pp.states.download(p_states, pp.N * pp.dim, ctx->stream);
	SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	API_END(ctx)
}

int spp_pose_restore_initial(spp_ctx_t ctx)
{
	API_BEGIN(ctx)
	PoseProblem &pp = ctx->pose;
	if(!pp.valid) throw invalid_error("no pose graph");
	SPP_CUDA(cudaMemcpyAsync(pp.states.p(), pp.states0.p(), pp.N * pp.dim * 8, cudaMemcpyDeviceToDevice, ctx->stream));
	pp.linearised = false;
	API_END(ctx)
}

int spp_pose_linearise(spp_ctx_t ctx)
{
	API_BEGIN(ctx)
	if(!ctx->pose.valid) throw invalid_error("no pose graph");
	pose_linearise(ctx);
	SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	API_END(ctx)
}

int spp_pose_get_lambda(spp_ctx_t ctx, uint64_t *p_n_block_cols, uint64_t *p_n_blocks, uint64_t *p_col_ptr,
	uint64_t *p_row_idx, double *p_values, double *p_eta)
{
	API_BEGIN(ctx)
	PoseProblem &pp = ctx->pose;
	if(!pp.valid) throw invalid_error("no pose graph");
	if(p_n_block_cols) *p_n_block_cols = pp.N;
	if(p_n_blocks) *p_n_blocks = pp.n_blocks;
	if(p_col_ptr) std::copy(pp.h_col_ptr.begin(), pp.h_col_ptr.end(), p_col_ptr);
	if(p_row_idx) std::copy(pp.h_row_idx.begin(), pp.h_row_idx.end(), p_row_idx);
	if(p_values || p_eta) {
		if(!pp.linearised) throw invalid_error("spp_pose_linearise() has not been called");
		if(p_values) pp.vals.download(p_values, pp.n_blocks * pp.dim * pp.dim, ctx->stream);
		if(p_eta) pp.eta.download(p_eta, pp.N * pp.dim, ctx->stream);
		SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	}
	API_END(ctx)
}

int spp_pose_chi2(spp_ctx_t ctx, double *p_chi2)
{
	API_BEGIN(ctx)
	if(!ctx->pose.valid || !p_chi2) throw invalid_error("no pose graph");
	*p_chi2 = pose_chi2(ctx);
	API_END(ctx)
}

int spp_pose_solve_step(spp_ctx_t ctx, double *p_dx)
{
	int rc = SPP_OK;
	API_BEGIN(ctx)
	PoseProblem &pp = ctx->pose;
	if(!pp.valid) throw invalid_error("no pose graph");
	if(!pp.linearised) pose_linearise(ctx);
	rc = pose_solve(ctx);
	if(rc == SPP_OK && p_dx) {
		pp.dx.download(p_dx, pp.N * pp.dim, ctx->stream);
		SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	}
	if(rc != SPP_OK) return rc;
	API_END(ctx)
}

int spp_pose_marginals(spp_ctx_t ctx, double *p_cov)
{
	int rc = SPP_OK;
	API_BEGIN(ctx)
	PoseProblem &pp = ctx->pose;
	if(!pp.valid) throw invalid_error("no pose graph");
	if(!p_cov) throw invalid_error("null argument");
	if(pp.N * pp.dim > 16384) throw invalid_error("pose marginals go through a dense inverse: at most 16384 unknowns");
	if(!pp.linearised) pose_linearise(ctx);
	DBuf<double> &d_cov = ctx->sys.cov_cam;
	d_cov.resize(pp.N * pp.dim * pp.dim);
	rc = pose_marginals(ctx, d_cov.p());
	if(rc != SPP_OK) return rc;
	d_cov.download(p_cov, pp.N * pp.dim * pp.dim, ctx->stream);
	SPP_CUDA(cudaStreamSynchronize(ctx->stream));
	API_END(ctx)
}

int spp_pose_optimize(spp_ctx_t ctx, size_t n_max_iterations, double f_min_dx_norm, spp_report_t *p_report)
{
	API_BEGIN(ctx)
	if(!ctx->pose.valid) throw invalid_error("no pose graph");
	spp_report_t local;
	pose_optimize(ctx, n_max_iterations, f_min_dx_norm, p_report? p_report : &local);
	API_END(ctx)
}

} // extern "C"
