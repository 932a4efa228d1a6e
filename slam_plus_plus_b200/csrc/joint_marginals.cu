// joint_marginals.cu -- joint marginal covariance of any set of bundle-adjustment vertices, on or off the block pattern of
// the reduced camera system, by multi-column forward solves on its Cholesky factor.
//
// In Schur order (lambda + alpha I) = [[U + alpha I, W], [W^T, V + alpha I]]; with C_p = V_p + alpha I, Y_a = W_a C_p^-1
// and S = U + alpha I - sum W C^-1 W^T, P S P^T = R^T R. Every vertex v gets a right-hand-side block b_v (6C x d_v):
//     camera i:   b_i = E_i                                  (its unit columns)
//     landmark p: b_p = -sum_{a in track(p)} E_{c_a} Y_a
// and for any two vertices
//     Sigma_uv = [u = v is a landmark] C_v^-1 + F_u^T F_v,     F_v = R^-T P b_v      (forward solve only)
// which reproduces Z = S^-1 on the camera blocks, -sum Z Y on the camera-landmark blocks and C^-1 + sum Y^T Z Y on the
// landmark blocks (marginals.cu), and gives every block off the pattern of S as well. This is the reference's own way to
// the landmark marginals (R^-T U D^-1, include/slam/BAMarginals.h:671-699) applied to any set of vertices, batched.
//
// F_v is structurally non-zero only on the reach of v: the supernodes that are ancestors-or-self, in the supernodal
// elimination tree, of the supernodes that hold its cameras. A batch of right-hand-side columns lives in a compact
// buffer that holds only the rows of the batch's reach (every supernode's own columns, padded to its panel's ld, in
// elimination order). Per reach supernode s, in elimination order, on one stream:
//     F_s = R11^-T B_s                 128-row block substitution with the diagonal-block inverses Rinv of the factor
//     B[rows of J] -= R12^T F_s        one GEMM, K = w, whose epilogue subtracts through the structure rows
// then per set K the Gram F_K^T F_K over the set's own reach rows (plus C_p^-1 on landmark diagonal blocks). All products
// are FP64 tensor-core GEMMs (mma.sync m8n8k4) of one kernel, k_joint_gemm.
//
// Determinism: a column of the forward solve depends on its own right-hand side only (every sum runs over k in a fixed
// order), and a column is exactly zero on the supernodes of the batch outside its own reach, so it gets the same bits in
// any batch. The Gram of a set sums over the rows of its own reach supernodes, segment by segment in elimination order,
// so its K-grouping is fixed by the set alone. Only the upper triangle is computed; the lower one is its exact
// transpose. No atomics.
//
// The dense reduced camera system is the case of one supernode (w = n, no structure).

#include "spp_ctx.h"
#include <cuda_pipeline_primitives.h>
#include <algorithm>
#include <chrono>
#include <stdlib.h>

namespace spp {

size_t dense_chol_ld(size_t n);
size_t dense_chol_storage(size_t n);
void schur_form_reduced_system(spp_ctx *ctx, double alpha, double alpha_diag, bool sparse_rcs);
void schur_fetch_host_pattern(spp_ctx *ctx);
void snode_symbolic(spp_ctx *ctx, size_t n, const std::vector<uint32_t> &blk_row, const std::vector<uint32_t> &blk_col);
void snode_factor(spp_ctx *ctx, const double *d_Sblk, const double *d_b);
void dense_chol_factor_panel(spp_ctx *ctx, double *A, size_t ld, size_t n_cols, double *Rinv, int *info, bool identity_tail);
void dense_chol_factor_dataflow(spp_ctx *ctx, double *A, size_t ld, size_t n_cols, double *Rinv, int *info);
bool dense_chol_dataflow_enabled();

#define LAUNCH_CHECK(ctx) do { ++ (ctx)->n_launches; SPP_CUDA(cudaGetLastError()); } while(0)

#define JM_NB 128   // panel granularity (= SN_NB of supernodal_chol.cu, CH_NB of dense_chol.cu)
#define JM_BM 128
#define JM_BN 64
#define JM_BK 16
#define JM_LDS (JM_BK + 4)
#define JM_STAGES 3
#define JM_THREADS 256

static const double JM_BUDGET_BYTES = 4e9; // device memory of the compact F of one batch (reach rows x batch columns)

enum { JM_SUB = 1 /* C -= A B (else C = A B) */, JM_A_LOWER = 2 /* A(i, k) = 0 for k > i */, JM_UPPER = 4 /* upper tiles only */ };

// C(i, j) = [C(i, j) -] sum_k A(i, k) B(k, j), i < M, j < N, K = 16 n_kt; A and B both k-contiguous:
//     A(i, k) = A[amap(i) lda + row(k)],  B(k, j) = B[bmap(j) ldb + row(k)],  C(i, j) = C[j ldc + crow(i)]
// amap / bmap: column lists (null: the identity); row(k) = kblk[k / 128] 128 + k % 128 (null: k); crow(i) =
// c_base[c_blk[i / 6]] + i % 6 (null: i).
struct JointGemm {
	const double *A, *B;
	double *C;
	const uint32_t *amap, *bmap, *kblk, *c_blk, *c_base;
	size_t lda, ldb, ldc;
	uint32_t M, N, n_kt;
	int flags;
};

__device__ __forceinline__ void dmma_jm(double &d0, double &d1, double a, double b)
{
	asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
		: "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

// Block tile 128 x 64, eight warps of 32 x 32, 3-stage cp.async pipeline over K; operand tiles [row][k] in shared memory
// with k padded by 4 (conflict-free fragment loads). Rows and columns past M / N load clamped operands and store nothing.
// MULTI: one problem per blockIdx.z from jobs (the Gram of many sets in one launch), else the problem g.
// In place (C = B) is allowed when M <= JM_BM: a CTA then owns its columns of C, and every read of B lands in shared
// memory before the epilogue.
template <bool MULTI>
__global__ void __launch_bounds__(JM_THREADS) k_joint_gemm(JointGemm g, const JointGemm *__restrict__ jobs)
{
	if(MULTI) g = jobs[blockIdx.z];
	const uint32_t i0 = blockIdx.y * JM_BM, j0 = blockIdx.x * JM_BN;
	if(i0 >= g.M || j0 >= g.N || ((g.flags & JM_UPPER) && i0 > j0 + (JM_BN - 1)))
		return;
	extern __shared__ double smem[];
	double (*As)[JM_BM][JM_LDS] = reinterpret_cast<double (*)[JM_BM][JM_LDS]>(smem);
	double (*Bs)[JM_BN][JM_LDS] = reinterpret_cast<double (*)[JM_BN][JM_LDS]>(smem + JM_STAGES * JM_BM * JM_LDS);
	const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
	const int wi = (warp >> 1) * 32, wj = (warp & 1) * 32;
	const int gq = lane >> 2, t = lane & 3;
	const double *A = g.A, *B = g.B;
	const size_t lda = g.lda, ldb = g.ldb;
	const uint32_t M = g.M, N = g.N;
	const uint32_t *amap = g.amap, *bmap = g.bmap, *kblk = g.kblk;

	auto stage_load = [&](int st, int kc) {
		const size_t r0 = kblk? (size_t)kblk[kc >> 3] * JM_NB + (kc & 7) * JM_BK : (size_t)kc * JM_BK;
		for(int idx = tid; idx < JM_BM * (JM_BK / 2); idx += JM_THREADS) {
			const int m = idx / (JM_BK / 2), q = idx % (JM_BK / 2);
			const uint32_t i = min(i0 + m, M - 1), c = amap? amap[i] : i;
			__pipeline_memcpy_async(&As[st][m][q * 2], A + (size_t)c * lda + r0 + q * 2, 16);
		}
		for(int idx = tid; idx < JM_BN * (JM_BK / 2); idx += JM_THREADS) {
			const int m = idx / (JM_BK / 2), q = idx % (JM_BK / 2);
			const uint32_t j = min(j0 + m, N - 1), c = bmap? bmap[j] : j;
			__pipeline_memcpy_async(&Bs[st][m][q * 2], B + (size_t)c * ldb + r0 + q * 2, 16);
		}
	};

	const int KT = (int)g.n_kt;
	#pragma unroll
	for(int s = 0; s < JM_STAGES - 1; ++ s) {
		if(s < KT) stage_load(s, s);
		__pipeline_commit();
	}
	const bool sub = (g.flags & JM_SUB) != 0, lower = (g.flags & JM_A_LOWER) != 0;
	uint32_t crow[4];
	#pragma unroll
	for(int a = 0; a < 4; ++ a) {
		const uint32_t i = i0 + wi + a * 8 + gq;
		crow[a] = (i >= M)? 0xffffffffu : g.c_blk? g.c_base[g.c_blk[i / 6]] + i % 6 : i;
	}
	// subtraction: the accumulators start from C and the A fragments are negated
	double acc[4][4][2];
	#pragma unroll
	for(int a = 0; a < 4; ++ a) {
		#pragma unroll
		for(int b = 0; b < 4; ++ b) {
			#pragma unroll
			for(int h = 0; h < 2; ++ h) {
				const uint32_t j = j0 + wj + b * 8 + 2 * t + h;
				acc[a][b][h] = (sub && crow[a] != 0xffffffffu && j < N)? g.C[(size_t)j * g.ldc + crow[a]] : 0.0;
			}
		}
	}
	for(int kt = 0; kt < KT; ++ kt) {
		__pipeline_wait_prior(JM_STAGES - 2);
		__syncthreads();
		if(kt + JM_STAGES - 1 < KT)
			stage_load((kt + JM_STAGES - 1) % JM_STAGES, kt + JM_STAGES - 1);
		__pipeline_commit();
		const int st = kt % JM_STAGES;
		#pragma unroll
		for(int k4 = 0; k4 < JM_BK; k4 += 4) {
			double fa[4], fb[4];
			#pragma unroll
			for(int a = 0; a < 4; ++ a) {
				const int m = wi + a * 8 + gq;
				double v = As[st][m][k4 + t];
				if(lower && kt * JM_BK + k4 + t > (int)i0 + m) v = 0;
				fa[a] = sub? -v : v;
			}
			#pragma unroll
			for(int b = 0; b < 4; ++ b)
				fb[b] = Bs[st][wj + b * 8 + gq][k4 + t];
			#pragma unroll
			for(int a = 0; a < 4; ++ a)
				#pragma unroll
				for(int b = 0; b < 4; ++ b)
					dmma_jm(acc[a][b][0], acc[a][b][1], fa[a], fb[b]);
		}
	}
	__pipeline_wait_prior(0);
	__syncthreads(); // in place: every read of B has landed before any store
	#pragma unroll
	for(int a = 0; a < 4; ++ a) {
		if(crow[a] == 0xffffffffu) continue;
		#pragma unroll
		for(int b = 0; b < 4; ++ b) {
			#pragma unroll
			for(int h = 0; h < 2; ++ h) {
				const uint32_t j = j0 + wj + b * 8 + 2 * t + h;
				if(j < N)
					g.C[(size_t)j * g.ldc + crow[a]] = acc[a][b][h];
			}
		}
	}
}

static size_t joint_gemm_smem() { return (size_t)JM_STAGES * (JM_BM + JM_BN) * JM_LDS * sizeof(double); }

// vertex / column descriptor: bit 31 landmark, bits 3 .. 30 camera / landmark index, bits 0 .. 2 component (a vertex: 0)

// one thread per right-hand-side column of the batch: I_6 columns for cameras, -Y_a of the track for landmarks (the
// cameras of a track are distinct, so no two writes meet). F is zero on entry.
__global__ void k_joint_rhs(size_t m, const uint32_t *__restrict__ desc, const uint32_t *__restrict__ cam_row,
	const uint32_t *__restrict__ pt_ptr, const uint32_t *__restrict__ obs_cam, const double *__restrict__ Y, double *__restrict__ F,
	size_t ldf)
{
	const size_t j = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(j >= m) return;
	const uint32_t d = desc[j], local = (d & 0x7fffffffu) >> 3, e = d & 7;
	double *f = F + j * ldf;
	if(!(d & 0x80000000u)) {
		f[cam_row[local] + e] = 1.0;
		return;
	}
	for(uint32_t a = pt_ptr[local]; a < pt_ptr[local + 1]; ++ a) {
		const uint32_t r = cam_row[obs_cam[a]];
		const double *y = Y + (size_t)a * 18 + e * 6; // column e of the column-major 6 x 3 block
		#pragma unroll
		for(int i = 0; i < 6; ++ i)
			f[r + i] = -y[i];
	}
}

// per set (D x D, column-major, at out + off[k]): the upper triangle plus C_p^-1 where both columns belong to the same
// landmark, written to (r, c) and, transposed, to (c, r). cols: the set's batch columns, from col_ptr[k].
__global__ void k_joint_finish(size_t n_sets, const uint64_t *__restrict__ off, const uint32_t *__restrict__ dim,
	const uint64_t *__restrict__ col_ptr, const uint32_t *__restrict__ cols, const uint32_t *__restrict__ desc,
	const double *__restrict__ Cinv, double *__restrict__ out)
{
	const uint64_t e = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if(e >= off[n_sets]) return;
	size_t lo = 0, hi = n_sets; // the set holding element e: off[lo] <= e < off[lo + 1]
	while(hi - lo > 1) {
		const size_t mid = (lo + hi) >> 1;
		if(off[mid] <= e) lo = mid; else hi = mid;
	}
	const uint32_t D = dim[lo];
	const uint64_t q = e - off[lo];
	const uint32_t c = (uint32_t)(q / D), r = (uint32_t)(q % D);
	if(r > c) return;
	double *o = out + off[lo];
	double v = o[(size_t)c * D + r];
	const uint32_t dr = desc[cols[col_ptr[lo] + r]], dc = desc[cols[col_ptr[lo] + c]];
	if((dr & 0x80000000u) && (dc & 0x80000000u) && (dr >> 3) == (dc >> 3))
		v += Cinv[(size_t)((dr & 0x7fffffffu) >> 3) * 9 + (dc & 7) * 3 + (dr & 7)];
	o[(size_t)c * D + r] = v;
	o[(size_t)r * D + c] = v;
}

// dense reduced camera system: identity on the padding of the diagonal
__global__ void k_joint_pad_identity(double *__restrict__ A, size_t ld, size_t n)
{
	const size_t i = n + blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(i < ld) A[i * ld + i] = 1.0;
}

// a factored "supernode" as the forward solve sees it
struct JmNode {
	const double *P;    // panel: R11 (ld x ld, upper), R12 (ld x h) right of it
	const double *Rinv; // [ld / 128][128 x 128] inverses of the diagonal blocks of R11, upper
	size_t ld, w, h;    // own columns padded / not, structure columns (scalars)
	uint32_t first;     // first permuted block column
	uint32_t parent;
	const uint32_t *d_rows; // structure block rows on the device (h / 6)
};

static inline size_t round_up(size_t x, size_t m) { return (x + m - 1) / m * m; }

static void joint_gemm(spp_ctx *ctx, const JointGemm &g)
{
	if(!g.M || !g.N || !g.n_kt) return;
	dim3 grid((unsigned)((g.N + JM_BN - 1) / JM_BN), (unsigned)((g.M + JM_BM - 1) / JM_BM));
	k_joint_gemm<false><<<grid, JM_THREADS, joint_gemm_smem(), ctx->stream>>>(g, 0);
	LAUNCH_CHECK(ctx);
}

static JointGemm jm_gemm(const double *A, size_t lda, const double *B, size_t ldb, double *C, size_t ldc, size_t M, size_t N,
	size_t K, int flags)
{
	JointGemm g;
	g.A = A; g.B = B; g.C = C;
	g.amap = g.bmap = g.kblk = g.c_blk = g.c_base = 0;
	g.lda = lda; g.ldb = ldb; g.ldc = ldc;
	g.M = (uint32_t)M; g.N = (uint32_t)N; g.n_kt = (uint32_t)(K / JM_BK);
	g.flags = flags;
	return g;
}

// Joint marginals of the system held as (U, V, W) (dense path: sparse == false). Sets k = verts[set_ptr[k] .. set_ptr[k +
// 1]], each vertex a descriptor (landmark, local index, component 0); p_cov receives the D_k x D_k matrices one after another. The caller
// has validated everything. budget_cols: > 0 forces the batch width (diagnostics). Returns SPP_OK / SPP_NOT_POSDEF.
int joint_marginals_to_host(spp_ctx *ctx, double alpha, bool sparse, const std::vector<uint64_t> &set_ptr,
	const std::vector<uint32_t> &verts, double *p_cov, bool timing)
{
	SchurSystem &s = ctx->sys;
	SupernodalChol &sc = ctx->snode;
	DenseChol &ch = ctx->chol;
	cudaStream_t st = ctx->stream;
	const size_t n_sets = set_ptr.size() - 1, C = s.C, n = 6 * C;
	static bool attr_done_on[64] = {false}; // the attribute belongs to the (kernel, device) pair
	bool &attr_done = attr_done_on[(ctx->device >= 0 && ctx->device < 64)? ctx->device : 0];
	if(!attr_done) {
		SPP_CUDA(cudaFuncSetAttribute(k_joint_gemm<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)joint_gemm_smem()));
		SPP_CUDA(cudaFuncSetAttribute(k_joint_gemm<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)joint_gemm_smem()));
		attr_done = true;
	}
	cudaEvent_t *ev = ctx->ev + 9; // [0 .. 6]: phase marks
	float ms[6] = {0, 0, 0, 0, 0, 0}; // forming + factorisation, plan, rhs, forward, Gram, copy
	double ms_plan = 0, flops = 0;
	auto t_host = std::chrono::steady_clock::now();

	// ---- form and factor
	if(sparse && !sc.valid) { // as schur_solve_current makes it (one rank)
		schur_fetch_host_pattern(ctx);
		snode_symbolic(ctx, C, s.h_blk_row, s.h_blk_col);
	}
	SPP_CUDA(cudaEventRecord(ev[0], st));
	std::vector<JmNode> nodes;
	std::vector<uint32_t> pos_of(C), col_super;
	ctx->h_scalars.resize(16);
	int *h_info = reinterpret_cast<int*>(ctx->h_scalars.p());
	if(sparse) {
		schur_form_reduced_system(ctx, alpha, alpha, true); // Cinv, Y and the block list of S at this damping
		s.sparse_solved = false; // the panels will hold the factor of this S, not the last solve's
		snode_factor(ctx, s.Sblk.p(), 0);
		SPP_CUDA(cudaMemcpyAsync(h_info, sc.d_info.p(), sizeof(int), cudaMemcpyDeviceToHost, st));
		const Supernodes &sn = sc.sn;
		const size_t ns = sn.n_super();
		nodes.resize(ns);
		for(size_t k = 0; k < ns; ++ k) {
			JmNode &q = nodes[k];
			q.P = sc.d_L.p() + sc.panel_off[k];
			q.Rinv = sc.d_Rinv.p() + (size_t)sc.rinv_first[k] * JM_NB * JM_NB;
			q.ld = sc.panel_ld[k];
			q.w = 6 * (size_t)(sn.first[k + 1] - sn.first[k]);
			q.h = 6 * (size_t)(sn.row_ptr[k + 1] - sn.row_ptr[k]);
			q.first = sn.first[k];
			q.parent = sn.parent[k];
			q.d_rows = sc.d_rows.p() + sn.row_ptr[k];
		}
		for(size_t i = 0; i < C; ++ i) pos_of[sc.h_order[i]] = (uint32_t)i;
		col_super = sn.col_super;
	} else {
		const size_t ld = dense_chol_ld(n), n_blk = ld / JM_NB;
		schur_form_reduced_system(ctx, alpha, alpha, false); // Cinv, Y and the dense S at this damping
		// factor a copy in the dense solve's layout (the marginals' scratch), as the solve does: the context's S stays
		s.Sinv.resize(std::max(s.Sinv.size(), dense_chol_storage(n)));
		SPP_CUDA(cudaMemcpyAsync(s.Sinv.p(), s.S.p(), dense_chol_storage(n) * sizeof(double), cudaMemcpyDeviceToDevice, st));
		ch.info.resize(1 + n_blk);
		SPP_CUDA(cudaMemsetAsync(ch.info.p(), 0, (1 + n_blk) * sizeof(int), st));
		if(ch.work.size() != n_blk * JM_NB * JM_NB) { // the diagonal-block kernel writes the upper triangles only
			ch.work.resize(n_blk * JM_NB * JM_NB);
			ch.work.zero(st);
		}
		if(ld > n) {
			k_joint_pad_identity<<<n_blocks(ld - n, 64), 64, 0, st>>>(s.Sinv.p(), ld, n);
			LAUNCH_CHECK(ctx);
		}
		if(dense_chol_dataflow_enabled())
			dense_chol_factor_dataflow(ctx, s.Sinv.p(), ld, ld + 64, ch.work.p(), ch.info.p());
		else
			dense_chol_factor_panel(ctx, s.Sinv.p(), ld, ld + JM_NB, ch.work.p(), ch.info.p(), false);
		SPP_CUDA(cudaMemcpyAsync(h_info, ch.info.p(), sizeof(int), cudaMemcpyDeviceToHost, st));
		nodes.resize(1);
		JmNode &q = nodes[0];
		q.P = s.Sinv.p(); q.Rinv = ch.work.p(); q.ld = ld; q.w = n; q.h = 0; q.first = 0; q.parent = 0xffffffffu; q.d_rows = 0;
		for(size_t i = 0; i < C; ++ i) pos_of[i] = (uint32_t)i;
		col_super.assign(C, 0);
	}
	SPP_CUDA(cudaEventRecord(ev[1], st));

	// ---- host plan
	const size_t ns = nodes.size();
	bool any_pt = false;
	for(size_t v = 0; v < verts.size(); ++ v) any_pt = any_pt || (verts[v] & 0x80000000u);
	std::vector<uint32_t> h_pt_ptr, h_obs_cam;
	if(any_pt) {
		h_pt_ptr.resize(s.P + 1);
		h_obs_cam.resize(s.O);
		s.pt_ptr.download(h_pt_ptr.data(), s.P + 1, st);
		s.obs_cam.download(h_obs_cam.data(), s.O, st);
	}
	SPP_CUDA(cudaStreamSynchronize(st)); // the status and the tracks
	if(*h_info < 0)
		throw cuda_error("dense Cholesky: the dataflow kernel's watchdog fired (a tile flag never arrived)");
	if(*h_info != 0)
		return SPP_NOT_POSDEF;
	t_host = std::chrono::steady_clock::now();
	std::vector<uint32_t> stamp(ns, 0xffffffffu), batch_stamp(ns, 0xffffffffu);
	uint32_t n_stamp = 0;
	// reach of a set (ascending: elimination order is a postorder, ancestors come later)
	auto set_reach = [&](size_t k, std::vector<uint32_t> &out) {
		out.clear();
		const uint32_t id = n_stamp ++;
		auto climb = [&](uint32_t cam) {
			for(uint32_t x = col_super[pos_of[cam]]; x != 0xffffffffu && stamp[x] != id; x = nodes[x].parent) {
				stamp[x] = id;
				out.push_back(x);
			}
		};
		for(uint64_t q = set_ptr[k]; q < set_ptr[k + 1]; ++ q) {
			const uint32_t v = verts[q], local = (v & 0x7fffffffu) >> 3;
			if(!(v & 0x80000000u))
				climb(local);
			else
				for(uint32_t a = h_pt_ptr[local]; a < h_pt_ptr[local + 1]; ++ a) climb(h_obs_cam[a]);
		}
		std::sort(out.begin(), out.end());
	};
	static const size_t forced_cols = getenv("SPP_JOINT_BATCH_COLS")? (size_t)atol(getenv("SPP_JOINT_BATCH_COLS")) : 0;
	std::vector<uint64_t> out_off(n_sets + 1, 0);
	for(size_t k = 0; k < n_sets; ++ k) {
		uint64_t D = 0;
		for(uint64_t q = set_ptr[k]; q < set_ptr[k + 1]; ++ q) D += (verts[q] & 0x80000000u)? 3 : 6;
		out_off[k + 1] = out_off[k] + D * D;
	}
	ms_plan += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_host).count();

	size_t n_batches = 0, total_cols = 0;
	std::vector<uint32_t> reach, b_reach;
	std::vector<std::vector<uint32_t> > reaches;
	size_t k0 = 0;
	while(k0 < n_sets) {
		t_host = std::chrono::steady_clock::now();
		// ---- greedy batch: whole sets in order while the compact F stays within the budget
		std::map<uint32_t, uint32_t> vcol; // vertex -> first batch column
		b_reach.clear();
		reaches.clear();
		size_t rows = 0, m = 0, k1 = k0;
		const uint32_t bid = (uint32_t)n_batches;
		while(k1 < n_sets) {
			set_reach(k1, reach);
			size_t add_rows = 0, add_cols = 0;
			for(uint32_t x : reach) if(batch_stamp[x] != bid) add_rows += nodes[x].ld;
			std::map<uint32_t, uint32_t> fresh;
			for(uint64_t q = set_ptr[k1]; q < set_ptr[k1 + 1]; ++ q)
				if(!vcol.count(verts[q]) && !fresh.count(verts[q])) {
					fresh[verts[q]] = 0;
					add_cols += (verts[q] & 0x80000000u)? 3 : 6;
				}
			const size_t r2 = rows + add_rows, m2 = m + add_cols;
			const bool fits = forced_cols? m2 <= forced_cols : (double)r2 * round_up(m2, JM_BN) * 8 <= JM_BUDGET_BYTES;
			if(k1 > k0 && !fits) break;
			for(uint32_t x : reach) if(batch_stamp[x] != bid) { batch_stamp[x] = bid; b_reach.push_back(x); }
			for(uint64_t q = set_ptr[k1]; q < set_ptr[k1 + 1]; ++ q)
				if(!vcol.count(verts[q])) {
					vcol[verts[q]] = (uint32_t)m;
					m += (verts[q] & 0x80000000u)? 3 : 6;
				}
			rows = r2;
			reaches.push_back(reach);
			++ k1;
		}
		std::sort(b_reach.begin(), b_reach.end());
		// compact rows, column descriptors, per-set columns and row blocks
		std::vector<uint64_t> row_off(ns, 0);
		size_t n_rows = 0;
		for(uint32_t x : b_reach) { row_off[x] = n_rows; n_rows += nodes[x].ld; }
		std::vector<uint32_t> h_idx; // [C pos_row | C cam_row | m desc | set columns | set row blocks]
		h_idx.assign(2 * C, 0xffffffffu);
		for(uint32_t x : b_reach) {
			const JmNode &q = nodes[x];
			for(size_t b = 0; b < q.w / 6; ++ b) h_idx[q.first + b] = (uint32_t)(row_off[x] + 6 * b);
		}
		for(size_t c = 0; c < C; ++ c) h_idx[C + c] = h_idx[pos_of[c]];
		const size_t desc_at = h_idx.size();
		h_idx.resize(desc_at + m);
		for(const auto &kv : vcol) {
			const uint32_t d = (kv.first & 0x80000000u)? 3 : 6;
			for(uint32_t e = 0; e < d; ++ e) h_idx[desc_at + kv.second + e] = kv.first | e;
		}
		const size_t nb_sets = k1 - k0;
		std::vector<uint64_t> col_ptr(nb_sets + 1, 0), kblk_at(nb_sets), fin_off(nb_sets + 1, 0);
		std::vector<uint32_t> dims(nb_sets);
		const size_t cols_at = h_idx.size();
		for(size_t k = 0; k < nb_sets; ++ k) {
			for(uint64_t q = set_ptr[k0 + k]; q < set_ptr[k0 + k + 1]; ++ q) {
				const uint32_t d = (verts[q] & 0x80000000u)? 3 : 6, c0 = vcol[verts[q]];
				for(uint32_t e = 0; e < d; ++ e) h_idx.push_back(c0 + e);
			}
			col_ptr[k + 1] = h_idx.size() - cols_at;
			dims[k] = (uint32_t)(col_ptr[k + 1] - col_ptr[k]);
			fin_off[k + 1] = out_off[k0 + k + 1] - out_off[k0];
		}
		for(size_t k = 0; k < nb_sets; ++ k) {
			kblk_at[k] = h_idx.size();
			for(uint32_t x : reaches[k])
				for(size_t b = 0; b < nodes[x].ld / JM_NB; ++ b) h_idx.push_back((uint32_t)(row_off[x] / JM_NB + b));
		}
		s.joint_idx.upload(h_idx, st);
		const uint32_t *d_idx = s.joint_idx.p();
		std::vector<JointGemm> jobs(nb_sets);
		s.joint_out.resize(std::max<uint64_t>(fin_off[nb_sets], 1));
		const size_t ldf = n_rows, mp = round_up(m, JM_BN);
		s.joint_F.resize(ldf * mp);
		uint32_t max_d = 0;
		for(size_t k = 0; k < nb_sets; ++ k) {
			const size_t K = (size_t)((k + 1 < nb_sets? kblk_at[k + 1] : h_idx.size()) - kblk_at[k]) * JM_NB;
			JointGemm &g = jobs[k];
			g = jm_gemm(s.joint_F.p(), ldf, s.joint_F.p(), ldf, s.joint_out.p() + fin_off[k], dims[k], dims[k], dims[k], K, JM_UPPER);
			g.amap = g.bmap = d_idx + cols_at + col_ptr[k];
			g.kblk = d_idx + kblk_at[k];
			max_d = std::max(max_d, dims[k]);
		}
		std::vector<uint64_t> h_fin(2 * (nb_sets + 1));
		std::copy(fin_off.begin(), fin_off.end(), h_fin.begin());
		std::copy(col_ptr.begin(), col_ptr.end(), h_fin.begin() + nb_sets + 1);
		s.joint_off.upload(h_fin, st);
		s.joint_dim.upload(dims, st);
		s.joint_jobs.upload(reinterpret_cast<const uint8_t*>(jobs.data()), jobs.size() * sizeof(JointGemm), st);
		ms_plan += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_host).count();

		// ---- right-hand side
		SPP_CUDA(cudaEventRecord(ev[2], st));
		SPP_CUDA(cudaMemsetAsync(s.joint_F.p(), 0, ldf * mp * sizeof(double), st));
		k_joint_rhs<<<n_blocks(m, 128), 128, 0, st>>>(m, d_idx + desc_at, d_idx + C, s.pt_ptr.p(), s.obs_cam.p(), s.Y.p(),
			s.joint_F.p(), ldf);
		LAUNCH_CHECK(ctx);
		SPP_CUDA(cudaEventRecord(ev[3], st));

		// ---- forward solve over the batch's reach, elimination order
		double *F = s.joint_F.p();
		for(uint32_t x : b_reach) {
			const JmNode &q = nodes[x];
			double *Bs = F + row_off[x];
			for(size_t r0 = 0; r0 < q.w; r0 += JM_NB) {
				const size_t kk = round_up(std::min<size_t>(JM_NB, q.w - r0), JM_BK), c1 = r0 + JM_NB;
				// F_i = Rinv_i^T B_i, in place
				joint_gemm(ctx, jm_gemm(q.Rinv + (r0 / JM_NB) * JM_NB * JM_NB, JM_NB, Bs + r0, ldf, Bs + r0, ldf, JM_NB, m, kk, JM_A_LOWER));
				// B_{>i} -= R11[i, >i]^T F_i
				if(c1 < q.w)
					joint_gemm(ctx, jm_gemm(q.P + c1 * q.ld + r0, q.ld, Bs + r0, ldf, Bs + c1, ldf, q.w - c1, m, kk, JM_SUB));
			}
			if(q.h) { // B[rows of J] -= R12^T F_s
				JointGemm g = jm_gemm(q.P + q.ld * q.ld, q.ld, Bs, ldf, F, ldf, q.h, m, round_up(q.w, JM_BK), JM_SUB);
				g.c_blk = q.d_rows;
				g.c_base = d_idx;
				joint_gemm(ctx, g);
			}
			flops += ((double)q.w * q.w + 2.0 * q.w * q.h) * m;
		}
		SPP_CUDA(cudaEventRecord(ev[4], st));

		// ---- Gram per set, then C^-1 and the lower triangles
		dim3 grid((unsigned)((max_d + JM_BN - 1) / JM_BN), (unsigned)((max_d + JM_BM - 1) / JM_BM), (unsigned)nb_sets);
		for(size_t z0 = 0; z0 < nb_sets; z0 += 65535) { // grid.z limit
			grid.z = (unsigned)std::min<size_t>(65535, nb_sets - z0);
			JointGemm dummy = jobs[0];
			k_joint_gemm<true><<<grid, JM_THREADS, joint_gemm_smem(), st>>>(dummy,
				reinterpret_cast<const JointGemm*>(s.joint_jobs.p()) + z0);
			LAUNCH_CHECK(ctx);
		}
		k_joint_finish<<<n_blocks(fin_off[nb_sets], 256), 256, 0, st>>>(nb_sets, s.joint_off.p(), s.joint_dim.p(),
			s.joint_off.p() + nb_sets + 1, d_idx + cols_at, d_idx + desc_at, s.Cinv.p(), s.joint_out.p());
		LAUNCH_CHECK(ctx);
		SPP_CUDA(cudaEventRecord(ev[5], st));

		// ---- to the host
		s.joint_out.download(p_cov + out_off[k0], fin_off[nb_sets], st);
		SPP_CUDA(cudaEventRecord(ev[6], st));
		SPP_CUDA(cudaStreamSynchronize(st));
		if(timing) {
			float t;
			if(!n_batches) { SPP_CUDA(cudaEventElapsedTime(&t, ev[0], ev[1])); ms[0] += t; }
			for(int i = 2; i < 6; ++ i) { SPP_CUDA(cudaEventElapsedTime(&t, ev[i], ev[i + 1])); ms[i] += t; }
		}
		++ n_batches;
		total_cols += m;
		k0 = k1;
	}
	if(timing && !n_batches) {
		float t;
		SPP_CUDA(cudaEventElapsedTime(&t, ev[0], ev[1]));
		ms[0] += t;
	}
	if(timing)
		fprintf(stderr, "[spp joint marginals] %s path: schur + factor %.3f ms, plan %.3f ms (host), rhs %.3f ms, forward solve %.3f ms "
			"(%.3e flops, %.2f TFLOP/s), gram %.3f ms, copy to host %.3f ms; %zu sets, %zu batches, %zu columns\n",
			sparse? "supernodal" : "dense", ms[0], ms_plan, ms[2], ms[3], flops, flops / std::max(ms[3], 1e-6f) * 1e-9, ms[4], ms[5],
			n_sets, n_batches, total_cols);
	return SPP_OK;
}

} // namespace spp
