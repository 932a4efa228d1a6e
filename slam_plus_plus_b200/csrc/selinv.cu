// selinv.cu -- selected inversion on the supernodal factor of a block-sparse reduced camera system: the entries of
// Z = S^-1 on the pattern of the factor R (P S P^T = R^T R), written over R in the panels. The marginal covariances
// (marginals.cu) read the camera blocks and, per landmark, the camera pairs of its track from there.
//
// Reference replaced: the reference recovers the marginals of a bundle adjustment from the factor of the Schur complement
// (CSchurComplement_Marginals::Schur_Marginals, include/slam/BAMarginals.h:579-760, called at the end of
// CNonlinearSolver_Lambda_LM::Optimize(), NonlinearSolver_Lambda_LM.h:1118-1350); it does so on a dense factor only.
//
// Takahashi recursion by supernodes: for supernode s with its own columns I (w of them, padded to ld) and its row
// structure J (h), the panel holds R11 = R_II and R12 = R_IJ. Root to leaves (every ancestor's Z is final before a
// descendant reads it):
//     W     = R11^-1                 upper; block back substitution from the 128 x 128 diagonal-block inverses Rinv
//                                    that the factorisation left: W_ii = Rinv_i, W_i,>i = -Rinv_i (R11_i,>i W_>i,>i)
//     X     = W R12
//     G     = Z_JJ                   gathered from the ancestors' panels through the update maps of s (the positions
//                                    the factorisation's updates s -> t scattered into), both triangles
//     Z_IJ  = -X G                   over R12
//     Z_II  = W W^T - Z_IJ X^T       over R11 (upper tiles; every diagonal-straddling tile in full)
// 2 w^3 / 3 + 2 w^2 h + 2 w h^2 flops, twice the factorisation's. Every product is one FP64 tensor-core GEMM
// (mma.sync m8n8k4, tcgen05 has no FP64 kind) with the triangular operands' zero tiles skipped. The schedule is the
// backward solve's: a supernode waits for its parent's event, independent subtrees run side by side on the side streams
// (narrow supernodes, each lane with its own scratch), the wide supernodes share one scratch on the main stream. Every
// sum has a fixed order: no atomics, bit-reproducible.

#include "spp_ctx.h"
#include <cuda_pipeline_primitives.h>
#include <algorithm>

namespace spp {

#define LAUNCH_CHECK(ctx) do { ++ (ctx)->n_launches; SPP_CUDA(cudaGetLastError()); } while(0)

#define SI_NB 128   // panel granularity (= SN_NB of supernodal_chol.cu)
#define SI_BM 128
#define SI_BN 64
#define SI_BK 16
#define SI_STAGES 3
#define SI_THREADS 256

__device__ __forceinline__ void dmma_si(double &d0, double &d1, double a, double b)
{
	asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
		: "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

enum { SI_A_UPPER = 1, SI_B_UPPER = 2, SI_BT_UPPER = 4, SI_C_UPPER = 8, SI_ACC = 16, SI_NEG = 32 };

// C (M x N, column-major, ldc) = [C +] (-)A op(B), K = the inner dimension; A column-major (element (m, k) at
// A[k lda + m]); TB = false: B(k, n) at B[n ldb + k], TB = true: op(B)(k, n) = B[k ldb + n]. M, N, K multiples of
// SI_BM, SI_BN, SI_BK. Flags: SI_A_UPPER A(m, k) = 0 for k < m; SI_B_UPPER B(k, n) = 0 for k > n (TB = false);
// SI_BT_UPPER op(B)(k, n) = 0 for k < n (TB = true); SI_C_UPPER tiles strictly below the diagonal are not computed.
// The zero tiles are skipped at tile granularity, so the operands' zero triangles inside a tile must be stored zeros.
// Block tile 128 x 64, eight warps of 32 x 32, 3-stage cp.async pipeline; operand tiles in shared memory with the
// fragment's contiguous dimension padded by 4 (conflict-free DMMA fragment loads).
template <bool TB>
__global__ void __launch_bounds__(SI_THREADS) k_selinv_gemm(size_t K, const double *__restrict__ A, size_t lda,
	const double *__restrict__ B, size_t ldb, double *__restrict__ C, size_t ldc, int flags)
{
	const size_t i0 = blockIdx.y * (size_t)SI_BM, j0 = blockIdx.x * (size_t)SI_BN;
	if((flags & SI_C_UPPER) && i0 > j0 + (SI_BN - 1))
		return;
	constexpr int A_LD = SI_BM + 4, B_LD = TB? SI_BN + 4 : SI_BK + 4, B_STAGE = TB? SI_BK * B_LD : SI_BN * B_LD;
	extern __shared__ double smem[];
	double *As = smem, *Bs = smem + SI_STAGES * SI_BK * A_LD;
	const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
	const int wi = (warp >> 1) * 32, wj = (warp & 1) * 32;
	const int g = lane >> 2, t = lane & 3;

	size_t kb = 0, ke = K;
	if(flags & SI_A_UPPER) kb = max(kb, i0);
	if(flags & SI_BT_UPPER) kb = max(kb, j0);
	if(flags & SI_B_UPPER) ke = min(ke, j0 + SI_BN);
	const int KT = (ke > kb)? (int)((ke - kb) / SI_BK) : 0;

	auto stage_load = [&](int st, int kc) {
		const size_t k0 = kb + (size_t)kc * SI_BK;
		double *as = As + st * SI_BK * A_LD, *bs = Bs + st * B_STAGE;
		for(int idx = tid; idx < SI_BK * SI_BM / 2; idx += SI_THREADS) { // (k, m pair)
			const int k = idx / (SI_BM / 2), q = idx % (SI_BM / 2);
			__pipeline_memcpy_async(as + k * A_LD + 2 * q, A + (k0 + k) * lda + i0 + 2 * q, 16);
		}
		if(TB) {
			for(int idx = tid; idx < SI_BK * SI_BN / 2; idx += SI_THREADS) { // (k, n pair)
				const int k = idx / (SI_BN / 2), q = idx % (SI_BN / 2);
				__pipeline_memcpy_async(bs + k * B_LD + 2 * q, B + (k0 + k) * ldb + j0 + 2 * q, 16);
			}
		} else {
			for(int idx = tid; idx < SI_BN * SI_BK / 2; idx += SI_THREADS) { // (n, k pair)
				const int n = idx / (SI_BK / 2), q = idx % (SI_BK / 2);
				__pipeline_memcpy_async(bs + n * B_LD + 2 * q, B + (j0 + n) * ldb + k0 + 2 * q, 16);
			}
		}
	};

	#pragma unroll
	for(int s = 0; s < SI_STAGES - 1; ++ s) {
		if(s < KT) stage_load(s, s);
		__pipeline_commit();
	}
	double acc[4][4][2];
	#pragma unroll
	for(int a = 0; a < 4; ++ a) {
		#pragma unroll
		for(int b = 0; b < 4; ++ b) {
			if(flags & SI_ACC) {
				const size_t c = j0 + wj + b * 8 + 2 * t, r = i0 + wi + a * 8 + g;
				acc[a][b][0] = C[c * ldc + r];
				acc[a][b][1] = C[(c + 1) * ldc + r];
			} else
				acc[a][b][0] = acc[a][b][1] = 0;
		}
	}
	const bool neg = (flags & SI_NEG) != 0;
	for(int kt = 0; kt < KT; ++ kt) {
		__pipeline_wait_prior(SI_STAGES - 2);
		__syncthreads();
		if(kt + SI_STAGES - 1 < KT)
			stage_load((kt + SI_STAGES - 1) % SI_STAGES, kt + SI_STAGES - 1);
		__pipeline_commit();
		const int st = kt % SI_STAGES;
		const double *as = As + st * SI_BK * A_LD, *bs = Bs + st * B_STAGE;
		#pragma unroll
		for(int k4 = 0; k4 < SI_BK; k4 += 4) {
			double fa[4], fb[4];
			#pragma unroll
			for(int a = 0; a < 4; ++ a) {
				const double v = as[(k4 + t) * A_LD + wi + a * 8 + g];
				fa[a] = neg? -v : v;
			}
			#pragma unroll
			for(int b = 0; b < 4; ++ b)
				fb[b] = TB? bs[(k4 + t) * B_LD + wj + b * 8 + g] : bs[(wj + b * 8 + g) * B_LD + k4 + t];
			#pragma unroll
			for(int a = 0; a < 4; ++ a)
				#pragma unroll
				for(int b = 0; b < 4; ++ b)
					dmma_si(acc[a][b][0], acc[a][b][1], fa[a], fb[b]);
		}
	}
	__pipeline_wait_prior(0);
	#pragma unroll
	for(int a = 0; a < 4; ++ a) {
		#pragma unroll
		for(int b = 0; b < 4; ++ b) {
			const size_t c = j0 + wj + b * 8 + 2 * t, r = i0 + wi + a * 8 + g;
			C[c * ldc + r] = acc[a][b][0];
			C[(c + 1) * ldc + r] = acc[a][b][1];
		}
	}
}

static size_t selinv_gemm_smem(bool tb)
{
	return (size_t)SI_STAGES * (SI_BK * (SI_BM + 4) + (tb? SI_BK * (SI_BN + 4) : SI_BN * (SI_BK + 4))) * sizeof(double);
}

// G(i, j) = Z_JJ of supernode s for the rows of one update s -> t: i < M (the part of the suffix inside t's own
// columns), i <= j < n_suffix; both triangles of G are written. cmap: block positions of the suffix in panel t (as the
// update scattered into them); row0: first scalar of the suffix in J. Threads run along the rows of one column.
__global__ void k_selinv_gather(uint32_t M, uint32_t n_suffix, uint32_t row0, const double *__restrict__ Pt, size_t ld_t,
	const uint32_t *__restrict__ cmap, double *__restrict__ G, size_t ldg)
{
	const uint32_t i = blockIdx.x * (uint32_t)blockDim.x + threadIdx.x, j = blockIdx.y;
	if(i >= M || j >= n_suffix || j < i) return;
	uint32_t rp = cmap[i / 6] + i % 6, cp = cmap[j / 6] + j % 6;
	if(rp > cp) { const uint32_t x = rp; rp = cp; cp = x; } // lower half of a diagonal block: its upper mirror
	const double v = Pt[(size_t)cp * ld_t + rp];
	const size_t gi = row0 + i, gj = row0 + j;
	G[gj * ldg + gi] = v;
	G[gi * ldg + gj] = v;
}

static void selinv_gemm(spp_ctx *ctx, cudaStream_t st, size_t M, size_t N, size_t K, const double *A, size_t lda,
	const double *B, size_t ldb, bool tb, double *C, size_t ldc, int flags)
{
	dim3 grid((unsigned)(N / SI_BN), (unsigned)(M / SI_BM));
	if(tb)
		k_selinv_gemm<true><<<grid, SI_THREADS, selinv_gemm_smem(true), st>>>(K, A, lda, B, ldb, C, ldc, flags);
	else
		k_selinv_gemm<false><<<grid, SI_THREADS, selinv_gemm_smem(false), st>>>(K, A, lda, B, ldb, C, ldc, flags);
	LAUNCH_CHECK(ctx);
}

// one supernode, enqueued on st; scratch (sized by snode_symbolic): [W, later G: max(ld^2, hp^2) | T: 128 ld | X: ld hp]
static void selinv_supernode(spp_ctx *ctx, cudaStream_t st, size_t s, double *scratch)
{
	SupernodalChol &sc = ctx->snode;
	const Supernodes &sn = sc.sn;
	const size_t ld = sc.panel_ld[s], nb = ld / SI_NB;
	const size_t hb = sn.row_ptr[s + 1] - sn.row_ptr[s], h = 6 * hb, hp = (h + SN_SEL_HP - 1) / SN_SEL_HP * SN_SEL_HP;
	double *P = sc.d_L.p() + sc.panel_off[s];
	const double *Rinv = sc.d_Rinv.p() + (size_t)sc.rinv_first[s] * SI_NB * SI_NB;
	double *W = scratch, *G = scratch, *T = scratch + std::max(ld * ld, hp * hp), *X = T + SI_NB * ld;
	// W = R11^-1, block row by block row from the bottom
	for(size_t bi = nb; bi > 0; -- bi) {
		const size_t i = bi - 1, r0 = i * SI_NB, c1 = r0 + SI_NB, m = ld - c1;
		SPP_CUDA(cudaMemcpy2DAsync(W + r0 * ld + r0, ld * sizeof(double), Rinv + i * SI_NB * SI_NB, SI_NB * sizeof(double),
			SI_NB * sizeof(double), SI_NB, cudaMemcpyDeviceToDevice, st));
		if(!m) continue;
		// T = R11[i, >i] W[>i, >i]; W[i, >i] = -Rinv_i T
		selinv_gemm(ctx, st, SI_NB, m, m, P + c1 * ld + r0, ld, W + c1 * ld + c1, ld, false, T, SI_NB, SI_B_UPPER);
		selinv_gemm(ctx, st, SI_NB, m, SI_NB, Rinv + i * SI_NB * SI_NB, SI_NB, T, SI_NB, false, W + c1 * ld + r0, ld,
			SI_A_UPPER | SI_NEG);
	}
	double *R12 = P + ld * ld;
	// X = W R12 (R12 is read for the last time)
	if(h)
		selinv_gemm(ctx, st, ld, hp, ld, W, ld, R12, ld, false, X, ld, SI_A_UPPER);
	// Z_II = W W^T over R11 (read for the last time by the W recursion); W is not needed after this
	selinv_gemm(ctx, st, ld, ld, ld, W, ld, W, ld, true, P, ld, SI_A_UPPER | SI_BT_UPPER | SI_C_UPPER);
	if(!h)
		return;
	// G = Z_JJ from the ancestors, zero padding, where W was
	SPP_CUDA(cudaMemsetAsync(G, 0, hp * hp * sizeof(double), st));
	size_t q = 0; // first structure block of the update
	for(uint64_t k = sc.upd_ptr[s]; k < sc.upd_ptr[s + 1]; ++ k) {
		const SnodeUpdate &u = sc.updates[k];
		const uint32_t n_suffix = u.N - 1; // without the right-hand-side column
		dim3 grid((u.M + 127) / 128, n_suffix);
		k_selinv_gather<<<grid, 128, 0, st>>>(u.M, n_suffix, (uint32_t)(6 * q), sc.d_L.p() + sc.panel_off[u.t], sc.panel_ld[u.t],
			sc.d_cmap.p() + u.map_off, G, hp);
		LAUNCH_CHECK(ctx);
		q += u.M / 6;
	}
	// Z_IJ = -X G over R12, then Z_II -= Z_IJ X^T
	selinv_gemm(ctx, st, ld, hp, hp, X, ld, G, hp, false, R12, ld, SI_NEG);
	selinv_gemm(ctx, st, ld, ld, hp, R12, ld, X, ld, true, P, ld, SI_C_UPPER | SI_ACC | SI_NEG);
}

// Selected inversion of the factor in the panels (snode_factor must have succeeded; ev_factor[ns - 1] marks its end on
// the context's stream). Enqueued; ends joined into the context's stream.
void snode_selected_inverse(spp_ctx *ctx)
{
	SupernodalChol &sc = ctx->snode;
	const Supernodes &sn = sc.sn;
	const size_t ns = sn.n_super();
	cudaStream_t st = ctx->stream;
	static bool attr_done_on[64] = {false}; // the attribute belongs to the (kernel, device) pair
	bool &attr_done = attr_done_on[(ctx->device >= 0 && ctx->device < 64)? ctx->device : 0];
	if(!attr_done) {
		SPP_CUDA(cudaFuncSetAttribute(k_selinv_gemm<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)selinv_gemm_smem(true)));
		SPP_CUDA(cudaFuncSetAttribute(k_selinv_gemm<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)selinv_gemm_smem(false)));
		attr_done = true;
	}
	sc.d_sel_main.resize(std::max<size_t>(sc.selinv_main_doubles, 1));
	sc.d_sel_lane.resize(std::max<size_t>(sc.selinv_lane_doubles * SupernodalChol::N_STREAMS, 1));
	bool lane_used[SupernodalChol::N_STREAMS] = {false};
	for(size_t ss = ns; ss > 0; -- ss) {
		const size_t s = ss - 1;
		const size_t ld = sc.panel_ld[s], h = 6 * (size_t)(sn.row_ptr[s + 1] - sn.row_ptr[s]);
		const bool on_lane = selinv_on_lane(ld, (h + SN_SEL_HP - 1) / SN_SEL_HP * SN_SEL_HP);
		const int lane = int(s % SupernodalChol::N_STREAMS);
		cudaStream_t ss_ = on_lane? sc.side[lane] : st;
		double *scratch = on_lane? sc.d_sel_lane.p() + (size_t)lane * sc.selinv_lane_doubles : sc.d_sel_main.p();
		if(sn.parent[s] != 0xffffffffu)
			SPP_CUDA(cudaStreamWaitEvent(ss_, sc.ev_x[sn.parent[s]], 0));
		else
			SPP_CUDA(cudaStreamWaitEvent(ss_, sc.ev_factor[ns - 1], 0));
		selinv_supernode(ctx, ss_, s, scratch);
		SPP_CUDA(cudaEventRecord(sc.ev_x[s], ss_));
		if(on_lane) lane_used[lane] = true;
	}
	for(int i = 0; i < SupernodalChol::N_STREAMS; ++ i) { // join the side lanes
		if(!lane_used[i]) continue;
		SPP_CUDA(cudaEventRecord(sc.ev_target[i % ns], sc.side[i]));
		SPP_CUDA(cudaStreamWaitEvent(st, sc.ev_target[i % ns], 0));
	}
}

} // namespace spp
