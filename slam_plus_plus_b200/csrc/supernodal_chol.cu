// supernodal_chol.cu -- stage 3 of the hot path for a reduced camera system (RCS) that is too large to be dense
// (BAL-13682 shape: 82 092 unknowns, 3-4 % block fill): supernodal block Cholesky S = R^T R under a fill-reducing
// ordering, forward solve riding along as an extra column, backward solve.
//
// Reference behaviour replaced (SURVEY 8(a) rows a14/a15): CLinearSolver_Schur first tries the dense solver and, when
// that throws std::bad_alloc, falls back to CLinearSolver_UberBlock on the block-sparse Schur complement
// (include/slam/LinearSolver_Schur.h:1836-1847): AMD ordering of the 6x6 block structure (CMatrixOrdering::
// p_BlockOrdering, src/slam/OrderingMagic.cpp:701-1033), elimination tree, up-looking block Cholesky
// (CUberBlockMatrix::CholeskyOf_FBS, include/slam/BlockMatrixFBS.inl:2341-2513) and two triangular solves
// (:2136-2275), all on one thread, block by block.
//
// Here the host does the integer work once per structure (block_ordering.cpp: ordering -- the caller's, i.e. the
// reference's own AMD permutation through the adapter, or the library's approximate minimum degree -- elimination
// tree, supernodes with relaxed amalgamation). A reduced camera system of a long sequence has FEW, WIDE supernodes
// (BAL shape: ~150 supernodes up to 17 000 columns wide with 10 000-row structures), so the numeric phase is dense
// FP64 tensor-core work on panels:
//   k_snode_assemble    scatter of the compact 6x6 block list of S (what the Schur kernels write and, on several
//                       GPUs, what the all-reduce sums) into the panels; rhs into the panels' rhs column
//   per supernode s, in elimination order:
//     dense_chol_factor_panel (dense_chol.cu)   potrf / TRSM / SYRK on the panel (R11, R12 = R11^-T A12, y = R11^-T b)
//     k_snode_update      for every ancestor t that owns rows of s: panel_t -= R_s[:, J]^T R_s[:, J..] as ONE DMMA
//                         GEMM (K = width of s) whose epilogue subtracts through the relative-index map -- stream
//                         order makes the sum order fixed: no atomics, bit-reproducible
//   backward, root to leaves: k_snode_gemv (y_s -= R12 x) + the dense backsolve on R11.

#include "spp_ctx.h"
#include <cuda_pipeline_primitives.h>
#include <algorithm>
#include <stdlib.h>

namespace spp {

void dense_chol_factor_panel(spp_ctx *ctx, double *A, size_t ld, size_t n_cols, double *Rinv, int *info, bool identity_tail = false);
void dense_chol_factor_single_panel(spp_ctx *ctx, cudaStream_t stream, double *A, size_t n_cols, double *Rinv, int *info);
void dense_chol_factor_dataflow(spp_ctx *ctx, double *A, size_t ld, size_t n_cols, double *Rinv, int *info);
bool dense_chol_dataflow_enabled();
void dense_chol_backsolve_panel(spp_ctx *ctx, cudaStream_t stream, const double *A, size_t ld, const double *Rinv, double *y, int *flags);
void schur_fetch_host_pattern(spp_ctx *ctx);
void allreduce_device(spp_ctx *ctx, double *d_ptr, size_t n);

#define LAUNCH_CHECK(ctx) do { ++ (ctx)->n_launches; SPP_CUDA(cudaGetLastError()); } while(0)

#define SN_NB 128   // panel granularity (= CH_NB of dense_chol.cu)
#define SN_BK 16
#define SN_LDS (SN_BK + 4)
#define SN_STAGES 3
#define SN_GEMV_COLS 64 // columns per CTA of the backward-solve GEMV: a short dependent chain per thread, many CTAs

// relaxed amalgamation (supernodal_symbolic): a supernode merges into its parent while the explicit zeros stay below this
// share of the merged panel, or while the merged width is at most this many block columns
static const double SN_RELAX_ZEROS = 0.05;
static const size_t SN_RELAX_SMALL = 16;
// supernodes at least this many columns wide are factored by the dataflow kernel (k_chol_dataflow), narrower ones by
// the look-ahead panel factorisation, whose panels were chain-bound on them
static const size_t SN_DATAFLOW_MIN = 1024;

static inline size_t round_up(size_t x, size_t m) { return (x + m - 1) / m * m; }

// the code path of a supernode and of an update, from the panel shapes: the numeric phase dispatches on these, the
// SPP_SNODE_VERBOSE line of the analysis counts them
static inline bool snode_on_side(size_t ld) { return ld == SN_NB; }               // one diagonal block: a side stream
static inline bool snode_dataflow(size_t ld) { return ld >= SN_DATAFLOW_MIN; }    // k_chol_dataflow (SPP_CHOL_DATAFLOW != 0)
static inline bool snode_update_tile128(const SnodeUpdate &u)                     // k_snode_update<128, 64>: two CTAs per SM
{
	return (size_t)((u.M + 127) / 128) * ((u.N + 127) / 128) >= 48;
}

// ---- host: symbolic -----------------------------------------------------------------------------------------

// blk_row / blk_col: the upper block list of the reduced camera system (i <= j, any order, diagonal blocks present)
void snode_symbolic(spp_ctx *ctx, size_t n, const std::vector<uint32_t> &blk_row, const std::vector<uint32_t> &blk_col)
{
	SupernodalChol &sc = ctx->snode;
	sc.valid = false;
	if(sc.sym_kept && sc.n == n && sc.sym_world == ctx->world && sc.sym_rank == ctx->rank && sc.sym_user_order == sc.user_order &&
	   sc.sym_row == blk_row && sc.sym_col == blk_col && !getenv("SPP_SNODE_NO_REUSE")) {
		sc.valid = true; // the same structure was uploaded again (new measurements / states): ordering, supernodes, maps and
		return;          // panel layout on the device are still the right ones
	}
	sc.sym_kept = false;
	sc.n = n;
	const size_t nb = blk_row.size();
	sc.n_s_blocks = nb;
	// upper block CSC, rows ascending
	std::vector<uint64_t> col_ptr(n + 1, 0), row_idx(nb);
	for(size_t b = 0; b < nb; ++ b) {
		if(blk_row[b] > blk_col[b] || blk_col[b] >= n)
			throw invalid_error("supernodal Cholesky: the block list must be upper triangular");
		++ col_ptr[blk_col[b] + 1];
	}
	for(size_t j = 0; j < n; ++ j) col_ptr[j + 1] += col_ptr[j];
	{
		std::vector<uint64_t> fill(col_ptr.begin(), col_ptr.end() - 1);
		for(size_t b = 0; b < nb; ++ b) row_idx[fill[blk_col[b]] ++] = blk_row[b];
		for(size_t j = 0; j < n; ++ j) std::sort(row_idx.begin() + col_ptr[j], row_idx.begin() + col_ptr[j + 1]);
	}
	// ordering
	if(!sc.user_order.empty()) {
		if(sc.user_order.size() != n)
			throw invalid_error("supernodal Cholesky: the ordering given by spp_schur_set_rcs_ordering has the wrong size");
		sc.h_order.assign(sc.user_order.begin(), sc.user_order.end());
	} else // approximate minimum degree, the reference's permutation (amd_exact.cpp)
		amd_exact_ordering(n, col_ptr.data(), row_idx.data(), sc.h_order);
	supernodal_symbolic(n, col_ptr.data(), row_idx.data(), sc.h_order, SN_RELAX_ZEROS, SN_RELAX_SMALL, (size_t)1 << 30, sc.sn);
	const Supernodes &sn = sc.sn;
	const size_t ns = sn.n_super();
	std::vector<uint32_t> inv(n);
	for(size_t i = 0; i < n; ++ i) inv[sc.h_order[i]] = (uint32_t)i;

	// panel layout
	sc.panel_off.resize(ns);
	sc.panel_ld.resize(ns);
	sc.panel_cols.resize(ns);
	sc.rinv_first.resize(ns);
	uint64_t total = 0;
	size_t n_rinv = 0;
	sc.factor_flops = 0;
	sc.max_part = 0;
	std::vector<uint64_t> pad_off;
	std::vector<uint32_t> pad_ld, pad_n0;
	for(size_t s = 0; s < ns; ++ s) {
		const size_t w = 6 * (size_t)(sn.first[s + 1] - sn.first[s]), h = 6 * (size_t)(sn.row_ptr[s + 1] - sn.row_ptr[s]);
		const size_t ld = round_up(w, SN_NB), cols = ld + round_up(h + 1, SN_NB);
		if(cols >= 0x7fffffffu)
			throw invalid_error("supernodal Cholesky: panel too wide for 32-bit column indices");
		sc.panel_off[s] = total;
		sc.panel_ld[s] = (uint32_t)ld;
		sc.panel_cols[s] = (uint32_t)cols;
		sc.rinv_first[s] = (uint32_t)n_rinv;
		total += (uint64_t)ld * cols;
		n_rinv += ld / SN_NB;
		sc.factor_flops += (double)w * w * w / 3 + (double)w * w * h + (double)w * h * h;
		if(ld > w) {
			pad_off.push_back(sc.panel_off[s]);
			pad_ld.push_back((uint32_t)ld);
			pad_n0.push_back((uint32_t)w);
		}
		if(h)
			sc.max_part = std::max(sc.max_part, ld * ((h + SN_GEMV_COLS - 1) / SN_GEMV_COLS));
	}
	sc.n_rinv_blocks = n_rinv;
	sc.factor_flops_total = sc.factor_flops;

	// ---- several ranks: who factors what. The work of a supernode (its panel and the updates it sends) is summed over
	// subtrees; supernodes whose subtree weighs more than a threshold stay with every rank ("shared": the top of the
	// tree, an upward-closed set), the subtrees hanging below them go to the least loaded rank, heaviest first. The
	// threshold is the one (of a few multiples of total / world) with the smallest predicted time = shared work + the
	// heaviest rank. Every rank computes the same plan from the same structure.
	sc.owner.assign(ns, -1);
	sc.distributed = false;
	if(ctx->world > 1 && ns > 1 && !getenv("SPP_SNODE_REPLICATED")) {
		std::vector<double> work;
		// a plan must save at least 3 % to be worth the exchange (SPP_SNODE_DISTRIBUTE_ALWAYS: any saving, for tests)
		const double f_predicted = plan_subtree_owners(sn, ctx->world, getenv("SPP_SNODE_DISTRIBUTE_ALWAYS")? 1e-9 : 0.03, sc.owner, work);
		const double f_total = sc.factor_flops_total, f_best = f_predicted * f_total;
		sc.distributed = f_predicted < 1.0;
		if(sc.distributed) {
			sc.factor_flops = 0;
			for(size_t s = 0; s < ns; ++ s)
				if(sc.owner[s] < 0 || sc.owner[s] == ctx->rank) sc.factor_flops += work[s];
		}
		if(getenv("SPP_SNODE_VERBOSE")) {
			size_t n_shared = 0;
			for(size_t s = 0; s < ns; ++ s) n_shared += sc.owner[s] < 0;
			fprintf(stderr, "[spp snode] rank %d of %d: %s, %zu of %zu supernodes shared, this rank executes %.3e of %.3e flops (predicted time %.1f %% of one rank's)\n",
				ctx->rank, ctx->world, sc.distributed? "subtrees distributed" : "replicated", n_shared, ns, sc.factor_flops, f_total,
				100 * f_best / f_total);
		}
	}

	// position of a block row inside panel t: own columns first, then the structure
	auto col_pos = [&](size_t t, uint32_t rb) -> uint32_t {
		if(rb < sn.first[t + 1])
			return (uint32_t)(6 * (rb - sn.first[t]));
		const uint32_t *beg = &sn.rows[sn.row_ptr[t]], *end = beg + (sn.row_ptr[t + 1] - sn.row_ptr[t]);
		const uint32_t *it = std::lower_bound(beg, end, rb);
		if(it == end || *it != rb)
			throw std::runtime_error("supernodal Cholesky: inconsistent symbolic structure");
		return (uint32_t)(sc.panel_ld[t] + 6 * (it - beg));
	};
	// destination of every block of S and of every camera's right-hand side
	std::vector<uint64_t> asm_dst(nb), rhs_dst(n);
	std::vector<uint32_t> asm_ld(nb);
	for(size_t b = 0; b < nb; ++ b) {
		const uint32_t pi = inv[blk_row[b]], pj = inv[blk_col[b]];
		const uint32_t lo = std::min(pi, pj), hi = std::max(pi, pj);
		const size_t t = sn.col_super[lo];
		const uint64_t ld = sc.panel_ld[t];
		uint64_t dst = sc.panel_off[t] + (uint64_t)col_pos(t, hi) * ld + 6 * (uint64_t)(lo - sn.first[t]);
		if(pi > pj)
			dst |= (uint64_t)1 << 63; // S(i, j) lands transposed
		asm_dst[b] = dst;
		asm_ld[b] = (uint32_t)ld;
	}
	for(size_t j = 0; j < n; ++ j) {
		const size_t t = sn.col_super[j];
		const uint64_t ld = sc.panel_ld[t], h = 6 * (uint64_t)(sn.row_ptr[t + 1] - sn.row_ptr[t]);
		rhs_dst[sc.h_order[j]] = sc.panel_off[t] + (ld + h) * ld + 6 * (uint64_t)(j - sn.first[t]);
	}
	// marginals: camera -> its diagonal block in the panels, and the block CSC (rows ascending, block id beside each row)
	// through which a landmark finds the block of any camera pair of its track
	std::vector<uint64_t> cam_diag(n);
	std::vector<uint32_t> cam_ld(n), csc_row(nb), csc_blk(nb);
	for(size_t c = 0; c < n; ++ c) {
		const uint32_t j = inv[c];
		const size_t t = sn.col_super[j];
		cam_diag[c] = sc.panel_off[t] + 6 * (uint64_t)(j - sn.first[t]) * (sc.panel_ld[t] + 1);
		cam_ld[c] = sc.panel_ld[t];
	}
	{
		std::vector<std::pair<uint32_t, uint32_t> > entries(nb);
		std::vector<uint64_t> fill(col_ptr.begin(), col_ptr.end() - 1);
		for(size_t b = 0; b < nb; ++ b) entries[fill[blk_col[b]] ++] = std::make_pair(blk_row[b], (uint32_t)b);
		for(size_t j = 0; j < n; ++ j) std::sort(entries.begin() + col_ptr[j], entries.begin() + col_ptr[j + 1]);
		for(size_t e = 0; e < nb; ++ e) { csc_row[e] = entries[e].first; csc_blk[e] = entries[e].second; }
	}
	// selected inversion: flops, and scratch (W = R11^-1 and later, in the same place, G = Z_JJ; T = one block row of the
	// W recursion; X = W R12). The supernodes with one diagonal block and a short structure run on the side lanes, each
	// lane with scratch of its own; every other supernode runs on the main stream and shares one set
	sc.selinv_flops = 0;
	sc.selinv_main_doubles = sc.selinv_lane_doubles = 0;
	for(size_t s = 0; s < ns; ++ s) {
		const double w = 6.0 * (sn.first[s + 1] - sn.first[s]), h = 6.0 * (sn.row_ptr[s + 1] - sn.row_ptr[s]);
		sc.selinv_flops += 2 * w * w * w / 3 + 2 * w * w * h + 2 * w * h * h;
		const size_t ld = sc.panel_ld[s], hp = round_up((size_t)h, SN_SEL_HP);
		const size_t need = std::max(ld * ld, hp * hp) + ld * (hp + SN_NB);
		size_t &slot = selinv_on_lane(ld, hp)? sc.selinv_lane_doubles : sc.selinv_main_doubles;
		slot = std::max(slot, need);
	}
	// updates s -> t with their relative-index maps
	sc.updates.clear();
	sc.upd_ptr.assign(ns + 1, 0);
	std::vector<uint32_t> cmap;
	for(size_t s = 0; s < ns; ++ s) {
		const size_t hb = sn.row_ptr[s + 1] - sn.row_ptr[s];
		const uint32_t *rows = hb? &sn.rows[sn.row_ptr[s]] : 0;
		size_t idx = 0;
		while(idx < hb) {
			const uint32_t t = sn.col_super[rows[idx]];
			size_t nJ = 1;
			while(idx + nJ < hb && sn.col_super[rows[idx + nJ]] == t) ++ nJ;
			SnodeUpdate u;
			u.s = (uint32_t)s; u.t = t;
			u.col0 = (uint32_t)(sc.panel_ld[s] + 6 * idx);
			u.M = (uint32_t)(6 * nJ);
			u.N = (uint32_t)(6 * (hb - idx) + 1);
			u.map_off = cmap.size();
			for(size_t q = idx; q < hb; ++ q)
				cmap.push_back(col_pos(t, rows[q]));
			cmap.push_back((uint32_t)(sc.panel_ld[t] + 6 * (sn.row_ptr[t + 1] - sn.row_ptr[t]))); // rhs column of t
			sc.updates.push_back(u);
			idx += nJ;
		}
		sc.upd_ptr[s + 1] = sc.updates.size();
	}

	cudaStream_t st = ctx->stream;
	sc.d_cmap.upload(cmap, st);
	sc.d_order.upload(sc.h_order, st);
	sc.d_rows.upload(sn.rows, st);
	sc.d_asm_dst.upload(asm_dst, st);
	sc.d_asm_ld.upload(asm_ld, st);
	sc.d_rhs_dst.upload(rhs_dst, st);
	sc.d_pad_off.upload(pad_off, st);
	sc.d_pad_ld.upload(pad_ld, st);
	sc.d_pad_n0.upload(pad_n0, st);
	sc.d_cam_diag.upload(cam_diag, st);
	sc.d_cam_ld.upload(cam_ld, st);
	sc.d_csc_ptr.upload(col_ptr, st);
	sc.d_csc_row.upload(csc_row, st);
	sc.d_csc_blk.upload(csc_blk, st);
	sc.d_L.resize(total);
	sc.d_Rinv.resize(n_rinv * SN_NB * SN_NB);
	sc.d_Rinv.zero(st); // the diagonal-block kernel writes upper triangles only
	sc.d_x.resize(n * 6);
	sc.d_part.resize(std::max<size_t>(sc.max_part, 1) * SupernodalChol::N_STREAMS);
	sc.d_info.resize(1 + n_rinv);
	sc.d_flag.resize(1);
	SPP_CUDA(cudaStreamSynchronize(st));
	if(getenv("SPP_SNODE_VERBOSE")) {
		size_t n_side = 0, n_look = 0, n_flow = 0, n_sel_lane = 0, max_ld = 0, max_h = 0, n_tile128 = 0;
		for(size_t s = 0; s < ns; ++ s) {
			const size_t ld = sc.panel_ld[s], h = 6 * (size_t)(sn.row_ptr[s + 1] - sn.row_ptr[s]);
			if(snode_on_side(ld)) ++ n_side; else if(snode_dataflow(ld)) ++ n_flow; else ++ n_look;
			n_sel_lane += selinv_on_lane(ld, round_up(h, SN_SEL_HP));
			max_ld = std::max(max_ld, ld);
			max_h = std::max(max_h, h);
		}
		for(const SnodeUpdate &u : sc.updates) n_tile128 += snode_update_tile128(u);
		fprintf(stderr, "[spp snode] n %zu, S blocks %zu, supernodes %zu, factor blocks %llu (exact %llu), panels %.2f GB, %.3e flops, %zu updates; "
			"supernodes on the side streams %zu, look-ahead %zu, dataflow %zu (ld >= %zu); largest ld %zu, largest h %zu; "
			"updates on 128x64 tiles %zu, on 64x64 tiles %zu; selected inversion on the side lanes %zu\n",
			n, nb, ns, (unsigned long long)sn.nnzb_factor, (unsigned long long)sn.nnzb_exact, total * 8e-9, sc.factor_flops,
			sc.updates.size(), n_side, n_look, n_flow, SN_DATAFLOW_MIN, max_ld, max_h, n_tile128, sc.updates.size() - n_tile128,
			n_sel_lane);
	}
	sc.sym_row = blk_row; sc.sym_col = blk_col; sc.sym_user_order = sc.user_order;
	sc.sym_world = ctx->world; sc.sym_rank = ctx->rank;
	sc.sym_kept = true;
	sc.valid = true;
}

// ---- device ----------------------------------------------------------------------------------------------

__device__ __forceinline__ void dmma884(double &d0, double &d1, double a, double b)
{
	asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
		: "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

__global__ void k_snode_pad_identity(size_t n_items, const uint64_t *__restrict__ off, const uint32_t *__restrict__ ld,
	const uint32_t *__restrict__ n0, double *__restrict__ L)
{
	const size_t it = blockIdx.x;
	if(it >= n_items) return;
	const size_t l = ld[it];
	double *P = L + off[it];
	for(size_t i = n0[it] + threadIdx.x; i < l; i += blockDim.x)
		P[i * l + i] = 1.0;
}

// thread per scalar of the compact block list
__global__ void k_snode_assemble(size_t n_vals, const double *__restrict__ Sblk, const uint64_t *__restrict__ dst,
	const uint32_t *__restrict__ ld, double *__restrict__ L)
{
	const size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(e >= n_vals) return;
	const size_t b = e / 36;
	const unsigned q = (unsigned)(e - b * 36), c = q / 6, r = q - c * 6;
	const uint64_t d = dst[b];
	const size_t l = ld[b];
	const bool tr = (d >> 63) != 0;
	double *P = L + (d & ~((uint64_t)1 << 63));
	P[tr? (size_t)r * l + c : (size_t)c * l + r] = Sblk[e];
}

__global__ void k_snode_assemble_rhs(size_t n_scalars, const double *__restrict__ b, const uint64_t *__restrict__ dst,
	double *__restrict__ L)
{
	const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(i >= n_scalars) return;
	L[dst[i / 6] + i % 6] = b[i];
}

// panel_t -= Ps[:, col0 + i]^T Ps[:, col0 + j], i < M, j < N, i <= j, scattered through cmap (block positions in panel
// t; rows of t are positions inside its own columns). Warp tile 32 x 32, DMMA m8n8k4, 3-stage cp.async pipeline over K.
template <int BM, int BN>
__global__ void __launch_bounds__((BM / 32) * (BN / 32) * 32) k_snode_update(const double *__restrict__ Ps, size_t ld_s,
	uint32_t col0, uint32_t max_col, uint32_t M, uint32_t N, uint32_t n_kt, double *__restrict__ Pt, size_t ld_t,
	const uint32_t *__restrict__ cmap)
{
	constexpr int WARPS_N = BN / 32, NT = (BM / 32) * (BN / 32) * 32;
	const uint32_t i0 = blockIdx.y * BM, j0 = blockIdx.x * BN;
	if(i0 > j0 + (BN - 1))
		return; // strictly below the diagonal of the update
	extern __shared__ double smem[];
	double (*As)[BM][SN_LDS] = reinterpret_cast<double (*)[BM][SN_LDS]>(smem);
	double (*Bs)[BN][SN_LDS] = reinterpret_cast<double (*)[BN][SN_LDS]>(smem + SN_STAGES * BM * SN_LDS);
	uint32_t *rpos = reinterpret_cast<uint32_t*>(smem + SN_STAGES * (BM + BN) * SN_LDS);
	uint32_t *cpos = rpos + BM;
	const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
	const int wi = (warp / WARPS_N) * 32, wj = (warp % WARPS_N) * 32;
	const int g = lane >> 2, t = lane & 3;

	for(int m = tid; m < BM; m += NT) {
		const uint32_t i = i0 + m;
		rpos[m] = (i < M)? cmap[i / 6] + i % 6 : 0xffffffffu;
	}
	for(int m = tid; m < BN; m += NT) {
		const uint32_t j = j0 + m;
		cpos[m] = (j < N)? cmap[j / 6] + j % 6 : 0xffffffffu;
	}

	auto stage_load = [&](int st, int kc) {
		for(int idx = tid; idx < BM * 8; idx += NT) {
			const int m = idx >> 3, q = idx & 7;
			const uint32_t c = min(col0 + i0 + m, max_col);
			__pipeline_memcpy_async(&As[st][m][q * 2], Ps + (size_t)c * ld_s + kc * SN_BK + q * 2, 16);
		}
		for(int idx = tid; idx < BN * 8; idx += NT) {
			const int m = idx >> 3, q = idx & 7;
			const uint32_t c = min(col0 + j0 + m, max_col);
			__pipeline_memcpy_async(&Bs[st][m][q * 2], Ps + (size_t)c * ld_s + kc * SN_BK + q * 2, 16);
		}
	};

	double acc[4][4][2];
	const int KT = (int)n_kt;
	#pragma unroll
	for(int s = 0; s < SN_STAGES - 1; ++ s) {
		if(s < KT) stage_load(s, s);
		__pipeline_commit();
	}
	// the accumulators start from the target entries (gathered through the map while the pipeline fills) and the A
	// fragments are negated below, so the epilogue is a plain scattered store instead of a read-modify-write
	__syncthreads(); // rpos / cpos
	#pragma unroll
	for(int a = 0; a < 4; ++ a) {
		const int mi = wi + a * 8 + g;
		const uint32_t rp = rpos[mi], i = i0 + mi;
		#pragma unroll
		for(int b = 0; b < 4; ++ b) {
			#pragma unroll
			for(int h = 0; h < 2; ++ h) {
				const int mj = wj + b * 8 + 2 * t + h;
				const uint32_t cp = cpos[mj];
				const bool ok = rp != 0xffffffffu && cp != 0xffffffffu && i <= j0 + mj;
				acc[a][b][h] = ok? Pt[(size_t)cp * ld_t + rp] : 0.0;
			}
		}
	}
	for(int kt = 0; kt < KT; ++ kt) {
		__pipeline_wait_prior(SN_STAGES - 2);
		__syncthreads();
		if(kt + SN_STAGES - 1 < KT)
			stage_load((kt + SN_STAGES - 1) % SN_STAGES, kt + SN_STAGES - 1);
		__pipeline_commit();
		const int st = kt % SN_STAGES;
		#pragma unroll
		for(int k4 = 0; k4 < SN_BK; k4 += 4) {
			double fa[4], fb[4];
			#pragma unroll
			for(int a = 0; a < 4; ++ a)
				fa[a] = -As[st][wi + a * 8 + g][k4 + t];
			#pragma unroll
			for(int b = 0; b < 4; ++ b)
				fb[b] = Bs[st][wj + b * 8 + g][k4 + t];
			#pragma unroll
			for(int a = 0; a < 4; ++ a)
				#pragma unroll
				for(int b = 0; b < 4; ++ b)
					dmma884(acc[a][b][0], acc[a][b][1], fa[a], fb[b]);
		}
	}
	__pipeline_wait_prior(0);
	#pragma unroll
	for(int a = 0; a < 4; ++ a) {
		const int mi = wi + a * 8 + g;
		const uint32_t rp = rpos[mi];
		if(rp == 0xffffffffu) continue;
		const uint32_t i = i0 + mi;
		#pragma unroll
		for(int b = 0; b < 4; ++ b) {
			#pragma unroll
			for(int h = 0; h < 2; ++ h) {
				const int mj = wj + b * 8 + 2 * t + h;
				const uint32_t cp = cpos[mj];
				if(cp != 0xffffffffu && i <= j0 + mj)
					Pt[(size_t)cp * ld_t + rp] = acc[a][b][h];
			}
		}
	}
}

template <int BM, int BN>
constexpr size_t snode_update_smem() { return (size_t)SN_STAGES * (BM + BN) * SN_LDS * sizeof(double) + (BM + BN) * sizeof(uint32_t); }

// backward solve, structure part: part[chunk][r] = sum over the chunk's structure columns of P[r, ld + c] x[row(c)]
__global__ void __launch_bounds__(128) k_snode_gemv(const double *__restrict__ P, size_t ld, size_t h /* scalar columns */,
	const uint32_t *__restrict__ rows /* block rows of the structure */, const double *__restrict__ x, double *__restrict__ part)
{
	__shared__ double xs[SN_GEMV_COLS];
	const size_t r = blockIdx.x * (size_t)128 + threadIdx.x;
	const size_t c0 = blockIdx.y * (size_t)SN_GEMV_COLS, c1 = min(c0 + SN_GEMV_COLS, h);
	for(size_t c = c0 + threadIdx.x; c < c1; c += 128)
		xs[c - c0] = x[(size_t)rows[c / 6] * 6 + c % 6];
	__syncthreads();
	const double *p = P + (ld + c0) * ld + r;
	double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
	const size_t nc = c1 - c0;
	size_t c = 0;
	for(; c + 8 <= nc; c += 8) { // eight independent loads in flight
		const double a0 = p[c * ld], a1 = p[(c + 1) * ld], a2 = p[(c + 2) * ld], a3 = p[(c + 3) * ld];
		const double a4 = p[(c + 4) * ld], a5 = p[(c + 5) * ld], a6 = p[(c + 6) * ld], a7 = p[(c + 7) * ld];
		s0 += a0 * xs[c]; s1 += a1 * xs[c + 1]; s2 += a2 * xs[c + 2]; s3 += a3 * xs[c + 3];
		s0 += a4 * xs[c + 4]; s1 += a5 * xs[c + 5]; s2 += a6 * xs[c + 6]; s3 += a7 * xs[c + 7];
	}
	for(; c < nc; ++ c)
		s0 += p[c * ld] * xs[c];
	part[blockIdx.y * ld + r] = (s0 + s1) + (s2 + s3);
}

__global__ void k_snode_gemv_reduce(size_t ld, size_t n_chunks, const double *__restrict__ part, double *__restrict__ y)
{
	const size_t r = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(r >= ld) return;
	double s = 0;
	for(size_t k = 0; k < n_chunks; ++ k)
		s += part[k * ld + r];
	y[r] -= s;
}

// x of the supernode's own columns: into the permuted solution (for the descendants) and, un-permuted, into dx
// (several ranks: the x of a shared supernode is the same everywhere and the increments are summed over the ranks at the
// end, so only rank 0 writes it to dx: b_write_dx)
__global__ void k_snode_store_x(size_t w, size_t first_scalar, const double *__restrict__ y, const uint32_t *__restrict__ order,
	double *__restrict__ x, double *__restrict__ dx, bool b_write_dx)
{
	const size_t r = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(r >= w) return;
	const double v = y[r];
	const size_t j = first_scalar + r;
	x[j] = v;
	if(b_write_dx)
		dx[(size_t)order[j / 6] * 6 + j % 6] = v;
}

// the status of the factorisation must be the same on every rank (a non-positive pivot in a subtree is seen by its owner
// only): flag = (info != 0), summed over the ranks, then info = its own value or "somewhere" (1)
__global__ void k_snode_info_to_flag(const int *__restrict__ info, double *__restrict__ flag)
{
	*flag = (*info != 0)? 1.0 : 0.0;
}
__global__ void k_snode_flag_to_info(const double *__restrict__ flag, int *__restrict__ info)
{
	if(*flag > 0 && *info == 0) *info = 1;
}

// ---- numeric phase ----------------------------------------------------------------------------------------

// Numeric factorisation, enqueued: assembly of d_Sblk (compact 6x6 block list of S in the order of the list given to
// snode_symbolic) and of d_b (reduced right-hand side, camera order; null: no right-hand side, the rhs columns stay zero)
// into the panels, the elimination-order loop with its side streams (joined back into the context's stream), and the
// status in d_info[0] (the same on every rank).
void snode_factor(spp_ctx *ctx, const double *d_Sblk, const double *d_b)
{
	SupernodalChol &sc = ctx->snode;
	if(!sc.valid)
		throw invalid_error("supernodal Cholesky: no symbolic factorisation");
	static bool attr_done_on[64] = {false}; // the attribute belongs to the (kernel, device) pair
	bool &attr_done = attr_done_on[(ctx->device >= 0 && ctx->device < 64)? ctx->device : 0];
	if(!attr_done) {
		SPP_CUDA(cudaFuncSetAttribute(k_snode_update<64, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)snode_update_smem<64, 64>()));
		SPP_CUDA(cudaFuncSetAttribute(k_snode_update<128, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)snode_update_smem<128, 64>()));
		attr_done = true;
	}
	const Supernodes &sn = sc.sn;
	const size_t ns = sn.n_super(), n = sc.n;
	cudaStream_t st = ctx->stream;
	if(!sc.side[0]) {
		int prio_lo = 0, prio_hi = 0;
		SPP_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
		for(int i = 0; i < SupernodalChol::N_STREAMS; ++ i)
			SPP_CUDA(cudaStreamCreateWithPriority(&sc.side[i], cudaStreamNonBlocking, prio_lo));
	}
	if(sc.ev_factor.size() < ns) {
		const size_t old = sc.ev_factor.size();
		sc.ev_factor.resize(ns); sc.ev_target.resize(ns); sc.ev_x.resize(ns);
		for(size_t i = old; i < ns; ++ i) {
			SPP_CUDA(cudaEventCreateWithFlags(&sc.ev_factor[i], cudaEventDisableTiming));
			SPP_CUDA(cudaEventCreateWithFlags(&sc.ev_target[i], cudaEventDisableTiming));
			SPP_CUDA(cudaEventCreateWithFlags(&sc.ev_x[i], cudaEventDisableTiming));
		}
	}
	std::vector<char> pending(ns, 0); // updates into panel t are in flight on its side stream
	double *L = sc.d_L.p();
	sc.d_L.zero(st);
	SPP_CUDA(cudaMemsetAsync(sc.d_info.p(), 0, sc.d_info.size() * sizeof(int), st));
	if(sc.d_pad_off.size()) {
		k_snode_pad_identity<<<(unsigned)sc.d_pad_off.size(), 128, 0, st>>>(sc.d_pad_off.size(), sc.d_pad_off.p(), sc.d_pad_ld.p(),
			sc.d_pad_n0.p(), L);
		LAUNCH_CHECK(ctx);
	}
	k_snode_assemble<<<n_blocks(sc.n_s_blocks * 36, 256), 256, 0, st>>>(sc.n_s_blocks * 36, d_Sblk, sc.d_asm_dst.p(), sc.d_asm_ld.p(), L);
	LAUNCH_CHECK(ctx);
	if(d_b) {
		k_snode_assemble_rhs<<<n_blocks(n * 6, 256), 256, 0, st>>>(n * 6, d_b, sc.d_rhs_dst.p(), L);
		LAUNCH_CHECK(ctx);
	}
	const bool dist = sc.distributed && ctx->world > 1;
	if(dist && ctx->rank != 0) { // the shared panels are summed over the ranks: S, the right-hand side and the identity
		for(size_t s = 0; s < ns; ++ s) { // padding come from rank 0 alone, the others contribute their subtrees' updates
			if(sc.owner[s] < 0)
				SPP_CUDA(cudaMemsetAsync(L + sc.panel_off[s], 0, (size_t)sc.panel_ld[s] * sc.panel_cols[s] * sizeof(double), st));
		}
	}
	char assembled_seen[SupernodalChol::N_STREAMS] = {0};
	int side_used[SupernodalChol::N_STREAMS] = {0};
	SPP_CUDA(cudaEventRecord(sc.ev_x[0], st)); // "panels assembled" (the backward solve re-records ev_x later)
	// factorisation, elimination order (a postorder: every descendant of t precedes t)
	auto factor_and_update = [&](size_t s) {
		double *Ps = L + sc.panel_off[s];
		const size_t ld = sc.panel_ld[s], cols = sc.panel_cols[s];
		// a supernode with a single diagonal block is factored on the side stream that carries the updates into it (no
		// event needed: same stream), so the many narrow supernodes of the lower tree levels run side by side; the wide
		// ones use the look-ahead panel factorisation on the main stream
		const bool on_side = snode_on_side(ld);
		cudaStream_t sf = on_side? sc.side[s % SupernodalChol::N_STREAMS] : st;
		if(on_side) {
			if(!assembled_seen[s % SupernodalChol::N_STREAMS]) { // the panels were assembled on the main stream
				SPP_CUDA(cudaStreamWaitEvent(sf, sc.ev_x[0], 0));
				assembled_seen[s % SupernodalChol::N_STREAMS] = 1;
			}
			dense_chol_factor_single_panel(ctx, sf, Ps, cols, sc.d_Rinv.p() + (size_t)sc.rinv_first[s] * SN_NB * SN_NB, sc.d_info.p());
		} else {
			if(pending[s]) // every update into this panel went to one side stream, in elimination order
				SPP_CUDA(cudaStreamWaitEvent(st, sc.ev_target[s], 0));
			// wide supernodes: the persistent dataflow factorisation (one kernel, no read-modify-write passes over the panel)
			if(snode_dataflow(ld) && dense_chol_dataflow_enabled())
				dense_chol_factor_dataflow(ctx, Ps, ld, cols, sc.d_Rinv.p() + (size_t)sc.rinv_first[s] * SN_NB * SN_NB, sc.d_info.p());
			else
				dense_chol_factor_panel(ctx, Ps, ld, cols, sc.d_Rinv.p() + (size_t)sc.rinv_first[s] * SN_NB * SN_NB, sc.d_info.p());
		}
		if(sc.upd_ptr[s + 1] > sc.upd_ptr[s] || on_side)
			SPP_CUDA(cudaEventRecord(sc.ev_factor[s], sf));
		if(on_side)
			side_used[s % SupernodalChol::N_STREAMS] = (int)s + 1; // joined before the backward solve
		const size_t w = 6 * (size_t)(sn.first[s + 1] - sn.first[s]);
		const uint32_t n_kt = (uint32_t)(round_up(w, SN_BK) / SN_BK);
		for(uint64_t q = sc.upd_ptr[s]; q < sc.upd_ptr[s + 1]; ++ q) {
			const SnodeUpdate &u = sc.updates[q];
			double *Pt = L + sc.panel_off[u.t];
			cudaStream_t su = sc.side[u.t % SupernodalChol::N_STREAMS];
			SPP_CUDA(cudaStreamWaitEvent(su, sc.ev_factor[s], 0));
			if(snode_update_tile128(u)) {
				dim3 grid((u.N + 63) / 64, (u.M + 127) / 128);
				k_snode_update<128, 64><<<grid, 256, snode_update_smem<128, 64>(), su>>>(Ps, ld, u.col0, (uint32_t)(cols - 1), u.M, u.N,
					n_kt, Pt, sc.panel_ld[u.t], sc.d_cmap.p() + u.map_off);
			} else {
				dim3 grid((u.N + 63) / 64, (u.M + 63) / 64);
				k_snode_update<64, 64><<<grid, 128, snode_update_smem<64, 64>(), su>>>(Ps, ld, u.col0, (uint32_t)(cols - 1), u.M, u.N,
					n_kt, Pt, sc.panel_ld[u.t], sc.d_cmap.p() + u.map_off);
			}
			LAUNCH_CHECK(ctx);
			SPP_CUDA(cudaEventRecord(sc.ev_target[u.t], su));
			pending[u.t] = 1;
		}
	};
	if(!dist) {
		for(size_t s = 0; s < ns; ++ s)
			factor_and_update(s);
	} else {
		// this rank's subtrees first (their updates reach their own panels and the shared ones) ...
		for(size_t s = 0; s < ns; ++ s)
			if(sc.owner[s] == ctx->rank) factor_and_update(s);
		// ... then the shared panels are summed over the ranks ...
		for(size_t s = 0; s < ns; ++ s) {
			if(sc.owner[s] >= 0) continue;
			if(pending[s]) {
				SPP_CUDA(cudaStreamWaitEvent(st, sc.ev_target[s], 0));
				pending[s] = 0;
			}
		}
		for(size_t s = 0; s < ns; ++ s)
			if(sc.owner[s] < 0) allreduce_device(ctx, L + sc.panel_off[s], (size_t)sc.panel_ld[s] * sc.panel_cols[s]);
		// side streams that factor narrow shared supernodes wait for the sums, not just for the assembly
		SPP_CUDA(cudaEventRecord(sc.ev_x[0], st));
		for(int i = 0; i < SupernodalChol::N_STREAMS; ++ i) assembled_seen[i] = 0;
		// ... and every rank factors the top of the tree
		for(size_t s = 0; s < ns; ++ s)
			if(sc.owner[s] < 0) factor_and_update(s);
	}
	for(int i = 0; i < SupernodalChol::N_STREAMS; ++ i) { // supernodes factored on the side streams (roots among them)
		if(side_used[i])
			SPP_CUDA(cudaStreamWaitEvent(st, sc.ev_factor[side_used[i] - 1], 0));
	}
	if(dist) { // one status for all ranks; the increments of the subtrees are summed at the end: start from zero
		k_snode_info_to_flag<<<1, 1, 0, st>>>(sc.d_info.p(), sc.d_flag.p());
		LAUNCH_CHECK(ctx);
		allreduce_device(ctx, sc.d_flag.p(), 1);
		k_snode_flag_to_info<<<1, 1, 0, st>>>(sc.d_flag.p(), sc.d_info.p());
		LAUNCH_CHECK(ctx);
	}
}

// d_Sblk: compact 6x6 block list of S in the order of the list given to snode_symbolic; d_b: reduced right-hand side
// (camera order); d_dx: camera increment out (camera order; may alias d_b). Returns SPP_OK / SPP_NOT_POSDEF.
int snode_factor_solve(spp_ctx *ctx, const double *d_Sblk, const double *d_b, double *d_dx)
{
	snode_factor(ctx, d_Sblk, d_b);
	SupernodalChol &sc = ctx->snode;
	const Supernodes &sn = sc.sn;
	const size_t ns = sn.n_super(), n = sc.n;
	cudaStream_t st = ctx->stream;
	double *L = sc.d_L.p();
	const bool dist = sc.distributed && ctx->world > 1;
	if(dist) // the increments of the subtrees are summed at the end: start from zero
		SPP_CUDA(cudaMemsetAsync(d_dx, 0, n * 6 * sizeof(double), st)); // (d_b, which d_dx may alias, went into the panels)
	SPP_CUDA(cudaEventRecord(sc.ev_factor[ns - 1], st)); // "factorisation complete"
	// backward solve, root to leaves; y_s sits in the rhs column of panel s. A supernode needs the x of its ancestors
	// only: supernodes go round-robin to the side streams and wait for their parent's event (which implies the
	// grandparents'), so independent subtrees are solved side by side
	for(size_t ss = ns; ss > 0; -- ss) {
		const size_t s = ss - 1;
		if(dist && sc.owner[s] >= 0 && sc.owner[s] != ctx->rank)
			continue; // another rank's subtree
		double *Ps = L + sc.panel_off[s];
		const size_t ld = sc.panel_ld[s], w = 6 * (size_t)(sn.first[s + 1] - sn.first[s]);
		const size_t h = 6 * (size_t)(sn.row_ptr[s + 1] - sn.row_ptr[s]);
		double *y = Ps + (ld + h) * ld;
		const int lane = int(s % SupernodalChol::N_STREAMS);
		cudaStream_t sb = sc.side[lane];
		double *part = sc.d_part.p() + (size_t)lane * std::max<size_t>(sc.max_part, 1);
		if(sn.parent[s] != 0xffffffffu)
			SPP_CUDA(cudaStreamWaitEvent(sb, sc.ev_x[sn.parent[s]], 0));
		else
			SPP_CUDA(cudaStreamWaitEvent(sb, sc.ev_factor[ns - 1], 0)); // the factorisation is complete (recorded above)
		if(h) {
			const size_t n_chunks = (h + SN_GEMV_COLS - 1) / SN_GEMV_COLS;
			k_snode_gemv<<<dim3((unsigned)(ld / 128), (unsigned)n_chunks), 128, 0, sb>>>(Ps, ld, h, sc.d_rows.p() + sn.row_ptr[s],
				sc.d_x.p(), part);
			LAUNCH_CHECK(ctx);
			k_snode_gemv_reduce<<<n_blocks(ld, 128), 128, 0, sb>>>(ld, n_chunks, part, y);
			LAUNCH_CHECK(ctx);
		}
		dense_chol_backsolve_panel(ctx, sb, Ps, ld, sc.d_Rinv.p() + (size_t)sc.rinv_first[s] * SN_NB * SN_NB, y,
			sc.d_info.p() + 1 + sc.rinv_first[s]);
		k_snode_store_x<<<n_blocks(w, 128), 128, 0, sb>>>(w, 6 * (size_t)sn.first[s], y, sc.d_order.p(), sc.d_x.p(), d_dx,
			!dist || sc.owner[s] >= 0 || ctx->rank == 0);
		LAUNCH_CHECK(ctx);
		SPP_CUDA(cudaEventRecord(sc.ev_x[s], sb));
	}
	for(int i = 0; i < SupernodalChol::N_STREAMS; ++ i) { // join the side streams
		SPP_CUDA(cudaEventRecord(sc.ev_target[i % ns], sc.side[i]));
		SPP_CUDA(cudaStreamWaitEvent(st, sc.ev_target[i % ns], 0));
	}
	if(dist)
		allreduce_device(ctx, d_dx, n * 6); // every rank needs all the camera increments
	if(ctx->async_mode && ctx->async_info) { // the caller synchronises later and reads the status there
		SPP_CUDA(cudaMemcpyAsync(ctx->async_info, sc.d_info.p(), sizeof(int), cudaMemcpyDeviceToHost, st));
		return SPP_OK;
	}
	ctx->h_scalars.resize(16);
	int *h_info = reinterpret_cast<int*>(ctx->h_scalars.p());
	SPP_CUDA(cudaMemcpyAsync(h_info, sc.d_info.p(), sizeof(int), cudaMemcpyDeviceToHost, st));
	SPP_CUDA(cudaStreamSynchronize(st));
	return (*h_info == 0)? SPP_OK : SPP_NOT_POSDEF;
}

} // namespace spp
