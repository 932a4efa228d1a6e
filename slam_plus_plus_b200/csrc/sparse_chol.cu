// sparse_chol.cu -- stage 3 of the hot path for block-sparse systems (pose graphs; the reference's fallback for a
// reduced camera system that is too large to be dense): fill-reducing ordering, symbolic analysis and the numeric
// block Cholesky with its two triangular solves.
//
// Reference functions replaced (SURVEY 8(a) row a15): CLinearSolver_UberBlock::SymbolicDecomposition_Blocky /
// Solve_PosDef_Blocky (include/slam/LinearSolver_UberBlock.h:272-296, 312-426): AMD ordering of the block structure
// (CMatrixOrdering::p_BlockOrdering, src/slam/OrderingMagic.cpp:701-1033), Permute_UpperTriangular_To, the elimination
// tree (src/slam/BlockMatrix.cpp:9403), the up-looking block Cholesky CholeskyOf_FBS
// (include/slam/BlockMatrixFBS.inl:2341-2513) and UpperTriangular[Transpose]_Solve_FBS (:2136-2275).
//
// The reference factors column by column on one thread (ereach + dense block kernels). Here the host does the
// integer work once per structure -- ordering (given by the caller, e.g. the reference's own AMD through the
// adapter, or the approximate minimum degree of block_ordering.cpp), elimination tree, column structures of the factor, and for
// every block L(i, j) the list of block pairs (L(i, k), L(j, k)) that update it -- and the device runs the numeric
// phase level by level of the elimination tree: all columns of a level are independent.
//   k_sparse_chol<B>    per level: (a) diagonal blocks: D = A_jj - sum_k L_jk L_jk^T, Cholesky + inverse of the
//                       B x B block, forward solve y_j; barrier; (b) off-diagonal blocks L_ij = (A_ij - sum_k L_ik
//                       L_jk^T) L_jj^-T; barrier. One warp per block, lanes over the block's elements.
//   k_sparse_backsolve<B> levels in reverse: x_j = L_jj^-T (y_j - sum_i L_ij^T x_i)
// The wide levels run as a cooperative grid (grid-wide barrier), the narrow tail of the tree on a single CTA
// (__syncthreads), so a chain-like tree does not pay a grid barrier per column.
// The factor is the lower-triangular L = R^T of the reference's upper factor R; its block pattern is the same.

#include "spp_ctx.h"
#include <cooperative_groups.h>
#include <algorithm>
#include <numeric>
#include <stdlib.h>

namespace cg = cooperative_groups;

namespace spp {

size_t dense_chol_ld(size_t n);
size_t dense_chol_storage(size_t n);
int dense_chol_solve_device(spp_ctx *ctx, double *A, size_t n, double *d_rhs_x);

#define LAUNCH_CHECK(ctx) do { ++ (ctx)->n_launches; SPP_CUDA(cudaGetLastError()); } while(0)
#define SC_WARPS 8
#define SC_ROOT_MAX_SCALARS 6144 // the dense root front is at most this wide

// ---- host: symbolic analysis ---------------------------------------------------------------------------

// Input: upper block structure in the caller's order (CSC, rows ascending, diagonal present), the ordering
// order[new] = old. Builds everything the numeric kernels need and uploads it; owner (SC_OWNER_SLOT / SC_OWNER_POSE)
// is recorded once the analysis is complete.
void sparse_chol_symbolic(spp_ctx *ctx, int owner, size_t n, size_t B, const uint64_t *col_ptr, const uint64_t *row_idx,
	const uint64_t *p_order_in)
{
	SparseChol &sc = ctx->schol;
	sc.valid = false;
	sc.owner = SC_OWNER_NONE;
	sc.n = n; sc.B = B;
	if(n >= 0x7fffffffu)
		throw invalid_error("sparse Cholesky: too many block columns for 32-bit indices");
	// ordering
	sc.h_order.resize(n);
	if(p_order_in) {
		std::vector<char> seen(n, 0);
		for(size_t i = 0; i < n; ++ i) {
			if(p_order_in[i] >= n || seen[p_order_in[i]])
				throw invalid_error("sparse Cholesky: the ordering is not a permutation");
			seen[p_order_in[i]] = 1;
			sc.h_order[i] = (uint32_t)p_order_in[i];
		}
	} else // approximate minimum degree, the reference's permutation (amd_exact.cpp)
		amd_exact_ordering(n, col_ptr, row_idx, sc.h_order);
	std::vector<uint32_t> inv(n);
	for(size_t i = 0; i < n; ++ i)
		inv[sc.h_order[i]] = (uint32_t)i;

	// permuted LOWER pattern by column, with the source of every block in the caller's value array
	const size_t BB = B * B;
	std::vector<std::vector<std::pair<uint32_t, int64_t> > > acol(n); // (row, +/-(source block index + 1)); negative = transposed
	{
		uint64_t blk = 0;
		for(size_t c = 0; c < n; ++ c) {
			for(uint64_t k = col_ptr[c]; k < col_ptr[c + 1]; ++ k, ++ blk) {
				const size_t r = row_idx[k];
				if(r > c || r >= n)
					throw invalid_error("sparse Cholesky: the matrix must be upper block-triangular");
				const uint32_t pr = inv[r], pc = inv[c];
				// the block A(r, c), r <= c, lands at (pr, pc); the lower factor wants row >= column:
				// A(r, c) = A(c, r)^T, so the lower entry (max, min) is the block itself transposed unless pr >= pc
				if(pr >= pc)
					acol[pc].push_back(std::make_pair(pr, (int64_t)(blk + 1)));      // lower(pr, pc) = A(r, c) as stored
				else
					acol[pr].push_back(std::make_pair(pc, -(int64_t)(blk + 1)));     // lower(pc, pr) = A(r, c)^T
			}
		}
		sc.n_a_blocks = blk;
	}
	for(size_t j = 0; j < n; ++ j) {
		std::sort(acol[j].begin(), acol[j].end());
		if(acol[j].empty() || acol[j][0].first != j)
			throw invalid_error("sparse Cholesky: missing diagonal block");
	}
	// elimination tree and column structures of L: struct(j) = pattern(A_j) U (struct(children) \ {child})
	std::vector<uint32_t> parent(n, 0xffffffffu);
	std::vector<std::vector<uint32_t> > lcol(n);
	{
		std::vector<std::vector<uint32_t> > children(n);
		std::vector<uint32_t> tmp;
		for(size_t j = 0; j < n; ++ j) {
			std::vector<uint32_t> &s = lcol[j];
			for(size_t q = 0; q < acol[j].size(); ++ q)
				s.push_back(acol[j][q].first);
			for(size_t q = 0; q < children[j].size(); ++ q) {
				const std::vector<uint32_t> &cs = lcol[children[j][q]];
				tmp.clear();
				std::set_union(s.begin(), s.end(), cs.begin() + 1, cs.end(), std::back_inserter(tmp)); // skip the child's diagonal
				// entries < j cannot occur: a child's structure below its diagonal starts at its parent = j
				s.swap(tmp);
			}
			if(s.size() > 1) {
				parent[j] = s[1];
				children[s[1]].push_back((uint32_t)j);
			}
		}
	}
	// block numbering: column by column, the diagonal block first
	std::vector<uint64_t> lptr(n + 1, 0);
	for(size_t j = 0; j < n; ++ j)
		lptr[j + 1] = lptr[j] + lcol[j].size();
	const size_t nb = lptr[n];
	std::vector<uint32_t> lrow(nb), lcolof(nb);
	for(size_t j = 0; j < n; ++ j) {
		std::copy(lcol[j].begin(), lcol[j].end(), lrow.begin() + lptr[j]);
		std::fill(lcolof.begin() + lptr[j], lcolof.begin() + lptr[j + 1], (uint32_t)j);
	}
	// source of every L block in A (0 = fill-in)
	std::vector<int64_t> src(nb, 0);
	for(size_t j = 0; j < n; ++ j) {
		size_t q = 0;
		for(size_t a = 0; a < acol[j].size(); ++ a) {
			while(lcol[j][q] != acol[j][a].first) ++ q;
			src[lptr[j] + q] = acol[j][a].second;
		}
	}
	// row structure: for every row j, the blocks L(j, k), k < j, in ascending k
	std::vector<uint64_t> rptr(n + 1, 0);
	for(size_t b = 0; b < nb; ++ b)
		if(lrow[b] != lcolof[b]) ++ rptr[lrow[b] + 1];
	for(size_t j = 0; j < n; ++ j)
		rptr[j + 1] += rptr[j];
	std::vector<uint32_t> rblk(rptr[n]);
	{
		std::vector<uint64_t> fill(rptr.begin(), rptr.end() - 1);
		for(size_t b = 0; b < nb; ++ b) // ascending block index = ascending column
			if(lrow[b] != lcolof[b]) rblk[fill[lrow[b]] ++] = (uint32_t)b;
	}
	// update lists: block (i, j) <- pairs (L(i, k), L(j, k)) for k in rowstruct(j) with L(i, k) present
	std::vector<uint64_t> uptr(nb + 1, 0);
	std::vector<uint32_t> ua, ub;
	for(size_t j = 0; j < n; ++ j) {
		for(uint64_t b = lptr[j]; b < lptr[j + 1]; ++ b) {
			const uint32_t i = lrow[b];
			for(uint64_t q = rptr[j]; q < rptr[j + 1]; ++ q) {
				const uint32_t bjk = rblk[q], k = lcolof[bjk];
				uint32_t bik;
				if(i == j)
					bik = bjk;
				else {
					std::vector<uint32_t>::const_iterator it = std::lower_bound(lcol[k].begin(), lcol[k].end(), i);
					if(it == lcol[k].end() || *it != i)
						continue;
					bik = (uint32_t)(lptr[k] + (it - lcol[k].begin()));
				}
				ua.push_back(bik);
				ub.push_back(bjk);
			}
			uptr[b + 1] = ua.size();
		}
	}
	// The top of the elimination tree is a long chain of wide columns (the top-level separators): level by level it
	// costs a barrier per column. Columns t0 .. n-1 (everything from the first column of a narrow level on) are
	// instead assembled into ONE dense front and factored by the dense DMMA Cholesky (dense_chol.cu).
	std::vector<uint32_t> level(n, 0);
	uint32_t n_levels_all = 0;
	for(size_t j = 0; j < n; ++ j) {
		if(parent[j] != 0xffffffffu)
			level[parent[j]] = std::max(level[parent[j]], level[j] + 1);
		n_levels_all = std::max(n_levels_all, level[j] + 1);
	}
	// root set: the columns of the narrow top levels (upward closed in the tree: the row structure of a root column
	// lies in the root set); ridx = dense index of a root column
	std::vector<uint32_t> ridx(n, 0xffffffffu);
	size_t m = 0;
	uint32_t narrow = n_levels_all; // first level of the narrow tail
	{
		std::vector<uint32_t> width(n_levels_all, 0);
		for(size_t j = 0; j < n; ++ j) ++ width[level[j]];
		while(narrow > 0 && width[narrow - 1] <= 2 * SC_WARPS) -- narrow;
		size_t cnt = 0;
		for(size_t j = 0; j < n; ++ j) cnt += level[j] >= narrow;
		if(n_levels_all - narrow < 8 || cnt * B > SC_ROOT_MAX_SCALARS || getenv("SPP_SPARSE_NO_ROOT"))
			narrow = n_levels_all; // not worth it / too large: everything level by level
		for(size_t j = 0; j < n; ++ j)
			if(level[j] >= narrow) ridx[j] = (uint32_t)m ++;
	}
	sc.n_root = m;
	// levels over the other columns
	const uint32_t n_levels = narrow;
	std::vector<uint32_t> lvl_ptr(n_levels + 1, 0), lvl_cols(n - m);
	for(size_t j = 0; j < n; ++ j) if(level[j] < narrow) ++ lvl_ptr[level[j] + 1];
	for(uint32_t l = 0; l < n_levels; ++ l) lvl_ptr[l + 1] += lvl_ptr[l];
	{
		std::vector<uint32_t> fill(lvl_ptr.begin(), lvl_ptr.end() - 1);
		for(size_t j = 0; j < n; ++ j) if(level[j] < narrow) lvl_cols[fill[level[j]] ++] = (uint32_t)j;
	}
	// off-diagonal blocks grouped by the level of their column (for the one-warp-per-block phase)
	std::vector<uint64_t> lvl_off_ptr(n_levels + 1, 0);
	std::vector<uint32_t> lvl_off_blk;
	lvl_off_blk.reserve(nb - n);
	for(uint32_t l = 0; l < n_levels; ++ l) {
		for(uint32_t q = lvl_ptr[l]; q < lvl_ptr[l + 1]; ++ q) {
			const uint32_t j = lvl_cols[q];
			for(uint64_t b = lptr[j] + 1; b < lptr[j + 1]; ++ b)
				lvl_off_blk.push_back((uint32_t)b);
		}
		lvl_off_ptr[l + 1] = lvl_off_blk.size();
	}
	// the tail of what is left (levels narrower than one CTA's warps) runs on a single CTA
	uint32_t tail = n_levels;
	while(tail > 0 && lvl_ptr[tail] - lvl_ptr[tail - 1] <= SC_WARPS && lvl_off_ptr[tail] - lvl_off_ptr[tail - 1] <= 4 * SC_WARPS)
		-- tail;
	// root front: its blocks with the update pairs that come from the other columns, and the row lists of the root
	// rows restricted to the other columns
	std::vector<uint32_t> root_blk, root_ua, root_ub, root_rblk, root_cols;
	std::vector<uint64_t> root_uptr(1, 0), root_rptr(1, 0);
	for(size_t j = 0; j < n; ++ j) {
		if(ridx[j] == 0xffffffffu)
			continue;
		root_cols.push_back((uint32_t)j);
		for(uint64_t b = lptr[j]; b < lptr[j + 1]; ++ b) {
			root_blk.push_back((uint32_t)b);
			for(uint64_t q = uptr[b]; q < uptr[b + 1]; ++ q) {
				if(ridx[lcolof[ub[q]]] == 0xffffffffu) {
					root_ua.push_back(ua[q]);
					root_ub.push_back(ub[q]);
				}
			}
			root_uptr.push_back(root_ua.size());
		}
		for(uint64_t q = rptr[j]; q < rptr[j + 1]; ++ q)
			if(ridx[lcolof[rblk[q]]] == 0xffffffffu) root_rblk.push_back(rblk[q]);
		root_rptr.push_back(root_rblk.size());
	}
	sc.h_ridx = ridx;
	sc.n_levels = n_levels;
	sc.tail_level = tail;
	sc.n_l_blocks = nb;
	sc.h_lptr.assign(lptr.begin(), lptr.end());
	sc.h_lrow = lrow;
	sc.h_parent = parent;

	cudaStream_t st = ctx->stream;
	std::vector<uint32_t> perm_scalar_src(n); // new position -> old block column
	sc.d_order.upload(sc.h_order, st);
	sc.d_lptr.upload(lptr, st);
	sc.d_lrow.upload(lrow, st);
	sc.d_lcolof.upload(lcolof, st);
	sc.d_src.upload(src, st);
	sc.d_rptr.upload(rptr, st);
	sc.d_rblk.upload(rblk, st);
	sc.d_uptr.upload(uptr, st);
	sc.d_ua.upload(ua, st);
	sc.d_ub.upload(ub, st);
	sc.d_lvl_ptr.upload(lvl_ptr, st);
	sc.d_lvl_cols.upload(lvl_cols, st);
	sc.d_lvl_off_ptr.upload(lvl_off_ptr, st);
	sc.d_lvl_off_blk.upload(lvl_off_blk, st);
	sc.n_root_blocks = root_blk.size();
	sc.d_root_blk.upload(root_blk, st);
	sc.d_root_uptr.upload(root_uptr, st);
	sc.d_root_ua.upload(root_ua, st);
	sc.d_root_ub.upload(root_ub, st);
	sc.d_root_rptr.upload(root_rptr, st);
	sc.d_root_rblk.upload(root_rblk, st);
	sc.d_root_cols.upload(root_cols, st);
	sc.d_ridx.upload(ridx, st);
	if(m) {
		sc.d_root_S.resize(dense_chol_storage(m * B));
		sc.d_root_rhs.resize(m * B);
	}
	sc.d_L.resize(nb * BB);
	sc.d_Linv.resize(n * BB);
	sc.d_y.resize(n * B);
	sc.d_info.resize(1);
	SPP_CUDA(cudaStreamSynchronize(st));
	if(getenv("SPP_SPARSE_VERBOSE"))
		fprintf(stderr, "[spp sparse chol] n %zu (B = %zu), A blocks %zu, L blocks %zu, levels %u (cooperative 0..%u, single CTA ..%u), "
			"dense root front %zu columns (%zu blocks)\n", n, B, sc.n_a_blocks, nb, n_levels_all, tail, n_levels, m, sc.n_root_blocks);
	sc.valid = true;
	sc.owner = owner;
}

// ---- device: numeric phase ------------------------------------------------------------------------------

template <bool GRID>
__device__ __forceinline__ void level_barrier()
{
	if(GRID)
		cg::this_grid().sync();
	else
		__syncthreads();
}

struct SparseCholArgs {
	const uint64_t *lptr;      // [n + 1] blocks of column j: lptr[j] (diagonal) .. lptr[j + 1]
	const uint32_t *lrow;      // [nb] block row
	const uint32_t *lcolof;    // [nb] block column
	const int64_t *src;        // [nb] +/-(block index in A + 1), 0 = fill-in
	const uint64_t *rptr;      // [n + 1] row structure: blocks L(j, k), k < j
	const uint32_t *rblk;
	const uint64_t *uptr;      // [nb + 1] update pairs of every block
	const uint32_t *ua, *ub;
	const uint32_t *lvl_ptr, *lvl_cols;
	const uint64_t *lvl_off_ptr;
	const uint32_t *lvl_off_blk;
	const uint32_t *order;     // [n] new position -> caller's block column
	const double *A;           // caller's values, blocks B x B column-major in structure order
	const double *rhs;         // caller's right-hand side (caller's order)
	double *L, *Linv, *y, *x;  // factor blocks, inverse diagonal blocks, forward / backward solution (new order / caller's)
	int *info;
};

// one warp: T(r, c) = A-part - sum over the update pairs of La(r, :) . Lb(c, :); lane e = r + B c (lanes >= B*B idle;
// B = 6 uses lanes 0..17 with two elements each: e and e + 18)
// b_given: the update pairs are pa / pb [pbeg, pend) instead of the block's own list. (A flag, not "pa != 0": a root front
// that covers the whole matrix has an EMPTY pair list, a null pointer, and must not fall back to the block's own list,
// whose L blocks are never formed for root columns.)
template <int B>
__device__ __forceinline__ void block_update(const SparseCholArgs &a, uint32_t blk, int lane, double (&t)[2],
	const uint32_t *pa = 0, const uint32_t *pb = 0, uint64_t pbeg = 0, uint64_t pend = 0, bool b_given = false)
{
	constexpr int BB = B * B, NE = (BB > 32)? 2 : 1, STEP = (BB > 32)? BB / 2 : 0;
	const int64_t s = a.src[blk];
	#pragma unroll
	for(int u = 0; u < NE; ++ u) {
		const int e = lane + u * STEP;
		t[u] = 0;
		if(e < BB && (NE == 1 || lane < STEP) && s) {
			const int r = e % B, c = e / B;
			const double *Ab = a.A + (size_t)((s > 0? s : -s) - 1) * BB;
			t[u] = (s > 0)? Ab[e] : Ab[c + B * r]; // transposed source
		}
	}
	const uint32_t *ua = b_given? pa : a.ua, *ub = b_given? pb : a.ub;
	const uint64_t beg = b_given? pbeg : a.uptr[blk], end = b_given? pend : a.uptr[blk + 1];
	for(uint64_t q = beg; q < end; ++ q) {
		const double *La = a.L + (size_t)ua[q] * BB, *Lb = a.L + (size_t)ub[q] * BB;
		#pragma unroll
		for(int u = 0; u < NE; ++ u) {
			const int e = lane + u * STEP;
			if(e < BB && (NE == 1 || lane < STEP)) {
				const int r = e % B, c = e / B;
				double acc = 0;
				#pragma unroll
				for(int k = 0; k < B; ++ k)
					acc += La[r + B * k] * Lb[c + B * k];
				t[u] -= acc;
			}
		}
	}
}

template <int B, bool GRID>
__global__ void __launch_bounds__(SC_WARPS * 32) k_sparse_chol(SparseCholArgs a, uint32_t level_begin, uint32_t level_end)
{
	constexpr int BB = B * B, NE = (BB > 32)? 2 : 1, STEP = (BB > 32)? BB / 2 : 0;
	__shared__ double scratch[SC_WARPS][BB];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const size_t gwarp = blockIdx.x * (size_t)SC_WARPS + warp, n_warps = gridDim.x * (size_t)SC_WARPS;
	double *sw = scratch[warp];
	for(uint32_t l = level_begin; l < level_end; ++ l) {
		// (a) diagonal blocks of the level's columns: update, Cholesky, inverse, forward solve
		for(size_t q = a.lvl_ptr[l] + gwarp; q < a.lvl_ptr[l + 1]; q += n_warps) {
			const uint32_t j = a.lvl_cols[q];
			const uint64_t bd = a.lptr[j];
			double t[2];
			block_update<B>(a, (uint32_t)bd, lane, t);
			#pragma unroll
			for(int u = 0; u < NE; ++ u) {
				const int e = lane + u * STEP;
				if(e < BB && (NE == 1 || lane < STEP)) sw[e] = t[u];
			}
			__syncwarp();
			// every lane factors the B x B block redundantly in registers (lower Cholesky D = G G^T) and inverts G
			double g[B][B], gi[B][B];
			#pragma unroll
			for(int c = 0; c < B; ++ c)
				#pragma unroll
				for(int r = 0; r < B; ++ r)
					g[r][c] = sw[r + B * c];
			bool bad = false;
			#pragma unroll
			for(int c = 0; c < B; ++ c) {
				double d = g[c][c];
				#pragma unroll
				for(int k = 0; k < c; ++ k)
					d -= g[c][k] * g[c][k];
				if(!(d > 0)) { bad = true; d = 1; }
				const double rd = rsqrt(d);
				g[c][c] = d * rd;
				#pragma unroll
				for(int r = c + 1; r < B; ++ r) {
					double v = g[r][c];
					#pragma unroll
					for(int k = 0; k < c; ++ k)
						v -= g[r][k] * g[c][k];
					g[r][c] = v * rd;
				}
				gi[c][c] = rd;
			}
			#pragma unroll
			for(int c = 0; c < B; ++ c) { // column c of G^-1 (lower triangular)
				#pragma unroll
				for(int r = c + 1; r < B; ++ r) {
					double v = 0;
					#pragma unroll
					for(int k = c; k < r; ++ k)
						v += g[r][k] * gi[k][c];
					gi[r][c] = -v * gi[r][r];
				}
			}
			if(bad && lane == 0)
				atomicCAS(a.info, 0, int(j) + 1);
			__syncwarp();
			#pragma unroll
			for(int u = 0; u < NE; ++ u) {
				const int e = lane + u * STEP;
				if(e < BB && (NE == 1 || lane < STEP)) {
					const int r = e % B, c = e / B;
					double vg = 0, vi = 0;
					#pragma unroll
					for(int rr = 0; rr < B; ++ rr)
						#pragma unroll
						for(int cc = 0; cc < B; ++ cc)
							if(rr == r && cc == c) { vg = (rr >= cc)? g[rr][cc] : 0.0; vi = (rr >= cc)? gi[rr][cc] : 0.0; }
					a.L[(size_t)bd * BB + e] = vg;
					a.Linv[(size_t)j * BB + e] = vi;
				}
			}
			// forward solve: y_j = G^-1 (b_j - sum_k L(j, k) y_k); lane r < B gathers its row, lanes exchange through scratch
			if(lane < B) {
				double v = a.rhs[(size_t)a.order[j] * B + lane];
				for(uint64_t p = a.rptr[j]; p < a.rptr[j + 1]; ++ p) {
					const uint32_t b = a.rblk[p];
					const double *Lb = a.L + (size_t)b * BB, *yk = a.y + (size_t)a.lcolof[b] * B;
					#pragma unroll
					for(int k = 0; k < B; ++ k)
						v -= Lb[lane + B * k] * yk[k];
				}
				sw[lane] = v;
			}
			__syncwarp();
			if(lane < B) {
				double v = 0;
				#pragma unroll
				for(int k = 0; k < B; ++ k) {
					double gik = 0;
					#pragma unroll
					for(int rr = 0; rr < B; ++ rr)
						if(rr == lane) gik = (rr >= k)? gi[rr][k] : 0.0;
					v += gik * sw[k];
				}
				a.y[(size_t)j * B + lane] = v;
			}
			__syncwarp();
		}
		level_barrier<GRID>();
		// (b) off-diagonal blocks of the level's columns: L_ij = (A_ij - sum_k L_ik L_jk^T) G_jj^-T
		for(uint64_t q = a.lvl_off_ptr[l] + gwarp; q < a.lvl_off_ptr[l + 1]; q += n_warps) {
			const uint32_t blk = a.lvl_off_blk[q], j = a.lcolof[blk];
			double t[2];
			block_update<B>(a, blk, lane, t);
			#pragma unroll
			for(int u = 0; u < NE; ++ u) {
				const int e = lane + u * STEP;
				if(e < BB && (NE == 1 || lane < STEP)) sw[e] = t[u];
			}
			__syncwarp();
			const double *Gi = a.Linv + (size_t)j * BB;
			#pragma unroll
			for(int u = 0; u < NE; ++ u) {
				const int e = lane + u * STEP;
				if(e < BB && (NE == 1 || lane < STEP)) {
					const int r = e % B, c = e / B;
					double v = 0; // (T G^-T)(r, c) = sum_k T(r, k) Ginv(c, k), k <= c
					#pragma unroll
					for(int k = 0; k < B; ++ k)
						v += sw[r + B * k] * Gi[c + B * k];
					a.L[(size_t)blk * BB + e] = v;
				}
			}
			__syncwarp();
		}
		level_barrier<GRID>();
	}
}

// levels in reverse: x_j = G_jj^-T (y_j - sum_{i > j} L_ij^T x_i); the result goes to the caller's order
template <int B, bool GRID>
__global__ void __launch_bounds__(SC_WARPS * 32) k_sparse_backsolve(SparseCholArgs a, uint32_t level_begin, uint32_t level_end)
{
	constexpr int BB = B * B;
	__shared__ double scratch[SC_WARPS][B];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const size_t gwarp = blockIdx.x * (size_t)SC_WARPS + warp, n_warps = gridDim.x * (size_t)SC_WARPS;
	for(uint32_t l = level_end; l -- > level_begin;) {
		for(size_t q = a.lvl_ptr[l] + gwarp; q < a.lvl_ptr[l + 1]; q += n_warps) {
			const uint32_t j = a.lvl_cols[q];
			if(lane < B) {
				double v = a.y[(size_t)j * B + lane];
				for(uint64_t b = a.lptr[j] + 1; b < a.lptr[j + 1]; ++ b) {
					const double *Lb = a.L + (size_t)b * BB, *xi = a.y + (size_t)a.lrow[b] * B; // x overwrites y
					#pragma unroll
					for(int k = 0; k < B; ++ k)
						v -= Lb[k + B * lane] * xi[k];
				}
				scratch[warp][lane] = v;
			}
			__syncwarp();
			if(lane < B) {
				const double *Gi = a.Linv + (size_t)j * BB;
				double v = 0; // (G^-T t)(r) = sum_k Ginv(k, r) t(k), k >= r
				#pragma unroll
				for(int k = 0; k < B; ++ k)
					v += Gi[k + B * lane] * scratch[warp][k];
				a.y[(size_t)j * B + lane] = v;
				a.x[(size_t)a.order[j] * B + lane] = v;
			}
			__syncwarp();
		}
		level_barrier<GRID>();
	}
}

struct SparseRootArgs {
	size_t n_blocks, m;
	const uint32_t *blk;        // [n_blocks] the root's blocks
	const uint64_t *uptr;       // [n_blocks + 1] update pairs from the non-root columns
	const uint32_t *ua, *ub;
	const uint64_t *rptr;       // [m + 1] per root row: its blocks in non-root columns
	const uint32_t *rblk;
	const uint32_t *cols;       // [m] root index -> column
	const uint32_t *ridx;       // [n] column -> root index
	double *S;                  // dense storage of the dense solver (upper triangle, column-major)
	size_t ld;
	double *rhs;                // [m * B]
};

// root front assembly: warp per block (i, j) of the root, S_upper(j, i) = (A_ij - sum_{k not in root} L_ik L_jk^T)^T
template <int B>
__global__ void __launch_bounds__(SC_WARPS * 32) k_root_assemble(SparseCholArgs a, SparseRootArgs ra)
{
	constexpr int BB = B * B, NE = (BB > 32)? 2 : 1, STEP = (BB > 32)? BB / 2 : 0;
	const int lane = threadIdx.x & 31;
	const size_t q = blockIdx.x * (size_t)SC_WARPS + (threadIdx.x >> 5);
	if(q >= ra.n_blocks) return;
	const uint32_t blk = ra.blk[q];
	const size_t i = ra.ridx[a.lrow[blk]], j = ra.ridx[a.lcolof[blk]];
	double t[2];
	block_update<B>(a, blk, lane, t, ra.ua, ra.ub, ra.uptr[q], ra.uptr[q + 1], true);
	#pragma unroll
	for(int u = 0; u < NE; ++ u) {
		const int e = lane + u * STEP;
		if(e < BB && (NE == 1 || lane < STEP)) {
			const int r = e % B, c = e / B; // element (r, c) of block (i, j) -> S(j B + c, i B + r)
			ra.S[(i * B + r) * ra.ld + j * B + c] = t[u];
		}
	}
}

// right-hand side of the root: thread per scalar row, rhs_i - sum_{k not in root} L(i, k) y_k
template <int B>
__global__ void k_root_rhs(SparseCholArgs a, SparseRootArgs ra)
{
	constexpr int BB = B * B;
	const size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(idx >= ra.m * B) return;
	const size_t ri = idx / B, i = ra.cols[ri];
	const int r = int(idx % B);
	double v = a.rhs[(size_t)a.order[i] * B + r];
	for(uint64_t p = ra.rptr[ri]; p < ra.rptr[ri + 1]; ++ p) {
		const uint32_t b = ra.rblk[p];
		const double *Lb = a.L + (size_t)b * BB, *yk = a.y + (size_t)a.lcolof[b] * B;
		#pragma unroll
		for(int k = 0; k < B; ++ k)
			v -= Lb[r + B * k] * yk[k];
	}
	ra.rhs[idx] = v;
}

template <int B>
__global__ void k_root_scatter(SparseCholArgs a, SparseRootArgs ra)
{
	const size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(idx >= ra.m * B) return;
	const size_t i = ra.cols[idx / B];
	const int r = int(idx % B);
	a.y[i * B + r] = ra.rhs[idx];
	a.x[(size_t)a.order[i] * B + r] = ra.rhs[idx];
}

template <int B>
static int sparse_chol_numeric_t(spp_ctx *ctx, SparseCholArgs &a)
{
	SparseChol &sc = ctx->schol;
	cudaStream_t st = ctx->stream;
	SPP_CUDA(cudaMemsetAsync(sc.d_info.p(), 0, sizeof(int), st));
	if(sc.coop_B != B) { // both cooperative kernels of this block size must be co-resident on the grid
		int per_sm = 0, per_sm_bs = 0, n_sm = 0, dev = 0;
		SPP_CUDA(cudaGetDevice(&dev));
		SPP_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
		SPP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_sparse_chol<B, true>, SC_WARPS * 32, 0));
		SPP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_bs, k_sparse_backsolve<B, true>, SC_WARPS * 32, 0));
		sc.max_coop_ctas = std::max(1, std::min(std::min(per_sm, per_sm_bs), 2) * n_sm);
		sc.coop_B = B;
	}
	uint32_t zero = 0, tail = sc.tail_level, nl = sc.n_levels;
	if(tail > 0) {
		void *args[] = {&a, &zero, &tail};
		SPP_CUDA(cudaLaunchCooperativeKernel((void*)k_sparse_chol<B, true>, dim3(sc.max_coop_ctas), dim3(SC_WARPS * 32), args, 0, st));
		LAUNCH_CHECK(ctx);
	}
	if(tail < nl) {
		k_sparse_chol<B, false><<<1, SC_WARPS * 32, 0, st>>>(a, tail, nl);
		LAUNCH_CHECK(ctx);
	}
	const size_t m = sc.n_root;
	if(m) { // the dense root front: assemble, factor + solve on the dense DMMA Cholesky, scatter
		const size_t nd = m * B;
		SparseRootArgs ra;
		ra.n_blocks = sc.n_root_blocks; ra.m = m; ra.blk = sc.d_root_blk.p(); ra.uptr = sc.d_root_uptr.p();
		ra.ua = sc.d_root_ua.p(); ra.ub = sc.d_root_ub.p(); ra.rptr = sc.d_root_rptr.p(); ra.rblk = sc.d_root_rblk.p();
		ra.cols = sc.d_root_cols.p(); ra.ridx = sc.d_ridx.p(); ra.S = sc.d_root_S.p(); ra.ld = dense_chol_ld(nd);
		ra.rhs = sc.d_root_rhs.p();
		sc.d_root_S.zero(st);
		k_root_assemble<B><<<n_blocks(sc.n_root_blocks, SC_WARPS), SC_WARPS * 32, 0, st>>>(a, ra);
		LAUNCH_CHECK(ctx);
		k_root_rhs<B><<<n_blocks(nd, 128), 128, 0, st>>>(a, ra);
		LAUNCH_CHECK(ctx);
		if(dense_chol_solve_device(ctx, sc.d_root_S.p(), nd, sc.d_root_rhs.p()) != SPP_OK)
			return SPP_NOT_POSDEF;
		k_root_scatter<B><<<n_blocks(nd, 128), 128, 0, st>>>(a, ra);
		LAUNCH_CHECK(ctx);
	}
	if(tail < nl) {
		k_sparse_backsolve<B, false><<<1, SC_WARPS * 32, 0, st>>>(a, tail, nl);
		LAUNCH_CHECK(ctx);
	}
	if(tail > 0) {
		void *args[] = {&a, &zero, &tail};
		SPP_CUDA(cudaLaunchCooperativeKernel((void*)k_sparse_backsolve<B, true>, dim3(sc.max_coop_ctas), dim3(SC_WARPS * 32), args, 0, st));
		LAUNCH_CHECK(ctx);
	}
	ctx->h_scalars.resize(16);
	int *h_info = reinterpret_cast<int*>(ctx->h_scalars.p());
	SPP_CUDA(cudaMemcpyAsync(h_info, sc.d_info.p(), sizeof(int), cudaMemcpyDeviceToHost, st));
	SPP_CUDA(cudaStreamSynchronize(st));
	return (*h_info == 0)? SPP_OK : SPP_NOT_POSDEF;
}

// d_A: the values of the structure given to sparse_chol_symbolic (device); d_rhs / d_x: caller's order (device)
int sparse_chol_solve_device(spp_ctx *ctx, const double *d_A, const double *d_rhs, double *d_x)
{
	SparseChol &sc = ctx->schol;
	if(!sc.valid)
		throw invalid_error("sparse Cholesky: no symbolic analysis");
	SparseCholArgs a;
	a.lptr = sc.d_lptr.p(); a.lrow = sc.d_lrow.p(); a.lcolof = sc.d_lcolof.p(); a.src = sc.d_src.p();
	a.rptr = sc.d_rptr.p(); a.rblk = sc.d_rblk.p(); a.uptr = sc.d_uptr.p(); a.ua = sc.d_ua.p(); a.ub = sc.d_ub.p();
	a.lvl_ptr = sc.d_lvl_ptr.p(); a.lvl_cols = sc.d_lvl_cols.p(); a.lvl_off_ptr = sc.d_lvl_off_ptr.p();
	a.lvl_off_blk = sc.d_lvl_off_blk.p(); a.order = sc.d_order.p();
	a.A = d_A; a.rhs = d_rhs; a.L = sc.d_L.p(); a.Linv = sc.d_Linv.p(); a.y = sc.d_y.p(); a.x = d_x; a.info = sc.d_info.p();
	if(sc.B == 3) return sparse_chol_numeric_t<3>(ctx, a);
	if(sc.B == 6) return sparse_chol_numeric_t<6>(ctx, a);
	if(sc.B == 2) return sparse_chol_numeric_t<2>(ctx, a);
	throw invalid_error("sparse Cholesky: block size must be 2, 3 or 6");
}

} // namespace spp
