// phb_nuc4.cu -- fused whole-tree walk kernels for 4-state (nucleotide) models on sm_100a.
//
// Replaces, for nstate == 4, the reference's one-node-at-a-time SSE path
// (update_partials_4_SSE treelikelihood4.c:1409, integrate_partials_4_SSE :822,
// node_log_likelihoods_4_SSE :882, update_upper_partials treelikelihood.c:2129,
// calculate_branch_partials_4_SSE treelikelihood4.c:1752, gradient_cat_branch_lengths
// treelikelihood.c:2793) by ONE kernel per evaluation:
//
//   * a thread owns PPT (pattern, rate category) pairs and walks the WHOLE tree: post-order for the
//     lower partials, root integration, then pre-order for upper partials and branch gradients;
//   * intermediate partials live in thread-private shared-memory slots; the host orders the walks so
//     that the number of live slots is the tree's Strahler number (<= log2(T) + 1);
//   * what travels between ops is the MESSAGE M_n = P_n L_n a node sends to its parent (L_n = M_a o M_b is formed and, if
//     needed, rescaled in registers): the post-order op of n multiplies by n's OWN matrix once, and that product is reused
//     three times -- by the parent's lower partial, by the sibling's upper partial and by n's own branch gradient
//     (4 mat-vecs per internal node and evaluation instead of the 7 a node-at-a-time formulation spends);
//   * the messages of internal nodes are streamed once to a CTA-private HBM scratch row (32 B per
//     (pattern, category) and node, coalesced 1 KB per warp) and read back once by the pre-order pass -- requested one op
//     ahead into alternating register sets and hinted into L2 three ops ahead; upper partials never leave the SM.  HBM traffic is ~2(T-1)*C*32 B per pattern instead of the
//     ~(5T-9)*C*32 B of node-at-a-time streaming (SURVEY.md 8d);
//   * transition matrices arrive in walk order through TMA bulk copies (cp.async.bulk + mbarrier,
//     double-buffered chunks of PHBC_WALK_CHUNK ops) and are read as warp-uniform broadcasts;
//   * dP/dt L is evaluated as Q (P L): dP/dt = Q P(t) for any rate matrix, so derivative matrices are
//     never built or staged; diag(f) Q sits in the kernel parameter (constant) bank;
//   * per-branch gradient terms are reduced with a paired warp butterfly (four branches per 6
//     shuffle rounds) and accumulated with no-return reductions into warp-private rows, which a second
//     tiny kernel sums in a fixed order (deterministic);
//   * GRAD = 2 additionally accumulates the 4 x 4 transition statistics of every branch (gstat_add), from which the
//     substitution-model parameter gradients of calculate_dlnl_dQ (treelikelihood.c:2337-2583) are 16-element contractions;
//   * GRAD = 3 (unscaled, exact form) additionally accumulates the diagonal of the branch-length Hessian: d2P/dt2 L = Q^2 (P L)
//     is one more product with a constant matrix (diag(pi) Q^2 in the parameter bank), and the (L'/L)^2 term takes each pattern's
//     L' summed over the categories through a shared-memory exchange per op.
//
// CTAs are persistent: grid = min(tiles, resident CTAs), each CTA loops over pattern tiles and owns
// its scratch, so device memory is independent of the pattern count.
#include "phb_ctx.cuh"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#define NUC4_CHUNK PHBC_WALK_CHUNK  // ops per TMA chunk
#define NUC4_NT 256   // threads per CTA
#ifndef NUC4_L2PF
#define NUC4_L2PF 1    // L2 prefetch hints two pre-order ops ahead
#endif

struct Nuc4Params {
	int T, N, C, P, PB, root;
	int n_post, n_pre, nslots, ntiles;
	int include_root_freqs, compat;
	int nbatch, phases;                   // branch-length samples sharing one launch; samples one CTA can touch
	long long mats_stride;                // doubles between the walk matrices of consecutive samples
	int post_first_tips, pre_first_tips;  // tip count of chunk 0 of each walk
	double threshold;
	const uint8_t *tip_codes;  // [2 walks][tiles][T][PB], rows in walk order
	const double *weights;
	const double *props;
	const phbc_post_op *post_ops;
	const phbc_pre_op *pre_ops;
	const double *post_mats;  // [n_post][3][C][16]: own (identity at the root) | child a | child b (tips only)
	const double *pre_mats;   // [n_pre][3][C][16]
	double *lower;            // [grid][n_post][C][PB][4]: messages P_n L_n
	double *gacc;             // [grid][phases][warps][N]
	double *gstat;            // GRAD == 2: [grid][warps][N][16] expected-transition statistics (see gstat_add)
	double *cta_lnl;          // [grid][phases][warps]
	double *pattern_lnl;      // [P]
	double freqs[4];
	double fq[4];     // weights of the gradient numerator: pi, or 1 when the root frequencies are folded into the uppers
	double wroot[4];  // upper message entering the root's children: 1, or pi (tlk->include_root_freqs)
	double FQ[16];    // diag(fq) Q: row i of the rate matrix times the weight of state i in the gradient numerator
	// GRAD == 3 only (appended: the layout above is that of the other variants)
	double FQ2[16];        // diag(pi) Q^2: weights of the second-derivative numerator
	const double *rates;   // [C] category rates
	double *hacc;          // [grid][warps][N] Hessian-diagonal rows
};

// ---------------------------------------------------------------------------------------------
// small dense helpers (everything in registers)
// ---------------------------------------------------------------------------------------------
// y = M x with M a 4x4 row-major matrix in shared memory (warp-uniform address => broadcast)
__device__ __forceinline__ void matvec_smem(const double *__restrict__ M, const double (&x)[4], double (&y)[4]) {
	const double2 *M2 = reinterpret_cast<const double2 *>(M);
#pragma unroll
	for (int i = 0; i < 4; i++) {
		const double2 a = M2[2 * i], b = M2[2 * i + 1];
		y[i] = fma(a.x, x[0], fma(a.y, x[1], fma(b.x, x[2], b.y * x[3])));
	}
}

// Tip codes: 0..3 a known state (gather one column), 4 missing with factor exactly 1 (state tips with
// state >= 4, treelikelihood4.c:1107-1150), 0x10 | mask an ambiguity set (tip partial vectors: sum of columns).
__device__ __forceinline__ void tip_message(const double *__restrict__ M, unsigned code, double (&y)[4]) {
	if (__all_sync(0xffffffffu, code < 4u)) {
#pragma unroll
		for (int i = 0; i < 4; i++) y[i] = M[4 * i + code];
	} else {
		double x[4];
#pragma unroll
		for (int j = 0; j < 4; j++) x[j] = (code < 4u ? code == (unsigned)j : ((code >> j) & 1u)) ? 1.0 : 0.0;
		matvec_smem(M, x, y);
		if (code == 4u) y[0] = y[1] = y[2] = y[3] = 1.0;
	}
}

#define NUC4_SLOT_BYTES (2 * NUC4_NT * 16)  // one slot: two halves of NT double2
#define NUC4_ROW_BYTES (NUC4_NT * 32)       // one lower-scratch row: same two-half layout

// thread-private 32-byte cells inside a [half][NT] double2 tile (conflict-free 128-bit accesses)
__device__ __forceinline__ void cell_load(const unsigned char *cell, double (&x)[4]) {
	const double2 lo = *reinterpret_cast<const double2 *>(cell);
	const double2 hi = *reinterpret_cast<const double2 *>(cell + NUC4_NT * 16);
	x[0] = lo.x, x[1] = lo.y, x[2] = hi.x, x[3] = hi.y;
}
__device__ __forceinline__ void cell_store(unsigned char *cell, const double (&x)[4]) {
	*reinterpret_cast<double2 *>(cell) = make_double2(x[0], x[1]);
	*reinterpret_cast<double2 *>(cell + NUC4_NT * 16) = make_double2(x[2], x[3]);
}
// lower-scratch rows use the same layout in global memory (streaming loads / stores: touched once each way)
__device__ __forceinline__ void row_load(const unsigned char *cell, double (&x)[4]) {
	const double2 lo = __ldcs(reinterpret_cast<const double2 *>(cell));
	const double2 hi = __ldcs(reinterpret_cast<const double2 *>(cell + NUC4_NT * 16));
	x[0] = lo.x, x[1] = lo.y, x[2] = hi.x, x[3] = hi.y;
}
__device__ __forceinline__ void row_store(unsigned char *cell, const double (&x)[4]) {
	__stcs(reinterpret_cast<double2 *>(cell), make_double2(x[0], x[1]));
	__stcs(reinterpret_cast<double2 *>(cell + NUC4_NT * 16), make_double2(x[2], x[3]));
}

// ---------------------------------------------------------------------------------------------
// the walk kernel
// ---------------------------------------------------------------------------------------------
// shared memory map (dynamic):
//   stage[2]: each 64 B (the two mbarriers live in stage 0's), CHUNK * 48 B of descriptors, CHUNK * 3*C*128 B of matrices,
//             2*CHUNK * PB B of tip codes
//   slots:    nslots * NUC4_SLOT_BYTES
//   xch:      exchange area for cross-category sums (C * PB doubles; 4 * C * PB under rescaling) + invLw[PB] + sfslot[nslots][NT]
// (C2's shape, Gamma-4, 5 slots and chunks of 6 ops: 64,256 B.  Four CTAs per SM at a 128-register budget were measured SLOWER than three at 160:
// 6.62 against 6.29 ms on the same box, round 1 h2.)
struct Nuc4Stage {
	uint32_t desc_off, mat_off, code_off, bytes;
};
__host__ __device__ constexpr Nuc4Stage nuc4_stage_layout(int C, int PB) {
	return Nuc4Stage{64u, (uint32_t)(64 + NUC4_CHUNK * 48), (uint32_t)(64 + NUC4_CHUNK * 48 + NUC4_CHUNK * 3 * C * 128),
	                 (uint32_t)((64 + NUC4_CHUNK * 48 + NUC4_CHUNK * 3 * C * 128 + 2 * NUC4_CHUNK * PB + 127) & ~127)};
}

// 4 values per lane -> 4 warp totals in 6 shuffle rounds: lane 0 gets v0, lane 8 v2, lane 16 v1, lane 24 v3
__device__ __forceinline__ double butterfly4(double v0, double v1, double v2, double v3, int lane) {
	const bool h16 = lane & 16, h8 = lane & 8;
	const double r01 = (h16 ? v1 : v0) + __shfl_xor_sync(0xffffffffu, h16 ? v0 : v1, 16);
	const double r23 = (h16 ? v3 : v2) + __shfl_xor_sync(0xffffffffu, h16 ? v2 : v3, 16);
	double r = (h8 ? r23 : r01) + __shfl_xor_sync(0xffffffffu, h8 ? r01 : r23, 8);
	r += __shfl_xor_sync(0xffffffffu, r, 4);
	r += __shfl_xor_sync(0xffffffffu, r, 2);
	r += __shfl_xor_sync(0xffffffffu, r, 1);
	return r;
}
// 2 values per lane: lane 0 gets v0, lane 16 gets v1
__device__ __forceinline__ double butterfly2(double v0, double v1, int lane) {
	const bool h16 = lane & 16;
	double r = (h16 ? v1 : v0) + __shfl_xor_sync(0xffffffffu, h16 ? v0 : v1, 16);
	r += __shfl_xor_sync(0xffffffffu, r, 8);
	r += __shfl_xor_sync(0xffffffffu, r, 4);
	r += __shfl_xor_sync(0xffffffffu, r, 2);
	r += __shfl_xor_sync(0xffffffffu, r, 1);
	return r;
}

// indicator vector of a tip code = the tip's L_n: a known state is one-hot, a missing state all ones (derivative matrices see their
// real row sums, treelikelihoodX.c:878-1001), an ambiguity set its mask
__device__ __forceinline__ void tip_vector(unsigned code, double (&x)[4]) {
#pragma unroll
	for (int j = 0; j < 4; j++) x[j] = (code < 4u ? code == (unsigned)j : (code == 4u || ((code >> j) & 1u))) ? 1.0 : 0.0;
}

// Expected-transition statistics of one branch: row[4 i + j] += sum over the warp's patterns of t[i] * x[j], with
// t = (w_k / L_k) f_i U_n[k, i] and x = L_n[k, .].  Any per-branch matrix M then contracts as sum_ij G[i][j] M[i][j] =
// sum_k w_k / L_k sum_i f_i U_n[k,i] (M L_n[k])_i -- the node sweep of calculate_dlnl_dQ (treelikelihood.c:2408-2478) for EVERY
// parameter at once, and without materialised upper partials.  16 values are reduced across 32 lanes by a transposing
// butterfly (8 + 4 + 2 + 1 + 1 shuffles); lane l ends up with element l >> 1.
template <int PPT>
__device__ __forceinline__ void gstat_add(const double (&t)[PPT][4], const double (&x)[PPT][4], double *row, int lane) {
	double v[16];
#pragma unroll
	for (int i = 0; i < 4; i++)
#pragma unroll
		for (int j = 0; j < 4; j++) {
			double a = t[0][i] * x[0][j];
#pragma unroll
			for (int u = 1; u < PPT; u++) a = fma(t[u][i], x[u][j], a);
			v[4 * i + j] = a;
		}
#pragma unroll
	for (int w = 8, off = 16; w >= 1; w >>= 1, off >>= 1) {
		const bool h = lane & off;
#pragma unroll
		for (int k = 0; k < w; k++) {
			const double keep = h ? v[w + k] : v[k], send = h ? v[k] : v[w + k];
			v[k] = keep + __shfl_xor_sync(0xffffffffu, send, off);
		}
	}
	v[0] += __shfl_xor_sync(0xffffffffu, v[0], 1);
	if (!(lane & 1)) red_add_f64(row + (lane >> 1), v[0]);
}

// y[u] = M x[u] for the PPT patterns of a thread: every matrix element is read from shared memory ONCE and feeds PPT
// independent FMA chains (half the LDS traffic and twice the instruction-level parallelism per pattern at PPT = 2)
template <int PPT>
__device__ __forceinline__ void matvec_smem_n(const double *__restrict__ M, const double (&x)[PPT][4], double (&y)[PPT][4]) {
	const double2 *M2 = reinterpret_cast<const double2 *>(M);
#pragma unroll
	for (int i = 0; i < 4; i++) {
		const double2 a = M2[2 * i], b = M2[2 * i + 1];
#pragma unroll
		for (int u = 0; u < PPT; u++) y[u][i] = fma(a.x, x[u][0], fma(a.y, x[u][1], fma(b.x, x[u][2], b.y * x[u][3])));
	}
}

// A thread owns PPT (pattern, category) cells of the tile: category c and patterns pl0 + u * PBT (PBT = PB / PPT), i.e. cell
// index c * PB + pl0 + u * PBT in every [half][NUC4_NT] cell array (slots, lower rows) -- the layouts do not depend on PPT.
// GRAD: 0 lnL only, 1 + branch gradients, 2 + expected-transition statistics per branch (substitution-model gradients),
// 3 + the diagonal of the branch-length Hessian (unscaled only; the extra accumulators do not fit the 168 / 80-register budgets of
// three CTAs per SM: two CTAs at PPT = 2, one at PPT = 1, so that nothing spills)
template <int C, bool SCALE, int GRAD, int PPT>
__global__ void __launch_bounds__(NUC4_NT / PPT, GRAD == 3 ? (PPT == 1 ? 1 : 2) : 3) k_nuc4_walk(const Nuc4Params prm) {
	extern __shared__ __align__(128) unsigned char smem_raw[];
	constexpr int PB = NUC4_NT / C;      // patterns per tile
	constexpr int NTHR = NUC4_NT / PPT;  // threads per CTA
	constexpr int PBT = PB / PPT;        // patterns per u-plane
	static_assert(PBT % 32 == 0 || PPT == 1, "a warp must not mix categories");
	static_assert(GRAD != 3 || !SCALE, "the Hessian walk is unscaled (rescaled evaluations take the resident-partials route)");
	constexpr bool RECOMP = GRAD == 1 && !SCALE;  // cherry recomputation (phb_cuda.h): the descriptors' flags are honoured by this variant only
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const int c = tid / PBT, pl0 = tid - c * PBT;
	const int cell0 = c * PB + pl0;  // cell index of u = 0; u adds u * PBT
	constexpr Nuc4Stage lay = nuc4_stage_layout(C, PB);
	uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw);  // inside stage 0's leading 64 bytes
	unsigned char *stage0 = smem_raw;
	unsigned char *slot_cell = stage0 + 2 * lay.bytes + cell0 * 16;  // this thread's first cell in slot 0
	double *xch = reinterpret_cast<double *>(stage0 + 2 * lay.bytes + (size_t)prm.nslots * NUC4_SLOT_BYTES);
	double *invLw = xch + (SCALE ? (GRAD == 2 ? 5 : 4) : (GRAD == 3 ? 2 : 1)) * C * PB;  // GRAD == 3: 1 / L_k follows at invLw + PB
	double *sfslot = invLw + PB;  // [nslots][NT] thread-private copies (SCALE only)
	const uint32_t my_mat = lay.mat_off + c * 128;  // this thread's category inside a staged matrix group
	const uint32_t my_code = lay.code_off + pl0;

	if (tid == 0) {
		mbar_init(&bars[0], 1);
		mbar_init(&bars[1], 1);
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
	}
	__syncthreads();

	uint32_t loads = 0;  // chunk loads consumed so far (CTA-uniform): stage = loads & 1, parity = (loads >> 1) & 1
	const double prop_c = (C == 1) ? 1.0 : prm.props[c];
	double cta_lnl = 0.0;
	unsigned char *row_cell = GRAD ? reinterpret_cast<unsigned char *>(prm.lower) + (size_t)blockIdx.x * prm.n_post * NUC4_ROW_BYTES + cell0 * 16 : nullptr;
	double *my_gacc = nullptr;
	double *my_gstat = GRAD == 2 ? prm.gstat + ((size_t)blockIdx.x * (NTHR / 32) + warp) * prm.N * 16 : nullptr;  // single sample only
	double *my_hacc = GRAD == 3 ? prm.hacc + ((size_t)blockIdx.x * (NTHR / 32) + warp) * prm.N : nullptr;          // single sample only
	const double rate_c = GRAD == 3 ? prm.rates[c] : 0.0;

	// L2 prefetch lanes of the pre-order pass (see pre_op): lane -> (row a | b, plane, half, 128-byte line)
	constexpr int PF_LPR = PPT * 2 * 4;  // lines per message row and warp
	const int pf_row = (lane / PF_LPR) & 1, pf_q = lane % PF_LPR;
	const bool pf_on = GRAD && lane < 2 * PF_LPR;
	const unsigned char *pf_base = GRAD ? row_cell - lane * 16 + ((pf_q >> 3) * PBT) * 16 + ((pf_q >> 2) & 1) * (NUC4_NT * 16) + (pf_q & 3) * 128 : nullptr;

	// work items = (sample, pattern tile), sample-major; a CTA owns a CONTIGUOUS range, so it touches at most
	// prm.phases consecutive samples and keeps one private accumulator row set per touched sample (deterministic sums)
	// (a single sample keeps the strided assignment: tiles are few and coarse, and the strided order spreads the CTAs that
	// get one tile more evenly over the SMs)
	const long long nitems = (long long)prm.ntiles * prm.nbatch;
	const bool strided = prm.nbatch == 1;
	const int item0 = strided ? (int)blockIdx.x : (int)(blockIdx.x * nitems / gridDim.x);
	const int item1 = strided ? (int)nitems : (int)((blockIdx.x + 1) * nitems / gridDim.x);
	const int item_step = strided ? (int)gridDim.x : 1;
	const int b_first = strided ? 0 : item0 / prm.ntiles;
	int cur_b = -1;
	auto flush_lnl = [&](int b) {
		if (lane == 0) prm.cta_lnl[((size_t)blockIdx.x * prm.phases + (b - b_first)) * (NTHR / 32) + warp] = (c == 0) ? cta_lnl : 0.0;  // one partial lnL per warp
	};

	for (int item = item0; item < item1; item += item_step) {
		const int bsmp = item / prm.ntiles, tile = item - bsmp * prm.ntiles;
		if (bsmp != cur_b) {
			if (cur_b >= 0) flush_lnl(cur_b);
			cur_b = bsmp;
			cta_lnl = 0.0;
			if (GRAD) my_gacc = prm.gacc + (((size_t)blockIdx.x * prm.phases + (bsmp - b_first)) * (NTHR / 32) + warp) * prm.N;
		}
		const uint8_t *tile_codes_post = prm.tip_codes + (size_t)tile * prm.T * PB;
		const uint8_t *tile_codes_pre = prm.tip_codes + ((size_t)prm.ntiles + tile) * prm.T * PB;

		// ------------------------------------------------------------------ post-order
		double out[PPT][4];
		double sf_acc[PPT];  // SCALE: log scaling factor of the value currently in `out`
#pragma unroll
		for (int u = 0; u < PPT; u++) out[u][0] = out[u][1] = out[u][2] = out[u][3] = 1.0, sf_acc[u] = 0.0;
		{
			const int nchunks = (prm.n_post + NUC4_CHUNK - 1) / NUC4_CHUNK;
			// one TMA stage: descriptors, walk-ordered matrices, walk-ordered tip codes of the chunk
			auto issue = [&](int ch, uint32_t ld, int tips) {
				const int first = ch * NUC4_CHUNK;
				const int cnt = min(NUC4_CHUNK, prm.n_post - first);
				unsigned char *dst = stage0 + (ld & 1) * lay.bytes;
				const uint32_t dbytes = cnt * (uint32_t)sizeof(phbc_post_op), mbytes = cnt * 3 * C * 128;
				const uint32_t cbytes = (tips & 31) * PB;
				mbar_expect_tx(&bars[ld & 1], dbytes + mbytes + cbytes);
				bulk_g2s(dst + lay.desc_off, prm.post_ops + first, dbytes, &bars[ld & 1]);
				bulk_g2s(dst + lay.mat_off, prm.post_mats + (size_t)cur_b * prm.mats_stride + (size_t)first * 3 * C * 16, mbytes, &bars[ld & 1]);
				if (cbytes) bulk_g2s(dst + lay.code_off, tile_codes_post + (size_t)(tips >> 5) * PB, cbytes, &bars[ld & 1]);
			};
			if (tid == 0) issue(0, loads, prm.post_first_tips);
			for (int ch = 0; ch < nchunks; ch++) {
				mbar_wait(&bars[loads & 1], (loads >> 1) & 1);
				const unsigned char *st = stage0 + (loads & 1) * lay.bytes;
				const phbc_post_op *desc = reinterpret_cast<const phbc_post_op *>(st + lay.desc_off);
				if (tid == 0 && ch + 1 < nchunks) issue(ch + 1, loads + 1, desc[0].next_tips);
				const unsigned char *mats = st + my_mat;
				const uint8_t *cds = st + my_code;
				const int first = ch * NUC4_CHUNK;
				const int cnt = min(NUC4_CHUNK, prm.n_post - first);
#pragma unroll 1
				for (int j = 0; j < cnt; j++) {
					const int kind = (desc[j].a_kind & 0xff) + desc[j].b_kind;
					// a cherry whose parent's pre-order op rebuilds its message (unscaled gradient walks only) keeps no row
					const bool keep_row = !(RECOMP && (desc[j].a_kind & PHBC_POST_NO_ROW));
					const int a_idx = desc[j].a_idx, b_idx = desc[j].b_idx, dst_slot = desc[j].dst_slot;
					const double *MN = reinterpret_cast<const double *>(mats + (j * 3 + 0) * C * 128);
					const double *MA = reinterpret_cast<const double *>(mats + (j * 3 + 1) * C * 128);
					const double *MB = reinterpret_cast<const double *>(mats + (j * 3 + 2) * C * 128);
					double ma[PPT][4], lw[PPT][4];
					double sf_in[PPT];
#pragma unroll
					for (int u = 0; u < PPT; u++) sf_in[u] = 0.0;
					// messages of the children: a tip's is a column (or column sum) of its matrix, an internal child's was formed by
					// its own op -- child b of kinds 1 and 2 is the previous op's result, still in `out`
					if (kind == 0) {
#pragma unroll
						for (int u = 0; u < PPT; u++) {
							tip_message(MA, cds[a_idx * PB + u * PBT], ma[u]);
							tip_message(MB, cds[b_idx * PB + u * PBT], out[u]);
						}
					} else {
						if (SCALE) {
#pragma unroll
							for (int u = 0; u < PPT; u++) sf_in[u] = sf_acc[u];
						}
						if (kind == 1) {
#pragma unroll
							for (int u = 0; u < PPT; u++) tip_message(MA, cds[a_idx * PB + u * PBT], ma[u]);
						} else {
#pragma unroll
							for (int u = 0; u < PPT; u++) {
								cell_load(slot_cell + a_idx * NUC4_SLOT_BYTES + u * PBT * 16, ma[u]);
								if (SCALE) sf_in[u] += sfslot[a_idx * NUC4_NT + cell0 + u * PBT];
							}
						}
					}
#pragma unroll
					for (int u = 0; u < PPT; u++)
#pragma unroll
						for (int i = 0; i < 4; i++) lw[u][i] = ma[u][i] * out[u][i];  // lower partial L_n
					if (SCALE) {
						// SingleTreeLikelihood_scalePartials (treelikelihood.c:1790-1836): max over categories and states
						double *mx = xch + ((first + j) & 1) * C * PB;
#pragma unroll
						for (int u = 0; u < PPT; u++) mx[cell0 + u * PBT] = fmax(fmax(lw[u][0], lw[u][1]), fmax(lw[u][2], lw[u][3]));
						__syncthreads();
#pragma unroll
						for (int u = 0; u < PPT; u++) {
							const int pl = pl0 + u * PBT;
							double m = mx[pl];
							for (int cc = 1; cc < C; cc++) m = fmax(m, mx[cc * PB + pl]);
							double sf = 0.0;
							if (m < prm.threshold) {
#pragma unroll
								for (int i = 0; i < 4; i++) lw[u][i] /= m;
								sf = log(m);
							}
							sf_acc[u] = sf + sf_in[u];
							if (dst_slot >= 0) sfslot[dst_slot * NUC4_NT + cell0 + u * PBT] = sf_acc[u];
						}
					}
					// the message to the parent: the node's OWN matrix (identity at the root, whose `out` feeds the root integration)
					matvec_smem_n<PPT>(MN, lw, out);
#pragma unroll
					for (int u = 0; u < PPT; u++) {
						if (dst_slot >= 0) cell_store(slot_cell + dst_slot * NUC4_SLOT_BYTES + u * PBT * 16, out[u]);  // parked for a later kind-2 op
						if (GRAD && keep_row) row_store(row_cell + (size_t)(unsigned)(first + j) * NUC4_ROW_BYTES + u * PBT * 16, out[u]);
					}
				}
				loads++;
				__syncthreads();  // everyone is done with this stage before it is refilled
			}
		}

		// ------------------------------------------------------------------ root integration
		// integrate_partials_4_SSE + node_log_likelihoods_4_SSE + weighted sum
		{
#pragma unroll
			for (int u = 0; u < PPT; u++) {
				double site = prm.freqs[0] * out[u][0] + prm.freqs[1] * out[u][1] + prm.freqs[2] * out[u][2] + prm.freqs[3] * out[u][3];
				xch[cell0 + u * PBT] = site * prop_c;
			}
			__syncthreads();
			if (c == 0) {
				double v = 0.0;
#pragma unroll
				for (int u = 0; u < PPT; u++) {
					const int pl = pl0 + u * PBT;
					const int p = tile * PB + pl;
					const bool live = p < prm.P;
					double L = xch[pl];
					for (int cc = 1; cc < C; cc++) L += xch[cc * PB + pl];
					double plk = log(L);
					if (SCALE) plk += sf_acc[u];
					const double w = live ? prm.weights[p] : 0.0;
					if (live && prm.nbatch == 1) prm.pattern_lnl[p] = plk;
					invLw[pl] = w / L;  // unscaled path: w_k / L_k; scaled paths use ratios instead
					if (GRAD == 3) invLw[PB + pl] = 1.0 / L;
					v += live ? plk * w : 0.0;
				}
				v = phb_warp_sum(v);
				if (lane == 0) cta_lnl += v;  // warps of category 0 only; summed below
			}
			__syncthreads();
		}

		// ------------------------------------------------------------------ pre-order + gradients
		if (GRAD) {
			double sgrad[PPT], wk[PPT], rinv[PPT];
#pragma unroll
			for (int u = 0; u < PPT; u++) {
				const int pl = pl0 + u * PBT;
				const int p = tile * PB + pl;
				sgrad[u] = invLw[pl];
				wk[u] = p < prm.P ? prm.weights[p] : 0.0;
				rinv[u] = GRAD == 3 ? invLw[PB + pl] : 0.0;
			}
			if (GRAD == 2) {
				// root entry of the statistics: sum_k w_k / L_k L_root[c, k, i] (the root term of the frequency parameters,
				// treelikelihood.c:2371-2404); `out` still holds the root op's result
				double r[4];
#pragma unroll
				for (int i = 0; i < 4; i++) {
					r[i] = sgrad[0] * out[0][i];
#pragma unroll
					for (int u = 1; u < PPT; u++) r[i] = fma(sgrad[u], out[u][i], r[i]);
				}
				const double tot = butterfly4(r[0], r[1], r[2], r[3], lane);  // lane 0: r0, lane 8: r2, lane 16: r1, lane 24: r3
				if ((lane & 7) == 0) red_add_f64(my_gstat + (size_t)prm.root * 16 + (((lane >> 4) & 1) | ((lane >> 2) & 2)), tot);
			}
			const int nchunks = (prm.n_pre + NUC4_CHUNK - 1) / NUC4_CHUNK;
			auto issue = [&](int ch, uint32_t ld, int tips) {
				const int first = ch * NUC4_CHUNK;
				const int cnt = min(NUC4_CHUNK, prm.n_pre - first);
				unsigned char *dst = stage0 + (ld & 1) * lay.bytes;
				const uint32_t dbytes = cnt * (uint32_t)sizeof(phbc_pre_op), mbytes = cnt * 3 * C * 128;
				const uint32_t cbytes = (tips & 31) * PB;
				mbar_expect_tx(&bars[ld & 1], dbytes + mbytes + cbytes);
				bulk_g2s(dst + lay.desc_off, prm.pre_ops + first, dbytes, &bars[ld & 1]);
				bulk_g2s(dst + lay.mat_off, prm.pre_mats + (size_t)cur_b * prm.mats_stride + (size_t)first * 3 * C * 16, mbytes, &bars[ld & 1]);
				if (cbytes) bulk_g2s(dst + lay.code_off, tile_codes_pre + (size_t)(tips >> 5) * PB, cbytes, &bars[ld & 1]);
			};
			// message rows of the internal children of one op (kind: 0 tip-tip, 1 tip-internal, 2 internal-internal)
			auto fetch = [&](const phbc_pre_op *d, double (&A)[PPT][4], double (&B)[PPT][4]) {
				const int kind = d->kind;
				const bool b_row = kind != 0 && !(RECOMP && (d->flags & PHBC_PRE_B_RECOMPUTE));
#pragma unroll
				for (int u = 0; u < PPT; u++) {
					if (kind == 2) row_load(row_cell + (size_t)(unsigned)d->a_row * NUC4_ROW_BYTES + u * PBT * 16, A[u]);
					if (b_row) row_load(row_cell + (size_t)(unsigned)d->b_row * NUC4_ROW_BYTES + u * PBT * 16, B[u]);
				}
			};
			// One op.  Its operands (message rows of the internal children) were loaded into xa / xb by the PREVIOUS op.  ALT: the first
			// thing this op does is to issue the loads of the NEXT op's rows into the other register set (na / nb), a full op ahead
			// of their use -- the two sets alternate between consecutive ops, no copies, and nothing tempts ptxas to sink the loads
			// towards their consumer.  The statistics variant (GRAD = 2) has no registers to spare for a second set: it copies its
			// operands out and refills the same set (na / nb alias xa / xb).  Returns the two gradient terms (and with GRAD == 3 the two
			// Hessian terms in ha / hb).
			constexpr bool ALT = GRAD != 2;
			constexpr bool L2PF = NUC4_L2PF && GRAD != 2;  // the statistics variant is issue-bound: the hints cost it more than they return
			auto pre_op = [&](const phbc_pre_op *desc, const unsigned char *mats, const uint8_t *cds, int j, int cnt, bool more_chunks,
			                  double (&xa)[PPT][4], double (&xb)[PPT][4], double (&na_)[PPT][4], double (&nb_)[PPT][4], double (&ureg)[PPT][4],
			                  double &va, double &vb, double &ha, double &hb) {
				const phbc_pre_op *d = desc + j;
				const int kind = d->kind;
				auto prefetch = [&]() {
					if (j + 1 < cnt) {
						fetch(d + 1, na_, nb_);
					} else if (more_chunks) {
						mbar_wait(&bars[(loads + 1) & 1], ((loads + 1) >> 1) & 1);
						fetch(reinterpret_cast<const phbc_pre_op *>(stage0 + ((loads + 1) & 1) * lay.bytes + lay.desc_off), na_, nb_);
					}
				};
				// Cherry recomputation: child b is a cherry and its op is the NEXT one.  Its two tip messages are formed here from that op's
				// staged matrices and codes, straight into the registers that op reads them from (na_ / nb_), and M_b = P_b (m_a' o m_b')
				// takes the place of the row the post-order pass would have written and this op would have waited for.
				auto recompute_b = [&]() {
					const bool same = j + 1 < cnt;
					const unsigned char *nst = same ? nullptr : stage0 + ((loads + 1) & 1) * lay.bytes;  // the next chunk's stage (its barrier was waited for in prefetch)
					const phbc_pre_op *dn = same ? d + 1 : reinterpret_cast<const phbc_pre_op *>(nst + lay.desc_off);
					const unsigned char *nm = same ? mats + (j + 1) * 3 * C * 128 : nst + my_mat;
					const uint8_t *nc = same ? cds : nst + my_code;
					const double *NP = reinterpret_cast<const double *>(nm);
					const double *NA = reinterpret_cast<const double *>(nm + C * 128);
					const double *NB = reinterpret_cast<const double *>(nm + 2 * C * 128);
					double lb[PPT][4];
#pragma unroll
					for (int u = 0; u < PPT; u++) {
						tip_message(NA, nc[dn->a_code * PB + u * PBT], na_[u]);
						tip_message(NB, nc[dn->b_code * PB + u * PBT], nb_[u]);
#pragma unroll
						for (int i = 0; i < 4; i++) lb[u][i] = na_[u][i] * nb_[u][i];
					}
					matvec_smem_n<PPT>(NP, lb, xb);
				};
				if (L2PF) {
					// the rows the op PHBC_PF_DIST positions later will read go to L2 now (the host put their indices into THIS op's
					// descriptor): the register prefetch above is one op -- about the loaded HBM latency -- ahead of its use, the hint
					// turns that load into an L2 hit.  One instruction per warp: lane l takes one 128-byte line of the warp's share
					// (2 rows x PPT planes x 2 halves x 512 bytes).
					const int r = reinterpret_cast<const int *>(&d->pf_a_row)[pf_row];
					if (pf_on && r >= 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(pf_base + (size_t)(unsigned)r * NUC4_ROW_BYTES));
				}
				const double *MP = reinterpret_cast<const double *>(mats + (j * 3 + 0) * C * 128);
				const double *MA = reinterpret_cast<const double *>(mats + (j * 3 + 1) * C * 128);
				const double *MB = reinterpret_cast<const double *>(mats + (j * 3 + 2) * C * 128);
				if (ALT) prefetch();
				if (RECOMP && (d->flags & PHBC_PRE_B_RECOMPUTE)) recompute_b();
				// W = P_p U_p, the part of the op that does not need the children's rows: computed FIRST, so that the wait for the rows
				// requested by the previous op (still 9 % of the stall samples with the L2 hints) sits behind 32 FP64 instructions
				double W[PPT][4];
				if (d->u_kind == PHBC_W_ROOT) {
					// children of the root: u = P_s L_s [o pi] (treelikelihood.c:2145-2154)
#pragma unroll
					for (int u = 0; u < PPT; u++)
#pragma unroll
						for (int i = 0; i < 4; i++) W[u][i] = prm.wroot[i];
				} else {
					if (d->u_kind == PHBC_W_SLOT) {
#pragma unroll
						for (int u = 0; u < PPT; u++) cell_load(slot_cell + d->u_slot * NUC4_SLOT_BYTES + u * PBT * 16, ureg[u]);  // else: left by the preceding op
					}
					matvec_smem_n<PPT>(MP, ureg, W);  // P_p u_p
				}
				// the op proper, on the messages P_x L_x of the children (ma, mb)
				auto body = [&](double (&ma)[PPT][4], double (&mb)[PPT][4]) {
				double ua[PPT][4], ub[PPT][4];
#pragma unroll
				for (int u = 0; u < PPT; u++)
#pragma unroll
					for (int i = 0; i < 4; i++) ua[u][i] = W[u][i] * mb[u][i], ub[u][i] = W[u][i] * ma[u][i];
				// numerators: sum_i f_i u_n[i] (dP_n L_n)[i] with dP_n L_n = Q (P_n L_n)
				double na[PPT], nb[PPT], da[PPT], db[PPT];
#pragma unroll
				for (int u = 0; u < PPT; u++) na[u] = nb[u] = da[u] = db[u] = 0.0;
#pragma unroll
				for (int i = 0; i < 4; i++) {
#pragma unroll
					for (int u = 0; u < PPT; u++) {
						// prm.FQ = diag(f) Q: the frequency weights ride on the rows of the rate matrix
						const double qa = fma(prm.FQ[4 * i], ma[u][0], fma(prm.FQ[4 * i + 1], ma[u][1], fma(prm.FQ[4 * i + 2], ma[u][2], prm.FQ[4 * i + 3] * ma[u][3])));
						const double qb = fma(prm.FQ[4 * i], mb[u][0], fma(prm.FQ[4 * i + 1], mb[u][1], fma(prm.FQ[4 * i + 2], mb[u][2], prm.FQ[4 * i + 3] * mb[u][3])));
						na[u] = fma(ua[u][i], qa, na[u]);
						nb[u] = fma(ub[u][i], qb, nb[u]);
						if (SCALE) {
							da[u] = fma(prm.fq[i] * ua[u][i], ma[u][i], da[u]);
							db[u] = fma(prm.fq[i] * ub[u][i], mb[u][i], db[u]);
						}
					}
				}
				va = vb = 0.0;
				// GRAD == 2: what multiplies f_i U[i] L[j] in the statistics of the three branches this op serves -- w_k / L_k, with
				// the site likelihood L_k taken in each branch's own scale under rescaling
				double coefa[PPT], coefb[PPT], coefp[PPT];
#pragma unroll
				for (int u = 0; u < PPT; u++) coefa[u] = coefb[u] = coefp[u] = sgrad[u];
				if (!SCALE) {
#pragma unroll
					for (int u = 0; u < PPT; u++) va = fma(na[u], sgrad[u], va), vb = fma(nb[u], sgrad[u], vb);
					if (GRAD == 3) {
						// row of category c, scaled by prop_c r_c in k_nuc4_finalize: w_k / L_k (r_c s_c - (L'_k / L_k) n_c) with s_c = sum_i
						// pi_i U[i] (Q^2 m)[i] and n_c = sum_i pi_i U[i] (Q m)[i]; summed over the categories that is
						// w_k (L"_k / L_k - (L'_k / L_k)^2), d2lnldt2_uppper (treelikelihood.c:2331)
						double lpa[PPT], lpb[PPT];
						if (C == 1) {
#pragma unroll
							for (int u = 0; u < PPT; u++) lpa[u] = rate_c * na[u] * rinv[u], lpb[u] = rate_c * nb[u] * rinv[u];
						} else {  // L'_k sums over the categories: exchange through two shared planes
							const double pr = prm.props[c] * rate_c;
							__syncthreads();  // previous op's readers are done
#pragma unroll
							for (int u = 0; u < PPT; u++) {
								const int ci = cell0 + u * PBT;
								xch[ci] = na[u] * pr;
								xch[C * PB + ci] = nb[u] * pr;
							}
							__syncthreads();
#pragma unroll
							for (int u = 0; u < PPT; u++) {
								const int pl = pl0 + u * PBT;
								double sa = 0.0, sb = 0.0;
								for (int cc = 0; cc < C; cc++) sa += xch[cc * PB + pl], sb += xch[C * PB + cc * PB + pl];
								lpa[u] = sa * rinv[u], lpb[u] = sb * rinv[u];
							}
						}
						ha = hb = 0.0;
#pragma unroll
						for (int u = 0; u < PPT; u++) {
							double sa = 0.0, sb = 0.0;
#pragma unroll
							for (int i = 0; i < 4; i++) {
								const double qa = fma(prm.FQ2[4 * i], ma[u][0], fma(prm.FQ2[4 * i + 1], ma[u][1], fma(prm.FQ2[4 * i + 2], ma[u][2], prm.FQ2[4 * i + 3] * ma[u][3])));
								const double qb = fma(prm.FQ2[4 * i], mb[u][0], fma(prm.FQ2[4 * i + 1], mb[u][1], fma(prm.FQ2[4 * i + 2], mb[u][2], prm.FQ2[4 * i + 3] * mb[u][3])));
								sa = fma(ua[u][i], qa, sa);
								sb = fma(ub[u][i], qb, sb);
							}
							ha = fma(sgrad[u], rate_c * sa - lpa[u] * na[u], ha);
							hb = fma(sgrad[u], rate_c * sb - lpb[u] * nb[u], hb);
						}
					}
				} else {
					// rescale the upper partials like the reference (their scale cancels in the ratios below)
					double *plane = xch;  // planes: max_a, max_b, den_a, den_b [, den_p]
					__syncthreads();      // previous op's readers are done
#pragma unroll
					for (int u = 0; u < PPT; u++) {
						const int ci = cell0 + u * PBT;
						plane[0 * C * PB + ci] = fmax(fmax(ua[u][0], ua[u][1]), fmax(ua[u][2], ua[u][3]));
						plane[1 * C * PB + ci] = fmax(fmax(ub[u][0], ub[u][1]), fmax(ub[u][2], ub[u][3]));
						plane[2 * C * PB + ci] = da[u] * prop_c;
						plane[3 * C * PB + ci] = db[u] * prop_c;
						if (GRAD == 2) {
							// site likelihood seen from the branch above this op's node, in the scale of (U_p, L_p = M_a o M_b):
							// sum_i f_i U_p[i] (P_p L_p)[i] = sum_j f_j L_p[j] (P_p U_p)[j] for a reversible model with f = pi, and
							// P_p U_p is W (the host sends a request here only then)
							double dp = 0.0;
#pragma unroll
							for (int i = 0; i < 4; i++) dp = fma(prm.fq[i] * W[u][i], ma[u][i] * mb[u][i], dp);
							plane[4 * C * PB + ci] = dp * prop_c;
						}
					}
					__syncthreads();
#pragma unroll
					for (int u = 0; u < PPT; u++) {
						const int pl = pl0 + u * PBT;
						double mxa = 0.0, mxb = 0.0, dta = 0.0, dtb = 0.0;
						for (int cc = 0; cc < C; cc++) {
							mxa = fmax(mxa, plane[0 * C * PB + cc * PB + pl]);
							mxb = fmax(mxb, plane[1 * C * PB + cc * PB + pl]);
							dta += plane[2 * C * PB + cc * PB + pl];
							dtb += plane[3 * C * PB + cc * PB + pl];
						}
						if (mxa < prm.threshold) {
#pragma unroll
							for (int i = 0; i < 4; i++) ua[u][i] /= mxa;
						}
						if (mxb < prm.threshold) {
#pragma unroll
							for (int i = 0; i < 4; i++) ub[u][i] /= mxb;
						}
						// exact: one site denominator shared by the categories; compat: per-category ratio
						// (gradient_cat_branch_lengths_aux, treelikelihood.c:2721-2738)
						va += prm.compat ? na[u] / da[u] * wk[u] : na[u] / dta * wk[u];
						vb += prm.compat ? nb[u] / db[u] * wk[u] : nb[u] / dtb * wk[u];
						if (GRAD == 2) {
							double dtp = 0.0;
							for (int cc = 0; cc < C; cc++) dtp += plane[4 * C * PB + cc * PB + pl];
							// ua / ub have just been divided by their maxima: the denominators belong to the undivided values
							coefa[u] = wk[u] / dta * (mxa < prm.threshold ? mxa : 1.0);
							coefb[u] = wk[u] / dtb * (mxb < prm.threshold ? mxb : 1.0);
							coefp[u] = wk[u] / dtp;
						}
					}
				}
				if (GRAD == 2 && d->u_kind != PHBC_W_ROOT) {  // the branch above this op's node: U_p is in ureg, L_p = M_a o M_b
					double tp[PPT][4], xp[PPT][4];
#pragma unroll
					for (int u = 0; u < PPT; u++)
#pragma unroll
						for (int i = 0; i < 4; i++) tp[u][i] = coefp[u] * prm.fq[i] * ureg[u][i], xp[u][i] = ma[u][i] * mb[u][i];
					gstat_add<PPT>(tp, xp, my_gstat + (size_t)d->node * 16, lane);
				}
				if (GRAD == 2 && kind != 2) {  // tip branches: L_n is the tip's indicator vector
					double tt[PPT][4], xt[PPT][4];
#pragma unroll
					for (int u = 0; u < PPT; u++) {
						tip_vector(cds[d->a_code * PB + u * PBT], xt[u]);
#pragma unroll
						for (int i = 0; i < 4; i++) tt[u][i] = coefa[u] * prm.fq[i] * ua[u][i];
					}
					gstat_add<PPT>(tt, xt, my_gstat + (size_t)d->a_node * 16, lane);
					if (kind == 0) {
#pragma unroll
						for (int u = 0; u < PPT; u++) {
							tip_vector(cds[d->b_code * PB + u * PBT], xt[u]);
#pragma unroll
							for (int i = 0; i < 4; i++) tt[u][i] = coefb[u] * prm.fq[i] * ub[u][i];
						}
						gstat_add<PPT>(tt, xt, my_gstat + (size_t)d->b_node * 16, lane);
					}
				}
#pragma unroll
				for (int u = 0; u < PPT; u++) {
					if (kind == 2) cell_store(slot_cell + d->a_slot * NUC4_SLOT_BYTES + u * PBT * 16, ua[u]);  // parked until its own op comes up
					// child b's op is the next one when b is internal; unconditional, so that ub is formed in ureg's registers (a
					// conditional hand-over costs 16 register moves per op) -- after a tip-tip op the next op reloads ureg from its slot
#pragma unroll
					for (int i = 0; i < 4; i++) ureg[u][i] = ub[u][i];
				}
				};
				// messages of the children: the prefetched rows for internal children, matrix columns (or column sums) for tips
				if (ALT) {
#pragma unroll
					const bool tips_ready = RECOMP && (d->flags & PHBC_PRE_TIPS_READY);  // a cherry whose tip messages the previous op left in xa / xb
					if (!tips_ready) {
#pragma unroll
						for (int u = 0; u < PPT; u++) {
							if (kind != 2) tip_message(MA, cds[d->a_code * PB + u * PBT], xa[u]);
							if (kind == 0) tip_message(MB, cds[d->b_code * PB + u * PBT], xb[u]);
						}
					}
					body(xa, xb);
				} else {
					double la[PPT][4], lb[PPT][4];
#pragma unroll
					for (int u = 0; u < PPT; u++) {
						if (kind == 2) {
#pragma unroll
							for (int i = 0; i < 4; i++) la[u][i] = xa[u][i];
						} else tip_message(MA, cds[d->a_code * PB + u * PBT], la[u]);
						if (kind == 0) tip_message(MB, cds[d->b_code * PB + u * PBT], lb[u]);
						else {
#pragma unroll
							for (int i = 0; i < 4; i++) lb[u][i] = xb[u][i];
						}
					}
					prefetch();
					body(la, lb);
				}
			};
			if (tid == 0) issue(0, loads, prm.pre_first_tips);
			mbar_wait(&bars[loads & 1], (loads >> 1) & 1);
			static_assert(NUC4_CHUNK % 2 == 0, "the two operand register sets alternate in pairs of ops");
			double xa[PPT][4], xb[PPT][4], ya[PPT][4], yb[PPT][4], ureg[PPT][4];
#pragma unroll
			for (int u = 0; u < PPT; u++)
#pragma unroll
				for (int i = 0; i < 4; i++) xa[u][i] = xb[u][i] = ya[u][i] = yb[u][i] = ureg[u][i] = 0.0;
			fetch(reinterpret_cast<const phbc_pre_op *>(stage0 + (loads & 1) * lay.bytes + lay.desc_off), xa, xb);
			for (int ch = 0; ch < nchunks; ch++) {
				const unsigned char *st = stage0 + (loads & 1) * lay.bytes;
				const phbc_pre_op *desc = reinterpret_cast<const phbc_pre_op *>(st + lay.desc_off);
				if (tid == 0 && ch + 1 < nchunks) issue(ch + 1, loads + 1, desc[0].next_tips);
				const unsigned char *mats = st + my_mat;
				const uint8_t *cds = st + my_code;
				const int first = ch * NUC4_CHUNK;
				const int cnt = min(NUC4_CHUNK, prm.n_pre - first);
				const bool more = ch + 1 < nchunks;
#pragma unroll 1
				for (int j = 0; j < cnt; j += 2) {
					// two ops (four branches) share one warp butterfly; partial sums go to warp-private rows
					double v0, v1, v2 = 0.0, v3 = 0.0;
					double h0 = 0.0, h1 = 0.0, h2 = 0.0, h3 = 0.0;  // GRAD == 3 only
					if (ALT) pre_op(desc, mats, cds, j, cnt, more, xa, xb, ya, yb, ureg, v0, v1, h0, h1);
					else pre_op(desc, mats, cds, j, cnt, more, xa, xb, xa, xb, ureg, v0, v1, h0, h1);
					if (j + 1 < cnt) {
						if (ALT) pre_op(desc, mats, cds, j + 1, cnt, more, ya, yb, xa, xb, ureg, v2, v3, h2, h3);
						else pre_op(desc, mats, cds, j + 1, cnt, more, xa, xb, xa, xb, ureg, v2, v3, h2, h3);
						const double r = butterfly4(v0, v1, v2, v3, lane);
						if ((lane & 7) == 0) {
							const phbc_pre_op *d = desc + j + ((lane >> 3) & 1);
							red_add_f64(my_gacc + ((lane & 16) ? d->b_node : d->a_node), r);
						}
						if (GRAD == 3) {
							const double rh = butterfly4(h0, h1, h2, h3, lane);
							if ((lane & 7) == 0) {
								const phbc_pre_op *d = desc + j + ((lane >> 3) & 1);
								red_add_f64(my_hacc + ((lane & 16) ? d->b_node : d->a_node), rh);
							}
						}
					} else {
						const double r = butterfly2(v0, v1, lane);
						if ((lane & 15) == 0) red_add_f64(my_gacc + ((lane & 16) ? desc[j].b_node : desc[j].a_node), r);
						if (GRAD == 3) {
							const double rh = butterfly2(h0, h1, lane);
							if ((lane & 15) == 0) red_add_f64(my_hacc + ((lane & 16) ? desc[j].b_node : desc[j].a_node), rh);
						}
					}
				}
				loads++;
				__syncthreads();
			}
		}
	}
	if (cur_b >= 0) flush_lnl(cur_b);
}

// ---------------------------------------------------------------------------------------------
// walk-ordered transition matrices: P(t) = |V exp(L t) V^-1| (substmodel.c:518-557), one thread per
// (matrix, category).  post entries: [op][own|a|b] (own = identity at the root); pre entries: [op][parent|a|b].
// Only tip children need their matrix at the parent's op; entries of internal children are left untouched.
// ---------------------------------------------------------------------------------------------
__global__ void k_nuc4_matrices(int T, int C, int root, int n_post, int n_pre, const phbc_post_op *__restrict__ post_ops,
                                const phbc_pre_op *__restrict__ pre_ops, const double *__restrict__ evec,
                                const double *__restrict__ eval, const double *__restrict__ ivec, const double *__restrict__ bl,
                                const double *__restrict__ rates, double *__restrict__ post_mats, double *__restrict__ pre_mats, int N,
                                long long mats_stride) {
	const int e = blockIdx.x * blockDim.x + threadIdx.x;
	const int total = (3 * n_post + 3 * n_pre) * C;
	if (e >= total) return;
	bl += (size_t)blockIdx.y * N;  // one branch-length vector and one matrix set per sample
	post_mats += (size_t)blockIdx.y * mats_stride;
	pre_mats += (size_t)blockIdx.y * mats_stride;
	const int c = e % C;
	const int m = e / C;
	int node, which;
	double *dst;
	if (m < 3 * n_post) {
		const phbc_post_op op = post_ops[m / 3];
		which = m % 3;
		node = which == 0 ? op.node : (which == 1 ? op.a_node : op.b_node);
		dst = post_mats + (size_t)e * 16;
	} else {
		const int mm = m - 3 * n_post;
		const phbc_pre_op op = pre_ops[mm / 3];
		which = mm % 3;
		node = which == 0 ? op.node : (which == 1 ? op.a_node : op.b_node);
		dst = pre_mats + ((size_t)mm * C + c) * 16;
	}
	if (which != 0 && node >= T) return;  // internal children bring their message along: no matrix needed here
	if (node == root) {
		const double diag = m < 3 * n_post ? 1.0 : 0.0;  // post-order: L_root passes through unchanged
#pragma unroll
		for (int k = 0; k < 16; k++) dst[k] = (k % 5 == 0) ? diag : 0.0;
		return;
	}
	const double t = bl[node] * rates[c];
	double ex[4];
#pragma unroll
	for (int k = 0; k < 4; k++) ex[k] = exp(eval[k] * t);
#pragma unroll
	for (int i = 0; i < 4; i++)
#pragma unroll
		for (int j = 0; j < 4; j++) {
			double acc = 0.0;
#pragma unroll
			for (int k = 0; k < 4; k++) acc = __dadd_rn(acc, __dmul_rn(__dmul_rn(ivec[k * 4 + j], ex[k]), evec[i * 4 + k]));  // substmodel.c:539-555 order
			dst[i * 4 + j] = fabs(acc);
		}
}

// tip encodings -> codes (see tip_message), laid out [walk][tile][k][PB] with row k = the k-th tip the walk consumes.
// states: s < 4 -> s, else 4 (missing).  partials: one-hot -> state, else 0x10 | mask with bit j set when partial[j] == 1;
// anything that is not a 0/1 vector raises *bad (the fused path then declines).  Padding patterns get code 4.
__global__ void k_nuc4_encode_tips(int T, int P, int PB, int ntiles, int tip_kind, const uint8_t *__restrict__ states,
                                   const double *__restrict__ partials, const int *__restrict__ post_order,
                                   const int *__restrict__ pre_order, uint8_t *__restrict__ codes, int *__restrict__ bad) {
	const size_t per_walk = (size_t)ntiles * T * PB;
	const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= 2 * per_walk) return;
	const int walk = i >= per_walk;
	const size_t r = i - walk * per_walk;
	const int pl = (int)(r % PB);
	const int k = (int)((r / PB) % T);
	const int tile = (int)(r / ((size_t)PB * T));
	const int p = tile * PB + pl;
	const int tip = walk ? pre_order[k] : post_order[k];
	unsigned code = 4;
	if (p < P) {
		if (tip_kind == PHBC_TIP_STATES) {
			const unsigned s = states[(size_t)tip * P + p];
			code = s < 4 ? s : 4;
		} else {
			unsigned mask = 0;
			for (int j = 0; j < 4; j++) {
				const double v = partials[((size_t)tip * P + p) * 4 + j];
				if (v == 1.0) mask |= 1u << j;
				else if (v != 0.0) *bad = 1;
			}
			// one-hot vectors become plain states; anything else keeps its mask (row sums for all-ones, treelikelihood4.c:1019-1025)
			code = __popc(mask) == 1 ? (unsigned)(__ffs(mask) - 1) : (0x10u | mask);
		}
	}
	codes[i] = (uint8_t)code;
}

// fixed-order final sums per sample: lnL, cat_grad[n][c] and d lnL / d bl (A11, treelikelihood.c:3129-3143) from the per-CTA /
// per-warp partials.  grid (ceil(N/32), nbatch), block (32, NUC4_FY): x = node, y strides over the CTAs of the walk launch
// that touched the sample (all of them for a single sample; contiguous item ranges for a batch, see k_nuc4_walk).
#define NUC4_FY 16
__global__ void __launch_bounds__(32 * NUC4_FY) k_nuc4_finalize(int N, int C, int nw /* warps per walk CTA */, int grid, int phases, int ntiles, int nbatch, int root,
                                                                const double *__restrict__ cta_lnl, const double *__restrict__ gacc, int want_grad,
                                                                const double *__restrict__ props, const double *__restrict__ rates,
                                                                double *__restrict__ cat_grad, double *__restrict__ result,
                                                                const double *__restrict__ hacc, double *__restrict__ hess) {
	constexpr int warps = NUC4_NT / 32;  // upper bound of nw
	__shared__ double red[NUC4_FY][warps][33];
	const int wpc = nw / C;  // warps per category
	const int tx = threadIdx.x, ty = threadIdx.y;
	const int b = blockIdx.y;
	const long long nitems = (long long)ntiles * nbatch;
	const long long lo = (long long)b * ntiles, hi = lo + ntiles;  // items of this sample
	// CTAs whose item range [c * nitems / grid, (c + 1) * nitems / grid) intersects [lo, hi); one sample: every CTA, phase 0
	int c_lo = 0, c_hi = grid;
	if (nbatch > 1) {
		c_lo = (int)(lo * grid / nitems);
		c_hi = (int)((hi * grid + nitems - 1) / nitems) + 1;
		while (c_lo > 0 && (long long)c_lo * nitems / grid > lo) c_lo--;
		if (c_hi > grid) c_hi = grid;
	}
	result += (size_t)b * (1 + N);
	cat_grad += (size_t)b * N * C;
	auto phase_of = [&](int cta) -> int {  // -1 when the CTA did not touch this sample
		if (nbatch == 1) return 0;
		const long long i0 = (long long)cta * nitems / grid, i1 = (long long)(cta + 1) * nitems / grid;
		if (i1 <= lo || i0 >= hi || i1 <= i0) return -1;
		return b - (int)(i0 / ntiles);
	};
	if (blockIdx.x == 0) {
		double s = 0.0;
		for (int cta = c_lo + ty; cta < c_hi; cta += NUC4_FY) {
			const int ph = phase_of(cta);
			if (ph >= 0 && tx < nw) s += cta_lnl[((size_t)cta * phases + ph) * nw + tx];
		}
		s = phb_warp_sum(s);
		if (tx == 0) red[ty][0][32] = s;
		__syncthreads();
		if (tx == 0 && ty == 0) {
			double tot = 0.0;
			for (int k = 0; k < NUC4_FY; k++) tot += red[k][0][32];
			result[0] = tot;
		}
		__syncthreads();
	}
	if (!want_grad) return;
	const int n = blockIdx.x * 32 + tx;
	// row set 0: gradient rows -> cat_grad, result[1 + n]; row set 1 (hacc != NULL, single sample): Hessian-diagonal rows -> hess[n],
	// the category rows weighted like the gradient's (the kernel folded the second rate factor in)
	for (int set = 0; set < (hacc ? 2 : 1); set++) {
		const double *rows = set ? hacc : gacc;
		double s8[warps];
#pragma unroll
		for (int w = 0; w < warps; w++) s8[w] = 0.0;
		if (n < N && n != root)
			for (int cta = c_lo + ty; cta < c_hi; cta += NUC4_FY) {
				const int ph = phase_of(cta);
				if (ph < 0) continue;
				const double *base = rows + ((size_t)cta * phases + ph) * nw * N + n;
#pragma unroll
				for (int w = 0; w < warps; w++)
					if (w < nw) s8[w] += base[(size_t)w * N];  // independent loads in flight
			}
#pragma unroll
		for (int w = 0; w < warps; w++) red[ty][w][tx] = s8[w];
		__syncthreads();
		if (ty < nw) {  // thread row w sums warp-row w over the CTA slices, fixed order
			double tot = 0.0;
			for (int k = 0; k < NUC4_FY; k++) tot += red[k][ty][tx];
			red[0][ty][tx] = tot;  // slice 0 of row ty is read only by this thread above
		}
		__syncthreads();
		if (ty == 0 && n < N) {
			double g = 0.0;
			for (int c = 0; c < C; c++) {
				double tot = 0.0;
				for (int w = 0; w < wpc; w++) tot += red[0][c * wpc + w][tx];
				if (set == 0) cat_grad[(size_t)n * C + c] = tot;
				if (C == 1) g = tot;
				else g = c == 0 ? tot * props[0] * rates[0] : g + tot * props[c] * rates[c];
			}
			if (set == 0) result[1 + n] = g;
			else hess[n] = C == 1 ? g * rates[0] : g;  // C == 1: the weighting above leaves the rate factor out
		}
		__syncthreads();  // red is reused by the next row set
	}
}

// G[n][c][e] = fixed-order sum of the per-(CTA, warp) statistics rows; warp w of a walk CTA works on category w / (nw / C).
// block (64, NUC4_GY): x = element of the [N][C][16] result, y strides over the (CTA, warp-of-category) rows
#define NUC4_GY 8
__global__ void __launch_bounds__(64 * NUC4_GY) k_nuc4_gstat_sum(int N, int C, int nw, int grid, const double *__restrict__ gstat, double *__restrict__ G) {
	__shared__ double red[NUC4_GY][64];
	const int idx = blockIdx.x * 64 + threadIdx.x;
	const bool live = idx < N * C * 16;
	const int e = idx & 15, c = live ? (idx >> 4) % C : 0, n = live ? (idx >> 4) / C : 0;
	const int wpc = nw / C, rows = grid * wpc;
	double s[4] = {0.0, 0.0, 0.0, 0.0};
	if (live) {
		const double *base = gstat + (size_t)n * 16 + e;
		int r = threadIdx.y;
		for (; r + 3 * NUC4_GY < rows; r += 4 * NUC4_GY) {
#pragma unroll
			for (int q = 0; q < 4; q++) {
				const int rr = r + q * NUC4_GY;
				s[q] += base[((size_t)(rr / wpc) * nw + c * wpc + rr % wpc) * N * 16];
			}
		}
		for (; r < rows; r += NUC4_GY) s[0] += base[((size_t)(r / wpc) * nw + c * wpc + r % wpc) * N * 16];
	}
	red[threadIdx.y][threadIdx.x] = (s[0] + s[1]) + (s[2] + s[3]);
	__syncthreads();
	if (threadIdx.y == 0 && live) {
		double tot = 0.0;
#pragma unroll
		for (int k = 0; k < NUC4_GY; k++) tot += red[k][threadIdx.x];
		G[idx] = tot;
	}
}

// out[k] = sum over nodes n (not the root, not `skip`), categories and matrix entries of props[c] * G[n][c][e] * M[k][n][c][e]
__global__ void k_nuc4_gstat_contract(int N, int C, int root, int skip, const double *__restrict__ G, const double *__restrict__ M /* [nsets][N][C][16] */,
                                      const double *__restrict__ props, double *__restrict__ out) {
	__shared__ double red[256];
	const double *Mk = M + (size_t)blockIdx.x * N * C * 16;
	double s = 0.0;
	for (int nc = threadIdx.x; nc < N * C; nc += blockDim.x) {
		const int n = nc / C, c = nc - n * C;
		if (n == root || n == skip) continue;
		double a = 0.0;
#pragma unroll
		for (int e = 0; e < 16; e++) a = fma(G[(size_t)nc * 16 + e], Mk[(size_t)nc * 16 + e], a);
		s += a * (C == 1 ? 1.0 : props[c]);
	}
	red[threadIdx.x] = s;
	__syncthreads();
	for (int w = blockDim.x / 2; w > 0; w >>= 1) {
		if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
		__syncthreads();
	}
	if (threadIdx.x == 0) out[blockIdx.x] = red[0];
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
// grad: phbc_eval_opts.want_gradient (2: statistics planes under rescaling; 3: two exchange planes and 1 / L_k, unscaled only)
static size_t nuc4_smem_bytes(int C, int PB, int nslots, bool scale, int grad) {
	const bool stat = grad == 2, hess = grad == 3 && !scale;
	return 2 * (size_t)nuc4_stage_layout(C, PB).bytes + (size_t)nslots * NUC4_SLOT_BYTES +
	       (size_t)((scale ? (stat ? 5 : 4) : (hess ? 2 : 1)) * C * PB + (hess ? 2 : 1) * PB + (scale ? nslots * NUC4_NT : 0)) * sizeof(double);
}

static int pattern_block(int C) {
	int pb = (NUC4_NT / C) & ~31;
	return pb;
}

bool phbc_nuc4_supported(const phbc_ctx *ctx, const phbc_eval_opts *o) {
	if (ctx->S != 4 || o->explicit_matrices || !ctx->have_eigen) return false;
	if (ctx->C != 1 && ctx->C != 2 && ctx->C != 4 && ctx->C != 8) return false;  // categories must tile the CTA exactly
	const int PB = pattern_block(ctx->C);
	const int nslots = ctx->post_slots > ctx->pre_slots ? ctx->post_slots : ctx->pre_slots;
	if (nuc4_smem_bytes(ctx->C, PB, nslots, o->scale != 0, o->want_gradient) > ctx->smem_optin) return false;
	return true;
}


static int nuc4_prepare_codes(phbc_ctx *ctx, int *usable);

int phbc_nuc4_evaluate(phbc_ctx *ctx, const phbc_eval_opts *o) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	const int C = ctx->C, N = ctx->N, T = ctx->T, P = ctx->P;
	const int PB = pattern_block(C);
	const int nslots = ctx->post_slots > ctx->pre_slots ? ctx->post_slots : ctx->pre_slots;
	const size_t smem = nuc4_smem_bytes(C, PB, nslots, o->scale != 0, o->want_gradient);
	const int ntiles = (P + PB - 1) / PB;
	// tip codes in walk order (once per tip upload / schedule change)
	{
		int usable = 0;
		const int prc = nuc4_prepare_codes(ctx, &usable);
		if (prc) return prc;
	}
	ctx->last_family = ctx->nuc4_codes_bad ? 1 : 2;
	if (ctx->nuc4_codes_bad) {  // non 0/1 tip partials: node-at-a-time kernels, one sample at a time
		phbc_eval_opts one = *o;
		one.batch_count = 1;
		for (int b = 0; b < (o->batch_count > 1 ? o->batch_count : 1); b++) {
			one.batch_index = o->batch_index + b;
			const int rc = phbc_generic_evaluate(ctx, &one);
			if (rc) return rc;
		}
		return 0;
	}

	// launch geometry: persistent CTAs, two per SM when shared memory allows
	// two patterns per thread (every matrix element read once feeds two FMA chains) wherever a warp still holds one category
	typedef void (*walk_fn)(const Nuc4Params);
	static const walk_fn table[4][2][2] = {
	    {{k_nuc4_walk<1, false, 0, 2>, k_nuc4_walk<1, false, 1, 2>}, {k_nuc4_walk<1, true, 0, 2>, k_nuc4_walk<1, true, 1, 2>}},
	    {{k_nuc4_walk<2, false, 0, 2>, k_nuc4_walk<2, false, 1, 2>}, {k_nuc4_walk<2, true, 0, 2>, k_nuc4_walk<2, true, 1, 2>}},
	    {{k_nuc4_walk<4, false, 0, 2>, k_nuc4_walk<4, false, 1, 2>}, {k_nuc4_walk<4, true, 0, 2>, k_nuc4_walk<4, true, 1, 2>}},
	    {{k_nuc4_walk<8, false, 0, 1>, k_nuc4_walk<8, false, 1, 1>}, {k_nuc4_walk<8, true, 0, 1>, k_nuc4_walk<8, true, 1, 1>}},
	};
	// unscaled walks that also accumulate the expected-transition statistics (phbc_nuc4_matrix_gradient)
	static const walk_fn table_stat[4][2] = {{k_nuc4_walk<1, false, 2, 2>, k_nuc4_walk<1, true, 2, 2>},
	                                         {k_nuc4_walk<2, false, 2, 2>, k_nuc4_walk<2, true, 2, 2>},
	                                         {k_nuc4_walk<4, false, 2, 2>, k_nuc4_walk<4, true, 2, 2>},
	                                         {k_nuc4_walk<8, false, 2, 1>, k_nuc4_walk<8, true, 2, 1>}};
	// unscaled walks that also accumulate the diagonal of the branch-length Hessian (phbc_nuc4_hessian)
	static const walk_fn table_hess[4] = {k_nuc4_walk<1, false, 3, 2>, k_nuc4_walk<2, false, 3, 2>, k_nuc4_walk<4, false, 3, 2>,
	                                      k_nuc4_walk<8, false, 3, 1>};
	const int ppt = C == 8 ? 1 : 2, nthr = NUC4_NT / ppt;
	const int ci = C == 1 ? 0 : (C == 2 ? 1 : (C == 4 ? 2 : 3));
	const bool want_stat = o->want_gradient == 2, want_hess = o->want_gradient == 3;
	if (want_stat && o->batch_count > 1) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "nuc4 walk: transition statistics need a single-sample evaluation");
		return -1;
	}
	if (want_hess && (o->batch_count > 1 || o->scale)) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "nuc4 walk: the Hessian diagonal needs a single unscaled evaluation");
		return -1;
	}
	walk_fn kern = want_hess ? table_hess[ci] : want_stat ? table_stat[ci][o->scale ? 1 : 0] : table[ci][o->scale ? 1 : 0][o->want_gradient ? 1 : 0];
	ctx->nuc4_G_valid = false;
	PHBC_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
	int per_sm = 0;
	PHBC_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, nthr, smem));
	if (per_sm < 1) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "nuc4 walk kernel does not fit on an SM (smem %zu)", smem);
		return -1;
	}
	const int nbatch = o->batch_count > 1 ? o->batch_count : 1;
	const long long nitems = (long long)ntiles * nbatch;
	int grid = per_sm * ctx->num_sms;
	if (grid > nitems) grid = (int)nitems;
	// samples one CTA can touch: its contiguous item range [c * nitems / grid, (c + 1) * nitems / grid)
	int phases = 1;
	for (int cta = 0; cta < grid; cta++) {
		const long long i0 = cta * nitems / grid, i1 = (cta + 1) * nitems / grid;
		if (i1 > i0) {
			const int ph = (int)((i1 - 1) / ntiles - i0 / ntiles) + 1;
			if (ph > phases) phases = ph;
		}
	}
	const int warps = nthr / 32;
	// scratch: walk matrices per sample, per-CTA lower rows, per-(CTA, sample phase, warp) gradient rows and lnL
	const long long mats_stride = (long long)(3 * ctx->n_post + 3 * ctx->n_pre) * C * 16;
	const size_t mats_bytes = (size_t)mats_stride * nbatch * sizeof(double);
	if (mats_bytes > ctx->walk_mats_bytes) {
		PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
		if (ctx->d_walk_mats) cudaFree(ctx->d_walk_mats);
		ctx->d_walk_mats = NULL;
		ctx->walk_mats_bytes = 0;
		PHBC_CHECK(cudaMalloc((void **)&ctx->d_walk_mats, mats_bytes));
		ctx->walk_mats_bytes = mats_bytes;
	}
	if (o->want_gradient) {
		const size_t lower_bytes = (size_t)grid * ctx->n_post * NUC4_ROW_BYTES;
		if (lower_bytes > ctx->walk_lower_bytes) {
			PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
			if (ctx->d_walk_lower) cudaFree(ctx->d_walk_lower);
			ctx->d_walk_lower = NULL;
			ctx->walk_lower_bytes = 0;
			PHBC_CHECK(cudaMalloc((void **)&ctx->d_walk_lower, lower_bytes));
			ctx->walk_lower_bytes = lower_bytes;
		}
		const size_t gacc_bytes = (size_t)grid * phases * warps * N * sizeof(double);
		if (gacc_bytes > ctx->walk_gacc_bytes) {
			PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
			if (ctx->d_walk_gacc) cudaFree(ctx->d_walk_gacc);
			ctx->d_walk_gacc = NULL;
			ctx->walk_gacc_bytes = 0;
			PHBC_CHECK(cudaMalloc((void **)&ctx->d_walk_gacc, gacc_bytes));
			ctx->walk_gacc_bytes = gacc_bytes;
		}
		PHBC_CHECK(cudaMemsetAsync(ctx->d_walk_gacc, 0, gacc_bytes, ctx->stream));
	}
	if (want_stat) {
		const size_t gstat_bytes = (size_t)grid * warps * N * 16 * sizeof(double);
		if (gstat_bytes > ctx->walk_gstat_bytes) {
			PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
			if (ctx->d_walk_gstat) cudaFree(ctx->d_walk_gstat);
			ctx->d_walk_gstat = NULL;
			ctx->walk_gstat_bytes = 0;
			PHBC_CHECK(cudaMalloc((void **)&ctx->d_walk_gstat, gstat_bytes));
			ctx->walk_gstat_bytes = gstat_bytes;
		}
		if (!ctx->d_nuc4_G) PHBC_CHECK(cudaMalloc((void **)&ctx->d_nuc4_G, (size_t)N * C * 16 * sizeof(double)));
		PHBC_CHECK(cudaMemsetAsync(ctx->d_walk_gstat, 0, gstat_bytes, ctx->stream));
	}
	if (want_hess) {
		const size_t hacc_bytes = (size_t)grid * warps * N * sizeof(double);
		if (hacc_bytes > ctx->walk_hacc_bytes) {
			PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
			if (ctx->d_walk_hacc) cudaFree(ctx->d_walk_hacc);
			ctx->d_walk_hacc = NULL;
			ctx->walk_hacc_bytes = 0;
			PHBC_CHECK(cudaMalloc((void **)&ctx->d_walk_hacc, hacc_bytes));
			ctx->walk_hacc_bytes = hacc_bytes;
		}
		if (!ctx->d_nuc4_hess) PHBC_CHECK(cudaMalloc((void **)&ctx->d_nuc4_hess, (size_t)N * sizeof(double)));
		PHBC_CHECK(cudaMemsetAsync(ctx->d_walk_hacc, 0, hacc_bytes, ctx->stream));
	}
	if (!ctx->d_nuc4_cta_lnl || ctx->nuc4_grid < grid * phases) {
		PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
		if (ctx->d_nuc4_cta_lnl) cudaFree(ctx->d_nuc4_cta_lnl);
		ctx->d_nuc4_cta_lnl = NULL;
		ctx->nuc4_grid = 0;
		PHBC_CHECK(cudaMalloc((void **)&ctx->d_nuc4_cta_lnl, (size_t)grid * phases * warps * sizeof(double)));
		ctx->nuc4_grid = grid * phases;
	}
	if (nbatch > ctx->cat_grad_cap) {  // cat_grad [sample][N][C]
		PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
		cudaFree(ctx->d_cat_grad);
		ctx->d_cat_grad = NULL;
		ctx->cat_grad_cap = 0;
		PHBC_CHECK(cudaMalloc((void **)&ctx->d_cat_grad, (size_t)nbatch * N * C * sizeof(double)));
		ctx->cat_grad_cap = nbatch;
	}
	double *post_mats = ctx->d_walk_mats;
	double *pre_mats = ctx->d_walk_mats + (size_t)3 * ctx->n_post * C * 16;
	{
		const int total = (3 * ctx->n_post + 3 * ctx->n_pre) * C;
		k_nuc4_matrices<<<dim3((total + 127) / 128, nbatch), 128, 0, ctx->stream>>>(T, C, ctx->root, ctx->n_post, ctx->n_pre, ctx->d_post_ops, ctx->d_pre_ops,
		                                                                          ctx->d_evec, ctx->d_eval, ctx->d_ivec,
		                                                                          ctx->d_bl + (size_t)o->batch_index * N, ctx->d_rates, post_mats, pre_mats,
		                                                                          N, mats_stride);
		ctx->launches++;
	}
	Nuc4Params prm;
	memset(&prm, 0, sizeof(prm));
	prm.T = T, prm.N = N, prm.C = C, prm.P = P, prm.PB = PB, prm.root = ctx->root;
	prm.n_post = ctx->n_post, prm.n_pre = ctx->n_pre, prm.nslots = nslots, prm.ntiles = ntiles;
	prm.include_root_freqs = o->include_root_freqs, prm.compat = o->compat_scaled_gradient;
	prm.nbatch = nbatch, prm.phases = phases, prm.mats_stride = mats_stride;
	prm.post_first_tips = ctx->post_first_tips, prm.pre_first_tips = ctx->pre_first_tips;
	prm.threshold = o->scaling_threshold;
	prm.tip_codes = ctx->d_nuc4_codes;
	prm.weights = ctx->d_weights;
	prm.props = ctx->d_props;
	prm.post_ops = ctx->d_post_ops;
	prm.pre_ops = ctx->d_pre_ops;
	prm.post_mats = post_mats;
	prm.pre_mats = pre_mats;
	prm.lower = ctx->d_walk_lower;
	prm.gacc = ctx->d_walk_gacc;
	prm.gstat = ctx->d_walk_gstat;
	prm.cta_lnl = ctx->d_nuc4_cta_lnl;
	prm.pattern_lnl = ctx->d_pattern_lnl;
	memcpy(prm.freqs, ctx->h_freqs, sizeof(prm.freqs));  // small model constants travel in the kernel parameter bank
	const bool irf = o->include_root_freqs && !want_hess;  // the Hessian diagonal is always in the exact form
	for (int i = 0; i < 4; i++) {
		prm.fq[i] = irf ? 1.0 : ctx->h_freqs[i];
		prm.wroot[i] = irf ? ctx->h_freqs[i] : 1.0;
		for (int j = 0; j < 4; j++) prm.FQ[4 * i + j] = prm.fq[i] * ctx->h_qmat[4 * i + j];
	}
	if (want_hess) {
		for (int i = 0; i < 4; i++)
			for (int j = 0; j < 4; j++) {
				double q2 = 0.0;
				for (int k = 0; k < 4; k++) q2 += ctx->h_qmat[4 * i + k] * ctx->h_qmat[4 * k + j];
				prm.FQ2[4 * i + j] = ctx->h_freqs[i] * q2;
			}
		prm.rates = ctx->d_rates;
		prm.hacc = ctx->d_walk_hacc;
	}
	int trc;
	if ((trc = phbc_time_begin(ctx))) return trc;
	kern<<<grid, nthr, smem, ctx->stream>>>(prm);
	ctx->launches++;
	if ((trc = phbc_time_end(ctx))) return trc;
	double *result = ctx->d_result + (size_t)o->batch_index * (1 + N);
	k_nuc4_finalize<<<dim3((N + 31) / 32, nbatch), dim3(32, NUC4_FY), 0, ctx->stream>>>(N, C, warps, grid, phases, ntiles, nbatch, ctx->root, ctx->d_nuc4_cta_lnl,
	                                                                         ctx->d_walk_gacc, o->want_gradient, ctx->d_props, ctx->d_rates,
	                                                                         ctx->d_cat_grad, result, want_hess ? ctx->d_walk_hacc : NULL,
	                                                                         want_hess ? ctx->d_nuc4_hess : NULL);
	ctx->launches++;
	if (want_stat) {
		k_nuc4_gstat_sum<<<(N * C * 16 + 63) / 64, dim3(64, NUC4_GY), 0, ctx->stream>>>(N, C, warps, grid, ctx->d_walk_gstat, ctx->d_nuc4_G);
		ctx->launches++;
		ctx->nuc4_G_valid = true;
	}
	PHBC_CHECK(cudaGetLastError());
	return 0;
}

// ---------------------------------------------------------------------------------------------
// substitution-model parameter gradients on the fused walk
// ---------------------------------------------------------------------------------------------
// makes sure the walk-ordered tip codes exist; *usable = 0 when the tips are not 0/1 vectors (the walk then declines)
static int nuc4_prepare_codes(phbc_ctx *ctx, int *usable) {
	const int C = ctx->C, T = ctx->T, P = ctx->P;
	const int PB = pattern_block(C);
	const int ntiles = (P + PB - 1) / PB;
	if (!ctx->d_nuc4_codes) {
		PHBC_CHECK(cudaMalloc((void **)&ctx->d_nuc4_codes, 2 * (size_t)ntiles * T * PB));
		PHBC_CHECK(cudaMalloc((void **)&ctx->d_nuc4_bad, sizeof(int)));
	}
	if (!ctx->nuc4_codes_valid) {
		const size_t n = 2 * (size_t)ntiles * T * PB;
		PHBC_CHECK(cudaMemsetAsync(ctx->d_nuc4_bad, 0, sizeof(int), ctx->stream));
		k_nuc4_encode_tips<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(T, P, PB, ntiles, ctx->tip_kind, ctx->d_tip_states, ctx->d_tip_partials,
		                                                                       ctx->d_post_tip_order, ctx->d_pre_tip_order, ctx->d_nuc4_codes,
		                                                                       ctx->d_nuc4_bad);
		ctx->launches++;
		int bad = 0;
		PHBC_CHECK(cudaMemcpyAsync(&bad, ctx->d_nuc4_bad, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
		PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
		ctx->nuc4_codes_bad = bad != 0;
		ctx->nuc4_codes_valid = true;
	}
	*usable = !ctx->nuc4_codes_bad;
	return 0;
}

/*
 * phbc_matrix_gradient on the fused walk: one GRAD = 2 launch leaves G[n][c][i][j] on the device, every matrix set is then a
 * 16-element contraction per (node, category).  Returns 1 (declined, nothing done) when the walk cannot serve the request:
 * tips that are not 0/1 vectors, a shape phbc_nuc4_supported refuses, or rescaling together with include_root_freqs, the
 * reference-compatible normalisation or a non-reversible model.
 */
int phbc_nuc4_matrix_gradient(phbc_ctx *ctx, const phbc_eval_opts *o, int nsets, const double *M_host, int skip_node, double *lnl, double *out_host) {
	phbc_eval_opts e = *o;
	e.want_gradient = 2;
	e.batch_count = 1;
	if (o->kernels == 1 || !phbc_nuc4_supported(ctx, &e)) return 1;
	if (o->scale) {
		// the scaled form takes each branch's site likelihood from P_p U_p (see the kernel): exact weights and a reversible model
		if (o->include_root_freqs || o->compat_scaled_gradient) return 1;
		double worst = 0.0, big = 0.0;
		for (int i = 0; i < 4; i++)
			for (int j = 0; j < 4; j++) {
				const double a = ctx->h_freqs[i] * ctx->h_qmat[4 * i + j], b = ctx->h_freqs[j] * ctx->h_qmat[4 * j + i];
				worst = fmax(worst, fabs(a - b));
				big = fmax(big, fabs(a));
			}
		if (!(worst <= 1e-12 * big)) return 1;
	}
	PHBC_CHECK(cudaSetDevice(ctx->device));
	int usable = 0, rc;
	if ((rc = nuc4_prepare_codes(ctx, &usable))) return rc;
	if (!usable) return 1;
	if ((rc = phbc_nuc4_evaluate(ctx, &e))) return rc;
	const size_t N = ctx->N, C = ctx->C, set = N * C * 16;
	// matrix sets and results travel through the grow-only reduction scratch (no allocation per request)
	if ((rc = phbc_ensure_scratch(ctx, ((size_t)nsets * set + nsets) * sizeof(double)))) return rc;
	double *d_M = ctx->d_scratch, *d_out = ctx->d_scratch + (size_t)nsets * set;
	PHBC_CHECK(cudaMemcpyAsync(d_M, M_host, (size_t)nsets * set * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
	k_nuc4_gstat_contract<<<nsets, 256, 0, ctx->stream>>>((int)N, (int)C, ctx->root, skip_node, ctx->d_nuc4_G, d_M, ctx->d_props, d_out);
	ctx->launches++;
	PHBC_CHECK(cudaMemcpyAsync(out_host, d_out, (size_t)nsets * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
	if (lnl) PHBC_CHECK(cudaMemcpyAsync(lnl, ctx->d_result + (size_t)e.batch_index * (1 + N), sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
	PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
	PHBC_CHECK(cudaGetLastError());
	return 0;
}

// Diagonal of the branch-length Hessian on the fused walk: one GRAD = 3 launch, then lnL, gradient and hess[N] to the host.  Returns 1
// (declined, nothing done) when the walk cannot serve it (see phb_cuda.h); the caller then takes the resident-partials route.
int phbc_nuc4_hessian(phbc_ctx *ctx, const phbc_eval_opts *o, double *lnl, double *grad, double *hess) {
	phbc_eval_opts e = *o;
	e.want_gradient = 3;
	e.batch_count = 1;
	e.include_root_freqs = 0;
	e.compat_scaled_gradient = 0;
	if (o->kernels == 1 || o->scale || o->batch_count > 1 || !phbc_nuc4_supported(ctx, &e)) return 1;
	PHBC_CHECK(cudaSetDevice(ctx->device));
	int usable = 0, rc;
	if ((rc = nuc4_prepare_codes(ctx, &usable))) return rc;
	if (!usable) return 1;
	if ((rc = phbc_nuc4_evaluate(ctx, &e))) return rc;
	PHBC_CHECK(cudaMemcpyAsync(hess, ctx->d_nuc4_hess, (size_t)ctx->N * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
	if ((rc = phbc_download_results(ctx, 1, lnl, grad))) return rc;  // synchronises the stream
	return 0;
}

// d lnL / d pi_i at fixed partials from the root entry of the statistics: sum_c prop_c G[root][c][i]
int phbc_nuc4_root_frequency_gradient(phbc_ctx *ctx, double *out_host) {
	if (!ctx->nuc4_G_valid) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "transition statistics are not resident");
		return -4;
	}
	PHBC_CHECK(cudaSetDevice(ctx->device));
	double g[8 * 16], props[8];
	const int C = ctx->C;
	PHBC_CHECK(cudaMemcpyAsync(g, ctx->d_nuc4_G + (size_t)ctx->root * C * 16, (size_t)C * 16 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
	PHBC_CHECK(cudaMemcpyAsync(props, ctx->d_props, (size_t)C * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
	PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
	for (int i = 0; i < 4; i++) {
		double s = 0.0;
		for (int c = 0; c < C; c++) s += (C == 1 ? 1.0 : props[c]) * g[c * 16 + i];
		out_host[i] = s;
	}
	return 0;
}

// The transition matrices of the last walk (first sample), from the walk-ordered set k_nuc4_matrices wrote: an internal node's matrix
// is entry 0 of its own post-order op, a tip's is entry 1 / 2 of its parent's op.  dP is what the walk contracts, Q P (see the kernel).
int phbc_nuc4_download_matrices(phbc_ctx *ctx, double *P, double *dP) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	if (!ctx->d_walk_mats) return -4;
	const int C = ctx->C, N = ctx->N, np = ctx->n_post;
	double *mats = (double *)malloc((size_t)3 * np * C * 16 * sizeof(double));
	phbc_post_op *ops = (phbc_post_op *)malloc((size_t)np * sizeof(phbc_post_op));
	double *Pl = P ? P : (double *)malloc((size_t)N * C * 16 * sizeof(double));
	if (!mats || !ops || !Pl) {
		free(mats), free(ops);
		if (!P) free(Pl);
		return -3;
	}
	cudaError_t e = cudaMemcpyAsync(mats, ctx->d_walk_mats, (size_t)3 * np * C * 16 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
	if (e == cudaSuccess) e = cudaMemcpyAsync(ops, ctx->d_post_ops, (size_t)np * sizeof(phbc_post_op), cudaMemcpyDeviceToHost, ctx->stream);
	if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
	if (e == cudaSuccess) {
		memset(Pl, 0, (size_t)N * C * 16 * sizeof(double));
		for (int k = 0; k < np; k++) {
			const int node[3] = {ops[k].node, (ops[k].a_kind & 0xff) == PHBC_W_TIP ? ops[k].a_node : -1, ops[k].b_kind == PHBC_W_TIP ? ops[k].b_node : -1};
			for (int w = 0; w < 3; w++)
				if (node[w] >= 0) memcpy(Pl + (size_t)node[w] * C * 16, mats + ((size_t)3 * k + w) * C * 16, (size_t)C * 16 * sizeof(double));
		}
		if (dP)
			for (int nc = 0; nc < N * C; nc++)
				for (int i = 0; i < 4; i++)
					for (int j = 0; j < 4; j++) {
						double acc = 0.0;
						for (int k = 0; k < 4; k++) acc += ctx->h_qmat[4 * i + k] * Pl[(size_t)nc * 16 + 4 * k + j];
						dP[(size_t)nc * 16 + 4 * i + j] = acc;
					}
	}
	free(mats), free(ops);
	if (!P) free(Pl);
	PHBC_CHECK(e);
	return 0;
}
