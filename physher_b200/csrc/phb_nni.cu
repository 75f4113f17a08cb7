// phb_nni.cu -- scores of nearest-neighbour interchanges on resident upper / lower partials.
//
// An NNI exchanges two subtrees x and y across the branch above v = parent[y] (the "central branch").  The exchanged tree's site
// likelihood is a contraction of four partials the move leaves unchanged, taken at the central branch:
//   kind R (x the sibling of v, p = parent[v]):         L = sum_c prop_c sum_i pi_i [A o M_y]_i       (P_v (M_keep o M_x))_i
//   kind C (across the root, x a child of w):             L = sum_c prop_c sum_i pi_i (P_w (A o M_y))_i (P_v (M_keep o M_x))_i
// with M_n = P_n L_n, keep the child of v that stays, A = P_p U_p (1 when p is the root) for kind R and A = M_keep_w (the child of w
// that stays) for kind C.  d/dt_v and d2/dt_v2 replace P_v by r_c P'_v and r_c^2 P"_v (the matrices k_branch_matrices builds).
// Under rescaling the per-pattern log factor is the sum of the cumulative factors of the four operands (tips carry none).
//
// Routes:
//   4 states   k_nni_score<4>: one thread per pattern, categories looped, both moves of a (v, x) group in one thread -- the
//              operand messages stay in registers, the group's matrices of one category are staged in shared memory;
//   any S      k_nni_operands writes A o M_y and M_keep o M_x of a chunk of moves to scratch, k_nni_contract contracts them.
// Per-CTA partial sums [move][3][tile] go through k_branch_sum (phb_branch.cu): fixed order, bit-identical from run to run.
#include "phb_score.cuh"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#define NNI_THREADS 128
#define NNI_SLOTS 11  // matrices of a group and category: P_x, P_y0, P_keep0, P_A, P_w, then P, P', P" of each of the two moves

// per-pattern log factor of a move's four operands
__device__ __forceinline__ double nni_log_factor(const Bufs &b, const phbc_nni_move &m, int p) {
	double s = 0.0;
	if (m.a >= b.T) s += b.sf[(size_t)m.a * b.P + p];  // U_p (index N + p) or L_keep_w
	if (m.keep >= b.T) s += b.sf[(size_t)m.keep * b.P + p];
	if (m.x >= b.T) s += b.sf[(size_t)m.x * b.P + p];
	if (m.y >= b.T) s += b.sf[(size_t)m.y * b.P + p];
	return s;
}

// out = M x_idx: state tips gather a column (an unknown state gives 1), tip partials and partials a matrix-vector product (message())
template <int S>
__device__ __forceinline__ void nni_message(const Bufs &b, int idx, int c, const double *M, int p, double *out) {
	if (is_state_tip(b, idx)) {
		const int s = b.tip_states[(size_t)idx * b.P + p];
#pragma unroll
		for (int i = 0; i < S; i++) out[i] = s < S ? M[i * S + s] : 1.0;
		return;
	}
	const double *xp = partial_ptr(b, idx, c) + (size_t)p * S;
	double x[S];
#pragma unroll
	for (int j = 0; j < S; j++) x[j] = xp[j];
#pragma unroll
	for (int i = 0; i < S; i++) {
		double acc = 0.0;
#pragma unroll
		for (int j = 0; j < S; j++) acc += M[i * S + j] * x[j];
		out[i] = acc;
	}
}

// source of shared-memory slot `slot` for category c: slots 0-4 the P of x, y, keep, A's owner and w (first matrix of the node's table
// entry), slots 5-10 P, P', P" of the central branch of each move; NULL for a slot the group does not use
template <int SS>
__device__ __forceinline__ const double *nni_slot(const double *mats, int C, int c, int slot, const phbc_nni_move &m0, const phbc_nni_move &m1,
                                                  bool two) {
	int item, q = 0;
	if (slot < 5) {
		item = slot == 0 ? m0.x : slot == 1 ? m0.y : slot == 2 ? m0.keep : slot == 3 ? (m0.a >= 0 ? m0.a_mat : -1) : m0.w;
	} else {
		const int j = (slot - 5) / 3;
		q = (slot - 5) % 3;
		item = j == 0 ? m0.cmat : (two ? m1.cmat : -1);
	}
	return item < 0 ? nullptr : mats + (((size_t)item * C + c) * 3 + q) * SS;
}

// grid (pattern tiles, groups of this launch); group g holds moves groups[g].x and groups[g].y (-1: none), which share x, v, A and
// w and exchange the same children of v (the second one possibly the other child); partial [move][3][tiles]
template <int S>
__global__ void __launch_bounds__(NNI_THREADS) k_nni_score(Bufs b, const int2 *__restrict__ groups, const phbc_nni_move *__restrict__ moves,
                                                         const double *__restrict__ mats, const double *__restrict__ freqs,
                                                         const double *__restrict__ props, const double *__restrict__ weights, int scale,
                                                         double *__restrict__ partial) {
	constexpr int SS = S * S;
	__shared__ double sm[NNI_SLOTS * SS];
	__shared__ double red[6][NNI_THREADS / 32];
	const int p = blockIdx.x * blockDim.x + threadIdx.x;
	const bool live = p < b.P;
	const int2 g = groups[blockIdx.y];
	const phbc_nni_move m0 = moves[g.x];
	const bool two = g.y >= 0;
	const phbc_nni_move m1 = moves[two ? g.y : g.x];
	const bool swap1 = m1.y != m0.y;  // the second move exchanges the other child of v
	const bool cross = m0.w >= 0;
	double acc[2][3] = {{0.0, 0.0, 0.0}, {0.0, 0.0, 0.0}};
	for (int c = 0; c < b.C; c++) {
		__syncthreads();
		for (int e = threadIdx.x; e < NNI_SLOTS * SS; e += blockDim.x) {
			const double *src = nni_slot<SS>(mats, b.C, c, e / SS, m0, m1, two);
			if (src) sm[e] = src[e % SS];
		}
		__syncthreads();
		if (!live) continue;
		double mx[S], my[S], mk[S], a[S];
		nni_message<S>(b, m0.x, c, sm, p, mx);
		nni_message<S>(b, m0.y, c, sm + SS, p, my);
		nni_message<S>(b, m0.keep, c, sm + 2 * SS, p, mk);
		if (m0.a >= 0) {
			nni_message<S>(b, m0.a, c, sm + 3 * SS, p, a);
		} else {
#pragma unroll
			for (int i = 0; i < S; i++) a[i] = 1.0;
		}
		const double pc = b.C == 1 ? 1.0 : props[c];
#pragma unroll
		for (int j = 0; j < 2; j++) {
			if (j == 1 && !two) break;
			const bool sw = j == 1 && swap1;
			double up[S], d[S];
#pragma unroll
			for (int i = 0; i < S; i++) up[i] = a[i] * (sw ? mk[i] : my[i]), d[i] = (sw ? my[i] : mk[i]) * mx[i];
			if (cross) {
				const double *W = sm + 4 * SS;
				double e[S];
#pragma unroll
				for (int i = 0; i < S; i++) {
					double s = 0.0;
#pragma unroll
					for (int k = 0; k < S; k++) s += W[i * S + k] * up[k];
					e[i] = s;
				}
#pragma unroll
				for (int i = 0; i < S; i++) up[i] = e[i];
			}
			const double *M0 = sm + (5 + 3 * j) * SS, *M1 = M0 + SS, *M2 = M1 + SS;
			double a0 = 0.0, a1 = 0.0, a2 = 0.0;
#pragma unroll
			for (int i = 0; i < S; i++) {
				double v0 = 0.0, v1 = 0.0, v2 = 0.0;
#pragma unroll
				for (int k = 0; k < S; k++) v0 += M0[i * S + k] * d[k], v1 += M1[i * S + k] * d[k], v2 += M2[i * S + k] * d[k];
				const double u = freqs[i] * up[i];
				a0 += u * v0, a1 += u * v1, a2 += u * v2;
			}
			acc[j][0] += pc * a0, acc[j][1] += pc * a1, acc[j][2] += pc * a2;
		}
	}
	double v[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
	if (live) {
		const double w = weights[p];
		for (int j = 0; j < 2; j++) {
			if (j == 1 && !two) break;
			const double L = acc[j][0];
			double plk = log(L);
			if (scale) plk += nni_log_factor(b, j ? m1 : m0, p);
			const double r1 = acc[j][1] / L;
			v[3 * j] = plk * w;
			v[3 * j + 1] = r1 * w;
			v[3 * j + 2] = (acc[j][2] / L - r1 * r1) * w;  // the ratio form of score_terms
		}
	}
	// the block sum of score_block_sum, six terms into two rows (written out: the shared helpers change this kernel's code)
	for (int q = 0; q < 6; q++) {
		const double s = phb_warp_sum(v[q]);
		if ((threadIdx.x & 31) == 0) red[q][threadIdx.x >> 5] = s;
	}
	__syncthreads();
	if (threadIdx.x < (two ? 6 : 3)) {
		double s = 0.0;
		for (int w = 0; w < NNI_THREADS / 32; w++) s += red[threadIdx.x][w];
		const int j = threadIdx.x / 3, q = threadIdx.x % 3;
		partial[((size_t)(j ? m1.out : m0.out) * 3 + q) * gridDim.x + blockIdx.x] = s;
	}
}

// any S, step 1: e = A o M_y and d = M_keep o M_x of a chunk of moves; grid (ceil(P / pblk), C, moves of the chunk); e, d [move][C][P][S]
__global__ void k_nni_operands(Bufs b, const phbc_nni_move *__restrict__ moves, const double *__restrict__ mats, int pblk,
                               double *__restrict__ e_out, double *__restrict__ d_out) {
	extern __shared__ double sm[];
	const int S = b.S, SS = S * S;
	double *mA = sm, *mY = sm + SS, *mK = sm + 2 * SS, *mX = sm + 3 * SS;
	const phbc_nni_move m = moves[blockIdx.z];
	const int c = blockIdx.y;
	const size_t stride = 3 * (size_t)SS;
	for (int e = threadIdx.x; e < SS; e += blockDim.x) {
		if (m.a >= 0) mA[e] = mats[((size_t)m.a_mat * b.C + c) * stride + e];
		mY[e] = mats[((size_t)m.y * b.C + c) * stride + e];
		mK[e] = mats[((size_t)m.keep * b.C + c) * stride + e];
		mX[e] = mats[((size_t)m.x * b.C + c) * stride + e];
	}
	__syncthreads();
	const size_t base = ((size_t)blockIdx.z * b.C + c) * b.P * S;
	const int p0 = blockIdx.x * pblk;
	for (int e = threadIdx.x; e < pblk * S; e += blockDim.x) {
		const int p = p0 + e / S, i = e % S;
		if (p >= b.P) break;
		double u = message(b, m.y, c, mY, p, i, true);
		if (m.a >= 0) u *= message(b, m.a, c, mA, p, i, true);
		e_out[base + (size_t)p * S + i] = u;
		d_out[base + (size_t)p * S + i] = message(b, m.keep, c, mK, p, i, true) * message(b, m.x, c, mX, p, i, true);
	}
}

// any S, step 2: grid (pattern tiles, moves of the chunk); one thread per pattern as k_branch_lnl, with the upper side (P_w) e for kind C
__global__ void __launch_bounds__(NNI_THREADS) k_nni_contract(Bufs b, const phbc_nni_move *__restrict__ moves, const double *__restrict__ mats,
                                                            const double *__restrict__ freqs, const double *__restrict__ props,
                                                            const double *__restrict__ weights, int scale, const double *__restrict__ e_in,
                                                            const double *__restrict__ d_in, double *__restrict__ partial) {
	extern __shared__ double sm[];
	__shared__ double red[3][NNI_THREADS / 32];
	const int S = b.S, SS = S * S;
	const int p = blockIdx.x * blockDim.x + threadIdx.x;
	const bool live = p < b.P;
	const phbc_nni_move m = moves[blockIdx.y];
	const bool cross = m.w >= 0;
	const size_t stride = 3 * (size_t)SS;
	double L = 0.0, dL = 0.0, d2L = 0.0;
	for (int c = 0; c < b.C; c++) {
		__syncthreads();
		const double *src = mats + ((size_t)m.cmat * b.C + c) * stride;
		for (int e = threadIdx.x; e < 3 * SS; e += blockDim.x) sm[e] = src[e];
		if (cross)
			for (int e = threadIdx.x; e < SS; e += blockDim.x) sm[3 * SS + e] = mats[((size_t)m.w * b.C + c) * stride + e];
		__syncthreads();
		if (!live) continue;
		const size_t off = (((size_t)blockIdx.y * b.C + c) * b.P + p) * S;
		const double *ev = e_in + off, *dv = d_in + off;
		double a0 = 0.0, a1 = 0.0, a2 = 0.0;
		for (int i = 0; i < S; i++) {
			const double *m0 = sm + i * S, *m1 = sm + SS + i * S, *m2 = sm + 2 * SS + i * S;
			double v0 = 0.0, v1 = 0.0, v2 = 0.0;
			for (int j = 0; j < S; j++) {
				const double xj = dv[j];
				v0 += m0[j] * xj, v1 += m1[j] * xj, v2 += m2[j] * xj;
			}
			double up;
			if (cross) {
				const double *wr = sm + 3 * SS + i * S;
				up = 0.0;
				for (int j = 0; j < S; j++) up += wr[j] * ev[j];
			} else {
				up = ev[i];
			}
			const double u = freqs[i] * up;
			a0 += u * v0, a1 += u * v1, a2 += u * v2;
		}
		const double pc = b.C == 1 ? 1.0 : props[c];
		L += pc * a0, dL += pc * a1, d2L += pc * a2;
	}
	double v[3] = {0.0, 0.0, 0.0};
	if (live) {
		const double w = weights[p];
		double plk = log(L);
		if (scale) plk += nni_log_factor(b, m, p);
		score_terms(plk, L, dL, d2L, w, v);
	}
	score_block_sum(red, v, NNI_THREADS / 32, m.out, partial);
}

// out_host [nmoves][3]; bl_host [N + nmoves]: every node's length (root entry unused), then each move's central length; ex_host
// (may be NULL) [N + nmoves][C][S] exp(eval * bl * rate); groups_host: the moves paired by (v, x), in launch order
extern "C" int phbc_nni_scores(phbc_ctx *ctx, const phbc_eval_opts *o, int nmoves, const phbc_nni_move *moves_host, int ngroups,
                               const int *groups_host, const double *bl_host, const double *ex_host, double *out_host) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	const size_t S = ctx->S, C = ctx->C, P = ctx->P, N = ctx->N;
	if (nmoves < 1) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "%d moves: at least one is needed", nmoves);
		return -1;
	}
	if (!ctx->have_eigen || o->explicit_matrices) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "NNI scores need the eigen system (explicit matrices cannot be re-evaluated at a new length)");
		return -4;
	}
	int rc;
	if ((rc = phbc_score_resident(ctx, o))) return rc;
	const size_t n = (size_t)nmoves, items = N + n;
	const size_t tiles = (P + NNI_THREADS - 1) / NNI_THREADS;
	ScoreScratch sc;
	if ((rc = phbc_score_scratch(ctx, items, n, 3, tiles, 2 * (size_t)ngroups * sizeof(int) + n * sizeof(phbc_nni_move), &sc))) return rc;
	int2 *d_groups = static_cast<int2 *>(sc.desc);  // the 32-byte descriptors follow
	phbc_nni_move *d_moves = reinterpret_cast<phbc_nni_move *>(d_groups + ngroups);
	PHBC_CHECK(cudaMemcpyAsync(d_moves, moves_host, n * sizeof(phbc_nni_move), cudaMemcpyHostToDevice, ctx->stream));
	if (ngroups > 0) PHBC_CHECK(cudaMemcpyAsync(d_groups, groups_host, 2 * (size_t)ngroups * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
	if ((rc = phbc_score_matrices(ctx, sc, items, bl_host, ex_host))) return rc;
	Bufs b = phbc_make_bufs(ctx);
	// any S: operand scratch of a chunk of moves, e and d [chunk][C][P][S], at most a quarter of the free memory and 4 GiB, allocated
	// before the timed window; PHB_NNI_CHUNK_MOVES caps the chunk (tests run the multi-chunk loop on small trees with it)
	const size_t per_move = 2 * C * P * S;
	size_t chunk = 0;
	double *d_vec = NULL;
	if (S != 4) {
		size_t free_b = 0, total_b = 0;
		PHBC_CHECK(cudaMemGetInfo(&free_b, &total_b));
		const size_t budget = free_b / 4 < ((size_t)4 << 30) ? free_b / 4 : ((size_t)4 << 30);
		chunk = budget / (per_move * sizeof(double));
		const char *cap = getenv("PHB_NNI_CHUNK_MOVES");
		if (cap && atol(cap) > 0 && (size_t)atol(cap) < chunk) chunk = (size_t)atol(cap);
		if (chunk < 1) chunk = 1;
		if (chunk > n) chunk = n;
		if (chunk > 65535) chunk = 65535;
		if ((rc = phbc_alloc(ctx, &d_vec, chunk * per_move, false))) return rc;
	}
	auto launch = [&]() -> int {
		int rc;
		if (S != 4) {
			const size_t osmem = 4 * S * S * sizeof(double), csmem = 4 * S * S * sizeof(double);
			if (osmem > 48 * 1024) PHBC_CHECK(cudaFuncSetAttribute(k_nni_operands, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)osmem));
			if (csmem > 48 * 1024) PHBC_CHECK(cudaFuncSetAttribute(k_nni_contract, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)csmem));
		}
		if ((rc = phbc_time_begin(ctx))) return rc;
		if (S == 4) {
			for (int g0 = 0; g0 < ngroups; g0 += 65535) {
				const int cnt = ngroups - g0 < 65535 ? ngroups - g0 : 65535;
				k_nni_score<4><<<dim3((unsigned)tiles, (unsigned)cnt), NNI_THREADS, 0, ctx->stream>>>(b, d_groups + g0, d_moves, sc.mats, ctx->d_freqs,
				                                                                                    ctx->d_props, ctx->d_weights, o->scale, sc.part);
				ctx->launches++;
			}
		} else {
			const int pblk = S <= 8 ? 512 : (S <= 32 ? 128 : 32);  // as k_generic_combine
			const size_t osmem = 4 * S * S * sizeof(double), csmem = 4 * S * S * sizeof(double);
			for (size_t m0 = 0; m0 < n; m0 += chunk) {
				const size_t cnt = n - m0 < chunk ? n - m0 : chunk;
				double *d_e = d_vec, *d_d = d_vec + cnt * C * P * S;
				k_nni_operands<<<dim3((unsigned)((P + pblk - 1) / pblk), (unsigned)C, (unsigned)cnt), 256, osmem, ctx->stream>>>(b, d_moves + m0, sc.mats,
				                                                                                                              pblk, d_e, d_d);
				k_nni_contract<<<dim3((unsigned)tiles, (unsigned)cnt), NNI_THREADS, csmem, ctx->stream>>>(b, d_moves + m0, sc.mats, ctx->d_freqs,
				                                                                                        ctx->d_props, ctx->d_weights, o->scale, d_e,
				                                                                                        d_d, sc.part);
				ctx->launches += 2;
			}
		}
		if ((rc = phbc_time_end(ctx))) return rc;
		return phbc_score_finish(ctx, sc, n, 3, tiles, out_host);
	};
	rc = launch();
	if (d_vec) {  // on every path: the stream is drained before the scratch goes
		const cudaError_t e = cudaStreamSynchronize(ctx->stream);
		cudaFree(d_vec);
		if (!rc && e != cudaSuccess) PHBC_CHECK(e);
	}
	return rc;
}

// ---------------------------------------------------------------------------------------------
// quintet scores: every move with its five branches free
// ---------------------------------------------------------------------------------------------
//
// Numbering the branches of the exchanged tree c = v (central), k = keep, x, y, o (kind R: p's own branch, o absent when p is the root;
// kind C: keep_w's branch), with M^d_n = P^d_n L_n for d = 0, 1, 2 (P, r P', r^2 P" at the move's own length of branch n):
//   B = M_k o M_x, B_k = M'_k o M_x, B_x = M_k o M'_x, B_kk = M"_k o M_x, B_xx = M_k o M"_x, B_kx = M'_k o M'_x     (v's end)
//   A = M_y o M_o and its six variants in y and o likewise, then P_w (w at its current length) applied to each for kind C (the far end)
//   L_ab = sum_c prop_c sum_i pi_i [A variant]_i (P^d_c [B variant])_i
// which takes the central products P_c {B, B_k, B_x, B_kk, B_xx, B_kx}, P'_c {B, B_k, B_x} and P"_c B.  21 sums per pattern: L, the
// five first derivatives (c, k, x, y, o) and the fifteen second derivatives of the upper triangle, row by row (cc ck cx cy co kk kx ky ko
// xx xy xo yy yo oo).  Matrix table: items cmat .. cmat + 4 are c, k, x, y, o of the move, item w is w at its current length.
//   4 states   k_nni_quintet<4>: one thread per pattern, categories looped, the sixteen matrices of one (move, category) staged in shared
//              memory (2 KiB), the operands and the twelve side vectors in registers.  The moves of one (v, x) group are not paired: two
//              moves' side vectors and sums do not fit the registers of a 128-thread CTA.
//   any S      k_nni_quintet_any: np patterns per CTA, 128 / np threads per pattern splitting the rows; the six B-side vectors (and for
//              kind C the six raw A-side vectors) of the CTA's patterns in shared memory, [vector][S][np], so that the central products
//              read whole vectors without a round trip through device memory; the matrices are read through the L1 cache, every
//              thread of a row group reading the same row.

#define QUINTET_TERMS 21
#define QUINTET_SLOTS 16  // P, P', P" of c, k, x, y, o, then P_w

// the 21 sums of one row i: a[6] the far-end variants (A, A_y, A_o, A_yy, A_oo, A_yo) at i times f = prop_c pi_i, cv[10] the central
// products at i (P B, P B_k, P B_x, P B_kk, P B_xx, P B_kx, P' B, P' B_k, P' B_x, P" B)
__device__ __forceinline__ void quintet_accumulate(double *acc, const double *a, const double *cv) {
	acc[0] += a[0] * cv[0];
	acc[1] += a[0] * cv[6], acc[2] += a[0] * cv[1], acc[3] += a[0] * cv[2], acc[4] += a[1] * cv[0], acc[5] += a[2] * cv[0];
	acc[6] += a[0] * cv[9], acc[7] += a[0] * cv[7], acc[8] += a[0] * cv[8], acc[9] += a[1] * cv[6], acc[10] += a[2] * cv[6];
	acc[11] += a[0] * cv[3], acc[12] += a[0] * cv[5], acc[13] += a[1] * cv[1], acc[14] += a[2] * cv[1];
	acc[15] += a[0] * cv[4], acc[16] += a[1] * cv[2], acc[17] += a[2] * cv[2];
	acc[18] += a[3] * cv[0], acc[19] += a[5] * cv[0], acc[20] += a[4] * cv[0];
}

// the weighted terms of one pattern in the ratio form of score_terms: w lnL, w L_a / L, w (L_ab / L - L_a L_b / L^2)
__device__ __forceinline__ void quintet_terms(double plk, const double *Ls, double w, double *v) {
	const double L = Ls[0];
	double r[5];
#pragma unroll
	for (int a = 0; a < 5; a++) r[a] = Ls[1 + a] / L, v[1 + a] = r[a] * w;
	v[0] = plk * w;
	int q = 6;
#pragma unroll
	for (int a = 0; a < 5; a++)
#pragma unroll
		for (int bb = a; bb < 5; bb++, q++) v[q] = (Ls[q] / L - r[a] * r[bb]) * w;
}

// the six products of two operands' messages m, n (each through P, r P', r^2 P"): m n, m' n, m n', m" n, m n", m' n'
__device__ __forceinline__ void quintet_side(const double *m, const double *n, double *out) {
	out[0] = m[0] * n[0], out[1] = m[1] * n[0], out[2] = m[0] * n[1], out[3] = m[2] * n[0], out[4] = m[0] * n[2], out[5] = m[1] * n[1];
}

// the three messages of operand idx through M, M + SS, M + 2 SS (P, r P', r^2 P"): state tips gather a column, an unknown state gives 1
// for P and the row sums for the derivatives, tip partials and partials are multiplied (message())
template <int S>
__device__ __forceinline__ void quintet_message(const Bufs &b, int idx, int c, const double *M, int p, double (&out)[3][S]) {
	constexpr int SS = S * S;
	if (is_state_tip(b, idx)) {
		const int s = b.tip_states[(size_t)idx * b.P + p];
#pragma unroll
		for (int d = 0; d < 3; d++)
#pragma unroll
			for (int i = 0; i < S; i++) {
				double r = 0.0;
#pragma unroll
				for (int j = 0; j < S; j++) r += M[d * SS + i * S + j];
				out[d][i] = s < S ? M[d * SS + i * S + s] : (d == 0 ? 1.0 : r);
			}
		return;
	}
	const double *xp = partial_ptr(b, idx, c) + (size_t)p * S;
	double x[S];
#pragma unroll
	for (int j = 0; j < S; j++) x[j] = xp[j];
#pragma unroll
	for (int d = 0; d < 3; d++)
#pragma unroll
		for (int i = 0; i < S; i++) {
			double acc = 0.0;
#pragma unroll
			for (int j = 0; j < S; j++) acc += M[d * SS + i * S + j] * x[j];
			out[d][i] = acc;
		}
}

// grid (pattern tiles, moves m0 .. m0 + gridDim.y - 1 in launch order); partial [move][21][tiles]
template <int S>
__global__ void __launch_bounds__(NNI_THREADS) k_nni_quintet(Bufs b, const phbc_nni_move *__restrict__ moves, int m0, const double *__restrict__ mats,
                                                           const double *__restrict__ freqs, const double *__restrict__ props,
                                                           const double *__restrict__ weights, int scale, double *__restrict__ partial) {
	constexpr int SS = S * S;
	__shared__ double sm[QUINTET_SLOTS * SS];
	__shared__ double red[QUINTET_TERMS][NNI_THREADS / 32];
	const int p = blockIdx.x * blockDim.x + threadIdx.x;
	const bool live = p < b.P;
	const phbc_nni_move m = moves[m0 + blockIdx.y];
	const bool cross = m.w >= 0;
	double tot[QUINTET_TERMS];
#pragma unroll
	for (int q = 0; q < QUINTET_TERMS; q++) tot[q] = 0.0;
	for (int c = 0; c < b.C; c++) {
		__syncthreads();
		for (int e = threadIdx.x; e < 15 * SS; e += blockDim.x) sm[e] = mats[((size_t)(m.cmat + e / (3 * SS)) * b.C + c) * 3 * SS + e % (3 * SS)];
		if (cross)
			for (int e = threadIdx.x; e < SS; e += blockDim.x) sm[15 * SS + e] = mats[((size_t)m.w * b.C + c) * 3 * SS + e];
		__syncthreads();
		if (!live) continue;
		double B[S][6], A[S][6];
		{
			double mk[3][S], mx[3][S];
			quintet_message<S>(b, m.keep, c, sm + 3 * SS, p, mk);
			quintet_message<S>(b, m.x, c, sm + 6 * SS, p, mx);
#pragma unroll
			for (int i = 0; i < S; i++) {
				const double u[3] = {mk[0][i], mk[1][i], mk[2][i]}, w[3] = {mx[0][i], mx[1][i], mx[2][i]};
				quintet_side(u, w, B[i]);
			}
		}
		{
			double my[3][S], mo[3][S];
			quintet_message<S>(b, m.y, c, sm + 9 * SS, p, my);
			if (m.a >= 0) {
				quintet_message<S>(b, m.a, c, sm + 12 * SS, p, mo);
			} else {  // p is the root: no fourth branch
#pragma unroll
				for (int i = 0; i < S; i++) mo[0][i] = 1.0, mo[1][i] = mo[2][i] = 0.0;
			}
#pragma unroll
			for (int i = 0; i < S; i++) {
				const double u[3] = {my[0][i], my[1][i], my[2][i]}, w[3] = {mo[0][i], mo[1][i], mo[2][i]};
				quintet_side(u, w, A[i]);
			}
		}
		if (cross) {  // the far end through P_w
			const double *W = sm + 15 * SS;
#pragma unroll
			for (int q = 0; q < 6; q++) {
				double e[S];
#pragma unroll
				for (int i = 0; i < S; i++) {
					double s = 0.0;
#pragma unroll
					for (int j = 0; j < S; j++) s += W[i * S + j] * A[j][q];
					e[i] = s;
				}
#pragma unroll
				for (int i = 0; i < S; i++) A[i][q] = e[i];
			}
		}
		const double pc = b.C == 1 ? 1.0 : props[c];
#pragma unroll
		for (int i = 0; i < S; i++) {
			double cv[10];
#pragma unroll
			for (int q = 0; q < 10; q++) cv[q] = 0.0;
#pragma unroll
			for (int j = 0; j < S; j++) {
				const double p0 = sm[i * S + j], p1 = sm[SS + i * S + j], p2 = sm[2 * SS + i * S + j];
#pragma unroll
				for (int q = 0; q < 6; q++) cv[q] += p0 * B[j][q];
#pragma unroll
				for (int q = 0; q < 3; q++) cv[6 + q] += p1 * B[j][q];
				cv[9] += p2 * B[j][0];
			}
			const double f = pc * freqs[i];
			double a[6];
#pragma unroll
			for (int q = 0; q < 6; q++) a[q] = f * A[i][q];
			quintet_accumulate(tot, a, cv);
		}
	}
	double v[QUINTET_TERMS];
#pragma unroll
	for (int q = 0; q < QUINTET_TERMS; q++) v[q] = 0.0;
	if (live) {
		double plk = log(tot[0]);
		if (scale) plk += nni_log_factor(b, m, p);
		quintet_terms(plk, tot, weights[p], v);
	}
	score_block_sum(red, v, 0, m.out, partial);
}

// one row of the three messages through P, r P', r^2 P" (rows m, m + SS, m + 2 SS) of an operand: a state tip gathers a column, an
// unknown state gives 1 for P and the row sums for the derivatives, partials are multiplied (message()); a NULL m (no fourth branch)
// gives 1, 0, 0
__device__ __forceinline__ void quintet_row(const double *__restrict__ m, int S, int SS, bool state, int code, const double *x, double *out) {
	out[0] = out[1] = out[2] = 0.0;
	if (!m) {
		out[0] = 1.0;
	} else if (state && code < S) {
		for (int d = 0; d < 3; d++) out[d] = __ldg(m + d * SS + code);
	} else if (state) {
		out[0] = 1.0;
		for (int j = 0; j < S; j++) out[1] += __ldg(m + SS + j), out[2] += __ldg(m + 2 * SS + j);
	} else {
		for (int j = 0; j < S; j++) {
			const double xj = x[j];
			out[0] += __ldg(m + j) * xj, out[1] += __ldg(m + SS + j) * xj, out[2] += __ldg(m + 2 * SS + j) * xj;
		}
	}
}

// any S: grid (pattern blocks of np, moves m0 ..), NNI_THREADS threads -- pattern blockIdx.x * np + threadIdx.x % np, rows
// threadIdx.x / np (mod NNI_THREADS / np); dynamic shared memory max(12 S np, 21 NNI_THREADS) doubles
__global__ void __launch_bounds__(NNI_THREADS) k_nni_quintet_any(Bufs b, const phbc_nni_move *__restrict__ moves, int m0, int np,
                                                               const double *__restrict__ mats, const double *__restrict__ freqs,
                                                               const double *__restrict__ props, const double *__restrict__ weights, int scale,
                                                               double *__restrict__ partial) {
	extern __shared__ double sm[];
	__shared__ double red[QUINTET_TERMS][NNI_THREADS / 32];
	const int S = b.S, SS = S * S, G = NNI_THREADS / np;
	const int pp = threadIdx.x % np, g = threadIdx.x / np;
	const int p = blockIdx.x * np + pp;
	const bool live = p < b.P;
	const phbc_nni_move m = moves[m0 + blockIdx.y];
	const bool cross = m.w >= 0;
	const int ids[4] = {m.keep, m.x, m.y, m.a};
	bool state[4];
	int code[4];
#pragma unroll
	for (int o = 0; o < 4; o++) {
		state[o] = ids[o] >= 0 && is_state_tip(b, ids[o]);
		code[o] = state[o] && live ? b.tip_states[(size_t)ids[o] * b.P + p] : 0;
	}
	double tot[QUINTET_TERMS];
#pragma unroll
	for (int q = 0; q < QUINTET_TERMS; q++) tot[q] = 0.0;
	const size_t stride = 3 * (size_t)SS;
	for (int c = 0; c < b.C; c++) {
		const double *Mc = mats + ((size_t)m.cmat * b.C + c) * stride;
		const double *Mn[4];  // keep, x, y, o
		const double *X[4];
#pragma unroll
	for (int o = 0; o < 4; o++) {
			Mn[o] = o == 3 && m.a < 0 ? nullptr : mats + ((size_t)(m.cmat + 1 + o) * b.C + c) * stride;
			X[o] = state[o] || ids[o] < 0 || !live ? nullptr : partial_ptr(b, ids[o], c) + (size_t)p * S;
		}
		__syncthreads();
		if (live) {
			for (int j = g; j < S; j += G) {
				double u[3], w[3], s6[6];
				quintet_row(Mn[0] + j * S, S, SS, state[0], code[0], X[0], u);
				quintet_row(Mn[1] + j * S, S, SS, state[1], code[1], X[1], w);
				quintet_side(u, w, s6);
#pragma unroll
				for (int q = 0; q < 6; q++) sm[((size_t)q * S + j) * np + pp] = s6[q];
				if (cross) {
					quintet_row(Mn[2] + j * S, S, SS, state[2], code[2], X[2], u);
					quintet_row(Mn[3] + j * S, S, SS, state[3], code[3], X[3], w);
					quintet_side(u, w, s6);
#pragma unroll
					for (int q = 0; q < 6; q++) sm[((size_t)(6 + q) * S + j) * np + pp] = s6[q];
				}
			}
		}
		__syncthreads();
		if (!live) continue;
		const double pc = b.C == 1 ? 1.0 : props[c];
		const double *W = cross ? mats + ((size_t)m.w * b.C + c) * stride : nullptr;
		for (int i = g; i < S; i += G) {
			double a[6];
			if (cross) {
#pragma unroll
				for (int q = 0; q < 6; q++) a[q] = 0.0;
				for (int j = 0; j < S; j++) {
					const double wj = __ldg(W + (size_t)i * S + j);
#pragma unroll
					for (int q = 0; q < 6; q++) a[q] += wj * sm[((size_t)(6 + q) * S + j) * np + pp];
				}
			} else {
				double u[3], w[3];
				quintet_row(Mn[2] + i * S, S, SS, state[2], code[2], X[2], u);
				quintet_row(Mn[3] ? Mn[3] + i * S : nullptr, S, SS, state[3], code[3], X[3], w);
				quintet_side(u, w, a);
			}
			double cv[10];
#pragma unroll
			for (int q = 0; q < 10; q++) cv[q] = 0.0;
			const double *r0 = Mc + (size_t)i * S, *r1 = r0 + SS, *r2 = r1 + SS;
			for (int j = 0; j < S; j++) {
				const double p0 = __ldg(r0 + j), p1 = __ldg(r1 + j), p2 = __ldg(r2 + j);
				double bv[6];
#pragma unroll
				for (int q = 0; q < 6; q++) bv[q] = sm[((size_t)q * S + j) * np + pp];
#pragma unroll
				for (int q = 0; q < 6; q++) cv[q] += p0 * bv[q];
#pragma unroll
				for (int q = 0; q < 3; q++) cv[6 + q] += p1 * bv[q];
				cv[9] += p2 * bv[0];
			}
			const double f = pc * freqs[i];
#pragma unroll
			for (int q = 0; q < 6; q++) a[q] *= f;
			quintet_accumulate(tot, a, cv);
		}
	}
	// the row groups' sums of each pattern, added in a fixed order
	__syncthreads();
#pragma unroll
	for (int q = 0; q < QUINTET_TERMS; q++) sm[q * NNI_THREADS + threadIdx.x] = tot[q];
	__syncthreads();
	double v[QUINTET_TERMS];
#pragma unroll
	for (int q = 0; q < QUINTET_TERMS; q++) v[q] = 0.0;
	if (live && g == 0) {
#pragma unroll
		for (int q = 0; q < QUINTET_TERMS; q++) {
			double s = 0.0;
			for (int h = 0; h < G; h++) s += sm[q * NNI_THREADS + h * np + pp];
			tot[q] = s;
		}
		double plk = log(tot[0]);
		if (scale) plk += nni_log_factor(b, m, p);
		quintet_terms(plk, tot, weights[p], v);
	}
	score_block_sum(red, v, 0, m.out, partial);
}

// patterns per CTA of the any-S kernel: the most of 32, 16, 8 whose twelve side vectors fit 48 KiB, else 8
static int quintet_np(int S) {
	for (int np = 32; np > 8; np /= 2)
		if (12 * (size_t)S * np * sizeof(double) <= 48 * 1024) return np;
	return 8;
}

static size_t quintet_smem(int S) {
	const size_t vec = 12 * (size_t)S * quintet_np(S), sums = QUINTET_TERMS * (size_t)NNI_THREADS;
	return (vec > sums ? vec : sums) * sizeof(double);
}

// out_host [nmoves][21]; moves_host in launch order (out = the output row), cmat the first of the move's five table items c, k, x, y,
// o; bl_host [N + 5 nmoves]: every node's length (root entry unused), then each move's five lengths; ex_host (may be NULL) their
// exponentials [N + 5 nmoves][C][S]
extern "C" int phbc_nni_quintet_scores(phbc_ctx *ctx, const phbc_eval_opts *o, int nmoves, const phbc_nni_move *moves_host, const double *bl_host,
                                       const double *ex_host, double *out_host) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	const size_t S = ctx->S, P = ctx->P, N = ctx->N;
	if (nmoves < 1) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "%d moves: at least one is needed", nmoves);
		return -1;
	}
	if (!ctx->have_eigen || o->explicit_matrices) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "NNI quintet scores need the eigen system (explicit matrices cannot be re-evaluated at a new length)");
		return -4;
	}
	int rc;
	if ((rc = phbc_score_resident(ctx, o))) return rc;
	const size_t n = (size_t)nmoves, items = N + 5 * n;
	const int np = S == 4 ? NNI_THREADS : quintet_np((int)S);
	const size_t tiles = (P + np - 1) / np, smem = S == 4 ? 0 : quintet_smem((int)S);
	ScoreScratch sc;
	if ((rc = phbc_score_scratch(ctx, items, n, QUINTET_TERMS, tiles, n * sizeof(phbc_nni_move), &sc))) return rc;
	phbc_nni_move *d_moves = static_cast<phbc_nni_move *>(sc.desc);
	PHBC_CHECK(cudaMemcpyAsync(d_moves, moves_host, n * sizeof(phbc_nni_move), cudaMemcpyHostToDevice, ctx->stream));
	if ((rc = phbc_score_matrices(ctx, sc, items, bl_host, ex_host))) return rc;
	// the dynamic size is always declared: the block-sum array's static bytes count toward the 48 KiB default too
	if (S != 4) PHBC_CHECK(cudaFuncSetAttribute(k_nni_quintet_any, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
	Bufs b = phbc_make_bufs(ctx);
	if ((rc = phbc_time_begin(ctx))) return rc;
	for (size_t m0 = 0; m0 < n; m0 += 65535) {
		const unsigned cnt = (unsigned)(n - m0 < 65535 ? n - m0 : 65535);
		if (S == 4)
			k_nni_quintet<4><<<dim3((unsigned)tiles, cnt), NNI_THREADS, 0, ctx->stream>>>(b, d_moves, (int)m0, sc.mats, ctx->d_freqs, ctx->d_props,
			                                                                           ctx->d_weights, o->scale, sc.part);
		else
			k_nni_quintet_any<<<dim3((unsigned)tiles, cnt), NNI_THREADS, smem, ctx->stream>>>(b, d_moves, (int)m0, np, sc.mats, ctx->d_freqs,
			                                                                               ctx->d_props, ctx->d_weights, o->scale, sc.part);
		ctx->launches++;
	}
	if ((rc = phbc_time_end(ctx))) return rc;
	return phbc_score_finish(ctx, sc, n, QUINTET_TERMS, tiles, out_host);
}
