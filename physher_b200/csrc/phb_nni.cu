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
	if ((rc = phbc_score_scratch(ctx, items, n, tiles, 2 * (size_t)ngroups * sizeof(int) + n * sizeof(phbc_nni_move), &sc))) return rc;
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
		return phbc_score_finish(ctx, sc, n, tiles, out_host);
	};
	rc = launch();
	if (d_vec) {  // on every path: the stream is drained before the scratch goes
		const cudaError_t e = cudaStreamSynchronize(ctx->stream);
		cudaFree(d_vec);
		if (!rc && e != cudaSuccess) PHBC_CHECK(e);
	}
	return rc;
}
