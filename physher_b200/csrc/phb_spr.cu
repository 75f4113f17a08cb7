// phb_spr.cu -- scores of subtree prune-and-regraft moves on the resident partials of the pruned tree.
//
// Prune the subtree of s together with p = parent[s] (the sibling b of s takes p's slot under g = parent[p]) and regraft it on the
// branch above a target e of the pruned tree: p takes e's slot, e and s become p's children.  With the pruned tree's upper and lower
// partials U~_e (buffer N + e, the upper_ops convention: P_sib L~_sib when e's pruned parent is the root) and L~_e (buffer e), the
// regrafted tree's site likelihood is one contraction at the pendant branch of s:
//   L = sum_c prop_c sum_i pi_i [(P_p U~_e) o (P_e L~_e)]_i (P_s L_s)_i
// d/dt_s and d2/dt_s2 replace P_s by r_c P'_s and r_c^2 P"_s (the matrices k_branch_matrices builds).  Under rescaling the per-pattern
// log factor is sf[N + e] + sf[e] + sf[s] (tips carry none).  The host writes the pruned tree's partials over the resident buffers
// first (phb_treelikelihood.c, spr_pass); this file holds the contraction only.
//
// Routes:
//   4 states   k_spr_score<4>: one thread per pattern, categories looped, the operand vectors in registers;
//   any S      k_spr_score_any: the same contraction row by row, operands read straight from the resident buffers (no scratch).
// Both stage the five matrices of one (target, category) -- P_p, P_e, and P_s, P'_s, P"_s at the pendant length -- in shared memory,
// take targets on grid.y (launches of at most 65,535) and write per-CTA sums [target][3][tile] that k_branch_sum (phb_branch.cu)
// reduces in a fixed order: bit-identical from run to run, no floating-point atomics.
#include "phb_score.cuh"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#define SPR_THREADS 128
#define SPR_ANY_THREADS_MAX 512

// source of shared-memory slot `slot` (0 P_p, 1 P_e, 2-4 P, P', P" of the pendant length) for target k and category c; the matrix
// table holds [item][C][3][S*S]: node n at its current length = item n, target k's pendant length = item N + k
__device__ __forceinline__ const double *spr_slot(const double *mats, int N, int C, int c, int slot, int p, int e, int k, int SS) {
	const int item = slot == 0 ? p : (slot == 1 ? e : N + k);
	const int q = slot < 2 ? 0 : slot - 2;
	return mats + (((size_t)item * C + c) * 3 + q) * SS;
}

// per-pattern log factor of the three operands
__device__ __forceinline__ double spr_log_factor(const Bufs &b, int s, int e, int p) {
	double f = b.sf[(size_t)(b.N + e) * b.P + p];
	if (e >= b.T) f += b.sf[(size_t)e * b.P + p];
	if (s >= b.T) f += b.sf[(size_t)s * b.P + p];
	return f;
}

// grid (pattern tiles, targets k0 .. k0 + gridDim.y - 1)
template <int S>
__global__ void __launch_bounds__(SPR_THREADS) k_spr_score(Bufs b, int s, int pn, const int *__restrict__ targets, int k0,
                                                         const double *__restrict__ mats, const double *__restrict__ freqs,
                                                         const double *__restrict__ props, const double *__restrict__ weights, int scale,
                                                         double *__restrict__ partial) {
	constexpr int SS = S * S;
	__shared__ double sm[5 * SS];
	__shared__ double red[3][SPR_THREADS / 32];
	const int p = blockIdx.x * blockDim.x + threadIdx.x;
	const bool live = p < b.P;
	const int k = k0 + blockIdx.y;
	const int e = targets[k];
	const bool s_state = is_state_tip(b, s), e_state = is_state_tip(b, e);
	const int s_code = s_state && live ? b.tip_states[(size_t)s * b.P + p] : 0;
	const int e_code = e_state && live ? b.tip_states[(size_t)e * b.P + p] : 0;
	double L = 0.0, dL = 0.0, d2L = 0.0;
	for (int c = 0; c < b.C; c++) {
		__syncthreads();
		for (int x = threadIdx.x; x < 5 * SS; x += blockDim.x) sm[x] = spr_slot(mats, b.N, b.C, c, x / SS, pn, e, k, SS)[x % SS];
		__syncthreads();
		if (!live) continue;
		const double *Pp = sm, *Pe = sm + SS, *M0 = sm + 2 * SS, *M1 = sm + 3 * SS, *M2 = sm + 4 * SS;
		double u[S], x[S], y[S], w[S];
		const double *up = partial_ptr(b, b.N + e, c) + (size_t)p * S;
#pragma unroll
		for (int j = 0; j < S; j++) u[j] = up[j];
		if (!e_state) {
			const double *xp = partial_ptr(b, e, c) + (size_t)p * S;
#pragma unroll
			for (int j = 0; j < S; j++) x[j] = xp[j];
		}
		if (!s_state) {
			const double *yp = partial_ptr(b, s, c) + (size_t)p * S;
#pragma unroll
			for (int j = 0; j < S; j++) y[j] = yp[j];
		}
#pragma unroll
		for (int i = 0; i < S; i++) {
			double a = 0.0;
#pragma unroll
			for (int j = 0; j < S; j++) a += Pp[i * S + j] * u[j];
			double m;
			if (e_state) {
				m = e_code < S ? Pe[i * S + e_code] : 1.0;
			} else {
				m = 0.0;
#pragma unroll
				for (int j = 0; j < S; j++) m += Pe[i * S + j] * x[j];
			}
			w[i] = freqs[i] * a * m;
		}
		double a0 = 0.0, a1 = 0.0, a2 = 0.0;
#pragma unroll
		for (int i = 0; i < S; i++) {
			double v0 = 0.0, v1 = 0.0, v2 = 0.0;
			if (s_state && s_code < S) {
				v0 = M0[i * S + s_code], v1 = M1[i * S + s_code], v2 = M2[i * S + s_code];
			} else if (s_state) {  // unknown state: 1 for P, the row sums of the derivative matrices (message())
				v0 = 1.0;
#pragma unroll
				for (int j = 0; j < S; j++) v1 += M1[i * S + j], v2 += M2[i * S + j];
			} else {
#pragma unroll
				for (int j = 0; j < S; j++) v0 += M0[i * S + j] * y[j], v1 += M1[i * S + j] * y[j], v2 += M2[i * S + j] * y[j];
			}
			a0 += w[i] * v0, a1 += w[i] * v1, a2 += w[i] * v2;
		}
		const double pc = b.C == 1 ? 1.0 : props[c];
		L += pc * a0, dL += pc * a1, d2L += pc * a2;
	}
	double v[3] = {0.0, 0.0, 0.0};
	if (live) {
		const double wt = weights[p];
		double plk = log(L);
		if (scale) plk += spr_log_factor(b, s, e, p);
		score_terms(plk, L, dL, d2L, wt, v);
	}
	score_block_sum(red, v, 0, k, partial);
}

// any S: grid (pattern tiles, targets k0 ..), dynamic shared memory 5 S^2 doubles; row i of every product is formed where it is used
__global__ void __launch_bounds__(SPR_ANY_THREADS_MAX) k_spr_score_any(Bufs b, int s, int pn, const int *__restrict__ targets, int k0,
                                                                     const double *__restrict__ mats, const double *__restrict__ freqs,
                                                                     const double *__restrict__ props, const double *__restrict__ weights,
                                                                     int scale, double *__restrict__ partial) {
	extern __shared__ double sm[];
	__shared__ double red[3][SPR_ANY_THREADS_MAX / 32];
	const int S = b.S, SS = S * S;
	const int p = blockIdx.x * blockDim.x + threadIdx.x;
	const bool live = p < b.P;
	const int k = k0 + blockIdx.y;
	const int e = targets[k];
	const bool s_state = is_state_tip(b, s);
	double L = 0.0, dL = 0.0, d2L = 0.0;
	for (int c = 0; c < b.C; c++) {
		__syncthreads();
		for (int x = threadIdx.x; x < 5 * SS; x += blockDim.x) sm[x] = spr_slot(mats, b.N, b.C, c, x / SS, pn, e, k, SS)[x % SS];
		__syncthreads();
		if (!live) continue;
		const double *U = partial_ptr(b, b.N + e, c) + (size_t)p * S;
		const double *Y = s_state ? nullptr : partial_ptr(b, s, c) + (size_t)p * S;
		double a0 = 0.0, a1 = 0.0, a2 = 0.0;
		for (int i = 0; i < S; i++) {
			const double *pp = sm + i * S, *m0 = sm + 2 * SS + i * S, *m1 = sm + 3 * SS + i * S, *m2 = sm + 4 * SS + i * S;
			double a = 0.0, v0 = 0.0, v1 = 0.0, v2 = 0.0;
			for (int j = 0; j < S; j++) a += pp[j] * U[j];
			const double m = message(b, e, c, sm + SS, p, i, true);
			if (s_state) {
				v0 = message(b, s, c, sm + 2 * SS, p, i, true);
				v1 = message(b, s, c, sm + 3 * SS, p, i, false);
				v2 = message(b, s, c, sm + 4 * SS, p, i, false);
			} else {
				for (int j = 0; j < S; j++) {
					const double yj = Y[j];
					v0 += m0[j] * yj, v1 += m1[j] * yj, v2 += m2[j] * yj;
				}
			}
			const double w = freqs[i] * a * m;
			a0 += w * v0, a1 += w * v1, a2 += w * v2;
		}
		const double pc = b.C == 1 ? 1.0 : props[c];
		L += pc * a0, dL += pc * a1, d2L += pc * a2;
	}
	double v[3] = {0.0, 0.0, 0.0};
	if (live) {
		const double wt = weights[p];
		double plk = log(L);
		if (scale) plk += spr_log_factor(b, s, e, p);
		score_terms(plk, L, dL, d2L, wt, v);
	}
	score_block_sum(red, v, 0, k, partial);
}

// threads per CTA of the score kernel: any S takes more where its five matrices leave room for one CTA per SM only
static int spr_threads(const phbc_ctx *ctx) {
	const size_t smem = 5 * (size_t)ctx->S * ctx->S * sizeof(double);
	return ctx->S == 4 ? SPR_THREADS : (smem > 48 * 1024 ? SPR_ANY_THREADS_MAX : SPR_THREADS);
}

// the scratch of one call (the layout of phb_score.cuh, descriptors = the targets), sized and allocated before the pruned pass
// overwrites anything, so that a state count the kernels cannot stage (-1) or a device too small for the matrix table (-3) is reported
// with the object unchanged
static int spr_scratch(phbc_ctx *ctx, int ntargets, ScoreScratch *sc) {
	const size_t S = ctx->S;
	const size_t smem = 5 * S * S * sizeof(double);
	if (S != 4 && smem > ctx->smem_optin) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "SPR scores: %zu states need %zu bytes of shared memory for five matrices (at most %zu)", S, smem,
		         ctx->smem_optin);
		return -1;
	}
	const size_t n = ntargets > 0 ? (size_t)ntargets : 1;
	const size_t tiles = ((size_t)ctx->P + spr_threads(ctx) - 1) / spr_threads(ctx);
	return phbc_score_scratch(ctx, ctx->N + n, n, tiles, n * sizeof(int), sc);
}

extern "C" int phbc_spr_reserve(phbc_ctx *ctx, int ntargets) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	ScoreScratch sc;
	return spr_scratch(ctx, ntargets, &sc);
}

// out_host [ntargets][3]; bl_host [N + ntargets]: every node's length (root entry unused), then each target's pendant length; ex_host
// (may be NULL) [N + ntargets][C][S] exp(eval * bl * rate).  The pruned tree's partials must be in the resident buffers.
extern "C" int phbc_spr_scores(phbc_ctx *ctx, const phbc_eval_opts *o, int s, int p, int ntargets, const int *targets_host,
                               const double *bl_host, const double *ex_host, double *out_host) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	const size_t S = ctx->S, P = ctx->P, N = ctx->N;
	if (ntargets < 1) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "%d targets: at least one is needed", ntargets);
		return -1;
	}
	if (!ctx->have_eigen || o->explicit_matrices) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "SPR scores need the eigen system (explicit matrices cannot be re-evaluated at a new length)");
		return -4;
	}
	int rc;
	if ((rc = phbc_score_resident(ctx, o))) return rc;
	ScoreScratch sc;
	if ((rc = spr_scratch(ctx, ntargets, &sc))) return rc;  // nothing to allocate when the caller reserved first
	const size_t smem = 5 * S * S * sizeof(double);
	const int threads = spr_threads(ctx);
	const size_t n = (size_t)ntargets;
	const size_t tiles = (P + threads - 1) / threads;
	const int *d_targets = static_cast<int *>(sc.desc);
	PHBC_CHECK(cudaMemcpyAsync(sc.desc, targets_host, n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
	if ((rc = phbc_score_matrices(ctx, sc, N + n, bl_host, ex_host))) return rc;
	if (S != 4 && smem > 48 * 1024) PHBC_CHECK(cudaFuncSetAttribute(k_spr_score_any, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
	Bufs b = phbc_make_bufs(ctx);
	if ((rc = phbc_time_begin(ctx))) return rc;
	for (size_t k0 = 0; k0 < n; k0 += 65535) {
		const unsigned cnt = (unsigned)(n - k0 < 65535 ? n - k0 : 65535);
		if (S == 4)
			k_spr_score<4><<<dim3((unsigned)tiles, cnt), threads, 0, ctx->stream>>>(b, s, p, d_targets, (int)k0, sc.mats, ctx->d_freqs, ctx->d_props,
			                                                                     ctx->d_weights, o->scale, sc.part);
		else
			k_spr_score_any<<<dim3((unsigned)tiles, cnt), threads, smem, ctx->stream>>>(b, s, p, d_targets, (int)k0, sc.mats, ctx->d_freqs, ctx->d_props,
			                                                                          ctx->d_weights, o->scale, sc.part);
		ctx->launches++;
	}
	if ((rc = phbc_time_end(ctx))) return rc;
	return phbc_score_finish(ctx, sc, n, tiles, out_host);
}
