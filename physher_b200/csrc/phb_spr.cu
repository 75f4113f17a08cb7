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
#include "phb_ctx.cuh"

#include <math.h>
#include <stdlib.h>
#include <string.h>

// phb_branch.cu
__global__ void k_branch_matrices(int S, int C, const double *__restrict__ evec, const double *__restrict__ eval, const double *__restrict__ ivec,
                                  const double *__restrict__ bl, const double *__restrict__ rates, const double *__restrict__ ex_host,
                                  double *__restrict__ mats);
__global__ void k_branch_sum(const double *__restrict__ partial, int n, double *__restrict__ out);

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

// block reduction of the three per-pattern terms into partial [target][3][tiles]
template <int WARPS>
__device__ __forceinline__ void spr_block_sum(double (*red)[WARPS], const double *v, int k, double *partial) {
	for (int q = 0; q < 3; q++) {
		const double s = phb_warp_sum(v[q]);
		if ((threadIdx.x & 31) == 0) red[q][threadIdx.x >> 5] = s;
	}
	__syncthreads();
	if (threadIdx.x < 3) {
		double s = 0.0;
		for (int w = 0; w < (int)(blockDim.x >> 5); w++) s += red[threadIdx.x][w];
		partial[((size_t)k * 3 + threadIdx.x) * gridDim.x + blockIdx.x] = s;
	}
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
		const double r1 = dL / L;
		v[0] = plk * wt;
		v[1] = r1 * wt;
		v[2] = (d2L / L - r1 * r1) * wt;
	}
	spr_block_sum<SPR_THREADS / 32>(red, v, k, partial);
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
		const double r1 = dL / L;
		v[0] = plk * wt;
		v[1] = r1 * wt;
		v[2] = (d2L / L - r1 * r1) * wt;
	}
	spr_block_sum<SPR_ANY_THREADS_MAX / 32>(red, v, k, partial);
}

// threads per CTA of the score kernel: any S takes more where its five matrices leave room for one CTA per SM only
static int spr_threads(const phbc_ctx *ctx) {
	const size_t smem = 5 * (size_t)ctx->S * ctx->S * sizeof(double);
	return ctx->S == 4 ? SPR_THREADS : (smem > 48 * 1024 ? SPR_ANY_THREADS_MAX : SPR_THREADS);
}

// the scratch of one call, sized and allocated before the pruned pass overwrites anything, so that a state count the kernels cannot
// stage (-1) or a device too small for the matrix table (-3) is reported with the object unchanged:
//   bl [items] | results [n][3] | matrices [items][C][3][S*S] | partial [n][3][tiles] | host exponentials [items][C][S] | targets
extern "C" int phbc_spr_reserve(phbc_ctx *ctx, int ntargets) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	const size_t S = ctx->S, C = ctx->C, P = ctx->P, N = ctx->N;
	const size_t smem = 5 * S * S * sizeof(double);
	if (S != 4 && smem > ctx->smem_optin) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "SPR scores: %zu states need %zu bytes of shared memory for five matrices (at most %zu)", S, smem,
		         ctx->smem_optin);
		return -1;
	}
	const size_t n = ntargets > 0 ? (size_t)ntargets : 1, items = N + n;
	const size_t tiles = (P + spr_threads(ctx) - 1) / spr_threads(ctx);
	const size_t need = (items * (1 + C * 3 * S * S + C * S) + n * (3 + 3 * tiles) + (n + 1) / 2) * sizeof(double);
	if (need <= ctx->branch_bytes) return 0;
	PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
	if (ctx->d_branch) cudaFree(ctx->d_branch);
	ctx->d_branch = NULL;
	ctx->branch_bytes = 0;
	const cudaError_t e = cudaMalloc((void **)&ctx->d_branch, need);
	if (e == cudaErrorMemoryAllocation) {
		(void)cudaGetLastError();
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "out of device memory: %.1f GB for the SPR matrix table and sums", need / 1e9);
		return -3;
	}
	PHBC_CHECK(e);
	ctx->branch_bytes = need;
	return 0;
}

// out_host [ntargets][3]; bl_host [N + ntargets]: every node's length (root entry unused), then each target's pendant length; ex_host
// (may be NULL) [N + ntargets][C][S] exp(eval * bl * rate).  The pruned tree's partials must be in the resident buffers.
extern "C" int phbc_spr_scores(phbc_ctx *ctx, const phbc_eval_opts *o, int s, int p, int ntargets, const int *targets_host,
                               const double *bl_host, const double *ex_host, double *out_host) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	const size_t S = ctx->S, C = ctx->C, P = ctx->P, N = ctx->N;
	if (ntargets < 1) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "%d targets: at least one is needed", ntargets);
		return -1;
	}
	if (!ctx->have_eigen || o->explicit_matrices) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "SPR scores need the eigen system (explicit matrices cannot be re-evaluated at a new length)");
		return -4;
	}
	if (!ctx->d_upper || !ctx->d_lower || (o->scale && !ctx->d_sf) || (ctx->tip_kind != PHBC_TIP_STATES && !ctx->d_tip_partials)) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "upper / lower partials are not resident");
		return -4;
	}
	int rc;
	if ((rc = phbc_spr_reserve(ctx, ntargets))) return rc;  // nothing to do when the caller reserved first
	const size_t smem = 5 * S * S * sizeof(double);
	const int threads = spr_threads(ctx);
	const size_t n = (size_t)ntargets, items = N + n;
	const size_t tiles = (P + threads - 1) / threads;
	double *d_bl = ctx->d_branch, *d_out = d_bl + items, *d_mats = d_out + 3 * n, *d_part = d_mats + items * C * 3 * S * S;
	double *d_exbuf = d_part + n * 3 * tiles;
	double *d_ex = ex_host ? d_exbuf : NULL;
	int *d_targets = reinterpret_cast<int *>(d_exbuf + items * C * S);
	PHBC_CHECK(cudaMemcpyAsync(d_bl, bl_host, items * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
	PHBC_CHECK(cudaMemcpyAsync(d_targets, targets_host, n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
	if (ex_host) PHBC_CHECK(cudaMemcpyAsync(d_ex, ex_host, items * C * S * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
	const int mthreads = S * S >= 256 ? 256 : (S * S >= 64 ? 64 : 32);
	k_branch_matrices<<<dim3((unsigned)items, (unsigned)C), mthreads, 3 * S * sizeof(double), ctx->stream>>>((int)S, (int)C, ctx->d_evec, ctx->d_eval,
	                                                                                                    ctx->d_ivec, d_bl, ctx->d_rates, d_ex, d_mats);
	ctx->launches++;
	if (S != 4 && smem > 48 * 1024) PHBC_CHECK(cudaFuncSetAttribute(k_spr_score_any, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
	Bufs b = phbc_make_bufs(ctx);
	if ((rc = phbc_time_begin(ctx))) return rc;
	for (size_t k0 = 0; k0 < n; k0 += 65535) {
		const unsigned cnt = (unsigned)(n - k0 < 65535 ? n - k0 : 65535);
		if (S == 4)
			k_spr_score<4><<<dim3((unsigned)tiles, cnt), threads, 0, ctx->stream>>>(b, s, p, d_targets, (int)k0, d_mats, ctx->d_freqs, ctx->d_props,
			                                                                     ctx->d_weights, o->scale, d_part);
		else
			k_spr_score_any<<<dim3((unsigned)tiles, cnt), threads, smem, ctx->stream>>>(b, s, p, d_targets, (int)k0, d_mats, ctx->d_freqs, ctx->d_props,
			                                                                          ctx->d_weights, o->scale, d_part);
		ctx->launches++;
	}
	if ((rc = phbc_time_end(ctx))) return rc;
	k_branch_sum<<<(unsigned)(3 * n), 256, 0, ctx->stream>>>(d_part, (int)tiles, d_out);
	ctx->launches++;
	PHBC_CHECK(cudaGetLastError());
	PHBC_CHECK(cudaMemcpyAsync(out_host, d_out, 3 * n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
	PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
	return 0;
}
