// phb_branch.cu -- single-branch fast path on resident upper / lower partials.
//
// Replaces, for one branch at a time, the reference's "upper likelihood" functions used by Brent / Newton branch optimisation,
// NNI / SPR and Model.d2logP:
//   _calculate_uppper        treelikelihood.c:2592-2686  lnL from U_n, L_n and a fresh P(t) of node n
//   calculate_dldt_uppper    treelikelihood.c:2195-2262  per-pattern dL/dt from r dP/dt
//   d2lnldt2_uppper          treelikelihood.c:2267-2335  d2 lnL / dt2 from r^2 d2P/dt2
// all three through calculate_branch_partials (treelikelihoodX.c:878-1001) + integrate_partials + a frequency-weighted sum:
//   L_k(t)  = sum_c prop_c sum_i pi_i U_n[c,k,i] (P(r_c t) L_n[c,k])_i          lnL   = sum_k w_k (log L_k + sf_k)
//   L'_k(t) = sum_c prop_c r_c   sum_i pi_i U_n[c,k,i] (P'(r_c t) L_n[c,k])_i   lnL'  = sum_k w_k L'_k / L_k
//   L"_k(t) = sum_c prop_c r_c^2 sum_i pi_i U_n[c,k,i] (P"(r_c t) L_n[c,k])_i   lnL"  = sum_k w_k (L"_k L_k - L'_k^2) / L_k^2
// The reference evaluates one candidate length per call, each a full pass over two partials buffers; here ONE launch takes a list
// of (node, length) items: one node at a vector of candidate lengths (a bracketing step or a line search, whose CTAs read the same
// two buffers concurrently and share them through L2), or every non-root node at its own length (the diagonal of the
// branch-length Hessian, phb_tlk_branch_hessian_diagonal, with the gradient and lnL of the same pass).
//
// Under rescaling the per-pattern log factor is sf_upper[n] + sf_lower[n] (the factors that were divided out of U_n and L_n);
// the derivative ratios are scale free.
#include "phb_ctx.cuh"

#include <math.h>
#include <stdlib.h>
#include <string.h>

// P(t), r P'(t), r^2 P"(t) for every (item, category): grid (nitems, C); mats [nitems][C][3][S*S]
// (p_t substmodel.c:518-557 with fabs, dp_dt :695-723, d2p_d2t :801-828; same operation order, no fused multiply-add)
__global__ void k_branch_matrices(int S, int C, const double *__restrict__ evec, const double *__restrict__ eval, const double *__restrict__ ivec,
                                  const double *__restrict__ bl, const double *__restrict__ rates, const double *__restrict__ ex_host,
                                  double *__restrict__ mats) {
	extern __shared__ double sm[];
	double *e0 = sm, *e1 = sm + S, *e2 = sm + 2 * S;
	const int k = blockIdx.x, c = blockIdx.y;
	const double r = rates[c];
	const double t = bl[k] * r;
	for (int q = threadIdx.x; q < S; q += blockDim.x) {
		const double l = eval[q];
		const double e = ex_host ? ex_host[((size_t)k * C + c) * S + q] : exp(l * t);  // see k_transition_matrices
		e0[q] = e;
		e1[q] = l * e;
		e2[q] = l * l * e;
	}
	__syncthreads();
	double *dst = mats + ((size_t)k * C + c) * 3 * S * S;
	for (int e = threadIdx.x; e < S * S; e += blockDim.x) {
		const int i = e / S, j = e % S;
		double p = 0.0, d = 0.0, d2 = 0.0;
		for (int q = 0; q < S; q++) {
			const double iv = ivec[q * S + j], ev = evec[i * S + q];
			p = __dadd_rn(p, __dmul_rn(__dmul_rn(iv, e0[q]), ev));
			d = __dadd_rn(d, __dmul_rn(__dmul_rn(iv, e1[q]), ev));
			d2 = __dadd_rn(d2, __dmul_rn(__dmul_rn(iv, e2[q]), ev));
		}
		dst[e] = fabs(p);
		dst[S * S + e] = d * r;             // treelikelihood.c:2235-2237
		dst[2 * S * S + e] = d2 * r * r;    // :2298-2300
	}
}

#define BR_THREADS 128

// grid (pattern tiles, nitems); one thread per pattern; item k is the branch above nodes[k]; partial [nitems][3][tiles]
__global__ void __launch_bounds__(BR_THREADS) k_branch_lnl(Bufs b, const int *__restrict__ nodes, const double *__restrict__ mats,
                                                        const double *__restrict__ freqs, const double *__restrict__ props,
                                                        const double *__restrict__ weights, int scale, double *__restrict__ partial) {
	extern __shared__ double sm[];
	__shared__ double red[3][BR_THREADS / 32];
	const int S = b.S, SS = S * S;
	const int p = blockIdx.x * blockDim.x + threadIdx.x;
	const bool live = p < b.P;
	const int k = blockIdx.y;
	const int node = nodes[k];
	const bool tip = is_state_tip(b, node);
	const int s_tip = (tip && live) ? b.tip_states[(size_t)node * b.P + p] : 0;
	double L = 0.0, dL = 0.0, d2L = 0.0;
	for (int c = 0; c < b.C; c++) {
		__syncthreads();
		const double *src = mats + ((size_t)k * b.C + c) * 3 * SS;
		for (int e = threadIdx.x; e < 3 * SS; e += blockDim.x) sm[e] = src[e];
		__syncthreads();
		if (!live) continue;
		const double *U = partial_ptr(b, b.N + node, c) + (size_t)p * S;
		const double *x = tip ? nullptr : partial_ptr(b, node, c) + (size_t)p * S;
		double a0 = 0.0, a1 = 0.0, a2 = 0.0;
		for (int i = 0; i < S; i++) {
			const double *m0 = sm + i * S, *m1 = sm + SS + i * S, *m2 = sm + 2 * SS + i * S;
			double v0 = 0.0, v1 = 0.0, v2 = 0.0;
			if (tip && s_tip < S) {
				v0 = m0[s_tip], v1 = m1[s_tip], v2 = m2[s_tip];
			} else if (tip) {  // unknown state: the row sums (treelikelihoodX.c:878-1001)
				for (int j = 0; j < S; j++) v0 += m0[j], v1 += m1[j], v2 += m2[j];
			} else {
				for (int j = 0; j < S; j++) {
					const double xj = x[j];
					v0 += m0[j] * xj, v1 += m1[j] * xj, v2 += m2[j] * xj;
				}
			}
			const double u = freqs[i] * U[i];
			a0 += u * v0, a1 += u * v1, a2 += u * v2;
		}
		const double pc = b.C == 1 ? 1.0 : props[c];
		L += pc * a0, dL += pc * a1, d2L += pc * a2;
	}
	double v[3] = {0.0, 0.0, 0.0};
	if (live) {
		const double w = weights[p];
		double plk = log(L);
		if (scale) {
			plk += b.sf[(size_t)(b.N + node) * b.P + p];
			if (!tip) plk += b.sf[(size_t)node * b.P + p];
		}
		v[0] = plk * w;
		const double r1 = dL / L;
		v[1] = r1 * w;
		// treelikelihood.c:2331 forms (L" L - L'^2) / L^2, which underflows to 0 / 0 once L_k < 1e-154 -- site likelihoods a tree of a
		// thousand taxa reaches without rescaling; the ratio form is the same value and stays finite
		v[2] = (d2L / L - r1 * r1) * w;
	}
	for (int q = 0; q < 3; q++) {
		const double s = phb_warp_sum(v[q]);
		if ((threadIdx.x & 31) == 0) red[q][threadIdx.x >> 5] = s;
	}
	__syncthreads();
	if (threadIdx.x < 3) {
		double s = 0.0;
		for (int w = 0; w < BR_THREADS / 32; w++) s += red[threadIdx.x][w];
		partial[((size_t)k * 3 + threadIdx.x) * gridDim.x + blockIdx.x] = s;
	}
}

// out[row] = sum of partial[row][0..n): one CTA per row, fixed order
__global__ void k_branch_sum(const double *__restrict__ partial, int n, double *__restrict__ out) {
	__shared__ double red[8];
	const double *in = partial + (size_t)blockIdx.x * n;
	double v = 0.0;
	for (int i = threadIdx.x; i < n; i += blockDim.x) v += in[i];
	v = phb_warp_sum(v);
	if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
	__syncthreads();
	if (threadIdx.x == 0) {
		double s = 0.0;
		for (int w = 0; w < (int)(blockDim.x >> 5); w++) s += red[w];
		out[blockIdx.x] = s;
	}
}

// out_host [nitems][3]: lnL, d lnL / dt, d2 lnL / dt2 of the branch above nodes[k] at length bl[k]; U and L of every listed node must be
// resident.  One node repeated: candidate lengths of one branch; distinct nodes: one entry per branch.
extern "C" int phbc_branch_lnl(phbc_ctx *ctx, const phbc_eval_opts *o, int nitems, const int *nodes_host, const double *bl_host, const double *ex_host,
                               double *out_host) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	const size_t S = ctx->S, C = ctx->C, P = ctx->P;
	if (nitems < 1 || nitems > 65535) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "%d branch items: out of range (1 .. 65535 per launch)", nitems);
		return -1;
	}
	if (!ctx->have_eigen || o->explicit_matrices) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "the single-branch path needs the eigen system (explicit matrices cannot be re-evaluated at a new length)");
		return -4;
	}
	for (int k = 0; k < nitems; k++) {
		const int node = nodes_host[k];
		if (node < 0 || node >= ctx->N || node == ctx->root) {
			snprintf(phbc_errbuf, sizeof(phbc_errbuf), "branch %d (root %d): out of range", node, ctx->root);
			return -1;
		}
		if (!ctx->d_upper || (node >= ctx->T && !ctx->d_lower) || (o->scale && !ctx->d_sf) ||
		    (node < ctx->T && ctx->tip_kind != PHBC_TIP_STATES && !ctx->d_tip_partials)) {
			snprintf(phbc_errbuf, sizeof(phbc_errbuf), "upper / lower partials are not resident");
			return -4;
		}
	}
	const size_t n = (size_t)nitems;
	const size_t tiles = (P + BR_THREADS - 1) / BR_THREADS;
	// scratch: bl [n] | results [n][3] | matrices [n][C][3][S*S] | partial [n][3][tiles] | host exponentials [n][C][S] | nodes [n] (int)
	const size_t need = (n * (4 + C * 3 * S * S + 3 * tiles + C * S) + (n + 1) / 2) * sizeof(double);
	if (need > ctx->branch_bytes) {
		PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
		if (ctx->d_branch) cudaFree(ctx->d_branch);
		ctx->d_branch = NULL;
		ctx->branch_bytes = 0;
		PHBC_CHECK(cudaMalloc((void **)&ctx->d_branch, need));
		ctx->branch_bytes = need;
	}
	double *d_bl = ctx->d_branch, *d_out = d_bl + n, *d_mats = d_out + 3 * n, *d_part = d_mats + n * C * 3 * S * S;
	double *d_exbuf = d_part + n * 3 * tiles;
	double *d_ex = ex_host ? d_exbuf : NULL;
	int *d_nodes = reinterpret_cast<int *>(d_exbuf + n * C * S);
	PHBC_CHECK(cudaMemcpyAsync(d_bl, bl_host, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
	PHBC_CHECK(cudaMemcpyAsync(d_nodes, nodes_host, n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
	if (ex_host) PHBC_CHECK(cudaMemcpyAsync(d_ex, ex_host, n * C * S * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
	const int mthreads = S * S >= 256 ? 256 : (S * S >= 64 ? 64 : 32);
	k_branch_matrices<<<dim3((unsigned)n, (unsigned)C), mthreads, 3 * S * sizeof(double), ctx->stream>>>((int)S, (int)C, ctx->d_evec, ctx->d_eval, ctx->d_ivec,
	                                                                                                d_bl, ctx->d_rates, d_ex, d_mats);
	const size_t smem = 3 * S * S * sizeof(double);
	if (smem > 48 * 1024) PHBC_CHECK(cudaFuncSetAttribute(k_branch_lnl, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
	Bufs b = phbc_make_bufs(ctx);
	k_branch_lnl<<<dim3((unsigned)tiles, (unsigned)n), BR_THREADS, smem, ctx->stream>>>(b, d_nodes, d_mats, ctx->d_freqs, ctx->d_props, ctx->d_weights,
	                                                                                   o->scale, d_part);
	k_branch_sum<<<(unsigned)(3 * n), 256, 0, ctx->stream>>>(d_part, (int)tiles, d_out);
	ctx->launches += 3;
	PHBC_CHECK(cudaGetLastError());
	PHBC_CHECK(cudaMemcpyAsync(out_host, d_out, 3 * n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
	PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
	return 0;
}
