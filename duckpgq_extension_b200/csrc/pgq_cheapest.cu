// pgq_cheapest.cu -- cheapest_path_length on the device CSR: the batched Bellman-Ford of
// cheapest_path_length.cpp:12-136 (TemplatedBatchBellmanFord: one lane per row, all lanes of an edge
// relaxed together, sweeps until nothing changes).  sm_100a only.
//
// The reference relaxes in place, sequentially, in CSR order; the distances it ends with are the least
// fixed point of  d[n] = min(d[n], d[v] + w(v,n))  -- for int64 exactly, for double because fl(a + w)
// is monotone in a -- and do not depend on the relaxation order.  The device relaxes in parallel with
// atomicMin and re-sweeps only the vertices whose distances improved, to the same fixed point,
// bit for bit.  "Unreachable" is the reference's own sentinel max/2 (l.15), added to like any other
// number (no guard, as UpdateOneLane l.29-36 has none).
//
// The fixed point needs every edge checked once from every vertex's final distance.  A vertex is
// re-swept after each improvement, so what remains is the first sweep: the reference relaxes every
// vertex there, even one still at the sentinel.  With weights >= 0 such a vertex lowers nothing
// (max/2 + w >= max/2 >= any distance), so only the sources start dirty.  With a negative weight
// max/2 + w can be below max/2 -- a target no source reaches then has a cost, and with DOUBLE
// weights (max/2 + -1e308) even a reached one can get cheaper -- so, when the CSR holds any weight
// below zero (w_negative, set at finalize), every vertex starts dirty.
#include <algorithm>
#include <cstring>

#include "pgq_tile.cuh"

#define BF_INF_I64 (0x7fffffffffffffffLL / 2)

// doubles are kept as order-preserving unsigned keys so that atomicMin works on them
__device__ __forceinline__ u64 f64_key(double d) {
	const u64 b = (u64)__double_as_longlong(d);
	return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_f64(u64 k) {
	const u64 b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
	return __longlong_as_double((long long)b);
}

template <bool F64>
__global__ void k_bf_init(int64_t count, u64 *dist) {
	const u64 inf = F64 ? f64_key(1.7976931348623157e308 / 2) : (u64)BF_INF_I64;
	for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
		dist[i] = inf;
	}
}

// dists[src][lane] = 0 for the rows of the batch (InitialiseBellmanFord, l.12-27)
template <bool F64>
__global__ void k_bf_sources(int b0, int cnt, int L, const int64_t *__restrict__ src, const uint8_t *__restrict__ src_valid,
                             const int32_t *__restrict__ perm, int64_t n, u64 *dist, uint32_t *dirty, int *err) {
	const int l = blockIdx.x * blockDim.x + threadIdx.x;
	if (l < cnt) {
		const int64_t row = b0 + l;
		if (!src_valid || src_valid[row]) {
			const int64_t s = src[row];
			if (s < 0 || s >= n) {
				*err = 1;
				return;
			}
			const int ps = perm[s];
			dist[(int64_t)ps * L + l] = F64 ? f64_key(0.0) : 0ull;
			atomicOr(&dirty[ps >> 5], 1u << (ps & 31));
		}
	}
}

// One sweep: a warp per dirty vertex relaxes all of its out-edges for all lanes (UpdateLanes, l.38-50).
template <bool F64>
__global__ void __launch_bounds__(256) k_bf_sweep(int64_t n, int L, const int32_t *__restrict__ off,
                                                  const int32_t *__restrict__ adj, const int64_t *__restrict__ w_bits,
                                                  u64 *dist, uint32_t *dirty, int *changed) {
	const int lane = threadIdx.x & 31;
	const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
	bool any = false;
	for (int64_t v = warp; v < n; v += nwarps) {
		const uint32_t bit = 1u << (v & 31);
		if (!(dirty[v >> 5] & bit)) {
			continue;
		}
		if (lane == 0) {
			atomicAnd(&dirty[v >> 5], ~bit); // cleared BEFORE the distances are read: a later improvement marks it again
		}
		__syncwarp();
		__threadfence();
		const int e0 = off[v], e1 = off[v + 1];
		for (int g = 0; g < L; g += 32) {
			const u64 dk = *reinterpret_cast<volatile u64 *>(&dist[v * L + g + lane]);
			for (int e = e0; e < e1; e++) {
				const int u = adj[e];
				u64 *slot = &dist[(int64_t)u * L + g + lane];
				bool better;
				if (F64) {
					// "better" is decided on the doubles, as the reference's nw < dists[n]: false for a NaN sum,
					// whose key (a NaN with the sign bit set, which the fp64 add passes through) sorts below
					// every number's
					const double c = key_f64(dk) + __longlong_as_double(w_bits[e]);
					const u64 nk = f64_key(c);
					better = c < key_f64(*reinterpret_cast<volatile u64 *>(slot)) && nk < atomicMin(slot, nk);
				} else {
					const u64 nk = (u64)((long long)dk + w_bits[e]);
					better = (long long)nk < *reinterpret_cast<volatile long long *>(slot) &&
					         (long long)nk < atomicMin(reinterpret_cast<long long *>(slot), (long long)nk);
				}
				if (__any_sync(FULL_MASK, better)) {
					if (lane == 0) {
						__threadfence();
						atomicOr(&dirty[u >> 5], 1u << (u & 31));
					}
					any = true;
				}
			}
		}
	}
	if (any && lane == 0) {
		*changed = 1;
	}
}

// result rows of the batch (l.73-101): max/2 -> NULL, NULL source / target -> NULL
template <bool F64>
__global__ void k_bf_results(int b0, int cnt, int L, const int64_t *__restrict__ dst, const uint8_t *__restrict__ src_valid,
                             const uint8_t *__restrict__ dst_valid, const int32_t *__restrict__ perm, int64_t n,
                             const u64 *__restrict__ dist, int64_t *out, uint8_t *out_valid, int *err) {
	const int l = blockIdx.x * blockDim.x + threadIdx.x;
	if (l < cnt) {
		const int64_t row = b0 + l;
		out_valid[row] = 0;
		out[row] = 0;
		if ((src_valid && !src_valid[row]) || (dst_valid && !dst_valid[row])) {
			return;
		}
		const int64_t d = dst[row];
		if (d < 0 || d >= n) {
			*err = 1;
			return;
		}
		const u64 k = dist[(int64_t)perm[d] * L + l];
		if (F64) {
			const double c = key_f64(k);
			if (c != 1.7976931348623157e308 / 2) {
				out[row] = __double_as_longlong(c);
				out_valid[row] = 1;
			}
		} else if ((long long)k != BF_INF_I64) {
			out[row] = (long long)k;
			out_valid[row] = 1;
		}
	}
}

template <bool F64>
static int run_bf(pgq_csr *csr, Workspace *ws, int64_t p, const int64_t *d_src, const int64_t *d_dst,
                  const uint8_t *d_sv, const uint8_t *d_dv, int64_t *d_out, uint8_t *d_ov, pgq_stats *st) {
	cudaStream_t s = ws->stream;
	const int64_t n = csr->n;
	// lanes per batch: as many as a 2 GB distance array allows, at most 256 (the reference's largest batch)
	int L = 256;
	while (L > 32 && (int64_t)L * std::max<int64_t>(n, 1) * 8 > ((int64_t)2 << 30)) {
		L >>= 1;
	}
	L = (int)std::min<int64_t>(L, ((p + 31) / 32) * 32);
	u64 *dist;
	uint32_t *dirty;
	int *flags, *h_flags;
	const size_t dist_elems = (size_t)std::max<int64_t>(n, 1) * L;
	const size_t dirty_bytes = ((size_t)n / 32 + 1) * sizeof(uint32_t);
	PGQ_TRY(pgq_ws_reserve(ws, 0, dist_elems * sizeof(u64), (void **)&dist));
	PGQ_TRY(pgq_ws_reserve(ws, 1, dirty_bytes, (void **)&dirty));
	PGQ_TRY(pgq_ws_reserve(ws, 2, 256, (void **)&flags)); // [0] changed, [1] range error
	PGQ_TRY(pgq_ws_pinned(ws, 256, (void **)&h_flags));
	PGQ_CUDA(cudaMemsetAsync(flags, 0, 2 * sizeof(int), s));
	const int sms = csr->ctx->sm_count;
	for (int64_t b0 = 0; b0 < p; b0 += L) {
		const int cnt = (int)std::min<int64_t>(L, p - b0);
		k_bf_init<F64><<<(unsigned)std::min<int64_t>((dist_elems + 255) / 256, (int64_t)sms * 16), 256, 0, s>>>(
		    (int64_t)dist_elems, dist);
		// with a negative weight every vertex is relaxed in the first sweep, sentinel or not (see the header);
		// the bits past n in the last word are never read, the sweep stops at v < n
		PGQ_CUDA(cudaMemsetAsync(dirty, csr->w_negative ? 0xff : 0, dirty_bytes, s));
		k_bf_sources<F64><<<(cnt + 127) / 128, 128, 0, s>>>((int)b0, cnt, L, d_src, d_sv, csr->perm, n, dist, dirty,
		                                                   flags + 1);
		st->batches++;
		st->kernel_launches += 2;
		for (;;) {
			PGQ_CUDA(cudaMemsetAsync(flags, 0, sizeof(int), s));
			k_bf_sweep<F64><<<(unsigned)std::max<int64_t>(1, std::min<int64_t>((n + 7) / 8, (int64_t)sms * 8)), 256, 0, s>>>(
			    n, L, csr->out.off, csr->out.adj, csr->w_bits, dist, dirty, flags);
			PGQ_CUDA(cudaGetLastError());
			PGQ_CUDA(cudaMemcpyAsync(h_flags, flags, 2 * sizeof(int), cudaMemcpyDeviceToHost, s));
			PGQ_CUDA(cudaStreamSynchronize(s));
			st->levels++;
			st->kernel_launches++;
			if (h_flags[1]) {
				return pgq_fail(PGQ_ERR_RANGE, "source rowid outside [0,%lld)", (long long)n);
			}
			if (!h_flags[0]) {
				break;
			}
		}
		k_bf_results<F64><<<(cnt + 127) / 128, 128, 0, s>>>((int)b0, cnt, L, d_dst, d_sv, d_dv, csr->perm, n, dist, d_out,
		                                                   d_ov, flags + 1);
		st->kernel_launches++;
	}
	PGQ_CUDA(cudaMemcpyAsync(h_flags, flags, 2 * sizeof(int), cudaMemcpyDeviceToHost, s));
	PGQ_CUDA(cudaStreamSynchronize(s));
	if (h_flags[1]) {
		return pgq_fail(PGQ_ERR_RANGE, "source or destination rowid outside [0,%lld)", (long long)n);
	}
	st->lanes = L;
	return PGQ_OK;
}

extern "C" int pgq_cheapest_path_length(pgq_csr *csr, int64_t p, const int64_t *src, const int64_t *dst,
                                        const uint8_t *src_valid, const uint8_t *dst_valid, void *out_cost,
                                        uint8_t *out_valid, pgq_stats *stats) {
	if (!csr) {
		return pgq_fail(PGQ_ERR_INVALID_ID, "%s", pgq_status_text(PGQ_ERR_INVALID_ID));
	}
	if (p < 0 || (p > 0 && (!src || !dst || !out_cost || !out_valid))) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "null or negative argument");
	}
	if (!csr->finalized || !csr->w_bits || csr->weight_type == 0) {
		// cheapest_path_length_function_data.cpp:22-24
		return pgq_fail(PGQ_ERR_NOT_INITIALIZED, "Need to initialize CSR before doing cheapest path");
	}
	pgq_stats st;
	memset(&st, 0, sizeof(st));
	if (p == 0) {
		if (stats) {
			*stats = st;
		}
		return PGQ_OK;
	}
	PGQ_CUDA(cudaSetDevice(csr->ctx->device));
	Workspace *ws;
	PGQ_TRY(pgq_ws_acquire(csr->ctx, &ws));
	cudaStream_t s = ws->stream;
	int rc = PGQ_OK;
	do {
		int64_t *d_src, *d_dst, *d_out;
		uint8_t *d_sv = nullptr, *d_dv = nullptr, *d_ov;
		const size_t b8 = (size_t)p * sizeof(int64_t);
		if ((rc = pgq_ws_reserve(ws, 6, b8, (void **)&d_src)) != PGQ_OK) break;
		if ((rc = pgq_ws_reserve(ws, 7, b8, (void **)&d_dst)) != PGQ_OK) break;
		if ((rc = pgq_ws_reserve(ws, 9, b8, (void **)&d_out)) != PGQ_OK) break;
		if ((rc = pgq_ws_reserve(ws, 10, (size_t)p, (void **)&d_ov)) != PGQ_OK) break;
		cudaMemcpyAsync(d_src, src, b8, cudaMemcpyHostToDevice, s);
		cudaMemcpyAsync(d_dst, dst, b8, cudaMemcpyHostToDevice, s);
		st.h2d_bytes = 2 * (int64_t)b8;
		if (src_valid) {
			if ((rc = pgq_ws_reserve(ws, 8, (size_t)p, (void **)&d_sv)) != PGQ_OK) break;
			cudaMemcpyAsync(d_sv, src_valid, (size_t)p, cudaMemcpyHostToDevice, s);
			st.h2d_bytes += p;
		}
		if (dst_valid) {
			if ((rc = pgq_ws_reserve(ws, 11, (size_t)p, (void **)&d_dv)) != PGQ_OK) break;
			cudaMemcpyAsync(d_dv, dst_valid, (size_t)p, cudaMemcpyHostToDevice, s);
			st.h2d_bytes += p;
		}
		rc = (csr->weight_type == 2) ? run_bf<true>(csr, ws, p, d_src, d_dst, d_sv, d_dv, d_out, d_ov, &st)
		                             : run_bf<false>(csr, ws, p, d_src, d_dst, d_sv, d_dv, d_out, d_ov, &st);
		if (rc != PGQ_OK) break;
		cudaMemcpyAsync(out_cost, d_out, b8, cudaMemcpyDeviceToHost, s);
		cudaMemcpyAsync(out_valid, d_ov, (size_t)p, cudaMemcpyDeviceToHost, s);
		st.d2h_bytes = (int64_t)b8 + p;
	} while (0);
	cudaError_t e = cudaStreamSynchronize(s); // (also on the error paths: nothing may outlive the call)
	if (rc == PGQ_OK && (e != cudaSuccess || (e = cudaGetLastError()) != cudaSuccess)) {
		rc = pgq_fail(PGQ_ERR_CUDA, "cheapest_path_length failed: %s", cudaGetErrorString(e));
	}
	cudaGetLastError();
	pgq_ws_release(csr->ctx, ws);
	if (rc == PGQ_OK && stats) {
		*stats = st;
	}
	return rc;
}
