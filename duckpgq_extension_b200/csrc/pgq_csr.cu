// pgq_csr.cu -- device-resident CSR: context/workspace plumbing, the device-side CSR build that
// replaces create_csr_vertex / create_csr_edge (reference: src/core/functions/scalar/csr_creation.cpp),
// the transposed (in-edge) CSC used by the bottom-up step, and the row-head metadata of the
// edge-tiled kernels.  sm_100a only.
#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "pgq_tile.cuh"

// ------------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

void pgq_set_error(const char *fmt, ...) {
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(g_err, sizeof(g_err), fmt, ap);
	va_end(ap);
}

int pgq_fail(int status, const char *fmt, ...) {
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(g_err, sizeof(g_err), fmt, ap);
	va_end(ap);
	return status;
}

extern "C" const char *pgq_last_error(void) {
	return g_err;
}

extern "C" int pgq_abi_version(void) {
	return PGQ_B200_ABI_VERSION;
}

extern "C" const char *pgq_status_text(int status) {
	switch (status) {
	case PGQ_OK:
		return "ok";
	case PGQ_ERR_CONSTRAINT: // csr_creation.cpp:122-124
		return "Non-existent/non-unique vertices detected. Make sure all vertices referred by edge tables exist "
		       "and are unique for path-finding queries.";
	case PGQ_ERR_INVALID_ID: // iterativelength.cpp:42
		return "Invalid ID";
	case PGQ_ERR_NOT_INITIALIZED: // iterativelength.cpp:46,50
		return "Need to initialize CSR before doing shortest path";
	case PGQ_ERR_INVALID_ARG:
		return "invalid argument";
	case PGQ_ERR_CUDA:
		return "CUDA error";
	case PGQ_ERR_OOM:
		return "out of memory";
	case PGQ_ERR_RANGE:
		return "vertex id or graph size out of range";
	case PGQ_ERR_UNSUPPORTED:
		return "unsupported";
	default:
		return "unknown status";
	}
}

// ------------------------------------------------------------------------------------------------
// context + workspace pool
// ------------------------------------------------------------------------------------------------
extern "C" int pgq_device_count(int *count) {
	if (!count) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "count is null");
	}
	// Load all kernels when the context is created instead of on first use: with CUDA's default lazy
	// loading the first query that needs a new lane width pays ~0.3 s in the middle of a statement.
	// (No effect if the process initialised CUDA before us, or if the user set the variable.)
	setenv("CUDA_MODULE_LOADING", "EAGER", 0);
	int c = 0;
	cudaError_t e = cudaGetDeviceCount(&c);
	if (e != cudaSuccess) {
		cudaGetLastError();
		*count = 0;
		return pgq_fail(PGQ_ERR_CUDA, "cudaGetDeviceCount failed: %s", cudaGetErrorString(e));
	}
	*count = c;
	return PGQ_OK;
}

extern "C" int pgq_ctx_create(int device, pgq_ctx **out) {
	if (!out) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "out is null");
	}
	*out = nullptr;
	int count = 0;
	PGQ_TRY(pgq_device_count(&count));
	if (device < 0 || device >= count) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "device %d not present (%d CUDA devices visible)", device, count);
	}
	PGQ_CUDA(cudaSetDevice(device));
	cudaDeviceProp prop;
	PGQ_CUDA(cudaGetDeviceProperties(&prop, device));
	if (prop.major < 10) {
		return pgq_fail(PGQ_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a only", device,
		                prop.major, prop.minor);
	}
	pgq_ctx *ctx = new (std::nothrow) pgq_ctx();
	if (!ctx) {
		return pgq_fail(PGQ_ERR_OOM, "host allocation failed");
	}
	ctx->device = device;
	ctx->sm_count = prop.multiProcessorCount;
	if (const char *env = getenv("PGQ_B200_MAX_WORKSPACES")) {
		ctx->max_ws = std::max(1, atoi(env));
	}
	if (const char *env = getenv("PGQ_B200_CSR_CACHE_MB")) {
		ctx->buf_cache_limit = (size_t)std::max(0, atoi(env)) << 20;
	}
	*out = ctx;
	return PGQ_OK;
}

static void ws_destroy(Workspace *ws) {
	for (int i = 0; i < PGQ_WS_SLOTS; i++) {
		if (ws->buf[i]) {
			cudaFree(ws->buf[i]);
		}
	}
	for (auto ev : ws->ev_pool) {
		cudaEventDestroy(ev);
	}
	if (ws->ev_begin) {
		cudaEventDestroy(ws->ev_begin);
	}
	if (ws->ev_end) {
		cudaEventDestroy(ws->ev_end);
	}
	if (ws->stream) {
		cudaStreamDestroy(ws->stream);
	}
	if (ws->pinned) {
		cudaFreeHost(ws->pinned);
	}
	delete ws;
}

extern "C" void pgq_ctx_destroy(pgq_ctx *ctx) {
	if (!ctx) {
		return;
	}
	cudaSetDevice(ctx->device);
	for (auto ws : ctx->free_ws) {
		ws_destroy(ws);
	}
	for (auto &kv : ctx->buf_cache) {
		cudaFree(kv.second);
	}
	delete ctx;
}

// The pool is bounded (pgq_ctx::max_ws, PGQ_B200_MAX_WORKSPACES): a host such as DuckDB calls the path
// functions from all of its worker threads at once, and every workspace holds three lane-mask arrays
// of the graph's size.  A caller that finds the budget used up waits for a workspace to come back.
static int ws_take(pgq_ctx *ctx, Workspace **out, bool block) {
	{
		std::unique_lock<std::mutex> g(ctx->mu);
		for (;;) {
			if (!ctx->free_ws.empty()) {
				*out = ctx->free_ws.back();
				ctx->free_ws.pop_back();
				return PGQ_OK;
			}
			if (ctx->live_ws < ctx->max_ws) {
				ctx->live_ws++;
				break;
			}
			if (!block) {
				return pgq_fail(PGQ_ERR_OOM, "all %d workspaces of the context are in use", ctx->max_ws);
			}
			ctx->cv.wait(g);
		}
	}
	Workspace *ws = new (std::nothrow) Workspace();
	cudaError_t e = ws ? cudaStreamCreateWithFlags(&ws->stream, cudaStreamNonBlocking) : cudaErrorMemoryAllocation;
	if (e == cudaSuccess) {
		e = cudaEventCreate(&ws->ev_begin);
	}
	if (e == cudaSuccess) {
		e = cudaEventCreate(&ws->ev_end);
	}
	if (e != cudaSuccess) {
		cudaGetLastError();
		if (ws) {
			ws_destroy(ws);
		}
		{
			std::lock_guard<std::mutex> g(ctx->mu);
			ctx->live_ws--;
		}
		ctx->cv.notify_one();
		return pgq_fail(ws ? PGQ_ERR_CUDA : PGQ_ERR_OOM, "workspace creation failed: %s", cudaGetErrorString(e));
	}
	*out = ws;
	return PGQ_OK;
}

int pgq_ws_acquire(pgq_ctx *ctx, Workspace **out) {
	return ws_take(ctx, out, true);
}

int pgq_ws_try_acquire(pgq_ctx *ctx, Workspace **out) {
	return ws_take(ctx, out, false);
}

void pgq_ws_release(pgq_ctx *ctx, Workspace *ws) {
	{
		std::lock_guard<std::mutex> g(ctx->mu);
		ctx->free_ws.push_back(ws);
	}
	ctx->cv.notify_one();
}

// pgq_ws_reserve that keeps the first keep_bytes of the slot's content when it has to grow
// (synchronises the stream in that case).
int pgq_ws_grow(Workspace *ws, int slot, size_t bytes, size_t keep_bytes, cudaStream_t s, void **out) {
	if (bytes == 0) {
		bytes = 256;
	}
	if (ws->cap[slot] < bytes) {
		const size_t want = std::max(bytes * 2, (size_t)4096);
		void *bigger = nullptr;
		cudaError_t e = cudaMalloc(&bigger, want);
		if (e != cudaSuccess) {
			cudaGetLastError();
			return pgq_fail(PGQ_ERR_OOM, "device allocation of %zu bytes failed: %s", want, cudaGetErrorString(e));
		}
		if (ws->buf[slot]) {
			if (keep_bytes > 0) {
				e = cudaMemcpyAsync(bigger, ws->buf[slot], std::min(keep_bytes, ws->cap[slot]), cudaMemcpyDeviceToDevice, s);
			}
			if (e == cudaSuccess) {
				e = cudaStreamSynchronize(s);
			}
			if (e != cudaSuccess) {
				cudaGetLastError();
				cudaFree(bigger);
				return pgq_fail(PGQ_ERR_CUDA, "growing a workspace buffer failed: %s", cudaGetErrorString(e));
			}
			cudaFree(ws->buf[slot]);
		}
		ws->buf[slot] = bigger;
		ws->cap[slot] = want;
	}
	*out = ws->buf[slot];
	return PGQ_OK;
}

int pgq_ws_reserve(Workspace *ws, int slot, size_t bytes, void **out) {
	if (bytes == 0) {
		bytes = 256;
	}
	if (ws->cap[slot] < bytes) {
		if (ws->buf[slot]) {
			PGQ_CUDA(cudaFree(ws->buf[slot]));
			ws->buf[slot] = nullptr;
			ws->cap[slot] = 0;
		}
		size_t want = bytes + bytes / 8; // a little slack so that slightly larger calls reuse it
		cudaError_t e = cudaMalloc(&ws->buf[slot], want);
		if (e != cudaSuccess) {
			cudaGetLastError();
			want = bytes;
			e = cudaMalloc(&ws->buf[slot], want);
		}
		if (e != cudaSuccess) {
			cudaGetLastError();
			return pgq_fail(PGQ_ERR_OOM, "device allocation of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
		}
		ws->cap[slot] = want;
	}
	*out = ws->buf[slot];
	return PGQ_OK;
}

int pgq_ws_pinned(Workspace *ws, size_t bytes, void **out) {
	if (ws->pinned_cap < bytes) {
		if (ws->pinned) {
			cudaFreeHost(ws->pinned);
			ws->pinned = nullptr;
			ws->pinned_cap = 0;
		}
		PGQ_CUDA(cudaHostAlloc(&ws->pinned, bytes, cudaHostAllocMapped)); // the GPU writes level statistics into it
		ws->pinned_cap = bytes;
	}
	*out = ws->pinned;
	return PGQ_OK;
}

// ------------------------------------------------------------------------------------------------
// exclusive prefix sum (int32), three-phase, 2048 items per block
// ------------------------------------------------------------------------------------------------
#define SCAN_THREADS 256
#define SCAN_ITEMS 8
#define SCAN_TILE (SCAN_THREADS * SCAN_ITEMS)

__device__ __forceinline__ int block_exclusive_scan(int x, int *total, int *smem /* >= 8 ints */) {
	int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	int incl = x;
#pragma unroll
	for (int d = 1; d < 32; d <<= 1) {
		int t = __shfl_up_sync(FULL_MASK, incl, d);
		if (lane >= d) {
			incl += t;
		}
	}
	if (lane == 31) {
		smem[warp] = incl;
	}
	__syncthreads();
	if (warp == 0) {
		int w = (lane < SCAN_THREADS / 32) ? smem[lane] : 0;
		int wi = w;
#pragma unroll
		for (int d = 1; d < 8; d <<= 1) {
			int t = __shfl_up_sync(FULL_MASK, wi, d);
			if (lane >= d) {
				wi += t;
			}
		}
		if (lane < SCAN_THREADS / 32) {
			smem[lane] = wi - w; // exclusive warp offsets
		}
		if (lane == SCAN_THREADS / 32 - 1) {
			smem[8] = wi;
		}
	}
	__syncthreads();
	*total = smem[8];
	return smem[warp] + incl - x;
}

__global__ void __launch_bounds__(SCAN_THREADS) k_scan_sums(const int32_t *__restrict__ in, int64_t count,
                                                            int32_t *__restrict__ sums) {
	__shared__ int smem[9];
	int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
	int s = 0;
#pragma unroll
	for (int j = 0; j < SCAN_ITEMS; j++) {
		if (base + j < count) {
			s += in[base + j];
		}
	}
	int total;
	block_exclusive_scan(s, &total, smem);
	if (threadIdx.x == 0) {
		sums[blockIdx.x] = total;
	}
}

__global__ void __launch_bounds__(SCAN_THREADS) k_scan_apply(const int32_t *in, int32_t *out, int64_t count,
                                                             const int32_t *__restrict__ block_offsets) {
	__shared__ int smem[9];
	int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
	int v[SCAN_ITEMS];
	int s = 0;
#pragma unroll
	for (int j = 0; j < SCAN_ITEMS; j++) {
		v[j] = (base + j < count) ? in[base + j] : 0;
		s += v[j];
	}
	int total;
	int excl = block_exclusive_scan(s, &total, smem) + (block_offsets ? block_offsets[blockIdx.x] : 0);
#pragma unroll
	for (int j = 0; j < SCAN_ITEMS; j++) {
		if (base + j < count) {
			out[base + j] = excl;
		}
		excl += v[j];
	}
}

size_t pgq_scan_tmp_elems(int64_t count) {
	size_t total = 0;
	int64_t c = count;
	while (c > SCAN_TILE) {
		c = (c + SCAN_TILE - 1) / SCAN_TILE;
		total += (size_t)c;
	}
	return total + 1;
}

// out may alias in.  block_tmp needs pgq_scan_tmp_elems(count) ints.
int pgq_scan_exclusive_i32(const int32_t *in, int32_t *out, int64_t count, int32_t *block_tmp, cudaStream_t s) {
	if (count <= 0) {
		return PGQ_OK;
	}
	int64_t nblocks = (count + SCAN_TILE - 1) / SCAN_TILE;
	if (nblocks == 1) {
		k_scan_apply<<<1, SCAN_THREADS, 0, s>>>(in, out, count, nullptr);
		PGQ_CUDA(cudaGetLastError());
		return PGQ_OK;
	}
	k_scan_sums<<<(unsigned)nblocks, SCAN_THREADS, 0, s>>>(in, count, block_tmp);
	PGQ_CUDA(cudaGetLastError());
	PGQ_TRY(pgq_scan_exclusive_i32(block_tmp, block_tmp, nblocks, block_tmp + nblocks, s));
	k_scan_apply<<<(unsigned)nblocks, SCAN_THREADS, 0, s>>>(in, out, count, block_tmp);
	PGQ_CUDA(cudaGetLastError());
	return PGQ_OK;
}

// ------------------------------------------------------------------------------------------------
// stable LSD radix sort of (int32 key, int32 value) pairs, 5 bits per pass
//   pass = per-tile digit histogram -> exclusive scan (digit-major, tile-minor) -> stable scatter.
// Stability is what makes the device CSR equal the reference's: edges of one source keep their
// arrival order (csr_creation.cpp:132-139 with one feeding thread).
// ------------------------------------------------------------------------------------------------
#define RS_BITS 5
#define RS_BINS (1 << RS_BITS)
#define RS_THREADS 256
#define RS_ITEMS 8
#define RS_TILE (RS_THREADS * RS_ITEMS)

__global__ void __launch_bounds__(RS_THREADS) k_rs_hist(const int32_t *__restrict__ keys, int64_t count, int shift,
                                                        int32_t *__restrict__ hist, int nblocks) {
	__shared__ int bins[RS_BINS];
	if (threadIdx.x < RS_BINS) {
		bins[threadIdx.x] = 0;
	}
	__syncthreads();
	const int64_t base = (int64_t)blockIdx.x * RS_TILE;
#pragma unroll
	for (int j = 0; j < RS_ITEMS; j++) {
		const int64_t i = base + j * RS_THREADS + threadIdx.x; // any order will do for counting
		if (i < count) {
			atomicAdd(&bins[(keys[i] >> shift) & (RS_BINS - 1)], 1);
		}
	}
	__syncthreads();
	if (threadIdx.x < RS_BINS) {
		hist[(int64_t)threadIdx.x * nblocks + blockIdx.x] = bins[threadIdx.x];
	}
}

__global__ void __launch_bounds__(RS_THREADS) k_rs_scatter(const int32_t *__restrict__ keys_in,
                                                           const int32_t *__restrict__ vals_in,
                                                           int32_t *__restrict__ keys_out, int32_t *__restrict__ vals_out,
                                                           int64_t count, int shift, const int32_t *__restrict__ offs,
                                                           int nblocks) {
	__shared__ int cnt[RS_BINS][RS_THREADS]; // per-thread digit counts, then prefixes over the threads
	const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
	const int64_t base = (int64_t)blockIdx.x * RS_TILE + (int64_t)t * RS_ITEMS; // a thread owns 8 consecutive pairs
	int k[RS_ITEMS], v[RS_ITEMS], local[RS_ITEMS];
#pragma unroll
	for (int d = 0; d < RS_BINS; d++) {
		cnt[d][t] = 0;
	}
#pragma unroll
	for (int j = 0; j < RS_ITEMS; j++) {
		if (base + j < count) {
			k[j] = keys_in[base + j];
			v[j] = vals_in[base + j];
			const int d = (k[j] >> shift) & (RS_BINS - 1);
			local[j] = cnt[d][t]; // rank among this thread's earlier pairs with the same digit
			cnt[d][t] = local[j] + 1;
		}
	}
	__syncthreads();
	// exclusive prefix over the 256 threads, one digit row at a time (4 rows per warp)
	for (int d = warp * (RS_BINS / 8); d < (warp + 1) * (RS_BINS / 8); d++) {
		int carry = 0;
		for (int c = 0; c < RS_THREADS / 32; c++) {
			const int x = cnt[d][c * 32 + lane];
			int incl = x;
#pragma unroll
			for (int s = 1; s < 32; s <<= 1) {
				int y = __shfl_up_sync(FULL_MASK, incl, s);
				if (lane >= s) {
					incl += y;
				}
			}
			cnt[d][c * 32 + lane] = carry + incl - x;
			carry += __shfl_sync(FULL_MASK, incl, 31);
		}
	}
	__syncthreads();
#pragma unroll
	for (int j = 0; j < RS_ITEMS; j++) {
		if (base + j < count) {
			const int d = (k[j] >> shift) & (RS_BINS - 1);
			const int64_t pos = (int64_t)offs[(int64_t)d * nblocks + blockIdx.x] + cnt[d][t] + local[j];
			keys_out[pos] = k[j];
			vals_out[pos] = v[j];
		}
	}
}

// Sorts by the low `end_bit` bits of the keys.  (keys_a, vals_a) hold the input and are clobbered;
// the result is in (*keys_res, *vals_res), which is either the a or the b pair.
static int radix_sort_pairs(Workspace *ws, int32_t *keys_a, int32_t *keys_b, int32_t *vals_a, int32_t *vals_b,
                            int64_t count, int end_bit, cudaStream_t s, int32_t **keys_res, int32_t **vals_res) {
	const int nblocks = (int)((count + RS_TILE - 1) / RS_TILE);
	const int64_t hist_elems = (int64_t)RS_BINS * nblocks;
	int32_t *hist, *scan_tmp;
	PGQ_TRY(pgq_ws_reserve(ws, 14, (size_t)(hist_elems + 1) * sizeof(int32_t), (void **)&hist));
	PGQ_TRY(pgq_ws_reserve(ws, 15, pgq_scan_tmp_elems(hist_elems) * sizeof(int32_t), (void **)&scan_tmp));
	int32_t *kin = keys_a, *kout = keys_b, *vin = vals_a, *vout = vals_b;
	for (int shift = 0; shift < end_bit; shift += RS_BITS) {
		k_rs_hist<<<nblocks, RS_THREADS, 0, s>>>(kin, count, shift, hist, nblocks);
		PGQ_CUDA(cudaGetLastError());
		PGQ_TRY(pgq_scan_exclusive_i32(hist, hist, hist_elems, scan_tmp, s));
		k_rs_scatter<<<nblocks, RS_THREADS, 0, s>>>(kin, vin, kout, vout, count, shift, hist, nblocks);
		PGQ_CUDA(cudaGetLastError());
		std::swap(kin, kout);
		std::swap(vin, vout);
	}
	*keys_res = kin;
	*vals_res = vin;
	return PGQ_OK;
}

// ------------------------------------------------------------------------------------------------
// small element-wise kernels
// ------------------------------------------------------------------------------------------------
static inline unsigned grid_for(int64_t count, int threads, int64_t cap = 1 << 20) {
	int64_t g = (count + threads - 1) / threads;
	return (unsigned)std::max<int64_t>(1, std::min<int64_t>(g, cap));
}

// int64 -> int32 with range check lo <= x < hi (err = 1 on violation)
__global__ void k_narrow(const int64_t *__restrict__ in, int32_t *__restrict__ out, int64_t count, int64_t lo,
                         int64_t hi, int *err) {
	for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
		int64_t x = in[i];
		if (x < lo || x >= hi) {
			*err = 1;
			x = lo;
		}
		out[i] = (int32_t)x;
	}
}

__global__ void k_widen(const int32_t *__restrict__ in, int64_t *__restrict__ out, int64_t count) {
	for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
		out[i] = in[i];
	}
}

__global__ void k_iota(int32_t *out, int64_t count) {
	for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
		out[i] = (int32_t)i;
	}
}

// cnt[dense_id[i]] = (int32) c[i]     (create_csr_vertex, csr_creation.cpp:103-109)
__global__ void k_set_counts(const int64_t *__restrict__ dense_id, const int64_t *__restrict__ c, int64_t count,
                             int64_t n, int32_t *cnt, int *err) {
	for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
		int64_t id = dense_id[i];
		int64_t x = c[i];
		if (id < 0 || id >= n || x < 0 || x > 0x7fffffffLL) {
			*err = 1;
		} else {
			cnt[id] = (int32_t)x;
		}
	}
}

__global__ void k_histogram(const int32_t *__restrict__ keys, int64_t count, int32_t *hist) {
	for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
		atomicAdd(&hist[keys[i]], 1);
	}
}

__global__ void k_compare_i32(const int32_t *__restrict__ a, const int32_t *__restrict__ b, int64_t count, int *err) {
	for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
		if (a[i] != b[i]) {
			*err = 1;
		}
	}
}

// out_adj[i] = dst[perm[i]], edge_ids[i] = eid[perm[i]]  (the stable scatter of create_csr_edge)
__global__ void k_gather_edges(const int32_t *__restrict__ perm, const int32_t *__restrict__ dst,
                               const int64_t *__restrict__ eid, const int64_t *__restrict__ w, int64_t count,
                               int32_t *__restrict__ adj, int64_t *__restrict__ edge_ids, int64_t *__restrict__ w_out) {
	for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
		int32_t p = perm[i];
		adj[i] = dst[p];
		edge_ids[i] = eid[p];
		if (w) {
			w_out[i] = w[p]; // w[pos-1] = weight, csr_creation.cpp:166,192
		}
	}
}

// *flag = 1 if some weight is below zero (cheapest_path_length then relaxes every vertex, pgq_cheapest.cu)
__global__ void k_any_negative(const int64_t *__restrict__ w_bits, int64_t count, bool f64, int *flag) {
	for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
		const int64_t b = w_bits[i];
		if (f64 ? __longlong_as_double(b) < 0.0 : b < 0) {
			*flag = 1;
		}
	}
}

// offsets must be non-decreasing, start at 0 and end at m
__global__ void k_check_offsets(const int32_t *__restrict__ off, int64_t n, int64_t m, int *err) {
	for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= n; i += (int64_t)gridDim.x * blockDim.x) {
		int32_t a = off[i];
		if (i == 0 && a != 0) {
			*err = 1;
		}
		if (i == n && a != m) {
			*err = 1;
		}
		if (i < n && off[i + 1] < a) {
			*err = 1;
		}
	}
}

// ---- internal vertex numbering ----------------------------------------------------------------------
// class 0: out > 0 and in > 0, 1: in only, 2: out only, 3: isolated.  Inside a class the vertices are
// ordered by DESCENDING degree (out-degree for the classes whose masks are gathered by the bottom-up
// level: the number of gathers that hit a vertex's mask per level IS its out-degree), ties in original
// order: the hot part of the gathered mask array becomes one contiguous, fully used range of sectors
// (R-MAT-22: the first 8 MB of the 256-lane mask array serve 85 % of all gathers), which is what lets it
// stay in L2 / L1 next to the streaming edge array.
#define PGQ_DEG_CLAMP 0x3FFFFF
__global__ void k_vertex_keys(const int32_t *__restrict__ outdeg, const int32_t *__restrict__ indeg, int64_t n,
                              int32_t *__restrict__ key, int32_t *__restrict__ val, int *class_count) {
	__shared__ int cnt[4];
	if (threadIdx.x < 4) {
		cnt[threadIdx.x] = 0;
	}
	__syncthreads();
	for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < n; v += (int64_t)gridDim.x * blockDim.x) {
		const int od = outdeg[v], id = indeg[v];
		const int c = (od > 0) ? (id > 0 ? 0 : 2) : (id > 0 ? 1 : 3);
		const int d = min(od > 0 ? od : id, PGQ_DEG_CLAMP);
		key[v] = (c << 22) | (PGQ_DEG_CLAMP - d);
		val[v] = (int32_t)v;
		atomicAdd(&cnt[c], 1);
	}
	__syncthreads();
	if (threadIdx.x < 4 && cnt[threadIdx.x]) {
		atomicAdd(&class_count[threadIdx.x], cnt[threadIdx.x]);
	}
}

// inv = the sorted vertex list; perm = its inverse
__global__ void k_invert_perm(const int32_t *__restrict__ sorted, int64_t n, int32_t *__restrict__ perm,
                              int32_t *__restrict__ inv) {
	for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
		const int32_t v = sorted[i];
		inv[i] = v;
		perm[v] = (int32_t)i;
	}
}

__global__ void k_apply_perm(int32_t *ids, int64_t count, const int32_t *__restrict__ perm) {
	for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
		ids[i] = perm[ids[i]];
	}
}

// src[e] = v for e in [off[v], off[v+1])  (a finished CSR back to edge rows, in CSR position order)
__global__ void k_rows_from_offsets(const int32_t *__restrict__ off, int64_t n, int32_t *__restrict__ src) {
	const int lane = threadIdx.x & 31;
	const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
	for (int64_t v = warp; v < n; v += nwarps) {
		for (int e = off[v] + lane; e < off[v + 1]; e += 32) {
			src[e] = (int32_t)v;
		}
	}
}

__global__ void k_iota64(int64_t *out, int64_t count) {
	for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
		out[i] = i;
	}
}

// degree of every ORIGINAL vertex, for the download in the reference's layout
__global__ void k_orig_degrees(const int32_t *__restrict__ off, const int32_t *__restrict__ perm, int64_t n,
                               int32_t *deg) {
	for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v <= n; v += (int64_t)gridDim.x * blockDim.x) {
		deg[v] = (v < n) ? off[perm[v] + 1] - off[perm[v]] : 0;
	}
}

// copies every original vertex's adjacency (internal ids -> original ids) and edge ids to its place
__global__ void k_orig_rows(const int32_t *__restrict__ off, const int32_t *__restrict__ adj,
                            const int64_t *__restrict__ edge_ids, const int32_t *__restrict__ perm,
                            const int32_t *__restrict__ inv, const int32_t *__restrict__ orig_off, int64_t n,
                            int64_t *e_out, int64_t *eid_out) {
	const int lane = threadIdx.x & 31;
	const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
	for (int64_t v = warp; v < n; v += nwarps) {
		const int p = perm[v];
		const int b = off[p], len = off[p + 1] - b, o = orig_off[v];
		for (int k = lane; k < len; k += 32) {
			if (e_out) {
				e_out[o + k] = inv[adj[b + k]];
			}
			if (eid_out) {
				eid_out[o + k] = edge_ids[b + k];
			}
		}
	}
}

// ---- row-head metadata ---------------------------------------------------------------------------
__global__ void k_mark_heads(const int32_t *__restrict__ off, int64_t n, uint32_t *head, int32_t *nzflag) {
	for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
		int32_t s = off[r], e = off[r + 1];
		int flag = e > s;
		nzflag[r] = flag;
		if (flag) {
			atomicOr(&head[s >> 5], 1u << (s & 31));
		}
	}
}

// nzidx = exclusive scan of nzflag.  Writes nzrow[rank] = r and the rank of every chunk start the
// row covers.
__global__ void k_fill_rows(const int32_t *__restrict__ off, const int32_t *__restrict__ nzidx, int64_t n,
                            int32_t *__restrict__ nzrow, int32_t *__restrict__ chunk_rank) {
	for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
		int32_t s = off[r], e = off[r + 1];
		if (e > s) {
			int32_t k = nzidx[r];
			nzrow[k] = (int32_t)r;
			for (int64_t c = ((int64_t)s + PGQ_CHUNK - 1) / PGQ_CHUNK; c * PGQ_CHUNK < e; c++) {
				chunk_rank[c] = k;
			}
		}
	}
}

// rowid[e] = source vertex of out-edge e (the out-CSR is sorted by source, so rowid is ascending)
__global__ void __launch_bounds__(256) k_edge_rows(DirGraph g, int64_t m, int32_t *__restrict__ rowid) {
	int lane = threadIdx.x & 31;
	int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
	for (int64_t c = warp; c < g.nchunks; c += nwarps) {
		ChunkWalker w(g, c, lane);
#pragma unroll
		for (int k = 0; k < PGQ_STEPS; k++) {
			uint32_t h = w.head_word(k);
			int rank = w.advance(h, lane);
			int64_t e = w.base + 32 * k + lane;
			if (e < m) {
				rowid[e] = g.nzrow[rank];
			}
		}
	}
}

// ---- the bottom-up layout (PullGraph) ------------------------------------------------------------------
// per row with in-edges: its contribution to the long part (deg or 0), long flag, short flag
__global__ void k_pull_classify(const int32_t *__restrict__ in_off, int64_t n_rows, int32_t *long_deg, int32_t *long_flag,
                                int32_t *short_flag) {
	for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r <= n_rows; r += (int64_t)gridDim.x * blockDim.x) {
		int d = 0;
		if (r < n_rows) {
			d = in_off[r + 1] - in_off[r];
		}
		const bool is_long = d >= PGQ_SHORT_DEG;
		long_deg[r] = is_long ? d : 0;
		long_flag[r] = is_long ? 1 : 0;
		short_flag[r] = (d > 0 && !is_long) ? 1 : 0;
	}
}

// long rows: copy the in-lists back to back (warp per row), rank -> row, compact offsets by rank
__global__ void __launch_bounds__(256) k_pull_long_fill(const int32_t *__restrict__ in_off, const int32_t *__restrict__ in_adj,
                                                        int64_t n_rows, const int32_t *__restrict__ long_pos,
                                                        const int32_t *__restrict__ long_rank, int32_t *adj, int32_t *row,
                                                        int32_t *off_by_rank) {
	const int lane = threadIdx.x & 31;
	const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
	for (int64_t r = warp; r < n_rows; r += nwarps) {
		const int b = in_off[r], d = in_off[r + 1] - b;
		if (d < PGQ_SHORT_DEG) {
			continue;
		}
		const int p = long_pos[r], k = long_rank[r];
		for (int j = lane; j < d; j += 32) {
			adj[p + j] = in_adj[b + j];
		}
		if (lane == 0) {
			row[k] = (int32_t)r;
			off_by_rank[k] = p;
		}
	}
}

// head bit + rank of every chunk start, from the offsets by rank (all rows non-empty)
__global__ void k_pull_long_meta(const int32_t *__restrict__ off_by_rank, int64_t n_long, uint32_t *head, int32_t *chunk_rank) {
	for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n_long; k += (int64_t)gridDim.x * blockDim.x) {
		const int32_t s = off_by_rank[k], e = off_by_rank[k + 1];
		atomicOr(&head[s >> 5], 1u << (s & 31));
		for (int64_t c = ((int64_t)s + PGQ_CHUNK - 1) / PGQ_CHUNK; c * PGQ_CHUNK < e; c++) {
			chunk_rank[c] = (int32_t)k;
		}
	}
}

// short rows: list them (ascending id) with the sort key 31 - degree
__global__ void k_pull_short_list(const int32_t *__restrict__ in_off, int64_t n_rows, const int32_t *__restrict__ short_pos,
                                  int32_t *key, int32_t *val) {
	for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_rows; r += (int64_t)gridDim.x * blockDim.x) {
		const int d = in_off[r + 1] - in_off[r];
		if (d > 0 && d < PGQ_SHORT_DEG) {
			key[short_pos[r]] = PGQ_SHORT_DEG - 1 - d;
			val[short_pos[r]] = (int32_t)r;
		}
	}
}

// width of every slice = degree of its first row (descending order) -> elements per slice
__global__ void k_pull_slice_width(const int32_t *__restrict__ sorted_key, int64_t n_short, int64_t n_slices, int32_t *elems) {
	for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s <= n_slices; s += (int64_t)gridDim.x * blockDim.x) {
		elems[s] = (s < n_slices) ? 32 * (PGQ_SHORT_DEG - 1 - sorted_key[s * 32]) : 0;
	}
}

__global__ void k_pull_short_fill(const int32_t *__restrict__ in_off, const int32_t *__restrict__ in_adj,
                                  const int32_t *__restrict__ sorted_row, int64_t n_short, int64_t n_slices,
                                  const int32_t *__restrict__ s_off, int32_t *s_adj, int32_t *s_row) {
	for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_slices * 32; i += (int64_t)gridDim.x * blockDim.x) {
		const int64_t s = i >> 5;
		const int lane = (int)(i & 31);
		const int begin = s_off[s], width = (s_off[s + 1] - begin) >> 5;
		int r = -1, b = 0, d = 0;
		if (i < n_short) {
			r = sorted_row[i];
			b = in_off[r];
			d = in_off[r + 1] - b;
		}
		s_row[i] = r;
		for (int j = 0; j < width; j++) {
			s_adj[begin + j * 32 + lane] = (j < d) ? in_adj[b + j] : -1;
		}
	}
}

// ------------------------------------------------------------------------------------------------
// host-side assembly
// ------------------------------------------------------------------------------------------------
static int dev_alloc(pgq_csr *csr, void **p, size_t bytes) {
	if (bytes == 0) {
		bytes = 256;
	}
	pgq_ctx *ctx = csr->ctx;
	*p = nullptr;
	{
		std::lock_guard<std::mutex> g(ctx->mu);
		auto it = ctx->buf_cache.find(bytes);
		if (it != ctx->buf_cache.end()) {
			*p = it->second;
			ctx->buf_cache.erase(it);
			ctx->buf_cache_bytes -= bytes;
		}
	}
	if (!*p) {
		cudaError_t e = cudaMalloc(p, bytes);
		if (e != cudaSuccess) { // give the cached buffers back to the driver and try once more
			cudaGetLastError();
			std::vector<void *> drop;
			{
				std::lock_guard<std::mutex> g(ctx->mu);
				for (auto &kv : ctx->buf_cache) {
					drop.push_back(kv.second);
				}
				ctx->buf_cache.clear();
				ctx->buf_cache_bytes = 0;
			}
			for (void *q : drop) {
				cudaFree(q);
			}
			e = cudaMalloc(p, bytes);
		}
		if (e != cudaSuccess) {
			cudaGetLastError();
			*p = nullptr;
			return pgq_fail(PGQ_ERR_OOM, "device allocation of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
		}
	}
	csr->allocs[*p] = bytes;
	csr->device_bytes += (int64_t)bytes;
	return PGQ_OK;
}

// Returns a buffer of the CSR to the context's cache (or to the driver when the cache is full).
template <typename T>
static void dev_free(pgq_csr *csr, T *&p) {
	if (!p) {
		return;
	}
	void *q = (void *)p;
	p = nullptr;
	auto it = csr->allocs.find(q);
	if (it == csr->allocs.end()) {
		cudaFree(q);
		return;
	}
	const size_t bytes = it->second;
	csr->allocs.erase(it);
	pgq_ctx *ctx = csr->ctx;
	{
		std::lock_guard<std::mutex> g(ctx->mu);
		if (ctx->buf_cache_bytes + bytes <= ctx->buf_cache_limit) {
			ctx->buf_cache.emplace(bytes, q);
			ctx->buf_cache_bytes += bytes;
			return;
		}
	}
	cudaFree(q);
}

static void free_dir(pgq_csr *csr, DirGraph &g) {
	dev_free(csr, g.off);
	dev_free(csr, g.adj);
	dev_free(csr, g.head);
	dev_free(csr, g.nzrow);
	dev_free(csr, g.chunk_rank);
	g = DirGraph();
}

static void free_pull(pgq_csr *csr) {
	PullGraph &g = csr->pull;
	dev_free(csr, g.adj);
	dev_free(csr, g.head);
	dev_free(csr, g.chunk_rank);
	dev_free(csr, g.row);
	dev_free(csr, g.s_adj);
	dev_free(csr, g.s_row);
	dev_free(csr, g.s_off);
	g = PullGraph();
}

static void free_staging(pgq_csr *csr) {
	dev_free(csr, csr->st_cnt);
	dev_free(csr, csr->st_src);
	dev_free(csr, csr->st_dst);
	dev_free(csr, csr->st_eid);
	dev_free(csr, csr->st_w);
}

// Waits for every chunk that is still on its way through a staging ring.
static int drain_rings(pgq_csr *csr, bool have_lock = false) {
	std::vector<std::shared_ptr<StageRing>> rings;
	if (have_lock) {
		rings.swap(csr->rings);
	} else {
		std::lock_guard<std::mutex> g(csr->mu);
		rings.swap(csr->rings);
	}
	cudaError_t bad = cudaSuccess;
	for (auto &r : rings) {
		cudaError_t e = cudaStreamSynchronize(r->stream);
		if (e != cudaSuccess) {
			bad = e;
		}
	}
	if (bad != cudaSuccess) {
		cudaGetLastError();
		return pgq_fail(PGQ_ERR_CUDA, "a create_csr chunk failed on the device: %s", cudaGetErrorString(bad));
	}
	return PGQ_OK;
}

extern "C" void pgq_csr_free(pgq_csr *csr) {
	if (!csr) {
		return;
	}
	cudaSetDevice(csr->ctx->device);
	drain_rings(csr); // (a CSR dropped half-way through its build, e.g. by the ConstraintException of csr_creation.cpp:121-125)
	free_dir(csr, csr->out);
	free_dir(csr, csr->in);
	free_pull(csr);
	dev_free(csr, csr->edge_ids);
	dev_free(csr, csr->perm);
	dev_free(csr, csr->inv);
	dev_free(csr, csr->w_bits);
	dev_free(csr, csr->d_err);
	free_staging(csr);
	delete csr;
}

// Reads a device error flag (synchronises the stream).
static int read_flag(int *d_flag, cudaStream_t s, int *value) {
	PGQ_CUDA(cudaMemcpyAsync(value, d_flag, sizeof(int), cudaMemcpyDeviceToHost, s));
	PGQ_CUDA(cudaStreamSynchronize(s));
	return PGQ_OK;
}

// Builds head / nzrow / chunk_rank for a direction whose off[] and adj[] are in place.
static int build_dir_metadata(pgq_csr *csr, DirGraph &g, Workspace *ws, cudaStream_t s) {
	int64_t n = csr->n, m = csr->m;
	g.nchunks = (m + PGQ_CHUNK - 1) / PGQ_CHUNK;
	size_t head_words = (size_t)std::max<int64_t>(g.nchunks, 1) * PGQ_STEPS;
	PGQ_TRY(dev_alloc(csr, (void **)&g.head, head_words * sizeof(uint32_t)));
	PGQ_TRY(dev_alloc(csr, (void **)&g.chunk_rank, (size_t)std::max<int64_t>(g.nchunks, 1) * sizeof(int32_t)));
	PGQ_CUDA(cudaMemsetAsync(g.head, 0, head_words * sizeof(uint32_t), s));
	PGQ_CUDA(cudaMemsetAsync(g.chunk_rank, 0, (size_t)std::max<int64_t>(g.nchunks, 1) * sizeof(int32_t), s));
	int32_t *nzflag, *scan_tmp;
	PGQ_TRY(pgq_ws_reserve(ws, 0, (size_t)(n + 1) * sizeof(int32_t), (void **)&nzflag));
	PGQ_TRY(pgq_ws_reserve(ws, 1, pgq_scan_tmp_elems(n + 1) * sizeof(int32_t), (void **)&scan_tmp));
	PGQ_CUDA(cudaMemsetAsync(nzflag, 0, (size_t)(n + 1) * sizeof(int32_t), s));
	if (n > 0) {
		k_mark_heads<<<grid_for(n, 256), 256, 0, s>>>(g.off, n, g.head, nzflag);
		PGQ_CUDA(cudaGetLastError());
	}
	PGQ_TRY(pgq_scan_exclusive_i32(nzflag, nzflag, n + 1, scan_tmp, s));
	int32_t nnz = 0;
	PGQ_CUDA(cudaMemcpyAsync(&nnz, nzflag + n, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
	PGQ_CUDA(cudaStreamSynchronize(s));
	g.nnz = nnz;
	PGQ_TRY(dev_alloc(csr, (void **)&g.nzrow, (size_t)std::max<int64_t>(nnz, 1) * sizeof(int32_t)));
	if (n > 0 && nnz > 0) {
		k_fill_rows<<<grid_for(n, 256), 256, 0, s>>>(g.off, nzflag, n, g.nzrow, g.chunk_rank);
		PGQ_CUDA(cudaGetLastError());
	}
	return PGQ_OK;
}

// The in-CSC once more in the layout of the fused bottom-up level (PullGraph): long rows chunk-walked,
// short rows in degree-sorted slices.  Rows [0, n_ab) are exactly the rows with in-edges.
static int build_pull_graph(pgq_csr *csr, Workspace *ws, cudaStream_t s) {
	PullGraph &g = csr->pull;
	const int64_t n_rows = csr->n_ab, m = csr->m;
	g = PullGraph();
	int32_t *long_deg, *long_flag, *short_flag, *scan_tmp;
	const size_t row_bytes = (size_t)(n_rows + 2) * sizeof(int32_t);
	PGQ_TRY(pgq_ws_reserve(ws, 0, row_bytes, (void **)&long_deg));
	PGQ_TRY(pgq_ws_reserve(ws, 9, row_bytes, (void **)&long_flag));
	PGQ_TRY(pgq_ws_reserve(ws, 10, row_bytes, (void **)&short_flag));
	PGQ_TRY(pgq_ws_reserve(ws, 1, pgq_scan_tmp_elems(std::max<int64_t>(n_rows, m / 32) + 2) * sizeof(int32_t), (void **)&scan_tmp));
	k_pull_classify<<<grid_for(n_rows + 1, 256, 148 * 8), 256, 0, s>>>(csr->in.off, n_rows, long_deg, long_flag, short_flag);
	PGQ_CUDA(cudaGetLastError());
	PGQ_TRY(pgq_scan_exclusive_i32(long_deg, long_deg, n_rows + 1, scan_tmp, s));
	PGQ_TRY(pgq_scan_exclusive_i32(long_flag, long_flag, n_rows + 1, scan_tmp, s));
	PGQ_TRY(pgq_scan_exclusive_i32(short_flag, short_flag, n_rows + 1, scan_tmp, s));
	int32_t totals[3] = {0, 0, 0};
	PGQ_CUDA(cudaMemcpyAsync(&totals[0], long_deg + n_rows, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
	PGQ_CUDA(cudaMemcpyAsync(&totals[1], long_flag + n_rows, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
	PGQ_CUDA(cudaMemcpyAsync(&totals[2], short_flag + n_rows, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
	PGQ_CUDA(cudaStreamSynchronize(s));
	g.m = totals[0];
	g.n_rows = totals[1];
	g.n_short = totals[2];
	g.nchunks = (g.m + PGQ_CHUNK - 1) / PGQ_CHUNK;
	g.n_slices = (g.n_short + 31) / 32;
	// ---- long part
	const size_t head_words = (size_t)std::max<int64_t>(g.nchunks, 1) * PGQ_STEPS;
	// (padded to whole ranges of 1024 positions: the bottom-up kernel fetches a range with one 4 KB bulk copy)
	const size_t adj_elems = (size_t)((std::max<int64_t>(g.m, 1) + 1023) / 1024) * 1024;
	PGQ_TRY(dev_alloc(csr, (void **)&g.adj, adj_elems * sizeof(int32_t)));
	PGQ_CUDA(cudaMemsetAsync(g.adj + adj_elems - 1024, 0xFF, 1024 * sizeof(int32_t), s));
	PGQ_TRY(dev_alloc(csr, (void **)&g.head, head_words * sizeof(uint32_t)));
	PGQ_TRY(dev_alloc(csr, (void **)&g.chunk_rank, (size_t)std::max<int64_t>(g.nchunks, 1) * sizeof(int32_t)));
	PGQ_TRY(dev_alloc(csr, (void **)&g.row, (size_t)std::max<int64_t>(g.n_rows, 1) * sizeof(int32_t)));
	PGQ_CUDA(cudaMemsetAsync(g.head, 0, head_words * sizeof(uint32_t), s));
	PGQ_CUDA(cudaMemsetAsync(g.chunk_rank, 0, (size_t)std::max<int64_t>(g.nchunks, 1) * sizeof(int32_t), s));
	if (g.n_rows > 0) {
		int32_t *off_by_rank;
		PGQ_TRY(pgq_ws_reserve(ws, 11, (size_t)(g.n_rows + 2) * sizeof(int32_t), (void **)&off_by_rank));
		k_pull_long_fill<<<grid_for(n_rows * 32, 256, 148 * 16), 256, 0, s>>>(csr->in.off, csr->in.adj, n_rows, long_deg,
		                                                                long_flag, g.adj, g.row, off_by_rank);
		const int32_t m_long = (int32_t)g.m;
		PGQ_CUDA(cudaMemcpyAsync(off_by_rank + g.n_rows, &m_long, sizeof(int32_t), cudaMemcpyHostToDevice, s));
		k_pull_long_meta<<<grid_for(g.n_rows, 256, 148 * 8), 256, 0, s>>>(off_by_rank, g.n_rows, g.head, g.chunk_rank);
		PGQ_CUDA(cudaGetLastError());
		PGQ_CUDA(cudaStreamSynchronize(s)); // (m_long lives on this frame)
	}
	// ---- short part: sort the short rows by descending degree (one stable radix pass: ties stay in id order)
	PGQ_TRY(dev_alloc(csr, (void **)&g.s_row, (size_t)std::max<int64_t>(g.n_slices * 32, 1) * sizeof(int32_t)));
	PGQ_TRY(dev_alloc(csr, (void **)&g.s_off, (size_t)(g.n_slices + 2) * sizeof(int32_t)));
	if (g.n_short > 0) {
		int32_t *key_a, *key_b, *val_a, *val_b, *key_res, *val_res;
		const size_t kv = (size_t)(g.n_slices * 32 + 32) * sizeof(int32_t);
		PGQ_TRY(pgq_ws_reserve(ws, 5, std::max(kv, ws->cap[5]), (void **)&key_a));
		PGQ_TRY(pgq_ws_reserve(ws, 6, std::max(kv, ws->cap[6]), (void **)&key_b));
		PGQ_TRY(pgq_ws_reserve(ws, 7, std::max(kv, ws->cap[7]), (void **)&val_a));
		PGQ_TRY(pgq_ws_reserve(ws, 12, kv, (void **)&val_b));
		k_pull_short_list<<<grid_for(n_rows, 256, 148 * 8), 256, 0, s>>>(csr->in.off, n_rows, short_flag, key_a, val_a);
		PGQ_CUDA(cudaGetLastError());
		PGQ_TRY(radix_sort_pairs(ws, key_a, key_b, val_a, val_b, g.n_short, 5, s, &key_res, &val_res));
		k_pull_slice_width<<<grid_for(g.n_slices + 1, 256, 148 * 8), 256, 0, s>>>(key_res, g.n_short, g.n_slices, g.s_off);
		PGQ_CUDA(cudaGetLastError());
		PGQ_TRY(pgq_scan_exclusive_i32(g.s_off, g.s_off, g.n_slices + 1, scan_tmp, s));
		int32_t total = 0;
		PGQ_CUDA(cudaMemcpyAsync(&total, g.s_off + g.n_slices, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
		PGQ_CUDA(cudaStreamSynchronize(s));
		g.s_total = total;
		PGQ_TRY(dev_alloc(csr, (void **)&g.s_adj, (size_t)std::max<int64_t>(g.s_total, 1) * sizeof(int32_t)));
		k_pull_short_fill<<<grid_for(g.n_slices * 32, 256, 148 * 16), 256, 0, s>>>(csr->in.off, csr->in.adj, val_res, g.n_short,
		                                                                    g.n_slices, g.s_off, g.s_adj, g.s_row);
		PGQ_CUDA(cudaGetLastError());
	} else {
		PGQ_CUDA(cudaMemsetAsync(g.s_off, 0, (size_t)(g.n_slices + 2) * sizeof(int32_t), s));
		PGQ_TRY(dev_alloc(csr, (void **)&g.s_adj, 256));
	}
	return PGQ_OK;
}

// out.off / out.adj (/ edge_ids) are in place: validate, build metadata, transpose, mark finalized.
static int finish_csr(pgq_csr *csr, Workspace *ws, cudaStream_t s) {
	int64_t n = csr->n, m = csr->m;
	int *d_err;
	PGQ_TRY(pgq_ws_reserve(ws, 2, 256, (void **)&d_err));
	PGQ_CUDA(cudaMemsetAsync(d_err, 0, sizeof(int), s));
	k_check_offsets<<<grid_for(n + 1, 256), 256, 0, s>>>(csr->out.off, n, m, d_err);
	PGQ_CUDA(cudaGetLastError());
	int flag = 0;
	PGQ_TRY(read_flag(d_err, s, &flag));
	if (flag) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "CSR offsets are not a non-decreasing sequence from 0 to m");
	}
	PGQ_TRY(build_dir_metadata(csr, csr->out, ws, s));

	// in-edge CSC: histogram of targets -> scan gives the offsets; a STABLE sort of (target, source)
	// over the source-ordered out-edges gives in-lists sorted by source id, which makes the
	// bottom-up gathers of neighbouring lanes fall into the same cache lines
	PGQ_TRY(dev_alloc(csr, (void **)&csr->in.off, (size_t)(n + 1) * sizeof(int32_t)));
	PGQ_TRY(dev_alloc(csr, (void **)&csr->in.adj, (size_t)std::max<int64_t>(m, 1) * sizeof(int32_t)));
	int32_t *scan_tmp;
	PGQ_TRY(pgq_ws_reserve(ws, 1, pgq_scan_tmp_elems(n + 1) * sizeof(int32_t), (void **)&scan_tmp));
	PGQ_CUDA(cudaMemsetAsync(csr->in.off, 0, (size_t)(n + 1) * sizeof(int32_t), s));
	if (m > 0) {
		k_histogram<<<grid_for(m, 256, 148 * 16), 256, 0, s>>>(csr->out.adj, m, csr->in.off);
		PGQ_CUDA(cudaGetLastError());
	}
	PGQ_TRY(pgq_scan_exclusive_i32(csr->in.off, csr->in.off, n + 1, scan_tmp, s));
	if (m > 0) {
		int32_t *rowid, *keys_out;
		PGQ_TRY(pgq_ws_reserve(ws, 5, (size_t)m * sizeof(int32_t), (void **)&keys_out));
		PGQ_TRY(pgq_ws_reserve(ws, 6, (size_t)m * sizeof(int32_t), (void **)&rowid));
		int end_bit = 1;
		while (end_bit < 31 && ((int64_t)1 << end_bit) < n) {
			end_bit++;
		}
		k_edge_rows<<<grid_for(csr->out.nchunks * 32, 256, 148 * 16), 256, 0, s>>>(csr->out, m, rowid);
		PGQ_CUDA(cudaGetLastError());
		int32_t *keys_a, *keys_res, *vals_res;
		PGQ_TRY(pgq_ws_reserve(ws, 7, (size_t)m * sizeof(int32_t), (void **)&keys_a));
		PGQ_CUDA(cudaMemcpyAsync(keys_a, csr->out.adj, (size_t)m * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
		PGQ_TRY(radix_sort_pairs(ws, keys_a, keys_out, rowid, csr->in.adj, m, end_bit, s, &keys_res, &vals_res));
		if (vals_res != csr->in.adj) {
			PGQ_CUDA(cudaMemcpyAsync(csr->in.adj, vals_res, (size_t)m * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
		}
	}
	PGQ_TRY(build_dir_metadata(csr, csr->in, ws, s));
	PGQ_TRY(build_pull_graph(csr, ws, s));
	PGQ_CUDA(cudaStreamSynchronize(s));
	static std::atomic<uint64_t> next_uid {1};
	csr->uid = next_uid++;
	csr->finalized = true;
	return PGQ_OK;
}

static int check_sizes(int64_t n, int64_t m) {
	if (n < 0 || m < 0) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "negative size");
	}
	if (n >= 0x7fffffffLL - 2 || m >= 0x7fffffffLL) {
		return pgq_fail(PGQ_ERR_RANGE, "n=%lld / m=%lld exceed the int32 device CSR", (long long)n, (long long)m);
	}
	return PGQ_OK;
}

extern "C" int pgq_csr_create(pgq_ctx *ctx, int64_t n, pgq_csr **out) {
	if (!ctx || !out) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "null argument");
	}
	*out = nullptr;
	PGQ_TRY(check_sizes(n, 0));
	PGQ_CUDA(cudaSetDevice(ctx->device));
	pgq_csr *csr = new (std::nothrow) pgq_csr();
	if (!csr) {
		return pgq_fail(PGQ_ERR_OOM, "host allocation failed");
	}
	csr->ctx = ctx;
	csr->n = n;
	int st = dev_alloc(csr, (void **)&csr->st_cnt, (size_t)(n + 1) * sizeof(int32_t));
	if (st == PGQ_OK) {
		st = dev_alloc(csr, (void **)&csr->d_err, 256);
	}
	if (st == PGQ_OK) {
		cudaError_t e = cudaMemset(csr->st_cnt, 0, (size_t)(n + 1) * sizeof(int32_t));
		if (e == cudaSuccess) {
			e = cudaMemset(csr->d_err, 0, 256);
		}
		if (e != cudaSuccess) {
			cudaGetLastError();
			st = pgq_fail(PGQ_ERR_CUDA, "cudaMemset failed: %s", cudaGetErrorString(e));
		}
	}
	if (st != PGQ_OK) {
		pgq_csr_free(csr);
		return st;
	}
	*out = csr;
	return PGQ_OK;
}

// Copies a host int64 column to the device in pieces and narrows it to int32 with a range check.
static int upload_narrow(Workspace *ws, const int64_t *host, int64_t count, int64_t lo, int64_t hi, int32_t *d_out,
                         int *d_err, cudaStream_t s) {
	const int64_t piece = (int64_t)1 << 24;
	int64_t *tmp;
	PGQ_TRY(pgq_ws_reserve(ws, 4, (size_t)std::min(piece, std::max<int64_t>(count, 1)) * sizeof(int64_t), (void **)&tmp));
	for (int64_t o = 0; o < count; o += piece) {
		int64_t c = std::min(piece, count - o);
		PGQ_CUDA(cudaMemcpyAsync(tmp, host + o, (size_t)c * sizeof(int64_t), cudaMemcpyHostToDevice, s));
		k_narrow<<<grid_for(c, 256, 148 * 8), 256, 0, s>>>(tmp, d_out + o, c, lo, hi, d_err);
		PGQ_CUDA(cudaGetLastError());
		PGQ_CUDA(cudaStreamSynchronize(s)); // tmp is reused by the next piece
	}
	return PGQ_OK;
}

// ---- staging rings ---------------------------------------------------------------------------------
#define STAGE_ROWS 4096 // rows per slot (a DuckDB DataChunk holds <= 2048)
#define STAGE_COLS 4    // src, dst, edge id, weight
#define STAGE_SLOTS 8

StageRing::~StageRing() {
	// (runs when the owning thread ends and no CSR refers to the ring any more)
	int cur = -1;
	cudaGetDevice(&cur);
	cudaSetDevice(device);
	if (stream) {
		cudaStreamSynchronize(stream);
	}
	for (auto e : ev) {
		cudaEventDestroy(e);
	}
	if (stream) {
		cudaStreamDestroy(stream);
	}
	if (pinned) {
		cudaFreeHost(pinned);
	}
	if (dev) {
		cudaFree(dev);
	}
	if (cur >= 0) {
		cudaSetDevice(cur);
	}
	cudaGetLastError();
}

static thread_local std::vector<std::shared_ptr<StageRing>> t_rings; // one per device this thread has fed

static int ring_for(pgq_csr *csr, std::shared_ptr<StageRing> *out) {
	const int device = csr->ctx->device;
	std::shared_ptr<StageRing> ring;
	for (auto &r : t_rings) {
		if (r->device == device) {
			ring = r;
		}
	}
	if (!ring) {
		ring = std::make_shared<StageRing>();
		ring->device = device;
		ring->slot_bytes = (size_t)STAGE_ROWS * STAGE_COLS * sizeof(int64_t);
		ring->nslots = STAGE_SLOTS;
		cudaError_t e = cudaStreamCreateWithFlags(&ring->stream, cudaStreamNonBlocking);
		if (e == cudaSuccess) {
			e = cudaHostAlloc((void **)&ring->pinned, ring->slot_bytes * ring->nslots, cudaHostAllocDefault);
		}
		if (e == cudaSuccess) {
			e = cudaMalloc((void **)&ring->dev, ring->slot_bytes * ring->nslots);
		}
		for (int i = 0; i < ring->nslots && e == cudaSuccess; i++) {
			cudaEvent_t ev;
			e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
			if (e == cudaSuccess) {
				ring->ev.push_back(ev);
			}
		}
		if (e != cudaSuccess) {
			cudaGetLastError();
			return pgq_fail(e == cudaErrorMemoryAllocation ? PGQ_ERR_OOM : PGQ_ERR_CUDA, "staging ring creation failed: %s",
			                cudaGetErrorString(e));
		}
		t_rings.push_back(ring);
	}
	{
		std::lock_guard<std::mutex> g(csr->mu);
		bool known = false;
		for (auto &r : csr->rings) {
			known |= (r.get() == ring.get());
		}
		if (!known) {
			csr->rings.push_back(ring);
		}
	}
	*out = ring;
	return PGQ_OK;
}

// claims the next slot of the ring (waits only if the device has not finished with it yet)
static int ring_slot(StageRing &ring, int *slot) {
	const int k = ring.next;
	ring.next = (ring.next + 1) % ring.nslots;
	cudaError_t e = cudaEventSynchronize(ring.ev[(size_t)k]); // immediately true for a never-recorded event
	if (e != cudaSuccess) {
		cudaGetLastError();
		return pgq_fail(PGQ_ERR_CUDA, "staging slot failed: %s", cudaGetErrorString(e));
	}
	*slot = k;
	return PGQ_OK;
}

__global__ void k_copy64(const int64_t *__restrict__ in, int64_t *__restrict__ out, int64_t count) {
	for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
		out[i] = in[i];
	}
}

extern "C" int pgq_csr_add_vertex_counts(pgq_csr *csr, int64_t count, const int64_t *dense_id, const int64_t *cnt,
                                         int64_t *sum_out) {
	if (!csr || count < 0 || (count > 0 && (!dense_id || !cnt))) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "null argument");
	}
	if (csr->finalized) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "CSR already finalized");
	}
	PGQ_CUDA(cudaSetDevice(csr->ctx->device));
	int64_t sum = 0;
	for (int64_t i = 0; i < count; i++) {
		sum += cnt[i];
	}
	if (count > 0) {
		std::shared_ptr<StageRing> ring;
		PGQ_TRY(ring_for(csr, &ring));
		for (int64_t o = 0; o < count; o += STAGE_ROWS) {
			const int64_t c = std::min<int64_t>(STAGE_ROWS, count - o);
			int slot;
			PGQ_TRY(ring_slot(*ring, &slot));
			int64_t *h = reinterpret_cast<int64_t *>(ring->pinned + (size_t)slot * ring->slot_bytes);
			int64_t *d = reinterpret_cast<int64_t *>(ring->dev + (size_t)slot * ring->slot_bytes);
			memcpy(h, dense_id + o, (size_t)c * sizeof(int64_t));
			memcpy(h + c, cnt + o, (size_t)c * sizeof(int64_t));
			PGQ_CUDA(cudaMemcpyAsync(d, h, (size_t)(2 * c) * sizeof(int64_t), cudaMemcpyHostToDevice, ring->stream));
			k_set_counts<<<grid_for(c, 256, 64), 256, 0, ring->stream>>>(d, d + c, c, csr->n, csr->st_cnt, csr->d_err);
			PGQ_CUDA(cudaGetLastError());
			PGQ_CUDA(cudaEventRecord(ring->ev[(size_t)slot], ring->stream));
		}
	}
	{
		std::lock_guard<std::mutex> g(csr->mu);
		csr->have_counts = true;
	}
	if (sum_out) {
		*sum_out += sum;
	}
	return PGQ_OK;
}

static int add_edges_impl(pgq_csr *csr, int64_t edge_size, int64_t edge_size_count, int64_t count, const int64_t *src,
                          const int64_t *dst, const int64_t *eid, const void *weights, int weight_type) {
	if (!csr || count < 0 || (count > 0 && (!src || !dst || !eid))) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "null argument");
	}
	if (edge_size != edge_size_count) { // csr_creation.cpp:121-125
		return pgq_fail(PGQ_ERR_CONSTRAINT, "%s", pgq_status_text(PGQ_ERR_CONSTRAINT));
	}
	if (csr->finalized) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "CSR already finalized");
	}
	PGQ_TRY(check_sizes(csr->n, edge_size));
	PGQ_CUDA(cudaSetDevice(csr->ctx->device));
	int64_t offset;
	{
		std::lock_guard<std::mutex> g(csr->mu); // CsrInitializeEdge runs once under csr_lock, csr_creation.cpp:43-61
		if (!csr->edge_init) {
			const size_t cap = (size_t)std::max<int64_t>(edge_size, 1);
			int32_t *a = nullptr, *b = nullptr;
			int64_t *c = nullptr, *w = nullptr;
			int st = dev_alloc(csr, (void **)&a, cap * sizeof(int32_t));
			if (st == PGQ_OK) st = dev_alloc(csr, (void **)&b, cap * sizeof(int32_t));
			if (st == PGQ_OK) st = dev_alloc(csr, (void **)&c, cap * sizeof(int64_t));
			if (st == PGQ_OK && weight_type) st = dev_alloc(csr, (void **)&w, cap * sizeof(int64_t)); // CsrInitializeWeight l.63-84
			if (st != PGQ_OK) { // commit all or nothing
				dev_free(csr, a);
				dev_free(csr, b);
				dev_free(csr, c);
				dev_free(csr, w);
				return st;
			}
			csr->st_src = a;
			csr->st_dst = b;
			csr->st_eid = c;
			csr->st_w = w;
			csr->weight_type = weight_type;
			csr->edge_size = edge_size;
			csr->m = edge_size;
			csr->edge_init = true;
		} else if (edge_size != csr->edge_size) {
			return pgq_fail(PGQ_ERR_INVALID_ARG, "edge_size changed between create_csr_edge chunks");
		} else if (weight_type != csr->weight_type) {
			return pgq_fail(PGQ_ERR_INVALID_ARG, "edge weight type changed between create_csr_edge chunks");
		}
		if (csr->staged + count > csr->edge_size) {
			return pgq_fail(PGQ_ERR_INVALID_ARG, "more edge rows (%lld) than edge_size (%lld)",
			                (long long)(csr->staged + count), (long long)csr->edge_size);
		}
		offset = csr->staged; // the arrival ticket of this chunk (pos = ++v[src+1] in the reference)
		csr->staged += count;
	}
	if (count == 0) {
		return PGQ_OK;
	}
	std::shared_ptr<StageRing> ring;
	PGQ_TRY(ring_for(csr, &ring));
	const int cols = weight_type ? 4 : 3;
	for (int64_t o = 0; o < count; o += STAGE_ROWS) {
		const int64_t c = std::min<int64_t>(STAGE_ROWS, count - o);
		int slot;
		PGQ_TRY(ring_slot(*ring, &slot));
		int64_t *h = reinterpret_cast<int64_t *>(ring->pinned + (size_t)slot * ring->slot_bytes);
		int64_t *d = reinterpret_cast<int64_t *>(ring->dev + (size_t)slot * ring->slot_bytes);
		memcpy(h, src + o, (size_t)c * sizeof(int64_t));
		memcpy(h + c, dst + o, (size_t)c * sizeof(int64_t));
		memcpy(h + 2 * c, eid + o, (size_t)c * sizeof(int64_t));
		if (weight_type) {
			memcpy(h + 3 * c, reinterpret_cast<const int64_t *>(weights) + o, (size_t)c * sizeof(int64_t));
		}
		cudaStream_t s = ring->stream;
		PGQ_CUDA(cudaMemcpyAsync(d, h, (size_t)(cols * c) * sizeof(int64_t), cudaMemcpyHostToDevice, s));
		const unsigned grid = grid_for(c, 256, 64);
		k_narrow<<<grid, 256, 0, s>>>(d, csr->st_src + offset + o, c, 0, csr->n, csr->d_err);
		k_narrow<<<grid, 256, 0, s>>>(d + c, csr->st_dst + offset + o, c, 0, csr->n, csr->d_err);
		k_copy64<<<grid, 256, 0, s>>>(d + 2 * c, csr->st_eid + offset + o, c);
		if (weight_type) {
			k_copy64<<<grid, 256, 0, s>>>(d + 3 * c, csr->st_w + offset + o, c);
		}
		PGQ_CUDA(cudaGetLastError());
		PGQ_CUDA(cudaEventRecord(ring->ev[(size_t)slot], s));
	}
	return PGQ_OK;
}

extern "C" int pgq_csr_add_edges(pgq_csr *csr, int64_t edge_size, int64_t edge_size_count, int64_t count,
                                 const int64_t *src, const int64_t *dst, const int64_t *eid) {
	return add_edges_impl(csr, edge_size, edge_size_count, count, src, dst, eid, nullptr, 0);
}

extern "C" int pgq_csr_add_edges_weighted(pgq_csr *csr, int64_t edge_size, int64_t edge_size_count, int64_t count,
                                          const int64_t *src, const int64_t *dst, const int64_t *eid,
                                          const int64_t *weight_i64, const double *weight_f64) {
	if (count > 0 && ((weight_i64 != nullptr) == (weight_f64 != nullptr))) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "exactly one of weight_i64 / weight_f64 must be given");
	}
	if (count == 0) { // nothing to stage (and no way to tell the weight type)
		if (edge_size != edge_size_count) {
			return pgq_fail(PGQ_ERR_CONSTRAINT, "%s", pgq_status_text(PGQ_ERR_CONSTRAINT));
		}
		return csr ? PGQ_OK : pgq_fail(PGQ_ERR_INVALID_ARG, "null argument");
	}
	if (weight_f64) {
		return add_edges_impl(csr, edge_size, edge_size_count, count, src, dst, eid, weight_f64, 2);
	}
	return add_edges_impl(csr, edge_size, edge_size_count, count, src, dst, eid, weight_i64, 1);
}

// The staged edge rows (original ids, arrival order) -> internal numbering -> out-CSR (stable by
// source: the order `pos = ++v[src+1]` yields when one thread feeds the rows, csr_creation.cpp:132-139)
// -> metadata, CSC.  Consumes csr->st_src / st_dst / st_eid.
static int finalize_from_rows(pgq_csr *csr, Workspace *ws, cudaStream_t s) {
	const int64_t n = csr->n, m = csr->m;
	int *d_err;
	int32_t *scan_tmp, *outdeg, *indeg, *flag;
	PGQ_TRY(pgq_ws_reserve(ws, 2, 256, (void **)&d_err));
	PGQ_TRY(pgq_ws_reserve(ws, 1, pgq_scan_tmp_elems(n + 1) * sizeof(int32_t), (void **)&scan_tmp));
	PGQ_TRY(pgq_ws_reserve(ws, 9, (size_t)(n + 1) * sizeof(int32_t), (void **)&outdeg));
	PGQ_TRY(pgq_ws_reserve(ws, 10, (size_t)(n + 1) * sizeof(int32_t), (void **)&indeg));
	PGQ_TRY(pgq_ws_reserve(ws, 0, (size_t)(n + 1) * sizeof(int32_t), (void **)&flag));
	PGQ_TRY(dev_alloc(csr, (void **)&csr->out.off, (size_t)(n + 1) * sizeof(int32_t)));
	PGQ_TRY(dev_alloc(csr, (void **)&csr->out.adj, (size_t)std::max<int64_t>(m, 1) * sizeof(int32_t)));
	PGQ_TRY(dev_alloc(csr, (void **)&csr->edge_ids, (size_t)std::max<int64_t>(m, 1) * sizeof(int64_t)));
	PGQ_TRY(dev_alloc(csr, (void **)&csr->perm, (size_t)std::max<int64_t>(n, 1) * sizeof(int32_t)));
	PGQ_TRY(dev_alloc(csr, (void **)&csr->inv, (size_t)std::max<int64_t>(n, 1) * sizeof(int32_t)));
	PGQ_CUDA(cudaMemsetAsync(d_err, 0, sizeof(int), s));
	PGQ_CUDA(cudaMemsetAsync(outdeg, 0, (size_t)(n + 1) * sizeof(int32_t), s));
	PGQ_CUDA(cudaMemsetAsync(indeg, 0, (size_t)(n + 1) * sizeof(int32_t), s));
	if (m > 0) {
		k_histogram<<<grid_for(m, 256, 148 * 16), 256, 0, s>>>(csr->st_src, m, outdeg);
		k_histogram<<<grid_for(m, 256, 148 * 16), 256, 0, s>>>(csr->st_dst, m, indeg);
	}
	// the degrees must equal the counts given to create_csr_vertex (the reference trusts them and
	// scatters out of place otherwise)
	if (csr->have_counts && n > 0) {
		k_compare_i32<<<grid_for(n, 256, 148 * 8), 256, 0, s>>>(outdeg, csr->st_cnt, n, d_err);
	}
	// internal numbering: one stable sort by (class, descending degree)
	int64_t class_size[4] = {0, 0, 0, 0};
	if (n > 0) {
		int32_t *key_a, *key_b, *val_a, *val_b, *key_res, *val_res;
		int *d_cls;
		const size_t kv_bytes = (size_t)std::max<int64_t>(std::max<int64_t>(n, m), 1) * sizeof(int32_t);
		PGQ_TRY(pgq_ws_reserve(ws, 5, kv_bytes, (void **)&key_a));
		PGQ_TRY(pgq_ws_reserve(ws, 6, kv_bytes, (void **)&key_b));
		PGQ_TRY(pgq_ws_reserve(ws, 7, kv_bytes, (void **)&val_a));
		PGQ_TRY(pgq_ws_reserve(ws, 11, (size_t)(n + 2) * sizeof(int32_t), (void **)&val_b));
		PGQ_TRY(pgq_ws_reserve(ws, 3, 256, (void **)&d_cls));
		PGQ_CUDA(cudaMemsetAsync(d_cls, 0, 4 * sizeof(int), s));
		k_vertex_keys<<<grid_for(n, 256, 148 * 8), 256, 0, s>>>(outdeg, indeg, n, key_a, val_a, d_cls);
		PGQ_CUDA(cudaGetLastError());
		PGQ_TRY(radix_sort_pairs(ws, key_a, key_b, val_a, val_b, n, 24, s, &key_res, &val_res));
		k_invert_perm<<<grid_for(n, 256, 148 * 8), 256, 0, s>>>(val_res, n, csr->perm, csr->inv);
		PGQ_CUDA(cudaGetLastError());
		int h_cls[4] = {0, 0, 0, 0};
		PGQ_CUDA(cudaMemcpyAsync(h_cls, d_cls, 4 * sizeof(int), cudaMemcpyDeviceToHost, s));
		PGQ_CUDA(cudaStreamSynchronize(s));
		for (int c = 0; c < 4; c++) {
			class_size[c] = h_cls[c];
		}
	}
	csr->n_a = class_size[0];
	csr->n_ab = class_size[0] + class_size[1];
	int flag_err = 0;
	PGQ_TRY(read_flag(d_err, s, &flag_err));
	if (flag_err) {
		return pgq_fail(PGQ_ERR_INVALID_ARG,
		                "create_csr_vertex counts do not match the degrees of the edges handed to create_csr_edge");
	}
	// row offsets of the internal out-CSR = CsrInitializeEdge's prefix sum (csr_creation.cpp:57-59)
	PGQ_CUDA(cudaMemsetAsync(csr->out.off, 0, (size_t)(n + 1) * sizeof(int32_t), s));
	if (m > 0) {
		k_apply_perm<<<grid_for(m, 256, 148 * 16), 256, 0, s>>>(csr->st_src, m, csr->perm);
		k_apply_perm<<<grid_for(m, 256, 148 * 16), 256, 0, s>>>(csr->st_dst, m, csr->perm);
		k_histogram<<<grid_for(m, 256, 148 * 16), 256, 0, s>>>(csr->st_src, m, csr->out.off);
	}
	PGQ_TRY(pgq_scan_exclusive_i32(csr->out.off, csr->out.off, n + 1, scan_tmp, s));
	if (m > 0) {
		int32_t *keys_out, *perm_in, *perm_out, *keys_res;
		PGQ_TRY(pgq_ws_reserve(ws, 5, (size_t)m * sizeof(int32_t), (void **)&keys_out));
		PGQ_TRY(pgq_ws_reserve(ws, 6, (size_t)m * sizeof(int32_t), (void **)&perm_in));
		PGQ_TRY(pgq_ws_reserve(ws, 7, (size_t)m * sizeof(int32_t), (void **)&perm_out));
		int end_bit = 1;
		while (end_bit < 31 && ((int64_t)1 << end_bit) < n) {
			end_bit++;
		}
		k_iota<<<grid_for(m, 256, 148 * 8), 256, 0, s>>>(perm_in, m);
		PGQ_CUDA(cudaGetLastError());
		// (st_src is staging and may be clobbered: the out-degree histogram above already used it)
		PGQ_TRY(radix_sort_pairs(ws, csr->st_src, keys_out, perm_in, perm_out, m, end_bit, s, &keys_res, &perm_out));
		if (csr->st_w) {
			PGQ_TRY(dev_alloc(csr, (void **)&csr->w_bits, (size_t)m * sizeof(int64_t)));
		}
		k_gather_edges<<<grid_for(m, 256, 148 * 16), 256, 0, s>>>(perm_out, csr->st_dst, csr->st_eid, csr->st_w, m,
		                                                       csr->out.adj, csr->edge_ids, csr->w_bits);
		PGQ_CUDA(cudaGetLastError());
		if (csr->w_bits) {
			PGQ_CUDA(cudaMemsetAsync(d_err, 0, sizeof(int), s));
			k_any_negative<<<grid_for(m, 256, 148 * 16), 256, 0, s>>>(csr->w_bits, m, csr->weight_type == 2, d_err);
			PGQ_CUDA(cudaGetLastError());
			int neg = 0;
			PGQ_TRY(read_flag(d_err, s, &neg));
			csr->w_negative = neg != 0;
		}
	}
	PGQ_TRY(finish_csr(csr, ws, s));
	PGQ_CUDA(cudaStreamSynchronize(s));
	return PGQ_OK;
}

extern "C" int pgq_csr_finalize(pgq_csr *csr) {
	if (!csr) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "null argument");
	}
	std::lock_guard<std::mutex> g(csr->mu);
	if (csr->finalized) {
		return PGQ_OK;
	}
	PGQ_CUDA(cudaSetDevice(csr->ctx->device));
	if (!csr->edge_init) { // vertices only: an edgeless graph (test/sql/path_finding/edgeless_graph.test)
		csr->edge_size = 0;
		csr->m = 0;
		csr->staged = 0;
	}
	// The undirected CSR CTE doubles BOTH counts (compressed_sparse_row.cpp:125-130,208-223): edge_size is then
	// twice the number of rows that arrive, the reference merely over-allocates e.  The edges are the rows that
	// came; their number must match the vertex counts, which finalize_from_rows checks.
	csr->m = csr->staged;
	PGQ_TRY(drain_rings(csr, true)); // every chunk has landed in the staging columns
	if (csr->d_err) {
		int flag = 0;
		PGQ_CUDA(cudaMemcpy(&flag, csr->d_err, sizeof(int), cudaMemcpyDeviceToHost));
		if (flag) {
			return pgq_fail(PGQ_ERR_RANGE, "create_csr_vertex / create_csr_edge: a rowid lies outside [0,%lld) or a count is negative",
			                (long long)csr->n);
		}
	}
	Workspace *ws;
	PGQ_TRY(pgq_ws_acquire(csr->ctx, &ws));
	int st = finalize_from_rows(csr, ws, ws->stream);
	pgq_ws_release(csr->ctx, ws);
	if (st == PGQ_OK) {
		free_staging(csr);
	}
	return st;
}

extern "C" int pgq_csr_build(pgq_ctx *ctx, int64_t n, int64_t m, const int64_t *src, const int64_t *dst,
                             const int64_t *eid, pgq_csr **out) {
	if (!ctx || !out || (m > 0 && (!src || !dst))) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "null argument");
	}
	*out = nullptr;
	PGQ_TRY(check_sizes(n, m));
	pgq_csr *csr = nullptr;
	PGQ_TRY(pgq_csr_create(ctx, n, &csr));
	int st = PGQ_OK;
	std::vector<int64_t> ids;
	if (!eid && m > 0) { // default edge rowids 0..m-1
		ids.resize((size_t)m);
		for (int64_t i = 0; i < m; i++) {
			ids[(size_t)i] = i;
		}
		eid = ids.data();
	}
	// bulk form: whole columns in large pieces (the chunk-wise staging rings are for DataChunk-sized calls)
	{
		std::lock_guard<std::mutex> g(csr->mu);
		const size_t cap = (size_t)std::max<int64_t>(m, 1);
		st = dev_alloc(csr, (void **)&csr->st_src, cap * sizeof(int32_t));
		if (st == PGQ_OK) st = dev_alloc(csr, (void **)&csr->st_dst, cap * sizeof(int32_t));
		if (st == PGQ_OK) st = dev_alloc(csr, (void **)&csr->st_eid, cap * sizeof(int64_t));
		csr->edge_size = m;
		csr->m = m;
		csr->staged = m;
		csr->edge_init = true;
	}
	if (st == PGQ_OK && m > 0) {
		Workspace *ws = nullptr;
		st = pgq_ws_acquire(ctx, &ws);
		if (st == PGQ_OK) {
			cudaStream_t s = ws->stream;
			st = upload_narrow(ws, src, m, 0, n, csr->st_src, csr->d_err, s);
			if (st == PGQ_OK) st = upload_narrow(ws, dst, m, 0, n, csr->st_dst, csr->d_err, s);
			if (st == PGQ_OK) {
				cudaError_t e = cudaMemcpyAsync(csr->st_eid, eid, (size_t)m * sizeof(int64_t), cudaMemcpyHostToDevice, s);
				if (e == cudaSuccess) {
					e = cudaStreamSynchronize(s);
				}
				if (e != cudaSuccess) {
					cudaGetLastError();
					st = pgq_fail(PGQ_ERR_CUDA, "edge upload failed: %s", cudaGetErrorString(e));
				}
			}
			pgq_ws_release(ctx, ws);
		}
	}
	if (st == PGQ_OK) {
		st = pgq_csr_finalize(csr);
	}
	if (st != PGQ_OK) {
		pgq_csr_free(csr);
		return st;
	}
	*out = csr;
	return PGQ_OK;
}

__global__ void k_range_check_i32(const int32_t *__restrict__ ids, int64_t count, int64_t n, int *err) {
	for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
		if (ids[i] < 0 || ids[i] >= n) {
			*err = 1;
		}
	}
}

extern "C" int pgq_csr_build_device(pgq_ctx *ctx, int64_t n, int64_t m, const int32_t *d_src, const int32_t *d_dst,
                                    const int64_t *d_eid, pgq_csr **out) {
	if (!ctx || !out || (m > 0 && (!d_src || !d_dst))) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "null argument");
	}
	*out = nullptr;
	PGQ_TRY(check_sizes(n, m));
	PGQ_CUDA(cudaSetDevice(ctx->device));
	pgq_csr *csr = new (std::nothrow) pgq_csr();
	if (!csr) {
		return pgq_fail(PGQ_ERR_OOM, "host allocation failed");
	}
	csr->ctx = ctx;
	csr->n = n;
	csr->m = m;
	csr->edge_size = m;
	csr->staged = m;
	csr->edge_init = true;
	Workspace *ws = nullptr;
	int st = pgq_ws_acquire(ctx, &ws);
	if (st != PGQ_OK) {
		delete csr;
		return st;
	}
	cudaStream_t s = ws->stream;
	do {
		int *d_err;
		const size_t cap = (size_t)std::max<int64_t>(m, 1);
		if ((st = pgq_ws_reserve(ws, 2, 256, (void **)&d_err)) != PGQ_OK) break;
		if ((st = dev_alloc(csr, (void **)&csr->st_src, cap * sizeof(int32_t))) != PGQ_OK) break;
		if ((st = dev_alloc(csr, (void **)&csr->st_dst, cap * sizeof(int32_t))) != PGQ_OK) break;
		if ((st = dev_alloc(csr, (void **)&csr->st_eid, cap * sizeof(int64_t))) != PGQ_OK) break;
		cudaMemsetAsync(d_err, 0, sizeof(int), s);
		// the columns may have been produced on any stream of the caller (torch's, cuDF's): the copies below
		// run on a stream of ours, so wait for the whole device once rather than race the producer
		cudaDeviceSynchronize();
		if (m > 0) {
			cudaMemcpyAsync(csr->st_src, d_src, (size_t)m * sizeof(int32_t), cudaMemcpyDeviceToDevice, s);
			cudaMemcpyAsync(csr->st_dst, d_dst, (size_t)m * sizeof(int32_t), cudaMemcpyDeviceToDevice, s);
			k_range_check_i32<<<grid_for(m, 256, 148 * 16), 256, 0, s>>>(csr->st_src, m, n, d_err);
			k_range_check_i32<<<grid_for(m, 256, 148 * 16), 256, 0, s>>>(csr->st_dst, m, n, d_err);
			if (d_eid) {
				cudaMemcpyAsync(csr->st_eid, d_eid, (size_t)m * sizeof(int64_t), cudaMemcpyDeviceToDevice, s);
			} else {
				k_iota64<<<grid_for(m, 256, 148 * 8), 256, 0, s>>>(csr->st_eid, m);
			}
		}
		int flag = 0;
		if ((st = read_flag(d_err, s, &flag)) != PGQ_OK) break;
		if (flag) {
			st = pgq_fail(PGQ_ERR_RANGE, "create_csr_edge: vertex rowid outside [0,%lld)", (long long)n);
			break;
		}
		st = finalize_from_rows(csr, ws, s);
	} while (0);
	pgq_ws_release(ctx, ws);
	if (st != PGQ_OK) {
		pgq_csr_free(csr);
		return st;
	}
	free_staging(csr);
	*out = csr;
	return PGQ_OK;
}

extern "C" int pgq_csr_upload(pgq_ctx *ctx, int64_t n, int64_t m, const int64_t *v, const int64_t *e,
                              const int64_t *edge_ids, pgq_csr **out) {
	if (!ctx || !out || !v || (m > 0 && !e)) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "null argument");
	}
	*out = nullptr;
	PGQ_TRY(check_sizes(n, m));
	PGQ_CUDA(cudaSetDevice(ctx->device));
	pgq_csr *csr = new (std::nothrow) pgq_csr();
	if (!csr) {
		return pgq_fail(PGQ_ERR_OOM, "host allocation failed");
	}
	csr->ctx = ctx;
	csr->n = n;
	csr->m = m;
	csr->edge_size = m;
	csr->staged = m;
	csr->edge_init = true;
	Workspace *ws = nullptr;
	int st = pgq_ws_acquire(ctx, &ws);
	if (st != PGQ_OK) {
		delete csr;
		return st;
	}
	cudaStream_t s = ws->stream;
	do {
		// the finished CSR is turned back into edge rows in CSR position order (which IS the arrival
		// order per source) and goes through the same pipeline as a device-side build
		int *d_err;
		int32_t *off_tmp;
		const size_t cap = (size_t)std::max<int64_t>(m, 1);
		if ((st = pgq_ws_reserve(ws, 2, 256, (void **)&d_err)) != PGQ_OK) break;
		if ((st = pgq_ws_reserve(ws, 11, (size_t)(n + 2) * sizeof(int32_t), (void **)&off_tmp)) != PGQ_OK) break;
		if ((st = dev_alloc(csr, (void **)&csr->st_src, cap * sizeof(int32_t))) != PGQ_OK) break;
		if ((st = dev_alloc(csr, (void **)&csr->st_dst, cap * sizeof(int32_t))) != PGQ_OK) break;
		if ((st = dev_alloc(csr, (void **)&csr->st_eid, cap * sizeof(int64_t))) != PGQ_OK) break;
		cudaMemsetAsync(d_err, 0, sizeof(int), s);
		// v[0..n] are the row offsets in the reference layout (v[n+1] == v[n] == m is padding)
		if ((st = upload_narrow(ws, v, n + 1, 0, m + 1, off_tmp, d_err, s)) != PGQ_OK) break;
		if (m > 0) {
			if ((st = upload_narrow(ws, e, m, 0, n, csr->st_dst, d_err, s)) != PGQ_OK) break;
		}
		k_check_offsets<<<grid_for(n + 1, 256), 256, 0, s>>>(off_tmp, n, m, d_err);
		int flag = 0;
		if ((st = read_flag(d_err, s, &flag)) != PGQ_OK) break;
		if (flag) {
			st = pgq_fail(PGQ_ERR_RANGE, "CSR arrays hold ids outside [0,n) or offsets that do not run from 0 to m");
			break;
		}
		if (m > 0) {
			k_rows_from_offsets<<<grid_for(n * 32, 256, 148 * 16), 256, 0, s>>>(off_tmp, n, csr->st_src);
			if (edge_ids) {
				cudaMemcpyAsync(csr->st_eid, edge_ids, (size_t)m * sizeof(int64_t), cudaMemcpyHostToDevice, s);
			} else {
				k_iota64<<<grid_for(m, 256, 148 * 8), 256, 0, s>>>(csr->st_eid, m);
			}
		}
		st = finalize_from_rows(csr, ws, s);
	} while (0);
	pgq_ws_release(ctx, ws);
	if (st != PGQ_OK) {
		pgq_csr_free(csr);
		return st;
	}
	free_staging(csr);
	*out = csr;
	return PGQ_OK;
}

extern "C" int pgq_csr_download(pgq_csr *csr, int64_t *v_out, int64_t *e_out, int64_t *edge_ids_out) {
	if (!csr) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "null argument");
	}
	if (!csr->finalized) {
		return pgq_fail(PGQ_ERR_NOT_INITIALIZED, "%s", pgq_status_text(PGQ_ERR_NOT_INITIALIZED));
	}
	PGQ_CUDA(cudaSetDevice(csr->ctx->device));
	int64_t n = csr->n, m = csr->m;
	Workspace *ws;
	PGQ_TRY(pgq_ws_acquire(csr->ctx, &ws));
	cudaStream_t s = ws->stream;
	int st = PGQ_OK;
	do {
		// back to the reference's layout: original vertex order, original ids
		int32_t *orig_off, *scan_tmp;
		int64_t *tmp_e, *tmp_id;
		if ((st = pgq_ws_reserve(ws, 0, (size_t)(n + 2) * sizeof(int32_t), (void **)&orig_off)) != PGQ_OK) break;
		if ((st = pgq_ws_reserve(ws, 1, pgq_scan_tmp_elems(n + 1) * sizeof(int32_t), (void **)&scan_tmp)) != PGQ_OK) break;
		if ((st = pgq_ws_reserve(ws, 4, (size_t)std::max<int64_t>(std::max<int64_t>(m, n + 2), 1) * sizeof(int64_t),
		                         (void **)&tmp_e)) != PGQ_OK) break;
		tmp_id = nullptr;
		if (edge_ids_out &&
		    (st = pgq_ws_reserve(ws, 5, (size_t)std::max<int64_t>(m, 1) * sizeof(int64_t), (void **)&tmp_id)) != PGQ_OK) break;
		k_orig_degrees<<<grid_for(n + 1, 256, 148 * 8), 256, 0, s>>>(csr->out.off, csr->perm, n, orig_off);
		if ((st = pgq_scan_exclusive_i32(orig_off, orig_off, n + 1, scan_tmp, s)) != PGQ_OK) break;
		if (m > 0 && (e_out || edge_ids_out)) {
			k_orig_rows<<<grid_for(n * 32, 256, 148 * 16), 256, 0, s>>>(csr->out.off, csr->out.adj, csr->edge_ids, csr->perm,
			                                                       csr->inv, orig_off, n, e_out ? tmp_e : nullptr,
			                                                       edge_ids_out ? tmp_id : nullptr);
			if (e_out) {
				cudaMemcpyAsync(e_out, tmp_e, (size_t)m * sizeof(int64_t), cudaMemcpyDeviceToHost, s);
			}
			if (edge_ids_out) {
				cudaMemcpyAsync(edge_ids_out, tmp_id, (size_t)m * sizeof(int64_t), cudaMemcpyDeviceToHost, s);
			}
			cudaStreamSynchronize(s);
		}
		if (v_out) {
			k_widen<<<grid_for(n + 1, 256, 148 * 8), 256, 0, s>>>(orig_off, tmp_e, n + 1);
			cudaMemcpyAsync(v_out, tmp_e, (size_t)(n + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, s);
			cudaStreamSynchronize(s);
			v_out[n + 1] = v_out[n]; // the reference's padding slot
		}
		cudaError_t e = cudaStreamSynchronize(s);
		if (e == cudaSuccess) {
			e = cudaGetLastError();
		}
		if (e != cudaSuccess) {
			st = pgq_fail(PGQ_ERR_CUDA, "CSR download failed: %s", cudaGetErrorString(e));
		}
	} while (0);
	pgq_ws_release(csr->ctx, ws);
	return st;
}

extern "C" int pgq_csr_info(pgq_csr *csr, int64_t *n, int64_t *m, int64_t *device_bytes) {
	if (!csr) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "null argument");
	}
	if (n) {
		*n = csr->n;
	}
	if (m) {
		*m = csr->m;
	}
	if (device_bytes) {
		*device_bytes = csr->device_bytes;
	}
	return PGQ_OK;
}

extern "C" int pgq_csr_weight_type(pgq_csr *csr, int *weight_type) {
	if (!csr || !weight_type) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "null argument");
	}
	*weight_type = csr->weight_type;
	return PGQ_OK;
}

extern "C" int pgq_csr_download_weights(pgq_csr *csr, void *w_out) {
	if (!csr || !w_out) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "null argument");
	}
	if (!csr->finalized) {
		return pgq_fail(PGQ_ERR_NOT_INITIALIZED, "%s", pgq_status_text(PGQ_ERR_NOT_INITIALIZED));
	}
	if (!csr->w_bits) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "the CSR has no edge weights");
	}
	PGQ_CUDA(cudaSetDevice(csr->ctx->device));
	const int64_t n = csr->n, m = csr->m;
	Workspace *ws;
	PGQ_TRY(pgq_ws_acquire(csr->ctx, &ws));
	cudaStream_t s = ws->stream;
	int st = PGQ_OK;
	do {
		int32_t *orig_off, *scan_tmp;
		int64_t *tmp_w;
		if ((st = pgq_ws_reserve(ws, 0, (size_t)(n + 2) * sizeof(int32_t), (void **)&orig_off)) != PGQ_OK) break;
		if ((st = pgq_ws_reserve(ws, 1, pgq_scan_tmp_elems(n + 1) * sizeof(int32_t), (void **)&scan_tmp)) != PGQ_OK) break;
		if ((st = pgq_ws_reserve(ws, 5, (size_t)std::max<int64_t>(m, 1) * sizeof(int64_t), (void **)&tmp_w)) != PGQ_OK) break;
		k_orig_degrees<<<grid_for(n + 1, 256, 148 * 8), 256, 0, s>>>(csr->out.off, csr->perm, n, orig_off);
		if ((st = pgq_scan_exclusive_i32(orig_off, orig_off, n + 1, scan_tmp, s)) != PGQ_OK) break;
		if (m > 0) {
			k_orig_rows<<<grid_for(n * 32, 256, 148 * 16), 256, 0, s>>>(csr->out.off, csr->out.adj, csr->w_bits, csr->perm,
			                                                       csr->inv, orig_off, n, nullptr, tmp_w);
			cudaMemcpyAsync(w_out, tmp_w, (size_t)m * sizeof(int64_t), cudaMemcpyDeviceToHost, s);
		}
		cudaError_t e = cudaStreamSynchronize(s);
		if (e == cudaSuccess) {
			e = cudaGetLastError();
		}
		if (e != cudaSuccess) {
			st = pgq_fail(PGQ_ERR_CUDA, "weight download failed: %s", cudaGetErrorString(e));
		}
	} while (0);
	pgq_ws_release(csr->ctx, ws);
	return st;
}
