// pgq_internal.h -- shared host-side declarations of libduckpgq_b200 (not part of the C ABI).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <condition_variable>
#include <map>
#include <memory>
#include <mutex>
#include <unordered_map>
#include <string>
#include <vector>

#include "duckpgq_b200.h"

typedef unsigned long long u64;

// ---- error plumbing: nothing throws across the C ABI -------------------------------------------
void pgq_set_error(const char *fmt, ...);
int pgq_fail(int status, const char *fmt, ...);

#define PGQ_CUDA(call)                                                                                      \
	do {                                                                                                    \
		cudaError_t _e = (call);                                                                            \
		if (_e != cudaSuccess) {                                                                            \
			cudaGetLastError();                                                                             \
			return pgq_fail(_e == cudaErrorMemoryAllocation ? PGQ_ERR_OOM : PGQ_ERR_CUDA, "%s failed: %s (%s:%d)", \
			                #call, cudaGetErrorString(_e), __FILE__, __LINE__);                             \
		}                                                                                                   \
	} while (0)

#define PGQ_TRY(call)           \
	do {                        \
		int _s = (call);        \
		if (_s != PGQ_OK) {     \
			return _s;          \
		}                       \
	} while (0)

// ---- geometry of the edge-tiled kernels --------------------------------------------------------
// A "chunk" is 256 consecutive positions of an adjacency array, processed by one warp as 8 steps
// of 32 lane-strided edges (perfectly coalesced 128 B loads).  Which row (vertex) an edge belongs
// to is recovered from a 1-bit-per-edge row-head bitmap plus one rank per chunk, so the kernels
// never binary-search the offsets and never see empty rows.
#define PGQ_CHUNK 256
#define PGQ_STEPS 8

// One direction of the graph: the out-CSR (row = source) or the in-CSC (row = destination).
struct DirGraph {
	int32_t *off = nullptr;        // [n+1] row offsets
	int32_t *adj = nullptr;        // [m]   neighbour ids
	uint32_t *head = nullptr;      // [nchunks*8] bit e = 1 iff position e is the first of its row
	int32_t *nzrow = nullptr;      // [nnz] ids of the non-empty rows, ascending
	int32_t *chunk_rank = nullptr; // [nchunks] index into nzrow of the row holding position 256*c
	int64_t nnz = 0;
	int64_t nchunks = 0;
};

// The in-edges in the layout of the fused bottom-up level (pgq_pull.cuh), built once per CSR next to the
// plain in-CSC (which path reconstruction keeps using):
//   long rows  (in-degree >= PGQ_SHORT_DEG): in-lists back to back in row order + head bitmap + chunk ranks;
//              `row` maps the rank of a long row to its vertex id
//   short rows (in-degree 1 .. PGQ_SHORT_DEG - 1): sorted by descending degree (ties by id), in slices of 32
//              rows stored column-major: s_adj[s_off[s] + j * 32 + l] = j-th in-neighbour of the slice's l-th row
//              (-1 = padding), s_row[s * 32 + l] = that row's vertex id (-1 = none)
#define PGQ_SHORT_DEG 32
struct PullGraph {
	int32_t *adj = nullptr;
	uint32_t *head = nullptr;
	int32_t *chunk_rank = nullptr;
	int32_t *row = nullptr;
	int64_t m = 0, nchunks = 0, n_rows = 0;
	int32_t *s_adj = nullptr;
	int32_t *s_row = nullptr;
	int32_t *s_off = nullptr;
	int64_t n_short = 0, n_slices = 0, s_total = 0;
};

#define PGQ_WS_SLOTS 32
// Scratch of one path-function call (mask arrays etc.), pooled per context and grown on demand.
struct Workspace {
	void *buf[PGQ_WS_SLOTS] = {};
	size_t cap[PGQ_WS_SLOTS] = {};
	cudaStream_t stream = nullptr; // owned stream for host-pointer calls
	cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
	std::vector<cudaEvent_t> ev_pool; // pairs around expansion kernels
	void *pinned = nullptr;           // small pinned status block
	size_t pinned_cap = 0;
	// The three lane-mask arrays are known to hold zeros from row clean_from on, for the CSR / lane width below
	// (a search only ever writes the rows of vertices WITH in-edges, which the internal numbering puts first):
	// a batch then clears just the first clean_from rows.  Reset whenever the arrays or their user change.
	uint64_t clean_csr_uid = 0;
	int clean_w = 0;
	int64_t clean_from = -1;
	const void *clean_ptr[3] = {nullptr, nullptr, nullptr};
};

struct pgq_ctx {
	int device = 0;
	int sm_count = 148;
	std::mutex mu;
	std::condition_variable cv;
	std::vector<Workspace *> free_ws;
	int live_ws = 0; // workspaces in existence (in use + pooled)
	int max_ws = 8;  // upper bound on them: a workspace holds three lane-mask arrays of the graph's size
	// Device buffers of freed CSRs, by exact size: DuckPGQ rebuilds a CSR of the same shape for every
	// query, so the ~20 cudaMalloc / cudaFree pairs of a CSR are paid once per shape, not once per query.
	std::multimap<size_t, void *> buf_cache;
	size_t buf_cache_bytes = 0;
	size_t buf_cache_limit = (size_t)16 << 30;
};

// Pinned staging ring + stream of one host thread for create_csr_vertex / create_csr_edge chunks:
// a chunk is copied into a pinned slot, sent to the device and narrowed / scattered asynchronously;
// nothing waits per chunk (a slot is waited for only when the ring wraps around onto a busy one).
struct StageRing {
	int device = 0;
	cudaStream_t stream = nullptr;
	char *pinned = nullptr; // nslots x slot_bytes
	char *dev = nullptr;    // nslots x slot_bytes
	size_t slot_bytes = 0;
	int nslots = 0;
	int next = 0;
	std::vector<cudaEvent_t> ev; // slot reusable once its event has completed
	~StageRing();
};

struct pgq_csr {
	pgq_ctx *ctx = nullptr;
	int64_t n = 0;
	int64_t m = 0;
	bool finalized = false;
	DirGraph out;
	DirGraph in;
	PullGraph pull; // the in-edges once more, laid out for the fused bottom-up level
	int64_t *edge_ids = nullptr; // [m] edge rowids in out-CSR order (the CSR position when none were given)
	// Internal vertex numbering: vertices are renumbered so that the ones whose masks are actually
	// gathered (out-degree > 0 and in-degree > 0) come first, then in-only, out-only and isolated
	// vertices, each class in its original order.  All device arrays use internal ids; perm/inv
	// translate at the boundary (pairs in, path vertices / downloaded CSR out).
	int32_t *perm = nullptr; // [n] original id -> internal id
	int32_t *inv = nullptr;  // [n] internal id -> original id
	int64_t n_a = 0;         // vertices with out- and in-edges (the randomly gathered part of the masks)
	int64_t n_ab = 0;        // ... plus vertices with only in-edges: the only ones a BFS level can reach
	uint64_t uid = 0;        // unique per CSR object of the process (workspaces remember whose zeros they hold)
	int64_t device_bytes = 0;
	// incremental build state (create_csr_vertex / create_csr_edge chunks)
	std::mutex mu;
	int32_t *st_cnt = nullptr; // [n] per-vertex counts from create_csr_vertex
	bool have_counts = false;
	bool edge_init = false;
	int64_t edge_size = 0;
	int64_t staged = 0;
	int32_t *st_src = nullptr; // [edge_size]
	int32_t *st_dst = nullptr;
	int64_t *st_eid = nullptr;
	int64_t *st_w = nullptr;   // [edge_size] raw 8-byte weights (create_csr_edge's BIGINT / DOUBLE overloads)
	int *d_err = nullptr;      // device flag: a chunk held an id outside [0, n)
	std::vector<std::shared_ptr<StageRing>> rings; // staging rings that still may hold chunks in flight
	// edge weights in out-CSR position order (CSR::w / CSR::w_double, compressed_sparse_row.hpp:32-40)
	int weight_type = 0; // 0 none, 1 BIGINT, 2 DOUBLE
	int64_t *w_bits = nullptr;
	bool w_negative = false; // some weight < 0 (-inf included; not -0.0 or a NaN), set at finalize
	std::unordered_map<void *, size_t> allocs; // every device buffer of this CSR with its size (buffer cache)
};

// ---- helpers implemented in pgq_csr.cu ---------------------------------------------------------
int pgq_ws_acquire(pgq_ctx *ctx, Workspace **out);     // blocks while the context's workspace budget is used up
int pgq_ws_try_acquire(pgq_ctx *ctx, Workspace **out); // PGQ_ERR_OOM instead of blocking
int pgq_ws_grow(Workspace *ws, int slot, size_t bytes, size_t keep_bytes, cudaStream_t s, void **out);
void pgq_ws_release(pgq_ctx *ctx, Workspace *ws);
int pgq_ws_reserve(Workspace *ws, int slot, size_t bytes, void **out);
int pgq_ws_pinned(Workspace *ws, size_t bytes, void **out);
int pgq_scan_exclusive_i32(const int32_t *in, int32_t *out, int64_t count, int32_t *block_tmp, cudaStream_t s);
size_t pgq_scan_tmp_elems(int64_t count);

// ---- BFS drivers implemented in pgq_bfs.cu -----------------------------------------------------
int pgq_bfs_lengths_device(pgq_csr *csr, Workspace *ws, int64_t p, const int64_t *d_src, const int64_t *d_dst,
                           const uint8_t *d_src_valid, const pgq_options *opts, int64_t *d_out_len,
                           uint8_t *d_out_valid, cudaStream_t stream, pgq_stats *stats);
int pgq_bfs_paths_device(pgq_csr *csr, Workspace *ws, int64_t p, const int64_t *d_src, const int64_t *d_dst,
                         const uint8_t *d_src_valid, const pgq_options *opts, int64_t *d_out_offsets,
                         int64_t *d_out_lengths, uint8_t *d_out_valid, int64_t **d_out_elems, int64_t *out_total,
                         cudaStream_t stream, pgq_stats *stats);
