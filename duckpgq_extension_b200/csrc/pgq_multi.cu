// pgq_multi.cu -- one process, several GPUs of one box (SURVEY.md section 8e): every search is independent given
// a read-only CSR, so the CSR is REPLICATED (peer copies over NVLink from the device that built it) and the
// search lanes of a call are dealt over the devices (pgq_options.shard_index / shard_count).  One persistent
// host thread per device runs its shard and writes the rows it answered straight into the caller's result
// columns -- no collective, no per-level exchange, no barrier besides the end of the call.
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstring>
#include <functional>
#include <thread>

#include "pgq_internal.h"

// ---- CSR replica on another device -------------------------------------------------------------------------
template <typename T>
static int clone_array(pgq_csr *dst, int dst_dev, T **out, const T *src, int src_dev, size_t count, cudaStream_t s) {
	*out = nullptr;
	if (!src) {
		return PGQ_OK;
	}
	const size_t bytes = std::max<size_t>(count, 1) * sizeof(T);
	void *p = nullptr;
	cudaError_t e = cudaMalloc(&p, bytes);
	if (e != cudaSuccess) {
		cudaGetLastError();
		return pgq_fail(PGQ_ERR_OOM, "device allocation of %zu bytes on device %d failed: %s", bytes, dst_dev,
		                cudaGetErrorString(e));
	}
	dst->allocs[p] = bytes;
	dst->device_bytes += (int64_t)bytes;
	*out = (T *)p;
	if (count > 0) {
		e = cudaMemcpyPeerAsync(p, dst_dev, src, src_dev, count * sizeof(T), s);
		if (e != cudaSuccess) {
			cudaGetLastError();
			return pgq_fail(PGQ_ERR_CUDA, "peer copy to device %d failed: %s", dst_dev, cudaGetErrorString(e));
		}
	}
	return PGQ_OK;
}

static int clone_dir(pgq_csr *dst, int dd, DirGraph &out, const DirGraph &in, int sd, int64_t n, int64_t m, cudaStream_t s) {
	out.nnz = in.nnz;
	out.nchunks = in.nchunks;
	PGQ_TRY(clone_array(dst, dd, &out.off, in.off, sd, (size_t)(n + 1), s));
	PGQ_TRY(clone_array(dst, dd, &out.adj, in.adj, sd, (size_t)std::max<int64_t>(m, 1), s));
	PGQ_TRY(clone_array(dst, dd, &out.head, in.head, sd, (size_t)std::max<int64_t>(in.nchunks, 1) * PGQ_STEPS, s));
	PGQ_TRY(clone_array(dst, dd, &out.nzrow, in.nzrow, sd, (size_t)std::max<int64_t>(in.nnz, 1), s));
	PGQ_TRY(clone_array(dst, dd, &out.chunk_rank, in.chunk_rank, sd, (size_t)std::max<int64_t>(in.nchunks, 1), s));
	return PGQ_OK;
}

extern "C" int pgq_csr_clone(pgq_csr *csr, pgq_ctx *target, pgq_csr **out) {
	if (!csr || !target || !out) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "null argument");
	}
	*out = nullptr;
	if (!csr->finalized) {
		return pgq_fail(PGQ_ERR_NOT_INITIALIZED, "%s", pgq_status_text(PGQ_ERR_NOT_INITIALIZED));
	}
	const int sd = csr->ctx->device, dd = target->device;
	PGQ_CUDA(cudaSetDevice(dd));
	if (sd != dd) {
		int can = 0;
		cudaDeviceCanAccessPeer(&can, dd, sd);
		if (can) {
			cudaError_t e = cudaDeviceEnablePeerAccess(sd, 0); // (copies also work without it, staged through the host)
			if (e != cudaSuccess) {
				cudaGetLastError();
			}
		}
	}
	pgq_csr *c = new (std::nothrow) pgq_csr();
	if (!c) {
		return pgq_fail(PGQ_ERR_OOM, "host allocation failed");
	}
	c->ctx = target;
	c->n = csr->n;
	c->m = csr->m;
	c->n_a = csr->n_a;
	c->n_ab = csr->n_ab;
	c->edge_size = csr->edge_size;
	c->staged = csr->staged;
	c->edge_init = true;
	c->weight_type = csr->weight_type;
	c->w_negative = csr->w_negative;
	Workspace *ws = nullptr;
	int st = pgq_ws_acquire(target, &ws);
	if (st != PGQ_OK) {
		delete c;
		return st;
	}
	cudaStream_t s = ws->stream;
	const int64_t n = csr->n, m = csr->m;
	do {
		if ((st = clone_dir(c, dd, c->out, csr->out, sd, n, m, s)) != PGQ_OK) break;
		if ((st = clone_dir(c, dd, c->in, csr->in, sd, n, m, s)) != PGQ_OK) break;
		{ // the bottom-up layout
			const PullGraph &g = csr->pull;
			PullGraph &o = c->pull;
			o = g; // sizes; every pointer is replaced below (nulled first: a failed clone must not free the source's arrays)
			o.adj = nullptr;
			o.head = nullptr;
			o.chunk_rank = nullptr;
			o.row = nullptr;
			o.s_adj = nullptr;
			o.s_row = nullptr;
			o.s_off = nullptr;
			if ((st = clone_array(c, dd, &o.adj, g.adj, sd, (size_t)((std::max<int64_t>(g.m, 1) + 1023) / 1024) * 1024, s)) != PGQ_OK) break;
			if ((st = clone_array(c, dd, &o.head, g.head, sd, (size_t)std::max<int64_t>(g.nchunks, 1) * PGQ_STEPS, s)) != PGQ_OK) break;
			if ((st = clone_array(c, dd, &o.chunk_rank, g.chunk_rank, sd, (size_t)std::max<int64_t>(g.nchunks, 1), s)) != PGQ_OK) break;
			if ((st = clone_array(c, dd, &o.row, g.row, sd, (size_t)std::max<int64_t>(g.n_rows, 1), s)) != PGQ_OK) break;
			if ((st = clone_array(c, dd, &o.s_adj, g.s_adj, sd, (size_t)std::max<int64_t>(g.s_total, 1), s)) != PGQ_OK) break;
			if ((st = clone_array(c, dd, &o.s_row, g.s_row, sd, (size_t)std::max<int64_t>(g.n_slices * 32, 1), s)) != PGQ_OK) break;
			if ((st = clone_array(c, dd, &o.s_off, g.s_off, sd, (size_t)(g.n_slices + 2), s)) != PGQ_OK) break;
		}
		if ((st = clone_array(c, dd, &c->edge_ids, csr->edge_ids, sd, (size_t)std::max<int64_t>(m, 1), s)) != PGQ_OK) break;
		if ((st = clone_array(c, dd, &c->perm, csr->perm, sd, (size_t)std::max<int64_t>(n, 1), s)) != PGQ_OK) break;
		if ((st = clone_array(c, dd, &c->inv, csr->inv, sd, (size_t)std::max<int64_t>(n, 1), s)) != PGQ_OK) break;
		if ((st = clone_array(c, dd, &c->w_bits, csr->w_bits, sd, (size_t)std::max<int64_t>(m, 1), s)) != PGQ_OK) break;
		cudaError_t e = cudaStreamSynchronize(s);
		if (e != cudaSuccess) {
			cudaGetLastError();
			st = pgq_fail(PGQ_ERR_CUDA, "CSR replication to device %d failed: %s", dd, cudaGetErrorString(e));
		}
	} while (0);
	pgq_ws_release(target, ws);
	if (st != PGQ_OK) {
		pgq_csr_free(c);
		return st;
	}
	static std::atomic<uint64_t> next_uid {(uint64_t)1 << 40}; // (disjoint from the ids of built CSRs)
	c->uid = next_uid++;
	c->finalized = true;
	*out = c;
	return PGQ_OK;
}

// ---- the device group -------------------------------------------------------------------------------------------
struct Worker {
	std::thread th;
	std::mutex mu;
	std::condition_variable cv;
	std::function<void()> job;
	bool has_job = false, done = false, quit = false;

	void loop() {
		std::unique_lock<std::mutex> g(mu);
		for (;;) {
			cv.wait(g, [&] { return has_job || quit; });
			if (quit) {
				return;
			}
			std::function<void()> f = std::move(job);
			has_job = false;
			g.unlock();
			f();
			g.lock();
			done = true;
			cv.notify_all();
		}
	}
	void submit(std::function<void()> f) {
		std::lock_guard<std::mutex> g(mu);
		job = std::move(f);
		has_job = true;
		done = false;
		cv.notify_all();
	}
	void wait() {
		std::unique_lock<std::mutex> g(mu);
		cv.wait(g, [&] { return done; });
	}
};

struct pgq_multi_csr {
	std::vector<int> devices;
	std::vector<pgq_ctx *> ctxs;     // [0] = the primary's context (not owned)
	std::vector<pgq_csr *> replicas; // [0] = the primary (not owned)
	std::vector<Worker *> workers;   // one per replica beyond the first (the caller's thread drives device 0)
	std::mutex call_mu;              // one multi-device call at a time per group
};

extern "C" void pgq_multi_csr_free(pgq_multi_csr *mc) {
	if (!mc) {
		return;
	}
	for (Worker *w : mc->workers) {
		{
			std::lock_guard<std::mutex> g(w->mu);
			w->quit = true;
			w->cv.notify_all();
		}
		if (w->th.joinable()) {
			w->th.join();
		}
		delete w;
	}
	for (size_t i = 1; i < mc->replicas.size(); i++) {
		pgq_csr_free(mc->replicas[i]);
	}
	for (size_t i = 1; i < mc->ctxs.size(); i++) {
		pgq_ctx_destroy(mc->ctxs[i]);
	}
	delete mc;
}

extern "C" int pgq_multi_csr_create(pgq_csr *primary, const int *devices, int n_devices, pgq_multi_csr **out) {
	if (!primary || !devices || n_devices < 1 || !out) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "null argument or empty device list");
	}
	*out = nullptr;
	if (devices[0] != primary->ctx->device) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "devices[0] must be the device the CSR lives on (%d)", primary->ctx->device);
	}
	for (int i = 0; i < n_devices; i++) {
		for (int j = 0; j < i; j++) {
			if (devices[i] == devices[j]) {
				return pgq_fail(PGQ_ERR_INVALID_ARG, "device %d listed twice", devices[i]);
			}
		}
	}
	pgq_multi_csr *mc = new (std::nothrow) pgq_multi_csr();
	if (!mc) {
		return pgq_fail(PGQ_ERR_OOM, "host allocation failed");
	}
	mc->devices.assign(devices, devices + n_devices);
	mc->ctxs.push_back(primary->ctx);
	mc->replicas.push_back(primary);
	for (int i = 1; i < n_devices; i++) {
		pgq_ctx *ctx = nullptr;
		int st = pgq_ctx_create(devices[i], &ctx);
		if (st == PGQ_OK) {
			mc->ctxs.push_back(ctx);
			pgq_csr *rep = nullptr;
			st = pgq_csr_clone(primary, ctx, &rep);
			if (st == PGQ_OK) {
				mc->replicas.push_back(rep);
			}
		}
		if (st != PGQ_OK) {
			std::string msg = pgq_last_error();
			pgq_multi_csr_free(mc);
			return pgq_fail(st, "%s", msg.c_str());
		}
		Worker *w = new Worker();
		w->th = std::thread([w]() { w->loop(); });
		mc->workers.push_back(w);
	}
	cudaSetDevice(primary->ctx->device);
	*out = mc;
	return PGQ_OK;
}

extern "C" int pgq_multi_csr_devices(pgq_multi_csr *mc, int *n_devices) {
	if (!mc || !n_devices) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "null argument");
	}
	*n_devices = (int)mc->replicas.size();
	return PGQ_OK;
}

extern "C" int pgq_multi_iterativelength(pgq_multi_csr *mc, int64_t p, const int64_t *src, const int64_t *dst,
                                         const uint8_t *src_valid, const pgq_options *opts, int64_t *out_len,
                                         uint8_t *out_valid, pgq_stats *stats /* nullable: [n_devices] */) {
	if (!mc) {
		return pgq_fail(PGQ_ERR_INVALID_ID, "%s", pgq_status_text(PGQ_ERR_INVALID_ID));
	}
	const int nd = (int)mc->replicas.size();
	if (nd == 1) {
		return pgq_iterativelength(mc->replicas[0], p, src, dst, src_valid, opts, out_len, out_valid, stats);
	}
	if (p < 0 || (p > 0 && (!src || !dst || !out_len || !out_valid))) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "null or negative argument");
	}
	if (opts && opts->shard_count > 1) {
		return pgq_fail(PGQ_ERR_INVALID_ARG, "pgq_multi_* shards the call itself: shard_index / shard_count must be 0");
	}
	std::lock_guard<std::mutex> call(mc->call_mu);
	for (int64_t i = 0; i < p; i++) { // rows nobody answers stay NULL
		out_len[i] = -1;
		out_valid[i] = 0;
	}
	std::vector<int> rcs((size_t)nd, PGQ_OK);
	std::vector<std::string> errs((size_t)nd);
	std::vector<std::vector<int64_t>> lens((size_t)nd);
	std::vector<std::vector<uint8_t>> valids((size_t)nd);
	auto run = [&](int d) {
		pgq_options o;
		memset(&o, 0, sizeof(o));
		if (opts) {
			o = *opts;
		}
		o.shard_index = d;
		o.shard_count = nd;
		std::vector<int64_t> &l = lens[(size_t)d];
		std::vector<uint8_t> &v = valids[(size_t)d];
		l.resize((size_t)std::max<int64_t>(p, 1));
		v.resize((size_t)std::max<int64_t>(p, 1));
		pgq_stats st;
		memset(&st, 0, sizeof(st));
		int rc = pgq_iterativelength(mc->replicas[(size_t)d], p, src, dst, src_valid, &o, l.data(), v.data(), &st);
		if (rc != PGQ_OK) {
			errs[(size_t)d] = pgq_last_error();
		} else {
			// the rows this device answered go straight into the caller's columns: a searched row belongs to exactly
			// one shard, and rows answered without a search (src == dst) get the same value from every device
			for (int64_t i = 0; i < p; i++) {
				if (v[(size_t)i]) {
					out_len[i] = l[(size_t)i];
					out_valid[i] = 1;
				}
			}
			if (stats) {
				stats[d] = st;
			}
		}
		rcs[(size_t)d] = rc;
	};
	for (int d = 1; d < nd; d++) {
		mc->workers[(size_t)d - 1]->submit([&run, d]() { run(d); });
	}
	run(0);
	for (int d = 1; d < nd; d++) {
		mc->workers[(size_t)d - 1]->wait();
	}
	cudaSetDevice(mc->ctxs[0]->device);
	for (int d = 0; d < nd; d++) {
		if (rcs[(size_t)d] != PGQ_OK) {
			return pgq_fail(rcs[(size_t)d], "device %d: %s", mc->devices[(size_t)d], errs[(size_t)d].c_str());
		}
	}
	return PGQ_OK;
}
