// at_runtime.cu -- host runtime behind include/aligntools_b200.h (sections A and C).
//
// A batch is sharded over the handle's devices as contiguous slices of pairs (no
// inter-GPU traffic, SURVEY.md 8e).  Each shard keeps its sequences resident in HBM,
// cuts its pairs into CHUNKS whose traceback-pointer blocks fit the pointer arena, and
// per chunk runs  fill (one launch per rows-per-lane class R)  ->  traceback count walk
// ->  exclusive scans  ->  traceback emit walk, all on one stream, timed with CUDA events.
// There is no CPU fallback anywhere in this file: without a usable sm_100 device every
// entry returns AT_E_CUDA.
#include "../../../include/aligntools_b200.h"
#include "at_kernels.cuh"
#include "at_devmem.h"

#include <cub/device/device_scan.cuh>
#include <thrust/iterator/transform_iterator.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

using namespace atb2;

// ------------------------------------------------------------------ handle ----
struct at_device {
	int id = 0;
	int sm_count = 0;
	cudaStream_t stream = nullptr;
	cudaStream_t pipe[4] = {nullptr, nullptr, nullptr, nullptr};   // at_batch_align's pipeline streams (created on first use)
	std::shared_ptr<BigCache> big = std::make_shared<BigCache>();
};

struct at_batch;
struct at_handle {
	std::vector<at_device> devs;
	std::string err;
	std::mutex mu;
	std::atomic<uint64_t> launches{0};
	// at_batch_align's pipeline: one workspace per (device, worker), kept for the life of the handle so
	// that after the first call a pipelined batch makes no CUDA allocator call at all
	std::vector<at_batch *> pipe_ws;
	std::vector<uint64_t> pipe_prefix;     // running cell counts of the batch in hand (kept: no page faults per call)
	std::mutex align_mu;
};

static void set_err(at_handle *h, const char *fmt, ...)
{
	char buf[512];
	va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
	if (h) { std::lock_guard<std::mutex> g(h->mu); h->err = buf; }
}

#define CU(h, call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { \
	set_err(h, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); return AT_E_CUDA; } } while (0)

extern "C" void at_default_params(at_params *p)
{
	if (!p) return;
	p->m = 1; p->u = -2; p->o = -5; p->e = -1; p->j = -10; p->jump = 0;   // init_opt, src/alignment.h:105-110
}

extern "C" const char *at_strerror(int rc)
{
	switch (rc) {
	case AT_OK: return "ok";
	case AT_E_ARG: return "parameter error";
	case AT_E_CUDA: return "CUDA error / no usable sm_100 device (there is no CPU fallback)";
	case AT_E_NOMEM: return "allocation failure";
	case AT_E_FITLEN: return "first sequence must be shorter than the second to do fitting alignment";
	case AT_E_NOSPACE: return "output buffer too small";
	case AT_E_RANGE: return "score range exceeds the int32 lanes";
	case AT_E_UNDEF: return "input undefined in the reference (empty record, or fit with l2 < 2)";
	default: return "unknown error";
	}
}

extern "C" const char *at_version(void) { return "aligntools-b200 0.1 (sm_100a)"; }

__global__ void at_unpack_2bit(const uint8_t *src, const uint64_t *src_off, const uint64_t *dst_off,
                               const uint32_t *len, uint32_t n_pairs, uint8_t *dst);

extern "C" int at_create(const int *devices, int n_devices, at_handle **out)
{
	if (!out) return AT_E_ARG;
	*out = nullptr;
	int count = 0;
	if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) return AT_E_CUDA;
	at_handle *h = new at_handle();
	std::vector<int> ids;
	if (!devices || n_devices <= 0) ids.push_back(0);
	else ids.assign(devices, devices + n_devices);
	for (int id : ids) {
		if (id < 0 || id >= count) { delete h; return AT_E_ARG; }
		cudaDeviceProp prop;
		if (cudaGetDeviceProperties(&prop, id) != cudaSuccess || prop.major < 10) { delete h; return AT_E_CUDA; }
		at_device d; d.id = id; d.sm_count = prop.multiProcessorCount;
		// host threads waiting for the device yield their core between polls: the pipelined path runs three
		// workers per GPU, and a multi-rank job (one process per GPU) must not starve them on a small host
		if (cudaSetDevice(id) == cudaSuccess && cudaSetDeviceFlags(cudaDeviceScheduleYield) != cudaSuccess) cudaGetLastError();
		if (cudaSetDevice(id) != cudaSuccess || cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking) != cudaSuccess) { delete h; return AT_E_CUDA; }
		cudaMemPool_t pool;
		if (cudaDeviceGetDefaultMemPool(&pool, id) == cudaSuccess) {
			uint64_t keep = UINT64_MAX;      // keep freed blocks cached in the pool (trimmed in at_destroy)
			cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
		}
		// The helper kernels ask for the same (maximal) shared-memory carve-out as the fill kernels: an
		// SM runs kernels of different carve-outs only one after the other, so without this every small
		// kernel of the pipelined path would wait for a persistent fill grid of another stream to drain.
		const void *helpers[] = {(const void *)at_traceback_walk<true>, (const void *)at_traceback_emit<true>, (const void *)at_scan_offsets,
		                         (const void *)at_symbol_set, (const void *)at_build_jmask, (const void *)at_unpack_2bit, (const void *)at_plan_uniform};
		for (const void *fn : helpers) cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
		h->devs.push_back(d);
	}
	*out = h;
	return AT_OK;
}

extern "C" void at_batch_free(at_batch *b);

extern "C" void at_destroy(at_handle *h)
{
	if (!h) return;
	for (at_batch *ws : h->pipe_ws) if (ws) at_batch_free(ws);
	h->pipe_ws.clear();
	for (auto &d : h->devs) {
		cudaSetDevice(d.id);
		if (d.stream) { cudaStreamSynchronize(d.stream); cudaStreamDestroy(d.stream); }
		for (auto &ps : d.pipe) if (ps) { cudaStreamSynchronize(ps); cudaStreamDestroy(ps); }
		d.big->drop_all();
		cudaMemPool_t pool;
		if (cudaDeviceGetDefaultMemPool(&pool, d.id) == cudaSuccess) cudaMemPoolTrimTo(pool, 0);
	}
	delete h;
}

extern "C" const char *at_last_error(const at_handle *h)
{
	if (!h) return "";
	static thread_local std::string copy;      // another thread of the handle may be rewriting h->err
	{ std::lock_guard<std::mutex> g(const_cast<at_handle *>(h)->mu); copy = h->err; }
	return copy.c_str();
}
extern "C" int at_device_count(const at_handle *h) { return h ? (int)h->devs.size() : 0; }
extern "C" uint64_t at_launch_count(const at_handle *h) { return h ? h->launches.load() : 0; }

// ------------------------------------------------------------------- batch ----
static const size_t AT_SEQ_SLACK = 1024;   // K2 stages 256-byte target tiles by TMA: the last tile may run past the last record

// A chunk of the shard's plan (at_plan.h) and its device buffers
struct Chunk : PlanChunk {
	explicit Chunk(PlanChunk &&p) : PlanChunk(std::move(p)) {}
	std::vector<DevBuf<FillJob>> d_jobs;       // [launch] K1 jobs ...
	std::vector<DevBuf<WaveTask>> d_tasks;     // ... or K2 tasks
	DevBuf<uint64_t> d_ptr_off, d_bnd_off, d_ops_off, d_cols_off, d_scratch_off;
	DevBuf<uint32_t> d_cigar; DevBuf<uint8_t> d_aln1, d_aln2;   // exact-size outputs of this chunk ...
	uint32_t *cigar = nullptr; uint8_t *aln1 = nullptr, *aln2 = nullptr;   // ... or the workspace's grow-only buffers (pipelined path); what fetch reads
	uint64_t tot_ops = 0, tot_cols = 0;
};

// Sub-slices of one device take turns (in pair order) on the host->device copy of their sequences.
struct UploadGate {
	std::mutex mu; std::condition_variable cv; uint64_t turn = 0;
	cudaEvent_t last = nullptr;      // recorded behind the previous turn's copies: the next turn's stream waits for it, not the host
	void wait_for(uint64_t k) { std::unique_lock<std::mutex> lk(mu); cv.wait(lk, [&] { return turn >= k; }); }
	void pass(uint64_t k) { std::lock_guard<std::mutex> lk(mu); if (turn < k + 1) { turn = k + 1; cv.notify_all(); } }    // idempotent
};

struct Shard {
	at_device *dev = nullptr;
	cudaStream_t stream = nullptr;      // the device's main stream, or a pipeline stream (at_batch_align)
	uint64_t p0 = 0, p1 = 0;            // pair range within the batch's input arrays
	uint64_t out_base = 0;              // index of pair p0 in the caller's output arrays
	uint32_t n = 0;
	DevBuf<uint8_t> d_q, d_t, d_jmask, d_rclass, d_end_state, d_q2, d_t2;
	DevBuf<uint64_t> d_q_off, d_t_off, d_site_off;
	DevBuf<uint32_t> d_q_len, d_t_len, d_end_i, d_end_j, d_beg_i, d_beg_j, d_n_ops, d_n_cols, d_counter;
	DevBuf<int32_t> d_score, d_sites;
	DevBuf<uint32_t> ws_cigar; DevBuf<uint8_t> ws_aln1, ws_aln2;     // pipeline workspace: outputs of the sub-slice, sized by their upper bound
	DevBuf<uint32_t> d_ptr, d_scratch, d_prog; DevBuf<uint8_t> d_bnd, d_scan_tmp; DevBuf<int32_t> d_chain;
	DevBuf<uint8_t> d_symmap; DevBuf<uint32_t> d_symset;
	bool prof = false; uint32_t syms = 0;      // query-profile variant of K1: the targets use <= 4 distinct bytes
	bool bits = false;                         // bit-parallel edit distance: `-u 1` and reads of <= 8 distinct bytes
	int bits_r = 1;                            // its 32-row blocks per lane (one launch per shard; fixes the edit-path pointer layout)
	bool twobit = false;                       // the sequences stay 2-bit packed in HBM (AT_SEQ_2BIT input consumed directly by K1 / K2 / K3)
	bool banded = false;                       // overlap / global with a per-pair band: d_band holds it clipped (at_band.h)
	DevBuf<int2> d_band;
	bool table = false;                        // substitution matrix, target alphabet of > 4 bytes: the TABLE variants of K1 / K2
	DevBuf<int8_t> d_subst;                    // substitution matrix, profile variants: the caller's 256 x 256 table
	DevBuf<int16_t> d_stab; DevBuf<uint32_t> d_qrow; DevBuf<uint16_t> d_tcol;      // ... table variants: SubstArgs
	uint32_t stab_bytes = 0;
	// what the substitution buffers above hold (a pipeline workspace keeps them from one sub-slice to the next): the matrix
	// the profile variants read, and the (scale, read set, target set, matrix) the table was built from
	std::vector<int8_t> up_matrix, up_table_matrix; std::vector<uint32_t> up_table_key;
	std::vector<uint64_t> h_t_rel;             // twobit + jump: device offsets of the packed targets (the jump masks copy their alignment)
	DevBuf<uint64_t> d_j_off;                  // twobit + jump: per-pair offsets into d_jmask (byte-encoded targets use d_t_off)
	BufCache cache;                            // released device blocks, reused by this shard's next allocations
	struct UploadGate *gate = nullptr; uint64_t gate_turn = 0;   // pipelined path: sub-slices upload their sequences one at a time, in pair order
	bool workspace = false;                    // pipeline workspace: reused for many sub-slices, buffers get head-room
	std::vector<Chunk> chunks;
	uint64_t cells = 0, ptr_bytes = 0, t_span = 0;   // t_span: bytes of d_t that hold the caller's target span
	cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
	cudaEvent_t evk[2] = {nullptr, nullptr};
	cudaEvent_t ev_up = nullptr;               // behind this shard's sequence upload (pipelined path: orders the sub-slices' copies)
	cudaEvent_t ev_sync = nullptr;             // shard_sync(): a sleeping wait for the stream
	// last-run timing
	double fill_ms = 0, tb_ms = 0, dev_ms = 0, domk_ms = 0; uint64_t domk_cells = 0, launches = 0; uint32_t domk_kind = 0, domk_r = 0, domk_flags = 0;
	int rc = AT_OK;
};

// How host threads wait for the device.  Default: spin with yields (the device's cudaDeviceScheduleYield flag) -- the lowest
// latency, and measured best even with 8 ranks x 3 pipeline workers on 32 cores (e2e C2 at N = 8: 37.0 ms spinning,
// 38.8 ms sleeping; profiles/bench_r02_n8*.json).  AT_SYNC=block makes the waits sleep on events created with
// cudaEventBlockingSync instead, for hosts where the cores are needed elsewhere.
static bool wait_blocking()
{
	static const bool v = [] { const char *e = getenv("AT_SYNC"); return e && (e[0] == 'b' || e[0] == 'B'); }();
	return v;
}
static cudaError_t event_create_timed(cudaEvent_t *e) { return cudaEventCreateWithFlags(e, wait_blocking() ? cudaEventBlockingSync : cudaEventDefault); }
static cudaError_t shard_sync(Shard &s)
{
	if (!wait_blocking()) return cudaStreamSynchronize(s.stream);
	if (!s.ev_sync) { cudaError_t e = cudaEventCreateWithFlags(&s.ev_sync, cudaEventBlockingSync | cudaEventDisableTiming); if (e != cudaSuccess) return e; }
	cudaError_t e = cudaEventRecord(s.ev_sync, s.stream);
	return e != cudaSuccess ? e : cudaEventSynchronize(s.ev_sync);
}

struct at_batch {
	at_handle *h = nullptr;
	int mode = 0; at_params prm; uint32_t out_flags = 0;
	std::vector<int8_t> subst;                 // substitution matrix (at_batch_*_scored): 256 x 256, empty = match / mismatch scoring
	uint64_t n = 0;
	bool traceback = false;
	std::vector<Shard> shards;
	bool ran = false;
};

__global__ void at_unpack_2bit(const uint8_t *src, const uint64_t *src_off, const uint64_t *dst_off,
                               const uint32_t *len, uint32_t n_pairs, uint8_t *dst)
{
	const uint32_t p = blockIdx.x;
	if (p >= n_pairs) return;
	const uint8_t *s = src + src_off[p];
	uint8_t *d = dst + dst_off[p];
	for (uint32_t k = threadIdx.x; k < len[p]; k += blockDim.x) {
		const uint32_t c = (s[k >> 2] >> (2 * (k & 3))) & 3u;
		d[k] = (uint8_t)("ACGT"[c]);
	}
}

// upload one side (reads or targets) of a shard; rewrites offsets relative to the device buffer
// `resident` (2-bit input only): the packed records stay as they are -- d_bytes receives them, d_off their byte
// offsets -- and the kernels read the codes directly; otherwise 2-bit input is expanded to bytes on the device.
static int upload_side(at_handle *h, Shard &s, uint32_t encoding, const uint8_t *src, const uint64_t *off,
                       const uint32_t *len, DevBuf<uint8_t> &d_bytes, DevBuf<uint8_t> &d_packed, DevBuf<uint64_t> &d_off,
                       DevBuf<uint32_t> &d_len, uint64_t *span_bytes, bool resident, std::vector<uint64_t> *keep_rel = nullptr)
{
	const uint32_t n = s.n;
	cudaStream_t st = s.stream;
	std::vector<uint64_t> rel(n), unp(n);
	uint64_t lo = UINT64_MAX, hi = 0, tot = 0;
	bool monotonic = true;
	for (uint32_t k = 0; k < n; ++k) {
		const uint64_t o = off[s.p0 + k];
		const uint64_t nbytes = encoding == AT_SEQ_2BIT ? ((uint64_t)len[s.p0 + k] + 3) / 4 : len[s.p0 + k];
		if (k && o < hi) monotonic = false;
		lo = std::min(lo, o); hi = std::max(hi, o + nbytes);
		unp[k] = tot; tot += len[s.p0 + k];
	}
	DevBuf<uint8_t> &raw = (encoding == AT_SEQ_2BIT && !resident) ? d_packed : d_bytes;
	if (monotonic && hi - lo <= 2 * tot + 64) {          // one bulk copy of the caller's span
		CU(h, raw.alloc(hi - lo + AT_SEQ_SLACK));
		CU(h, cudaMemcpyAsync(raw.p, src + lo, hi - lo, cudaMemcpyHostToDevice, st));
		for (uint32_t k = 0; k < n; ++k) rel[k] = off[s.p0 + k] - lo;
		*span_bytes = hi - lo;
	} else {                                             // scattered records: repack on the host first
		std::vector<uint8_t> stage;
		uint64_t pos = 0;
		for (uint32_t k = 0; k < n; ++k) {
			const uint64_t nbytes = encoding == AT_SEQ_2BIT ? ((uint64_t)len[s.p0 + k] + 3) / 4 : len[s.p0 + k];
			rel[k] = pos; stage.resize(pos + nbytes);
			memcpy(stage.data() + pos, src + off[s.p0 + k], nbytes); pos += nbytes;
		}
		CU(h, raw.alloc(pos + AT_SEQ_SLACK));
		CU(h, cudaMemcpyAsync(raw.p, stage.data(), pos, cudaMemcpyHostToDevice, st));      // pageable source: staged before the call returns
		*span_bytes = pos;
	}
	CU(h, d_off.alloc(n)); CU(h, d_len.alloc(n));
	CU(h, cudaMemcpyAsync(d_len.p, len + s.p0, n * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
	if (encoding == AT_SEQ_2BIT && !resident) {
		DevBuf<uint64_t> d_src_off;
		CU(h, d_src_off.alloc(n));
		CU(h, cudaMemcpyAsync(d_src_off.p, rel.data(), n * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
		CU(h, cudaMemcpyAsync(d_off.p, unp.data(), n * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
		CU(h, d_bytes.alloc(tot + AT_SEQ_SLACK));
		at_unpack_2bit<<<n, 128, 0, st>>>(d_packed.p, d_src_off.p, d_off.p, d_len.p, n, d_bytes.p);
		CU(h, cudaGetLastError());
		h->launches++;
		d_src_off.release();      // stream-ordered: reused only by later work of this stream
		*span_bytes = tot;
	} else {
		CU(h, cudaMemcpyAsync(d_off.p, rel.data(), n * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
		if (keep_rel) keep_rel->swap(rel);      // (the copy above has staged the pageable vector already)
	}
	// No synchronisation here: `rel` / `unp` / `stage` are pageable, so the runtime has staged them by the time
	// cudaMemcpyAsync returns; the caller's (possibly pinned) sequence buffers stay valid until setup_shard's one
	// synchronisation at its end.
	return AT_OK;
}

// give the per-chunk buffers back to the pool (stream-ordered: the same stream reuses them at once)
static void release_chunks(Shard &s)
{
	for (auto &c : s.chunks) {
		c.d_ptr_off.release(); c.d_bnd_off.release(); for (auto &d : c.d_jobs) d.release(); for (auto &d : c.d_tasks) d.release();
		c.d_ops_off.release(); c.d_cols_off.release(); c.d_scratch_off.release(); c.d_cigar.release(); c.d_aln1.release(); c.d_aln2.release();
	}
	s.chunks.clear();
}

static void free_shard(Shard &s)
{
	if (s.dev) { cudaSetDevice(s.dev->id); tl_stream = s.stream; tl_big = s.dev->big.get(); }
	tl_cache = &s.cache;
	s.d_q.release(); s.d_t.release(); s.d_jmask.release(); s.d_j_off.release(); s.d_rclass.release(); s.d_end_state.release();
	s.d_q2.release(); s.d_t2.release();
	s.d_q_off.release(); s.d_t_off.release(); s.d_site_off.release();
	s.d_q_len.release(); s.d_t_len.release(); s.d_end_i.release(); s.d_end_j.release(); s.d_beg_i.release();
	s.d_beg_j.release(); s.d_n_ops.release(); s.d_n_cols.release(); s.d_counter.release();
	s.ws_cigar.release(); s.ws_aln1.release(); s.ws_aln2.release();
	s.d_score.release(); s.d_sites.release(); s.d_ptr.release(); s.d_scratch.release(); s.d_bnd.release(); s.d_scan_tmp.release();
	s.d_prog.release(); s.d_chain.release(); s.d_symmap.release(); s.d_symset.release(); s.d_band.release();
	s.d_subst.release(); s.d_stab.release(); s.d_qrow.release(); s.d_tcol.release();
	s.up_matrix.clear(); s.up_table_matrix.clear(); s.up_table_key.clear();
	release_chunks(s);
	for (auto &e : s.ev) if (e) cudaEventDestroy(e);
	for (auto &e : s.evk) if (e) cudaEventDestroy(e);
	if (s.ev_up) cudaEventDestroy(s.ev_up);
	if (s.ev_sync) cudaEventDestroy(s.ev_sync);
	s.cache.flush(s.stream);
	tl_cache = nullptr; tl_big = nullptr;
}

extern "C" void at_batch_free(at_batch *b)
{
	if (!b) return;
	for (auto &s : b->shards) free_shard(s);
	delete b;
}

// Which bytes occur in a device buffer (at_symbol_set): 256-bit set, read back to the host.
static int scan_alphabet(at_handle *h, Shard &s, const uint8_t *d_bytes, uint64_t n_bytes, uint32_t set8[8])
{
	cudaStream_t st = s.stream;
	CU(h, s.d_symset.alloc(8));
	CU(h, cudaMemsetAsync(s.d_symset.p, 0, 8 * sizeof(uint32_t), st));
	at_symbol_set<<<(int)std::min<uint64_t>(s.dev->sm_count * 8, (n_bytes + 4095) / 4096 + 1), 256, 0, st>>>(d_bytes, n_bytes, s.d_symset.p);
	CU(h, cudaGetLastError());
	h->launches++;
	CU(h, cudaMemcpyAsync(set8, s.d_symset.p, 8 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
	CU(h, shard_sync(s));
	return AT_OK;
}

static int upload_symmap(at_handle *h, Shard &s, const uint8_t map[256])
{
	CU(h, s.d_symmap.alloc(256));
	CU(h, cudaMemcpyAsync(s.d_symmap.p, map, 256, cudaMemcpyHostToDevice, s.stream));      // `map` is pageable stack memory: staged before the call returns
	return AT_OK;
}

// Kernel variants of the shard, from the alphabets of its sequences:
//   s.prof  query-profile variant of K1 / K2 -- the TARGETS use at most 4 distinct bytes (symmap: target byte -> 0..3);
//   s.bits  bit-parallel kernel for `edit -u 1` -- the READS use at most 8 distinct bytes (symmap: read byte -> 0..7,
//           anything else -> 8).  The two are exclusive: symmap describes one side.
//   s.table substitution matrix with more than 4 target bytes: the table variants (upload_subst_table).
static int upload_subst_table(at_batch *b, Shard &s, uint64_t q_span, const uint32_t *tset);
static int choose_variants(at_batch *b, Shard &s, const at_batch_input *in, uint64_t q_span)
{
	at_handle *h = b->h;
	int rc;
	s.prof = false; s.bits = false; s.syms = 0; s.table = false;
	const bool two_bit = in->encoding == AT_SEQ_2BIT;                  // the alphabet is ACGT by construction
	uint32_t set8[8];
	uint8_t map[256];
	if (b->mode == AT_EDIT && b->prm.u == 1 && !getenv("AT_NO_BITPAR")) {
		memset(map, 8, sizeof map);
		int nsym = 0;
		if (two_bit) { map['A'] = 0; map['C'] = 1; map['G'] = 2; map['T'] = 3; nsym = 4; }
		else {
			if ((rc = scan_alphabet(h, s, s.d_q.p, q_span, set8))) return rc;
			for (int c = 0; c < 256; ++c)
				if (set8[c >> 5] >> (c & 31) & 1u) { if (nsym < 8) map[c] = (uint8_t)nsym; ++nsym; }
		}
		if (nsym >= 1 && nsym <= 8) { s.bits = true; return upload_symmap(h, s, map); }
		return AT_OK;                                                  // large read alphabet: cell-by-cell kernel, xor/min variant
	}
	const bool scored = !b->subst.empty();
	// AT_NO_PROFILE: a scored batch takes the table variants whatever its alphabet.  They read byte-encoded sequences, which
	// setup_shard guarantees: AT_NO_PROFILE also turns 2-bit residency off (2-bit input is expanded to bytes on upload).
	if (getenv("AT_NO_PROFILE")) return scored ? upload_subst_table(b, s, q_span, nullptr) : AT_OK;
	memset(map, 0, sizeof map);
	int nsym = 0; uint32_t syms = 0;
	if (two_bit) { map['C'] = 1; map['G'] = 2; map['T'] = 3; nsym = 4; syms = (uint32_t)'A' | ((uint32_t)'C' << 8) | ((uint32_t)'G' << 16) | ((uint32_t)'T' << 24); }
	else {
		// d_t holds the caller's span: every byte of it is a target byte or a gap between records (which can only add symbols)
		if ((rc = scan_alphabet(h, s, s.d_t.p, s.t_span, set8))) return rc;
		for (int c = 0; c < 256; ++c)
			if (set8[c >> 5] >> (c & 31) & 1u) { if (nsym < 4) { map[c] = (uint8_t)nsym; syms |= (uint32_t)c << (8 * nsym); } ++nsym; }
	}
	if (nsym < 1 || nsym > 4) return scored ? upload_subst_table(b, s, q_span, set8) : AT_OK;      // (2-bit input has nsym = 4: set8 is the scan's)
	for (int c = nsym; c < 4; ++c) syms |= (syms & 255u) << (8 * c);   // unused codes repeat a used symbol (they are never looked up)
	s.syms = syms; s.prof = true;
	if (scored && !(s.d_subst.p && s.up_matrix == b->subst)) {      // the profile variants build their profiles from the matrix itself
		CU(h, s.d_subst.alloc(65536));
		CU(h, cudaMemcpyAsync(s.d_subst.p, b->subst.data(), 65536, cudaMemcpyHostToDevice, s.stream));      // pageable: staged before the call returns
		s.up_matrix = b->subst;
	}
	return upload_symmap(h, s, map);
}

// Substitution matrix, target alphabet of more than 4 bytes: the shard's read and target alphabets compacted to codes (in
// byte order) and one int16 table [read code][target code] of what the kernels add per cell -- 8 s for the affine kernels, 4 s
// for overlap's -- with the byte offsets of every read byte's row and every target byte's column.  The kernels copy the table
// into shared memory (up to 128 KB for 256 x 256 symbols; a few hundred bytes for protein).  `tset`: the target alphabet when the
// caller has scanned it already (NULL: scanned here).  A shard that already holds the table of the same alphabets and matrix
// (the next sub-slice of a pipeline workspace) keeps it.
static int upload_subst_table(at_batch *b, Shard &s, uint64_t q_span, const uint32_t *tset)
{
	at_handle *h = b->h;
	int rc;
	const int scale = b->mode == AT_OVERLAP ? 4 : 8;
	std::vector<uint32_t> key(17);      // scale, read set, target set
	key[0] = (uint32_t)scale;
	if ((rc = scan_alphabet(h, s, s.d_q.p, q_span, key.data() + 1))) return rc;
	if (tset) std::copy(tset, tset + 8, key.begin() + 9);
	else if ((rc = scan_alphabet(h, s, s.d_t.p, s.t_span, key.data() + 9))) return rc;
	s.table = true;
	if (s.d_stab.p && key == s.up_table_key && b->subst == s.up_table_matrix) return AT_OK;
	const uint32_t *qset = key.data() + 1, *tst = key.data() + 9;
	std::vector<int> qb, tb;      // the bytes of each code
	for (int c = 0; c < 256; ++c) { if (qset[c >> 5] >> (c & 31) & 1u) qb.push_back(c); if (tst[c >> 5] >> (c & 31) & 1u) tb.push_back(c); }
	if (qb.empty()) qb.push_back(0);
	if (tb.empty()) tb.push_back(0);
	const size_t nq = qb.size(), nt = tb.size();
	std::vector<int16_t> tab(((nq * nt * 2 + 15) & ~(size_t)15) / 2, 0);
	for (size_t x = 0; x < nq; ++x)
		for (size_t y = 0; y < nt; ++y) tab[x * nt + y] = (int16_t)(scale * b->subst[qb[x] * 256 + tb[y]]);
	std::vector<uint32_t> qrow(256, 0);      // bytes outside the alphabet never occur: row 0
	std::vector<uint16_t> tcol(256, 0);
	for (size_t x = 0; x < nq; ++x) qrow[qb[x]] = (uint32_t)(x * nt * 2);
	for (size_t y = 0; y < nt; ++y) tcol[tb[y]] = (uint16_t)(y * 2);
	s.stab_bytes = (uint32_t)(tab.size() * 2);
	CU(h, s.d_stab.alloc(tab.size())); CU(h, s.d_qrow.alloc(256)); CU(h, s.d_tcol.alloc(256));
	cudaStream_t st = s.stream;      // pageable host vectors: each copy is staged before cudaMemcpyAsync returns
	CU(h, cudaMemcpyAsync(s.d_stab.p, tab.data(), s.stab_bytes, cudaMemcpyHostToDevice, st));
	CU(h, cudaMemcpyAsync(s.d_qrow.p, qrow.data(), 256 * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
	CU(h, cudaMemcpyAsync(s.d_tcol.p, tcol.data(), 256 * sizeof(uint16_t), cudaMemcpyHostToDevice, st));
	s.up_table_key.swap(key); s.up_table_matrix = b->subst;
	return AT_OK;
}

// max |s(a, b)| of a substitution matrix (256 x 256)
static int64_t subst_maxabs(const int8_t *mat)
{
	int64_t v = 0;
	for (int k = 0; k < 65536; ++k) v = std::max<int64_t>(v, mat[k] < 0 ? -(int64_t)mat[k] : mat[k]);
	return v;
}

// fit+jump: the per-pair blacklists as a byte mask aligned with the target bytes (at_build_jmask)
static int build_jump_mask(at_batch *b, Shard &s, const at_batch_input *in)
{
	at_handle *h = b->h;
	cudaStream_t st = s.stream;
	const uint32_t n = s.n;
	// params.jump == 2 (junction WHITELIST, the semantics of the comment at src/alignment.h:542-544): entering J is
	// barred everywhere except on the listed indices -- the mask starts as all ones and the sites clear it
	const bool whitelist = b->prm.jump == 2;
	// byte-encoded targets: the mask is indexed like the targets (same offsets, same 16-byte alignment for the TMA tiles of
	// K2).  2-bit resident targets: one mask byte per SYMBOL, each pair's mask placed so that it has the alignment K2's
	// ring gives the expanded target -- 4 x (packed address mod 16) past a 16-byte boundary.
	uint64_t mask_bytes = s.d_t.n;
	if (s.twobit) {
		std::vector<uint64_t> jo(n);
		uint64_t cur = 0;
		for (uint32_t k = 0; k < n; ++k) {
			jo[k] = cur + 4 * (((uintptr_t)s.d_t.p + s.h_t_rel[k]) & 15u);
			cur = (jo[k] + in->t_len[s.p0 + k] + 15u) & ~(uint64_t)15u;
		}
		mask_bytes = cur + AT_SEQ_SLACK;
		CU(h, s.d_j_off.alloc(n));
		CU(h, cudaMemcpyAsync(s.d_j_off.p, jo.data(), n * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
	}
	const uint64_t *d_j_off = s.twobit ? s.d_j_off.p : s.d_t_off.p;
	CU(h, s.d_jmask.alloc(mask_bytes));
	CU(h, cudaMemsetAsync(s.d_jmask.p, whitelist ? 1 : 0, mask_bytes, st));
	if (!in->sites || !in->site_off) return AT_OK;
	const uint64_t lo = in->site_off[s.p0], hi = in->site_off[s.p1];
	std::vector<uint64_t> so(n + 1);
	for (uint32_t k = 0; k <= n; ++k) so[k] = in->site_off[s.p0 + k] - lo;
	CU(h, s.d_sites.alloc(hi - lo + 1)); CU(h, s.d_site_off.alloc(n + 1));
	if (hi > lo) CU(h, cudaMemcpyAsync(s.d_sites.p, in->sites + lo, (hi - lo) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
	CU(h, cudaMemcpyAsync(s.d_site_off.p, so.data(), (n + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
	at_build_jmask<<<n, 64, 0, st>>>(s.d_sites.p, s.d_site_off.p, d_j_off, s.d_t_len.p, n, s.d_jmask.p, whitelist ? 0 : 1);
	CU(h, cudaGetLastError());
	h->launches++;
	return AT_OK;
}


// AT_WAVE_START_LAG (columns, default 0): a K2 stripe starts only once the stripe above it is this far ahead (A/B knob)
static uint32_t wave_start_lag() { static const uint32_t v = [] { const char *e = getenv("AT_WAVE_START_LAG"); return e && *e ? (uint32_t)strtoul(e, nullptr, 10) : 0u; }(); return v; }

// `band` (NULL: unbanded): the caller's band arrays, indexed like `in` (band->lo[s.p0 + k] is the shard's pair k)
static int setup_shard(at_batch *b, Shard &s, const at_batch_input *in, const at_band *band)
{
	at_handle *h = b->h;
	CU(h, cudaSetDevice(s.dev->id));
	cudaStream_t st = s.stream;
	tl_stream = st;
	tl_cache = &s.cache; tl_big = s.dev->big.get();
	const uint32_t n = s.n;
	int rc;
	// AT_PIPE_TRACE=2: host timeline of this function's phases (ms since entry) on stderr
	static const bool trace_setup = getenv("AT_PIPE_TRACE") && atoi(getenv("AT_PIPE_TRACE")) >= 2;
	const auto t_enter = std::chrono::steady_clock::now();
	std::string tl_;
	auto mark = [&](const char *what) {
		if (!trace_setup) return;
		char buf[64];
		snprintf(buf, sizeof buf, " %s %.2f", what, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_enter).count());
		tl_ += buf;
	};
	uint64_t q_span = 0;
	{
		// a pipeline worker waits for the uploads of the sub-slices before its own: the first (small) sub-slice's
		// sequences are not held up behind a later, larger one sharing the copy engine, and its fill starts early
		// 2-bit input stays packed in HBM: K1 reads the codes with 128-bit / byte loads (the code IS the query-profile
		// index), K2 stages 64-byte tiles by TMA and expands them into its shared-memory ring once per 256 columns, the
		// traceback decodes them; no expansion kernel, a quarter of the sequence bytes in HBM and over PCIe.  (The alphabet
		// is ACGT by construction, so the query-profile variants always apply; AT_NO_PROFILE falls back to expanding.)
		s.twobit = in->encoding == AT_SEQ_2BIT && !getenv("AT_NO_PROFILE") && !getenv("AT_NO_2BIT_RESIDENT");
		if (s.gate) {
			s.gate->wait_for(s.gate_turn);
			if (s.gate->last) CU(h, cudaStreamWaitEvent(st, s.gate->last, 0));      // copy engine: earlier sub-slices first
		}
		rc = upload_side(h, s, in->encoding, in->q, in->q_off, in->q_len, s.d_q, s.d_q2, s.d_q_off, s.d_q_len, &q_span, s.twobit);
		if (!rc) rc = upload_side(h, s, in->encoding, in->t, in->t_off, in->t_len, s.d_t, s.d_t2, s.d_t_off, s.d_t_len, &s.t_span, s.twobit,
		                          s.twobit && b->mode == AT_FIT && b->prm.jump ? &s.h_t_rel : nullptr);
		if (!s.ev_up) CU(h, cudaEventCreateWithFlags(&s.ev_up, cudaEventDisableTiming | (wait_blocking() ? cudaEventBlockingSync : 0)));
		if (!rc) CU(h, cudaEventRecord(s.ev_up, st));      // behind the sequence copies: what must complete before the caller's buffers are free
		if (s.gate) {
			if (!rc) s.gate->last = s.ev_up;
			s.gate->pass(s.gate_turn);
		}
		if (rc) return rc;
	}
	s.d_q2.release(); s.d_t2.release();
	mark("upload");
	const bool jump = b->mode == AT_FIT && b->prm.jump;
	s.banded = band != nullptr;
	std::vector<PairBand> bands;
	if (s.banded) {
		bands.resize(n);
		for (uint32_t k = 0; k < n; ++k) band_clip(in->q_len[s.p0 + k], in->t_len[s.p0 + k], band->lo[s.p0 + k], band->hi[s.p0 + k], bands[k].lo, bands[k].hi);
		CU(h, s.d_band.alloc(n));
		CU(h, cudaMemcpyAsync(s.d_band.p, bands.data(), n * sizeof(int2), cudaMemcpyHostToDevice, st));      // staged before the set-up's synchronisation
	}
	if ((rc = choose_variants(b, s, in, q_span))) return rc;
	if (jump && (rc = build_jump_mask(b, s, in))) return rc;
	s.bits_r = s.bits ? (int)choose_bits_r(in->q_len + s.p0, n, (uint64_t)s.dev->sm_count * 8 * AT_WAVE_WARPS) : 1;
	mark("alphabet+jmask");
	PlanIn pin;
	pin.n = n; pin.l1 = in->q_len + s.p0; pin.l2 = in->t_len + s.p0;
	pin.mode = b->mode; pin.traceback = b->traceback; pin.jump = jump;
	pin.band = s.banded ? bands.data() : nullptr;
	pin.bits = s.bits; pin.bits_r = (uint32_t)s.bits_r;
	// substitution matrix: packed lanes only with the profile variant (the table variant runs on int32 lanes)
	if (b->subst.empty()) pin.p16 = p16_rule(b->mode, b->prm, jump, getenv("AT_NO_P16") != nullptr);
	else if (s.prof) pin.p16 = p16_rule(b->mode, b->prm, jump, getenv("AT_NO_P16") != nullptr, subst_maxabs(b->subst.data()));
	pin.allow_uniform = !getenv("AT_NO_UNIFORM_PLAN");
	static const bool pair_major = [] { const char *e = getenv("AT_WAVE_ORDER"); return e && !strcmp(e, "pair"); }();
	pin.pair_major = pair_major;
	// ---- pointer-arena budget ----
	// The whole shard's pointer blocks in one chunk if they fit the arena this shard already owns (a
	// pipeline workspace after its first sub-slice); otherwise ask the driver what is free.
	// cudaMemGetInfo is kept off the steady-state path: with other threads driving the device it was
	// seen to block for tens of milliseconds.
	const uint64_t need = need_words(pin);
	size_t free_b = 0, total_b = 0;
	const bool owned = need <= s.d_ptr.n && !getenv("AT_PTR_BUDGET_MB");
	if (!owned && need) {
		CU(h, cudaMemGetInfo(&free_b, &total_b));
		// blocks cached in the stream-ordered pool are reusable by this batch: count them as free
		cudaMemPool_t pool; uint64_t reserved = 0, used = 0;
		if (cudaDeviceGetDefaultMemPool(&pool, s.dev->id) == cudaSuccess &&
		    cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &reserved) == cudaSuccess &&
		    cudaMemPoolGetAttribute(pool, cudaMemPoolAttrUsedMemCurrent, &used) == cudaSuccess && reserved > used)
			free_b += (size_t)(reserved - used);
		free_b += s.d_ptr.bytes;      // the arena this shard holds is re-sized, not added to
		free_b += s.dev->big->cached_bytes();      // arena-sized blocks cached in the handle are dropped on demand
	}
	pin.budget_words = owned ? std::max<uint64_t>(s.d_ptr.n, 1) : (uint64_t)(free_b * 0.45) / 4;
	if (!need) pin.budget_words = UINT64_MAX;
	if (const char *env = getenv("AT_PTR_BUDGET_MB")) pin.budget_words = (uint64_t)atoll(env) * (1ull << 20) / 4;
	mark("meminfo");
	Plan plan = make_plan(pin);
	if (plan.fail_pair != UINT32_MAX) {
		set_err(h, "pair %llu needs %llu MB of traceback pointers; arena budget is %llu MB", (unsigned long long)(s.p0 + plan.fail_pair),
		        (unsigned long long)(plan.fail_words >> 18), (unsigned long long)(pin.budget_words >> 18));
		return AT_E_NOMEM;
	}
	mark("plan");
	// ---- device buffers: results, then what the plan says ----
	CU(h, s.d_score.alloc(n)); CU(h, s.d_end_i.alloc(n)); CU(h, s.d_end_j.alloc(n)); CU(h, s.d_end_state.alloc(n));
	CU(h, s.d_beg_i.alloc(n)); CU(h, s.d_beg_j.alloc(n)); CU(h, s.d_n_ops.alloc(n + 1)); CU(h, s.d_n_cols.alloc(n + 1));
	CU(h, cudaMemsetAsync(s.d_n_ops.p, 0, (n + 1) * sizeof(uint32_t), st));
	CU(h, cudaMemsetAsync(s.d_n_cols.p, 0, (n + 1) * sizeof(uint32_t), st));
	CU(h, cudaMemsetAsync(s.d_beg_i.p, 0, n * sizeof(uint32_t), st));
	CU(h, cudaMemsetAsync(s.d_beg_j.p, 0, n * sizeof(uint32_t), st));
	CU(h, s.d_counter.alloc(64));
	CU(h, s.d_rclass.alloc(n));
	release_chunks(s);      // a pipeline worker reuses its shard (and the shard-level buffers) for every sub-slice
	s.cells = plan.cells; s.ptr_bytes = 0;
	// pageable host vectors: each copy is staged before cudaMemcpyAsync returns
	auto upload = [&](auto &d, const auto &v) -> cudaError_t { return v.empty() ? cudaSuccess : cudaMemcpyAsync(d.p, v.data(), v.size() * sizeof(v[0]), cudaMemcpyHostToDevice, st); };
	for (PlanChunk &pc : plan.chunks) {
		s.chunks.emplace_back(std::move(pc));
		Chunk &c = s.chunks.back();
		const uint32_t nc = c.k1 - c.k0;
		c.d_jobs.resize(c.launches.size()); c.d_tasks.resize(c.launches.size());
		for (size_t li = 0; li < c.launches.size(); ++li) {
			const PlanLaunch &l = c.launches[li];
			if (l.kind >= LK_WAVE) { CU(h, c.d_tasks[li].alloc(l.n)); CU(h, upload(c.d_tasks[li], l.tasks)); }
			else { CU(h, c.d_jobs[li].alloc(l.n)); CU(h, upload(c.d_jobs[li], l.jobs)); }
		}
		CU(h, c.d_ptr_off.alloc(nc)); CU(h, upload(c.d_ptr_off, c.ptr_off));
		CU(h, c.d_bnd_off.alloc(nc)); CU(h, upload(c.d_bnd_off, c.bnd_off));
		if (b->traceback) {
			CU(h, c.d_ops_off.alloc(nc + 1)); CU(h, c.d_cols_off.alloc(nc + 1));
			CU(h, c.d_scratch_off.alloc(nc)); CU(h, upload(c.d_scratch_off, c.scratch_off));
		}
		s.ptr_bytes += c.ptr_words * 4;
	}
	if (plan.uniform) {
		// on this stream, behind the uploads; the host does not wait for it (it may sit behind another sub-slice's fill)
		Chunk &c = s.chunks[0];
		at_plan_uniform<<<(n + 255) / 256, 256, 0, st>>>(n, plan.u, c.d_jobs[0].p, c.d_ptr_off.p, c.d_bnd_off.p, b->traceback ? c.d_scratch_off.p : nullptr, s.d_rclass.p);
		CU(h, cudaGetLastError());
		h->launches++;
	} else CU(h, upload(s.d_rclass, plan.rclass));
	mark("jobs");
	const bool linear = b->mode >= AT_OVERLAP;      // the single-plane kernels' boundary slabs hold 8-byte elements
	if (plan.max_bnd_elems && s.d_bnd.alloc(plan.max_bnd_elems * (linear ? sizeof(uint64_t) : sizeof(int4)) + 64) != cudaSuccess) { set_err(h, "stripe boundary slabs of %llu MB", (unsigned long long)((plan.max_bnd_elems * (linear ? 8 : 16)) >> 20)); return AT_E_NOMEM; }
	if (!plan.max_bnd_elems) CU(h, s.d_bnd.alloc(64));
	CU(h, s.d_prog.alloc(plan.max_prog_words + 1));
	CU(h, s.d_chain.alloc(4ull * plan.max_pairs + 4));
	if (plan.max_scratch_words && s.d_scratch.alloc(plan.max_scratch_words) != cudaSuccess) { set_err(h, "traceback scratch of %llu MB", (unsigned long long)(plan.max_scratch_words >> 18)); return AT_E_NOMEM; }
	if (plan.max_chunk_words) {
		cudaError_t e = s.d_ptr.alloc(plan.max_chunk_words + (s.workspace && plan.max_chunk_words > s.d_ptr.n ? plan.max_chunk_words / 16 : 0));
		if (e != cudaSuccess) { set_err(h, "pointer arena of %llu MB: %s", (unsigned long long)(plan.max_chunk_words >> 18), cudaGetErrorString(e)); return AT_E_NOMEM; }
	}
	for (auto &e : s.ev) if (!e) CU(h, event_create_timed(&e));
	for (auto &e : s.evk) if (!e) CU(h, event_create_timed(&e));
	mark("arena");
	// the ONE synchronisation of the set-up: every upload has left the caller's buffers (they may be reused or freed once
	// at_batch_create / the sub-slice's set-up returns) and the plan's host vectors.  A uniform plan uploads nothing from
	// the host: the sequence copies are all it waits for, not the plan kernel (which may be queued behind another fill).
	CU(h, plan.uniform ? cudaEventSynchronize(s.ev_up) : shard_sync(s));
	mark("sync");
	if (trace_setup) fprintf(stderr, "[at setup] pairs %u:%s\n", n, tl_.c_str());
	return AT_OK;
}

// argument checks shared by at_batch_create and the pipelined at_batch_align; mirrors the reference's own failure modes
// `prefix` (optional): receives the running cell counts, prefix[k] = sum of l1*l2 over pairs < k (n_pairs + 1 entries),
// so that the one-shot path validates, counts and slices a million-pair batch in one pass
// `wave_tasks` (optional): number of K2 tasks -- (pair, stripe of 256 rows) -- the batch will run as, 0 for pairs that go to K1:
// the one-shot path sizes its sub-slices so that each still fills the GPU several times over
// `sc` (optional): a substitution matrix, whose largest entry stands for m and u in the score-range bound
static int validate_batch(at_handle *h, int mode, const at_params *p, const at_batch_input *in, std::vector<uint64_t> *prefix = nullptr,
                          uint64_t *wave_tasks = nullptr, const at_scoring *sc = nullptr)
{
	if (mode < AT_GLOBAL || mode > AT_EDIT) { set_err(h, "bad mode %d", mode); return AT_E_ARG; }
	if (!in->n_pairs || !in->q || !in->q_off || !in->q_len || !in->t || !in->t_off || !in->t_len) { set_err(h, "align: parameter error"); return AT_E_ARG; }
	if (in->encoding != AT_SEQ_BYTES && in->encoding != AT_SEQ_2BIT) return AT_E_ARG;
	if ((in->sites == nullptr) != (in->site_off == nullptr)) return AT_E_ARG;
	if (in->n_pairs >= (1ull << 31)) return AT_E_ARG;
	if (in->site_off) {      // per-pair slices of `sites`: ascending offsets (build_jump_mask indexes with their differences)
		for (uint64_t k = 0; k < in->n_pairs; ++k)
			if (in->site_off[k + 1] < in->site_off[k] || in->site_off[k + 1] - in->site_off[0] > (1ull << 40)) { set_err(h, "site_off is not ascending at pair %llu", (unsigned long long)k); return AT_E_ARG; }
	}
	int64_t maxabs = std::max<int64_t>({llabs((long long)p->m), llabs((long long)p->u), llabs((long long)p->o), llabs((long long)p->e), llabs((long long)p->j), 1});
	if (sc) maxabs = std::max<int64_t>({subst_maxabs(sc->matrix), llabs((long long)p->o), llabs((long long)p->e), llabs((long long)p->j), 1});
	// Score lanes hold values x8.  With B = 8 (l1 + l2 + 2) maxabs bounding every finite value, a -inf stand-in
	// (AT_NEG = -2^29, at_kernels.cuh) that has drifted by up to B must still lose against every finite value:
	// AT_NEG + B < -B  <=>  (l1 + l2 + 2) * maxabs < 2^25.  (AT_NEG_INIT - B stays above INT32_MIN with room to spare.)
	const uint64_t max_sum = (uint64_t)(((1ll << 25) - 1) / maxabs);
	uint64_t *pre = nullptr;
	if (prefix) { prefix->resize(in->n_pairs + 1); pre = prefix->data(); pre[0] = 0; }
	// one pair's checks, in the reference's order of failure; `report` false = only say whether it fails
	auto check = [&](uint64_t k, uint64_t l1, uint64_t l2, bool report) -> int {
		if (l1 == 0 || l2 == 0) { if (report) set_err(h, "pair %llu: empty record", (unsigned long long)k); return AT_E_UNDEF; }
		if (mode == AT_FIT && l1 > l2) { if (report) set_err(h, "pair %llu: first sequence must be shorter than the second to do fitting alignment", (unsigned long long)k); return AT_E_FITLEN; }
		if (mode == AT_FIT && l2 < 2) { if (report) set_err(h, "pair %llu: fit with l2 < 2 is undefined in the reference", (unsigned long long)k); return AT_E_UNDEF; }
		/* + 40: K1's lanes run up to 34 columns past l2 (their cells obey the same bounds) */
		if (l1 + l2 + 42 > max_sum) { if (report) set_err(h, "pair %llu: score range", (unsigned long long)k); return AT_E_RANGE; }
		return AT_OK;
	};
	// ranges of pairs: checks and the range's cell total in one pass (a few host threads on a large batch),
	// the running cell counts in a second pass once every range knows its base
	const uint64_t n = in->n_pairs;
	const size_t parts = n >= (1u << 17) ? 4 : 1;
	std::vector<uint64_t> lo(parts + 1), sum(parts, 0), bad(parts, UINT64_MAX), tasks(parts, 0);
	const bool all_wave = mode >= AT_OVERLAP;
	for (size_t r = 0; r <= parts; ++r) lo[r] = n * r / parts;
	auto pass1 = [&](size_t r) {
		uint64_t acc = 0, tk = 0;
		for (uint64_t k = lo[r]; k < lo[r + 1]; ++k) {
			const uint64_t l1 = in->q_len[k], l2 = in->t_len[k];
			if (check(k, l1, l2, false)) { bad[r] = k; break; }
			acc += l1 * l2;
			if (all_wave || l1 > 32u * MAXR) tk += (l1 + 32u * MAXR - 1) / (32u * MAXR);
		}
		sum[r] = acc; tasks[r] = tk;
	};
	auto pass2 = [&](size_t r, uint64_t acc) {
		for (uint64_t k = lo[r]; k < lo[r + 1]; ++k) { acc += (uint64_t)in->q_len[k] * in->t_len[k]; pre[k + 1] = acc; }
	};
	auto each_range = [&](const std::function<void(size_t)> &fn) {
		if (parts == 1) { fn(0); return; }
		std::vector<std::thread> th;
		for (size_t r = 1; r < parts; ++r) th.emplace_back(fn, r);
		fn(0);
		for (auto &t : th) t.join();
	};
	each_range(pass1);
	for (size_t r = 0; r < parts; ++r)
		if (bad[r] != UINT64_MAX) return check(bad[r], in->q_len[bad[r]], in->t_len[bad[r]], true);   // the first failing pair, as a serial scan would report
	if (wave_tasks) { *wave_tasks = 0; for (size_t r = 0; r < parts; ++r) *wave_tasks += tasks[r]; }
	if (pre) {
		std::vector<uint64_t> base(parts, 0);
		for (size_t r = 1; r < parts; ++r) base[r] = base[r - 1] + sum[r - 1];
		each_range([&](size_t r) { pass2(r, base[r]); });
	}
	return AT_OK;
}

extern "C" int at_plan_slices(const uint32_t *q_len, const uint32_t *t_len, uint64_t n_pairs, uint32_t parts, uint64_t *cut)
{
	if (!q_len || !t_len || !cut || parts == 0) return AT_E_ARG;
	std::vector<uint64_t> prefix(n_pairs + 1, 0), c;
	for (uint64_t k = 0; k < n_pairs; ++k) prefix[k + 1] = prefix[k] + (uint64_t)q_len[k] * t_len[k];
	cut_by_prefix(prefix, 0, n_pairs, parts, c);
	for (uint32_t k = 0; k <= parts; ++k) cut[k] = c[k];
	return AT_OK;
}

// whether a run walks the pointers: any output beyond the score; edit only when the path is asked for as well
// (AT_OUT_EDIT_PATH: without it edit stays score-only, whatever else the flags say)
static bool wants_traceback(int mode, uint32_t out_flags)
{
	if (!(out_flags & (AT_OUT_CIGAR | AT_OUT_ALN))) return false;
	return mode != AT_EDIT || (out_flags & AT_OUT_EDIT_PATH);
}

static at_batch *new_batch(at_handle *h, int mode, const at_params *p, uint32_t out_flags, uint64_t n, const at_scoring *sc = nullptr)
{
	at_batch *b = new at_batch();
	b->h = h; b->mode = mode; b->prm = *p; b->out_flags = out_flags; b->n = n;
	b->traceback = wants_traceback(mode, out_flags);
	if (sc) b->subst.assign(sc->matrix, sc->matrix + 65536);
	return b;
}

// a substitution matrix is for global, local, fit and overlap, and must be there
static int validate_scoring(at_handle *h, int mode, const at_scoring *sc)
{
	if (!sc) return AT_OK;
	if (mode == AT_EDIT) { set_err(h, "scoring: edit distance takes no substitution matrix"); return AT_E_ARG; }
	if (!sc->matrix) { set_err(h, "scoring: matrix is NULL"); return AT_E_ARG; }
	return AT_OK;
}

// a band is for AT_OVERLAP and AT_GLOBAL, with both arrays and lo[p] <= hi[p] for every pair; a global pair's band must
// hold its end diagonal l2 - l1 (then every in-band cell is finite and a banded global result always exists)
static int validate_band(at_handle *h, int mode, const at_batch_input *in, const at_band *band)
{
	if (!band) return AT_OK;
	if (mode != AT_OVERLAP && mode != AT_GLOBAL) { set_err(h, "band: only overlap alignment takes a band (mode %d)", mode); return AT_E_ARG; }
	if (!band->lo || !band->hi) { set_err(h, "band: %s is NULL", band->lo ? "hi" : "lo"); return AT_E_ARG; }
	for (uint64_t k = 0; k < in->n_pairs; ++k) {
		if (band->lo[k] > band->hi[k]) { set_err(h, "band: lo > hi at pair %llu (%d > %d)", (unsigned long long)k, band->lo[k], band->hi[k]); return AT_E_ARG; }
		const int64_t d = (int64_t)in->t_len[k] - (int64_t)in->q_len[k];
		if (mode == AT_GLOBAL && (d < band->lo[k] || d > band->hi[k])) {
			set_err(h, "band: pair %llu: global alignment's end diagonal l2 - l1 = %lld lies outside the band [%d, %d]",
			        (unsigned long long)k, (long long)d, band->lo[k], band->hi[k]);
			return AT_E_ARG;
		}
	}
	return AT_OK;
}

// K2 tasks of a banded global batch: every pair runs on K2, one task per queued stripe of 256 rows (at_plan.h)
static uint64_t banded_global_tasks(const at_batch_input *in, const at_band *band)
{
	uint64_t n = 0;
	for (uint64_t k = 0; k < in->n_pairs; ++k) {
		const uint32_t l1 = in->q_len[k], l2 = in->t_len[k], RPP = 32u * MAXR;
		PairBand bd;
		band_clip(l1, l2, band->lo[k], band->hi[k], bd.lo, bd.hi);
		for (uint32_t s = 0; s < (l1 + RPP - 1) / RPP; ++s) n += band_stripe_queued(l1, l2, bd, RPP, s);
	}
	return n;
}

extern "C" int at_batch_create(at_handle *h, int mode, const at_params *p, const at_batch_input *in,
                               uint32_t out_flags, at_batch **out)
{
	return at_batch_create_banded(h, mode, p, in, nullptr, out_flags, out);
}

static int create_batch(at_handle *h, int mode, const at_params *p, const at_batch_input *in, const at_band *band, const at_scoring *sc,
                        uint32_t out_flags, at_batch **out);

extern "C" int at_batch_create_banded(at_handle *h, int mode, const at_params *p, const at_batch_input *in,
                                      const at_band *band, uint32_t out_flags, at_batch **out)
{
	return create_batch(h, mode, p, in, band, nullptr, out_flags, out);
}

extern "C" int at_batch_create_scored(at_handle *h, int mode, const at_params *p, const at_batch_input *in,
                                      const at_scoring *sc, uint32_t out_flags, at_batch **out)
{
	if (!h || !p || !in || !out) return AT_E_ARG;
	*out = nullptr;
	if (int rc = validate_scoring(h, mode, sc)) return rc;
	return create_batch(h, mode, p, in, nullptr, sc, out_flags, out);
}

// `band` / `sc` (NULL: none): at most one of the two is given
static int create_batch(at_handle *h, int mode, const at_params *p, const at_batch_input *in, const at_band *band, const at_scoring *sc,
                        uint32_t out_flags, at_batch **out)
{
	if (!h || !p || !in || !out) return AT_E_ARG;
	*out = nullptr;
	// contiguous slices balanced by cells (one device: no running cell counts needed)
	const size_t nd = h->devs.size();
	std::vector<uint64_t> prefix, cut;
	if (int rc = validate_batch(h, mode, p, in, nd > 1 ? &prefix : nullptr, nullptr, sc)) return rc;
	if (int rc = validate_band(h, mode, in, band)) return rc;
	at_batch *b = new_batch(h, mode, p, out_flags, in->n_pairs, sc);
	cut_by_prefix(prefix, 0, b->n, nd, cut);
	b->shards.resize(nd);
	std::vector<std::thread> th;
	for (size_t d = 0; d < nd; ++d) {
		Shard &s = b->shards[d];
		s.dev = &h->devs[d]; s.stream = s.dev->stream; s.p0 = cut[d]; s.p1 = cut[d + 1]; s.out_base = s.p0; s.n = (uint32_t)(s.p1 - s.p0);
	}
	auto work = [&](size_t d) { Shard &s = b->shards[d]; s.rc = s.n ? setup_shard(b, s, in, band) : AT_OK; };
	if (nd == 1) work(0);
	else { for (size_t d = 0; d < nd; ++d) th.emplace_back(work, d); for (auto &t : th) t.join(); }
	for (auto &s : b->shards) if (s.rc) { int rc = s.rc; at_batch_free(b); return rc; }
	*out = b;
	return AT_OK;
}

// ------------------------------------------------------------------ launch ----
// Kernel tables.  K1 (at_fill_affine): mode variant x rows-per-lane x lanes; kind: 0 global, 1 local,
// 2 fit, 3 fit+jump on int32 lanes, 4 / 5 / 6 local / global / fit on packed s16x2 lanes.  K2 (at_wave_*): affine modes
// with R = 8, single-plane modes (overlap / edit) with R = 1..8.
typedef void (*fill2_fn)(const FillArgs2);
typedef void (*wave_fn)(const WaveArgs);

// SCORED: substitution-matrix scoring (the table variant, !PROF, has no packed kinds: p16 is off for it)
template <int R, bool PROF, bool SCORED = false> static fill2_fn affine_fn(int kind)
{
	constexpr bool PK = !SCORED || PROF;      // packed kinds exist
	switch (kind) {
	case 0: return at_fill_affine<MODE_GLOBAL, R, false, false, PROF, SCORED>;
	case 1: return at_fill_affine<MODE_LOCAL, R, false, false, PROF, SCORED>;
	case 2: return at_fill_affine<MODE_FIT, R, false, false, PROF, SCORED>;
	case 3: return at_fill_affine<MODE_FIT, R, true, false, PROF, SCORED>;
	case 4: return at_fill_affine<MODE_LOCAL, R, false, PK, PROF, SCORED>;
	case 5: return at_fill_affine<MODE_GLOBAL, R, false, PK, PROF, SCORED>;
	default: return at_fill_affine<MODE_FIT, R, false, PK, PROF, SCORED>;
	}
}
template <bool PROF, bool SCORED = false> static fill2_fn affine_kernel_r(int kind, int R)
{
	switch (R) {
	case 1: return affine_fn<1, PROF, SCORED>(kind); case 2: return affine_fn<2, PROF, SCORED>(kind); case 3: return affine_fn<3, PROF, SCORED>(kind);
	case 4: return affine_fn<4, PROF, SCORED>(kind); case 5: return affine_fn<5, PROF, SCORED>(kind); case 6: return affine_fn<6, PROF, SCORED>(kind);
	case 7: return affine_fn<7, PROF, SCORED>(kind); default: return affine_fn<8, PROF, SCORED>(kind);
	}
}
static fill2_fn affine_kernel(int kind, int R, bool prof, bool scored)
{
	if (scored) return prof ? affine_kernel_r<true, true>(kind, R) : affine_kernel_r<false, true>(kind, R);
	return prof ? affine_kernel_r<true>(kind, R) : affine_kernel_r<false>(kind, R);
}
template <int MODE, bool PROF, bool BANDED = false, bool PTR = false, bool SCORED = false> static wave_fn wave_linear_fn(int R)
{
	switch (R) {
	case 1: return at_wave_linear<MODE, 1, PROF, BANDED, PTR, SCORED>; case 2: return at_wave_linear<MODE, 2, PROF, BANDED, PTR, SCORED>; case 3: return at_wave_linear<MODE, 3, PROF, BANDED, PTR, SCORED>;
	case 4: return at_wave_linear<MODE, 4, PROF, BANDED, PTR, SCORED>; case 5: return at_wave_linear<MODE, 5, PROF, BANDED, PTR, SCORED>; case 6: return at_wave_linear<MODE, 6, PROF, BANDED, PTR, SCORED>;
	case 7: return at_wave_linear<MODE, 7, PROF, BANDED, PTR, SCORED>; default: return at_wave_linear<MODE, 8, PROF, BANDED, PTR, SCORED>;
	}
}
// banded overlap / global (validate_band admits a band with AT_OVERLAP and AT_GLOBAL only)
static wave_fn wave_banded_kernel(int mode, int R, bool prof)
{
	if (mode == AT_GLOBAL) return prof ? at_wave_affine<MODE_GLOBAL, false, true, true> : at_wave_affine<MODE_GLOBAL, false, false, true>;
	return prof ? wave_linear_fn<MODE_OVERLAP, true, true>(R) : wave_linear_fn<MODE_OVERLAP, false, true>(R);
}
// edit paths (AT_OUT_EDIT_PATH): the PTR instantiations, which also store the pointers
static wave_fn bits_kernel(int R, bool path)
{
	if (path) return R == 1 ? at_wave_edit_bits<1, true> : (R == 2 ? at_wave_edit_bits<2, true> : at_wave_edit_bits<4, true>);
	return R == 1 ? at_wave_edit_bits<1> : (R == 2 ? at_wave_edit_bits<2> : at_wave_edit_bits<4>);
}
static wave_fn wave_kernel(int mode, bool jump, int R, bool prof, bool path)
{
	if (mode == AT_EDIT && path) return prof ? wave_linear_fn<MODE_EDIT, true, false, true>(R) : wave_linear_fn<MODE_EDIT, false, false, true>(R);
	switch (mode) {
	case AT_GLOBAL: return prof ? at_wave_affine<MODE_GLOBAL, false, true> : at_wave_affine<MODE_GLOBAL, false, false>;
	case AT_LOCAL: return prof ? at_wave_affine<MODE_LOCAL, false, true> : at_wave_affine<MODE_LOCAL, false, false>;
	case AT_FIT: return jump ? (prof ? at_wave_affine<MODE_FIT, true, true> : at_wave_affine<MODE_FIT, true, false>)
	                         : (prof ? at_wave_affine<MODE_FIT, false, true> : at_wave_affine<MODE_FIT, false, false>);
	case AT_OVERLAP: return prof ? wave_linear_fn<MODE_OVERLAP, true>(R) : wave_linear_fn<MODE_OVERLAP, false>(R);
	default: return prof ? wave_linear_fn<MODE_EDIT, true>(R) : wave_linear_fn<MODE_EDIT, false>(R);
	}
}

// substitution-matrix scoring (global, local, fit, overlap; validate_scoring): the SCORED instantiations
static wave_fn wave_scored_kernel(int mode, bool jump, int R, bool prof)
{
	switch (mode) {
	case AT_GLOBAL: return prof ? at_wave_affine<MODE_GLOBAL, false, true, false, true> : at_wave_affine<MODE_GLOBAL, false, false, false, true>;
	case AT_LOCAL: return prof ? at_wave_affine<MODE_LOCAL, false, true, false, true> : at_wave_affine<MODE_LOCAL, false, false, false, true>;
	case AT_FIT: return jump ? (prof ? at_wave_affine<MODE_FIT, true, true, false, true> : at_wave_affine<MODE_FIT, true, false, false, true>)
	                         : (prof ? at_wave_affine<MODE_FIT, false, true, false, true> : at_wave_affine<MODE_FIT, false, false, false, true>);
	default: return prof ? wave_linear_fn<MODE_OVERLAP, true, false, false, true>(R) : wave_linear_fn<MODE_OVERLAP, false, false, false, true>(R);
	}
}

struct CastU64 { __host__ __device__ uint64_t operator()(const uint32_t &x) const { return (uint64_t)x; } };

static SubstArgs subst_args(const Shard &s)
{
	SubstArgs a;
	a.matrix = s.d_subst.p; a.table = s.d_stab.p; a.qrow = s.d_qrow.p; a.tcol = s.d_tcol.p; a.table_bytes = s.table ? s.stab_bytes : 0;
	return a;
}

// `fills_done` (optional) is called once, when the next sub-slice of the pipelined one-shot path may
// launch its fill: after this shard's last traceback kernel has been enqueued (score-only: after its
// fills completed), so the device runs fill, traceback, next fill back to back while this shard's
// D2H copies and host work overlap the next fill.
static int run_shard(at_batch *b, Shard &s, const std::function<void()> *fills_done = nullptr)
{
	at_handle *h = b->h;
	CU(h, cudaSetDevice(s.dev->id));
	cudaStream_t st = s.stream;
	tl_stream = st;
	tl_cache = &s.cache; tl_big = s.dev->big.get();
	const bool jump = b->mode == AT_FIT && b->prm.jump;
	static const bool tb_overlap = getenv("AT_PIPE_TB_OVERLAP") != nullptr;
	s.fill_ms = s.tb_ms = s.dev_ms = s.domk_ms = 0; s.domk_cells = 0; s.launches = 0;
	// dominant (most cells) fill launch of the whole shard -> per-launch timing for the roofline
	int dom_chunk = -1, dom_launch = -1; uint64_t dom_cells = 0;
	for (size_t ci = 0; ci < s.chunks.size(); ++ci)
		for (size_t li = 0; li < s.chunks[ci].launches.size(); ++li)
			if (s.chunks[ci].launches[li].cells > dom_cells) { dom_cells = s.chunks[ci].launches[li].cells; dom_chunk = (int)ci; dom_launch = (int)li; }

	cudaEvent_t e_begin = s.ev[0], e_fill = s.ev[1], e_tb = s.ev[2];
	float ms = 0;
	bool first = true;
	cudaEvent_t e_first = s.ev[3];
	for (size_t ci = 0; ci < s.chunks.size(); ++ci) {
		Chunk &c = s.chunks[ci];
		const uint32_t nc = c.k1 - c.k0;
		CU(h, cudaMemsetAsync(s.d_counter.p, 0, 64 * sizeof(uint32_t), st));
		if (c.prog_words) CU(h, cudaMemsetAsync(s.d_prog.p, 0, c.prog_words * sizeof(uint32_t), st));
		if (b->mode >= AT_OVERLAP && c.bnd_elems) CU(h, cudaMemsetAsync(s.d_bnd.p, 0, c.bnd_elems * sizeof(uint64_t), st));   // tagged hand-off words of the single-plane kernels
		CU(h, cudaEventRecord(e_begin, st));
		if (first) { CU(h, cudaEventRecord(e_first, st)); first = false; }
		for (size_t li = 0; li < c.launches.size(); ++li) {
			const PlanLaunch &l = c.launches[li];
			const bool scored = !b->subst.empty();
			const void *fn = l.kind == LK_BITS ? (const void *)bits_kernel(l.r, b->traceback)
			               : l.kind == LK_WAVE ? (s.banded ? (const void *)wave_banded_kernel(b->mode, l.r, s.prof)
			                                     : scored ? (const void *)wave_scored_kernel(b->mode, jump, l.r, s.prof)
			                                     : (const void *)wave_kernel(b->mode, jump, l.r, s.prof, b->traceback))
			               : (const void *)affine_kernel(l.kind == LK_PACKED ? (b->mode == AT_LOCAL ? 4 : b->mode == AT_GLOBAL ? 5 : 6) : (b->mode == AT_FIT ? (jump ? 3 : 2) : b->mode), l.r, s.prof, scored);
			const int warps = l.kind >= LK_WAVE ? AT_WAVE_WARPS : AT_FILL_WARPS;
			const size_t dyn_smem = l.kind >= LK_WAVE ? (s.table ? wave_smem_bytes_table(s.stab_bytes) : 0)
			                      : s.table ? fill_smem_bytes_table(l.r, s.stab_bytes) : fill_smem_bytes(l.r, l.kind == LK_PACKED, s.prof);
			// the opt-in above 48 KB counts static and dynamic shared memory together: the K2 table variants have both, so every
			// table launch states its dynamic size (K1 has no static shared memory)
			if (dyn_smem > 48 * 1024 || s.table) CU(h, cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn_smem));
			int occ = 0;
			CU(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, 32 * warps, dyn_smem));
			if (occ < 1) { set_err(h, "fill kernel (mode %d, R %d) cannot be resident: not an sm_100 build?", b->mode, l.r); return AT_E_CUDA; }
			// AT_PIPE_TB_OVERLAP (older scheme, kept for A/B runs): traceback kernels run beside the next sub-slice's
			// fill, which must then leave them shared memory and registers (a K1 grid at full occupancy fills an SM)
			if (tb_overlap && s.workspace && l.kind != LK_WAVE && l.kind != LK_BITS && occ > 4) occ = 4;
			int blocks = (int)std::min<uint64_t>((uint64_t)s.dev->sm_count * occ, (l.n + warps - 1) / warps);
			if (blocks < 1) blocks = 1;
			const bool dom = (int)ci == dom_chunk && (int)li == dom_launch;
			if (dom) CU(h, cudaEventRecord(s.evk[0], st));
			if (l.kind >= LK_WAVE) {
				WaveArgs wa;
				wa.symmap = s.d_symmap.p; wa.syms = s.syms;
				wa.q = s.d_q.p; wa.q_off = s.d_q_off.p; wa.q_len = s.d_q_len.p;
				wa.t = s.d_t.p; wa.t_off = s.d_t_off.p; wa.t_len = s.d_t_len.p;
				wa.jmask = s.d_jmask.p; wa.j_off = s.twobit && jump ? s.d_j_off.p : s.d_t_off.p; wa.twobit = s.twobit ? 1 : 0; wa.start_lag = wave_start_lag(); wa.tasks = c.d_tasks[li].p; wa.n_tasks = l.n;
				wa.counter = s.d_counter.p + (l.kind == LK_BITS ? 48 : 32) + l.r; wa.prog = s.d_prog.p + l.prog_base;
				wa.ptr = s.d_ptr.p; wa.ptr_off = c.d_ptr_off.p; wa.pair_base = c.k0;
				wa.bnd = s.d_bnd.p; wa.bnd_off = c.d_bnd_off.p; wa.chain = s.d_chain.p;
				wa.score = s.d_score.p; wa.end_i = s.d_end_i.p; wa.end_j = s.d_end_j.p; wa.end_state = s.d_end_state.p;
				wa.m = b->prm.m; wa.u = b->prm.u; wa.o = b->prm.o; wa.e = b->prm.e; wa.jp = b->prm.j;
				wa.want_ptr = b->traceback ? 1 : 0;
				wa.k_and = cell_k_and<false>(); wa.k_or = cell_k_or<false>();
				wa.band = s.banded ? s.d_band.p : nullptr;
				wa.sub = subst_args(s);
				void *kargs[] = {(void *)&wa};
				CU(h, cudaLaunchKernel(fn, dim3(blocks), dim3(32 * warps), kargs, dyn_smem, st));
			} else {
				FillArgs2 fa;
				fa.q = s.d_q.p; fa.q_off = s.d_q_off.p; fa.q_len = s.d_q_len.p;
				fa.t = s.d_t.p; fa.t_off = s.d_t_off.p; fa.t_len = s.d_t_len.p;
				fa.jmask = s.d_jmask.p; fa.j_off = s.twobit && jump ? s.d_j_off.p : s.d_t_off.p; fa.symmap = s.d_symmap.p; fa.syms = s.syms;
				fa.jobs = c.d_jobs[li].p; fa.n_jobs = l.n;
				fa.counter = s.d_counter.p + (l.kind == LK_PACKED ? 16 : 0) + l.r; fa.ptr = s.d_ptr.p; fa.ptr_off = c.d_ptr_off.p; fa.pair_base = c.k0;
				fa.score = s.d_score.p; fa.end_i = s.d_end_i.p; fa.end_j = s.d_end_j.p; fa.end_state = s.d_end_state.p;
				fa.m = b->prm.m; fa.u = b->prm.u; fa.o = b->prm.o; fa.e = b->prm.e; fa.jp = b->prm.j;
				fa.want_ptr = b->traceback ? 1 : 0; fa.twobit = s.twobit ? 1 : 0;
				fa.k_and = l.kind == LK_PACKED ? cell_k_and<true>() : cell_k_and<false>(); fa.k_or = l.kind == LK_PACKED ? cell_k_or<true>() : cell_k_or<false>();
				fa.sub = subst_args(s);
				void *kargs[] = {(void *)&fa};
				CU(h, cudaLaunchKernel(fn, dim3(blocks), dim3(32 * warps), kargs, dyn_smem, st));
			}
			if (dom) CU(h, cudaEventRecord(s.evk[1], st));
			s.launches++;
		}
		CU(h, cudaEventRecord(e_fill, st));
		const bool last_chunk = ci + 1 == s.chunks.size();
		// pipelined one-shot path: the SMs go to the next sub-slice once this one's traceback kernels are in the
		// queue ahead of its fill -- the fill runs at full occupancy and the (short) traceback is not squeezed
		// beside it; copies and host round trips still overlap the neighbours' fills
		const bool tb_first = fills_done && last_chunk && b->traceback && !tb_overlap;
		if (fills_done && last_chunk && !tb_first) { CU(h, cudaEventSynchronize(e_fill)); (*fills_done)(); }
		if (b->traceback) {
			TraceArgs ta;
			ta.q = s.d_q.p; ta.q_off = s.d_q_off.p; ta.q_len = s.d_q_len.p;
			ta.t = s.d_t.p; ta.t_off = s.d_t_off.p; ta.t_len = s.d_t_len.p;
			ta.ptr = s.d_ptr.p; ta.ptr_off = c.d_ptr_off.p; ta.rclass = s.d_rclass.p;
			ta.pair_base = c.k0; ta.n_pairs = nc;
			ta.end_i = s.d_end_i.p; ta.end_j = s.d_end_j.p; ta.end_state = s.d_end_state.p;
			ta.beg_i = s.d_beg_i.p; ta.beg_j = s.d_beg_j.p; ta.n_ops = s.d_n_ops.p; ta.n_cols = s.d_n_cols.p;
			ta.ops_off = c.d_ops_off.p; ta.cols_off = c.d_cols_off.p;
			ta.scratch = s.d_scratch.p; ta.scratch_off = c.d_scratch_off.p;
			ta.cigar = nullptr; ta.aln1 = nullptr; ta.aln2 = nullptr;
			ta.mode = b->mode == AT_EDIT ? MODE_GLOBAL : b->mode;      // an edit path is emitted as global's: from (0, 0)
			ta.jump = jump ? 1 : 0; ta.twobit = s.twobit ? 1 : 0;
			ta.band = s.banded ? s.d_band.p : nullptr;
			// few long walks: one walker per warp, prefetching ahead; with many walks, or short ones (a few hundred
			// steps: nothing to prefetch far ahead of), the chase is throughput-bound and the prefetches only add traffic
			ta.lookahead = nc < 32768u && c.scratch_words / nc >= 2048 ? 1 : 0;
			const int walk_blocks = ta.lookahead ? (int)(((uint64_t)nc * 32 + 127) / 128) : (int)((nc + 127) / 128);   // one walker per warp | per thread
			if (b->mode == AT_EDIT && s.bits) at_traceback_walk<false, false, EDIT_WALK_BITS><<<walk_blocks, 128, 0, st>>>(ta);
			else if (b->mode == AT_EDIT) at_traceback_walk<false, false, EDIT_WALK_LIN><<<walk_blocks, 128, 0, st>>>(ta);
			else if (s.banded) at_traceback_walk<false, true><<<walk_blocks, 128, 0, st>>>(ta);
			else if (s.workspace && tb_overlap) at_traceback_walk<true><<<walk_blocks, 128, 0, st>>>(ta);
			else at_traceback_walk<false><<<walk_blocks, 128, 0, st>>>(ta);
			CU(h, cudaGetLastError());
			s.launches++;
			// exclusive offsets of n_ops / n_cols: offsets[0] = 0, offsets[1..nc] inclusive sums
			if (s.workspace && nc <= (1u << 18)) {      // pipelined path: must be able to run beside another stream's fill
				at_scan_offsets<<<2, 256, 0, st>>>(s.d_n_ops.p + c.k0, s.d_n_cols.p + c.k0, nc, c.d_ops_off.p, c.d_cols_off.p);
				CU(h, cudaGetLastError());
				s.launches++;
			} else {
				size_t tmp_bytes = 0;
				auto it_ops = thrust::make_transform_iterator((const uint32_t *)(s.d_n_ops.p + c.k0), CastU64());
				auto it_cols = thrust::make_transform_iterator((const uint32_t *)(s.d_n_cols.p + c.k0), CastU64());
				CU(h, cub::DeviceScan::InclusiveSum(nullptr, tmp_bytes, it_ops, c.d_ops_off.p + 1, (int)nc, st));
				CU(h, s.d_scan_tmp.alloc(tmp_bytes + 16));
				CU(h, cudaMemsetAsync(c.d_ops_off.p, 0, sizeof(uint64_t), st));
				CU(h, cudaMemsetAsync(c.d_cols_off.p, 0, sizeof(uint64_t), st));
				CU(h, cub::DeviceScan::InclusiveSum(s.d_scan_tmp.p, tmp_bytes, it_ops, c.d_ops_off.p + 1, (int)nc, st));
				CU(h, cub::DeviceScan::InclusiveSum(s.d_scan_tmp.p, tmp_bytes, it_cols, c.d_cols_off.p + 1, (int)nc, st));
			}
			const bool want_cig = b->out_flags & AT_OUT_CIGAR, want_aln = b->out_flags & AT_OUT_ALN;
			auto out_buffers = [&](uint64_t ops, uint64_t cols) -> int {
				// tb_first: the workspace's own buffers, kept across sub-slices and calls (grow-only) -- upper-bound sized
				// blocks are too large to go through the allocator in the steady state
				DevBuf<uint32_t> &cg = tb_first ? s.ws_cigar : c.d_cigar;
				DevBuf<uint8_t> &a1 = tb_first ? s.ws_aln1 : c.d_aln1, &a2 = tb_first ? s.ws_aln2 : c.d_aln2;
				if (want_cig) { if (cg.alloc(ops + 1) != cudaSuccess) { set_err(h, "cigar buffer"); return AT_E_NOMEM; } }
				if (want_aln) { if (a1.alloc(cols + 1) != cudaSuccess || a2.alloc(cols + 1) != cudaSuccess) { set_err(h, "alignment buffer"); return AT_E_NOMEM; } }
				ta.cigar = c.cigar = want_cig ? cg.p : nullptr;
				ta.aln1 = c.aln1 = want_aln ? a1.p : nullptr; ta.aln2 = c.aln2 = want_aln ? a2.p : nullptr;
				return AT_OK;
			};
			uint64_t tot[2] = {0, 0};
			if (tb_first) {
				// no host round trip between the walk and the emit: the outputs are sized by their upper bound
				// (an alignment has at most l1 + l2 columns; the workspace keeps the buffers), the totals follow later
				// (rounded up generously: sub-slices differ by a few pairs, and a request just above every cached
				// block would go to the CUDA allocator, which waits for the fills already in the queue)
				const uint64_t cap = (c.scratch_words + c.scratch_words / 8 + (1u << 22)) & ~(uint64_t)((1u << 22) - 1);
				if (int rc = out_buffers(cap, cap)) return rc;
			} else {
				CU(h, cudaMemcpyAsync(&tot[0], c.d_ops_off.p + nc, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
				CU(h, cudaMemcpyAsync(&tot[1], c.d_cols_off.p + nc, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
				CU(h, shard_sync(s));
				if (int rc = out_buffers(tot[0], tot[1])) return rc;
			}
			if (s.workspace && tb_overlap) at_traceback_emit<true><<<(int)(((uint64_t)nc * 32 + 127) / 128), 128, 0, st>>>(ta);
			else at_traceback_emit<false><<<(int)(((uint64_t)nc * 32 + 127) / 128), 128, 0, st>>>(ta);
			CU(h, cudaGetLastError());
			s.launches++;
			if (tb_first) {
				// the next fill is launched once this one has COMPLETED: launched earlier it would take the SMs
				// as this fill's blocks retire, and this sub-slice's traceback (and its workspace) would wait a whole
				// fill behind it -- the workers then fall into lockstep
				CU(h, cudaEventSynchronize(e_fill));
				(*fills_done)();
				CU(h, cudaMemcpyAsync(&tot[0], c.d_ops_off.p + nc, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
				CU(h, cudaMemcpyAsync(&tot[1], c.d_cols_off.p + nc, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
				CU(h, shard_sync(s));
			}
			c.tot_ops = tot[0]; c.tot_cols = tot[1];
		}
		CU(h, cudaEventRecord(e_tb, st));
		CU(h, shard_sync(s));
		CU(h, cudaEventElapsedTime(&ms, e_begin, e_fill)); s.fill_ms += ms;
		CU(h, cudaEventElapsedTime(&ms, e_fill, e_tb)); s.tb_ms += ms;
		if ((int)ci == dom_chunk) {
			CU(h, cudaEventElapsedTime(&ms, s.evk[0], s.evk[1])); s.domk_ms = ms; s.domk_cells = dom_cells;
			const PlanLaunch &dl = c.launches[dom_launch];
			s.domk_kind = (uint32_t)dl.kind; s.domk_r = (uint32_t)dl.r; s.domk_flags = (s.prof ? 1u : 0u) | (jump ? 2u : 0u) | (s.twobit ? 4u : 0u) | (b->subst.empty() ? 0u : 8u);
		}
		if (ci + 1 == s.chunks.size()) { CU(h, cudaEventElapsedTime(&ms, e_first, e_tb)); s.dev_ms = ms; }
	}
	h->launches += s.launches;
	return AT_OK;
}

extern "C" int at_batch_run(at_batch *b, at_timing *timing)
{
	if (!b) return AT_E_ARG;
	const size_t nd = b->shards.size();
	auto work = [&](size_t d) { Shard &s = b->shards[d]; s.rc = s.n ? run_shard(b, s) : AT_OK; };
	if (nd == 1) work(0);
	else { std::vector<std::thread> th; for (size_t d = 0; d < nd; ++d) th.emplace_back(work, d); for (auto &t : th) t.join(); }
	for (auto &s : b->shards) if (s.rc) return s.rc;
	b->ran = true;
	if (timing) {
		memset(timing, 0, sizeof *timing);
		for (auto &s : b->shards) {
			timing->fill_ms = std::max(timing->fill_ms, s.fill_ms);
			timing->traceback_ms = std::max(timing->traceback_ms, s.tb_ms);
			timing->device_ms = std::max(timing->device_ms, s.dev_ms);
			timing->cells += s.cells; timing->launches += s.launches; timing->ptr_bytes += b->traceback ? s.ptr_bytes : 0;
			if (s.domk_cells > timing->fill_kernel_cells) { timing->fill_kernel_cells = s.domk_cells; timing->fill_kernel_ms = s.domk_ms; timing->fill_kernel_kind = s.domk_kind; timing->fill_kernel_rows = s.domk_r; timing->fill_kernel_flags = s.domk_flags; }
		}
	}
	return AT_OK;
}

extern "C" int at_batch_sizes(const at_batch *b, uint64_t *cigar_ops, uint64_t *aln_bytes)
{
	if (!b || !b->ran) return AT_E_ARG;
	uint64_t o = 0, c = 0;
	for (auto &s : b->shards) for (auto &ch : s.chunks) { o += ch.tot_ops; c += ch.tot_cols; }
	if (cigar_ops) *cigar_ops = (b->out_flags & AT_OUT_CIGAR) ? o : 0;
	if (aln_bytes) *aln_bytes = (b->out_flags & AT_OUT_ALN) ? c : 0;
	return AT_OK;
}

// D2H of one shard's results into the caller's arrays.  base_ops / base_cols: position of the
// shard's first op / column in the dense outputs (advanced past this shard on return).  The
// offset arrays receive entries [out_base, out_base + n) here; the final entry [n_total] is the
// caller's job.
static int fetch_shard(at_batch *b, Shard &s, at_batch_output *out, bool want_cig, bool want_aln,
                       uint64_t &base_ops, uint64_t &base_cols)
{
	at_handle *h = b->h;
	if (!s.n) return AT_OK;
	CU(h, cudaSetDevice(s.dev->id));
	cudaStream_t st = s.stream;
	const uint64_t ob = s.out_base;
	CU(h, cudaMemcpyAsync(out->score + ob, s.d_score.p, s.n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
	if (out->end_i) CU(h, cudaMemcpyAsync(out->end_i + ob, s.d_end_i.p, s.n * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
	if (out->end_j) CU(h, cudaMemcpyAsync(out->end_j + ob, s.d_end_j.p, s.n * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
	if (out->beg_i) CU(h, cudaMemcpyAsync(out->beg_i + ob, s.d_beg_i.p, s.n * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
	if (out->beg_j) CU(h, cudaMemcpyAsync(out->beg_j + ob, s.d_beg_j.p, s.n * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
	for (auto &c : s.chunks) {
		const uint32_t nc = c.k1 - c.k0;
		if (want_cig) {
			CU(h, cudaMemcpyAsync(out->cigar_off + ob + c.k0, c.d_ops_off.p, nc * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
			if (c.tot_ops) CU(h, cudaMemcpyAsync(out->cigar + base_ops, c.cigar, c.tot_ops * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
		}
		if (want_aln) {
			CU(h, cudaMemcpyAsync(out->aln_off + ob + c.k0, c.d_cols_off.p, nc * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
			if (c.tot_cols) {
				CU(h, cudaMemcpyAsync(out->aln1 + base_cols, c.aln1, c.tot_cols, cudaMemcpyDeviceToHost, st));
				CU(h, cudaMemcpyAsync(out->aln2 + base_cols, c.aln2, c.tot_cols, cudaMemcpyDeviceToHost, st));
			}
		}
		CU(h, shard_sync(s));
		// chunk-local offsets -> global
		if (want_cig && base_ops) for (uint32_t k = 0; k < nc; ++k) out->cigar_off[ob + c.k0 + k] += base_ops;
		if (want_aln && base_cols) for (uint32_t k = 0; k < nc; ++k) out->aln_off[ob + c.k0 + k] += base_cols;
		base_ops += c.tot_ops; base_cols += c.tot_cols;
	}
	CU(h, shard_sync(s));
	return AT_OK;
}

extern "C" int at_batch_fetch(at_batch *b, at_batch_output *out)
{
	if (!b || !out || !b->ran || !out->score) return AT_E_ARG;
	at_handle *h = b->h;
	const bool want_cig = b->traceback && (b->out_flags & AT_OUT_CIGAR) && out->cigar;
	const bool want_aln = b->traceback && (b->out_flags & AT_OUT_ALN) && out->aln1 && out->aln2;
	if (want_cig && !out->cigar_off) return AT_E_ARG;
	if (want_aln && !out->aln_off) return AT_E_ARG;
	uint64_t tot_ops = 0, tot_cols = 0;
	at_batch_sizes(b, &tot_ops, &tot_cols);
	if (want_cig && tot_ops > out->cigar_cap) { set_err(h, "cigar buffer too small: need %llu ops", (unsigned long long)tot_ops); return AT_E_NOSPACE; }
	if (want_aln && tot_cols > out->aln_cap) { set_err(h, "alignment buffer too small: need %llu bytes", (unsigned long long)tot_cols); return AT_E_NOSPACE; }
	uint64_t base_ops = 0, base_cols = 0;
	for (auto &s : b->shards)
		if (int rc = fetch_shard(b, s, out, want_cig, want_aln, base_ops, base_cols)) return rc;
	if (want_cig) out->cigar_off[b->n] = base_ops;
	if (want_aln) out->aln_off[b->n] = base_cols;
	if (!b->traceback) {
		if (out->cigar_off) for (uint64_t k = 0; k <= b->n; ++k) out->cigar_off[k] = 0;
		if (out->aln_off) for (uint64_t k = 0; k <= b->n; ++k) out->aln_off[k] = 0;
	}
	return AT_OK;
}

#include "at_pipeline.inl"      // at_batch_align: the pipelined one-shot path (same translation unit)

extern "C" void *at_host_alloc(size_t bytes)
{
	void *p = nullptr;
	if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
	return p;
}

extern "C" void at_host_free(void *p) { if (p) cudaFreeHost(p); }

extern "C" int at_host_register(void *p, size_t bytes)
{
	if (!p || !bytes) return AT_E_ARG;
	if (cudaHostRegister(p, bytes, cudaHostRegisterPortable) != cudaSuccess) { cudaGetLastError(); return AT_E_CUDA; }
	return AT_OK;
}

extern "C" int at_host_unregister(void *p)
{
	if (!p) return AT_E_ARG;
	if (cudaHostUnregister(p) != cudaSuccess) { cudaGetLastError(); return AT_E_CUDA; }
	return AT_OK;
}

extern "C" int64_t at_pack_2bit(const char *seq, uint64_t n, uint8_t *dst)
{
	if (!seq || !dst) return -1;
	const uint64_t nb = (n + 3) / 4;
	memset(dst, 0, nb);
	for (uint64_t k = 0; k < n; ++k) {
		uint8_t c;
		switch (seq[k]) { case 'A': c = 0; break; case 'C': c = 1; break; case 'G': c = 2; break; case 'T': c = 3; break; default: return -1; }
		dst[k >> 2] |= (uint8_t)(c << (2 * (k & 3)));
	}
	return (int64_t)nb;
}

extern "C" int64_t at_cigar_to_string(const uint32_t *ops, uint64_t n_ops, char *dst, uint64_t cap)
{
	if (!dst || (!ops && n_ops)) return -1;
	uint64_t pos = 0;
	for (uint64_t k = 0; k < n_ops; ++k) {
		char buf[16];
		const uint32_t code = ops[k] & 15u;      // the format reserves four bits for the op code
		if (code > AT_CIG_N) return -1;
		const int len = snprintf(buf, sizeof buf, "%u%c", ops[k] >> 4, "MIDN"[code]);
		if (pos + len + 1 > cap) return -1;
		memcpy(dst + pos, buf, len); pos += len;
	}
	if (pos + 1 > cap) return -1;
	dst[pos] = 0;
	return (int64_t)pos;
}
