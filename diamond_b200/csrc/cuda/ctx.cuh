// ctx.cuh -- shared definitions of the CUDA K layer (libdmnd_b200.so): context, block residency, scratch arena,
// event-based phase timing.  sm_100a only; no fallback of any kind.
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>
#include "../../../include/dmnd_b200.h"
#include "dev_params.h"

namespace dmnd_cuda {

void set_error(const std::string& m);

#define DMND_CUDA_CHECK(expr)                                                                             \
	do {                                                                                                  \
		cudaError_t _e = (expr);                                                                          \
		if (_e != cudaSuccess) {                                                                          \
			dmnd_cuda::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e) + " (" + __FILE__ + ":" + std::to_string(__LINE__) + ")"); \
			return 1;                                                                                     \
		}                                                                                                 \
	} while (0)

// Grow-only device buffer (the library owns all device memory; nothing is allocated per launch in steady state).
struct DevBuf {
	void* p = nullptr;
	size_t cap = 0;
	int ensure(size_t bytes) {
		if (bytes <= cap) return 0;
		if (p) cudaFree(p);
		p = nullptr; cap = 0;
		const size_t want = bytes + bytes / 4 + 256;
		cudaError_t e = cudaMalloc(&p, want);
		if (e != cudaSuccess) { set_error(std::string("cudaMalloc(") + std::to_string(want) + "): " + cudaGetErrorString(e)); return 1; }
		cap = want;
		return 0;
	}
	// grow and keep the first `keep` bytes (device-to-device copy; cudaFree synchronises, so the copy is complete before the old buffer goes)
	int ensure_keep(size_t bytes, size_t keep) {
		if (bytes <= cap) return 0;
		void* old = p;
		const size_t want = bytes + bytes / 2 + 256;
		void* np = nullptr;
		cudaError_t e = cudaMalloc(&np, want);
		if (e != cudaSuccess) { set_error(std::string("cudaMalloc(") + std::to_string(want) + "): " + cudaGetErrorString(e)); return 1; }
		if (old && keep) cudaMemcpy(np, old, keep < cap ? keep : cap, cudaMemcpyDeviceToDevice);
		if (old) cudaFree(old);
		p = np; cap = want;
		return 0;
	}
	void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
	template<typename T> T* as() const { return (T*)p; }
};

enum Phase { PH_SEED = 0, PH_DP_SCORE, PH_DP_TRACE, PH_H2D, PH_D2H, PH_COUNT };

}  // namespace dmnd_cuda

namespace dmnd_cuda {
// Seed index of a reference block for one shape: sorted 40-bit key mixes + locations, bucket directory, Bloom filter.
struct RefIndex {
	DevBuf keys, locs, bucket, bloom, bitmap;
	unsigned long long nref = 0;
	int sid = -1, shift = 0;
	uint32_t bloom_blocks = 0;
	uint32_t bitmap_mask = 0;  // bits of the first-level filter - 1
	bool valid = false;
	uint64_t content_epoch = 0, params_hash = 0;  // what the index was built from: the block's content epoch and the context's parameters
	void release() { keys.release(); locs.release(); bucket.release(); bloom.release(); bitmap.release(); valid = false; }
};

// Content epochs are unique in the process, not per block: a block allocated where a freed one lived (same address) never
// matches an index cached for the old one's contents.
inline uint64_t new_content_epoch() {
	static std::atomic<uint64_t> next{ 1 };
	return next.fetch_add(1, std::memory_order_relaxed);
}
}  // namespace dmnd_cuda

struct dmnd_block {
	dmnd_cuda::RefIndex idx;             // built by dmnd_block_build_index (reference side), reused by every lane
	size_t cap_bytes = 0, cap_seqs = 0;  // allocated sizes (the block pool matches on them)
	int8_t* letters = nullptr;  // device
	int8_t* bias = nullptr;     // device, same offsets as letters
	int64_t* limits = nullptr;  // device
	uint32_t* soft = nullptr;   // device, one bit per letter: inside a MaskingTable entry (abundant motif), see dmnd_block_mask
	bool has_soft = false;      // dmnd_block_mask(MOTIF) has run: dmnd_search_shape reads `soft`
	size_t raw_len = 0;
	uint32_t nseq = 0;
	uint64_t content_epoch = dmnd_cuda::new_content_epoch();  // renewed whenever letters or the soft table change (dmnd_block_mask): a cached index of an older epoch is rebuilt
	std::vector<int64_t> h_limits;  // host copy (problem binning needs lengths)
	std::vector<cudaEvent_t> range_ready;  // dmnd_block_upload_ranges: one event per uploaded sequence range
	std::vector<uint32_t> range_cuts;      // [nranges + 1] sequence boundaries of those ranges
};

struct dmnd_hits {
	dmnd_hit* d = nullptr;  // device, grouped by query; lives in the context's hit arena (no per-call cudaMalloc/cudaFree:
	size_t n = 0;           // cudaFree synchronises the whole device and would stall the other lanes)
};

struct dmnd_ctx {
	int device = 0;
	dmnd_params params;
	dmnd_cuda::DevParams h_dev_params;
	dmnd_cuda::DevParams* d_params = nullptr;
	uint8_t* d_matcher[DMND_MAX_SHAPES + 1] = {};  // PatternMatcher tables
	uint32_t matcher_minlen[DMND_MAX_SHAPES + 1] = {}, matcher_suffix[DMND_MAX_SHAPES + 1] = {};
	cudaStream_t stream = nullptr, copy_stream = nullptr;
	cudaEvent_t ev_copy = nullptr;
	int sm_count = 148;
	// scratch
	dmnd_cuda::DevBuf b_keys, b_keys2, b_vals, b_vals2, b_cub, b_bucket, b_entries, b_pairs, b_hits, b_hits2, b_counters;
	dmnd_cuda::DevBuf b_surv;  // stage-1 survivors of one index chunk (seed.cu)
	unsigned long long last_pairs_bound = 0;  // (q, s) pairs of the last search slice (sizes the next one)
	dmnd_cuda::DevBuf b_probs, b_results, b_order, b_trace, b_trace_off, b_tr, b_work, b_prep, b_bloom;
	dmnd_cuda::DevBuf b_mask_pb, b_mask_scale, b_mask_pos, b_mask_pos2, b_mask_cov, b_mask_flag, b_mask_seqs, b_mask_zinv, b_mask_need;  // dmnd_block_mask scratch
	uint64_t mask_n = 0;  // letters hard-masked by the last dmnd_block_mask on this context (sorted offsets in b_mask_pos)
	std::vector<uint64_t> h_excl;  // host copy of the trace prefix (slicing)
	void* comm = nullptr; int comm_rank = 0, comm_size = 1;  // NCCL communicator of dmnd_comm_init (comm.cu)
	bool force_generic_dp = false;
	bool force_int32_dp = false;     // the packed 16-bit kernel overflowed: this call runs on the int32 kernels
	uint8_t* d_s16_table = nullptr;   // global image of the score table of swipe16_kernel (swipe16.cuh), built once per context
	bool s16_ok = false;
	uint64_t dp_overflows = 0;       // calls repeated on the int32 kernels
	uint64_t dp_cells_score = 0, dp_cells_trace = 0, dp_cells_padded = 0;  // cells of the problems LAUNCHED (score-only / traceback kernels) and what the register tiles evaluate for them
	std::vector<dmnd_ctx*> lanes;  // owned lane contexts (dmnd_ctx_lane)
	dmnd_cuda::RefIndex own_index;  // private reference index when the block carries none
	const dmnd_block* own_index_block = nullptr;  // ... and the block it was built from (own_index.content_epoch = that block's epoch; the pair
	                                              // identifies the contents even when a later block reuses the address)
	dmnd_cuda::DevBuf b_chain_probs;  // dmnd_hits_chain: the DP problems of the device-chained queries (read in place by dmnd_banded_swipe_chained)
	dmnd_chain_query* chain_q = nullptr; dmnd_dp_problem* chain_probs = nullptr; dmnd_hit* chain_fb_hits = nullptr; dmnd_segment* chain_fb_segs = nullptr; dmnd_hit_site* chain_fb_sites = nullptr;
	size_t chain_counts[3] = {};
	dmnd_cuda::DevBuf b_hits_out;  // hit arena handed out by dmnd_search_shape (one live dmnd_hits per context)
	struct FreeBlock { int8_t *letters, *bias; int64_t* limits; uint32_t* soft; size_t cap_bytes, cap_seqs; dmnd_cuda::RefIndex idx; };
	std::vector<FreeBlock> block_pool;  // device memory of freed blocks, reused by dmnd_block_upload
	void* h_pinned = nullptr;  // small pinned staging for counters
	size_t h_pinned_cap = 0;
	// timing
	cudaEvent_t ev_a = nullptr, ev_b = nullptr;
	cudaEvent_t ev_sync = nullptr;  // cudaEventBlockingSync: host waits sleep instead of spinning (the host pool owns the CPU quota)
	double phase_ms[dmnd_cuda::PH_COUNT] = {};
	uint64_t launches = 0, h2d_bytes = 0, d2h_bytes = 0;
};

namespace dmnd_cuda {

// Host wait for everything queued on `st`: sleeps on a blocking event.  cudaStreamSynchronize spins under the default
// schedule flags, and a spinning lane thread burns one CPU of the container's quota that the worker pool needs.
inline cudaError_t stream_wait(dmnd_ctx* c, cudaStream_t st) {
	cudaError_t e = cudaEventRecord(c->ev_sync, st);
	if (e != cudaSuccess) return e;
	return cudaEventSynchronize(c->ev_sync);
}

struct PhaseTimer {  // CUDA events on the library's stream, accumulated per phase
	dmnd_ctx* c; Phase ph;
	PhaseTimer(dmnd_ctx* c, Phase ph) : c(c), ph(ph) { cudaEventRecord(c->ev_a, c->stream); }
	void stop() {
		cudaEventRecord(c->ev_b, c->stream);
		cudaEventSynchronize(c->ev_b);
		float ms = 0;
		cudaEventElapsedTime(&ms, c->ev_a, c->ev_b);
		c->phase_ms[ph] += ms;
	}
	// split form for phases with a host decision in the middle: mark_end() closes the interval on the stream without
	// waiting, collect() adds it up once the stream is known to have passed the mark, restart() opens the next interval --
	// the host gap between the two intervals is not counted as device time
	void mark_end() { cudaEventRecord(c->ev_b, c->stream); }
	void collect() {
		float ms = 0;
		if (cudaEventElapsedTime(&ms, c->ev_a, c->ev_b) == cudaSuccess) c->phase_ms[ph] += ms;
	}
	void restart() { cudaEventRecord(c->ev_a, c->stream); }
};

int search_shape_impl(dmnd_ctx* ctx, dmnd_block* query, const dmnd_block* ref, int sid, uint32_t q_begin, uint32_t q_end, dmnd_hits** out, dmnd_stage_counters* counters);
int build_ref_index(dmnd_ctx* ctx, const dmnd_block* ref, int sid, RefIndex& ix);
int debug_left_most_impl(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, int sid, int chunk, uint32_t qloc, uint32_t sloc, unsigned long long* out30);
int hits_xdrop_impl(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, const dmnd_hits* h, int raw_xdrop, dmnd_segment* host, dmnd_hit_site* sites, size_t cap);
int hits_gapped_filter_impl(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, const dmnd_hits* h, uint8_t* pass, size_t cap);
int block_mask_impl(dmnd_ctx* ctx, dmnd_block* b, int algo, uint32_t s_begin, uint32_t s_end, uint64_t* n_hard);
int block_mask_fetch_impl(dmnd_ctx* ctx, uint64_t* positions, size_t cap);
}  // namespace dmnd_cuda
extern "C" int dmnd_block_alloc_empty(dmnd_ctx* ctx, size_t raw_len, uint32_t nseq, dmnd_block** out);
namespace dmnd_cuda {
int launch_xdrop(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, const dmnd_hits* h, int raw_xdrop, dmnd_segment* d_segs, dmnd_hit_site* d_sites);
int hits_chain_impl(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, const dmnd_hits* h, int raw_xdrop, int band_slow, int max_targets, dmnd_chain_out* out);
int hits_chain_fetch_impl(dmnd_ctx* ctx, dmnd_chain_query* queries, dmnd_dp_problem* problems, dmnd_hit* hits, dmnd_segment* segs, dmnd_hit_site* sites);
int s16_table_build(dmnd_ctx* ctx);
int banded_swipe_impl(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, const dmnd_dp_problem* problems, const dmnd_dp_problem* d_problems, size_t n, int mode,
                      dmnd_dp_result* results, uint8_t* transcripts, size_t transcript_cap);

}  // namespace dmnd_cuda
