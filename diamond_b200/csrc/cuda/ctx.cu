// ctx.cu -- context, block residency and the extern "C" K-layer entry points of libdmnd_b200.so.
#include "ctx.cuh"
#include <cmath>
#include <cstring>

namespace dmnd_cuda {
static thread_local std::string g_err;
void set_error(const std::string& m) { g_err = m; }
}  // namespace dmnd_cuda
using namespace dmnd_cuda;

static __global__ void clear_seed_mask_kernel(int8_t* letters, size_t begin, size_t end) {
	// 16 B per thread over [begin, end); every byte keeps its low 7 bits (delimiter 31 is unaffected).  Chunks that
	// straddle the range ends are handled byte by byte so that bytes of a neighbouring query range are never rewritten.
	const size_t c0 = (begin / 16) * 16 + ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 16;
	if (c0 >= end) return;
	if (c0 >= begin && c0 + 16 <= end) {
		uint4* p = reinterpret_cast<uint4*>(letters + c0);
		uint4 v = *p;
		v.x &= 0x7f7f7f7fu; v.y &= 0x7f7f7f7fu; v.z &= 0x7f7f7f7fu; v.w &= 0x7f7f7f7fu;
		*p = v;
	}
	else
		for (size_t k = (c0 > begin ? c0 : begin); k < c0 + 16 && k < end; ++k) letters[k] &= 0x7f;
}

// HauserCorrection (stats/hauser_correction.cpp:53-109), one thread per sequence running the reference's own five-phase
// sliding-window loop.  The window sums are integers; the three float operations per position (int->float, divide,
// subtract) and the half-away-from-zero rounding use the explicit round-to-nearest intrinsics, so the int8 results are
// bit-identical to the host's scalar code (no FMA contraction, IEEE division).
// Memory: the 128 sequences of a block are contiguous in the block image, so the block stages their letters through
// shared memory with coalesced 16-byte loads, works on the staged copy in place (letter -> bias) and writes the range
// back coalesced; a range that does not fit (long sequences) is processed straight from global memory.
#define HAUSER_STAGE_BYTES (40 * 1024)
static __global__ void __launch_bounds__(128) hauser_kernel(const int8_t* __restrict__ letters, const int64_t* __restrict__ limits, uint32_t nseq,
                                     const DevParams* __restrict__ P, int8_t* __restrict__ bias) {
	__shared__ int8_t s_score[32 * 20];
	__shared__ float s_bg[20];
	__shared__ __align__(16) int8_t s_stage[HAUSER_STAGE_BYTES];
	for (int i = threadIdx.x; i < 32 * 20; i += blockDim.x) s_score[i] = P->score[(i / 20) * 32 + (i % 20)];
	if (threadIdx.x < 20) s_bg[threadIdx.x] = P->background_scores_f32[threadIdx.x];
	const uint32_t s0 = blockIdx.x * blockDim.x, s1 = min(nseq, s0 + blockDim.x);
	const int64_t rbeg = limits[s0] & ~(int64_t)15, rend = limits[s1];  // [rbeg, rend) covers the block's sequences (+ delimiters)
	const bool staged = (rend - rbeg) <= HAUSER_STAGE_BYTES;
	if (staged)
		for (int64_t x = (int64_t)threadIdx.x * 16; x < rend - rbeg; x += (int64_t)blockDim.x * 16)
			*reinterpret_cast<uint4*>(s_stage + x) = *reinterpret_cast<const uint4*>(letters + rbeg + x);  // block images are 16 B aligned and padded
	__syncthreads();
	const uint32_t sidx = s0 + threadIdx.x;
	if (sidx < nseq) {
		const int64_t beg = limits[sidx];
		const int len = (int)(limits[sidx + 1] - beg - 1);
		if (len > 0) {
			const int8_t* seq = staged ? s_stage + (beg - rbeg) : letters + beg;
			int8_t* out = staged ? s_stage + (beg - rbeg) : bias + beg;  // in place when staged: position m is read before it is overwritten
			int scores[20];
#pragma unroll
			for (int i = 0; i < 20; ++i) scores[i] = 0;
			const unsigned window = 40, l = (unsigned)len, window_half = min(window / 2, l - 1);
			unsigned n = 0, h = 0, m = 0, t = 0;
			auto add = [&](int letter) { const int8_t* row = s_score + letter * 20;
#pragma unroll
				for (int i = 0; i < 20; ++i) scores[i] += row[i]; };
			auto sub = [&](int letter) { const int8_t* row = s_score + letter * 20;
#pragma unroll
				for (int i = 0; i < 20; ++i) scores[i] -= row[i]; };
			// the in-place update destroys letters behind m, but the trailing edge t <= m - 20 still needs them: keep the last
			// 41 letters in a small ring (registers / local) -- simpler: a ring buffer of the window's letters
			uint8_t ring[64];
			auto letter_at = [&](unsigned pos) -> int { return staged ? (int)ring[pos & 63] : (int)(seq[pos] & 31); };
			auto emit = [&](unsigned pos) {
				const int r = letter_at(pos);
				int8_t v = 0;
				if (r < 20) {
					int sr = 0;
#pragma unroll
					for (int i = 0; i < 20; ++i) if (i == r) sr = scores[i];
					const float f = __fsub_rn(s_bg[r], __fdiv_rn(__int2float_rn(sr - (int)s_score[r * 20 + r]), __uint2float_rn(n - 1)));
					v = (int8_t)(f < 0.0f ? __fsub_rn(f, 0.5f) : __fadd_rn(f, 0.5f));
				}
				out[pos] = v;
			};
			auto take = [&](unsigned pos) -> int { const int L = seq[pos] & 31; if (staged) ring[pos & 63] = (uint8_t)L; return L; };  // h runs ahead of m and t
			while (n < window_half && h < l) { ++n; add(take(h)); ++h; }
			while (n < (window + 1) && h < l) { ++n; add(take(h)); emit(m); ++h; ++m; }
			while (h < l) { add(take(h)); sub(letter_at(t)); emit(m); ++h; ++t; ++m; }
			while (m < l && n > (window_half + 1)) { --n; sub(letter_at(t)); emit(m); ++t; ++m; }
			while (m < l) { emit(m); ++m; }
		}
	}
	__syncthreads();
	if (staged) {
		// delimiters (and the 0..15 leading bytes of the previous block's tail) must stay 0 in the bias array
		for (int64_t x = threadIdx.x; x < rend - rbeg; x += blockDim.x) {
			const int64_t g = rbeg + x;
			if (g >= limits[s0]) bias[g] = (letters[g] == DMND_DELIMITER) ? (int8_t)0 : s_stage[x];
		}
	}
}

// Issue-rate micro-benchmark: 8 independent chains of one DPX instruction per thread, enough warps to fill every SMSP.
// PACKED = false: VIADDMNMX (one 32-bit cell per lane), true: VIADDMNMX.S16x2 (two 16-bit cells per lane, swipe16.cuh).
template<bool PACKED>
static __global__ void __launch_bounds__(256) int_peak_kernel(int* out, int iters, int b) {
	int a[8];
#pragma unroll
	for (int k = 0; k < 8; ++k) a[k] = threadIdx.x + k;
	for (int i = 0; i < iters; ++i) {
#pragma unroll
		for (int k = 0; k < 8; ++k) a[k] = PACKED ? (int)__viaddmax_s16x2((unsigned)a[k], (unsigned)b, (unsigned)(k - i)) : __viaddmax_s32(a[k], b, k - i);
	}
	int s = 0;
#pragma unroll
	for (int k = 0; k < 8; ++k) s += a[k];
	out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

extern "C" {

static int measure_peak(dmnd_ctx* ctx, bool packed, double* lane_instr_per_s) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	const int blocks = ctx->sm_count * 8, threads = 256, iters = 1 << 15;
	if (ctx->b_work.ensure((size_t)blocks * threads * sizeof(int))) return 1;
	if (packed) int_peak_kernel<true><<<blocks, threads, 0, ctx->stream>>>(ctx->b_work.as<int>(), 1024, -1);  // warm-up
	else int_peak_kernel<false><<<blocks, threads, 0, ctx->stream>>>(ctx->b_work.as<int>(), 1024, -1);
	cudaEventRecord(ctx->ev_a, ctx->stream);
	if (packed) int_peak_kernel<true><<<blocks, threads, 0, ctx->stream>>>(ctx->b_work.as<int>(), iters, -1);
	else int_peak_kernel<false><<<blocks, threads, 0, ctx->stream>>>(ctx->b_work.as<int>(), iters, -1);
	cudaEventRecord(ctx->ev_b, ctx->stream);
	DMND_CUDA_CHECK(cudaEventSynchronize(ctx->ev_b));
	float ms = 0;
	cudaEventElapsedTime(&ms, ctx->ev_a, ctx->ev_b);
	*lane_instr_per_s = (double)blocks * threads * (double)iters * 8.0 / (ms * 1e-3);
	return 0;
}
int dmnd_measure_int_peak(dmnd_ctx* ctx, double* lane_instr_per_s) { return measure_peak(ctx, false, lane_instr_per_s); }
int dmnd_measure_int_peak_packed(dmnd_ctx* ctx, double* lane_instr_per_s) { return measure_peak(ctx, true, lane_instr_per_s); }

const char* dmnd_last_error(void) { return g_err.c_str(); }
void dmnd_set_last_error(const char* m) { g_err = m ? m : ""; }
const char* dmnd_backend(void) { return "cuda-sm100a"; }
const dmnd_params* dmnd_ctx_params(const dmnd_ctx* ctx) { return &ctx->params; }

int dmnd_create(int device, const dmnd_params* params, dmnd_ctx** out) {
	int ndev = 0;
	if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
		set_error("dmnd_create: no CUDA device visible -- libdmnd_b200.so has no CPU path");
		return 1;
	}
	if (device < 0 || device >= ndev) { set_error("dmnd_create: bad device index"); return 1; }
	DMND_CUDA_CHECK(cudaSetDevice(device));
	cudaDeviceProp prop;
	DMND_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
	if (prop.major < 10) { set_error(std::string("dmnd_create: device ") + prop.name + " is not sm_100 class; this library is built for sm_100a only"); return 1; }
	dmnd_ctx* c = new dmnd_ctx();
	c->device = device;
	c->params = *params;
	c->sm_count = prop.multiProcessorCount;
	{
		int least = 0, greatest = 0;
		DMND_CUDA_CHECK(cudaDeviceGetStreamPriorityRange(&least, &greatest));
		DMND_CUDA_CHECK(cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, greatest));
	}
	DMND_CUDA_CHECK(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
	DMND_CUDA_CHECK(cudaEventCreateWithFlags(&c->ev_copy, cudaEventDisableTiming));
	DMND_CUDA_CHECK(cudaEventCreate(&c->ev_a));
	DMND_CUDA_CHECK(cudaEventCreateWithFlags(&c->ev_b, cudaEventBlockingSync));
	DMND_CUDA_CHECK(cudaEventCreateWithFlags(&c->ev_sync, cudaEventBlockingSync | cudaEventDisableTiming));
	DevParams& d = c->h_dev_params;
	std::memset(&d, 0, sizeof d);
	d.one = 1; d.k65536 = 65536; d.neg2 = 0x80008000u;
	std::memcpy(d.score, params->score, 1024);
	std::memcpy(d.reduction, params->reduction, 32);
	std::memcpy(d.map8, params->map8, 32);
	std::memcpy(d.map8b, params->map8b, 32);
	std::memcpy(d.shape_pos, params->shape_pos, sizeof d.shape_pos);
	std::memcpy(d.shape_mask, params->shape_mask, sizeof d.shape_mask);
	std::memcpy(d.shape_len, params->shape_len, sizeof d.shape_len);
	d.n_shapes = params->n_shapes; d.shape_weight = params->shape_weight; d.reduction_size = params->reduction_size;
	d.hamming_id = params->hamming_id; d.seedp_bits = params->seedp_bits; d.index_chunks = params->index_chunks;
	d.left_most_interval = params->left_most_interval; d.ungapped_window = params->ungapped_window;
	d.gap_open = params->gap_open; d.gap_extend = params->gap_extend; d.seed_cut = params->seed_cut;
	std::memcpy(d.background_scores_f32, params->background_scores_f32, sizeof d.background_scores_f32);
	std::memcpy(d.ungapped_cutoff, params->ungapped_cutoff, sizeof d.ungapped_cutoff);
	d.short_query_ungapped_cutoff = params->short_query_ungapped_cutoff; d.short_query_max_len = params->short_query_max_len;
	d.query_contexts = params->query_contexts > 1 ? params->query_contexts : 1; std::memcpy(d.ungapped_cutoff_short, params->ungapped_cutoff_short, sizeof d.ungapped_cutoff_short);
	std::memcpy(d.gapped_cutoff1, params->gapped_cutoff1, sizeof d.gapped_cutoff1); std::memcpy(d.gapped_cutoff2, params->gapped_cutoff2, sizeof d.gapped_cutoff2);
	d.gapped_filter_diag_score = params->gapped_filter_diag_score; d.gapped_filter_window = params->gapped_filter_window;
	std::memcpy(d.tantan_lr, params->tantan_lr, sizeof d.tantan_lr);
	std::memcpy(d.tantan_d, params->tantan_d, sizeof d.tantan_d);
	d.tantan_b2b = params->tantan_b2b; d.tantan_f2f = params->tantan_f2f; d.tantan_p_repeat_end = params->tantan_p_repeat_end;
	d.tantan_p_mask = params->tantan_p_mask; d.max_motif_len = params->max_motif_len;
	{
		unsigned long long pw = 1;
		for (int i = 0; i < params->shape_weight; ++i) pw *= (unsigned long long)params->reduction_size;
		int bits = 0;
		for (unsigned long long x = pw - 1; x > 0; x >>= 1) ++bits;
		d.seed_bits = bits;
	}
	// ln(n!) rounded to 6 decimals, as tabulated by the reference (lib/blast/blast_seg.cpp:54-58)
	static const double LNFACT[13] = { 0.000000, 0.000000, 0.693147, 1.791759, 3.178054, 4.787492, 6.579251, 8.525161,
		10.604603, 12.801827, 15.104413, 17.502308, 19.987214 };
	std::memcpy(d.lnfact, LNFACT, sizeof LNFACT);
	DMND_CUDA_CHECK(cudaMalloc(&c->d_params, sizeof(DevParams)));
	DMND_CUDA_CHECK(cudaMemcpy(c->d_params, &d, sizeof d, cudaMemcpyHostToDevice));
	// PatternMatcher tables (util/algo/pattern_matcher.h:25-45): matcher[k] over shapes [0,k)
	for (int k = 0; k <= params->n_shapes; ++k) {
		uint32_t minl = 32, maxl = 0;
		for (int i = 0; i < k; ++i) {
			const uint32_t len = 32 - (uint32_t)__builtin_clz(params->shape_mask[i]);
			maxl = len > maxl ? len : maxl;
			minl = len < minl ? len : minl;
		}
		c->matcher_minlen[k] = minl;
		c->matcher_suffix[k] = (1u << maxl) - 1;
		std::vector<uint8_t> t((size_t)c->matcher_suffix[k] + 1, 0);
		for (uint32_t s = 0; s <= c->matcher_suffix[k]; ++s)
			for (int i = 0; i < k; ++i)
				if ((s & params->shape_mask[i]) == params->shape_mask[i]) t[s] = 1;
		DMND_CUDA_CHECK(cudaMalloc(&c->d_matcher[k], t.size()));
		DMND_CUDA_CHECK(cudaMemcpy(c->d_matcher[k], t.data(), t.size(), cudaMemcpyHostToDevice));
	}
	c->h_pinned_cap = 1 << 16;
	DMND_CUDA_CHECK(cudaMallocHost(&c->h_pinned, c->h_pinned_cap));
	if (dmnd_cuda::s16_table_build(c)) return 1;
	*out = c;
	return 0;
}

int dmnd_ctx_lane(dmnd_ctx* ctx, int lane, dmnd_ctx** out) {
	if (lane < 0 || lane > 15) { set_error("dmnd_ctx_lane: lane index out of range"); return 1; }
	while ((int)ctx->lanes.size() <= lane) {
		dmnd_ctx* c = nullptr;
		if (dmnd_create(ctx->device, &ctx->params, &c)) return 1;
		// lanes run staggered: an earlier lane is further along, so its kernels go first (lower lane = higher priority)
		int least = 0, greatest = 0;
		DMND_CUDA_CHECK(cudaDeviceGetStreamPriorityRange(&least, &greatest));
		cudaStreamDestroy(c->stream);
		DMND_CUDA_CHECK(cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, std::min(least, greatest + 1 + (int)ctx->lanes.size())));
		ctx->lanes.push_back(c);
	}
	*out = ctx->lanes[(size_t)lane];
	return 0;
}

void dmnd_destroy(dmnd_ctx* c) {
	if (!c) return;
	for (dmnd_ctx* l : c->lanes) dmnd_destroy(l);
	c->lanes.clear();
	cudaSetDevice(c->device);
	cudaStreamSynchronize(c->stream);
	DevBuf* bufs[] = { &c->b_keys, &c->b_keys2, &c->b_vals, &c->b_vals2, &c->b_cub, &c->b_bucket, &c->b_entries, &c->b_pairs, &c->b_hits,
		&c->b_hits2, &c->b_counters, &c->b_probs, &c->b_results, &c->b_order, &c->b_trace, &c->b_trace_off, &c->b_tr, &c->b_work, &c->b_prep, &c->b_bloom,
		&c->b_mask_pb, &c->b_mask_scale, &c->b_mask_pos, &c->b_mask_pos2, &c->b_mask_cov, &c->b_mask_flag, &c->b_mask_seqs, &c->b_mask_zinv, &c->b_mask_need };
	for (DevBuf* b : bufs) b->release();
	for (auto& f : c->block_pool) { cudaFree(f.letters); cudaFree(f.bias); cudaFree(f.limits); cudaFree(f.soft); f.idx.release(); }
	c->b_hits_out.release();
	c->own_index.release();
	for (int k = 0; k <= c->params.n_shapes; ++k) if (c->d_matcher[k]) cudaFree(c->d_matcher[k]);
	if (c->d_s16_table) cudaFree(c->d_s16_table);
	dmnd_comm_destroy(c);
	if (c->d_params) cudaFree(c->d_params);
	if (c->h_pinned) cudaFreeHost(c->h_pinned);
	cudaEventDestroy(c->ev_a); cudaEventDestroy(c->ev_b); cudaEventDestroy(c->ev_sync);
	cudaStreamDestroy(c->stream);
	cudaStreamDestroy(c->copy_stream);
	cudaEventDestroy(c->ev_copy);
	delete c;
}

static int block_alloc(dmnd_ctx* ctx, size_t raw_len, const int64_t* limits, uint32_t nseq, const char* who, dmnd_block** out, size_t* padded_out) {
	if (raw_len < 2 * DMND_PERIMETER_PADDING || limits[0] != DMND_PERIMETER_PADDING || (size_t)limits[nseq] + DMND_PERIMETER_PADDING != raw_len) {
		set_error((std::string(who) + ": not a block image (256 B padding + sequences + 256 B padding)").c_str());
		return 1;
	}
	dmnd_block* b = new dmnd_block();
	b->raw_len = raw_len; b->nseq = nseq;
	b->h_limits.assign(limits, limits + nseq + 1);
	const size_t padded = (raw_len + 63) & ~(size_t)63;  // 16 B vector loads may touch the tail
	// reuse the device memory of a freed block when one is large enough (steady-state uploads allocate nothing)
	for (size_t k = 0; k < ctx->block_pool.size(); ++k) {
		const dmnd_ctx::FreeBlock& f = ctx->block_pool[k];
		if (f.cap_bytes >= padded + 64 && f.cap_seqs >= (size_t)nseq + 1 && f.cap_bytes <= 2 * (padded + 64) + (1 << 20)) {
			b->letters = f.letters; b->bias = f.bias; b->limits = f.limits; b->soft = f.soft; b->cap_bytes = f.cap_bytes; b->cap_seqs = f.cap_seqs;
			b->idx = f.idx; b->idx.valid = false;  // keeps the index buffers' capacity, not their contents
			ctx->block_pool.erase(ctx->block_pool.begin() + (ptrdiff_t)k);
			break;
		}
	}
	if (!b->letters) {
		b->cap_bytes = padded + 64; b->cap_seqs = (size_t)nseq + 1;
		if (cudaMalloc(&b->letters, b->cap_bytes) != cudaSuccess || cudaMalloc(&b->bias, b->cap_bytes) != cudaSuccess
		    || cudaMalloc(&b->limits, sizeof(int64_t) * b->cap_seqs) != cudaSuccess
		    || cudaMalloc(&b->soft, b->cap_bytes / 8 + 16) != cudaSuccess) {
			cudaFree(b->letters); cudaFree(b->bias); cudaFree(b->limits); cudaFree(b->soft); delete b;
			set_error((std::string(who) + ": cudaMalloc failed").c_str());
			return 1;
		}
	}
	*out = b; *padded_out = padded;
	return 0;
}

int dmnd_block_geometry(const dmnd_block* b, size_t* raw_len, uint32_t* nseq) { *raw_len = b->raw_len; *nseq = b->nseq; return 0; }
int dmnd_block_download_limits(dmnd_ctx* ctx, const dmnd_block* b, int64_t* limits, size_t count) {
	(void)ctx;
	if (count != (size_t)b->nseq + 1) { set_error("dmnd_block_download_limits: count must be nseq + 1"); return 1; }
	std::memcpy(limits, b->h_limits.data(), count * sizeof(int64_t));
	return 0;
}

// A block of the given geometry with nothing in it yet (dmnd_block_broadcast fills it from another rank): delimiters, zero bias, empty soft table.
int dmnd_block_alloc_empty(dmnd_ctx* ctx, size_t raw_len, uint32_t nseq, dmnd_block** out) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	if (raw_len < 2 * DMND_PERIMETER_PADDING) { set_error("dmnd_block_alloc_empty: not a block image"); return 1; }
	std::vector<int64_t> lim((size_t)nseq + 1, (int64_t)DMND_PERIMETER_PADDING);
	lim[nseq] = (int64_t)(raw_len - DMND_PERIMETER_PADDING);  // placeholder limits that pass block_alloc's shape check; overwritten by the broadcast
	dmnd_block* b = nullptr;
	size_t padded = 0;
	if (block_alloc(ctx, raw_len, lim.data(), nseq, "dmnd_block_alloc_empty", &b, &padded)) return 1;
	DMND_CUDA_CHECK(cudaMemsetAsync(b->letters, DMND_DELIMITER, padded + 64, ctx->stream));
	DMND_CUDA_CHECK(cudaMemsetAsync(b->bias, 0, padded + 64, ctx->stream));
	DMND_CUDA_CHECK(cudaMemsetAsync(b->soft, 0, b->cap_bytes / 8 + 16, ctx->stream));
	DMND_CUDA_CHECK(stream_wait(ctx, ctx->stream));
	*out = b;
	return 0;
}

int dmnd_block_upload(dmnd_ctx* ctx, const int8_t* letters, size_t raw_len, const int64_t* limits, uint32_t nseq, dmnd_block** out) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	dmnd_block* b = nullptr;
	size_t padded = 0;
	if (block_alloc(ctx, raw_len, limits, nseq, "dmnd_block_upload", &b, &padded)) return 1;
	PhaseTimer t(ctx, PH_H2D);
	DMND_CUDA_CHECK(cudaMemsetAsync(b->letters, DMND_DELIMITER, padded + 64, ctx->stream));
	DMND_CUDA_CHECK(cudaMemcpyAsync(b->letters, letters, raw_len, cudaMemcpyHostToDevice, ctx->stream));
	DMND_CUDA_CHECK(cudaMemcpyAsync(b->limits, limits, sizeof(int64_t) * ((size_t)nseq + 1), cudaMemcpyHostToDevice, ctx->stream));
	DMND_CUDA_CHECK(cudaMemsetAsync(b->bias, 0, padded + 64, ctx->stream));
	DMND_CUDA_CHECK(cudaMemsetAsync(b->soft, 0, b->cap_bytes / 8 + 16, ctx->stream));
	t.stop();
	DMND_CUDA_CHECK(stream_wait(ctx, ctx->stream));  // the copy is complete on return, independent of the timer
	ctx->h2d_bytes += raw_len + sizeof(int64_t) * ((size_t)nseq + 1);
	*out = b;
	return 0;
}

int dmnd_block_upload_ranges(dmnd_ctx* ctx, const int8_t* letters, size_t raw_len, const int64_t* limits, uint32_t nseq,
                             const uint32_t* cuts, int nranges, dmnd_block** out) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	if (nranges < 1 || nranges > 64 || cuts[0] != 0 || cuts[nranges] != nseq) { set_error("dmnd_block_upload_ranges: cuts must run from 0 to nseq in 1..64 ranges"); return 1; }
	for (int k = 0; k < nranges; ++k) if (cuts[k] > cuts[k + 1]) { set_error("dmnd_block_upload_ranges: cuts not ascending"); return 1; }
	dmnd_block* b = nullptr;
	size_t padded = 0;
	if (block_alloc(ctx, raw_len, limits, nseq, "dmnd_block_upload_ranges", &b, &padded)) return 1;
	cudaStream_t cs = ctx->copy_stream;
	// order the copy stream behind whatever the compute streams still do with a recycled buffer: block_free synchronised them
	DMND_CUDA_CHECK(cudaMemsetAsync(b->letters, DMND_DELIMITER, padded + 64, cs));
	DMND_CUDA_CHECK(cudaMemsetAsync(b->bias, 0, padded + 64, cs));
	DMND_CUDA_CHECK(cudaMemsetAsync(b->soft, 0, b->cap_bytes / 8 + 16, cs));
	DMND_CUDA_CHECK(cudaMemcpyAsync(b->limits, limits, sizeof(int64_t) * ((size_t)nseq + 1), cudaMemcpyHostToDevice, cs));
	b->range_ready.resize((size_t)nranges, nullptr);
	b->range_cuts.assign(cuts, cuts + nranges + 1);
	for (int k = 0; k < nranges; ++k) {
		// range k: from its first sequence (the head padding with range 0) to 256 bytes past its last one: the seed windows,
		// fingerprints and left-most filter of a range read a little beyond its end (into the next range's first letters)
		const size_t lo = k == 0 ? 0 : (size_t)limits[cuts[k]];
		const size_t hi = std::min(raw_len, (size_t)limits[cuts[k + 1]] + DMND_PERIMETER_PADDING);
		if (hi > lo) DMND_CUDA_CHECK(cudaMemcpyAsync(b->letters + lo, letters + lo, hi - lo, cudaMemcpyHostToDevice, cs));
		DMND_CUDA_CHECK(cudaEventCreateWithFlags(&b->range_ready[(size_t)k], cudaEventDisableTiming));
		DMND_CUDA_CHECK(cudaEventRecord(b->range_ready[(size_t)k], cs));
	}
	ctx->h2d_bytes += raw_len + sizeof(int64_t) * ((size_t)nseq + 1);
	*out = b;
	return 0;
}

int dmnd_block_range_wait(dmnd_ctx* ctx, const dmnd_block* b, uint32_t s_begin, uint32_t s_end) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	if (b->range_ready.empty() || s_begin >= s_end) return 0;  // uploaded synchronously: everything is there
	for (size_t k = 0; k < b->range_ready.size(); ++k)
		if (b->range_cuts[k] < s_end && b->range_cuts[k + 1] > s_begin)  // range k holds some of the sequences
			DMND_CUDA_CHECK(cudaStreamWaitEvent(ctx->stream, b->range_ready[k], 0));
	return 0;
}

void dmnd_block_free(dmnd_ctx* ctx, dmnd_block* b) {
	if (!b) return;
	cudaSetDevice(ctx->device);
	cudaStreamSynchronize(ctx->stream);
	for (dmnd_ctx* l : ctx->lanes) cudaStreamSynchronize(l->stream);
	cudaStreamSynchronize(ctx->copy_stream);
	for (cudaEvent_t e : b->range_ready) if (e) cudaEventDestroy(e);
	if (ctx->block_pool.size() < 4) ctx->block_pool.push_back(dmnd_ctx::FreeBlock{ b->letters, b->bias, b->limits, b->soft, b->cap_bytes, b->cap_seqs, b->idx });
	else { cudaFree(b->letters); cudaFree(b->bias); cudaFree(b->limits); cudaFree(b->soft); b->idx.release(); }
	delete b;
}

int dmnd_block_set_bias(dmnd_ctx* ctx, dmnd_block* b, const int8_t* bias, size_t raw_len) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	if (raw_len != b->raw_len) { set_error("dmnd_block_set_bias: length mismatch"); return 1; }
	PhaseTimer t(ctx, PH_H2D);
	if (bias) { DMND_CUDA_CHECK(cudaMemcpyAsync(b->bias, bias, raw_len, cudaMemcpyHostToDevice, ctx->stream)); ctx->h2d_bytes += raw_len; }
	else DMND_CUDA_CHECK(cudaMemsetAsync(b->bias, 0, raw_len, ctx->stream));
	t.stop();
	DMND_CUDA_CHECK(stream_wait(ctx, ctx->stream));  // the copy is complete on return, independent of the timer
	return 0;
}

int dmnd_block_build_index(dmnd_ctx* ctx, dmnd_block* b, int sid) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	if (sid < 0 || sid >= ctx->params.n_shapes) { set_error("dmnd_block_build_index: bad shape id"); return 1; }
	// FNV-1a over the parameters: an index is only reused by contexts with the same shapes / reduction / mode
	uint64_t ph = 1469598103934665603ull;
	for (size_t k = 0; k < sizeof ctx->params; ++k) { ph ^= ((const unsigned char*)&ctx->params)[k]; ph *= 1099511628211ull; }
	if (b->idx.valid && b->idx.sid == sid && b->idx.content_epoch == b->content_epoch && b->idx.params_hash == ph) return 0;  // resident block, unchanged: keep the index
	PhaseTimer t(ctx, PH_SEED);
	const int rc = build_ref_index(ctx, b, sid, b->idx);
	b->idx.content_epoch = b->content_epoch; b->idx.params_hash = ph;
	t.stop();
	DMND_CUDA_CHECK(stream_wait(ctx, ctx->stream));  // the copy is complete on return, independent of the timer
	return rc;
}

int dmnd_block_compute_bias_range(dmnd_ctx* ctx, dmnd_block* b, int mode, uint32_t s_begin, uint32_t s_end) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	if (mode != 0 && mode != 1) { set_error("dmnd_block_compute_bias: unknown mode"); return 1; }
	if (s_begin > s_end || s_end > b->nseq) { set_error("dmnd_block_compute_bias_range: sequence range out of bounds"); return 1; }
	if (s_begin == s_end) return 0;
	PhaseTimer t(ctx, PH_SEED);
	const size_t lo = (size_t)b->h_limits[s_begin], hi = (size_t)b->h_limits[s_end];
	DMND_CUDA_CHECK(cudaMemsetAsync(b->bias + lo, 0, hi - lo, ctx->stream));
	if (mode == 1) {
		const uint32_t n = s_end - s_begin;
		hauser_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(b->letters, b->limits + s_begin, n, ctx->d_params, b->bias);
		++ctx->launches;
		DMND_CUDA_CHECK(cudaGetLastError());
	}
	t.stop();
	DMND_CUDA_CHECK(stream_wait(ctx, ctx->stream));  // the copy is complete on return, independent of the timer
	return 0;
}

int dmnd_block_compute_bias(dmnd_ctx* ctx, dmnd_block* b, int mode) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	if (mode != 0 && mode != 1) { set_error("dmnd_block_compute_bias: unknown mode"); return 1; }
	DMND_CUDA_CHECK(cudaMemsetAsync(b->bias, 0, b->raw_len, ctx->stream));  // padding included
	return dmnd_block_compute_bias_range(ctx, b, mode, 0, b->nseq);
}

int dmnd_block_download_bias(dmnd_ctx* ctx, const dmnd_block* b, int8_t* bias, size_t raw_len) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	if (raw_len != b->raw_len) { set_error("dmnd_block_download_bias: length mismatch"); return 1; }
	DMND_CUDA_CHECK(cudaMemcpyAsync(bias, b->bias, raw_len, cudaMemcpyDeviceToHost, ctx->stream));
	DMND_CUDA_CHECK(stream_wait(ctx, ctx->stream));
	ctx->d2h_bytes += raw_len;
	return 0;
}

int dmnd_block_download_bias_async(dmnd_ctx* ctx, const dmnd_block* b, int8_t* bias, size_t raw_len) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	if (raw_len != b->raw_len) { set_error("dmnd_block_download_bias_async: length mismatch"); return 1; }
	// the copy stream waits for everything issued so far on the compute stream (the bias kernel), then runs beside it
	DMND_CUDA_CHECK(cudaEventRecord(ctx->ev_copy, ctx->stream));
	DMND_CUDA_CHECK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_copy, 0));
	DMND_CUDA_CHECK(cudaMemcpyAsync(bias, b->bias, raw_len, cudaMemcpyDeviceToHost, ctx->copy_stream));
	ctx->d2h_bytes += raw_len;
	return 0;
}

int dmnd_copy_wait(dmnd_ctx* ctx) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	DMND_CUDA_CHECK(stream_wait(ctx, ctx->copy_stream));
	return 0;
}

void* dmnd_host_alloc(dmnd_ctx* ctx, size_t bytes) {
	cudaSetDevice(ctx->device);
	void* p = nullptr;
	if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) { set_error("dmnd_host_alloc: cudaMallocHost failed"); return nullptr; }
	return p;
}

void dmnd_host_free(dmnd_ctx* ctx, void* p) {
	cudaSetDevice(ctx->device);
	if (p) cudaFreeHost(p);
}

int dmnd_hits_xdrop(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, const dmnd_hits* h, int raw_xdrop, dmnd_segment* host, size_t cap) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	return hits_xdrop_impl(ctx, query, ref, h, raw_xdrop, host, nullptr, cap);
}

int dmnd_hits_xdrop_sites(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, const dmnd_hits* h, int raw_xdrop, dmnd_segment* host,
                          dmnd_hit_site* sites, size_t cap) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	return hits_xdrop_impl(ctx, query, ref, h, raw_xdrop, host, sites, cap);
}

int dmnd_hits_gapped_filter(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, const dmnd_hits* h, uint8_t* pass, size_t cap) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	return hits_gapped_filter_impl(ctx, query, ref, h, pass, cap);
}

int dmnd_block_download_letters(dmnd_ctx* ctx, const dmnd_block* b, int8_t* letters, size_t raw_len) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	if (raw_len != b->raw_len) { set_error("dmnd_block_download_letters: length mismatch"); return 1; }
	DMND_CUDA_CHECK(cudaMemcpyAsync(letters, b->letters, raw_len, cudaMemcpyDeviceToHost, ctx->stream));
	DMND_CUDA_CHECK(stream_wait(ctx, ctx->stream));
	ctx->d2h_bytes += raw_len;
	return 0;
}

int dmnd_debug_block_soft(dmnd_ctx* ctx, const dmnd_block* b, uint8_t* out, size_t raw_len) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	if (raw_len != b->raw_len) { set_error("dmnd_debug_block_soft: length mismatch"); return 1; }
	std::vector<uint32_t> bits(raw_len / 32 + 1);
	DMND_CUDA_CHECK(cudaMemcpyAsync(bits.data(), b->soft, bits.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
	DMND_CUDA_CHECK(stream_wait(ctx, ctx->stream));
	for (size_t p = 0; p < raw_len; ++p) out[p] = b->has_soft ? (uint8_t)((bits[p >> 5] >> (p & 31)) & 1u) : 0;
	return 0;
}

int dmnd_debug_ref_index(dmnd_ctx* ctx, const dmnd_block* ref, int sid, uint64_t* keys, uint32_t* locs, size_t cap, size_t* n) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	if (sid < 0 || sid >= ctx->params.n_shapes) { set_error("dmnd_debug_ref_index: bad shape id"); return 1; }
	dmnd_cuda::RefIndex& ix = ctx->own_index;
	ctx->own_index_block = nullptr;  // the private index is rebuilt here without a record of its block: the next search rebuilds it again
	if (dmnd_cuda::build_ref_index(ctx, ref, sid, ix)) return 1;
	*n = (size_t)ix.nref;
	if (cap < *n) { set_error("dmnd_debug_ref_index: buffer too small"); return 1; }
	if (*n) {
		DMND_CUDA_CHECK(cudaMemcpyAsync(keys, ix.keys.p, *n * 8, cudaMemcpyDeviceToHost, ctx->stream));
		DMND_CUDA_CHECK(cudaMemcpyAsync(locs, ix.locs.p, *n * 4, cudaMemcpyDeviceToHost, ctx->stream));
		DMND_CUDA_CHECK(stream_wait(ctx, ctx->stream));
	}
	return 0;
}

int dmnd_debug_left_most(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, int sid, int chunk, uint32_t qloc, uint32_t sloc, unsigned long long* out30) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	if (sid < 0 || sid >= ctx->params.n_shapes || chunk < 0) { set_error("dmnd_debug_left_most: bad shape id / chunk"); return 1; }
	return dmnd_cuda::debug_left_most_impl(ctx, query, ref, sid, chunk, qloc, sloc, out30);
}

static int clear_range(dmnd_ctx* ctx, dmnd_block* b, size_t begin, size_t end) {
	if (end <= begin) return 0;
	const size_t threads = (end - (begin / 16) * 16 + 15) / 16;
	clear_seed_mask_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, ctx->stream>>>(b->letters, begin, end);
	++ctx->launches;
	DMND_CUDA_CHECK(cudaGetLastError());
	return 0;
}

int dmnd_block_clear_seed_mask(dmnd_ctx* ctx, dmnd_block* b) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	return clear_range(ctx, b, 0, b->raw_len);
}

int dmnd_block_clear_seed_mask_range(dmnd_ctx* ctx, dmnd_block* b, uint32_t q_begin, uint32_t q_end) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	if (q_begin > q_end || q_end > b->nseq) { set_error("dmnd_block_clear_seed_mask_range: bad range"); return 1; }
	return clear_range(ctx, b, (size_t)b->h_limits[q_begin], (size_t)b->h_limits[q_end]);
}

int dmnd_block_mask(dmnd_ctx* ctx, dmnd_block* b, int algo, uint32_t s_begin, uint32_t s_end, uint64_t* n_hard) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	return block_mask_impl(ctx, b, algo, s_begin, s_end, n_hard);
}
int dmnd_block_mask_fetch(dmnd_ctx* ctx, uint64_t* positions, size_t cap) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	return block_mask_fetch_impl(ctx, positions, cap);
}

int dmnd_search_shape(dmnd_ctx* ctx, dmnd_block* query, const dmnd_block* ref, int sid, dmnd_hits** out, dmnd_stage_counters* counters) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	return search_shape_impl(ctx, query, ref, sid, 0, query->nseq, out, counters);
}

int dmnd_search_shape_range(dmnd_ctx* ctx, dmnd_block* query, const dmnd_block* ref, int sid, uint32_t q_begin, uint32_t q_end,
                            dmnd_hits** out, dmnd_stage_counters* counters) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	if (q_begin > q_end || q_end > query->nseq) { set_error("dmnd_search_shape_range: bad query range"); return 1; }
	return search_shape_impl(ctx, query, ref, sid, q_begin, q_end, out, counters);
}

size_t dmnd_hits_count(const dmnd_hits* h) { return h->n; }

int dmnd_hits_download(dmnd_ctx* ctx, const dmnd_hits* h, dmnd_hit* host, size_t cap) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	if (cap < h->n) { set_error("dmnd_hits_download: buffer too small"); return 1; }
	if (h->n == 0) return 0;
	PhaseTimer t(ctx, PH_D2H);
	DMND_CUDA_CHECK(cudaMemcpyAsync(host, h->d, h->n * sizeof(dmnd_hit), cudaMemcpyDeviceToHost, ctx->stream));
	t.stop();
	DMND_CUDA_CHECK(stream_wait(ctx, ctx->stream));  // the copy is complete on return, independent of the timer
	ctx->d2h_bytes += h->n * sizeof(dmnd_hit);
	return 0;
}

void dmnd_hits_free(dmnd_ctx* ctx, dmnd_hits* h) {
	if (!h) return;
	(void)ctx;
	delete h;  // the records live in the context's hit arena
}

int dmnd_banded_swipe(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, const dmnd_dp_problem* problems, size_t n, int mode,
                      dmnd_dp_result* results, uint8_t* transcripts, size_t transcript_cap) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	return banded_swipe_impl(ctx, query, ref, problems, nullptr, n, mode, results, transcripts, transcript_cap);
}

int dmnd_hits_chain(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, const dmnd_hits* h, int raw_xdrop, int band_slow, int max_targets, dmnd_chain_out* out) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	if (ctx->params.query_contexts > 1) { set_error("dmnd_hits_chain: one query context only"); return 1; }
	return hits_chain_impl(ctx, query, ref, h, raw_xdrop, band_slow, max_targets, out);
}
int dmnd_hits_chain_fetch(dmnd_ctx* ctx, dmnd_chain_query* queries, dmnd_dp_problem* problems, dmnd_hit* hits, dmnd_segment* segs, dmnd_hit_site* sites) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	return hits_chain_fetch_impl(ctx, queries, problems, hits, segs, sites);
}
int dmnd_banded_swipe_chained(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, size_t n, int mode, dmnd_dp_result* results, uint8_t* transcripts, size_t transcript_cap) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	if (n != ctx->chain_counts[1]) { set_error("dmnd_banded_swipe_chained: n is not the problem count of the last dmnd_hits_chain"); return 1; }
	return banded_swipe_impl(ctx, query, ref, nullptr, ctx->chain_probs, n, mode, results, transcripts, transcript_cap);
}

int dmnd_timing_fetch(dmnd_ctx* ctx, dmnd_timing* out, int flags) {
	std::memset(out, 0, sizeof *out);
	auto take = [&](dmnd_ctx* c) {
		out->seed_ms += c->phase_ms[PH_SEED]; out->dp_score_ms += c->phase_ms[PH_DP_SCORE]; out->dp_trace_ms += c->phase_ms[PH_DP_TRACE];
		out->h2d_ms += c->phase_ms[PH_H2D]; out->d2h_ms += c->phase_ms[PH_D2H];
		out->launches += c->launches; out->h2d_bytes += c->h2d_bytes; out->d2h_bytes += c->d2h_bytes;
		out->dp_cells_score += c->dp_cells_score; out->dp_cells_trace += c->dp_cells_trace; out->dp_cells_padded += c->dp_cells_padded; out->dp_overflow_reruns += c->dp_overflows;
		if (flags & DMND_TIMING_RESET) {
			for (double& x : c->phase_ms) x = 0;
			c->launches = 0; c->h2d_bytes = 0; c->d2h_bytes = 0;
			c->dp_cells_score = c->dp_cells_trace = c->dp_cells_padded = 0; c->dp_overflows = 0;
		}
	};
	take(ctx);
	if (!(flags & DMND_TIMING_THIS_CONTEXT))
		for (dmnd_ctx* l : ctx->lanes) take(l);
	return 0;
}

}  // extern "C"

