// pipeline.cpp -- P layer: one (query block, reference block) pass of blastp on top of the K layer.
//
// Host restatement of the reference's control flow around its two hot kernels, batched across queries so that every
// GPU launch sees the DP problems of ALL queries at once (the reference batches only within one query):
//   search/setup.cpp:306-309,338-402       seedp_bits, setup_search (sensitivity traits -> parameters)
//   run/double_indexed.cpp:102-252         run_ref_chunk: search_shape per shape, then align_queries
//   align/align.cpp:203-269                align_queries (sort by query, per-query extend)
//   align/load_hits.h:44-122               load_hits
//   align/extend.cpp:79-119,226-387        ranking_chunk_size, ranking_terminate, extend (chunk loop)
//   align/ungapped.cpp:62-118              ungapped_stage
//   align/gapped_score.cpp:41-72,107-246   band, add_dp_targets, round-1 align
//   align/gapped_final.cpp:64-158          round-2 align
//   align/culling.cpp:34-202               inner_culling, culling, append_hits, output_range
//   dp/dp.h:47-52,121-124                  banded_cols, cells
// Every per-query extend() is a small state machine (produce DP problems -> wait -> consume results), so the chunked
// ranking loop of the reference is replayed exactly while the DP itself runs in device-wide waves.
//
// Memory: a query's state is plain data; its variable-length lists live in the bump arena of the worker thread that
// owns the query (static block partition, so no list is ever touched by two threads), and every large buffer is kept
// in a process-wide workspace between calls -- a steady-state step performs no heap allocation and no page faults.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cfloat>
#include <climits>
#include <map>
#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>
#include "../../../include/dmnd_b200.h"
#include "chaining.h"
#include "range_cover.h"
#include "scoring.h"

namespace {

using namespace dmnd;
using Clock = std::chrono::steady_clock;
static double ms_since(Clock::time_point t0) { return std::chrono::duration<double, std::milli>(Clock::now() - t0).count(); }

// DMND_PROFILE=1: wall-clock of the host phases on stderr (development aid)
static Clock::time_point g_prof_epoch = Clock::now();  // start of the current dmnd_blastp call (timestamps of the laps)
struct Prof {
	bool on = std::getenv("DMND_PROFILE") != nullptr;
	int lane = -1;
	Clock::time_point t = Clock::now();
	void lap(const char* what) {
		if (!on) return;
		std::fprintf(stderr, "[dmnd profile] lane %2d %-34s %8.2f ms  (ends at %8.2f)\n", lane, what, ms_since(t), ms_since(g_prof_epoch));
		t = Clock::now();
	}
};

// CPUs this process may actually use: min(hardware threads, cgroup v2/v1 CFS quota).  Oversubscribing a quota-limited
// container (128 visible CPUs, 16 allowed) throttles every worker, so the pool is sized to the quota.
int effective_cpus() {
	int n = (int)std::thread::hardware_concurrency();
	if (n < 1) n = 1;
	auto read2 = [](const char* path, long long& a, long long& b) {
		FILE* f = std::fopen(path, "r");
		if (!f) return false;
		char s1[64] = { 0 }, s2[64] = { 0 };
		const int k = std::fscanf(f, "%63s %63s", s1, s2);
		std::fclose(f);
		if (k < 1 || std::strcmp(s1, "max") == 0) return false;
		a = std::atoll(s1); b = k > 1 ? std::atoll(s2) : 0;
		return true;
	};
	long long q = 0, per = 0;
	if (read2("/sys/fs/cgroup/cpu.max", q, per) && q > 0 && per > 0) n = std::min<long long>(n, std::max<long long>(1, (q + per - 1) / per));
	else {
		long long q1 = 0, p1 = 0, d = 0;
		if (read2("/sys/fs/cgroup/cpu/cpu.cfs_quota_us", q1, d) && q1 > 0 && read2("/sys/fs/cgroup/cpu/cpu.cfs_period_us", p1, d) && p1 > 0)
			n = std::min<long long>(n, std::max<long long>(1, (q1 + p1 - 1) / p1));
	}
	return n;
}

// ---- fork-join pool: threads persist between calls, run(f) executes f(t) for t in [0, T) ---------------------------
class Pool {
public:
	explicit Pool(int n) : n_(n) {
		for (int t = 1; t < n; ++t) th_.emplace_back([this] { loop(); });
	}
	~Pool() {
		{ std::lock_guard<std::mutex> l(m_); stop_ = true; ++gen_; }
		cv_.notify_all();
		for (auto& t : th_) t.join();
	}
	int size() const { return n_; }
	// Runs f(0) .. f(size() - 1), each once.  Tasks are claimed by whichever thread is free (the caller included) rather than
	// tied to one worker each: on a host shared with other processes a worker that is descheduled before it starts does not
	// hold up the call, another thread takes its task.  Callers index their outputs by the task, so results do not depend on
	// which thread ran it.
	// Lanes take turns: whoever has host work gets every worker; among waiting lanes the lowest id (the one furthest
	// along in the staggered pipeline) goes first.
	void run(const std::function<void(int)>& f, int prio = 0) {
		{
			std::unique_lock<std::mutex> l(turn_m_);
			waiting_.push_back(prio);
			turn_cv_.wait(l, [&] { return !busy_ && *std::min_element(waiting_.begin(), waiting_.end()) == prio; });
			busy_ = true;
			waiting_.erase(std::find(waiting_.begin(), waiting_.end(), prio));
		}
		// exceptions (std::bad_alloc from a growing list is the realistic one) are caught per thread, the first is rethrown here after
		// every worker has finished with `f` and the turn has been handed on -- a throw must neither leave workers inside the
		// caller's std::function nor the other lanes blocked on the turn
		std::exception_ptr first;
		auto guarded = [&](int t) { try { f(t); } catch (...) { std::lock_guard<std::mutex> l(err_m_); if (!first) first = std::current_exception(); } };
		const std::function<void(int)> g(guarded);
		if (n_ == 1) g(0);
		else {
			uint64_t gen;
			{
				std::lock_guard<std::mutex> l(m_);
				fn_ = &g; gen = ++gen_;
				left_.store(n_, std::memory_order_relaxed);
				claim_.store(gen << 32, std::memory_order_release);
			}
			cv_.notify_all();
			work(gen, g);
			std::unique_lock<std::mutex> l(m_);
			done_.wait(l, [this] { return left_.load(std::memory_order_acquire) == 0; });
		}
		{ std::lock_guard<std::mutex> l(turn_m_); busy_ = false; }
		turn_cv_.notify_all();
		if (first) std::rethrow_exception(first);
	}
private:
	// claim_ = (generation << 32) | next task.  A claim only succeeds for the generation the thread read fn_ with, and run() returns
	// only after every task of its generation has finished, so fn_ is alive whenever a claimed task calls it.
	void work(uint64_t gen, const std::function<void(int)>& f) {
		for (;;) {
			uint64_t c = claim_.load(std::memory_order_acquire);
			if ((c >> 32) != (gen & 0xffffffffull) || (c & 0xffffffffull) >= (uint64_t)n_) return;
			if (!claim_.compare_exchange_weak(c, c + 1, std::memory_order_acq_rel)) continue;
			f((int)(c & 0xffffffffull));
			if (left_.fetch_sub(1, std::memory_order_acq_rel) == 1) { std::lock_guard<std::mutex> l(m_); done_.notify_one(); }
		}
	}
	void loop() {
		uint64_t seen = 0;
		for (;;) {
			const std::function<void(int)>* f;
			{
				std::unique_lock<std::mutex> l(m_);
				cv_.wait(l, [&] { return gen_ != seen; });
				seen = gen_;
				if (stop_) return;
				f = fn_;
			}
			work(seen, *f);
		}
	}
	int n_;
	std::vector<std::thread> th_;
	std::mutex m_, turn_m_, err_m_;
	std::condition_variable cv_, done_, turn_cv_;
	std::vector<int> waiting_;
	bool busy_ = false;
	const std::function<void(int)>* fn_ = nullptr;
	std::atomic<uint64_t> claim_{ 0 };
	std::atomic<int> left_{ 0 };
	uint64_t gen_ = 0;
	bool stop_ = false;
};

// ---- bump arena ---------------------------------------------------------------------------------------------------
class Arena {
public:
	void reset() { cur_ = 0; used_ = 0; }
	void* alloc(size_t bytes) {
		bytes = (bytes + 15) & ~(size_t)15;
		while (cur_ < blocks_.size() && used_ + bytes > sizes_[cur_]) { ++cur_; used_ = 0; }
		if (cur_ == blocks_.size()) {
			const size_t sz = std::max<size_t>(bytes, (size_t)4 << 20);
			blocks_.emplace_back(new char[sz]);
			sizes_.push_back(sz);
		}
		void* p = blocks_[cur_].get() + used_;
		used_ += bytes;
		return p;
	}
private:
	std::vector<std::unique_ptr<char[]>> blocks_;
	std::vector<size_t> sizes_;
	size_t cur_ = 0, used_ = 0;
};

template<typename T>
struct List {  // trivially-copyable elements only
	T* p = nullptr;
	uint32_t n = 0, cap = 0;
	void reserve(Arena& a, uint32_t c) {
		if (c <= cap) return;
		T* np = (T*)a.alloc(sizeof(T) * c);
		if (n) std::memcpy(np, p, sizeof(T) * n);
		p = np; cap = c;
	}
	void push(Arena& a, const T& v) {
		if (n == cap) reserve(a, cap ? cap * 2 : 4);
		p[n++] = v;
	}
	T* begin() const { return p; }
	T* end() const { return p + n; }
	void clear() { n = 0; }
};

struct SeedHit { int i, j, score; dmnd_segment seg; uint8_t gf;  /* gf: the hit passes the gapped filter (modes that have one) */ uint8_t frame;  /* query context of the hit (0 for blastp), align/load_hits.h:86 */ bool operator<(const SeedHit& x) const { const int d1 = i - j, d2 = x.i - x.j; return d1 < d2 || (d1 == d2 && j < x.j); } };
struct TargetScore { uint32_t target; uint16_t score; bool operator<(const TargetScore& x) const { return score > x.score || (score == x.score && target < x.target); } };

struct HspLite { int score; double evalue; int d_begin, d_end; uint32_t ctx;  /* query block id of the frame that aligned (= the query for blastp) */ };
inline bool hsp_less(const HspLite& a, const HspLite& b) {  // basic/match.h:199-202 (query_source_range.begin_ is 0 in round 1)
	return a.score > b.score || (a.score == b.score && a.d_begin < b.d_begin);
}
struct Target {  // align/target.h:83-144 after inner_culling (max_hsps == 1): only the best HSP is kept
	uint32_t block_id; int tlen; int filter_score; double filter_evalue; HspLite hsp; bool has_hsp;
	uint32_t hsp_prob;  // fused queries: index (within the query's problem slice) of the problem that produced `hsp`
	static bool comp_score(const Target& t, const Target& u) { return t.filter_score > u.filter_score || (t.filter_score == u.filter_score && t.block_id < u.block_id); }  // align/target.h:128-130
	static bool comp_evalue(const Target& t, const Target& u) {
		return t.filter_evalue < u.filter_evalue || (t.filter_evalue == u.filter_evalue && (t.filter_score > u.filter_score || (t.filter_score == u.filter_score && t.block_id < u.block_id)));
	}
};
struct Match {  // align/extend.h:36-70
	uint32_t target_block_id; int tlen; int filter_score; double filter_evalue; bool has_hsp; HspLite h; dmnd_dp_result r;
	uint64_t tr_off; uint32_t tr_len;  // into the owner thread's transcript buffer
	uint32_t end_frame;                // frameshift mode: 1 + context offset (0..5) of the frame the alignment ends in; 0 otherwise
	static bool cmp_score(const Match& m, const Match& n) { return m.filter_score > n.filter_score || (m.filter_score == n.filter_score && m.target_block_id < n.target_block_id); }  // align/extend.h:50-52
	static bool cmp_evalue(const Match& m, const Match& n) {
		return m.filter_evalue < n.filter_evalue || (m.filter_evalue == n.filter_evalue && (m.filter_score > n.filter_score || (m.filter_score == n.filter_score && m.target_block_id < n.target_block_id)));
	}
};

int band_for(int len, bool slow) {  // Extension::band, align/gapped_score.cpp:41-72
	if (!slow) {  // Mode::BANDED_FAST
		if (len < 50) return 12;
		if (len < 100) return 16;
		if (len < 250) return 30;
		if (len < 350) return 40;
		return 64;
	}
	if (len < 50) return 15;  // Mode::BANDED_SLOW
	if (len < 100) return 20;
	if (len < 150) return 30;
	if (len < 200) return 50;
	if (len < 250) return 60;
	if (len < 350) return 100;
	if (len < 500) return 120;
	return 150;
}
inline int banded_cols(int qlen, int tlen, int d_begin, int d_end) {  // dp/dp.h:47-52
	const int pos = std::max(d_end - 1, 0) - (d_end - 1);
	return std::min(qlen - 1 - d_begin, tlen - 1) + 1 - pos;
}

// Host view of a block whose letters were hard-masked on the device (dmnd_block_mask): the caller's letter image stays
// const; sequences that contain masked letters get a patched private copy (with the delimiter on either side, as the
// x-drop and chaining loops expect), every other sequence is read in place.  Read-only after build().
struct PatchSet {
	std::vector<uint64_t> bits;      // one bit per sequence: has a patched copy
	std::vector<uint32_t> ids;       // ascending sequence ids with a copy
	std::vector<size_t> off;         // start of the copy (its leading delimiter) in `arena`
	std::vector<int8_t> arena;
	bool empty() const { return ids.empty(); }
	// pos[0..n): ascending offsets of masked letters in the block image; [s_begin, s_end) = the sequences they can lie in
	void build(const int8_t* letters, const int64_t* limits, uint32_t nseq, uint32_t s_begin, uint32_t s_end, const uint64_t* pos, size_t n) {
		bits.assign(((size_t)nseq + 63) / 64, 0); ids.clear(); off.clear(); arena.clear();
		const int64_t* lb = limits + s_begin;
		for (size_t k = 0; k < n;) {
			const uint32_t sid = (uint32_t)(std::upper_bound(lb, limits + s_end + 1, (int64_t)pos[k]) - limits) - 1;
			const int64_t b = limits[sid], e = limits[sid + 1];  // [b, e - 1) letters, e - 1 = delimiter
			const size_t o = arena.size();
			arena.resize(o + (size_t)(e - b) + 1);
			std::memcpy(arena.data() + o, letters + b - 1, (size_t)(e - b) + 1);
			for (; k < n && (int64_t)pos[k] < e; ++k) arena[o + 1 + (size_t)((int64_t)pos[k] - b)] = MASK_LETTER;
			bits[sid >> 6] |= (uint64_t)1 << (sid & 63);
			ids.push_back(sid); off.push_back(o);
			lb = limits + sid + 1;
		}
	}
	const int8_t* find(uint32_t sid) const {  // patched copy of the sequence, or nullptr
		if (bits.empty() || !((bits[sid >> 6] >> (sid & 63)) & 1)) return nullptr;
		const size_t k = (size_t)(std::lower_bound(ids.begin(), ids.end(), sid) - ids.begin());
		return arena.data() + off[k] + 1;
	}
};

struct Env {
	const Scoring* sc;
	const int8_t *q_letters, *r_letters;
	const PatchSet *q_patch = nullptr, *r_patch = nullptr;  // hard-masked sequences (dmnd_blastp with masking); null = read in place
	bool band_slow = false;      // Extension::Mode::BANDED_SLOW band table (align/extend.cpp:62-75, gapped_score.cpp:41-72)
	double ranking_letters = 2e9; // ranking_chunk_size's default_letters (align/extend.cpp:86)
	bool gapped_filter = false;  // Extension::gapped_filter before the ungapped stage (align/extend.cpp:205-214)
	int n_shapes = 1;   // shapes of the sensitivity mode (search/setup.cpp:80-304): one dmnd_search_shape per shape
	int mask_algo = 0;  // DMND_MASK_* bits a lane applies to its own query range before searching (0: blocks arrive masked)
	uint32_t contexts = 1;  // align_mode.query_contexts: 6 = blastx, the query block holds the six frames of every query back to back
	int frame_shift = 0;    // config.frame_shift: > 0 = frameshift alignment mode, the legacy extension pipeline (align/align.cpp:168-172)
	bool range_culling = false; double range_cover = 50.0;  // config.query_range_culling / query_range_cover (frameshift mode only, basic/config.cpp:824-825)
	const int8_t* qseq(uint32_t q) const { const int8_t* p = q_patch ? q_patch->find(q) : nullptr; return p ? p : q_letters + q_limits[q]; }
	const int8_t* rseq(uint32_t t) const { const int8_t* p = r_patch ? r_patch->find(t) : nullptr; return p ? p : r_letters + r_limits[t]; }
	const int64_t *q_limits, *r_limits;
	uint32_t nq, nr;
	int64_t ref_letters;
	int max_target_seqs;  // cfg.max_target_seqs: -k, or "all" (INT_MAX) for -k 0 (output/output_format.cpp:236-245)
	double top = -1.0;    // --top (config.toppercent): >= 0 = report the targets within this percentage of the best bit score; -1 = not given
	int outer_limit;      // config.max_target_seqs_ as given (0 for -k 0): the bound of extend()'s outer loop (align/extend.cpp:336)
	double max_evalue;
	double min_bit_score = 0.0;  // --min-score (config.min_bit_score): replaces the e-value bound of ScoreMatrix::report_cutoff (stats/score_matrix.cpp:234-239)
	bool report_cutoff(int score, double evalue) const { return min_bit_score != 0.0 ? sc->bitscore(score) >= min_bit_score : evalue <= max_evalue; }
	bool hauser, want_transcript;
	bool fuse;  // see Driver::start
	// The bridge from hits to DP problems runs on the device (dmnd_hits_chain) for single-shape blastp without a gapped filter: the hits
	// never come to the host, the round-1 problem list of every query with <= 64 targets is produced and aligned in HBM, and only
	// queries with ranking chunks (or pairs beyond the device code's capacities) take the host code.
	bool bridge = false;
	// --id / --query-cover / --subject-cover (config.min_id, query_cover, subject_cover): with any of them set the reference only SORTS the
	// targets after round 1 (first_round_culling = !have_filters || --top, align/extend.cpp:94-96,288) and runs round 2 in steps
	double min_id = 0.0, query_cover = 0.0, subject_cover = 0.0, approx_min_id = 0.0;
	bool have_filters = false, first_round_culling = true;
	double min_length_ratio = 0.0;  // Search::Config::min_length_ratio (run/config.cpp:156-164)
	const uint32_t* self_targets = nullptr;  // --no-self-hits: per query (source query for translated searches) the target whose HSP Match::apply_filters removes
	int qlen(uint32_t q) const { return (int)(q_limits[q + 1] - q_limits[q] - 1); }
	int tlen(uint32_t t) const { return (int)(r_limits[t + 1] - r_limits[t] - 1); }
};

template<typename It>
It output_range(It begin, It end, const Env& e) {  // align/culling.cpp:90-109
	if (end <= begin) return begin;
	It i = begin;
	if (i->filter_evalue == DBL_MAX) return begin;
	if (e.top >= 0.0) {  // --top: everything within `top` percent of the best bit score
		const double cutoff = std::max((1.0 - e.top / 100.0) * e.sc->bitscore(begin->filter_score), 1.0);
		while (i < end && e.sc->bitscore(i->filter_score) >= cutoff) ++i;
		return i;
	}
	i += std::min<ptrdiff_t>((ptrdiff_t)e.max_target_seqs, end - begin);
	while (--i > begin && i->filter_evalue == DBL_MAX);
	++i;
	return i;
}

enum Phase : uint8_t { PH_ROUND1_PRODUCE, PH_ROUND1_CONSUME, PH_ROUND2_PRODUCE, PH_ROUND2_CONSUME, PH_DONE };

struct QueryState {
	uint32_t qid;  // block id of the query's first context (the query itself for blastp)
	int qlen;      // length of that context (query_seq[0].length() in the reference)
	Phase phase;
	bool new_hits_ev;
	bool fused;
	bool bridged;  // its round-1 problems came from dmnd_hits_chain (no SeedHitList on the host)
	// SeedHitList (align/target.h:160-165): slices of the owner thread's flat arrays
	uint32_t sh_off, tgt_off, n_targets;  // hit_begin[tgt_off + k] (n_targets + 1 entries), block ids / scores [ts_off..]
	uint32_t ts_off;
	// extend() loop state (align/extend.cpp:259-336)
	int64_t chunk_size, i0, i1;
	int tail_score, previous_tail_score;
	List<Target> aligned_targets, r1;
	List<Match> matches, r2;
	List<uint32_t> prob_target;  // per DP problem in flight: index into r1 / r2
	uint32_t r2_it, r2_begin, r2_prev;  // round 2 in steps (filters): next target of aligned_targets, first match of this step, matches before the round
	size_t prob_begin;           // offset in the owner thread's problem list of this wave
	uint32_t prob_count;
};

struct ThreadCtx {
	Arena arena;
	std::vector<SeedHit> seed_hits;
	std::vector<uint32_t> hit_begin, target_block_ids;
	std::vector<TargetScore> target_scores;
	std::vector<dmnd_dp_problem> p1, p2;
	std::vector<uint8_t> trbuf;
	// scratch
	std::vector<SeedHit> hits;
	std::vector<Segment> segs;
	std::vector<Chain> chains;
	std::vector<int8_t> cbs;
	std::vector<Target> tmp_targets;
	std::vector<uint32_t> unaligned;  // queries of this thread that had seed hits but no alignment
	uint64_t cells1 = 0, cells2 = 0, n_targets = 0, n_matches = 0, n_aligned = 0, n_extended = 0;
	uint64_t fused_r1 = 0, fused_r2 = 0, fused_r1_wave = 0;  // fused queries: round-1 problems traced, round-2 problems answered from them
	void reset() {
		arena.reset(); seed_hits.clear(); hit_begin.clear(); target_block_ids.clear(); target_scores.clear();
		p1.clear(); p2.clear(); trbuf.clear(); unaligned.clear(); cells1 = cells2 = n_targets = n_matches = n_aligned = n_extended = 0; fused_r1 = fused_r2 = fused_r1_wave = 0;
	}
};

// Grow-only plain host buffer WITHOUT value initialisation (std::vector::resize would memset tens of MB on one thread);
// kept alive between calls so that steady-state steps touch no fresh pages.
template<typename T> struct RawBuf {
	T* p = nullptr;
	size_t n = 0, cap = 0;
	RawBuf() = default;
	RawBuf(const RawBuf&) = delete;
	RawBuf& operator=(const RawBuf&) = delete;
	~RawBuf() { std::free(p); }
	void resize(size_t count) {
		if (count > cap) {
			std::free(p);
			cap = count + count / 8 + 4096;
			p = static_cast<T*>(std::malloc(cap * sizeof(T)));
			if (!p) { cap = n = 0; throw std::bad_alloc(); }
		}
		n = count;
	}
	T* data() { return p; }
	const T* data() const { return p; }
	size_t size() const { return n; }
	T& operator[](size_t i) { return p[i]; }
	const T& operator[](size_t i) const { return p[i]; }
};

// Grow-only page-locked host buffer (dmnd_host_alloc): device<->host copies of hits, DP problems, results and
// transcripts run as real DMA at link speed instead of staged pageable copies.  Contents are not preserved by resize().
template<typename T> struct HostBuf {
	T* p = nullptr;
	size_t n = 0, cap = 0;
	int resize(dmnd_ctx* ctx, size_t count) {
		if (count > cap) {
			if (p) dmnd_host_free(ctx, p);
			cap = count + count / 4 + 1024;
			p = static_cast<T*>(dmnd_host_alloc(ctx, cap * sizeof(T)));
			if (!p) { cap = n = 0; return 1; }
		}
		n = count;
		return 0;
	}
	T* data() { return p; }
	const T* data() const { return p; }
	size_t size() const { return n; }
	bool empty() const { return n == 0; }
	T& operator[](size_t i) { return p[i]; }
	const T& operator[](size_t i) const { return p[i]; }
	const T* begin() const { return p; }
	const T* end() const { return p + n; }
};

// Everything that survives between calls (buffers keep their capacity: no page faults in steady state).
struct Workspace {
	Pool* pool = nullptr;
	int lane = 0;  // turn priority on the shared pool
	void run(const std::function<void(int)>& f) { pool->run(f, lane); }
	std::vector<ThreadCtx> tc;
	HostBuf<dmnd_hit> hv;
	HostBuf<dmnd_segment> segv;
	HostBuf<dmnd_hit_site> sitev;
	struct HitSeg { dmnd_hit h; dmnd_segment s; dmnd_hit_site site; uint8_t gf; };
	std::vector<HitSeg> hs;
	// hits [b, e) of hv / segv / sitev / gfv as the records load_hits and legacy_init take (built in place in hs)
	HitSeg* gather(size_t b, size_t e) {
		for (size_t x = b; x < e; ++x) hs[x] = HitSeg{ hv[x], segv[x], sitev[x], gfv[x] };
		return hs.data() + b;
	}
	std::vector<size_t> qstart;
	std::vector<QueryState> qs;
	HostBuf<dmnd_dp_problem> p1, p2, cprobs;  // cprobs / cres / cq: dmnd_hits_chain's problem list, its results, its per-query records
	HostBuf<dmnd_dp_result> res1, res2, cres;
	HostBuf<dmnd_chain_query> cq;
	HostBuf<uint8_t> tr;
	RawBuf<dmnd_match> out_matches;   // lane output when several lanes run (copied into the result afterwards)
	RawBuf<uint8_t> out_transcripts;
	std::vector<dmnd_hit> acc_hits; std::vector<dmnd_segment> acc_segs; std::vector<dmnd_hit_site> acc_sites; std::vector<uint8_t> acc_gf;  // hits of all shapes (several shapes only)
	std::vector<uint8_t> gfv;         // per hit of hv: passes the gapped filter (1 where the mode has none)
	std::vector<uint64_t> mask_pos;   // letters of this lane's query range that dmnd_block_mask turned into X
	PatchSet q_patch;
};
// Process-wide: the worker pool and one workspace per lane.
struct Shared {
	std::mutex mtx;
	std::unique_ptr<Pool> pool;
	std::vector<std::unique_ptr<Workspace>> lanes;
	std::vector<uint64_t> r_mask_pos;  // reference-block counterpart of Workspace::mask_pos / q_patch
	PatchSet r_patch;
	void ensure(int threads, int nlanes) {
		if (!pool || pool->size() != threads) { pool.reset(new Pool(threads)); lanes.clear(); }
		while ((int)lanes.size() < nlanes) lanes.emplace_back(new Workspace());
		for (auto& w : lanes) { w->pool = pool.get(); if ((int)w->tc.size() != threads) { w->tc.clear(); w->tc.resize((size_t)threads); } }
	}
};
Shared& shared() { static Shared s; return s; }

struct Driver {
	dmnd_ctx* ctx;
	dmnd_block* qb;
	const dmnd_block* rb;
	Env env;
	Workspace* ws;
	int T;
	dmnd_run_stats stats;

	size_t nq_hit = 0;
	size_t block_begin(int t) const { return nq_hit * (size_t)t / (size_t)T; }

	void load_hits(QueryState& q, ThreadCtx& tc, Workspace::HitSeg* begin, Workspace::HitSeg* end);
	void start(QueryState& q, ThreadCtx& tc);
	void start_bridged(QueryState& q, ThreadCtx& tc, const dmnd_chain_query& cq, const dmnd_dp_problem* probs);
	void produce_round1(QueryState& q, ThreadCtx& tc);
	void produce_round2(QueryState& q, ThreadCtx& tc);
	void consume_round1(QueryState& q, ThreadCtx& tc, const dmnd_dp_problem* probs, const dmnd_dp_result* res);
	void consume_round2(QueryState& q, ThreadCtx& tc, const dmnd_dp_problem* probs, const dmnd_dp_result* res, const uint8_t* tr);
	void consume_fused(QueryState& q, ThreadCtx& tc, const dmnd_dp_problem* probs, const dmnd_dp_result* res, const uint8_t* tr);
	bool filtered_out(const QueryState& q, const Match& m) const;
	void take_round2_result(QueryState& q, ThreadCtx& tc, Match& m, const dmnd_dp_problem& pr, const dmnd_dp_result& r, const uint8_t* tr, double known_evalue = -1.0);
	void finish_round2(QueryState& q, ThreadCtx& tc);
	void finish_outer(QueryState& q);
	int run_waves();
	// frameshift alignment mode (legacy.inc)
	std::vector<struct LegacyQuery> lq;
	void legacy_init(size_t k, QueryState& q, ThreadCtx& tc, Workspace::HitSeg* begin, Workspace::HitSeg* end);
	void legacy_produce(LegacyQuery& L, const QueryState& q, ThreadCtx& tc, bool score_only);
	void legacy_consume_scores(LegacyQuery& L, const QueryState& q, const dmnd_fs_result* res);
	void legacy_consume_trace(LegacyQuery& L, QueryState& q, ThreadCtx& tc, const dmnd_fs_result* res, const uint8_t* tr);
	int run_legacy();
};

// std::stable_sort without its temporary-buffer allocation for the short lists that dominate (insertion sort is stable)
template<typename T, typename Cmp> static void stable_small_sort(std::vector<T>& v, Cmp cmp) {
	if (v.size() > 24) { std::stable_sort(v.begin(), v.end(), cmp); return; }
	for (size_t i = 1; i < v.size(); ++i) {
		size_t j = i;
		if (!cmp(v[i], v[i - 1])) continue;
		const T x = v[i];
		while (j > 0 && cmp(x, v[j - 1])) { v[j] = v[j - 1]; --j; }
		v[j] = x;
	}
}

void Driver::load_hits(QueryState& q, ThreadCtx& tc, Workspace::HitSeg* begin, Workspace::HitSeg* end) {
	// align/load_hits.h:44-122 (each hit carries its precomputed x-drop segment and its site in the reference block along)
	std::sort(begin, end, [](const Workspace::HitSeg& x, const Workspace::HitSeg& y) {
		const dmnd_hit &a = x.h, &b = y.h;
		const uint64_t sa = DMND_HIT_SUBJECT(a), sb = DMND_HIT_SUBJECT(b);
		return sa < sb || (sa == sb && (a.query < b.query || (a.query == b.query && a.seed_offset < b.seed_offset)));
	});
	q.sh_off = (uint32_t)tc.seed_hits.size();
	q.tgt_off = (uint32_t)tc.hit_begin.size();
	q.ts_off = (uint32_t)tc.target_scores.size();
	uint32_t target = UINT32_MAX, ntg = 0;
	uint16_t score = 0;
	for (Workspace::HitSeg* hsp = begin; hsp < end; ++hsp) {
		const dmnd_hit* h = &hsp->h;
		// SequenceSet::local_position of the subject position: delivered with the hit (dmnd_hits_xdrop_sites)
		const uint32_t t = hsp->site.target;
		if (t != target) {
			if (target != UINT32_MAX) { tc.target_scores.push_back({ ntg - 1, score }); score = 0; }
			tc.hit_begin.push_back((uint32_t)tc.seed_hits.size());
			target = t;
			tc.target_block_ids.push_back(t);
			++ntg;
		}
		const uint16_t hs = (uint16_t)DMND_HIT_SCORE(*h);
		tc.seed_hits.push_back({ h->seed_offset, hsp->site.j, (int)hs, hsp->s, hsp->gf, (uint8_t)(h->query - q.qid) });
		score = std::max(score, hs);
	}
	if (target != UINT32_MAX) tc.target_scores.push_back({ ntg - 1, score });
	tc.hit_begin.push_back((uint32_t)tc.seed_hits.size());
	q.n_targets = ntg;
}

void Driver::start(QueryState& q, ThreadCtx& tc) {
	// align/extend.cpp:346-387 then :226-258
	const Env& e = env;
	q.qlen = e.qlen(q.qid);
	q.bridged = false;
	q.new_hits_ev = false; q.tail_score = q.previous_tail_score = 0;
	q.aligned_targets = {}; q.r1 = {}; q.matches = {}; q.r2 = {}; q.prob_target = {};
	q.prob_begin = 0; q.prob_count = 0;
	const int64_t target_count = q.n_targets;
	tc.n_targets += (uint64_t)target_count;
	if (target_count == 0) { q.phase = PH_DONE; return; }
	const int64_t block_mult = std::max<int64_t>((int64_t)std::round((double)e.ref_letters / e.ranking_letters), 1);
	const int64_t mm = ((int64_t)e.max_target_seqs + 31) / 32 * 32;  // make_multiple(max_target_seqs, 32)
	q.chunk_size = e.top >= 0.0 ? 128 * block_mult : std::max<int64_t>(128, std::min<int64_t>(mm, 400)) * block_mult;  // ranking_chunk_size, align/extend.cpp:79-92
	TargetScore* ts = tc.target_scores.data() + q.ts_off;
	if (q.chunk_size < target_count) std::sort(ts, ts + target_count);
	q.i0 = 0;
	q.i1 = std::min<int64_t>(q.chunk_size, target_count);
	if (e.top < 0.0 && e.min_bit_score == 0.0 && (q.i1 - q.i0) < e.max_target_seqs)  // align/extend.cpp:262
		while (q.i1 < target_count && e.sc->evalue(ts[q.i1].score, (unsigned)q.qlen, 50) <= e.max_evalue)
			q.i1 += std::min<int64_t>(16, target_count - q.i1);
	// Fused rounds: round 2 re-evaluates, with traceback, exactly the (query, target, band) problem of round 1 that gave
	// each surviving target its HSP (gapped_final.cpp:64-78 takes hsp.d_begin/d_end).  With 180 GB of HBM the trace of
	// round 1 can simply be kept: a query whose targets mostly survive culling (<= 64 targets, one ranking chunk, at most
	// max_target_seqs = 25 culled away) sends its round-1 problems through the traceback kernel once and answers round 2
	// from those results -- one device round trip instead of two, 13 instead of 9 + 13 lane-ops per surviving cell.
	q.fused = e.fuse && e.contexts == 1 && target_count <= 64 && target_count <= q.chunk_size;
	q.phase = PH_ROUND1_PRODUCE;
}

// A query whose round-1 problem list was produced on the device (dmnd_hits_chain): the state start() + produce_round1() would
// have left for a fused query, minus the SeedHitList.  Targets without a problem are not listed: consume_round1 drops them anyway.
void Driver::start_bridged(QueryState& q, ThreadCtx& tc, const dmnd_chain_query& cq, const dmnd_dp_problem* probs) {
	const Env& e = env;
	q.qid = cq.query;
	q.qlen = e.qlen(q.qid);
	q.bridged = true; q.fused = true;
	q.new_hits_ev = false; q.tail_score = q.previous_tail_score = 0;
	q.aligned_targets = {}; q.r1 = {}; q.matches = {}; q.r2 = {}; q.prob_target = {};
	q.sh_off = q.tgt_off = q.ts_off = 0;
	q.n_targets = cq.n_targets;
	q.prob_begin = 0; q.prob_count = cq.n_problems;
	tc.n_targets += cq.n_targets; tc.n_extended += cq.n_targets;
	const int64_t block_mult = std::max<int64_t>((int64_t)std::round((double)e.ref_letters / e.ranking_letters), 1);
	const int64_t mm = ((int64_t)e.max_target_seqs + 31) / 32 * 32;
	q.chunk_size = e.top >= 0.0 ? 128 * block_mult : std::max<int64_t>(128, std::min<int64_t>(mm, 400)) * block_mult;
	q.i0 = 0; q.i1 = q.n_targets;  // one ranking chunk (n_targets <= 64 < chunk_size)
	q.r1.reserve(tc.arena, cq.n_problems);
	uint32_t last = UINT32_MAX;
	for (uint32_t k = 0; k < cq.n_problems; ++k) {
		const dmnd_dp_problem& pr = probs[k];
		if (pr.target != last) {
			q.r1.push(tc.arena, Target{ pr.target, e.tlen(pr.target), 0, DBL_MAX, HspLite{ 0, 0.0, 0, 0, q.qid }, false, 0 });
			last = pr.target;
		}
		q.prob_target.push(tc.arena, q.r1.n - 1);
		tc.cells1 += (uint64_t)(pr.d_end - pr.d_begin) * (uint64_t)banded_cols(q.qlen, e.tlen(pr.target), pr.d_begin, pr.d_end);
	}
	tc.fused_r1 += cq.n_problems;
	q.phase = PH_ROUND1_CONSUME;
}

void Driver::produce_round1(QueryState& q, ThreadCtx& tc) {
	// extend_chunk -> ungapped_stage -> align (round 1)
	const Env& e = env;
	q.r1.clear();
	q.r1.reserve(tc.arena, (uint32_t)(q.i1 - q.i0));
	q.prob_target.clear();
	std::vector<dmnd_dp_problem>& plist = q.fused ? tc.p2 : tc.p1;  // fused: straight into the traceback batch
	q.prob_begin = plist.size();
	const int band = band_for(q.qlen, e.band_slow);  // Extension::band(query_seq->length(), mode): the first context's length
	const TargetScore* ts = tc.target_scores.data() + q.ts_off;
	const uint32_t* hb = tc.hit_begin.data() + q.tgt_off;
	const uint32_t* ids = tc.target_block_ids.data() + q.ts_off;
	for (int64_t k = q.i0; k < q.i1; ++k) {
		const uint32_t tix = ts[k].target;
		const uint32_t block_id = ids[tix];
		const int slen = e.tlen(block_id);
		const int8_t* subject = e.rseq(block_id);
		q.r1.push(tc.arena, Target{ block_id, slen, 0, DBL_MAX, HspLite{ 0, 0.0, 0, 0, q.qid }, false, 0 });
		tc.hits.assign(tc.seed_hits.begin() + hb[tix], tc.seed_hits.begin() + hb[tix + 1]);
		if (e.gapped_filter && !(e.contexts > 1 && q.qlen < 85)) {  // Extension::gapped_filter (align/gapped_filter.cpp:41-63): a target stays iff one of its hits passes; translated queries whose first frame is < GAPPED_FILTER_MIN_QLEN = 85 skip it (align/extend.cpp:197-206)
			bool any = false;
			for (const SeedHit& h : tc.hits) any |= h.gf != 0;
			if (!any) continue;
		}
		++tc.n_extended;
		// translated queries: a target with ONE seed hit skips the x-drop extension and chaining, its band is centred on the
		// hit's diagonal (align/ungapped.cpp:76-80)
		const bool single = e.contexts > 1 && tc.hits.size() == 1;
		if (!single) std::sort(tc.hits.begin(), tc.hits.end());
		for (uint32_t f = 0; f < e.contexts; ++f) {  // ungapped_stage + add_dp_targets, one frame after the other (ungapped.cpp:110-116, gapped_score.cpp:119)
			const uint32_t ctx = q.qid + f;
			tc.chains.clear();
			int qlen_f = q.qlen;
			if (single) {
				if (tc.hits[0].frame != f) continue;
				qlen_f = e.qlen(ctx);
				Chain c; c.d_min = c.d_max = tc.hits[0].i - tc.hits[0].j; c.score = tc.hits[0].score;
				tc.chains.push_back(c);
			}
			else {
				tc.segs.clear();
				for (const SeedHit& h : tc.hits) {  // align/ungapped.cpp:81-91
					if (h.frame != f) continue;
					if (!tc.segs.empty() && tc.segs.back().diag() == h.i - h.j && tc.segs.back().subject_end() >= h.j) continue;
					// xdrop_ungapped(query, cbs, target, hit.i, hit.j) was evaluated for every hit on the device (dmnd_hits_xdrop)
					const Segment d{ h.seg.i, h.seg.j, h.seg.len, h.seg.score };
					if (d.score > 0) tc.segs.push_back(d);
				}
				if (tc.segs.empty()) continue;
				if (e.contexts > 1) qlen_f = e.qlen(ctx);
				stable_small_sort(tc.segs, [](const Segment& x, const Segment& y) { return x.diag() < y.diag() || (x.diag() == y.diag() && x.j < y.j); });
				chain_segments(*e.sc, e.qseq(ctx), qlen_f, subject, slen, tc.segs, tc.chains);
				stable_small_sort(tc.chains, [](const Chain& x, const Chain& y) { return x.d_min < y.d_min; });
			}
			// add_dp_targets, align/gapped_score.cpp:107-180
			int d0 = INT_MAX, d1 = INT_MIN;
			auto emit = [&] {
				plist.push_back(dmnd_dp_problem{ ctx, block_id, d0, d1 });
				q.prob_target.push(tc.arena, q.r1.n - 1);
				tc.cells1 += (uint64_t)(d1 - d0) * (uint64_t)banded_cols(qlen_f, slen, d0, d1);
			};
			for (const Chain& h : tc.chains) {
				const int b0 = std::max(h.d_min - band, -(slen - 1)), b1 = std::min(h.d_max + 1 + band, qlen_f);
				bool merge = false;
				if (d0 != INT_MAX) {
					const int ib = std::max(d0, b0), ie = std::min(d1, b1);
					const double overlap = ie > ib ? ie - ib : 0;
					merge = overlap / (d1 - d0) > 0.0 || overlap / (b1 - b0) > 0.0;
				}
				if (merge) { d0 = std::min(d0, b0); d1 = std::max(d1, b1); }
				else {
					if (d0 != INT_MAX) emit();
					d0 = b0; d1 = b1;
				}
			}
			if (!tc.chains.empty()) emit();
		}
	}
	q.prob_count = (uint32_t)(plist.size() - q.prob_begin);
	if (q.fused) { tc.fused_r1 += q.prob_count; tc.fused_r1_wave += q.prob_count; }
	q.phase = PH_ROUND1_CONSUME;
}

static void culling_targets(List<Target>& targets, bool sort_only, const Env& e) {  // align/culling.cpp:92-94,187-191
	if (e.top >= 0.0) std::sort(targets.begin(), targets.end(), Target::comp_score); else std::sort(targets.begin(), targets.end(), Target::comp_evalue);
	if (!sort_only) targets.n = (uint32_t)(output_range(targets.begin(), targets.end(), e) - targets.begin());
}

void Driver::consume_round1(QueryState& q, ThreadCtx& tc, const dmnd_dp_problem* probs, const dmnd_dp_result* res) {
	const Env& e = env;
	// tail of align() round 1 (gapped_score.cpp:231-246): add_hit + inner_culling (max_hsps == 1 keeps the first HSP in
	// Hsp::operator< order; list::sort is stable, so among equal keys the earliest-added wins)
	for (uint32_t k = 0; k < q.prob_count; ++k) {
		const int score = res[k].score;
		Target& t = q.r1.p[q.prob_target.p[k]];
		const uint32_t ctx = probs[k].query;
		const double ev = e.sc->evalue(score, (unsigned)(ctx == q.qid ? q.qlen : e.qlen(ctx)), (unsigned)t.tlen);
		if (score > 0 && e.report_cutoff(score, ev)) {  // banded_swipe.h:341-342, ScoreMatrix::report_cutoff
			const HspLite h{ score, ev, probs[k].d_begin, probs[k].d_end, ctx };
			// Target::add_hit(list,it), target.h:104-112: a strictly higher score moves filter_score AND best_context to this HSP's
			// frame (frames arrive in ascending order, as the reference's loop over the frames delivers them); inner_culling keeps
			// the best HSP of best_context only (culling.cpp:58-67)
			if (score > t.filter_score) { t.filter_evalue = ev; t.filter_score = score; t.hsp = h; t.hsp_prob = k; }
			else if (t.has_hsp && ctx == t.hsp.ctx && hsp_less(h, t.hsp)) { t.hsp = h; t.hsp_prob = k; }
			t.has_hsp = true;
		}
	}
	// keep targets with hits (gapped_score.cpp:236-243)
	tc.tmp_targets.clear();
	for (const Target& t : q.r1) if (t.filter_evalue != DBL_MAX) tc.tmp_targets.push_back(t);
	q.r1.clear();
	std::vector<Target>& v = tc.tmp_targets;
	// align/extend.cpp:307-320
	const TargetScore* ts = tc.target_scores.data() + q.ts_off;
	const int64_t n_targets = q.n_targets;
	const bool multi_chunk = (q.i1 - q.i0) < n_targets;
	bool new_hits = q.new_hits_ev = !v.empty();
	if (multi_chunk) {
		// append_hits, align/culling.cpp:111-141 (with_culling = first_round_culling = true)
		if (v.empty()) new_hits = false;
		else {
			new_hits = e.top < 0.0 && (int64_t)q.aligned_targets.n < e.max_target_seqs;
			bool append = !e.first_round_culling || new_hits;
			culling_targets(q.aligned_targets, append, e);
			double min_evalue = DBL_MAX;
			int max_score = 0;
			for (const Target& t : v) { min_evalue = std::min(min_evalue, t.filter_evalue); max_score = std::max(max_score, t.filter_score); }
			Target* range_end = output_range(q.aligned_targets.begin(), q.aligned_targets.end(), e);
			if (q.aligned_targets.n == 0 || (e.top < 0.0 && min_evalue <= (range_end - 1)->filter_evalue)
			    || (e.top >= 0.0 && max_score >= (int)((1.0 - e.top / 100.0) * (range_end - 1)->filter_score))) { append = true; new_hits = true; }  // top_cutoff_score<int>, basic/config.h:452-455
			if (append) for (const Target& t : v) q.aligned_targets.push(tc.arena, t);
		}
	}
	else {
		q.aligned_targets.clear();
		q.aligned_targets.reserve(tc.arena, (uint32_t)v.size());
		for (const Target& t : v) q.aligned_targets.push(tc.arena, t);
	}
	q.i0 = q.i1;
	q.i1 += std::min<int64_t>(q.chunk_size, n_targets - q.i1);
	q.previous_tail_score = q.tail_score;
	if (new_hits && !q.bridged) q.tail_score = ts[q.i1 - 1].score;  // (a bridged query has one ranking chunk: the tail score is never read)
	bool terminate = false;
	if (q.i0 < n_targets) {  // ranking_terminate, align/extend.cpp:111-119
		const int tscore = ts[q.i1 - 1].score;
		terminate = !new_hits && (q.previous_tail_score == 0 || double(tscore) / (double)q.previous_tail_score <= 0.95 || e.sc->bitscore(tscore) < 25.0);
	}
	if (q.i0 < n_targets && !terminate) { q.phase = PH_ROUND1_PRODUCE; return; }
	culling_targets(q.aligned_targets, !e.first_round_culling, e);  // extend.cpp:331
	if (q.aligned_targets.n == 0) finish_outer(q);  // round 2 over nothing returns no matches
	else { q.phase = PH_ROUND2_PRODUCE; q.r2.clear(); q.r2_it = 0; q.r2_prev = q.matches.n; }
}

void Driver::produce_round2(QueryState& q, ThreadCtx& tc) {
	// round-2 problems (gapped_final.cpp:64-78,118-124): one per kept HSP of every culled target.  With filters and without --top the
	// targets are taken in steps (:107-111): max(k - matches so far, 16) rounded up to a multiple of 16, until k matches passed the filters
	const Env& e = env;
	q.prob_begin = tc.p2.size();
	q.prob_target.clear();
	uint32_t step = q.aligned_targets.n - q.r2_it;
	if (!e.first_round_culling && e.top < 0.0) {
		const int64_t want = std::max<int64_t>((int64_t)e.max_target_seqs - (int64_t)q.r2.n, 16);
		step = (uint32_t)std::min<int64_t>((want + 15) / 16 * 16, (int64_t)step);
	}
	q.r2.reserve(tc.arena, q.r2.n + step);
	q.r2_begin = q.r2.n;
	for (uint32_t k = q.r2_it; k < q.r2_it + step; ++k) {
		const Target& tg = q.aligned_targets.p[k];
		if (tg.has_hsp) {
			tc.p2.push_back(dmnd_dp_problem{ tg.hsp.ctx, tg.block_id, tg.hsp.d_begin, tg.hsp.d_end });
			q.prob_target.push(tc.arena, q.r2.n);
			tc.cells2 += (uint64_t)(tg.hsp.d_end - tg.hsp.d_begin) * (uint64_t)banded_cols(tg.hsp.ctx == q.qid ? q.qlen : env.qlen(tg.hsp.ctx), tg.tlen, tg.hsp.d_begin, tg.hsp.d_end);
		}
		Match m;
		std::memset(&m, 0, sizeof m);
		m.target_block_id = tg.block_id; m.tlen = tg.tlen; m.filter_score = 0; m.filter_evalue = DBL_MAX; m.has_hsp = false;
		q.r2.push(tc.arena, m);
	}
	q.r2_it += step;
	q.prob_count = (uint32_t)(tc.p2.size() - q.prob_begin);
	q.phase = PH_ROUND2_CONSUME;
}

void Driver::take_round2_result(QueryState& q, ThreadCtx& tc, Match& m, const dmnd_dp_problem& pr, const dmnd_dp_result& r, const uint8_t* tr, double known_evalue) {
	// gapped_final.cpp:140-149; known_evalue >= 0: the e-value of (r.score, qlen, tlen) was already computed in round 1
	const Env& e = env;
	const double ev = known_evalue >= 0.0 ? known_evalue : e.sc->evalue(r.score, (unsigned)(pr.query == q.qid ? q.qlen : e.qlen(pr.query)), (unsigned)m.tlen);
	if (r.score > 0 && e.report_cutoff(r.score, ev)) {
		const HspLite h{ r.score, ev, pr.d_begin, pr.d_end, pr.query };
		if (!m.has_hsp || hsp_less(h, m.h)) {
			m.h = h; m.r = r;
			m.tr_off = 0; m.tr_len = 0;
			if (e.want_transcript && r.status == 0 && tr) {
				m.tr_off = tc.trbuf.size(); m.tr_len = r.transcript_len;
				tc.trbuf.insert(tc.trbuf.end(), tr + r.transcript_off, tr + r.transcript_off + r.transcript_len);
			}
		}
		m.has_hsp = true;
	}
}

bool Driver::filtered_out(const QueryState& q, const Match& m) const {
	// filter_hsp, align/culling.cpp:144-170 (Hsp::id_percent / query_cover_percent / subject_cover_percent, basic/match.h:208-221); the
	// query range is the HSP's range on the DNA read for translated queries: three letters per codon (basic/translated_position.h:120-135)
	const Env& e = env;
	const dmnd_dp_result& r = m.r;
	const int source_query_len = e.contexts == 6 ? e.qlen(q.qid) + e.qlen(q.qid + 1) + e.qlen(q.qid + 2) + 2 : q.qlen;
	const int q_range = (r.q_end - r.q_begin) * (e.contexts == 6 ? 3 : 1);
	const double qcov = (double)q_range * 100 / (unsigned)source_query_len, tcov = (double)(r.t_end - r.t_begin) * 100 / (unsigned)m.tlen;
	if (e.approx_min_id > 0.0) {  // hsp.approx_id (banded_swipe.h:185): 100 for identical stretches, else the linear estimate from score per column
		const int ql = r.q_end - r.q_begin, tl = r.t_end - r.t_begin;
		const int8_t *qs = e.qseq(m.h.ctx) + r.q_begin, *ts = e.rseq(m.target_block_id) + r.t_begin;
		bool identical = ql == tl;
		for (int i = 0; identical && i < ql; ++i) identical = (qs[i] & 31) == (ts[i] & 31);
		const int mx = std::max(ql, tl);
		const double approx = identical ? 100.0 : (mx == 0 ? 100.0 : std::min(std::max(std::fma((double)r.score / mx, 16.56, 11.41), 0.0), 100.0));
		if (approx < e.approx_min_id) return true;
	}
	return (double)r.identities * 100.0 / (double)r.length < e.min_id || qcov < e.query_cover || tcov < e.subject_cover;
}

void Driver::finish_round2(QueryState& q, ThreadCtx& tc) {
	const Env& e = env;
	for (Match* m = q.r2.begin() + q.r2_begin; m < q.r2.end(); ++m) {
		if (m->has_hsp) { m->filter_evalue = m->h.evalue; m->filter_score = m->h.score; }  // Match::inner_culling
		if (m->has_hsp && ((e.have_filters && filtered_out(q, *m)) || (e.self_targets && e.self_targets[q.qid / e.contexts] == m->target_block_id))) { m->has_hsp = false; m->filter_evalue = DBL_MAX; m->filter_score = 0; }  // Match::apply_filters, culling.cpp:172-185
	}
	if (e.top >= 0.0) std::sort(q.r2.begin(), q.r2.end(), Match::cmp_score); else std::sort(q.r2.begin(), q.r2.end(), Match::cmp_evalue);  // culling(r, cfg), culling.cpp:199-202
	q.r2.n = (uint32_t)(output_range(q.r2.begin(), q.r2.end(), e) - q.r2.begin());
	// the next step of the filtered schedule (gapped_final.cpp:156: it < targets.end() && goon())
	if (q.r2_it < q.aligned_targets.n && (e.top >= 0.0 || (int64_t)q.r2.n + (int64_t)q.r2_prev < (int64_t)e.max_target_seqs)) { q.phase = PH_ROUND2_PRODUCE; return; }
	for (const Match& m : q.r2) q.matches.push(tc.arena, m);
	q.r2.clear();
	q.aligned_targets.clear();
	finish_outer(q);
}

void Driver::consume_round2(QueryState& q, ThreadCtx& tc, const dmnd_dp_problem* probs, const dmnd_dp_result* res, const uint8_t* tr) {
	for (uint32_t k = 0; k < q.prob_count; ++k) take_round2_result(q, tc, q.r2.p[q.prob_target.p[k]], probs[k], res[k], tr);
	finish_round2(q, tc);
}

void Driver::consume_fused(QueryState& q, ThreadCtx& tc, const dmnd_dp_problem* probs, const dmnd_dp_result* res, const uint8_t* tr) {
	// round 1 over the traceback results (their scores are the score-only kernel's), then round 2 answered from them
	consume_round1(q, tc, probs, res);
	if (q.phase != PH_ROUND2_PRODUCE) return;  // nothing survived, or (never for a fused query) another ranking chunk
	q.r2.clear();
	q.r2.reserve(tc.arena, q.aligned_targets.n);
	q.r2_begin = 0; q.r2_it = q.aligned_targets.n;  // (fused queries never run with filters: one step)
	for (const Target& tg : q.aligned_targets) {
		Match m;
		std::memset(&m, 0, sizeof m);
		m.target_block_id = tg.block_id; m.tlen = tg.tlen; m.filter_score = 0; m.filter_evalue = DBL_MAX; m.has_hsp = false;
		if (tg.has_hsp) {  // the round-2 problem of this target IS round-1 problem hsp_prob (gapped_final.cpp:64-78)
			const dmnd_dp_problem& pr = probs[tg.hsp_prob];
			tc.cells2 += (uint64_t)(pr.d_end - pr.d_begin) * (uint64_t)banded_cols(q.qlen, tg.tlen, pr.d_begin, pr.d_end);
			++tc.fused_r2;
			// same problem, same score: the e-value of round 1 (tg.hsp) is the e-value of round 2
			take_round2_result(q, tc, m, pr, res[tg.hsp_prob], tr, res[tg.hsp_prob].score == tg.hsp.score ? tg.hsp.evalue : -1.0);
		}
		q.r2.push(tc.arena, m);
	}
	finish_round2(q, tc);
}

void Driver::finish_outer(QueryState& q) {
	// outer do-while of extend(), align/extend.cpp:336, then the final culling (:341)
	const Env& e = env;
	if (e.top < 0.0 && (int64_t)q.matches.n < e.outer_limit && q.i0 < (int64_t)q.n_targets && q.new_hits_ev) { q.phase = PH_ROUND1_PRODUCE; return; }
	if (e.top >= 0.0) std::sort(q.matches.begin(), q.matches.end(), Match::cmp_score); else std::sort(q.matches.begin(), q.matches.end(), Match::cmp_evalue);
	q.matches.n = (uint32_t)(output_range(q.matches.begin(), q.matches.end(), e) - q.matches.begin());
	q.phase = PH_DONE;
}

// Transcript bytes the traceback kernel may need for problems p[0, n): qlen + tlen per problem.
static size_t transcript_cap(const Env& e, const dmnd_dp_problem* p, size_t n) {
	size_t cap = 0;
	for (size_t k = 0; k < n; ++k) cap += (size_t)e.qlen(p[k].query) + (size_t)e.tlen(p[k].target);
	return cap;
}

int Driver::run_waves() {
	Workspace& w = *ws;
	Prof prof;
	std::vector<size_t> off1((size_t)T + 1), off2((size_t)T + 1);
	for (;;) {
		auto t0 = Clock::now();
		// ---- produce: every active query emits the DP problems of its next step into its owner's list
		ws->run([&](int t) {
			ThreadCtx& tc = w.tc[(size_t)t];
			tc.p1.clear(); tc.p2.clear();
			for (size_t k = block_begin(t), en = block_begin(t + 1); k < en; ++k) {
				QueryState& q = w.qs[k];
				if (q.phase == PH_ROUND1_PRODUCE) produce_round1(q, tc);
				else if (q.phase == PH_ROUND2_PRODUCE) produce_round2(q, tc);
			}
		});
		off1[0] = off2[0] = 0;
		for (int t = 0; t < T; ++t) { off1[(size_t)t + 1] = off1[(size_t)t] + w.tc[(size_t)t].p1.size(); off2[(size_t)t + 1] = off2[(size_t)t] + w.tc[(size_t)t].p2.size(); }
		if (off1[(size_t)T] + off2[(size_t)T] == 0) break;  // nothing in flight: every query is done
		if (w.p1.resize(ctx, off1[(size_t)T]) || w.p2.resize(ctx, off2[(size_t)T]) || w.res1.resize(ctx, off1[(size_t)T]) || w.res2.resize(ctx, off2[(size_t)T])) return 1;
		ws->run([&](int t) {
			const ThreadCtx& tc = w.tc[(size_t)t];
			if (!tc.p1.empty()) std::memcpy(w.p1.data() + off1[(size_t)t], tc.p1.data(), tc.p1.size() * sizeof(dmnd_dp_problem));
			if (!tc.p2.empty()) std::memcpy(w.p2.data() + off2[(size_t)t], tc.p2.data(), tc.p2.size() * sizeof(dmnd_dp_problem));
		});
		// problem counts in the reference's terms: a fused query's round-1 problems sit in the traceback batch, its round-2
		// problems are answered from their results (counted in consume_fused)
		uint64_t fused_wave = 0;
		for (ThreadCtx& tc : w.tc) { fused_wave += tc.fused_r1_wave; tc.fused_r1_wave = 0; }
		stats.dp_problems_round1 += w.p1.size() + fused_wave; stats.dp_problems_round2 += w.p2.size() - fused_wave;
		stats.host_bridge_ms += ms_since(t0);
		prof.lap("  wave: produce + concat");
		// ---- device waves
		t0 = Clock::now();
		if (!w.p1.empty() && dmnd_banded_swipe(ctx, qb, rb, w.p1.data(), w.p1.size(), DMND_DP_SCORE_ONLY, w.res1.data(), nullptr, 0)) return 1;
		stats.dp1_ms += ms_since(t0);
		t0 = Clock::now();
		uint8_t* trp = nullptr;
		if (!w.p2.empty()) {
			size_t cap = 0;
			if (env.want_transcript) {
				cap = transcript_cap(env, w.p2.data(), w.p2.size());
				if (w.tr.resize(ctx, cap)) return 1;
				trp = w.tr.data();
			}
			if (dmnd_banded_swipe(ctx, qb, rb, w.p2.data(), w.p2.size(), DMND_DP_TRACEBACK, w.res2.data(), trp, cap)) return 1;
		}
		stats.dp2_ms += ms_since(t0);
		prof.lap("  wave: banded_swipe x2");
		t0 = Clock::now();
		// ---- consume
		ws->run([&](int t) {
			ThreadCtx& tc = w.tc[(size_t)t];
			const dmnd_dp_problem *P1 = w.p1.data() + off1[(size_t)t], *P2 = w.p2.data() + off2[(size_t)t];
			const dmnd_dp_result *R1 = w.res1.data() + off1[(size_t)t], *R2 = w.res2.data() + off2[(size_t)t];
			for (size_t k = block_begin(t), en = block_begin(t + 1); k < en; ++k) {
				QueryState& q = w.qs[k];
				if (q.phase == PH_ROUND1_CONSUME) {
					if (q.fused) consume_fused(q, tc, P2 + q.prob_begin, R2 + q.prob_begin, trp);
					else consume_round1(q, tc, P1 + q.prob_begin, R1 + q.prob_begin);
				}
				else if (q.phase == PH_ROUND2_CONSUME) consume_round2(q, tc, P2 + q.prob_begin, R2 + q.prob_begin, trp);
			}
		});
		stats.host_bridge_ms += ms_since(t0);
		prof.lap("  wave: consume");
	}
	return 0;
}

#include "legacy.inc"

}  // namespace

// ------------------------------------------------------------------------------------------------------------
struct dmnd_result {
	RawBuf<dmnd_match> matches;
	RawBuf<uint8_t> transcripts;
	dmnd_run_stats stats;
	std::vector<uint64_t> masked[2];  // hard-masked letters of the query / reference block (dmnd_blastp with masking)
	std::vector<uint32_t> unaligned;  // queries (first context) with seed hits and no alignment, ascending
};
// dmnd_result_free parks up to two results here; the next call reuses their (already touched) memory.
struct ResultPool {
	std::mutex m;
	std::vector<dmnd_result*> free_list;
	dmnd_result* take() {
		std::lock_guard<std::mutex> l(m);
		if (free_list.empty()) return new dmnd_result();
		dmnd_result* r = free_list.back(); free_list.pop_back();
		return r;
	}
	void give(dmnd_result* r) {
		{
			std::lock_guard<std::mutex> l(m);
			if (free_list.size() < 2) { free_list.push_back(r); return; }
		}
		delete r;
	}
};
static ResultPool& result_pool() { static ResultPool p; return p; }

extern "C" {

// Sensitivity::{FAST, DEFAULT, MID_SENSITIVE, SENSITIVE, MORE_SENSITIVE, VERY_SENSITIVE, ULTRA_SENSITIVE}: sensitivity_traits
// (search/setup.cpp:40-54), shape_codes (:80-304), default_ext_mode (align/extend.cpp:62-75), ranking_chunk_size's default_letters
// (align/extend.cpp:86).  The shape codes are the reference's (spaced-seed patterns are data of the method, like BLOSUM62).
struct ModeTraits {
	int n_shapes; const char* const* codes;
	int min_identities; double ungapped_evalue, ungapped_evalue_short, gapped_filter_evalue; int index_chunks; double seed_cut;
	bool motif_masking, band_slow; double ranking_letters;
};
static const ModeTraits* mode_traits(int sensitivity) {
	static const char* const fast[] = { "1101110101101111" };
	static const char* const dflt[] = { "111101110111", "111011010010111" };
	static const char* const mid[] = { "11110110111", "1101100111101", "1110010101111", "11010101100111", "11101110001011", "1110100100010111", "1101000011010111", "1110011000011011" };
	static const char* const sens[] = { "1011110111", "110100100010111", "11001011111", "101110001111", "11011101100001", "1111010010101", "111001001001011", "10101001101011",
		"111101010011", "1111000010000111", "1100011011011", "1101010000011011", "1110001010101001", "110011000110011", "11011010001101", "1101001100010011" };
	static const char* const very[] = { "11101111", "110110111", "111111001", "1010111011", "11110001011", "110100101011", "110110001101", "1010101000111", "1100101001011",
		"1101010101001", "1110010010011", "110110000010011", "111001000100011", "1101000100010011" };
	static const char* const ultra[] = { "1111111", "11101111", "110011111", "110110111", "111111001", "1010111011", "1011110101", "1111000111", "10011110011", "10101101101",
		"10111010101", "11001010111", "11001100111", "11010101101", "11110001011", "100111010011", "101100110101", "101110000111", "110100101011", "110110001101", "111000110011",
		"1010001011011", "1010101000111", "1010110100011", "1100100110011", "1100101001011", "1101001100101", "1101010101001", "1110001010101", "1110010010011", "10100001101101",
		"11000100010111", "11010000100111", "11010100110001", "11101000011001", "11110000001101", "11110100000011", "101001000001111", "110000100101011", "110010010000111",
		"110101100001001", "110110000010011", "111001000100011", "111100000100101", "1000110010010101", "1001000100101101", "1001000110011001", "1010001001001011",
		"1010001010010011", "1010010001010101", "1010010100010011", "1010010101001001", "1010100000101011", "1010100011000101", "1011000010001011", "1100010000111001",
		"1100010010001011", "1100100001001011", "1100100100100011", "1100110000001101", "1101000100010011", "1101000110000101", "1110000001010011", "1110100000010101" };
	static const ModeTraits t[7] = {
		//  shapes        minid ug_ev     ug_ev_s  gf_ev chunks seed_cut motif  slow   ranking letters
		{ 1, fast,  11, 0.0,      0.0,     0.0, 4, 0.9, true,  false, 2e9 },
		{ 2, dflt,  11, 10000.0,  10000.0, 0.0, 4, 0.8, true,  false, 2e9 },
		{ 8, mid,   11, 10000.0,  10000.0, 0.0, 4, 1.0, true,  false, 2e9 },
		{ 16, sens, 11, 10000.0,  10000.0, 1.0, 4, 1.0, true,  false, 2e9 },
		{ 16, sens, 11, 10000.0,  10000.0, 1.0, 4, 1.0, false, true,  2e9 },   // MORE_SENSITIVE: the shapes of SENSITIVE, no motif masking, BANDED_SLOW
		{ 14, very,  9, 100000.0, 30000.0, 1.0, 1, 1.0, false, true,  800e6 },
		{ 64, ultra, 9, 300000.0, 30000.0, 1.0, 1, 1.0, false, true,  800e6 },
	};
	return sensitivity >= 0 && sensitivity <= 6 ? &t[sensitivity] : nullptr;
}
extern "C" int dmnd_alignment_stats(int32_t raw_score, uint32_t query_len, uint32_t target_len, uint64_t db_letters, double* evalue, double* bit_score) {
	Scoring sc;
	sc.db_letters = (double)db_letters;
	if (evalue) *evalue = sc.evalue(raw_score, query_len, target_len);
	if (bit_score) *bit_score = sc.bitscore(raw_score);
	return 0;
}
extern "C" int dmnd_mode_motif_masking(int sensitivity) { const ModeTraits* t = mode_traits(sensitivity); return t ? (int)t->motif_masking : -1; }

void dmnd_search_opts_default(dmnd_search_opts* o) {
	std::memset(o, 0, sizeof *o);
	o->sensitivity = 0; o->threads = 8; o->index_chunks = 0; o->comp_based_stats = 1; o->max_target_seqs = 25;
	o->max_evalue = 0.001; o->db_letters = 0; o->want_transcript = 0;
	o->query_contexts = 1; o->top_percent = -1.0;
	o->masking = 1; o->motif_masking = 1;  // the reference's defaults for blastp --fast (run/config.cpp:126-135, search/setup.cpp:43)
}

int dmnd_params_init(const dmnd_search_opts* o, dmnd_params* p) {
	std::memset(p, 0, sizeof *p);
	Scoring sc;
	std::memcpy(p->score, sc.m8, sizeof p->score);
	p->gap_open = sc.gap_open; p->gap_extend = sc.gap_extend;
	for (int i = 0; i < 20; ++i) p->background_scores_f32[i] = (float)sc.background_scores[i];
	// Reduction("A KR EDNQ C G H ILVM FYW P ST"), stats/stats.cpp:48, basic/basic.cpp:267-296
	static const char* groups[10] = { "A", "KR", "EDNQ", "C", "G", "H", "ILVM", "FYW", "P", "ST" };
	const char* alph = letter_alphabet();
	for (int c = 0; c < 10; ++c)
		for (const char* s = groups[c]; *s; ++s) {
			const int l = (int)(std::strchr(alph, *s) - alph);
			p->reduction[l] = (uint8_t)c; p->map8[l] = (uint8_t)c; p->map8b[l] = (uint8_t)c;
		}
	p->reduction[MASK_LETTER] = MASK_LETTER; p->reduction[STOP_LETTER] = MASK_LETTER;
	p->map8[MASK_LETTER] = p->map8[STOP_LETTER] = p->map8[DMND_DELIMITER] = 10;
	p->map8b[MASK_LETTER] = p->map8b[STOP_LETTER] = p->map8b[DMND_DELIMITER] = 11;
	p->reduction_size = 10;
	const ModeTraits* mt = mode_traits(o->sensitivity);
	if (!mt) { dmnd_set_last_error("sensitivity must be 0 (--fast) .. 6 (--ultra-sensitive)"); return 1; }
	p->n_shapes = mt->n_shapes;
	for (int s = 0; s < p->n_shapes; ++s) {
		int w = 0, len = 0;
		for (const char* c = mt->codes[s]; *c; ++c, ++len)
			if (*c == '1') { p->shape_pos[s][w++] = len; p->shape_mask[s] |= 1u << len; }
		p->shape_len[s] = len; p->shape_weight = w;
	}
	p->hamming_id = std::max(mt->min_identities, o->approx_min_id >= 90.0 ? 30 : o->approx_min_id >= 50.0 ? 20 : 0);  // hamming_id_cutoff(config.approx_min_id), search/setup.cpp:70-79,343
	p->index_chunks = o->index_chunks > 0 ? o->index_chunks : mt->index_chunks;
	{  // seedp_bits, search/setup.cpp:306-309
		auto bit_length = [](int64_t x) { int n = 0; while (x > 0) { ++n; x >>= 1; } return n; };
		int64_t pw = 1; for (int i = 0; i < p->shape_weight; ++i) pw *= p->reduction_size;
		const int threads = o->threads > 0 ? o->threads : 1;
		p->seedp_bits = std::max(std::max(bit_length(pw - 1) - 32, bit_length((int64_t)threads * 4 * p->index_chunks - 1)), 8);
	}
	p->seed_cut = mt->seed_cut * std::log(2.0) * p->shape_weight;  // traits seed_cut (search/setup.cpp:43-49)
	p->left_most_interval = 32; p->ungapped_window = 48;
	p->ungapped_evalue = mt->ungapped_evalue;
	p->short_query_max_len = 60;
	p->short_query_ungapped_cutoff = sc.rawscore(25.0);
	if (p->ungapped_evalue > 0.0)
		for (int b = 1; b <= 31; ++b)  // CutoffTable: rawscore(bitscore_norm(evalue, 2^(b-1))), stats/score_matrix.h:133-151
			p->ungapped_cutoff[b] = sc.rawscore(-std::log(p->ungapped_evalue / 1e9 / (double)(1u << (b - 1))) / std::log(2.0));
	p->query_contexts = o->query_contexts > 1 ? o->query_contexts : 1;
	if (mt->ungapped_evalue_short > 0.0)  // cfg.cutoff_table_short (search/setup.cpp:375), read for translated frames of 61..85 letters
		for (int b = 1; b <= 31; ++b)
			p->ungapped_cutoff_short[b] = sc.rawscore(-std::log(mt->ungapped_evalue_short / 1e9 / (double)(1u << (b - 1))) / std::log(2.0));
	p->gapped_filter_evalue = mt->gapped_filter_evalue;
	p->gapped_filter_window = 200;
	p->gapped_filter_diag_score = sc.rawscore(12.0);
	if (p->gapped_filter_evalue > 0.0) {
		// CutoffTable2D::calc_min_score (util/scores/cutoff_table.h:69-74) over ScoreMatrix::evalue_norm (stats/score_matrix.cpp:222-225:
		// the e-value against a 10^9-letter database)
		Scoring norm; norm.db_letters = 1e9;
		auto min_score = [&](unsigned qlen, unsigned slen, double evalue) {
			for (int i = 10; i < 1000; ++i) if (norm.evalue(i, qlen, slen) <= evalue) return i;
			return 1000;
		};
		for (int b1 = 1; b1 <= 31; ++b1)
			for (int b2 = 1; b2 <= 31; ++b2) {
				p->gapped_cutoff1[b1][b2] = (int16_t)min_score(1u << (b1 - 1), 1u << (b2 - 1), 2000.0);  // config.gapped_filter_evalue1
				p->gapped_cutoff2[b1][b2] = (int16_t)min_score(1u << (b1 - 1), 1u << (b2 - 1), p->gapped_filter_evalue);
			}
	}
	{	// tantan constants, masking/masking.cpp:133-153 and masking/tantan.cpp:131-142, evaluated in the reference's types.
		// lambda is what cbrc::LambdaCalculator (lib/tantan, a randomised root search seeded by the C library's default
		// rand() state) returns for BLOSUM62's 20 x 20 core; tests/test_masking.py re-derives it from the reference's own
		// LambdaCalculator.cc (oracle/ref_build lambda probe) and requires this exact double.
		const double lambda = 0x1.4bcf16a672882p-2;  // 0.32403216734804385
		// masking.cpp:146-151 fills the ratio for the whole 26-letter alphabet (value_traits.alphabet_size), X * _ included
		for (int a = 0; a < 26; ++a)
			for (int b = 0; b < 26; ++b) p->tantan_lr[a * 32 + b] = (float)std::exp(lambda * (double)sc.m8[a * 32 + b]);
		const float p_repeat = 0.005f, p_repeat_end = 0.05f;
		volatile float growth_rt = 1.0f / 0.9f;  // run-time value: powf below must be the C library's, as in the reference,
		const float repeat_growth = growth_rt;   // not a compile-time folding of it
		const int W = 50;
		const float b2f0 = p_repeat * (1.0f - repeat_growth) / (1.0f - std::pow(repeat_growth, (float)W));
		p->tantan_d[W - 1] = b2f0;
		for (int i = W - 2; i >= 0; --i) p->tantan_d[i] = p->tantan_d[i + 1] * repeat_growth;
		p->tantan_b2b = 1.0f - p_repeat; p->tantan_f2f = 1.0f - p_repeat_end; p->tantan_p_repeat_end = p_repeat_end;
		p->tantan_p_mask = (float)0.9;  // config.tantan_minMaskProb (basic/config.cpp:402)
		p->max_motif_len = 30;
	}
	return 0;
}

// One lane: the whole pipeline for the queries [q_begin, q_end) on its own lane context (stream + scratch).  Lanes run
// on their own host threads; while one lane waits for its kernels the other one owns the worker pool, so the host
// bridge of one query range overlaps the device work of the other.
struct LaneOut {
	RawBuf<dmnd_match>* matches = nullptr;  // the result's buffers (one lane) or the lane workspace's (several)
	RawBuf<uint8_t>* transcripts = nullptr;
	dmnd_run_stats stats;
	std::vector<uint32_t> unaligned;
	std::string error;
	int rc = 0;
};

// Seed stages of the lanes are issued one after the other, in lane order: lane 0 gets its hits after 1/nlanes of the
// seed time instead of sharing the device with everybody, which staggers the lanes into a pipeline (host bridge of
// lane k overlaps the seed stage of lane k+1 and the DP kernels of lane k-1).
struct SeedTurn {
	std::mutex m;
	std::condition_variable cv;
	int turn = 0;
	// A lane masks its own query range in place before it searches, and the 48-byte fingerprints of a lane's LAST sequence read into
	// the first letters of the next lane's range (search/hamming/finger_print.h:59-96 crosses sequence borders): lane k may only
	// search once lane k + 1 has finished masking, as the reference masks the whole block before any search
	// (run/double_indexed.cpp:737-741).  masked[l] is set when lane l's masking is on the device and complete (or was not asked for).
	std::vector<char> masked;
	void set_masked(int lane) { { std::lock_guard<std::mutex> l(m); if ((size_t)lane < masked.size()) masked[(size_t)lane] = 1; } cv.notify_all(); }
	void wait_masked(int lane) { std::unique_lock<std::mutex> l(m); cv.wait(l, [&] { return (size_t)lane >= masked.size() || masked[(size_t)lane]; }); }
	void wait_for(int lane) { std::unique_lock<std::mutex> l(m); cv.wait(l, [&] { return turn >= lane; }); }
	void pass(int lane) { { std::lock_guard<std::mutex> l(m); turn = std::max(turn, lane + 1); } cv.notify_all(); }
};

// However a lane leaves (error or exception), the lanes behind it must not wait for its masking or its seed turn.
struct TurnRelease { SeedTurn& turn; int lane; ~TurnRelease() { turn.set_masked(lane); turn.pass(lane); } };

struct HitsGuard {  // the hits of one search, freed on every way out of the scope that searched
	dmnd_ctx* ctx; dmnd_hits* h = nullptr;
	explicit HitsGuard(dmnd_ctx* c) : ctx(c) {}
	HitsGuard(const HitsGuard&) = delete;
	~HitsGuard() { dmnd_hits_free(ctx, h); }
};

static void add_counters(dmnd_stage_counters& a, const dmnd_stage_counters& b) {
	a.seeds_hit += b.seeds_hit; a.seed_hits += b.seed_hits; a.tentative_matches1 += b.tentative_matches1;
	a.tentative_matches2 += b.tentative_matches2; a.tentative_matches3 += b.tentative_matches3; a.masked_seeds += b.masked_seeds;
}

// The device time, launch and byte counters between two snapshots of a context's timing (the DP cell counters stay 0).
static dmnd_timing device_delta(const dmnd_timing& t1, const dmnd_timing& t0) {
	dmnd_timing d{};
	d.seed_ms = t1.seed_ms - t0.seed_ms; d.dp_score_ms = t1.dp_score_ms - t0.dp_score_ms; d.dp_trace_ms = t1.dp_trace_ms - t0.dp_trace_ms;
	d.h2d_ms = t1.h2d_ms - t0.h2d_ms; d.d2h_ms = t1.d2h_ms - t0.d2h_ms;
	d.launches = t1.launches - t0.launches; d.h2d_bytes = t1.h2d_bytes - t0.h2d_bytes; d.d2h_bytes = t1.d2h_bytes - t0.d2h_bytes;
	return d;
}

// Waits for the lane's query range (dmnd_block_upload_ranges), masks it ("Masking queries", run/double_indexed.cpp:737-741, + the query
// block's motif table: the host only learns WHICH letters became X and patches private copies of those sequences), computes its
// composition bias, then waits for the next lane's masking and for this lane's seed turn.
static int prepare_range(Driver& d, uint32_t q_begin, uint32_t q_end, int lane, SeedTurn& turn, Prof& prof) {
	Workspace& w = *d.ws;
	const Env& env = d.env;
	int rc = dmnd_block_range_wait(d.ctx, d.qb, q_begin, q_end);
	if (!rc && env.mask_algo) {
		uint64_t n_hard = 0;
		rc = dmnd_block_mask(d.ctx, d.qb, env.mask_algo, q_begin, q_end, &n_hard);
		w.mask_pos.resize((size_t)n_hard);
		if (!rc && n_hard) rc = dmnd_block_mask_fetch(d.ctx, w.mask_pos.data(), w.mask_pos.size());
		if (!rc) { w.q_patch.build(env.q_letters, env.q_limits, env.nq, q_begin, q_end, w.mask_pos.data(), w.mask_pos.size()); d.env.q_patch = &w.q_patch; }
	}
	turn.set_masked(lane);  // (dmnd_block_mask returns when the range is masked on the device; also set on failure so nobody waits forever)
	rc = rc || dmnd_block_compute_bias_range(d.ctx, d.qb, env.hauser ? 1 : 0, q_begin, q_end);
	turn.wait_masked(lane + 1);
	prof.lap("wait, mask, bias");
	turn.wait_for(lane);
	prof.lap("wait for the seed turn");
	return rc;
}

// Seed stage of the bridged mode (Env::bridge): the search, then dmnd_hits_chain turns the hits into the round-1 problem list on the
// device.  Only the per-query records, the problems and the hits of DMND_CHAIN_HOST queries come back.
static int seed_bridged(Driver& d, uint32_t q_begin, uint32_t q_end, int lane, SeedTurn& turn, Clock::time_point t0, dmnd_chain_out& co, Prof& prof) {
	Workspace& w = *d.ws;
	HitsGuard hits(d.ctx);
	const int rc = dmnd_search_shape_range(d.ctx, d.qb, d.rb, 0, q_begin, q_end, &hits.h, &d.stats.seed);
	turn.pass(lane);
	if (rc) return 1;
	prof.lap("search_shape");
	d.stats.hits = dmnd_hits_count(hits.h);
	d.stats.seed_ms = ms_since(t0);
	t0 = Clock::now();
	if (dmnd_hits_chain(d.ctx, d.qb, d.rb, hits.h, d.env.sc->raw_ungapped_xdrop, d.env.band_slow ? 1 : 0, 64, &co)) return 1;
	const size_t nh = (size_t)co.n_host_hits;
	if (w.cq.resize(d.ctx, (size_t)co.n_queries) || w.cprobs.resize(d.ctx, (size_t)co.n_problems) || w.cres.resize(d.ctx, (size_t)co.n_problems)
	    || w.hv.resize(d.ctx, nh) || w.segv.resize(d.ctx, nh) || w.sitev.resize(d.ctx, nh))
		return 1;
	if (dmnd_hits_chain_fetch(d.ctx, w.cq.data(), w.cprobs.data(), w.hv.data(), w.segv.data(), w.sitev.data())) return 1;
	d.stats.host_bridge_ms += ms_since(t0);
	prof.lap("hits_chain (device bridge)");
	w.gfv.assign(nh, 1);  // (the mode has no gapped filter)
	return 0;
}

// Seed stage of every other mode, run_ref_chunk's loop over the shapes (run/double_indexed.cpp:185-214): SEED_MASK bits set by one shape
// stay visible to the next ones.  Every hit comes with its x-drop segment (align/ungapped.cpp:88), its site in the reference block and,
// where the mode has one, its gapped-filter verdict.  The hits of all shapes feed one extension: the shapes' query-grouped lists are
// merged into one (counting sort by query, stable).  Leaves the lane's hits in hv / segv / sitev / gfv [0, nh).
static int seed_host(Driver& d, uint32_t q_begin, uint32_t q_end, int lane, SeedTurn& turn, size_t& nh, Prof& prof) {
	Workspace& w = *d.ws;
	const Env& env = d.env;
	const int n_shapes = env.n_shapes;
	w.acc_hits.clear(); w.acc_segs.clear(); w.acc_sites.clear(); w.acc_gf.clear(); w.gfv.clear();
	for (int sid = 0; sid < n_shapes; ++sid) {
		HitsGuard hits(d.ctx);
		dmnd_stage_counters cn;
		if (dmnd_search_shape_range(d.ctx, d.qb, d.rb, sid, q_begin, q_end, &hits.h, &cn)) return 1;
		if (n_shapes == 1) turn.pass(lane);  // (with several shapes the turn passes once every shape's hits are down)
		add_counters(d.stats.seed, cn);
		const size_t n = dmnd_hits_count(hits.h);
		std::vector<uint8_t>& gf = n_shapes == 1 ? w.gfv : w.acc_gf;  // this shape's gapped-filter verdicts go to its end
		gf.resize(gf.size() + n, 1);
		if (w.hv.resize(d.ctx, n) || w.segv.resize(d.ctx, n) || w.sitev.resize(d.ctx, n)) return 1;
		if (n && (dmnd_hits_download(d.ctx, hits.h, w.hv.data(), n) || dmnd_hits_xdrop_sites(d.ctx, d.qb, d.rb, hits.h, env.sc->raw_ungapped_xdrop, w.segv.data(), w.sitev.data(), n)))
			return 1;
		if (n && env.gapped_filter && dmnd_hits_gapped_filter(d.ctx, d.qb, d.rb, hits.h, gf.data() + gf.size() - n, n)) return 1;  // align/gapped_filter.cpp, per hit
		if (n_shapes > 1) {
			w.acc_hits.insert(w.acc_hits.end(), w.hv.begin(), w.hv.end()); w.acc_segs.insert(w.acc_segs.end(), w.segv.begin(), w.segv.end());
			w.acc_sites.insert(w.acc_sites.end(), w.sitev.begin(), w.sitev.end());
		}
	}
	turn.pass(lane);
	prof.lap("search_shape + hits download (every shape)");
	nh = w.hv.size();
	if (n_shapes > 1) {
		const std::vector<dmnd_hit>& ah = w.acc_hits;
		nh = ah.size();
		if (w.hv.resize(d.ctx, nh) || w.segv.resize(d.ctx, nh) || w.sitev.resize(d.ctx, nh)) return 1;
		std::vector<size_t> off((size_t)(q_end - q_begin) + 1, 0);
		for (const dmnd_hit& h : ah) ++off[(size_t)(h.query - q_begin) + 1];
		for (size_t k = 1; k < off.size(); ++k) off[k] += off[k - 1];
		w.gfv.resize(nh);
		for (size_t k = 0; k < nh; ++k) {
			const size_t o = off[(size_t)(ah[k].query - q_begin)]++;
			w.hv[o] = ah[k]; w.segv[o] = w.acc_segs[k]; w.sitev[o] = w.acc_sites[k]; w.gfv[o] = w.acc_gf[k];
		}
	}
	if (env.min_length_ratio > 0.0) {
		// mutual-coverage seed stage (search/hamming/kernel_mutual_cov.h:28-52, chosen by stage1_dispatch when min_length_ratio > 0): over
		// length-sorted blocks its two cursors admit exactly the (query, target) pairs with qlen / tlen >= mlr and tlen / qlen >= mlr.
		// Every later step of the seed stage is per pair, so dropping the other pairs' hits here gives the same hit list.
		const double mlr = env.min_length_ratio;
		size_t o = 0;
		for (size_t x = 0; x < nh; ++x) {
			const int ql = env.qlen(w.hv[x].query), tl = env.tlen(w.sitev[x].target);
			if ((double)ql / tl < mlr || (double)tl / ql < mlr) continue;
			if (o != x) { w.hv[o] = w.hv[x]; w.segv[o] = w.segv[x]; w.sitev[o] = w.sitev[x]; w.gfv[o] = w.gfv[x]; }
			++o;
		}
		nh = o;
	}
	d.stats.hits = nh;
	return 0;
}

// Bridged mode: the device-chained problem list is aligned where it lies and the host only scores and culls (consume_fused); the
// queries the device code left to the host load their hits as on the host path.
static int load_bridged(Driver& d, const dmnd_chain_out& co, Prof& prof) {
	Workspace& w = *d.ws;
	const Env& env = d.env;
	const size_t T = (size_t)d.T;
	auto t0 = Clock::now();
	const size_t np = (size_t)co.n_problems, nqh = (size_t)co.n_queries;
	uint8_t* trp = nullptr;
	size_t cap = 0;
	if (np && env.want_transcript) {
		std::vector<size_t> part(T, 0);
		w.run([&](int t) {
			const size_t b = np * (size_t)t / T, e = np * (size_t)(t + 1) / T;
			part[(size_t)t] = transcript_cap(env, w.cprobs.data() + b, e - b);
		});
		for (size_t c : part) cap += c;
		if (w.tr.resize(d.ctx, cap)) return 1;
		trp = w.tr.data();
	}
	if (np && dmnd_banded_swipe_chained(d.ctx, d.qb, d.rb, np, DMND_DP_TRACEBACK, w.cres.data(), trp, cap)) return 1;
	d.stats.dp2_ms += ms_since(t0);
	d.stats.dp_problems_round1 += np;
	prof.lap("banded_swipe (chained list)");
	t0 = Clock::now();
	d.nq_hit = nqh;
	w.qs.resize(nqh);
	w.hs.resize((size_t)co.n_host_hits);
	std::atomic<int> bad(0);
	w.run([&](int t) {
		ThreadCtx& tc = w.tc[(size_t)t];
		tc.reset();
		for (size_t k = d.block_begin(t), en = d.block_begin(t + 1); k < en; ++k) {
			QueryState& q = w.qs[k];
			const dmnd_chain_query& cq = w.cq[k];
			if (k > 0 && cq.query <= w.cq[k - 1].query) bad = 1;
			if (cq.flags & DMND_CHAIN_HOST) {
				q.qid = cq.query;
				Workspace::HitSeg* hs = w.gather(cq.first, (size_t)cq.first + cq.n_hits);
				d.load_hits(q, tc, hs, hs + cq.n_hits);
				d.start(q, tc);
			}
			else {
				d.start_bridged(q, tc, cq, w.cprobs.data() + cq.first);
				d.consume_fused(q, tc, w.cprobs.data() + cq.first, w.cres.data() + cq.first, trp);
			}
		}
	});
	if (bad) { dmnd_set_last_error("dmnd_blastp: dmnd_hits_chain records not in ascending query order"); return 1; }
	d.stats.host_bridge_ms += ms_since(t0);
	prof.lap("consume chained queries (parallel)");
	return 0;
}

// Host path: hv [0, nh) is grouped by ascending query id; one group per query = all its contexts (search/hit.h:71-78), boundaries found
// in parallel.  Every query then loads its hits (load_hits + start, or legacy_init in frameshift mode).
static int load_host(Driver& d, size_t nh, Prof& prof) {
	Workspace& w = *d.ws;
	const Env& env = d.env;
	const size_t T = (size_t)d.T;
	const uint32_t C = env.contexts;
	auto t0 = Clock::now();
	std::vector<std::vector<size_t>> tl_bounds(T);
	std::atomic<int> bad(0);
	w.run([&](int t) {
		auto& v = tl_bounds[(size_t)t];
		v.clear();
		for (size_t i = nh * (size_t)t / T, en = nh * (size_t)(t + 1) / T; i < en; ++i)
			if (i == 0 || w.hv[i].query / C != w.hv[i - 1].query / C) {
				if (i > 0 && w.hv[i].query < w.hv[i - 1].query) bad = 1;
				v.push_back(i);
			}
	});
	if (bad) { dmnd_set_last_error("dmnd_blastp: hits not grouped by ascending query"); return 1; }
	w.qstart.clear();
	for (const auto& v : tl_bounds) w.qstart.insert(w.qstart.end(), v.begin(), v.end());
	w.qstart.push_back(nh);
	const size_t nqh = w.qstart.size() - 1;
	d.nq_hit = nqh;
	w.qs.resize(nqh);
	w.hs.resize(nh);
	if (env.frame_shift) { d.lq.clear(); d.lq.resize(nqh); }
	prof.lap("group queries");
	w.run([&](int t) {
		ThreadCtx& tc = w.tc[(size_t)t];
		tc.reset();
		for (size_t k = d.block_begin(t), en = d.block_begin(t + 1); k < en; ++k) {
			QueryState& q = w.qs[k];
			q.qid = w.hv[w.qstart[k]].query / C * C;
			Workspace::HitSeg* hs = w.gather(w.qstart[k], w.qstart[k + 1]);
			Workspace::HitSeg* he = hs + (w.qstart[k + 1] - w.qstart[k]);
			if (env.frame_shift) { d.legacy_init(k, q, tc, hs, he); continue; }
			d.load_hits(q, tc, hs, he);
			d.start(q, tc);
		}
	});
	d.stats.host_bridge_ms += ms_since(t0);
	prof.lap("load_hits (parallel)");
	return 0;
}

// Emit: per-thread counts -> offsets -> parallel fill of the lane's output (matches grouped by ascending query), with the counters the
// threads kept.
static void emit_matches(Driver& d, LaneOut& lo, Prof& prof) {
	Workspace& w = *d.ws;
	const Scoring& sc = *d.env.sc;
	const size_t T = (size_t)d.T;
	auto t0 = Clock::now();
	std::vector<size_t> moff(T + 1, 0), troff(T + 1, 0);
	w.run([&](int t) {
		ThreadCtx& tc = w.tc[(size_t)t];
		for (size_t k = d.block_begin(t), en = d.block_begin(t + 1); k < en; ++k) {
			tc.n_matches += w.qs[k].matches.n;
			if (w.qs[k].matches.n) ++tc.n_aligned;
			else tc.unaligned.push_back(w.qs[k].qid);
		}
	});
	for (size_t t = 0; t < T; ++t) {
		const ThreadCtx& tc = w.tc[t];
		moff[t + 1] = moff[t] + tc.n_matches;
		troff[t + 1] = troff[t] + tc.trbuf.size();
		d.stats.targets += tc.n_targets; d.stats.queries_aligned += tc.n_aligned;
		d.stats.cells_round1 += tc.cells1; d.stats.cells_round2 += tc.cells2;
		d.stats.dp_problems_round2 += tc.fused_r2; d.stats.dp_problems_fused += tc.fused_r1;
		d.stats.targets_extended += tc.n_extended;
		lo.unaligned.insert(lo.unaligned.end(), tc.unaligned.begin(), tc.unaligned.end());  // threads own ascending query ranges
	}
	lo.matches->resize(moff[T]);
	lo.transcripts->resize(troff[T]);
	w.run([&](int t) {
		const ThreadCtx& tc = w.tc[(size_t)t];
		dmnd_match* o = lo.matches->data() + moff[(size_t)t];
		if (!tc.trbuf.empty()) std::memcpy(lo.transcripts->data() + troff[(size_t)t], tc.trbuf.data(), tc.trbuf.size());
		for (size_t k = d.block_begin(t), en = d.block_begin(t + 1); k < en; ++k) {
			const QueryState& q = w.qs[k];
			for (const Match& m : q.matches) {
				std::memset(o, 0, sizeof *o);
				o->query = m.h.ctx; o->target = m.target_block_id; o->score = m.h.score; o->evalue = m.h.evalue;
				o->bit_score = sc.bitscore(m.h.score);
				o->q_begin = m.r.q_begin; o->q_end = m.r.q_end; o->t_begin = m.r.t_begin; o->t_end = m.r.t_end;
				o->identities = m.r.identities; o->mismatches = m.r.mismatches; o->gap_openings = m.r.gap_openings;
				o->length = m.r.length; o->gaps = m.r.gaps; o->positives = m.r.positives;
				o->transcript_off = troff[(size_t)t] + m.tr_off; o->transcript_len = m.tr_len;
				o->reserved = m.end_frame;
				++o;
			}
		}
	});
	d.stats.matches = lo.matches->size();
	d.stats.host_bridge_ms += ms_since(t0);
	prof.lap("emit matches");
}

// The stages of one lane.  Wall time up to the end of the seed stage is seed_ms (the bridged mode's seed stage ends with its search),
// the DP calls go to dp1_ms / dp2_ms, and the host work between them (dmnd_hits_chain included) to host_bridge_ms.
static int lane_run(dmnd_ctx* ctx, dmnd_block* qb, const dmnd_block* rb, const Env& env, uint32_t q_begin, uint32_t q_end,
                    Workspace& w, int host_threads, LaneOut& lo, int lane, SeedTurn& turn) {
	TurnRelease release{ turn, lane };
	auto t_total = Clock::now();
	Driver d;
	d.ctx = ctx; d.qb = qb; d.rb = rb; d.ws = &w; d.T = host_threads; d.env = env;
	std::memset(&d.stats, 0, sizeof d.stats);
	w.lane = lane;
	dmnd_timing tm0, tm1;
	dmnd_timing_fetch(ctx, &tm0, DMND_TIMING_THIS_CONTEXT);  // snapshot: the device counters of this call are reported as a delta
	Prof prof;
	prof.lane = lane;
	const auto t_seed = Clock::now();
	if (prepare_range(d, q_begin, q_end, lane, turn, prof)) return 1;
	dmnd_chain_out co{};
	size_t nh = 0;
	if (env.bridge ? seed_bridged(d, q_begin, q_end, lane, turn, t_seed, co, prof) : seed_host(d, q_begin, q_end, lane, turn, nh, prof)) return 1;
	if (dmnd_block_clear_seed_mask_range(ctx, qb, q_begin, q_end)) return 1;  // run/double_indexed.cpp:211-212
	prof.lap("clear seed mask");
	if (!env.bridge) d.stats.seed_ms = ms_since(t_seed);
	if (env.bridge ? load_bridged(d, co, prof) : load_host(d, nh, prof)) return 1;
	if (env.frame_shift ? d.run_legacy() : d.run_waves()) return 1;
	prof.lap("run_waves");
	emit_matches(d, lo, prof);
	d.stats.total_ms = ms_since(t_total);
	dmnd_timing_fetch(ctx, &tm1, DMND_TIMING_THIS_CONTEXT);
	d.stats.device = device_delta(tm1, tm0);
	lo.stats = d.stats;
	return 0;
}

static void add_stats(dmnd_run_stats& a, const dmnd_run_stats& b) {
	add_counters(a.seed, b.seed);
	a.hits += b.hits; a.targets += b.targets; a.dp_problems_round1 += b.dp_problems_round1; a.dp_problems_round2 += b.dp_problems_round2;
	a.cells_round1 += b.cells_round1; a.cells_round2 += b.cells_round2; a.queries_aligned += b.queries_aligned; a.matches += b.matches;
	a.dp_problems_fused += b.dp_problems_fused; a.targets_extended += b.targets_extended;
	// wall-clock phase times of concurrent lanes overlap: report the longest lane
	a.seed_ms = std::max(a.seed_ms, b.seed_ms); a.host_bridge_ms = std::max(a.host_bridge_ms, b.host_bridge_ms);
	a.dp1_ms = std::max(a.dp1_ms, b.dp1_ms); a.dp2_ms = std::max(a.dp2_ms, b.dp2_ms);
	a.device.seed_ms += b.device.seed_ms; a.device.dp_score_ms += b.device.dp_score_ms; a.device.dp_trace_ms += b.device.dp_trace_ms;
	a.device.h2d_ms += b.device.h2d_ms; a.device.d2h_ms += b.device.d2h_ms; a.device.launches += b.device.launches;
	a.device.h2d_bytes += b.device.h2d_bytes; a.device.d2h_bytes += b.device.d2h_bytes;
}

// Host threads, number of staggered query lanes and their contiguous, letter-balanced query ranges
// (SequenceSet::partition, data/sequence_set.cpp:57-75, is the reference's analogue for its threads).
struct LanePlan {
	int host_threads = 1, nlanes = 1;
	std::vector<uint32_t> cut;
};
static LanePlan plan_lanes(uint32_t nq, const int64_t* q_limits, uint32_t contexts) {
	LanePlan p;
	p.host_threads = effective_cpus();
	if (const char* ev = std::getenv("DMND_HOST_THREADS")) p.host_threads = std::max(1, std::atoi(ev));
	// staggered query lanes (see SeedTurn): small inputs gain nothing; with the host bridge on the device 4 lanes measured best at 10^6
	// queries on 16 host CPUs (profiles/lane_sweep_r2.txt: 3 / 4 / 6 / 8 lanes = 64.5 / 49.4 / 58.2 / 67.6 ms per step)
	p.nlanes = nq < 40000u ? 1 : (int)std::min<uint32_t>(4u, std::max<uint32_t>(2u, nq / 250000u));
	if (const char* ev = std::getenv("DMND_LANES")) p.nlanes = std::max(1, std::min(8, std::atoi(ev)));
	p.nlanes = (int)std::min<uint32_t>((uint32_t)p.nlanes, std::max<uint32_t>(nq, 1));
	p.cut.assign((size_t)p.nlanes + 1, nq);
	p.cut[0] = 0;
	for (int l = 1; l < p.nlanes; ++l) {
		const int64_t want = q_limits[0] + (q_limits[nq] - q_limits[0]) * l / p.nlanes;
		p.cut[(size_t)l] = (uint32_t)(std::lower_bound(q_limits, q_limits + nq + 1, want) - q_limits);
		p.cut[(size_t)l] = p.cut[(size_t)l] / contexts * contexts;  // a query's contexts stay in one lane
		p.cut[(size_t)l] = std::min(std::max(p.cut[(size_t)l], p.cut[(size_t)l - 1]), nq);
	}
	return p;
}

static int mask_bits(const dmnd_search_opts* o) { return (o->masking ? DMND_MASK_TANTAN : 0) | (o->motif_masking ? DMND_MASK_MOTIF : 0); }

// mask_algo != 0: the blocks arrive unmasked (dmnd_blastp); the reference block is masked here, every lane masks its own
// query range.  mask_algo == 0: resident blocks, already in their searched state.
static int blastp_impl(dmnd_ctx* ctx, dmnd_block* qb, const dmnd_block* rb, const int8_t* q_letters, const int64_t* q_limits,
                       uint32_t nq, const int8_t* r_letters, const int64_t* r_limits, uint32_t nr, const dmnd_search_opts* opts,
                       int mask_algo, dmnd_result** out) {
	auto t_total = Clock::now();
	if (opts->masking < 0 || opts->masking > 1 || opts->motif_masking < 0 || opts->motif_masking > 1) {
		dmnd_set_last_error("dmnd_blastp: masking / motif_masking must be 0 or 1 (SEG masking is not part of this build)");
		return 1;
	}
	Shared& sh = shared();
	std::lock_guard<std::mutex> guard(sh.mtx);
	struct PoolReturn { void operator()(dmnd_result* r) const { result_pool().give(r); } };
	std::unique_ptr<dmnd_result, PoolReturn> res(result_pool().take());
	res->matches.resize(0); res->transcripts.resize(0);
	res->masked[0].clear(); res->masked[1].clear(); res->unaligned.clear();
	std::memset(&res->stats, 0, sizeof res->stats);
	Scoring sc;
	int64_t ref_letters = 0;
	for (uint32_t i = 0; i < nr; ++i) ref_letters += r_limits[i + 1] - r_limits[i] - 1;
	sc.db_letters = opts->db_letters ? (double)opts->db_letters : (double)ref_letters;
	const uint32_t contexts = opts->query_contexts > 1 ? (uint32_t)opts->query_contexts : 1u;
	if ((contexts != 1 && contexts != 6) || nq % contexts != 0) {
		dmnd_set_last_error("dmnd_blastp: query_contexts must be 1 or 6 with nq a multiple of it");
		return 1;
	}
	if ((uint32_t)std::max(dmnd_ctx_params(ctx)->query_contexts, 1) != contexts) {
		dmnd_set_last_error("dmnd_blastp: the context was created for another query_contexts (dmnd_params_init copies it from the options)");
		return 1;
	}
	const LanePlan plan = plan_lanes(nq, q_limits, contexts);
	const int host_threads = plan.host_threads, nlanes = plan.nlanes;
	sh.ensure(host_threads, nlanes);

	Env e;
	e.sc = &sc; e.q_letters = q_letters; e.r_letters = r_letters;
	e.q_limits = q_limits; e.r_limits = r_limits; e.nq = nq; e.nr = nr; e.ref_letters = ref_letters;
	e.max_target_seqs = opts->max_target_seqs == 0 ? INT_MAX : opts->max_target_seqs; e.outer_limit = opts->max_target_seqs; e.max_evalue = opts->max_evalue;
	if (opts->top_percent > 100.0) { dmnd_set_last_error("dmnd_blastp: top_percent must lie in [0, 100] (negative = not given)"); return 1; }
	if (opts->top_percent >= 0.0 && opts->top_percent < 100.0) e.top = opts->top_percent;
	else if (opts->top_percent == 100.0) e.max_target_seqs = INT_MAX;  // output/output_format.cpp:233-240: --top 100 = every target, ranked by e-value
	e.hauser = opts->comp_based_stats == 1; e.want_transcript = opts->want_transcript != 0;
	e.frame_shift = opts->frame_shift;
	if (e.frame_shift < 0 || (e.frame_shift > 0 && contexts != 6)) { dmnd_set_last_error("dmnd_blastp: frame_shift needs translated queries (query_contexts = 6) and a positive penalty"); return 1; }
	e.range_culling = opts->range_culling != 0;
	if (opts->range_cover < 0.0 || opts->range_cover > 100.0) { dmnd_set_last_error("dmnd_blastp: range_cover is a percentage (0 = the default, 50)"); return 1; }
	if (opts->range_cover > 0.0) e.range_cover = opts->range_cover;
	if (e.range_culling && !e.frame_shift) { dmnd_set_last_error("dmnd_blastp: query range culling is only supported in frameshift alignment mode"); return 1; }  // basic/config.cpp:824-825
	if (e.frame_shift) {
		// the legacy pipeline extends without composition bias (align/legacy/query_mapper.cpp:131: xdrop_ungapped(.., nullptr, ..);
		// banded_3frame_swipe takes no bias at all) and always keeps the transcript (output/output_format.cpp:256-257)
		e.hauser = false; e.want_transcript = true;
	}
	e.fuse = std::getenv("DMND_NO_FUSE") == nullptr;
	e.mask_algo = mask_algo; e.contexts = contexts;
	if (opts->ext_mode < 0 || opts->ext_mode > 2) { dmnd_set_last_error("dmnd_blastp: ext_mode is 0 (mode default), 1 (banded-fast) or 2 (banded-slow)"); return 1; }
	e.self_targets = opts->self_targets;
	e.min_bit_score = opts->min_bit_score;
	if (!(e.min_bit_score >= 0.0)) { dmnd_set_last_error("dmnd_blastp: min_bit_score must not be negative (0 = the e-value bound applies)"); return 1; }
	if (e.min_bit_score != 0.0) e.fuse = false;  // (the device bridge admits one ranking chunk of <= 64 targets: unaffected, but keep the tested host schedule)
	e.min_id = opts->min_id; e.query_cover = opts->query_cover; e.subject_cover = opts->subject_cover; e.approx_min_id = opts->approx_min_id;
	if (e.approx_min_id != 0.0 && e.min_id != 0.0) { dmnd_set_last_error("Incompatible options: --approx-id, --id."); return 1; }  // run/config.cpp:168-169
	if (!(e.min_id >= 0.0 && e.min_id <= 100.0) || !(e.query_cover >= 0.0 && e.query_cover <= 100.0) || !(e.subject_cover >= 0.0 && e.subject_cover <= 100.0) || !(e.approx_min_id >= 0.0 && e.approx_min_id <= 100.0)) {
		dmnd_set_last_error("dmnd_blastp: min_id, query_cover and subject_cover are percentages (0 = no filter)");
		return 1;
	}
	e.have_filters = e.min_id > 0.0 || e.query_cover > 0.0 || e.subject_cover > 0.0 || e.approx_min_id > 0.0;
	e.first_round_culling = !e.have_filters || e.top >= 0.0;  // align/extend.cpp:288 (config.toppercent.present(): --top 100 counts, see below)
	if (e.have_filters) e.fuse = false;  // fused rounds and the device bridge assume round 2 = the culled targets of round 1, in one step
	if (e.query_cover >= 50.0 && e.query_cover == e.subject_cover && contexts == 1) e.min_length_ratio = std::max(e.query_cover / 100 - 0.05, 0.0);  // run/config.cpp:156-159
	{
		const ModeTraits* mt = mode_traits(opts->sensitivity);
		if (!mt) { dmnd_set_last_error("dmnd_blastp: bad sensitivity"); return 1; }
		e.n_shapes = mt->n_shapes; e.gapped_filter = mt->gapped_filter_evalue > 0.0; e.band_slow = opts->ext_mode == 0 ? mt->band_slow : opts->ext_mode == 2; e.ranking_letters = mt->ranking_letters;  // --ext (search/setup.cpp:377-384)
		if (e.frame_shift) e.gapped_filter = false;  // Extension::gapped_filter belongs to Extension::extend, which frameshift mode does not run
	}
	e.bridge = e.n_shapes == 1 && e.fuse && e.contexts == 1 && !e.gapped_filter && !e.frame_shift;
	if (mask_algo) {
		// "Masking reference" (run/double_indexed.cpp:122-127) and the reference block's motif table, before its seed index
		uint64_t n_hard = 0;
		if (dmnd_block_mask(ctx, const_cast<dmnd_block*>(rb), mask_algo, 0, nr, &n_hard)) return 1;
		sh.r_mask_pos.resize((size_t)n_hard);
		if (n_hard && dmnd_block_mask_fetch(ctx, sh.r_mask_pos.data(), sh.r_mask_pos.size())) return 1;
		sh.r_patch.build(r_letters, r_limits, nr, 0, nr, sh.r_mask_pos.data(), sh.r_mask_pos.size());
		e.r_patch = &sh.r_patch;
	}

	// (the per-position composition bias of the queries is computed on the device by each lane for its own range)
	// reference side of the seed join, once per call, shared by the lanes (the reference rebuilds it per run as well)
	g_prof_epoch = Clock::now();
	if (dmnd_block_build_index(ctx, const_cast<dmnd_block*>(rb), 0)) return 1;

	const std::vector<uint32_t>& cut = plan.cut;
	std::vector<LaneOut> lo((size_t)nlanes);
	for (int l = 0; l < nlanes; ++l) {
		lo[(size_t)l].matches = nlanes == 1 ? &res->matches : &sh.lanes[(size_t)l]->out_matches;
		lo[(size_t)l].transcripts = nlanes == 1 ? &res->transcripts : &sh.lanes[(size_t)l]->out_transcripts;
	}
	std::vector<dmnd_ctx*> lctx((size_t)nlanes, ctx);
	for (int l = 1; l < nlanes; ++l)
		if (dmnd_ctx_lane(ctx, l - 1, &lctx[(size_t)l])) return 1;
	SeedTurn seed_turn;
	seed_turn.masked.assign((size_t)nlanes, 0);
	auto body = [&](int l) {
		LaneOut& o = lo[(size_t)l];
		try {
			o.rc = lane_run(lctx[(size_t)l], qb, rb, e, cut[(size_t)l], cut[(size_t)l + 1], *sh.lanes[(size_t)l], host_threads, o, l, seed_turn);
			if (o.rc) o.error = dmnd_last_error();  // the error text is thread-local in the CUDA library
		}
		catch (const std::exception& ex) { o.rc = 1; o.error = std::string("dmnd_blastp: ") + ex.what(); }
	};
	std::vector<std::thread> th;
	for (int l = 1; l < nlanes; ++l) th.emplace_back(body, l);
	body(0);
	for (auto& t : th) t.join();
	for (int l = 0; l < nlanes; ++l)
		if (lo[(size_t)l].rc) { dmnd_set_last_error(lo[(size_t)l].error.c_str()); return 1; }

	// ---- concatenate lanes (ascending query ranges); a single lane hands its vectors over, several are copied in parallel
	if (nlanes == 1) add_stats(res->stats, lo[0].stats);  // the lane wrote straight into the result
	else {
		std::vector<size_t> mo((size_t)nlanes + 1, 0), to((size_t)nlanes + 1, 0);
		for (int l = 0; l < nlanes; ++l) { mo[(size_t)l + 1] = mo[(size_t)l] + lo[(size_t)l].matches->size(); to[(size_t)l + 1] = to[(size_t)l] + lo[(size_t)l].transcripts->size(); }
		res->matches.resize(mo[(size_t)nlanes]);
		res->transcripts.resize(to[(size_t)nlanes]);
		const int T = host_threads;
		sh.pool->run([&](int t) {
			for (int l = 0; l < nlanes; ++l) {
				const LaneOut& o = lo[(size_t)l];
				const size_t n = o.matches->size(), b = n * (size_t)t / (size_t)T, e = n * (size_t)(t + 1) / (size_t)T;
				dmnd_match* dst = res->matches.data() + mo[(size_t)l];
				for (size_t k = b; k < e; ++k) { dst[k] = (*o.matches)[k]; dst[k].transcript_off += to[(size_t)l]; }
				const size_t nt = o.transcripts->size(), tb = nt * (size_t)t / (size_t)T, te = nt * (size_t)(t + 1) / (size_t)T;
				if (te > tb) std::memcpy(res->transcripts.data() + to[(size_t)l] + tb, o.transcripts->data() + tb, te - tb);
			}
		});
		for (int l = 0; l < nlanes; ++l) add_stats(res->stats, lo[(size_t)l].stats);
	}
	for (int l = 0; l < nlanes; ++l) res->unaligned.insert(res->unaligned.end(), lo[(size_t)l].unaligned.begin(), lo[(size_t)l].unaligned.end());
	if (mask_algo) {  // lanes cover ascending query ranges and report ascending offsets: concatenation is sorted
		for (int l = 0; l < nlanes; ++l) res->masked[0].insert(res->masked[0].end(), sh.lanes[(size_t)l]->mask_pos.begin(), sh.lanes[(size_t)l]->mask_pos.end());
		res->masked[1] = sh.r_mask_pos;
	}
	res->stats.total_ms = ms_since(t_total);
	*out = res.release();
	return 0;
}

int dmnd_blastp_resident(dmnd_ctx* ctx, dmnd_block* query, const dmnd_block* ref, const int8_t* q_letters, const int64_t* q_limits,
                         uint32_t nq, const int8_t* r_letters, const int64_t* r_limits, uint32_t nr, const dmnd_search_opts* opts,
                         dmnd_result** out) {
	return blastp_impl(ctx, query, ref, q_letters, q_limits, nq, r_letters, r_limits, nr, opts, 0, out);
}

int dmnd_blastp(dmnd_ctx* ctx, const int8_t* q_letters, size_t q_raw_len, const int64_t* q_limits, uint32_t nq,
                const int8_t* r_letters, size_t r_raw_len, const int64_t* r_limits, uint32_t nr, const dmnd_search_opts* opts,
                dmnd_result** out) {
	dmnd_block *qb = nullptr, *rb = nullptr;
	Prof prof;
	// the reference block first (the index build needs it), then the query block range by range on the copy stream: lane 0
	// starts as soon as ITS range is there, the other ranges travel while it already searches
	if (dmnd_block_upload(ctx, r_letters, r_raw_len, r_limits, nr, &rb)) return 1;
	const LanePlan plan = plan_lanes(nq, q_limits, opts->query_contexts > 1 ? (uint32_t)opts->query_contexts : 1u);
	if (dmnd_block_upload_ranges(ctx, q_letters, q_raw_len, q_limits, nq, plan.cut.data(), plan.nlanes, &qb)) { dmnd_block_free(ctx, rb); return 1; }
	prof.lap("e2e: block uploads (queries in flight)");
	const int rc = blastp_impl(ctx, qb, rb, q_letters, q_limits, nq, r_letters, r_limits, nr, opts, mask_bits(opts), out);
	prof.t = Clock::now();
	dmnd_block_free(ctx, qb); dmnd_block_free(ctx, rb);
	prof.lap("e2e: block frees");
	return rc;
}

const dmnd_match* dmnd_result_matches(const dmnd_result* r, size_t* n) { *n = r->matches.size(); return r->matches.data(); }
const uint8_t* dmnd_result_transcripts(const dmnd_result* r, size_t* n) { *n = r->transcripts.size(); return r->transcripts.data(); }
const dmnd_run_stats* dmnd_result_stats(const dmnd_result* r) { return &r->stats; }
const uint64_t* dmnd_result_masked_positions(const dmnd_result* r, int side, size_t* n) {
	const std::vector<uint64_t>& v = r->masked[side ? 1 : 0];
	*n = v.size();
	return v.data();
}
const uint32_t* dmnd_result_unaligned(const dmnd_result* r, size_t* n) { *n = r->unaligned.size(); return r->unaligned.data(); }
void dmnd_result_free(dmnd_result* r) { if (r) result_pool().give(r); }

}  // extern "C"
