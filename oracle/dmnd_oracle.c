/* dmnd_oracle.c -- CPU restatement (plain C) of the K layer of include/dmnd_b200.h.
 *
 * TEST INFRASTRUCTURE ONLY.  This file is the parity oracle for the CUDA kernels: it restates, loop by loop, what
 * the reference (bbuchfink/diamond v2.2.2, AVX2 dispatch) computes on the hot path, in scalar C.  It is linked only
 * by tests/ (and by __graft_entry__.smoke() / bench.py's cpu_baseline leg as the checker); the product library
 * libdmnd_b200.so contains none of it and fails loudly without a CUDA device.
 *
 * Pinned against the reference itself: tests/test_oracle_vs_reference.py links this file under the host pipeline
 * (diamond_b200/csrc/host) and requires byte-identical fmt-6 output with oracle/_ref/diamond (the unmodified
 * reference compiled by oracle/ref_build/Makefile) plus equal --log stage counters, on the committed fixtures: every
 * blastp sensitivity mode (--fast .. --ultra-sensitive), with and without the reference's default masking, tabular output
 * incl. the CIGAR / BTOP / gapped-sequence fields and the pairwise format (tests/golden/make_golden.py lists the levels).
 *
 * Reference sections restated (file:line in /root/reference/src):
 *   seed packing            basic/shape.h:113-171, basic/reduction.h:98-105, search/seed_array/enum_seeds.h:56-89
 *   partition / chunk order basic/seed.h:35-51, util/algo/partition.h:23-58, search/stage0.cpp:101-121
 *   join                    util/algo/hash_join.h:174-226 (semantics only: equi-join on the packed seed)
 *   entropy masking         search/seed_complexity.cpp:37-51,77-127
 *   stage 1 (Hamming)       search/hamming/kernel.h:29-75, search/hamming/finger_print.h:180-215
 *   stage 2 (left-most)     search/stage2.h:73-154, search/left_most.h:30-110, search/sse_dist.h:105-190 (SSE branch),
 *                           util/algo/pattern_matcher.h:23-65, util/sequence/sequence.h:30-40
 *   stage 2 (ungapped win.) search/stage2.h:41-57,104-154, dp/ungapped_align.cpp:244-257, dp/ungapped_simd.cpp:32-88 (call size -> 255 cap),
 *                           search/hamming/kernel.h:61-74 + hit_field.h:44-57 (1024-subject tiles, ascending survivors), util/scores/cutoff_table.h
 *   masking                 masking/tantan.cpp:43-214 (AVX2 object's fp32 order), masking/masking.cpp:76-166 (motif table, MaskingTable),
 *                           util/kmer/kmer.h:62-117, data/block/block.cpp:162-178, search/seed_array/enum_seeds.h:255-270
 *   gapped filter           align/gapped_filter.cpp:33-63, dp/scan_diags.cpp:30-297, dp/score_profile.cpp:32-65
 *   banded SWIPE            dp/swipe/banded_swipe.h:189-351, dp/swipe/cell_update.h:103-141,
 *                           dp/swipe/banded_matrix.h:313-445, dp/swipe/target_iterator.h:59-173, dp/dp.h:47-52
 *   traceback walk          dp/swipe/banded_swipe.h:127-187, basic/hssp.cpp:260-290
 */
#include "../include/dmnd_b200.h"
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>
#include "../diamond_b200/csrc/host/motif_table.h"

static char g_err[512];
const char* dmnd_last_error(void) { return g_err; }
void dmnd_set_last_error(const char* m) { snprintf(g_err, sizeof g_err, "%s", m); }
const char* dmnd_backend(void) { return "oracle-cpu"; }
struct dmnd_ctx;
const dmnd_params* dmnd_ctx_params(const dmnd_ctx* ctx);
static int fail(const char* m) { snprintf(g_err, sizeof g_err, "%s", m); return 1; }

struct dmnd_block {
	int8_t* letters;
	int8_t* bias;
	uint8_t* soft_buf; /* 1 = letter inside a MaskingTable entry (abundant motif) */
	uint8_t* soft;     /* == soft_buf once dmnd_block_mask(MOTIF) has run, NULL before */
	size_t raw_len;
	int64_t* limits;
	uint32_t nseq;
};
struct dmnd_ctx {
	dmnd_params p;
	uint8_t* matcher[DMND_MAX_SHAPES + 1]; /* matcher[k] = PatternMatcher over shapes [0,k) */
	uint32_t m_minlen[DMND_MAX_SHAPES + 1], m_suffix[DMND_MAX_SHAPES + 1];
};
struct dmnd_hits { dmnd_hit* h; size_t n; };
const dmnd_params* dmnd_ctx_params(const dmnd_ctx* ctx) { return &ctx->p; }
/* letters hard-masked by the calling thread's last dmnd_block_mask (lanes share one oracle context but run on their own threads) */
static __thread uint64_t* t_mask_pos; static __thread size_t t_mask_n, t_mask_cap;

/* ---------------------------------------------------------------------------------------------------------- */
/* util/algo/pattern_matcher.h:25-45 */
static void build_matcher(dmnd_ctx* c, int k) {
	uint32_t minl = 32, maxl = 0;
	for (int i = 0; i < k; ++i) {
		uint32_t len = 32 - (uint32_t)__builtin_clz(c->p.shape_mask[i]);
		if (len > maxl) maxl = len;
		if (len < minl) minl = len;
	}
	c->m_minlen[k] = minl;
	c->m_suffix[k] = (1u << maxl) - 1;
	size_t sz = (size_t)c->m_suffix[k] + 1;
	c->matcher[k] = (uint8_t*)calloc(sz, 1);
	for (uint32_t s = 0; s <= c->m_suffix[k]; ++s)
		for (int i = 0; i < k; ++i)
			if ((s & c->p.shape_mask[i]) == c->p.shape_mask[i]) c->matcher[k][s] = 1;
}
/* util/algo/pattern_matcher.h:47-57 */
static uint32_t matcher_hit(const dmnd_ctx* c, int k, uint32_t h, uint32_t len) {
	if (len < c->m_minlen[k]) return 0;
	const uint32_t end = len - c->m_minlen[k] + 1;
	uint32_t r = 0;
	for (uint32_t i = 0; i < end; ++i) {
		r |= (uint32_t)c->matcher[k][h & c->m_suffix[k]] << i;
		h >>= 1;
	}
	return r;
}

int dmnd_create(int device, const dmnd_params* params, dmnd_ctx** out) {
	(void)device;
	dmnd_ctx* c = (dmnd_ctx*)calloc(1, sizeof *c);
	c->p = *params;
	for (int k = 0; k <= params->n_shapes; ++k) build_matcher(c, k);
	*out = c;
	return 0;
}
int dmnd_ctx_lane(dmnd_ctx* ctx, int lane, dmnd_ctx** out) { (void)lane; *out = ctx; return 0; } /* the CPU restatement is stateless per call */
void dmnd_destroy(dmnd_ctx* c) {
	if (!c) return;
	for (int k = 0; k <= c->p.n_shapes; ++k) free(c->matcher[k]);
	free(c);
}

int dmnd_block_upload(dmnd_ctx* ctx, const int8_t* letters, size_t raw_len, const int64_t* limits, uint32_t nseq,
                      dmnd_block** out) {
	(void)ctx;
	dmnd_block* b = (dmnd_block*)calloc(1, sizeof *b);
	b->letters = (int8_t*)malloc(raw_len);
	memcpy(b->letters, letters, raw_len);
	b->bias = (int8_t*)calloc(raw_len, 1);
	b->soft_buf = (uint8_t*)calloc(raw_len, 1);
	b->raw_len = raw_len;
	b->limits = (int64_t*)malloc(sizeof(int64_t) * ((size_t)nseq + 1));
	memcpy(b->limits, limits, sizeof(int64_t) * ((size_t)nseq + 1));
	b->nseq = nseq;
	*out = b;
	return 0;
}
int dmnd_block_upload_ranges(dmnd_ctx* ctx, const int8_t* letters, size_t raw_len, const int64_t* limits, uint32_t nseq,
                             const uint32_t* cuts, int nranges, dmnd_block** out) {
	if (nranges < 1 || nranges > 64 || cuts[0] != 0 || cuts[nranges] != nseq) return fail("dmnd_block_upload_ranges: cuts must run from 0 to nseq in 1..64 ranges");
	return dmnd_block_upload(ctx, letters, raw_len, limits, nseq, out); /* nothing to overlap on the CPU */
}
int dmnd_block_range_wait(dmnd_ctx* ctx, const dmnd_block* b, uint32_t s_begin, uint32_t s_end) { (void)ctx; (void)b; (void)s_begin; (void)s_end; return 0; }
void dmnd_block_free(dmnd_ctx* ctx, dmnd_block* b) {
	(void)ctx;
	if (!b) return;
	free(b->letters); free(b->bias); free(b->soft_buf); free(b->limits); free(b);
}
int dmnd_block_set_bias(dmnd_ctx* ctx, dmnd_block* b, const int8_t* bias, size_t raw_len) {
	(void)ctx;
	if (raw_len != b->raw_len) return fail("dmnd_block_set_bias: length mismatch");
	if (bias) memcpy(b->bias, bias, raw_len); else memset(b->bias, 0, raw_len);
	return 0;
}
/* stats/hauser_correction.cpp:53-109 (same loop structure: five phases of the sliding 40-letter window) */
static void hauser_one(const dmnd_params* p, const int8_t* seq, int len, int8_t* out) {
	int scores[20];
	memset(scores, 0, sizeof scores);
	const unsigned window = 40, l = (unsigned)len, window_half = (window / 2 < l - 1) ? window / 2 : l - 1;
	unsigned n = 0, h = 0, m = 0, t = 0;
	memset(out, 0, (size_t)len);
#define SC(a, b) ((int)p->score[(a) * 32 + (b)])
#define ADD(pos) do { const int _l = seq[pos] & 31; for (int _i = 0; _i < 20; ++_i) scores[_i] += SC(_l, _i); } while (0)
#define SUB(pos) do { const int _l = seq[pos] & 31; for (int _i = 0; _i < 20; ++_i) scores[_i] -= SC(_l, _i); } while (0)
#define EMIT(pos) do { const int _r = seq[pos] & 31; if (_r < 20) { const float _f = p->background_scores_f32[_r] - (float)(scores[_r] - SC(_r, _r)) / (float)(n - 1); \
		out[pos] = (int8_t)(_f < 0.0f ? _f - 0.5f : _f + 0.5f); } } while (0)
	while (n < window_half && h < l) { ++n; ADD(h); ++h; }
	while (n < (window + 1) && h < l) { ++n; ADD(h); EMIT(m); ++h; ++m; }
	while (h < l) { ADD(h); SUB(t); EMIT(m); ++h; ++t; ++m; }
	while (m < l && n > (window_half + 1)) { --n; SUB(t); EMIT(m); ++t; ++m; }
	while (m < l) { EMIT(m); ++m; }
#undef SC
#undef ADD
#undef SUB
#undef EMIT
}
int dmnd_block_build_index(dmnd_ctx* ctx, dmnd_block* b, int sid) { (void)ctx; (void)b; (void)sid; return 0; } /* the restatement joins per call */
int dmnd_block_compute_bias_range(dmnd_ctx* ctx, dmnd_block* b, int mode, uint32_t s_begin, uint32_t s_end) {
	if (mode != 0 && mode != 1) return fail("dmnd_block_compute_bias: unknown mode");
	if (s_begin > s_end || s_end > b->nseq) return fail("dmnd_block_compute_bias_range: sequence range out of bounds");
	if (s_begin == s_end) return 0;
	memset(b->bias + b->limits[s_begin], 0, (size_t)(b->limits[s_end] - b->limits[s_begin]));
	if (mode == 0) return 0;
	for (uint32_t i = s_begin; i < s_end; ++i) {
		const int64_t beg = b->limits[i];
		const int len = (int)(b->limits[i + 1] - beg - 1);
		if (len > 0) hauser_one(&ctx->p, b->letters + beg, len, b->bias + beg);
	}
	return 0;
}
int dmnd_block_compute_bias(dmnd_ctx* ctx, dmnd_block* b, int mode) {
	if (mode != 0 && mode != 1) return fail("dmnd_block_compute_bias: unknown mode");
	memset(b->bias, 0, b->raw_len);
	return dmnd_block_compute_bias_range(ctx, b, mode, 0, b->nseq);
}
int dmnd_block_download_bias(dmnd_ctx* ctx, const dmnd_block* b, int8_t* bias, size_t raw_len) {
	(void)ctx;
	if (raw_len != b->raw_len) return fail("dmnd_block_download_bias: length mismatch");
	memcpy(bias, b->bias, raw_len);
	return 0;
}
int dmnd_block_download_bias_async(dmnd_ctx* ctx, const dmnd_block* b, int8_t* bias, size_t raw_len) { return dmnd_block_download_bias(ctx, b, bias, raw_len); }
int dmnd_copy_wait(dmnd_ctx* ctx) { (void)ctx; return 0; }
void* dmnd_host_alloc(dmnd_ctx* ctx, size_t bytes) { (void)ctx; return malloc(bytes ? bytes : 1); }
void dmnd_host_free(dmnd_ctx* ctx, void* p) { (void)ctx; free(p); }
int dmnd_block_download_letters(dmnd_ctx* ctx, const dmnd_block* b, int8_t* letters, size_t raw_len) {
	(void)ctx;
	if (raw_len != b->raw_len) return fail("dmnd_block_download_letters: length mismatch");
	memcpy(letters, b->letters, raw_len);
	return 0;
}
/* ---------------------------------------------------------------------------------------------------------- */
/* Masking.  masking/tantan.cpp:43-214 as the AVX2 dispatch object evaluates it (oracle/ref_build compiles that object
 * with -mavx2 and without -mfma, so Traits<float>::LANES == 8 and fmadd(a,b,c) == add(mul(a,b),c),
 * util/simd/vector8_avx2.h:124-139): every product and sum is a separate IEEE fp32 operation, horizontal sums go
 * through hsum's ((a0+a4)+(a1+a5)) + ((a2+a6)+(a3+a7)) tree, register sums are accumulated left to right, the two tail
 * elements 48 and 49 last.  Compile with -ffp-contract=off (Makefile). */
#define TT_W 50
static float tt_hsum8(const float* a) { const float s0 = a[0] + a[4], s1 = a[1] + a[5], s2 = a[2] + a[6], s3 = a[3] + a[7]; return (s0 + s1) + (s2 + s3); }
/* util/simd/vector.h:37-48 sum(x, 50) */
static float tt_sum50(const float* x) {
	float acc[8];
	for (int k = 0; k < 8; ++k) acc[k] = 0.0f;
	for (int r = 0; r < 6; ++r) for (int k = 0; k < 8; ++k) acc[k] = acc[k] + x[8 * r + k];
	float sum = tt_hsum8(acc);
	sum += x[48]; sum += x[49];
	return sum;
}
/* e_seg[off] of tantan.cpp:163-171,181: the likelihood ratio of letter i against the letter off+1 positions before it */
static float tt_e(const dmnd_params* p, const int8_t* seq, int i, int ltr, int off) {
	const int j = i - 1 - off;
	return j >= 0 ? p->tantan_lr[ltr * 32 + (seq[j] & DMND_LETTER_MASK)] : 0.0f;
}
/* Util::tantan::mask(seq, len, ..., mask_mode 1): returns the number of letters set to MASK_LETTER, their offsets
 * (base + i) are appended to ctx->mask_pos. */
static size_t tantan_one(const dmnd_params* p, int8_t* seq, int len, uint64_t base, float* log2_ratio) {
	if (len == 0) return 0;
	const float* d = p->tantan_d;
	const float b2b = p->tantan_b2b, f2f = p->tantan_f2f, p_repeat_end = p->tantan_p_repeat_end, p_mask = p->tantan_p_mask;
	float f[TT_W];
	float* pb = (float*)malloc(sizeof(float) * (size_t)len);
	float* scale = (float*)malloc(sizeof(float) * (size_t)((len - 1) / 16 + 1));
	for (int k = 0; k < TT_W; ++k) f[k] = 0.0f;
	float b = 1.0f, f_sum = 0.0f;
	float log2_unscale = 0.0f; /* test-only: log2 of the product of the b's the rescaling divided by (see dmnd_oracle_tantan_log2_ratio) */
	for (int i = 0; i < len; ++i) {
		const int ltr = seq[i] & DMND_LETTER_MASK;
		/* forward_step, tantan.cpp:43-76 */
		const float b_old = b;
		float f_sum_new = 0.0f;
		for (int r = 0; r < 6; ++r) {
			for (int k = 0; k < 8; ++k) {
				const int off = 8 * r + k;
				const float tmp = f[off] * f2f + b_old * d[off];
				f[off] = tmp * tt_e(p, seq, i, ltr, off);
			}
			f_sum_new += tt_hsum8(f + 8 * r);
		}
		for (int off = 48; off < 50; ++off) {
			float vf = f[off];
			vf = (vf * f2f + b_old * d[off]) * tt_e(p, seq, i, ltr, off);
			f[off] = vf;
			f_sum_new += vf;
		}
		b = b_old * b2b + f_sum * p_repeat_end;
		f_sum = f_sum_new;
		if ((i & 15) == 15) {
			const float s = 1.0f / b;
			log2_unscale += log2f(b);
			scale[i / 16] = s;
			b *= s;
			for (int k = 0; k < TT_W; ++k) f[k] = f[k] * s;
			f_sum *= s;
		}
		pb[i] = b;
	}
	const float z = b * b2b + tt_sum50(f) * p_repeat_end;
	const float zinv = 1.0f / z;
	if (log2_ratio) *log2_ratio = log2f(z) + log2_unscale - (float)(len + 1) * log2f(b2b);
	b = b2b;
	for (int k = 0; k < TT_W; ++k) f[k] = p_repeat_end;
	size_t n = 0;
	for (int i = len - 1; i >= 0; --i) {
		const float pf = 1.0f - (pb[i] * b * zinv);
		if ((i & 15) == 15) {
			const float s = scale[i / 16];
			b *= s;
			for (int k = 0; k < TT_W; ++k) f[k] = f[k] * s;
		}
		const int ltr = seq[i] & DMND_LETTER_MASK;
		/* backward_step, tantan.cpp:78-111 */
		const float vC = p_repeat_end * b;
		float tsum = 0.0f;
		for (int r = 0; r < 6; ++r) {
			float vt[8];
			for (int k = 0; k < 8; ++k) {
				const int off = 8 * r + k;
				const float vf = f[off] * tt_e(p, seq, i, ltr, off);
				vt[k] = vf * d[off];
				f[off] = vf * f2f + vC;
			}
			tsum += tt_hsum8(vt);
		}
		for (int off = 48; off < 50; ++off) {
			float vf = f[off] * tt_e(p, seq, i, ltr, off);
			tsum += vf * d[off];
			vf = vf * f2f + p_repeat_end * b;
			f[off] = vf;
		}
		b = b2b * b + tsum;
		if (pf >= p_mask) {
			seq[i] = 23; /* value_traits.mask_char: MASK_LETTER */
			if (t_mask_n == t_mask_cap) { t_mask_cap = t_mask_cap ? t_mask_cap * 2 : 1024; t_mask_pos = (uint64_t*)realloc(t_mask_pos, t_mask_cap * sizeof(uint64_t)); }
			t_mask_pos[t_mask_n++] = base + (uint64_t)i;
			++n;
		}
	}
	free(pb); free(scale);
	return n;
}
static int cmp_u64(const void* a, const void* b) { const uint64_t x = *(const uint64_t*)a, y = *(const uint64_t*)b; return x < y ? -1 : x > y; }
/* masking/masking.cpp:110-131 mask_motifs: util/kmer/kmer.h:62-117 KmerIterator<8> (letters >= 20 restart the k-mer),
 * Mask::Ranges::push_back merging (masking/def.h:73-79), the >= 50 % rule and config.max_motif_len. */
static void motifs_one(const dmnd_params* p, const int8_t* seq, int len, uint8_t* soft) {
	if (len < DMND_MOTIF_LEN) return;
	uint8_t* cov = (uint8_t*)calloc((size_t)len, 1);
	long n = 0;
	for (int i = 0; i + DMND_MOTIF_LEN <= len; ++i) {
		uint64_t code = 0;
		int ok = 1;
		for (int k = 0; k < DMND_MOTIF_LEN; ++k) {
			const int l = seq[i + k] & DMND_LETTER_MASK;
			if (l >= 20) { ok = 0; break; }
			code = code * 20 + (uint64_t)l;
		}
		if (!ok || !bsearch(&code, DMND_MOTIF_CODES, DMND_MOTIF_COUNT, sizeof(uint64_t), cmp_u64)) continue;
		for (int k = 0; k < DMND_MOTIF_LEN; ++k) cov[i + k] = 1;
	}
	for (int i = 0; i < len; ++i) n += cov[i];
	if ((double)n / len < 0.5)
		for (int i = 0; i < len;) {
			if (!cov[i]) { ++i; continue; }
			int e = i;
			while (e < len && cov[e]) ++e;
			if (e - i <= p->max_motif_len) memset(soft + i, 1, (size_t)(e - i));
			i = e;
		}
	free(cov);
}
int dmnd_block_mask(dmnd_ctx* ctx, dmnd_block* b, int algo, uint32_t s_begin, uint32_t s_end, uint64_t* n_hard) {
	if (s_begin > s_end || s_end > b->nseq) return fail("dmnd_block_mask: bad sequence range");
	if (algo & ~(DMND_MASK_TANTAN | DMND_MASK_MOTIF)) return fail("dmnd_block_mask: unknown masking algorithm");
	t_mask_n = 0;
	if (algo & DMND_MASK_TANTAN)
		for (uint32_t i = s_begin; i < s_end; ++i)
			tantan_one(&ctx->p, b->letters + b->limits[i], (int)(b->limits[i + 1] - b->limits[i] - 1), (uint64_t)b->limits[i], NULL);
	if (t_mask_n) qsort(t_mask_pos, t_mask_n, sizeof(uint64_t), cmp_u64);
	if (algo & DMND_MASK_MOTIF) {
		__atomic_store_n(&b->soft, b->soft_buf, __ATOMIC_RELAXED); /* (query lanes mask their own ranges of one block concurrently: same value from every lane) */
		for (uint32_t i = s_begin; i < s_end; ++i) {
			const int len = (int)(b->limits[i + 1] - b->limits[i] - 1);
			memset(b->soft_buf + b->limits[i], 0, (size_t)len);
			motifs_one(&ctx->p, b->letters + b->limits[i], len, b->soft_buf + b->limits[i]);
		}
	}
	if (n_hard) *n_hard = t_mask_n;
	return 0;
}
int dmnd_block_mask_fetch(dmnd_ctx* ctx, uint64_t* positions, size_t cap) {
	(void)ctx;
	if (cap < t_mask_n) return fail("dmnd_block_mask_fetch: buffer too small");
	if (t_mask_n) memcpy(positions, t_mask_pos, t_mask_n * sizeof(uint64_t));
	return 0;
}
int dmnd_block_clear_seed_mask_range(dmnd_ctx* ctx, dmnd_block* b, uint32_t q_begin, uint32_t q_end) {
	(void)ctx;
	if (q_begin > q_end || q_end > b->nseq) return fail("dmnd_block_clear_seed_mask_range: bad range");
	for (int64_t i = b->limits[q_begin]; i < b->limits[q_end]; ++i)
		if (b->letters[i] != DMND_DELIMITER) b->letters[i] &= 0x7f;
	return 0;
}
int dmnd_block_clear_seed_mask(dmnd_ctx* ctx, dmnd_block* b) {
	(void)ctx;
	for (size_t i = 0; i < b->raw_len; ++i)
		if (b->letters[i] != DMND_DELIMITER) b->letters[i] &= 0x7f; /* only bit 7 is ever added */
	return 0;
}
int dmnd_measure_int_peak(dmnd_ctx* ctx, double* v) { (void)ctx; *v = 0; return fail("oracle: no device to measure"); }
int dmnd_measure_int_peak_packed(dmnd_ctx* ctx, double* v) { (void)ctx; *v = 0; return fail("oracle: no device to measure"); }
int dmnd_timing_fetch(dmnd_ctx* ctx, dmnd_timing* out, int reset) {
	(void)ctx; (void)reset;
	memset(out, 0, sizeof *out);
	return 0;
}

/* ---------------------------------------------------------------------------------------------------------- */
/* Seed stage                                                                                                  */
typedef struct { uint64_t seed; uint64_t loc; } entry;
static int cmp_entry(const void* a, const void* b) {
	const entry *x = (const entry*)a, *y = (const entry*)b;
	if (x->seed != y->seed) return x->seed < y->seed ? -1 : 1;
	return x->loc < y->loc ? -1 : (x->loc > y->loc);
}

/* basic/shape.h:113-171 on a sequence reduced by basic/reduction.h:98-105: invalid iff any class == MASK (23). */
static int seed_at(const dmnd_params* p, int sid, const int8_t* s, const uint8_t* soft, uint64_t* out) {
	uint64_t v = 0;
	for (int k = 0; k < p->shape_weight; ++k) {
		const int pos = p->shape_pos[sid][k];
		/* a soft-masked letter reads as MASK_LETTER while the seeds are enumerated (Block::soft_mask, data/block/block.cpp:162-171) */
		const unsigned r = (soft && soft[pos]) ? 23u : p->reduction[s[pos] & DMND_LETTER_MASK];
		if (r == 23) return 0;
		v = v * (uint64_t)p->reduction_size + r;
	}
	*out = v;
	return 1;
}
/* basic/shape.h:73-96 Shape::set_seed (un-reduced input, is_amino_acid test) -- used by verify_hit only. */
static int seed_at_unreduced(const dmnd_params* p, int sid, const int8_t* s, uint64_t* out) {
	uint64_t v = 0;
	for (int k = 0; k < p->shape_weight; ++k) {
		const int l = s[p->shape_pos[sid][k]] & DMND_LETTER_MASK;
		if (l == 23 || l == 31 || l == 24) return 0;
		v = v * (uint64_t)p->reduction_size + p->reduction[l];
	}
	*out = v;
	return 1;
}

static size_t enum_seeds(const dmnd_params* p, int sid, const dmnd_block* b, uint32_t pbegin, uint32_t pend, uint32_t s_begin, uint32_t s_end, entry** out) {
	const uint64_t mask = ((uint64_t)1 << p->seedp_bits) - 1;
	const int span = p->shape_len[sid];
	size_t n = 0, cap = 1024;
	entry* e = (entry*)malloc(cap * sizeof *e);
	for (uint32_t i = s_begin; i < s_end; ++i) {
		const int64_t beg = b->limits[i], len = b->limits[i + 1] - b->limits[i] - 1;
		for (int64_t j = 0; j + span <= len; ++j) {
			uint64_t s;
			if (!seed_at(p, sid, b->letters + beg + j, b->soft ? b->soft + beg + j : NULL, &s)) continue;
			const uint32_t part = (uint32_t)(s & mask);
			if (part < pbegin || part >= pend) continue;
			if (n == cap) { cap *= 2; e = (entry*)realloc(e, cap * sizeof *e); }
			e[n].seed = s; e[n].loc = (uint64_t)(beg + j); ++n;
		}
	}
	qsort(e, n, sizeof *e, cmp_entry);
	*out = e;
	return n;
}

/* lib/blast/blast_seg.cpp:54-58: ln(n!) rounded to 6 decimals, as tabulated by the reference. */
static const double LNFACT[13] = { 0.000000, 0.000000, 0.693147, 1.791759, 3.178054, 4.787492, 6.579251, 8.525161,
	10.604603, 12.801827, 15.104413, 17.502308, 19.987214 };
/* search/seed_complexity.cpp:37-51 */
static int seed_is_complex(const dmnd_params* p, int sid, const int8_t* seq) {
	unsigned count[20] = { 0 };
	for (int k = 0; k < p->shape_weight; ++k) {
		const int l = seq[p->shape_pos[sid][k]] & DMND_LETTER_MASK;
		if (l >= 20) return 0;
		++count[p->reduction[l]];
	}
	double entropy = LNFACT[p->shape_weight];
	for (int c = 0; c < p->reduction_size; ++c) entropy -= LNFACT[count[c]];
	return entropy >= p->seed_cut;
}

/* search/hamming/finger_print.h:180-202: 48 bytes at [loc-16, loc+32), & 31, count equal bytes. */
static unsigned fingerprint_match(const int8_t* q, const int8_t* s) {
	unsigned n = 0;
	for (int k = -16; k < 32; ++k) n += (q[k] & DMND_LETTER_MASK) == (s[k] & DMND_LETTER_MASK);
	return n;
}

/* util/sequence/sequence.h:30-40 */
static void clip(const int8_t* seq, int len, int anchor, const int8_t** obegin, const int8_t** oend) {
	const int8_t *a = seq + anchor, *begin = seq, *end = seq + len;
	for (;;) {
		const int8_t* p = (const int8_t*)memchr(begin, DMND_DELIMITER, (size_t)(end - begin));
		if (!p) { *obegin = begin; *oend = end; return; }
		if (p >= a) { *obegin = begin; *oend = p; return; }
		begin = p + 1;
	}
}

/* search/sse_dist.h:137-155 (SSE branch: map8 on the query side, map8b on the subject side, no amino-acid test) */
static uint64_t reduced_match(const dmnd_params* p, const int8_t* q, const int8_t* s, int len) {
	uint64_t m = 0;
	for (int k = 0; k < len && k < 64; ++k)
		if (p->map8[q[k] & DMND_LETTER_MASK] == p->map8b[s[k] & DMND_LETTER_MASK]) m |= (uint64_t)1 << k;
	return m;
}
/* search/sse_dist.h:157-170 */
static uint64_t seed_mask_bits(const int8_t* s, int len) {
	uint64_t m = 0;
	for (int k = 0; k < len && k < 64; ++k)
		if (s[k] & DMND_SEED_MASK) m |= (uint64_t)1 << k;
	return m;
}

typedef struct { const dmnd_ctx* c; int sid; int chunked; uint32_t range_begin, range_end; } lm_ctx;

/* search/left_most.h:30-49 */
static int verify_hit(const lm_ctx* x, const int8_t* q, const int8_t* s, int left, uint32_t match_mask) {
	const dmnd_params* p = &x->c->p;
	if (x->chunked) {
		if ((p->shape_mask[x->sid] & match_mask) == p->shape_mask[x->sid]) {
			uint64_t seed;
			if (!seed_at_unreduced(p, x->sid, s, &seed)) return 0;
			const uint32_t part = (uint32_t)(seed & (((uint64_t)1 << p->seedp_bits) - 1));
			if (left && !(part < x->range_end)) return 0;
			if (!left && !(part < x->range_begin)) return 0;
		}
	}
	return fingerprint_match(q, s) >= (unsigned)p->hamming_id;
}
/* search/left_most.h:51-60 */
static int verify_hits(const lm_ctx* x, uint32_t mask, const int8_t* q, const int8_t* s, int left, uint32_t match_mask) {
	int shift = 0;
	while (mask != 0) {
		const int i = __builtin_ctz(mask);
		if (verify_hit(x, q + i + shift, s + i + shift, left, match_mask >> (i + shift))) return 1;
		mask >>= i; mask >>= 1; /* (i + 1) may be 32 */
		shift += i + 1;
	}
	return 0;
}
/* search/left_most.h:62-110 */
static int left_most_filter(const lm_ctx* x, const int8_t* query, int query_len, const int8_t* subject, int seed_offset,
                            int seed_len) {
	const dmnd_ctx* c = x->c;
	const int first_shape = x->sid == 0;
	int d = seed_offset - 16 > 0 ? seed_offset - 16 : 0, window_left = seed_offset < 16 ? seed_offset : 16;
	const int8_t *q = query + d, *s = subject + d;
	int window = query_len - d;
	if (window > window_left + 1 + 32) window = window_left + 1 + 32;
	const int8_t *cb, *ce;
	clip(s, window, window_left, &cb, &ce);
	window -= (int)(s + window - ce);
	d = (int)(cb - s);
	q += d; s += d; window_left -= d; window -= d;

	const uint64_t match_mask = reduced_match(&c->p, q, s, window), query_seed_mask = ~seed_mask_bits(q, window);
	const uint32_t len_left = (uint32_t)(window_left + seed_len - 1),
		match_mask_left = (uint32_t)((((uint64_t)1 << len_left) - 1) & match_mask),
		query_mask_left = (uint32_t)((((uint64_t)1 << len_left) - 1) & query_seed_mask);
	const int cur = x->sid + 1, prev = x->sid;
	const uint32_t left_hit = matcher_hit(c, cur, match_mask_left, len_left) & query_mask_left;
	if (first_shape && !x->chunked)
		return left_hit == 0 || !verify_hits(x, left_hit, q, s, 1, match_mask_left);
	const uint32_t len_right = (uint32_t)(window - window_left - 1),
		match_mask_right = (uint32_t)(match_mask >> (window_left + 1)),
		query_mask_right = (uint32_t)(query_seed_mask >> (window_left + 1));
	const uint32_t right_hit = matcher_hit(c, x->chunked ? cur : prev, match_mask_right, len_right) & query_mask_right;
	return (left_hit == 0 || !verify_hits(x, left_hit, q, s, 1, match_mask_left))
		&& (right_hit == 0 || !verify_hits(x, right_hit, q + window_left + 1, s + window_left + 1, 0, match_mask_right));
}

static uint32_t seq_of(const dmnd_block* b, uint64_t loc) { /* SequenceSet::local_position: last i with limits[i] <= loc */
	uint32_t lo = 0, hi = b->nseq;
	while (hi - lo > 1) { uint32_t mid = lo + (hi - lo) / 2; if ((uint64_t)b->limits[mid] <= loc) lo = mid; else hi = mid; }
	return lo;
}

/* MaskingTable::remove(template_len, add_bit_mask = true) after the query enumeration (masking/masking.cpp:96-107,
 * search/seed_array/enum_seeds.h:255-260 with EnumCfg::mask_seeds of the query side, search/stage0.cpp:139-142):
 * every table entry [b, e) leaves SEED_MASK on [max(b - shape_len + 1, 0), e).  Entries are the maximal runs of `soft`. */
static void motif_seed_mask(const dmnd_params* p, dmnd_block* query, int sid, uint32_t q_begin, uint32_t q_end) {
	const int tl = p->shape_len[sid];
	for (uint32_t qi = q_begin; qi < q_end; ++qi) {
		const int64_t beg = query->limits[qi];
		const int len = (int)(query->limits[qi + 1] - beg - 1);
		for (int i = 0; i < len;) {
			if (!query->soft[beg + i]) { ++i; continue; }
			int e = i;
			while (e < len && query->soft[beg + e]) ++e;
			for (int j = (i - tl + 1 > 0 ? i - tl + 1 : 0); j < e; ++j) query->letters[beg + j] |= (int8_t)DMND_SEED_MASK;
			i = e;
		}
	}
}
/* ---- dmnd_hits_chain (test twin of cuda/chain.cu): the same records from the host code of diamond_b200/csrc/host (load_hits order,
 * segment filter, chaining.cpp, band merge) through dmnd_host_chain_pair.  No fixed capacities: only queries with more than
 * max_targets targets carry DMND_CHAIN_HOST. */
int dmnd_host_chain_pair(const int32_t* hit_i, const int32_t* hit_j, const dmnd_segment* hit_seg, int nh, const int8_t* query, int qlen,
                         const int8_t* subject, int slen, int band, int32_t* d0_out, int32_t* d1_out, int cap);
typedef struct { dmnd_chain_query* q; size_t nq; dmnd_dp_problem* probs; size_t np, pcap; dmnd_hit* fh; dmnd_segment* fs; dmnd_hit_site* ft; size_t nf, fcap; } chain_state;
static __thread chain_state t_chain;
static const dmnd_hit* g_sort_hits; static const dmnd_hit_site* g_sort_sites;
static __thread const dmnd_hit* t_sort_hits; static __thread const dmnd_hit_site* t_sort_sites;
static int cmp_chain_idx(const void* a, const void* b) {
	const uint32_t x = *(const uint32_t*)a, y = *(const uint32_t*)b;
	const dmnd_hit *hx = t_sort_hits + x, *hy = t_sort_hits + y;
	if (hx->query != hy->query) return hx->query < hy->query ? -1 : 1;
	if (t_sort_sites[x].target != t_sort_sites[y].target) return t_sort_sites[x].target < t_sort_sites[y].target ? -1 : 1;
	return x < y ? -1 : (x > y);
}
static int chain_band_for(int len, int slow) {
	if (!slow) return len < 50 ? 12 : len < 100 ? 16 : len < 250 ? 30 : len < 350 ? 40 : 64;
	return len < 50 ? 15 : len < 100 ? 20 : len < 150 ? 30 : len < 200 ? 50 : len < 250 ? 60 : len < 350 ? 100 : len < 500 ? 120 : 150;
}
int dmnd_hits_chain(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, const dmnd_hits* h, int raw_xdrop, int band_slow, int max_targets, dmnd_chain_out* out) {
	(void)g_sort_hits; (void)g_sort_sites;
	memset(out, 0, sizeof *out);
	chain_state* c = &t_chain;
	c->nq = c->np = c->nf = 0;
	const size_t n = h->n;
	if (n == 0) return 0;
	dmnd_segment* segs = (dmnd_segment*)malloc(n * sizeof *segs);
	dmnd_hit_site* sites = (dmnd_hit_site*)malloc(n * sizeof *sites);
	uint32_t* idx = (uint32_t*)malloc(n * sizeof *idx);
	if (dmnd_hits_xdrop_sites(ctx, query, ref, h, raw_xdrop, segs, sites, n)) { free(segs); free(sites); free(idx); return 1; }
	for (size_t k = 0; k < n; ++k) idx[k] = (uint32_t)k;
	t_sort_hits = h->h; t_sort_sites = sites;
	qsort(idx, n, sizeof *idx, cmp_chain_idx);
	free(c->q); c->q = (dmnd_chain_query*)malloc(n * sizeof *c->q);
	if (c->fcap < n) { free(c->fh); free(c->fs); free(c->ft); c->fh = (dmnd_hit*)malloc(n * sizeof *c->fh); c->fs = (dmnd_segment*)malloc(n * sizeof *c->fs); c->ft = (dmnd_hit_site*)malloc(n * sizeof *c->ft); c->fcap = n; }
	size_t npairs = 0;
	int32_t *hi = (int32_t*)malloc(n * sizeof *hi), *hj = (int32_t*)malloc(n * sizeof *hj);
	dmnd_segment* hs = (dmnd_segment*)malloc(n * sizeof *hs);
	for (size_t qb = 0; qb < n;) {
		const uint32_t qid = h->h[idx[qb]].query;
		size_t qe = qb;
		uint32_t ntg = 0, last = 0xffffffffu;
		while (qe < n && h->h[idx[qe]].query == qid) { if (sites[idx[qe]].target != last) { ++ntg; last = sites[idx[qe]].target; } ++qe; }
		npairs += ntg;
		dmnd_chain_query q; memset(&q, 0, sizeof q);
		q.query = qid; q.n_targets = ntg; q.n_hits = (uint32_t)(qe - qb);
		if ((int)ntg > max_targets) {
			q.flags = DMND_CHAIN_HOST; q.first = (uint32_t)c->nf;
			for (size_t k = qb; k < qe; ++k) { c->fh[c->nf] = h->h[idx[k]]; c->fs[c->nf] = segs[idx[k]]; c->ft[c->nf] = sites[idx[k]]; ++c->nf; }
		}
		else {
			q.first = (uint32_t)c->np;
			const int64_t qo = query->limits[qid];
			const int qlen = (int)(query->limits[qid + 1] - qo - 1);
			for (size_t pb = qb; pb < qe;) {
				const uint32_t tg = sites[idx[pb]].target;
				size_t pe = pb;
				int nh = 0;
				while (pe < qe && sites[idx[pe]].target == tg) { hi[nh] = h->h[idx[pe]].seed_offset; hj[nh] = sites[idx[pe]].j; hs[nh] = segs[idx[pe]]; ++nh; ++pe; }
				const int64_t to = ref->limits[tg];
				const int slen = (int)(ref->limits[tg + 1] - to - 1);
				int32_t d0[64], d1[64];
				const int np = dmnd_host_chain_pair(hi, hj, hs, nh, query->letters + qo, qlen, ref->letters + to, slen, chain_band_for(qlen, band_slow), d0, d1, 64);
				if (np < 0) { free(segs); free(sites); free(idx); free(hi); free(hj); free(hs); return fail("dmnd_hits_chain: more than 64 bands for one target"); }
				if (c->np + (size_t)np > c->pcap) { c->pcap = (c->np + (size_t)np) * 2 + 1024; c->probs = (dmnd_dp_problem*)realloc(c->probs, c->pcap * sizeof *c->probs); }
				for (int k = 0; k < np; ++k) { dmnd_dp_problem pr; pr.query = qid; pr.target = tg; pr.d_begin = d0[k]; pr.d_end = d1[k]; c->probs[c->np++] = pr; }
				q.n_problems += (uint32_t)np;
				pb = pe;
			}
		}
		c->q[c->nq++] = q;
		qb = qe;
	}
	free(segs); free(sites); free(idx); free(hi); free(hj); free(hs);
	out->n_queries = c->nq; out->n_pairs = npairs; out->n_problems = c->np; out->n_host_hits = c->nf;
	return 0;
}
int dmnd_hits_chain_fetch(dmnd_ctx* ctx, dmnd_chain_query* queries, dmnd_dp_problem* problems, dmnd_hit* hits, dmnd_segment* segs, dmnd_hit_site* sites) {
	(void)ctx;
	const chain_state* c = &t_chain;
	if (c->nq) memcpy(queries, c->q, c->nq * sizeof *queries);
	if (c->np) memcpy(problems, c->probs, c->np * sizeof *problems);
	if (c->nf) { memcpy(hits, c->fh, c->nf * sizeof *hits); memcpy(segs, c->fs, c->nf * sizeof *segs); memcpy(sites, c->ft, c->nf * sizeof *sites); }
	return 0;
}
int dmnd_banded_swipe_chained(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, size_t n, int mode, dmnd_dp_result* results, uint8_t* transcripts, size_t transcript_cap) {
	if (n != t_chain.np) return fail("dmnd_banded_swipe_chained: n is not the problem count of the last dmnd_hits_chain");
	return dmnd_banded_swipe(ctx, query, ref, t_chain.probs, n, mode, results, transcripts, transcript_cap);
}

/* multi-GPU entry points: nothing to broadcast on a CPU (the sharding logic is tested with gloo through diamond_b200/shard.py) */
int dmnd_comm_unique_id(void* out128) { (void)out128; return fail("oracle: no NCCL on the CPU"); }
int dmnd_comm_init(dmnd_ctx* ctx, int rank, int nranks, const void* id) { (void)ctx; (void)rank; (void)nranks; (void)id; return fail("oracle: no NCCL on the CPU"); }
void dmnd_comm_destroy(dmnd_ctx* ctx) { (void)ctx; }
int dmnd_block_broadcast(dmnd_ctx* ctx, int root, dmnd_block* src, dmnd_block** out) { (void)ctx; (void)root; (void)src; (void)out; return fail("oracle: no NCCL on the CPU"); }
int dmnd_block_alloc_empty(dmnd_ctx* ctx, size_t raw_len, uint32_t nseq, dmnd_block** out) { (void)ctx; (void)raw_len; (void)nseq; (void)out; return fail("oracle: not implemented"); }
int dmnd_block_geometry(const dmnd_block* b, size_t* raw_len, uint32_t* nseq) { *raw_len = b->raw_len; *nseq = b->nseq; return 0; }
int dmnd_block_download_limits(dmnd_ctx* ctx, const dmnd_block* b, int64_t* limits, size_t count) {
	(void)ctx;
	if (count != (size_t)b->nseq + 1) return fail("dmnd_block_download_limits: count must be nseq + 1");
	memcpy(limits, b->limits, count * sizeof *limits);
	return 0;
}

/* Diagnostics twin of the device library's dmnd_debug_left_most (tools/seed_stage_diag.py): same out30 layout. */
int dmnd_debug_left_most(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, int sid, int chunk, uint32_t qloc, uint32_t sloc, unsigned long long* out) {
	const dmnd_params* p = &ctx->p;
	const uint32_t parts_total = 1u << p->seedp_bits;
	const uint32_t nchunks = (uint32_t)p->index_chunks < parts_total ? (uint32_t)p->index_chunks : parts_total;
	const uint32_t psize = parts_total / nchunks, prem = parts_total % nchunks, bsel = (uint32_t)chunk < prem ? (uint32_t)chunk : prem;
	const uint32_t pb = bsel * (psize + 1) + ((uint32_t)chunk - bsel) * psize, pe = pb + ((uint32_t)chunk < prem ? psize + 1 : psize);
	lm_ctx x; x.c = ctx; x.sid = sid; x.chunked = p->index_chunks > 1; x.range_begin = pb; x.range_end = pe;
	memset(out, 0, 30 * sizeof *out);
	const int8_t *qp = query->letters + qloc, *sp = ref->letters + sloc;
	const uint32_t qid = seq_of(query, qloc);
	const int seed_offset0 = (int)((int64_t)qloc - query->limits[qid]);
	const int window0 = p->ungapped_window;
	const int8_t *cb, *ce;
	clip(qp - window0, window0 * 2, window0, &cb, &ce);
	const int window_left0 = (int)(qp - cb), window_clipped = (int)(ce - cb);
	const int interval_mod = p->left_most_interval > 0 ? seed_offset0 % p->left_most_interval : window_left0;
	const int overhang = window_left0 - interval_mod > 0 ? window_left0 - interval_mod : 0;
	const int8_t *qry = cb + overhang, *subject = sp - window_left0 + overhang;
	const int query_len = window_clipped - overhang, seed_offset = window_left0 - overhang, seed_len = p->shape_len[sid];
	out[0] = (unsigned long long)left_most_filter(&x, qry, query_len, subject, seed_offset, seed_len);
	int d = seed_offset - 16 > 0 ? seed_offset - 16 : 0, window_left = seed_offset < 16 ? seed_offset : 16;
	const int8_t *q = qry + d, *s = subject + d;
	int window = query_len - d;
	if (window > window_left + 1 + 32) window = window_left + 1 + 32;
	clip(s, window, window_left, &cb, &ce);
	window -= (int)(s + window - ce);
	d = (int)(cb - s);
	q += d; s += d; window_left -= d; window -= d;
	const uint64_t match_mask = reduced_match(p, q, s, window), seed_bits = seed_mask_bits(q, window), query_seed_mask = ~seed_bits;
	const uint32_t len_left = (uint32_t)(window_left + seed_len - 1), match_mask_left = (uint32_t)((((uint64_t)1 << len_left) - 1) & match_mask),
		query_mask_left = (uint32_t)((((uint64_t)1 << len_left) - 1) & query_seed_mask);
	const uint32_t raw_left = matcher_hit(ctx, sid + 1, match_mask_left, len_left), left_hit = raw_left & query_mask_left;
	const uint32_t len_right = (uint32_t)(window - window_left - 1), match_mask_right = (uint32_t)(match_mask >> (window_left + 1)), query_mask_right = (uint32_t)(query_seed_mask >> (window_left + 1));
	const uint32_t right_hit = matcher_hit(ctx, x.chunked ? sid + 1 : sid, match_mask_right, len_right) & query_mask_right;
	out[1] = match_mask; out[2] = seed_bits; out[3] = ((uint64_t)raw_left << 32) | left_hit; out[4] = right_hit;
	out[5] = ((uint64_t)(uint32_t)seed_offset << 32) | (uint32_t)window_left; out[6] = ((uint64_t)(uint32_t)window << 32) | len_left;
	out[7] = left_hit ? (unsigned long long)verify_hits(&x, left_hit, q, s, 1, match_mask_left) : 2;
	out[8] = right_hit ? (unsigned long long)verify_hits(&x, right_hit, q + window_left + 1, s + window_left + 1, 0, match_mask_right) : 2;
	int n = 0;
	for (int pos = 0; pos < 32 && n < 20; ++pos) {
		if (!((left_hit >> pos) & 1u)) continue;
		const uint32_t mm = match_mask_left >> pos;
		uint64_t seed = 0; int valid = 1;
		for (int k = 0; k < p->shape_weight; ++k) { const int l = s[pos + p->shape_pos[sid][k]] & DMND_LETTER_MASK; if (l == 23 || l == 31 || l == 24) valid = 0; seed = seed * (uint64_t)p->reduction_size + p->reduction[l]; }
		const uint32_t part = (uint32_t)(seed & (((uint64_t)1 << p->seedp_bits) - 1));
		out[9 + n] = ((uint64_t)pos << 56) | ((uint64_t)verify_hit(&x, q + pos, s + pos, 1, mm) << 48) | ((uint64_t)((p->shape_mask[sid] & mm) == p->shape_mask[sid]) << 40)
			| ((uint64_t)valid << 36) | ((uint64_t)fingerprint_match(q + pos, s + pos) << 24) | part;
		++n;
	}
	out[29] = (unsigned long long)n;
	return 0;
}
/* Test-only: tantan on every sequence of the block (letters are masked in place); out_ratio[i] = log2(Z / W_bg) of
 * sequence i as the device's forward kernel computes it (diamond_b200/csrc/cuda/mask_kernels.cuh: sequences with a ratio
 * below 3 skip the backward pass there), out_masked[i] = letters tantan masked in it.  tests/test_masking.py checks the
 * implication "ratio < 3  =>  nothing masked" on real and synthetic proteins. */
int dmnd_oracle_tantan_log2_ratio(dmnd_ctx* ctx, dmnd_block* b, float* out_ratio, uint32_t* out_masked) {
	t_mask_n = 0;
	for (uint32_t i = 0; i < b->nseq; ++i) {
		out_ratio[i] = 0.0f;
		out_masked[i] = (uint32_t)tantan_one(&ctx->p, b->letters + b->limits[i], (int)(b->limits[i + 1] - b->limits[i] - 1), (uint64_t)b->limits[i], out_ratio + i);
	}
	return 0;
}
/* Test-only views for tests/emu_mask.cpp (not part of include/dmnd_b200.h): the soft-masking table as one byte per letter,
 * and the SEED_MASK marking above on its own. */
int dmnd_oracle_block_soft(const dmnd_block* b, uint8_t* out, size_t raw_len) {
	if (raw_len != b->raw_len) return fail("dmnd_oracle_block_soft: length mismatch");
	if (b->soft) memcpy(out, b->soft, raw_len); else memset(out, 0, raw_len);
	return 0;
}
int dmnd_debug_block_soft(dmnd_ctx* ctx, const dmnd_block* b, uint8_t* out, size_t raw_len) { (void)ctx; return dmnd_oracle_block_soft(b, out, raw_len); }
/* every seed of the block for shape sid, sorted by (seed, location): what the reference's seed arrays hold (key = the packed seed) */
int dmnd_debug_ref_index(dmnd_ctx* ctx, const dmnd_block* ref, int sid, uint64_t* keys, uint32_t* locs, size_t cap, size_t* n) {
	if (sid < 0 || sid >= ctx->p.n_shapes) return fail("dmnd_debug_ref_index: bad shape id");
	entry* e;
	*n = enum_seeds(&ctx->p, sid, ref, 0, (uint32_t)1 << ctx->p.seedp_bits, 0, ref->nseq, &e);
	if (cap < *n) { free(e); return fail("dmnd_debug_ref_index: buffer too small"); }
	for (size_t k = 0; k < *n; ++k) { keys[k] = e[k].seed; locs[k] = (uint32_t)e[k].loc; }
	free(e);
	return 0;
}
int dmnd_oracle_motif_seed_mask(dmnd_ctx* ctx, dmnd_block* b, int sid, uint32_t q_begin, uint32_t q_end) {
	if (b->soft) motif_seed_mask(&ctx->p, b, sid, q_begin, q_end);
	return 0;
}

int dmnd_search_shape(dmnd_ctx* ctx, dmnd_block* query, const dmnd_block* ref, int sid, dmnd_hits** out,
                      dmnd_stage_counters* counters) {
	return dmnd_search_shape_range(ctx, query, ref, sid, 0, query->nseq, out, counters);
}
int dmnd_search_shape_range(dmnd_ctx* ctx, dmnd_block* query, const dmnd_block* ref, int sid, uint32_t q_begin, uint32_t q_end,
                            dmnd_hits** out, dmnd_stage_counters* counters) {
	const dmnd_params* p = &ctx->p;
	if (q_begin > q_end || q_end > query->nseq) return fail("dmnd_search_shape_range: bad query range");
	dmnd_stage_counters cn; memset(&cn, 0, sizeof cn);
	size_t nh = 0, hcap = 1024;
	dmnd_hit* hits = (dmnd_hit*)malloc(hcap * sizeof *hits);
	const uint32_t parts_total = (uint32_t)1 << p->seedp_bits;
	const uint32_t nchunks = (uint32_t)p->index_chunks < parts_total ? (uint32_t)p->index_chunks : parts_total;
	const uint32_t psize = parts_total / nchunks, prem = parts_total % nchunks;
	if (query->soft) motif_seed_mask(p, query, sid, q_begin, q_end);
	for (uint32_t chunk = 0; chunk < nchunks; ++chunk) {
		const uint32_t bsel = chunk < prem ? chunk : prem;
		const uint32_t pb = bsel * (psize + 1) + (chunk - bsel) * psize, pe = pb + (chunk < prem ? psize + 1 : psize);
		entry *re, *qe;
		const size_t nr = enum_seeds(p, sid, ref, pb, pe, 0, ref->nseq, &re), nq = enum_seeds(p, sid, query, pb, pe, q_begin, q_end, &qe);
		/* pass 1: entropy masking of every shared key of this chunk (search/stage0.cpp:173 runs before the search) */
		size_t i = 0, j = 0;
		uint8_t* erased = (uint8_t*)calloc(nq + 1, 1); /* marks first entry of an erased query run */
		while (i < nq && j < nr) {
			if (qe[i].seed < re[j].seed) { ++i; continue; }
			if (qe[i].seed > re[j].seed) { ++j; continue; }
			size_t i2 = i, j2 = j;
			while (i2 < nq && qe[i2].seed == qe[i].seed) ++i2;
			while (j2 < nr && re[j2].seed == re[j].seed) ++j2;
			if (!seed_is_complex(p, sid, query->letters + qe[i].loc)) {
				for (size_t k = i; k < i2; ++k) query->letters[qe[k].loc] |= (int8_t)DMND_SEED_MASK;
				erased[i] = 1;
				++cn.masked_seeds;
			}
			i = i2; j = j2;
		}
		/* pass 2: stage 1 + stage 2 per shared key */
		lm_ctx x = { ctx, sid, p->index_chunks > 1, pb, pe };
		i = 0; j = 0;
		while (i < nq && j < nr) {
			if (qe[i].seed < re[j].seed) { ++i; continue; }
			if (qe[i].seed > re[j].seed) { ++j; continue; }
			size_t i2 = i, j2 = j;
			while (i2 < nq && qe[i2].seed == qe[i].seed) ++i2;
			while (j2 < nr && re[j2].seed == re[j].seed) ++j2;
			if (!erased[i]) {
				++cn.seeds_hit;
				cn.seed_hits += (uint64_t)(i2 - i) * (uint64_t)(j2 - j);
				for (size_t a = i; a < i2; ++a) {
					const int8_t* qp = query->letters + qe[a].loc;
					const uint32_t qid = seq_of(query, qe[a].loc);
					const int seed_offset = (int)((int64_t)qe[a].loc - query->limits[qid]);
					/* search/stage2.h:92-103; ungapped_window(query_len) :58-63: a translated frame of <= 85 letters uses its whole length */
					const int query_len = (int)(query->limits[qid + 1] - query->limits[qid] - 1);
					const int short_frame = p->query_contexts > 1 && query_len <= 85;
					const int window = short_frame ? query_len : p->ungapped_window;
					const int8_t *cb, *ce;
					clip(qp - window, window * 2, window, &cb, &ce);
					const int window_left = (int)(qp - cb), window_clipped = (int)(ce - cb);
					const int interval_mod = p->left_most_interval > 0 ? seed_offset % p->left_most_interval : window_left;
					const int overhang = window_left - interval_mod > 0 ? window_left - interval_mod : 0;
					/* search/stage2.h:41-57 ungapped_cutoff */
					int score_cutoff = 0;
					if (p->ungapped_evalue != 0.0) {
						if (query_len <= p->short_query_max_len) score_cutoff = p->short_query_ungapped_cutoff;
						else if (short_frame) score_cutoff = p->ungapped_cutoff_short[32 - __builtin_clz((uint32_t)query_len)];
						else score_cutoff = p->ungapped_cutoff[32 - __builtin_clz((uint32_t)query_len)];
					}
					/* search/hamming/kernel.h:61-74: the key's subject locations are visited in tiles of config.tile_size = 1024;
					 * per query location the stage-1 survivors of a tile (ascending, hit_field.h:44-57) go through
					 * window_ungapped_best in batches of 32 (search/stage2.h:114-120, AVX2 int8 channels) */
					for (size_t tile = j; tile < j2; tile += 1024) {
						const size_t tile_end = tile + 1024 < j2 ? tile + 1024 : j2;
						size_t surv[1024], ns = 0;
						for (size_t bb = tile; bb < tile_end; ++bb)
							if (fingerprint_match(qp, ref->letters + re[bb].loc) >= (unsigned)p->hamming_id) surv[ns++] = bb;
						cn.tentative_matches1 += ns;
						for (size_t b0 = 0; b0 < ns; b0 += 32) {
							const size_t nb = ns - b0 < 32 ? ns - b0 : 32;
							for (size_t k = 0; k < nb; ++k) {
								const size_t bb = surv[b0 + k];
								const int8_t* sp = ref->letters + re[bb].loc;
								int score = 0x7fffffff; /* INT_MAX when the ungapped stage is skipped: (uint16_t) -> 0xFFFF */
								if (score_cutoff) {
									/* dp/ungapped_align.cpp:244-257 ungapped_window over the clipped query window; batches of >= 4
									 * subjects take the int8 kernel instead (dp/ungapped_simd.cpp:32-88), whose biased saturating
									 * lanes cap the running score at 255 (score_vector_int8.h) -- same floor at 0, same maximum below it */
									int st = 0, best = 0;
									const int8_t* sw = sp - window_left;
									for (int t = 0; t < window_clipped; ++t) {
										st += (int)p->score[(cb[t] & DMND_LETTER_MASK) * 32 + (sw[t] & DMND_LETTER_MASK)];
										if (st < 0) st = 0;
										if (st > best) best = st;
									}
									score = (nb >= 4 && best > 255) ? 255 : best;
								}
								if (!(score > score_cutoff)) continue;
								++cn.tentative_matches2;
								if (left_most_filter(&x, cb + overhang, window_clipped - overhang, sp - window_left + overhang,
								                     window_left - overhang, p->shape_len[sid])) {
									++cn.tentative_matches3;
									if (nh == hcap) { hcap *= 2; hits = (dmnd_hit*)realloc(hits, hcap * sizeof *hits); }
									hits[nh].query = qid;
									hits[nh].seed_offset = seed_offset;
									hits[nh].subject_score = re[bb].loc | ((uint64_t)(uint16_t)score << 48);
									++nh;
								}
							}
						}
					}
				}
			}
			i = i2; j = j2;
		}
		free(erased); free(re); free(qe);
	}
	/* group by query (stable), as the ABI promises */
	dmnd_hits* h = (dmnd_hits*)calloc(1, sizeof *h);
	h->n = nh;
	h->h = (dmnd_hit*)malloc((nh ? nh : 1) * sizeof(dmnd_hit));
	{
		size_t* cnt = (size_t*)calloc((size_t)query->nseq + 1, sizeof(size_t));
		for (size_t k = 0; k < nh; ++k) ++cnt[hits[k].query + 1];
		for (uint32_t k = 0; k < query->nseq; ++k) cnt[k + 1] += cnt[k];
		for (size_t k = 0; k < nh; ++k) h->h[cnt[hits[k].query]++] = hits[k];
		free(cnt);
	}
	free(hits);
	*out = h;
	if (counters) *counters = cn;
	return 0;
}
size_t dmnd_hits_count(const dmnd_hits* h) { return h->n; }
int dmnd_hits_download(dmnd_ctx* ctx, const dmnd_hits* h, dmnd_hit* host, size_t cap) {
	(void)ctx;
	if (cap < h->n) return fail("dmnd_hits_download: buffer too small");
	memcpy(host, h->h, h->n * sizeof(dmnd_hit));
	return 0;
}
/* dp/ungapped_align.cpp:150-214 (ScoreOnly) */
int dmnd_hits_xdrop_sites(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, const dmnd_hits* h, int raw_xdrop,
                          dmnd_segment* host, dmnd_hit_site* sites, size_t cap) {
	const dmnd_params* p = &ctx->p;
	if (cap < h->n) return fail("dmnd_hits_xdrop: buffer too small");
	for (size_t k = 0; k < h->n; ++k) {
		const dmnd_hit* hit = &h->h[k];
		const uint64_t sloc = DMND_HIT_SUBJECT(*hit);
		const uint32_t t = seq_of(ref, sloc);
		const int8_t *qs = query->letters + query->limits[hit->query], *cb = query->bias + query->limits[hit->query], *ss = ref->letters + ref->limits[t];
		const int qa = hit->seed_offset, sa = (int)((int64_t)sloc - ref->limits[t]);
		int score = 0, st = 0, n = 1, delta = 0, len = 0, ql, sl;
		int q = qa - 1, s = sa - 1;
		while (score - st < raw_xdrop && (ql = qs[q] & 31) != DMND_DELIMITER && (sl = ss[s] & 31) != DMND_DELIMITER) {
			st += p->score[ql * 32 + sl] + cb[q];
			if (st > score) { score = st; delta = n; }
			--q; --s; ++n;
		}
		q = qa; s = sa; st = score; n = 1;
		while (score - st < raw_xdrop && (ql = qs[q] & 31) != DMND_DELIMITER && (sl = ss[s] & 31) != DMND_DELIMITER) {
			st += p->score[ql * 32 + sl] + cb[q];
			if (st > score) { score = st; len = n; }
			++q; ++s; ++n;
		}
		host[k].i = qa - delta; host[k].j = sa - delta; host[k].len = len + delta; host[k].score = score;
		if (sites) { sites[k].target = t; sites[k].j = sa; }
	}
	return 0;
}
/* ---------------------------------------------------------------------------------------------------------- */
/* Gapped filter.  DP::make_profile8 (dp/score_profile.cpp:32-65, AVX2 branch): profile(l, i) = sat8(matrix8[l][query[i]] +
 * bias[i]) for true amino acids l (no bias for l >= 20), -1 in the 128 positions of padding on either side.
 * DP::scan_diags64/128 (dp/scan_diags.cpp:30-275): per diagonal d_begin + k the running score, floored at 0 and saturating
 * at 255 (biased int8 lanes), over the target columns [j0, j1); the maximum per diagonal.  DP::diag_alignment (:277-297). */
static int gf_profile(const dmnd_params* p, const int8_t* q, const int8_t* cbs, int qlen, int l, int i) {
	if (i < 0 || i >= qlen) return -1;
	int v = p->score[l * 32 + (q[i] & DMND_LETTER_MASK)];
	if (l < 20) { v += cbs[i]; if (v > 127) v = 127; if (v < -128) v = -128; }
	return v;
}
static void gf_scan(const dmnd_params* p, const int8_t* q, const int8_t* cbs, int qlen, const int8_t* t, int band, int d_begin, int j_begin, int j_end, int* out) {
	int v[128];
	for (int k = 0; k < band; ++k) { v[k] = 0; out[k] = 0; }
	const int j0 = j_begin > -(d_begin + band - 1) ? j_begin : -(d_begin + band - 1), j1 = (qlen - d_begin) < j_end ? (qlen - d_begin) : j_end;
	for (int j = j0, i = d_begin + j0; j < j1; ++j, ++i) {
		const int l = t[j] & DMND_LETTER_MASK;
		for (int k = 0; k < band; ++k) {
			int x = v[k] + gf_profile(p, q, cbs, qlen, l, i + k);
			if (x < 0) x = 0;
			if (x > 255) x = 255;
			v[k] = x;
			if (x > out[k]) out[k] = x;
		}
	}
}
static int gf_diag_alignment(const dmnd_params* p, const int* s, int count) {
	int best = 0, best_gap = -p->gap_open, d = -1;
	for (int i = 0; i < count; ++i) {
		if (s[i] < p->gapped_filter_diag_score) continue;
		const int gap_score = -p->gap_extend * (i - d) + best_gap;
		int n = s[i];
		if (gap_score + s[i] > best) best = n = gap_score + s[i];
		if (s[i] > best) best = n = s[i];
		const int open_score = -p->gap_open + n;
		if (open_score > gap_score) { best_gap = open_score; d = i; }
	}
	return best;
}
static int gf_one(const dmnd_params* p, const int8_t* q, const int8_t* cbs, int qlen, const int8_t* t, int slen, int hi, int hj, int band, int window) {
	const int diag = hi - hj;
	const int d = diag - band / 2 > -(slen - 1) ? diag - band / 2 : -(slen - 1);
	const int j0 = hj - window > 0 ? hj - window : 0, j1 = hj + window < slen ? hj + window : slen;
	int scores[128];
	gf_scan(p, q, cbs, qlen, t, band, d, j0, j1, scores);
	return gf_diag_alignment(p, scores, band);
}
static int bit_len(int x) { return 32 - __builtin_clz((uint32_t)x); }
int dmnd_hits_gapped_filter(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, const dmnd_hits* h, uint8_t* pass, size_t cap) {
	const dmnd_params* p = &ctx->p;
	if (cap < h->n) return fail("dmnd_hits_gapped_filter: buffer too small");
	for (size_t k = 0; k < h->n; ++k) {
		const dmnd_hit* hit = &h->h[k];
		const uint64_t sloc = DMND_HIT_SUBJECT(*hit);
		const uint32_t t = seq_of(ref, sloc);
		const int8_t *qs = query->letters + query->limits[hit->query], *cb = query->bias + query->limits[hit->query], *ss = ref->letters + ref->limits[t];
		const int qlen = (int)(query->limits[hit->query + 1] - query->limits[hit->query] - 1), slen = (int)(ref->limits[t + 1] - ref->limits[t] - 1);
		const int hi = hit->seed_offset, hj = (int)((int64_t)sloc - ref->limits[t]);
		pass[k] = 0;
		/* align/gapped_filter.cpp:44-63; `qlen` there is query_profile->length(), the length of the query's FIRST context, whatever
		 * frame the hit lies in; translated queries shorter than MIN_STAGE2_QLEN = 100 pass after the first scan */
		const int translated = p->query_contexts > 1;
		const uint32_t q0 = translated ? hit->query / (uint32_t)p->query_contexts * (uint32_t)p->query_contexts : hit->query;
		const int qlen0 = (int)(query->limits[q0 + 1] - query->limits[q0] - 1);
		const int f1 = gf_one(p, qs, cb, qlen, ss, slen, hi, hj, 64, 100);
		if (qlen0 > 0 && f1 > p->gapped_cutoff1[bit_len(qlen0)][bit_len(slen)]) {
			if (translated && qlen0 < 100) { pass[k] = 1; continue; }
			const int f2 = gf_one(p, qs, cb, qlen, ss, slen, hi, hj, 128, p->gapped_filter_window);
			if (f2 > p->gapped_cutoff2[bit_len(qlen0)][bit_len(slen)]) pass[k] = 1;
		}
	}
	return 0;
}
int dmnd_hits_xdrop(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, const dmnd_hits* h, int raw_xdrop,
                    dmnd_segment* host, size_t cap) {
	return dmnd_hits_xdrop_sites(ctx, query, ref, h, raw_xdrop, host, NULL, cap);
}
void dmnd_hits_free(dmnd_ctx* ctx, dmnd_hits* h) { (void)ctx; if (h) { free(h->h); free(h); } }

/* ---------------------------------------------------------------------------------------------------------- */
/* Banded SWIPE                                                                                                */
static inline int imax(int a, int b) { return a > b ? a : b; }
static inline int imin(int a, int b) { return a < b ? a : b; }

/* Stats-only passes (round 2 when band*cols > max_swipe_dp and no transcript is requested: swipe_wrapper.cpp:89-96 puts
 * such targets into bins 3..5, dispatch_swipe :177-199 runs ForwardCell in round 0 and BackwardCell in the reversed
 * round 1).  A cell is {v, a, b}: ForwardCell a = ident, b = len; BackwardCell a = mismatch, b = gapopen
 * (stat_cell.h:46-160).  Ties copy the statistics of the max() argument (set_max, stat_cell.h:258-272), in the order
 * hgap, vgap for the current cell and `open` for the gaps (cell_update.h:113-136). */
typedef struct { int v, a, b; } scell;
static inline void scell_max(scell* x, const scell* y) { /* set_max: v = max; if (v == y.v) take y's statistics */
	if (y->v > x->v) x->v = y->v;
	if (x->v == y->v) { x->a = y->a; x->b = y->b; }
}
typedef struct { int best, max_col, max_band_row, a, b; } stats_out;
static void stats_pass(const dmnd_params* p, const int8_t* q, const int8_t* cbs, int qlen, const int8_t* t, int tlen, int d_begin, int d_end,
                       int backward, stats_out* o) {
	const int band = d_end - d_begin;
	const int i1 = imax(d_end - 1, 0), i0 = i1 + 1 - band, j0 = i1 - (d_end - 1);
	const int cols = imin(qlen - 1 - d_begin, tlen - 1) + 1 - j0;
	memset(o, 0, sizeof *o);
	if (band <= 0 || cols <= 0) return;
	const int go = p->gap_open + p->gap_extend, ge = p->gap_extend;
	scell* score = (scell*)calloc((size_t)band, sizeof(scell));
	scell* hgap = (scell*)calloc((size_t)band + 1, sizeof(scell));
	for (int c = 0; c < cols; ++c) {
		const int j = j0 + c;
		const int r_begin = imax(i0 + c, 0) - (i0 + c), r_end = imin(i1 + c, qlen - 1) + 1 - (i0 + c);
		if (r_begin >= r_end) break;
		const int tl = t[j] & DMND_LETTER_MASK;
		scell vgap = { 0, 0, 0 };
		int col_best = 0, i_max = 0;
		for (int r = r_begin; r < r_end; ++r) {
			const int i = i0 + c + r;
			scell hg = hgap[r + 1];
			const int ql = q[i] & DMND_LETTER_MASK;
			scell cur = score[r];
			cur.v += p->score[ql * 32 + tl] + cbs[i];
			const int id = ql == tl; /* VectorIdMask, stat_cell.h:38-44 */
			if (!backward) { cur.a += id; cur.b += 1; hg.b += 1; vgap.b += 1; } /* update_stats, :225-232 */
			else cur.a += 1 - id;                                                /* :234-237 */
			scell_max(&cur, &hg); scell_max(&cur, &vgap);
			if (cur.v < 0) cur.v = 0;
			col_best = imax(col_best, cur.v);
			if (col_best == cur.v) i_max = r;
			vgap.v = imax(vgap.v - ge, 0); hg.v = imax(hg.v - ge, 0);
			scell open = cur;
			open.v = imax(cur.v - go, 0);
			if (backward) open.b += 1;                /* update_open, :250-257 */
			if (cur.v == 0) { cur.a = 0; cur.b = 0; } /* :243-257 */
			scell_max(&hg, &open); scell_max(&vgap, &open);
			hgap[r] = hg;
			score[r] = cur;
		}
		if (col_best > o->best) { /* banded_swipe.h:321-326 */
			o->best = col_best; o->max_col = c; o->max_band_row = i_max;
			o->a = score[i_max].a; o->b = score[i_max].b;
		}
	}
	free(score); free(hgap);
}

/* One problem; values use the reference's int8/int16 lane semantics: every score, hgap and vgap is floored at 0
 * (saturating arithmetic around DELTA, dp/score_vector_int8.h:263-346,421-436).  trace nibble per cell:
 * bit0 cur==vgap, bit1 cur==hgap (cell_update.h:76-79), bit2 vgap'==open, bit3 hgap'==open (:85-88). */
static int swipe_one(const dmnd_ctx* ctx, const int8_t* q, const int8_t* cbs, int qlen, const int8_t* t, int tlen, int d_begin,
                     int d_end, int mode, dmnd_dp_result* res, uint8_t* tr, size_t tr_cap, size_t* tr_used) {
	const dmnd_params* p = &ctx->p;
	const int band = d_end - d_begin;
	const int i1 = imax(d_end - 1, 0), i0 = i1 + 1 - band, j0 = i1 - (d_end - 1);
	const int cols = imin(qlen - 1 - d_begin, tlen - 1) + 1 - j0; /* dp/dp.h:47-52 */
	memset(res, 0, sizeof *res);
	if (band <= 0 || cols <= 0) return 0;
	if (mode == DMND_DP_TRACEBACK && tr == NULL && (int64_t)band * (int64_t)cols > DMND_MAX_SWIPE_DP) {
		/* forward statistics, then the reversed pass over (reversed query) x (reversed target prefix [0, t_end)) in the
		 * mirrored band: recompute_reversed, swipe_wrapper.cpp:364-444; result assembly banded_swipe.h:86-122 */
		stats_out f, b;
		stats_pass(p, q, cbs, qlen, t, tlen, d_begin, d_end, 0, &f);
		if (f.best <= 0) return 0;
		const int q_end = i0 + f.max_col + f.max_band_row + 1, t_end = j0 + f.max_col + 1;
		int8_t* rq = (int8_t*)malloc((size_t)qlen), *rc = (int8_t*)malloc((size_t)qlen), *rt = (int8_t*)malloc((size_t)t_end);
		for (int i = 0; i < qlen; ++i) { rq[i] = q[qlen - 1 - i]; rc[i] = cbs[qlen - 1 - i]; }
		for (int j = 0; j < t_end; ++j) rt[j] = t[t_end - 1 - j];
		const int rd0 = -(d_end - 1) + qlen - t_end, rd1 = -d_begin + qlen - t_end + 1; /* Geo::rev_diag */
		stats_pass(p, rq, rc, qlen, rt, t_end, rd0, rd1, 1, &b);
		free(rq); free(rc); free(rt);
		if (b.best <= 0) return 0;
		const int ri1 = imax(rd1 - 1, 0), ri0 = ri1 + 1 - band, rj0 = ri1 - (rd1 - 1);
		res->score = b.best;
		res->q_end = q_end; res->t_end = t_end;
		res->q_begin = qlen - (ri0 + b.max_col + b.max_band_row + 1);
		res->t_begin = t_end - (rj0 + b.max_col + 1);
		res->identities = f.a; res->length = f.b;
		res->mismatches = b.a; res->gap_openings = b.b;
		res->gaps = res->length - res->identities - res->mismatches; /* assign_stats, stat_cell.h:215-219 */
		return 0;
	}
	const int go = p->gap_open + p->gap_extend, ge = p->gap_extend;
	int* score = (int*)calloc((size_t)band, sizeof(int));
	int* hgap = (int*)calloc((size_t)band + 1, sizeof(int));
	uint8_t* trace = mode == DMND_DP_TRACEBACK ? (uint8_t*)calloc((size_t)band * (size_t)cols, 1) : NULL;
	int best = 0, max_col = 0, max_band_row = 0;
	for (int c = 0; c < cols; ++c) {
		const int j = j0 + c;
		const int r_begin = imax(i0 + c, 0) - (i0 + c), r_end = imin(i1 + c, qlen - 1) + 1 - (i0 + c);
		if (r_begin >= r_end) break;
		const int tl = t[j] & DMND_LETTER_MASK;
		int vgap = 0, col_best = 0, i_max = 0;
		for (int r = r_begin; r < r_end; ++r) {
			const int i = i0 + c + r;
			int hg = hgap[r + 1];
			const int m = p->score[(q[i] & DMND_LETTER_MASK) * 32 + tl] + cbs[i];
			int cur = score[r] + m;
			cur = imax(cur, hg); cur = imax(cur, vgap); cur = imax(cur, 0);
			uint8_t nib = (uint8_t)((cur == vgap ? 1 : 0) | (cur == hg ? 2 : 0));
			col_best = imax(col_best, cur);
			if (col_best == cur) i_max = r; /* VectorRowCounter::inc, cell_update.h:43-46 */
			vgap = imax(vgap - ge, 0); hg = imax(hg - ge, 0);
			const int open = imax(cur - go, 0);
			hg = imax(hg, open); vgap = imax(vgap, open);
			nib |= (uint8_t)((vgap == open ? 4 : 0) | (hg == open ? 8 : 0));
			if (trace) trace[(size_t)c * band + r] = nib;
			hgap[r] = hg;
			score[r] = cur;
		}
		if (col_best > best) { best = col_best; max_col = c; max_band_row = i_max; } /* banded_swipe.h:321-326 */
	}
	res->score = best;
	if (mode == DMND_DP_TRACEBACK && best > 0) {
		/* banded_swipe.h:127-187 + banded_matrix.h:357-402 */
		int c = max_col, r = max_band_row;
		int i = i0 + max_col + max_band_row, j = j0 + max_col;
		res->q_end = i + 1; res->t_end = j + 1;
		int sc = 0;
		size_t n = 0, base = *tr_used;
		int overflow = 0;
#define PUSH(op, letter) do { if (tr) { if (base + n < tr_cap) tr[base + n] = (uint8_t)(((op) << 6) | ((letter) & 63)); else overflow = 1; } ++n; } while (0)
		while (i >= 0 && j >= 0 && sc < best) {
			const uint8_t nib = trace[(size_t)c * band + r];
			if ((nib & 3) == 0) {
				const int ql = q[i] & DMND_LETTER_MASK, sl = t[j] & DMND_LETTER_MASK;
				const int m = p->score[ql * 32 + sl];
				sc += m + cbs[i];
				if (ql == sl) { PUSH(DMND_OP_MATCH, 0); ++res->identities; ++res->positives; }
				else { PUSH(DMND_OP_SUBSTITUTION, sl); ++res->mismatches; if (m > 0) ++res->positives; }
				++res->length;
				--i; --j; --c; /* walk_diagonal: same band row, previous column */
			} else if (nib & 1) {
				int l = 0;
				do { ++l; --i; --r; } while ((trace[(size_t)c * band + r] & 4) == 0 && i > 0);
				++res->gap_openings; res->length += l; res->gaps += l;
				for (int k = 0; k < l; ++k) PUSH(DMND_OP_INSERTION, 0);
				sc -= p->gap_open + l * p->gap_extend;
			} else {
				int l = 0;
				do { ++l; --j; --c; ++r; } while ((trace[(size_t)c * band + r] & 8) == 0 && j > 0);
				++res->gap_openings; res->length += l; res->gaps += l;
				for (int k = 0; k < l; ++k) PUSH(DMND_OP_DELETION, t[j + l - k] & DMND_LETTER_MASK); /* hssp.cpp:283: subject[-i] from it.j + len */
				sc -= p->gap_open + l * p->gap_extend;
			}
		}
#undef PUSH
		if (sc != best) { free(score); free(hgap); free(trace); return fail("oracle: Traceback error."); }
		res->q_begin = i + 1; res->t_begin = j + 1;
		if (tr) {
			if (overflow) res->status = 1;
			else {
				for (size_t a = 0, b = n; a + 1 < b; ++a, --b) { uint8_t x = tr[base + a]; tr[base + a] = tr[base + b - 1]; tr[base + b - 1] = x; }
				res->transcript_off = (uint32_t)base; res->transcript_len = (uint32_t)n;
				*tr_used = base + n;
			}
		}
	}
	free(score); free(hgap); free(trace);
	return 0;
}

int dmnd_banded_swipe(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, const dmnd_dp_problem* problems,
                      size_t n, int mode, dmnd_dp_result* results, uint8_t* transcripts, size_t transcript_cap) {
	size_t used = 0;
	for (size_t k = 0; k < n; ++k) {
		const dmnd_dp_problem* pr = &problems[k];
		if (pr->query >= query->nseq || pr->target >= ref->nseq) return fail("dmnd_banded_swipe: sequence index out of range");
		const int64_t qo = query->limits[pr->query], to = ref->limits[pr->target];
		const int qlen = (int)(query->limits[pr->query + 1] - qo - 1), tlen = (int)(ref->limits[pr->target + 1] - to - 1);
		if (swipe_one(ctx, query->letters + qo, query->bias + qo, qlen, ref->letters + to, tlen, pr->d_begin, pr->d_end, mode,
		              &results[k], transcripts, transcript_cap, &used))
			return 1;
	}
	return 0;
}

/* ---- frameshift alignment: banded_3frame_swipe<int32_t, ...> for ONE target (dp/swipe/banded_3frame_swipe.cpp:392-520) ----------
 * Buffers as the reference keeps them: Banded3FrameSwipeTracebackMatrix (:118-296) = one column of 3*band + 1 scores per target
 * letter (+ a zero column in front), band index p = 3 * (i - i0(column)) + frame, the last entry of a column stays 0; hgap_ of
 * 3*band + 3 entries, read at p + 3 and written at p.  The score-only matrix (:43-115) overwrites one column in place and yields
 * the same cell values (every value is read before its slot is rewritten), so both modes run this one function.  Cell update:
 * dp/swipe/swipe.h:57-83 on int32_t (saturate = max with 0).  Entries the reference never writes (rows before the query start
 * other than the three that set_zero clears, rows past the query end) are uninitialised memory there; they are 0 here. */
static int fs_swipe_one(const dmnd_ctx* ctx, const int8_t* const q[3], const int ql[3], int dna_len, const int8_t* t, int tlen,
                        int d_begin, int d_end, int F, int mode, dmnd_fs_result* res, uint8_t* tr, size_t tr_cap, size_t* tr_used) {
	const dmnd_params* p = &ctx->p;
	memset(res, 0, sizeof *res);
	const int band = d_end - d_begin, B3 = band * 3, W = B3 + 1;
	const int i1s = imax(d_end - 1, 0), i0s = i1s + 1 - band, pos0 = i1s - (d_end - 1); /* :410-421, TargetIterator (target_iterator.h:68-92) */
	const int qlen = ql[0];
	if (band <= 0 || qlen <= 0 || tlen - pos0 <= 0) return 0;
	const int ncol = tlen - pos0;
	int* S = (int*)calloc((size_t)W * ((size_t)ncol + 1), sizeof(int));
	int* hgap = (int*)calloc((size_t)B3 + 3, sizeof(int));
	if (!S || !hgap) { free(S); free(hgap); return fail("oracle: out of memory (3-frame swipe)"); }
	const int go = p->gap_open + p->gap_extend, ge = p->gap_extend;
	int best = 0, max_col = 0;
	for (int j = 0, i0 = i0s, i1 = i1s; j < ncol; ++j, ++i0, ++i1) {
		const int i0_ = imax(i0, 0), i1_ = imin(i1, qlen - 1);
		if (i0_ > i1_) break;
		const int* old = S + (size_t)j * W;
		int* cur = S + (size_t)(j + 1) * W;
		int pidx = (i0_ - i0) * 3;
		if (pidx > 0) cur[pidx - 1] = cur[pidx - 2] = cur[pidx - 3] = 0; /* ColumnIterator::set_zero */
		const int tl = t[pos0 + j] & DMND_LETTER_MASK;
		int vg[3] = { 0, 0, 0 }, col_best = 0;
		int sm4 = 0, sm3 = old[pidx], sm2 = old[pidx + 1];
		int stop = 0;
		for (int i = i0_; i <= i1_ && !stop; ++i)
			for (int f = 0; f < 3; ++f) {
				if (f > 0 && i >= ql[f]) { stop = 1; break; } /* :469,477: `break` leaves the row loop */
				int hg = hgap[pidx + 3];
				const int sc = p->score[(q[f][i] & DMND_LETTER_MASK) * 32 + tl];
				int c = sm3 + sc;
				const int fs = sc - F;
				c = imax(c, sm4 + fs); c = imax(c, sm2 + fs);
				c = imax(imax(c, vg[f]), hg);
				c = imax(c, 0);
				col_best = imax(col_best, c);
				vg[f] -= ge; hg -= ge;
				const int open = c - go;
				vg[f] = imax(vg[f], open); hg = imax(hg, open);
				hgap[pidx] = hg; cur[pidx] = c;
				++pidx;
				sm4 = sm3; sm3 = sm2; sm2 = old[pidx + 1 <= B3 ? pidx + 1 : B3];
			}
		if (col_best > best) { best = col_best; max_col = j; }
	}
	res->score = best;
	if (best > 0) res->t_end = pos0 + max_col + 1; /* score only: the first column that reaches the score (the reference's max_col, :495-498) */
	if (mode != DMND_DP_TRACEBACK || best <= 0) { free(S); free(hgap); return 0; }
	/* traceback(): :338-390, dp.traceback :257-267 */
	const long total = (long)W * ((long)ncol + 1);
#define SV(x) (((x) >= 0 && (x) < total) ? S[(x)] : 0)
	const int col = max_col + 1, i0c = i0s + max_col;
	long idx = -1;
	for (int x = imax(-i0c, 0) * 3, xe = imin(B3, dna_len - 2 - i0c * 3); x < xe; ++x)
		if (S[(size_t)col * W + x] == best) { idx = (long)col * W + x; break; }
	if (idx < 0) { free(S); free(hgap); res->status = 2; return 0; }
	int fr = (int)((idx - (long)col * W) % 3), i = i0c + (int)((idx - (long)col * W) / 3), j = pos0 + max_col;
	res->q_end = i + 1; res->t_end = j + 1; res->frame_end = fr;
	size_t n = 0, base = *tr_used;
	int overflow = 0, err = 0;
#define PUSHB(b) do { if (tr) { if (base + n < tr_cap) tr[base + n] = (uint8_t)(b); else overflow = 1; } ++n; } while (0)
#define PUSH_MATCH() do { if (qa == sa) { PUSHB(DMND_OP_MATCH << 6); ++res->identities; ++res->positives; } \
		else { PUSHB((DMND_OP_SUBSTITUTION << 6) | sa); ++res->mismatches; if (m > 0) ++res->positives; } ++res->length; } while (0)
	while (SV(idx) > 0 && !err) {
		if (i < 0 || j < 0 || i >= ql[fr]) { err = 1; break; }
		const int qa = q[fr][i] & DMND_LETTER_MASK, sa = t[j] & DMND_LETTER_MASK;
		const int m = p->score[qa * 32 + sa], sc = SV(idx);
		if (sc == SV(idx - W) + m) { PUSH_MATCH(); idx -= W; --i; --j; }
		else if (sc == SV(idx - (W + 1)) + m - F) { /* walk_forward_shift :180-191 */
			PUSH_MATCH(); PUSHB(DMND_TR_FRAMESHIFT_FWD);
			idx -= W + 1; --i; --j; --fr;
			if (fr == -1) { fr = 2; --i; }
		}
		else if (sc == SV(idx - (W - 1)) + m - F) { /* walk_reverse_shift :192-203 */
			PUSH_MATCH(); PUSHB(DMND_TR_FRAMESHIFT_REV);
			idx -= W - 1; --i; --j; ++fr;
			if (fr == 3) { fr = 0; ++i; }
		}
		else { /* walk_gap(d_begin, d_end) :204-244 */
			const int i0g = imax(d_begin + j, 0), j0g = imax(i - d_end, -1);
			const long hstep = B3 - 2;
			long h = idx - hstep, h0 = idx - (long)(j - j0g) * hstep, v = idx - 3, v0 = idx - (long)(i - i0g + 1) * 3;
			int g = go, l = 1, found = 0;
			while (v > v0 && h > h0) {
				if (sc + g == SV(h)) { found = 2; break; }
				else if (sc + g == SV(v)) { found = 1; break; }
				h -= hstep; v -= 3; ++l; g += ge;
			}
			if (!found) while (v > v0) { if (sc + g == SV(v)) { found = 1; break; } v -= 3; ++l; g += ge; }
			if (!found) while (h > h0) { if (sc + g == SV(h)) { found = 2; break; } h -= hstep; ++l; g += ge; }
			if (!found) { err = 1; break; }
			++res->gap_openings; res->length += l; res->gaps += l; /* Hsp::push_gap */
			if (found == 1) { idx = v; i -= l; for (int k = 0; k < l; ++k) PUSHB(DMND_OP_INSERTION << 6); }
			else { idx = h; j -= l; for (int k = 0; k < l; ++k) PUSHB((DMND_OP_DELETION << 6) | (t[j + l - k] & DMND_LETTER_MASK)); }
		}
	}
#undef PUSH_MATCH
#undef PUSHB
#undef SV
	free(S); free(hgap);
	if (err) { res->status = 2; return 0; }
	res->q_begin = i + 1; res->t_begin = j + 1; res->frame_begin = fr;
	if (tr) {
		if (overflow) res->status = 1;
		else {
			for (size_t a = 0, b = n; a + 1 < b; ++a, --b) { uint8_t x = tr[base + a]; tr[base + a] = tr[base + b - 1]; tr[base + b - 1] = x; }
			res->transcript_off = (uint32_t)base; res->transcript_len = (uint32_t)n;
			*tr_used = base + n;
		}
	}
	return 0;
}

int dmnd_banded_3frame_swipe(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, const dmnd_dp_problem* problems, size_t n,
                             int frame_shift, int mode, dmnd_fs_result* results, uint8_t* transcripts, size_t transcript_cap) {
	size_t used = 0;
	for (size_t k = 0; k < n; ++k) {
		const dmnd_dp_problem* pr = &problems[k];
		if ((uint64_t)pr->query + 3 > query->nseq || pr->target >= ref->nseq) return fail("dmnd_banded_3frame_swipe: sequence index out of range");
		const int8_t* q[3]; int ql[3];
		for (int f = 0; f < 3; ++f) {
			const int64_t o = query->limits[pr->query + f];
			q[f] = query->letters + o; ql[f] = (int)(query->limits[pr->query + f + 1] - o - 1);
		}
		const int dna_len = ql[0] + ql[1] + ql[2] + 2; /* frame f holds (dna_len - f) / 3 codons (basic/translated_position.h:47-50) */
		const int64_t to = ref->limits[pr->target];
		const int tlen = (int)(ref->limits[pr->target + 1] - to - 1);
		if (fs_swipe_one(ctx, q, ql, dna_len, ref->letters + to, tlen, pr->d_begin, pr->d_end, frame_shift, mode, &results[k], transcripts,
		                 transcript_cap, &used))
			return 1;
	}
	return 0;
}
