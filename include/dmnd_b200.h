/* dmnd_b200.h -- C ABI of the B200-native DIAMOND seed-and-extend hot path.
 *
 * Two layers, both plain C (pointers + sizes, no C++/torch types, no exceptions across the boundary):
 *
 *  K layer ("kernel ABI")   batch-oriented replacements for the reference's three SIMD dispatch seams
 *                           (util/simd/dispatch.h:46-116):
 *                             Search::search_shape          search/search.h:80,   search/stage0.cpp:101-228
 *                             DP::BandedSwipe::swipe        dp/dp.h:287,          dp/swipe/swipe_wrapper.cpp:446-470
 *                           plus block residency (data/string_set.h:26-275 layout, re-used byte for byte).
 *                           Implemented by hand-written sm_100a CUDA in libdmnd_b200.so.  The CPU restatement under
 *                           oracle/ implements the SAME symbols and is linked in their place only by tests/.
 *
 *  P layer ("pipeline ABI") host C++ restating run_ref_chunk -> search_shape -> align_queries
 *                           (run/double_indexed.cpp:102-252, align/align.cpp:203-269, align/extend.cpp:226-387)
 *                           on top of the K layer: what a `diamond blastp` maintainer would call instead of
 *                           Search::run for one (query block, reference block) pair.
 *
 * Every function returns 0 on success, non-zero on failure; the message is available from dmnd_last_error().
 * Caller owns all host buffers; the library owns device memory behind the opaque handles.  Calls on one
 * dmnd_ctx must be serialised by the caller.  There is NO CPU fallback: dmnd_create fails without a CUDA device.
 */
#ifndef DMND_B200_H
#define DMND_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define DMND_MAX_SHAPES 64
#define DMND_MAX_WEIGHT 12
#define DMND_PERIMETER_PADDING 256 /* data/string_set.h:34 */
#define DMND_DELIMITER 31          /* basic/value.h:62 */
#define DMND_LETTER_MASK 31        /* basic/value.h:63 */
#define DMND_SEED_MASK 0x80        /* basic/value.h:64 (bit 7 of a query letter) */

typedef struct dmnd_ctx dmnd_ctx;
typedef struct dmnd_block dmnd_block;
typedef struct dmnd_hits dmnd_hits;

/* Everything the kernels need that the reference keeps in globals (`config`, `score_matrix`, `shapes`,
 * Reduction::instance): filled by dmnd_params_init() from the host restatement of search/setup.cpp:338-402. */
typedef struct dmnd_params {
	int8_t score[32 * 32];            /* matrix8 layout [a*32+b], out-of-alphabet = -128 (stats/score_matrix.h:35-44) */
	int32_t gap_open, gap_extend;     /* 11 / 1 */
	uint8_t reduction[32];            /* Reduction::map_  (basic/basic.cpp:267-296): letter -> class, MASK/STOP -> 23 */
	uint8_t map8[32], map8b[32];      /* Reduction::map8_/map8b_: distinct sentinels for masked letters */
	int32_t reduction_size;           /* 10 (murphy10) */
	int32_t n_shapes, shape_weight;
	int32_t shape_len[DMND_MAX_SHAPES];
	uint32_t shape_mask[DMND_MAX_SHAPES];                 /* Shape::mask_  bit i = position i is a '1' */
	int32_t shape_pos[DMND_MAX_SHAPES][DMND_MAX_WEIGHT];  /* Shape::positions_ */
	int32_t hamming_id;               /* Search::Config::hamming_filter_id (11; 9 very-sensitive) */
	int32_t seedp_bits, index_chunks; /* search/setup.cpp:306-309, :42-53 */
	double seed_cut;                  /* seed_complexity_cut = cut * ln2 * weight (search/setup.cpp:369-370) */
	int32_t left_most_interval;       /* config.left_most_interval = 32 */
	int32_t ungapped_window;          /* config.ungapped_window = 48 */
	double ungapped_evalue;           /* 0 => stage-2 ungapped window filter skipped (--fast); > 0: Search::Config::ungapped_evalue */
	int32_t ungapped_cutoff[32];      /* Util::Scores::CutoffTable(ungapped_evalue) (util/scores/cutoff_table.h:26-47): raw score
	                                     cutoff by bit length of the query length; all 0 when ungapped_evalue == 0 */
	int32_t short_query_ungapped_cutoff; /* score_matrix.rawscore(config.short_query_ungapped_bitscore = 25) (search/stage0.cpp:187) */
	int32_t short_query_max_len;      /* config.short_query_max_len = 60 (basic/config.cpp:566) */
	/* gapped filter of the modes from --sensitive upwards (align/gapped_filter.cpp:33-63, dp/scan_diags.cpp) */
	double gapped_filter_evalue;      /* 0 => no gapped filter; 1.0 for --sensitive (search/setup.cpp:49) */
	int16_t gapped_cutoff1[32][32];   /* Util::Scores::CutoffTable2D(config.gapped_filter_evalue1 = 2000) by bit lengths of (query, target) length */
	int16_t gapped_cutoff2[32][32];   /* CutoffTable2D(gapped_filter_evalue) (run/double_indexed.cpp:302-305) */
	int32_t gapped_filter_diag_score; /* score_matrix.rawscore(config.gapped_filter_diag_bit_score = 12) (search/setup.cpp:368) */
	int32_t gapped_filter_window;     /* config.gapped_filter_window = 200 (basic/config.cpp:560) */
	float background_scores_f32[20];  /* (float)ScoreMatrix::background_scores_ (stats/score_matrix.cpp:241-248), for Hauser */
	/* tantan repeat masking (masking/tantan.cpp:121-214, called from masking/masking.cpp:162 with p_repeat 0.005,
	 * p_repeat_end 0.05, growth 1/0.9, min. mask probability config.tantan_minMaskProb 0.9): every constant the
	 * forward-backward pass uses, evaluated once on the host exactly as the reference evaluates it (fp32). */
	float tantan_lr[32 * 32];         /* Masking::likelihoodRatioMatrixf_ [a*32+b] = (float)exp(lambda * score(a,b)), a,b < 26 (whole alphabet, X * _ included); 0 elsewhere (masking.cpp:133-153) */
	float tantan_d[50];               /* d[49] = b2f0, d[i] = d[i+1] * growth (tantan.cpp:136-142) */
	float tantan_b2b, tantan_f2f, tantan_p_repeat_end, tantan_p_mask;
	int32_t max_motif_len;            /* config.max_motif_len = 30 (basic/config.cpp:602) */
	/* translated queries (blastx): the three places where the K layer asks align_mode.query_translated */
	int32_t query_contexts;           /* 1, or 6: the query block holds six frames per query; a frame of <= 85 letters then takes the stage-2
	                                     window over its whole length and ungapped_cutoff_short (search/stage2.h:41-63), and the gapped filter
	                                     reads its cutoffs at the length of the query's FIRST frame and stops after its first scan when that is
	                                     < 100 (align/gapped_filter.cpp:44-55) */
	int32_t ungapped_cutoff_short[32]; /* CutoffTable(traits.ungapped_evalue_short), search/setup.cpp:345,375 */
} dmnd_params;

/* Search::Hit (search/hit.h:30-48) as a fixed 16-byte record. */
typedef struct dmnd_hit {
	uint32_t query;       /* frame-level query id */
	int32_t seed_offset;  /* offset of the seed in the query sequence */
	uint64_t subject_score; /* bits 0..47 = global offset of the seed in the reference block (PackedLoc),
	                           bits 48..63 = score_ (0xFFFF when the ungapped stage is skipped) */
} dmnd_hit;
#define DMND_HIT_SUBJECT(h) ((h).subject_score & 0xFFFFFFFFFFFFull)
#define DMND_HIT_SCORE(h) ((uint32_t)((h).subject_score >> 48))

/* Counters printed by the reference under --log (basic/basic.cpp:186-190). */
typedef struct dmnd_stage_counters {
	uint64_t seeds_hit;          /* shared keys                      "Seeds hit" */
	uint64_t seed_hits;          /* sum nq*ns                        "Hits (filter stage 0)" */
	uint64_t tentative_matches1; /* passed Hamming                   "Hits (filter stage 1)" */
	uint64_t tentative_matches2; /* passed ungapped (== 1 for fast)  "Hits (filter stage 2)" */
	uint64_t tentative_matches3; /* passed left-most                 "Hits (filter stage 3)" */
	uint64_t masked_seeds;       /* keys erased by the entropy cut */
} dmnd_stage_counters;

/* One banded DP problem == one DpTarget (dp/dp.h:34-146) of one (query, frame). */
typedef struct dmnd_dp_problem {
	uint32_t query;   /* sequence index in the query block */
	uint32_t target;  /* sequence index in the reference block */
	int32_t d_begin;  /* band = diagonals [d_begin, d_end), diagonal = i - j */
	int32_t d_end;
} dmnd_dp_problem;

/* config.max_swipe_dp (basic/config.cpp:595): a round-2 problem with band * cols above this is not traced back unless
 * a transcript is requested; its coordinates and counts come from two statistics passes (swipe_wrapper.cpp:89-96). */
#define DMND_MAX_SWIPE_DP 1000000
enum { DMND_DP_SCORE_ONLY = 0, /* round 1: HspValues::NONE, banded_swipe.h:189-351 with DummyRowCounter */
       DMND_DP_TRACEBACK = 1   /* round 2: TracebackVectorMatrix kernel + walk, banded_swipe.h:127-187 */ };

typedef struct dmnd_dp_result {
	int32_t score;
	int32_t q_begin, q_end, t_begin, t_end; /* half-open, 0-based (Hsp::query_range / subject_range) */
	int32_t identities, mismatches, gap_openings, length, gaps, positives; /* basic/hssp.cpp:260-290 */
	uint32_t transcript_off, transcript_len; /* into the transcript buffer; 0/0 if not requested */
	int32_t status; /* 0 ok; 1 = transcript buffer too small */
} dmnd_dp_result;

/* Transcript bytes (forward order): one byte per edit operation.
 *   0x00 | n  (n=1)  is not used; encoding is: high 2 bits = op (0 match, 1 insertion(gap in subject),
 *   2 deletion(gap in query), 3 substitution), low 6 bits = letter of the subject for deletion/substitution,
 *   0 for match/insertion.  One byte per alignment column (insertions of length n are n bytes). */
enum { DMND_OP_MATCH = 0, DMND_OP_INSERTION = 1, DMND_OP_DELETION = 2, DMND_OP_SUBSTITUTION = 3 };

const char* dmnd_last_error(void);
void dmnd_set_last_error(const char* msg);
/* "cuda-sm100a" for the product library, "oracle-cpu" for the test stand-in under oracle/. */
const char* dmnd_backend(void);
/* The parameters a context was created with (dmnd_blastp checks that its options describe the same kind of query block). */
const dmnd_params* dmnd_ctx_params(const dmnd_ctx* ctx);

/* ---- K layer ---------------------------------------------------------------------------------------------- */
int dmnd_create(int device, const dmnd_params* params, dmnd_ctx** out);
void dmnd_destroy(dmnd_ctx* ctx);
/* Lane contexts: independent stream + scratch memory on the same device and parameters, owned by `ctx` (destroyed with
 * it).  Blocks uploaded through `ctx` may be used with any of its lanes; calls on DIFFERENT lanes may run concurrently
 * from different host threads (the P layer overlaps the host bridge of one query range with the kernels of another). */
int dmnd_ctx_lane(dmnd_ctx* ctx, int lane, dmnd_ctx** out);

/* `letters` is the reference's block image (256 B delimiter padding + sum(seq + 1 delimiter) + 256 B padding),
 * raw_len bytes long; limits[0..nseq] are the sequence start offsets into it (limits[0] == 256).  Copies to HBM. */
int dmnd_block_upload(dmnd_ctx* ctx, const int8_t* letters, size_t raw_len, const int64_t* limits, uint32_t nseq,
                      dmnd_block** out);
/* Same, but the letters travel asynchronously on the library's copy stream in `nranges` consecutive sequence ranges
 * [cuts[k], cuts[k+1]) (cuts[0] == 0, cuts[nranges] == nseq); the call returns while the copies are in flight.
 * dmnd_block_range_wait(ctx_or_lane, b, s_begin, s_end) makes that context's stream wait until the sequences
 * [s_begin, s_end) (and the 256 bytes after them, which their seed windows may read) have arrived -- the P layer starts
 * lane 0 while the other ranges are still uploading.  A no-op for blocks uploaded with dmnd_block_upload.
 * `letters` must stay valid (and should be page-locked) until every range has been waited for or the block is freed. */
int dmnd_block_upload_ranges(dmnd_ctx* ctx, const int8_t* letters, size_t raw_len, const int64_t* limits, uint32_t nseq,
                             const uint32_t* cuts, int nranges, dmnd_block** out);
int dmnd_block_range_wait(dmnd_ctx* ctx, const dmnd_block* b, uint32_t s_begin, uint32_t s_end);
void dmnd_block_free(dmnd_ctx* ctx, dmnd_block* b);
/* Per-position int8 composition bias (HauserCorrection::int8, stats/hauser_correction.cpp:53-109), laid out at the
 * same offsets as the block's letters.  NULL => all zero (--comp-based-stats 0). */
int dmnd_block_set_bias(dmnd_ctx* ctx, dmnd_block* b, const int8_t* bias, size_t raw_len);
/* Builds (or rebuilds) the block's seed index for shape `sid` (reference side of the join: packed seeds, sorted, with a
 * bucket directory and a Bloom filter).  dmnd_search_shape[_range] uses it when present -- every lane shares it -- and
 * builds a private one otherwise.  The index is a cache: it does not change any result. */
int dmnd_block_build_index(dmnd_ctx* ctx, dmnd_block* b, int sid);
/* Fills the block's bias array on the device: mode 1 = HauserCorrection of every sequence (stats/hauser_correction.cpp:
 * 53-109, window 40, fp32, rounded half away from zero), mode 0 = zeros (--comp-based-stats 0). */
int dmnd_block_compute_bias(dmnd_ctx* ctx, dmnd_block* b, int mode);
/* Same for the sequences [s_begin, s_end) only, on `ctx`'s stream (a lane computes the bias of its own query range); complete on return. */
int dmnd_block_compute_bias_range(dmnd_ctx* ctx, dmnd_block* b, int mode, uint32_t s_begin, uint32_t s_end);
/* Reads back the block's bias array. */
int dmnd_block_download_bias(dmnd_ctx* ctx, const dmnd_block* b, int8_t* bias, size_t raw_len);
/* Same, on the library's copy stream: returns at once, dmnd_copy_wait() blocks until `bias` is complete.  Overlaps with
 * kernels issued afterwards (the bias must have been computed before).  `bias` should come from dmnd_host_alloc(). */
int dmnd_block_download_bias_async(dmnd_ctx* ctx, const dmnd_block* b, int8_t* bias, size_t raw_len);
int dmnd_copy_wait(dmnd_ctx* ctx);
/* Page-locked host memory for buffers that cross the bus every step. */
void* dmnd_host_alloc(dmnd_ctx* ctx, size_t bytes);
void dmnd_host_free(dmnd_ctx* ctx, void* p);
/* Reads back the block's letters (query letters carry SEED_MASK bits set by dmnd_search_shape). */
int dmnd_block_download_letters(dmnd_ctx* ctx, const dmnd_block* b, int8_t* letters, size_t raw_len);
/* ---- multi-GPU (SURVEY 8e): one process per GPU, queries sharded, the packed reference block broadcast once over NVLink ------
 * The 128-byte NCCL unique id is created on one rank (dmnd_comm_unique_id) and handed to every rank by the caller's own means
 * (torch.distributed, MPI, a file); dmnd_comm_init joins the communicator.  dmnd_block_broadcast sends the root's RESIDENT block --
 * letters as they are (masked if the root masked them), limits, soft-masking table, bias -- straight into a new block on every other
 * rank (device to device, no host bounce); the root gets its own block back in *out.  This is the only collective of the path. */
int dmnd_comm_unique_id(void* out128);
int dmnd_comm_init(dmnd_ctx* ctx, int rank, int nranks, const void* unique_id128);
void dmnd_comm_destroy(dmnd_ctx* ctx);
int dmnd_block_broadcast(dmnd_ctx* ctx, int root, dmnd_block* src_on_root, dmnd_block** out);
/* An empty block of the given geometry (what dmnd_block_broadcast allocates on the receiving ranks). */
int dmnd_block_alloc_empty(dmnd_ctx* ctx, size_t raw_len, uint32_t nseq, dmnd_block** out);
/* Geometry and limits of a resident block (a rank that received its reference block by broadcast reads them back from here). */
int dmnd_block_geometry(const dmnd_block* b, size_t* raw_len, uint32_t* nseq);
int dmnd_block_download_limits(dmnd_ctx* ctx, const dmnd_block* b, int64_t* limits, size_t count);

/* ---- diagnostics: intermediate state of the seed stage for tests and tools/seed_stage_diag.py (not on the path) ----
 * dmnd_debug_block_soft: the block's soft-masking table after dmnd_block_mask(MOTIF) (Block::soft_mask, data/block/block.cpp:162-178),
 *   one byte per letter of the block image, 1 = inside an abundant motif.
 * dmnd_debug_ref_index: the reference side of the seed join for shape sid as the search reads it: *n (key, location) records in
 *   index order -- keys ascending; inside a key the locations ascend in the modes with the stage-2 window filter (their order decides
 *   which survivors share a window_ungapped_best call).  The key is an implementation detail (equal keys <=> equal seeds). */
int dmnd_debug_block_soft(dmnd_ctx* ctx, const dmnd_block* b, uint8_t* out, size_t raw_len);
int dmnd_debug_ref_index(dmnd_ctx* ctx, const dmnd_block* ref, int sid, uint64_t* keys, uint32_t* locs, size_t cap, size_t* n);
/* dmnd_debug_left_most: the left-most filter (search/left_most.h:62-110) of one (query location, reference location) pair of shape sid in
 *   index chunk `chunk`, on the block's current SEED_MASK state: out30[0] = pass, [1] match mask, [2] SEED_MASK bits of the window,
 *   [3] matcher hits left (raw << 32 | masked), [4] right, [5..6] window geometry, [7..8] verify_hits left / right (2 = not evaluated),
 *   [9..28] per left candidate: pos << 56 | verify_hit << 48 | current-shape match << 40 | valid << 36 | fingerprint << 24 | partition, [29] count. */
int dmnd_debug_left_most(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, int sid, int chunk, uint32_t qloc, uint32_t sloc, unsigned long long* out30);
/* Clears the SEED_MASK bits (run/double_indexed.cpp:211-212). */
int dmnd_block_clear_seed_mask(dmnd_ctx* ctx, dmnd_block* b);
int dmnd_block_clear_seed_mask_range(dmnd_ctx* ctx, dmnd_block* b, uint32_t q_begin, uint32_t q_end);

/* Sequence masking, a property of the resident block (MaskingAlgo bits, masking/def.h:27).
 *   DMND_MASK_TANTAN  hard masking: every letter whose tantan repeat probability is >= params.tantan_p_mask becomes
 *                     MASK_LETTER (X = 23) in place, as mask_seqs(seqs, Masking::get(), true, TANTAN) does when the
 *                     reference loads a query or reference block (run/double_indexed.cpp:122-127, :737-741;
 *                     masking/tantan.cpp:113-214, AVX2 dispatch: the fp32 evaluation order of that path is kept).
 *   DMND_MASK_MOTIF   soft masking: builds the block's MaskingTable of abundant 8-mer motifs (masking/masking.cpp:110-131:
 *                     merged ranges of table hits, none if they cover >= half of the sequence, only ranges of
 *                     <= params.max_motif_len letters).  dmnd_search_shape then enumerates seeds of either side with those
 *                     letters read as X (Block::soft_mask, search/seed_array/enum_seeds.h:262-270) and sets SEED_MASK on
 *                     the query positions MaskingTable::remove(template_len, add_bit_mask) marks (masking.cpp:96-107).
 * Sequences [s_begin, s_end) are processed on `ctx`'s stream (a lane masks its own query range).  TANTAN runs before
 * MOTIF when both bits are given (the reference builds the motif table from the hard-masked letters).  *n_hard receives
 * the number of letters hard-masked by this call; dmnd_block_mask_fetch() then copies their offsets into the block image
 * (ascending) so that the caller can keep its host copy of the letters in step. */
enum { DMND_MASK_NONE = 0, DMND_MASK_TANTAN = 1, DMND_MASK_MOTIF = 4 };
int dmnd_block_mask(dmnd_ctx* ctx, dmnd_block* b, int algo, uint32_t s_begin, uint32_t s_end, uint64_t* n_hard);
int dmnd_block_mask_fetch(dmnd_ctx* ctx, uint64_t* positions, size_t cap);

/* Stages 0-2 for shape `sid`, all index chunks in reference order; hits are grouped by query (ascending),
 * order inside a query unspecified (the reference's is thread-dependent; consumers sort, align/load_hits.h:45).
 * Sets SEED_MASK bits in the query block exactly like Search::mask_seeds (search/seed_complexity.cpp:77-127). */
int dmnd_search_shape(dmnd_ctx* ctx, dmnd_block* query, const dmnd_block* ref, int sid, dmnd_hits** out,
                      dmnd_stage_counters* counters);
/* Same for the queries [q_begin, q_end) only (query sharding inside one block); SEED_MASK bits are set in that range only. */
int dmnd_search_shape_range(dmnd_ctx* ctx, dmnd_block* query, const dmnd_block* ref, int sid, uint32_t q_begin, uint32_t q_end,
                            dmnd_hits** out, dmnd_stage_counters* counters);
size_t dmnd_hits_count(const dmnd_hits* h);
/* x-drop ungapped extension of every hit (xdrop_ungapped, dp/ungapped_align.cpp:150-214, score-only variant with the
 * query block's bias): out[k] belongs to hit k of dmnd_hits_download().  `raw_xdrop` = config.raw_ungapped_xdrop.
 * The caller applies the reference's "covered by the previous segment on this diagonal" skip (align/ungapped.cpp:84)
 * itself; the extension of one hit does not depend on any other hit. */
typedef struct dmnd_segment { int32_t i, j, len, score; } dmnd_segment; /* DiagonalSegment, util/geo/diagonal_segment.h */
int dmnd_hits_xdrop(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, const dmnd_hits* h, int raw_xdrop,
                    dmnd_segment* host, size_t cap);
/* Same, and also where each hit lies in the reference block: the sequence holding its subject position
 * (SequenceSet::local_position, data/string_set.h) and the position inside that sequence -- load_hits (align/load_hits.h:
 * 44-122) needs exactly this per hit, and the extension kernel has it at hand.  `sites` may be NULL. */
typedef struct dmnd_hit_site { uint32_t target; int32_t j; } dmnd_hit_site;
int dmnd_hits_xdrop_sites(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, const dmnd_hits* h, int raw_xdrop,
                          dmnd_segment* host, dmnd_hit_site* sites, size_t cap);
/* Gapped filter of every hit (Extension::gapped_filter, align/gapped_filter.cpp:33-63): pass[k] = 1 iff hit k's 64-diagonal
 * scan (window 100) scores above gapped_cutoff1 AND its 128-diagonal scan (window gapped_filter_window) above gapped_cutoff2,
 * both through DP::diag_alignment (dp/scan_diags.cpp:277-297) on the int8 query profile with the block's Hauser bias
 * (DP::make_profile8, dp/score_profile.cpp:32-65).  The caller keeps a target iff any of its hits passes.  Same order as
 * dmnd_hits_download(). */
int dmnd_hits_gapped_filter(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, const dmnd_hits* h, uint8_t* pass, size_t cap);
int dmnd_hits_download(dmnd_ctx* ctx, const dmnd_hits* h, dmnd_hit* host, size_t cap);
void dmnd_hits_free(dmnd_ctx* ctx, dmnd_hits* h);

/* ---- the host bridge on the device: hits -> DP problems without leaving HBM ------------------------------------------------
 * dmnd_hits_chain replaces, for every query of `h`, load_hits (align/load_hits.h:44-122: hits grouped by target), the ungapped
 * stage (align/ungapped.cpp:62-118: x-drop segment of every hit, covered hits skipped), Chaining::run (chaining/greedy_align.cpp:
 * 482-497) and add_dp_targets (align/gapped_score.cpp:107-180: band = chain diagonals +- Extension::band(query length), overlapping
 * bands merged): one record per query that has hits, ascending query ids, and the queries' banded DP problems in (query, target,
 * band) order -- exactly the round-1 problem list of a query whose targets fit one ranking chunk.  Queries with more than
 * `max_targets` targets (ranking chunks, align/extend.cpp:79-119) or with a (query, target) pair beyond the implementation's fixed
 * capacities carry DMND_CHAIN_HOST and no problems: their hits, segments and sites are returned instead (dmnd_hits_chain_fetch) and
 * the caller runs the reference's per-query logic on them.  The problem list stays on the device: dmnd_banded_swipe_chained aligns
 * it in place.  Single query context only (blastp).  `band_slow`: Extension::Mode::BANDED_SLOW band table. */
typedef struct dmnd_chain_query {
	uint32_t query, n_targets, n_problems;
	uint32_t first;   /* index of the query's first DP problem, or (DMND_CHAIN_HOST) of its first hit in the host-path arrays */
	uint32_t n_hits, flags;
} dmnd_chain_query;
enum { DMND_CHAIN_HOST = 1 };
typedef struct dmnd_chain_out { uint64_t n_queries, n_pairs, n_problems, n_host_hits; } dmnd_chain_out;
int dmnd_hits_chain(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, const dmnd_hits* h, int raw_xdrop, int band_slow,
                    int max_targets, dmnd_chain_out* out);
/* Copies the last dmnd_hits_chain's records to the host: `queries` [n_queries], `problems` [n_problems], and the hits / segments /
 * sites [n_host_hits] of the DMND_CHAIN_HOST queries (grouped by query, a query's hits ordered by target). */
int dmnd_hits_chain_fetch(dmnd_ctx* ctx, dmnd_chain_query* queries, dmnd_dp_problem* problems, dmnd_hit* hits, dmnd_segment* segs,
                          dmnd_hit_site* sites);
/* dmnd_banded_swipe over the problem list the last dmnd_hits_chain left on the device (n = its n_problems), results in list order. */
int dmnd_banded_swipe_chained(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, size_t n, int mode, dmnd_dp_result* results,
                              uint8_t* transcripts, size_t transcript_cap);

/* Banded affine-gap local alignment of n problems.  `transcripts` may be NULL (no edit transcript wanted). */
int dmnd_banded_swipe(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, const dmnd_dp_problem* problems,
                      size_t n, int mode, dmnd_dp_result* results, uint8_t* transcripts, size_t transcript_cap);

/* ---- frameshift alignment (blastx -F): 3-frame banded DP ------------------------------------------------------------------
 * banded_3frame_swipe (dp/swipe/banded_3frame_swipe.cpp:392-520, cell update dp/swipe/swipe.h:57-83): one DP over the three reading
 * frames of one strand of a DNA query against a protein target.  problems[k].query = block id of the strand's first frame (6q for
 * the forward strand, 6q + 3 for the reverse strand; the next two sequences of the query block are its frames +1 and +2),
 * d_begin / d_end = band of translated diagonals (i - j, i = codon index).  Cell (codon start x = 3i + f, column j):
 *   H = max(0, H(x-3, j-1) + s, H(x-4, j-1) + s - F, H(x-2, j-1) + s - F, hgap from (x, j-1), vgap from (x-3, j)),
 * F = frame_shift, no composition bias (the reference's legacy pipeline passes none).  DMND_DP_SCORE_ONLY fills `score` and `t_end`
 * (1 + the first target position whose column reaches the score: the reference's max_col; the caller passes the band its int16 SIMD
 * batch would have had, see host/legacy.inc); DMND_DP_TRACEBACK keeps the score
 * matrix and walks it back exactly as the reference does (:338-390, TracebackIterator :152-250), incl. its gap search order.
 * Transcript bytes as dmnd_banded_swipe, plus DMND_TR_FRAMESHIFT_FWD / _REV (op_frameshift_forward / _reverse; in forward
 * order such a byte precedes the match column that was reached through the shift). */
typedef struct dmnd_fs_result {
	int32_t score;
	int32_t q_begin, q_end;          /* Hsp::query_range: codon indices, q_begin in frame_begin, q_end in frame_end */
	int32_t frame_begin, frame_end;  /* frame offsets 0..2 inside the strand (Hsp::set_begin / set_end, basic/hssp.cpp:197-217) */
	int32_t t_begin, t_end;
	int32_t identities, mismatches, gap_openings, length, gaps, positives; /* Hsp::push_match / push_gap, basic/hssp.cpp:260-290 */
	uint32_t transcript_off, transcript_len;
	int32_t status;                  /* 0 ok; 1 = transcript buffer too small; 2 = "Traceback error" of the reference */
} dmnd_fs_result;
#define DMND_TR_FRAMESHIFT_FWD 0x41 /* '\' in the reference's pairwise and btop output */
#define DMND_TR_FRAMESHIFT_REV 0x42 /* '/' */
int dmnd_banded_3frame_swipe(dmnd_ctx* ctx, const dmnd_block* query, const dmnd_block* ref, const dmnd_dp_problem* problems, size_t n,
                             int frame_shift, int mode, dmnd_fs_result* results, uint8_t* transcripts, size_t transcript_cap);

/* Device time (ms) spent in the library's own kernels since the last reset, and the number of kernel launches: filled
 * from CUDA events recorded on the context's stream.  A root context reports itself plus its lanes; lanes run
 * concurrently, so their stream times overlap (a serial kernel time needs a single-lane run). */
typedef struct dmnd_timing {
	double seed_ms, dp_score_ms, dp_trace_ms, h2d_ms, d2h_ms;
	uint64_t launches;
	uint64_t h2d_bytes, d2h_bytes;
	uint64_t dp_cells_score, dp_cells_trace; /* algorithmic cells (band x cols) of the problems the score-only / traceback kernels were LAUNCHED on:
	                                            a fused query's problems are evaluated once, by the traceback kernel */
	uint64_t dp_cells_padded;                /* cells those kernels evaluate incl. the padding of their register tiles and wavefront */
	uint64_t dp_overflow_reruns;             /* dmnd_banded_swipe calls repeated on the int32 kernels (int16 range / bias table left) */
} dmnd_timing;
enum { DMND_TIMING_RESET = 1, DMND_TIMING_THIS_CONTEXT = 2 /* do not add the lanes */ };
int dmnd_timing_fetch(dmnd_ctx* ctx, dmnd_timing* out, int flags);
/* Roofline denominator for the DP kernels: measured issue rate (lane-instructions / s, whole GPU) of the three-input
 * integer DPX instructions (VIADDMNMX / VIMNMX3) the recurrence is built from.  Runs a ~20 ms micro-benchmark. */
int dmnd_measure_int_peak(dmnd_ctx* ctx, double* lane_instr_per_s);
/* Same for the packed form VIADDMNMX.S16x2 (two 16-bit cells per lane and instruction) the 16-bit kernel is built from. */
int dmnd_measure_int_peak_packed(dmnd_ctx* ctx, double* lane_instr_per_s);

/* ---- P layer ---------------------------------------------------------------------------------------------- */
typedef struct dmnd_search_opts {
	int32_t sensitivity;       /* 0 = --fast, 1 = default, 2 = --mid-sensitive, 3 = --sensitive, 4 = --more-sensitive, 5 = --very-sensitive,
	                              6 = --ultra-sensitive (search/setup.cpp:40-54).  Call dmnd_search_opts_default() first: a zeroed struct is
	                              not the default (top_percent 0 means --top 0).  Device status of the modes above 0: see DESIGN.md 7. */
	int32_t threads;           /* reference -p: fixes seedp_bits (search/setup.cpp:306-309); host worker threads */
	int32_t index_chunks;      /* reference -c; 0 = mode default (4) */
	int32_t comp_based_stats;  /* 0 or 1 (Hauser) */
	int32_t max_target_seqs;   /* -k, default 25; 0 = report all targets (as the reference reads -k 0) */
	double max_evalue;         /* -e, default 0.001 */
	uint64_t db_letters;       /* 0 = letters of the reference block */
	int32_t want_transcript;   /* 1 = keep edit transcripts (fmt 0) */
	int32_t masking;           /* --masking: 1 = tantan (reference default), 0 = none */
	int32_t motif_masking;     /* --motif-masking: 1 = soft-mask abundant motifs (reference default for --fast), 0 = off */
	int32_t query_contexts;    /* 1 = blastp; 6 = blastx (align_mode.query_contexts, basic/basic.cpp:42-47): the query block holds the six
	                              translated frames of every DNA query as consecutive sequences (context id = 6 * query + frame,
	                              data/block/block.cpp:86-100), nq is a multiple of 6, dmnd_match.query is the CONTEXT that aligned and
	                              q_begin / q_end are positions in that frame's translation.  0 is read as 1.  dmnd_params_init copies it
	                              into dmnd_params.query_contexts: create the context from the same options. */
	double top_percent;        /* --top: report the targets whose bit score lies within this percentage of the query's best one instead of the
	                              best max_target_seqs (config.toppercent; align/culling.cpp:90-141, align/extend.cpp:79-92,336); negative = not given */
	int32_t frame_shift;       /* blastx -F: frame shift penalty (config.frame_shift, 15 when given as 0 in long-read mode); > 0 selects the reference's
	                              frameshift alignment mode: the legacy extension pipeline (align/align.cpp:168-172, align/legacy/) -- ungapped
	                              ranking, 3-frame banded DP over seed-hit bands (dmnd_banded_3frame_swipe), no composition bias.  Needs
	                              query_contexts == 6.  dmnd_match then reports the frame the alignment BEGINS in (query), codon positions in the
	                              begin / end frames (q_begin, q_end) and the END frame in `reserved` (1 + context offset 0..5); transcripts are
	                              always kept and may hold DMND_TR_FRAMESHIFT_* bytes.  0 = off */
	int32_t range_culling;     /* --range-culling (config.query_range_culling, frameshift mode only): targets are ranked and culled per query RANGE --
	                              a target is dropped when half of the read range of its HSPs is already covered by better targets
	                              (align/legacy/banded_swipe_pipeline.cpp:139-154, output/target_culling.h:110-160).  --long-reads = this + top 10 + -F 15 */
	double min_id;             /* --id: minimum identity percentage of a reported alignment (config.min_id), 0 = no filter */
	double query_cover;        /* --query-cover: minimum percentage of the query (of the DNA read for translated searches) an alignment spans */
	double subject_cover;      /* --subject-cover: the same for the target.  Any of the three filters switches the extension to the reference's
	                              filtered schedule (align/extend.cpp:95,288: targets are only sorted, not culled, after round 1; round 2 runs in
	                              steps of max_target_seqs targets with Match::apply_filters after each, align/gapped_final.cpp:107-158,
	                              align/culling.cpp:144-184) -- without it a filter would merely thin out the best max_target_seqs targets.
	                              Equal query and subject covers >= 50 in a protein search also set the reference's min_length_ratio
	                              (run/config.cpp:156-159): seed hits between sequences whose length ratio lies below cover/100 - 0.05 are dropped */
	double min_bit_score;      /* --min-score: minimum bit score of a reported alignment; when set it REPLACES the e-value bound (ScoreMatrix::report_cutoff,
	                              stats/score_matrix.cpp:234-239) and the ranking loop no longer widens its first chunk by e-value (align/extend.cpp:262) */
	double approx_min_id;      /* --approx-id: minimum APPROXIMATE identity percentage, min(max(16.56 * score / max(query range, target range) + 11.41, 0), 100),
	                              100 for an alignment of identical stretches (Stats::approx_id, stats/stats.cpp:113-118; Hsp::approx_id_percent,
	                              basic/hssp.cpp:381-392).  A report filter like min_id; 50 / 90 and above also raise the Hamming cutoff of seed stage 1 to
	                              20 / 30 identities (search/setup.cpp:70-79,343: dmnd_params_init copies that into dmnd_params.hamming_id) */
	const uint32_t* self_targets; /* --no-self-hits: NULL, or one entry per query (per DNA query for translated searches): the reference sequence whose alignment with
	                              this query is not reported (UINT32_MAX = none).  The reference drops an HSP when query and target have the same title and the same
	                              letters (filter_hsp, align/culling.cpp:166-168, part of Match::apply_filters after round 2); titles live with the caller, so the
	                              caller names the pairs.  Unlike the other filters this one does not change the extension's schedule (align/extend.cpp:94-96) */
	double range_cover;        /* --range-cover: with range_culling, the percentage of a target's query range that better targets must cover before it is dropped
	                              (config.query_range_cover, default 50); 0 = the default */
	int32_t ext_mode;          /* --ext: 0 = the sensitivity mode's own extension mode (align/extend.cpp:62-75), 1 = banded-fast, 2 = banded-slow (the band table of
	                              Extension::band, align/gapped_score.cpp:41-72); the reference's full / global / none modes are not on this path */
} dmnd_search_opts;

typedef struct dmnd_match {
	uint32_t query, target;
	int32_t score;
	double evalue, bit_score;
	int32_t q_begin, q_end, t_begin, t_end;
	int32_t identities, mismatches, gap_openings, length, gaps, positives;
	uint64_t transcript_off;
	uint32_t transcript_len;
	uint32_t reserved;
} dmnd_match;

typedef struct dmnd_run_stats {
	dmnd_stage_counters seed;
	uint64_t hits, targets, dp_problems_round1, dp_problems_round2;
	uint64_t cells_round1, cells_round2; /* algorithmic cells = sum (d_end-d_begin)*cols, dp/dp.h:121-124 */
	uint64_t queries_aligned, matches;
	uint64_t dp_problems_fused; /* round-1 problems evaluated once WITH traceback; their queries' round-2 problems were
	                               answered from those results (counted in dp_problems_round2 / cells_round2 all the same) */
	uint64_t targets_extended;  /* targets that enter the ungapped stage, i.e. after the gapped filter where the mode has one:
	                               "Target hits (stage 3)" of the reference's --log (align/extend.cpp:215) */
	double seed_ms, host_bridge_ms, dp1_ms, dp2_ms, total_ms; /* wall clock, host */
	dmnd_timing device;
} dmnd_run_stats;

typedef struct dmnd_result dmnd_result;

void dmnd_search_opts_default(dmnd_search_opts* o);
/* The sensitivity mode's default for --motif-masking (SensitivityTraits::motif_masking, search/setup.cpp:40-54): 1, 0, or -1 for a bad mode. */
int dmnd_mode_motif_masking(int sensitivity);
/* E-value and bit score of a raw alignment score under the path's scoring system (BLOSUM62 11/1, ScoreMatrix::evalue / bitscore,
 * stats/score_matrix.cpp:217-254 with the ALP area correction) for a database of db_letters letters: what a reader of stored alignments
 * (`view` over a DAA file) needs to print the columns the search computed. */
int dmnd_alignment_stats(int32_t raw_score, uint32_t query_len, uint32_t target_len, uint64_t db_letters, double* evalue, double* bit_score);
/* Fills a dmnd_params for BLOSUM62 11/1 and the given options (host restatement of setup_search). */
int dmnd_params_init(const dmnd_search_opts* o, dmnd_params* out);
/* One (query block, reference block) pass of blastp: seed search, extension rounds, culling.
 * Matches come back grouped by query in ascending query order, inside a query in the reference's report order. */
int dmnd_blastp(dmnd_ctx* ctx, const int8_t* q_letters, size_t q_raw_len, const int64_t* q_limits, uint32_t nq,
                const int8_t* r_letters, size_t r_raw_len, const int64_t* r_limits, uint32_t nr,
                const dmnd_search_opts* opts, dmnd_result** out);
/* Same, with both blocks already resident (used by the bench's device-resident timing and by multi-GPU shards).
 * Resident blocks are in the state the reference holds a loaded block in: with opts->masking / motif_masking set the
 * caller has already run dmnd_block_mask() on both, and q_letters / r_letters are the equally masked host images
 * (dmnd_block_download_letters); dmnd_blastp() does all of that itself inside the call. */
int dmnd_blastp_resident(dmnd_ctx* ctx, dmnd_block* query, const dmnd_block* ref, const int8_t* q_letters,
                         const int64_t* q_limits, uint32_t nq, const int8_t* r_letters, const int64_t* r_limits,
                         uint32_t nr, const dmnd_search_opts* opts, dmnd_result** out);
const dmnd_match* dmnd_result_matches(const dmnd_result* r, size_t* n);
const uint8_t* dmnd_result_transcripts(const dmnd_result* r, size_t* n);
const dmnd_run_stats* dmnd_result_stats(const dmnd_result* r);
/* Offsets (ascending) into the caller's block image of the letters dmnd_blastp hard-masked (tantan, opts->masking): side 0 =
 * query block, 1 = reference block.  The reference prints MASKED sequences in its sequence-bearing output fields (btop,
 * qseq_gapped, ...: output/blast_tab_format.cpp:365-398, align/output.cpp:80-90); a caller that formats those patches its copy
 * with these.  Empty for dmnd_blastp_resident (the caller masked the blocks itself). */
const uint64_t* dmnd_result_masked_positions(const dmnd_result* r, int side, size_t* n);
/* Queries (block id of their first context) that had seed hits but ended without an alignment, ascending: the queries the reference's
 * output stage still visits (align/align.cpp:167-181, align/output.cpp:32-54) and formats with DEFAULT_REPORT_UNALIGNED (PAF, SAM) or
 * --unal 1 report as unaligned.  Queries without any seed hit are not listed, as the reference does not report them either. */
const uint32_t* dmnd_result_unaligned(const dmnd_result* r, size_t* n);
void dmnd_result_free(dmnd_result* r);

#ifdef __cplusplus
}
#endif
#endif
