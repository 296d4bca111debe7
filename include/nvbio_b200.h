/* nvbio_b200.h -- C ABI of the B200-native replacement for nvbio's two data-parallel hot paths.
 *
 * Plain C: pointers, sizes, PODs.  No torch / thrust / nvbio types in any signature.
 * All `d_` pointers are DEVICE memory owned by the caller; all calls are asynchronous on `stream`
 * (a cudaStream_t passed as void*; NULL = the legacy default stream) unless stated otherwise.
 * Return value: 0 on success, a positive cudaError_t value, or a negative NVB_E_* code.
 *
 * Every entry point names the reference interface it replaces (paths relative to the nvbio tree).
 * INTEGRATION.md shows the reference-side binding for each.
 *
 * Threads and devices.  Every call works on the CURRENT device of the calling thread (cudaSetDevice), and all `d_` pointers must
 * belong to it.  The library keeps no state between calls except, per device, lazily-created profiling events and kernel
 * attributes (both guarded; a host that drives several GPUs from one process -- nvBowtie's one compute thread per device -- may
 * call from all of its threads at once).  Two concurrent calls must not share output or temp buffers.
 */
#ifndef NVBIO_B200_H
#define NVBIO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NVB_VERSION 100

/* error codes (negative; positive values are cudaError_t) */
#define NVB_OK              0
#define NVB_E_INVALID      -1   /* bad argument (unsupported band length, bits, NULL pointer, ...) */
#define NVB_E_TEMP_SIZE    -2   /* temp buffer too small: *temp_bytes holds the required size */
#define NVB_E_CAPACITY     -3   /* an output buffer capacity would be exceeded */
#define NVB_E_UNSUPPORTED  -4   /* valid request that this build does not implement */

typedef struct nvb_uint2 { uint32_t x, y; } nvb_uint2;

/* score of an alignment sink that received no report: nvbio's Field_traits<int32>::min() (nvbio/basic/numbers.h:832-836), the value
 * aln::BestSink<int32> / Best2Sink<int32> are constructed with (sink_inl.h:40,73-78) */
#define NVB_SINK_MIN (-(1 << 30))

/* ---------------------------------------------------------------------------------------------
 * Data views
 * ------------------------------------------------------------------------------------------- */

/* FM-index in the reference's production layout (nvbio/io/fmindex/fmindex.h:302-319,
 * nvbio/io/fmindex/fmindex_impl.cu:308-322): block k = 32 bytes at byte offset 32k =
 * { uint4 bwt = 64 symbols, 2-bit big-endian ; uint4 occ = #A,#C,#G,#T in bwt[0,64k) }.
 * Mirrors nvbio::fm_index<rank_dictionary<2,64,...>, SSA_index_multiple_context<16>>
 * (nvbio/fmindex/fmindex.h:341-387): {m_length, m_primary, m_L2, m_rank_dict, m_sa}. */
typedef struct nvb_fm_index {
    const void*     d_bwt_occ;   /* ceil(length/64) blocks of 32 bytes, 32-byte aligned            */
    const uint32_t* d_ssa;       /* (length+I)/I words: SA[r] for r%I==0, ssa[0]=0xFFFFFFFF; may be
                                    NULL when only rank/match are used                             */
    uint32_t        length;      /* text length n (number of BWT symbols)                          */
    uint32_t        primary;     /* row of the `$` suffix                                          */
    uint32_t        L2[5];       /* exclusive prefix sums of the symbol counts                     */
    /* ---- optional B200 extensions; zero-initialise for an index in the reference's format ---- */
    uint32_t        sa_interval; /* I: 0 or 16 = the reference's SA_INT (FMIndexDataCore::SA_INT);
                                    any power of two down to 1 (= the full suffix array, 4 bytes per
                                    base: 12 GB at 3 Gbp, nothing on a 180 GB part) shortens locate  */
    const nvb_uint2* d_ktab;     /* 4^ktab_k inclusive SA ranges of every k-mer (index = the k symbols
                                    as a 2k-bit number, first symbol most significant), built by
                                    nvb_fm_build_ktab; replaces the first k LF steps of match()     */
    uint32_t        ktab_k;      /* 0 = no table */
    uint32_t        ktab_located;/* 0: d_ktab holds 8-byte entries {x, y};  1: 16-byte entries {x, y, SA[x], SA[y]} built by
                                    nvb_fm_build_ktab_located (SA[x] valid when y == x, both when y == x + 1): a seed whose
                                    k-mer occurs once or twice is located by the look-up + a text comparison, without walking the
                                    range on;  2: the same table built by nvb_fm_build_ktab_context -- the last word of a ONE-row
                                    entry (y == x) holds the 16 text symbols before SA[x] instead, so that such a seed (up to k + 16
                                    symbols long) is resolved by the look-up alone; and, when length < 0xC0000000, a TWO-row entry is
                                    stored as {x, 0xC0000000 | a | b << 14, SA[x], SA[x+1]} (y = x + 1 implied; a, b = the 7 symbols before
                                    SA[x], SA[x+1]), which resolves seeds up to k + 7 symbols the same way.  Ranges are identical in
                                    every case.  */
} nvb_fm_index;

/* A set of strings stored in one packed symbol stream (nvbio PackedStream semantics,
 * nvbio/basic/packedstream_inl.h:336-372): `bits` per symbol in {2,4,8}; big_endian = symbol 0 of a
 * word sits in its TOP bits (nvbio's BIG_ENDIAN_T).  String i spans symbols
 * [off_i, off_i+len_i) of the stream, with
 *     off_i = d_offsets ? d_offsets[i] : i * stride,   len_i = d_lengths ? d_lengths[i] : length.
 * This covers ConcatenatedStringSet / SparseStringSet / fixed-stride sets over a packed stream
 * (nvbio/strings/string_set.h) and the infix sets built by extract_seeds (nvbio/strings/seeds.h). */
typedef struct nvb_string_set {
    const uint32_t* d_words;
    uint32_t        bits;
    uint32_t        big_endian;
    const uint32_t* d_offsets;
    const uint32_t* d_lengths;
    uint32_t        stride;
    uint32_t        length;
} nvb_string_set;

/* alignment type, values of nvbio::aln::AlignmentType (nvbio/alignment/alignment_base.h:54) */
#define NVB_GLOBAL      0
#define NVB_LOCAL       1
#define NVB_SEMI_GLOBAL 2

/* Gotoh scoring scheme.  With d_qual_table == NULL this is aln::SimpleGotohScheme
 * (nvbio/alignment/utils.h:114-135: substitution = r==q ? match : mismatch).  With a table it is
 * nvBowtie's SmithWatermanScoringScheme<QualCost,ConstantCost>::substitution
 * (nvBowtie/bowtie2/cuda/scoring.h:281): r==q ? table[2*qual] : table[2*qual+1]; the caller evaluates
 * the reference's float expression (scoring.h:96-100) on the host into the 256x2 int32 table so that
 * fast-math differences cannot leak in.  All gap costs are negative. */
typedef struct nvb_gotoh_scheme {
    int32_t        match, mismatch;
    int32_t        pattern_gap_open, pattern_gap_ext;
    int32_t        text_gap_open, text_gap_ext;
    const int32_t* d_qual_table;     /* device, 512 int32, or NULL */
    int32_t        qual_table_min;   /* bounds of the table's values (host knowledge of device data): they admit the */
    int32_t        qual_table_max;   /* packed 16-bit DPX path; 0,0 = unknown -> the int32 kernel scores the batch   */
} nvb_gotoh_scheme;

int         nvb_version(void);
const char* nvb_error_string(int err);

/* ---------------------------------------------------------------------------------------------
 * HP-A  FM-index
 * ------------------------------------------------------------------------------------------- */

/* out[i] = rank(fmi, k[i], c[i]) : occurrences of c in bwt rows [0,k], `$`-aware.
 * Replaces nvbio::rank(fm_index,k,c)  (nvbio/fmindex/fmindex_inl.h:36-57 ->
 * rank_dictionary_inl.h:500-511 dispatch_rank<2,64,...,uint4,uint4>::run). */
int nvb_fm_rank(const nvb_fm_index* fmi, const uint32_t* d_k, const uint8_t* d_c, uint32_t n,
                uint32_t* d_out, void* stream);

/* d_out4[4*i + c] = rank(fmi, k[i], c) for c = A,C,G,T at once (16-byte aligned output).
 * Replaces nvbio::rank4(fm_index,k) / rank_all (nvbio/fmindex/fmindex_inl.h:107-133,194-222 ->
 * rank_dictionary_inl.h:539-573, the count-table popc_2bit_all path used by nvBowtie's 1-mismatch mapper). */
int nvb_fm_rank4(const nvb_fm_index* fmi, const uint32_t* d_k, uint32_t n, uint32_t* d_out4, void* stream);

/* Generic rank dictionary (SURVEY 8a row a6): a PLAIN big-endian 2-bit packed text over 32- or 64-bit words with a separate
 * occurrence table sampled every K symbols (K a multiple of the symbols per word), 32- or 64-bit counters -- the form the
 * reference's tests and its 64-bit indices instantiate.  Replaces dispatch_rank<2,K,PackedStream<...,2,true,index_type>,Occ,CT,
 * word_type,index_type>::run / run4 (nvbio/fmindex/rank_dictionary_inl.h:243-422) and build_occurrence_table<2,K> (:42-77).
 *   d_occ[4k + c]    = #c in text[0, kK)          (index_bits wide)
 *   nvb_dict_rank    d_out[t] = #c[t] in text[0, i[t]]  (i and out index_bits wide; i == all ones -> 0)
 *   nvb_dict_rank4   d_out4[4t + c] for c = A,C,G,T
 *   nvb_dict_build_occ  builds d_occ (ceil(n/K) * 4 counters) on the device; h_counts (optional) = the four symbol totals */
int nvb_dict_rank(const void* d_text, uint32_t word_bits, const void* d_occ, uint32_t index_bits, uint32_t K,
                  const void* d_i, const uint8_t* d_c, uint32_t n, void* d_out, void* stream);
int nvb_dict_rank4(const void* d_text, uint32_t word_bits, const void* d_occ, uint32_t index_bits, uint32_t K,
                   const void* d_i, uint32_t n, void* d_out4, void* stream);
int nvb_dict_build_occ(const void* d_text, uint32_t word_bits, uint64_t n_symbols, uint32_t K, uint32_t index_bits, void* d_occ, uint64_t h_counts[4],
                       void* d_temp, size_t* temp_bytes, void* stream);

#define NVB_MATCH_FORWARD_ORDER 1u  /* consume the query left-to-right instead of right-to-left   */
#define NVB_MATCH_COMPLEMENT    2u  /* complement each symbol (c<4 ? 3-c : c) before ranking      */
/* FORWARD_ORDER|COMPLEMENT is how nvBowtie searches the reverse-complement strand of a seed over the
 * forward index (nvBowtie/bowtie2/cuda/mapping_inl.h:292-309). */

/* Exact backward search of n queries: d_ranges[i] = inclusive SA range (x,y), empty iff x>y;
 * a query symbol > 3 yields (1,0).
 * Replaces nvbio::match(fm_index,pattern,len) (nvbio/fmindex/fmindex_inl.h:280-341), nvBowtie's
 * match_range (nvBowtie/bowtie2/cuda/mapping_inl.h:83-97) and the thrust::transform(rank_functor) of
 * FMIndexFilter::rank (nvbio/fmindex/filter_inl.h:283-287). */
int nvb_fm_match(const nvb_fm_index* fmi, const nvb_string_set* queries, uint32_t n, uint32_t flags,
                 nvb_uint2* d_ranges, void* stream);

/* One-mismatch seed search: nvBowtie's map<find_exact>(query, len1, len2, index, ...) as a batch primitive
 * (nvBowtie/bowtie2/cuda/mapping_inl.h:128-220, the rank4-based core of the APPROX / CASE_PRUNING seed mappers,
 * :318-429).  For query i: every SA range of the query with exactly one substitution among its consumed symbols
 * [exact_len, len) (none in the first exact_len), in the reference's push order (position ascending, substituted
 * symbol ascending), followed by the perfect match when find_exact; an N inside the exact region or a second N yields
 * nothing, a single later N ends exact matching there.  "Consumed symbols" are the stream's symbols in order with
 * NVB_MATCH_FORWARD_ORDER (nvBowtie's forward reader over its reversed reads), reversed without it.
 * d_ranges[i*max_out + k] = k-th inclusive range (k < min(count, max_out)); d_counts[i] = pushes; d_range_sums[i]
 * (optional) = sum of the range sizes (the reference's range_sum; range_count = count).
 * The bounded priority deque the reference feeds (seed_hit_deque_array.h) stays with the caller. */
int nvb_fm_match_approx(const nvb_fm_index* fmi, const nvb_string_set* queries, uint32_t n, uint32_t flags,
                        uint32_t exact_len, int find_exact, uint32_t max_out,
                        nvb_uint2* d_ranges, uint32_t* d_counts, uint32_t* d_range_sums, void* stream);

/* -------------------------------------------------------------------------------------------
 * nvBowtie's seed-mapping stage (SURVEY 8a row a10 / 8f-2): for every queued read, the seeds at symbol offsets
 *     begin + retry * (seed_freq / (max_reseed + 1)) + k * seed_freq      while the seed fits
 * are searched on both strands -- exactly (EXACT) or with one substitution outside the first subseed_len consumed symbols
 * (APPROX) -- and their SA ranges kept in a BOUNDED per-read priority deque of at most max_hits SeedHits ordered by range
 * size.  Replaces map_queues_kernel<EXACT_MAPPING|APPROX_MAPPING> (nvBowtie/bowtie2/cuda/mapping_inl.h:229-366, 539-591),
 * the entry points map / map_exact / map_approx (mapping.cu:63-188) and the deque storage (seed_hit_deque_array.h:157-204).
 * CASE_PRUNING mapping needs the reverse index and is not implemented.
 *   reads            4-bit (DNA_N) or 2-bit big-endian strings; nvBowtie reads the forward strand of a seed front to back
 *                    (NVB_MATCH_FORWARD_ORDER) and the other strand back to front, complemented (mapping_inl.h:263-309)
 *                    A seed containing an N is skipped by both mappers (as the reference's N test does, mapping_inl.h:258,346).
 *   d_queue          read ids to process (PingPongQueuesView::in_queue), or NULL = 0 .. n_queue-1
 *   d_seed_freq      optional per-read seed interval (nvBowtie evaluates SimpleFunc(read length) in float on the device,
 *                    params.cpp:157-158: evaluate it on the host); NULL = params->seed_freq for every read
 *   d_hits           arena of max_hits slots per READ ID: the read's hits sorted by range size (ascending, stable in push
 *                    order = the order pop_top() yields); d_counts[read id] = their number
 *   d_reseed[i]      (optional) 1 when queue entry i found no range or range_sum >= rep_seeds * range_count (:586-588)
 *   d_range_stats    (optional) [2*i] = range_sum, [2*i+1] = range_count of queue entry i
 * A full deque drops a largest range before every further push, as the reference does (pop_bottom, then push); among equally
 * large ranges the most recently pushed one goes (an interval heap's choice depends on its layout): the kept range SIZES, the
 * statistics and -- whenever a read pushes at most max_hits hits -- the complete hit sets equal the reference's. */
typedef struct nvb_seed_hit {          /* bowtie2::cuda::SeedHit, seed_hit.h:54-98,230-232 (8 bytes) */
    uint32_t range_begin;              /* SA range [range_begin, range_begin + delta) -- EXCLUSIVE end */
    uint32_t bits;                     /* delta:20 | pos_in_read:10 | rc:1 | index_dir:1 (low to high) */
} nvb_seed_hit;
#define NVB_MAP_EXACT  0u
#define NVB_MAP_APPROX 1u
#define NVB_MAP_MAX_PUSHES 100u        /* an approximate seed of length L pushes at most 3 L + 1 ranges: L <= 33 */
typedef struct nvb_map_params {
    uint32_t algorithm;                /* NVB_MAP_EXACT | NVB_MAP_APPROX */
    uint32_t seed_len, seed_freq;      /* ParamsPOD::seed_len, seed_freq(read_len) evaluated on the host */
    uint32_t max_hits, max_reseed, rep_seeds, subseed_len, min_read_len;
    uint32_t fw, rc;                   /* search the forward / the reverse-complement strand */
} nvb_map_params;
int nvb_map_seeds(const nvb_fm_index* fmi, const nvb_string_set* reads, const uint32_t* d_queue, uint32_t n_queue, uint32_t retry,
                  const nvb_map_params* params, const uint32_t* d_seed_freq,
                  nvb_seed_hit* d_hits, uint32_t* d_counts, uint8_t* d_reseed, uint32_t* d_range_stats, void* stream);

/* Two-phase locate of queued SA rows (nvBowtie/bowtie2/cuda/locate_inl.h:122-210; nvbio/fmindex/fmindex_inl.h:502-569
 * locate_ssa_iterator / lookup_ssa_iterator): init walks LF to the next sampled row, lookup adds the sampled position.
 * d_idx (optional) is the sorting permutation nvBowtie passes as idx_queue: entry t works on element d_idx[t] of the arrays. */
int nvb_fm_locate_init(const nvb_fm_index* fmi, const uint32_t* d_rows, const uint32_t* d_idx, uint32_t n,
                       uint32_t* d_sampled_row, uint32_t* d_steps, void* stream);
int nvb_fm_locate_lookup(const nvb_fm_index* fmi, const uint32_t* d_sampled_row, const uint32_t* d_steps, const uint32_t* d_idx, uint32_t n,
                         uint32_t* d_pos, void* stream);
/* locate with the rows radix-sorted first "to gather locality" (aligner_best_approx.h:737-756): same positions as nvb_fm_locate,
 * returned in the input order. */
int nvb_fm_locate_sorted(const nvb_fm_index* fmi, const uint32_t* d_rows, uint32_t n, uint32_t* d_pos,
                         void* d_temp, size_t* temp_bytes, void* stream);

/* d_pos[i] = text position of SA row d_rows[i]  (row 0 -> 0xFFFFFFFF as in the reference).
 * Replaces nvbio::locate(fm_index,i) (nvbio/fmindex/fmindex_inl.h:471-499) with
 * SSA_index_multiple_context<16>::fetch (nvbio/fmindex/ssa_inl.h:487-504). */
int nvb_fm_locate(const nvb_fm_index* fmi, const uint32_t* d_rows, uint32_t n, uint32_t* d_pos, void* stream);

/* FMIndexFilter<device_tag>::rank (nvbio/fmindex/filter_inl.h:268-300): match every query, then
 * d_slots = inclusive scan of the range sizes (uint64).  The total hit count is d_slots[n-1]; if
 * h_n_hits != NULL the call synchronises the stream and stores it there (the reference returns it). */
int nvb_fm_filter_rank(const nvb_fm_index* fmi, const nvb_string_set* queries, uint32_t n, uint32_t flags,
                       nvb_uint2* d_ranges, uint64_t* d_slots, uint64_t* h_n_hits,
                       void* d_temp, size_t* temp_bytes, void* stream);

/* FMIndexFilter<device_tag>::locate(begin,end,hits) (nvbio/fmindex/filter_inl.h:306-402):
 * for global hit index h in [begin,end): d_hits[h-begin] = (text position, query id). */
int nvb_fm_filter_locate(const nvb_fm_index* fmi, const nvb_uint2* d_ranges, const uint64_t* d_slots,
                         uint32_t n_queries, uint64_t begin, uint64_t end, nvb_uint2* d_hits, void* stream);

/* ---------------------------------------------------------------------------------------------
 * HP-B  batched banded Gotoh score
 * ------------------------------------------------------------------------------------------- */

/* For i < n: banded DP of patterns[i] (rows) against texts[i] (band anchored at text offset 0),
 * d_score[i] / d_sink[i] = BestSink<int32>{score, sink=(text_end, pattern_end)}; an alignment with
 * text_len < pattern_len leaves the sink at its defaults (NVB_SINK_MIN, (-1,-1)).
 * band_len in {3,5,7,15,31,63}.  d_quals (one byte per pattern symbol, indexed like the pattern
 * stream) may be NULL (trivial_quality_string).
 * Replaces aln::BatchedBandedAlignmentScore<BAND_LEN,stream,DeviceThreadScheduler>::enact and
 * aln::batch_banded_alignment_score<BAND_LEN> with GotohAligner (nvbio/alignment/batched_banded_inl.h:
 * 78-162, nvbio/alignment/batched_inl.h:1067-1101 -> gotoh/gotoh_banded_inl.h:406-658).
 * Temp storage follows the reference's min_temp_storage/enact(temp_size,temp) convention
 * (nvbio/alignment/batched.h:333-353): call with d_temp==NULL to query *temp_bytes. */
int nvb_banded_gotoh_score(int band_len, int type, const nvb_gotoh_scheme* scheme,
                           const nvb_string_set* patterns, const uint8_t* d_quals,
                           const nvb_string_set* texts, uint32_t n,
                           int32_t* d_score, nvb_uint2* d_sink,
                           void* d_temp, size_t* temp_bytes, void* stream);

/* same, reading the number of alignments from device memory (*d_n <= n_max): lets a pipeline chain
 * locate -> extend without a host round trip. */
int nvb_banded_gotoh_score_indirect(int band_len, int type, const nvb_gotoh_scheme* scheme,
                           const nvb_string_set* patterns, const uint8_t* d_quals,
                           const nvb_string_set* texts, const uint32_t* d_n, uint32_t n_max,
                           int32_t* d_score, nvb_uint2* d_sink,
                           void* d_temp, size_t* temp_bytes, void* stream);

/* Windowed banded Gotoh score (SURVEY 8a row b7, second half): rows [window_begin, min(window_end, pattern length)) of every
 * alignment still alive, the (H, F) band carried between calls in d_checkpoints (band_len short2 per alignment, clamped at
 * SHRT_MIN+32 when stored), the BestSink in d_score / d_sink (in/out) and the reference's bool result in d_alive
 * (0 = text shorter than pattern, or the band maximum can no longer reach d_min_score[i] + remaining_rows * match; such
 * alignments are skipped by later passes).  window_begin == 0 initialises score / sink / alive.  d_min_score may be NULL
 * (= INT_MIN: never give up).  Scoring a pattern in consecutive windows yields exactly nvb_banded_gotoh_score's result.
 * Replaces aln::banded_alignment_score<BAND_LEN>(aligner, pattern, quals, text, min_score, window_begin, window_end, sink,
 * checkpoint) (nvbio/alignment/banded_inl.h:178-218, gotoh_banded_inl.h:132-199,616-634,706-739), the per-pass body of
 * BatchedBandedAlignmentScore<..., DeviceStagedThreadScheduler> (batched_banded_inl.h:170-241).  bands 3, 5, 7, 15, 31. */
int nvb_banded_gotoh_score_window(int band_len, int type, const nvb_gotoh_scheme* scheme,
                                  const nvb_string_set* patterns, const uint8_t* d_quals, const nvb_string_set* texts, uint32_t n,
                                  uint32_t window_begin, uint32_t window_end, const int32_t* d_min_score,
                                  int16_t* d_checkpoints, int32_t* d_score, nvb_uint2* d_sink, uint8_t* d_alive, void* stream);

/* Banded Gotoh score with aln::Best2Sink<int32>(distinct_dist) (nvbio/alignment/sink.h:114-147, sink_inl.h:70-116) instead of BestSink: the
 * best alignment (last maximal report wins) and the best one whose text end is more than distinct_dist away from it -- the second-best
 * score a MAPQ estimate needs.  d_out6[6*i ..] = (score1, sink1.x, sink1.y, score2, sink2.x, sink2.y); unset entries keep the sink's
 * defaults (NVB_SINK_MIN, 0xFFFFFFFF).  Every report the reference makes reaches the sink in its order (LOCAL: every cell, row by row).
 * One alignment per thread on the int32 kernel; bands 3, 5, 7, 15, 31, 63. */
int nvb_banded_gotoh_score_best2(int band_len, int type, const nvb_gotoh_scheme* scheme,
                                 const nvb_string_set* patterns, const uint8_t* d_quals, const nvb_string_set* texts, uint32_t n,
                                 uint32_t distinct_dist, int32_t* d_out6, void* stream);

/* Full-matrix (un-banded) Gotoh score (SURVEY 8f-3): every pattern against the WHOLE of its text.
 * d_score / d_sink = BestSink<int32>{score, (text end, pattern end)}; pattern and text lengths must be >= 1 and
 * `patterns->length` / `texts->length` must bound them (<= 65535; the text bound sizes the boundary-column scratch).
 * Replaces aln::alignment_score / aln::BatchedAlignmentScore<stream,DeviceThreadScheduler> with
 * GotohAligner<TYPE,SimpleGotohScheme> (default PatternBlockingTag; nvbio/alignment/alignment_inl.h:95-125,
 * gotoh/gotoh_inl.h:459-960, batched_inl.h:236-605) -- the DP sw-benchmark times (sw-benchmark.cu:592-641) and nvBowtie's
 * opposite-mate scoring.  LOCAL ties resolve in the reference's (8-column stripe, row, column) order.
 * d_quals (one byte per pattern symbol, indexed like the pattern offsets; may be NULL) and scheme->d_qual_table select the
 * quality-dependent substitution scores as in nvb_banded_gotoh_score; such batches run on the int32 kernel. */
int nvb_gotoh_score(int type, const nvb_gotoh_scheme* scheme, const nvb_string_set* patterns, const uint8_t* d_quals, const nvb_string_set* texts, uint32_t n,
                    int32_t* d_score, nvb_uint2* d_sink, void* d_temp, size_t* temp_bytes, void* stream);

/* Same, with the number of alignments read from device memory (*d_n, clamped to n_max): lets a producer kernel decide
 * the batch size without a host round trip (the opposite-mate stage of nvb_seed_extend_paired). */
int nvb_gotoh_score_indirect(int type, const nvb_gotoh_scheme* scheme, const nvb_string_set* patterns, const uint8_t* d_quals, const nvb_string_set* texts,
                             const uint32_t* d_n, uint32_t n_max,
                             int32_t* d_score, nvb_uint2* d_sink, void* d_temp, size_t* temp_bytes, void* stream);

/* Full-matrix Gotoh traceback: score + sink as nvb_gotoh_score, plus the alignment itself.
 *   d_ops[i*max_ops ..]  the backtracer's pushes in END -> START order (0 = SUBSTITUTION 'M', 1 = INSERTION 'I' (pattern symbol
 *                        against a gap), 2 = DELETION 'D'), d_n_ops[i] their number (may exceed max_ops: then truncated)
 *   d_source[i]          = (text begin, pattern begin) of the alignment; the soft clips of the pattern are
 *                          pattern_len - sink.y at the end and source.y at the start
 * Replaces aln::alignment_traceback<MAX_PATTERN_LEN,MAX_TEXT_LEN,CHECKPOINTS> with a Gotoh aligner (generic driver
 * nvbio/alignment/alignment_inl.h:365-530; state machine gotoh/gotoh_inl.h:1806-1871) and its batched form
 * BatchedAlignmentTraceback (batched_inl.h:607-860).  No checkpoints: d_temp holds the whole direction matrix, 4 bits per cell
 * (max_text_len * ceil(max_pattern_len/32) * 16 bytes per alignment). */
int nvb_gotoh_traceback(int type, const nvb_gotoh_scheme* scheme, const nvb_string_set* patterns, const uint8_t* d_quals, const nvb_string_set* texts, uint32_t n,
                        int32_t* d_score, nvb_uint2* d_sink, nvb_uint2* d_source,
                        uint8_t* d_ops, uint32_t max_ops, uint32_t* d_n_ops,
                        void* d_temp, size_t* temp_bytes, void* stream);

/* Banded Gotoh traceback (SURVEY 8f-4).  For i < n: score, sink (end cells) as nvb_banded_gotoh_score, plus the
 * source (start cells) and the alignment as the backtracer's pushes in END -> START order, one byte per op
 * (0 = SUBSTITUTION 'M', 1 = INSERTION 'I', 2 = DELETION 'D'; nvbio::aln::DirectionVector) at d_ops[i*max_ops ..];
 * d_n_ops[i] = number of ops (ops beyond max_ops are counted, not stored; max_ops >= pattern length + band_len always
 * suffices).  The soft clips the reference passes to Backtracer::clip are (pattern_len - sink.y) and source.y.
 * `patterns->length` must bound the pattern lengths (it sizes the per-alignment direction matrix in d_temp).
 * Replaces aln::banded_alignment_traceback<BAND_LEN,MAX_PATTERN_LEN,CHECKPOINTS> and
 * BatchedBandedAlignmentTraceback (nvbio/alignment/banded_inl.h:352-489, gotoh/gotoh_banded_inl.h:763-962,
 * batched_banded_inl.h:248-451): instead of 32-row checkpoints + window recomputation the whole 4-bit direction
 * matrix of every alignment is kept in HBM and walked once. */
int nvb_banded_gotoh_traceback(int band_len, int type, const nvb_gotoh_scheme* scheme,
                               const nvb_string_set* patterns, const uint8_t* d_quals, const nvb_string_set* texts, uint32_t n,
                               int32_t* d_score, nvb_uint2* d_sink, nvb_uint2* d_source,
                               uint8_t* d_ops, uint32_t max_ops, uint32_t* d_n_ops,
                               void* d_temp, size_t* temp_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Index construction on the device (SURVEY 8f-1; needed to run any of the above on synthetic data)
 * ------------------------------------------------------------------------------------------- */

/* Build occ + interleave: d_bwt holds n 2-bit big-endian BWT symbols (ceil(n/64)*4 words, padding
 * ignored); writes ceil(n/64) 32-byte blocks to d_bwt_occ and the L2 table to h_L2 (synchronises).
 * Replaces nvbio::build_occurrence_table<2,64> + the interleave loop
 * (nvbio/fmindex/rank_dictionary_inl.h:42-77, nvbio/io/fmindex/fmindex_impl.cu:263-331). */
int nvb_fm_build_occ(const uint32_t* d_bwt, uint32_t n, void* d_bwt_occ, uint32_t h_L2[5],
                     void* d_temp, size_t* temp_bytes, void* stream);

/* Suffix-sort a 2-bit big-endian packed text of n symbols on the device and emit the BWT (nvbio
 * convention: `$` row removed, nvbio/fmindex/bwt.h:51-63), the primary row, the sampled SA
 * (every sa_interval-th row, ssa[0]=0xFFFFFFFF; sa_interval 0 means 16) and optionally the full SA with
 * the `$` row (n+1 entries, d_sa may be NULL).
 * d_bwt must hold ceil(n/64)*4 words, d_ssa (n+I)/I words.  Synchronises. */
int nvb_fm_build_bwt(const uint32_t* d_text, uint32_t n, uint32_t* d_bwt, uint32_t* h_primary,
                     uint32_t* d_ssa, uint32_t sa_interval, uint32_t* d_sa,
                     void* d_temp, size_t* temp_bytes, void* stream);

/* Fill d_ktab[4^k] with match() of every k-mer (level by level: 4^k * 4/3 LF steps in total).
 * k in [1,16] (8.6 GB at k=15, 34 GB at k=16).  fmi->d_ktab / ktab_k are ignored on input. */
int nvb_fm_build_ktab(const nvb_fm_index* fmi, uint32_t k, nvb_uint2* d_ktab, void* stream);

/* The same table with 16-byte entries {x, y, SA[x], SA[y]} (d_ktab16: 4^k * 16 bytes, 16-byte aligned; 69 GB at k = 16 -- HBM capacity
 * traded for dependent gathers).  The SA values are filled for ranges of one row (x == y) or two (y == x + 1) and need the full suffix array
 * (fmi->sa_interval == 1), else NVB_E_UNSUPPORTED.  Use with nvb_fm_index.d_ktab = d_ktab16, ktab_located = 1. */
int nvb_fm_build_ktab_located(const nvb_fm_index* fmi, uint32_t k, void* d_ktab16, void* stream);

/* nvb_fm_build_ktab_located + text context: for every one-row entry the unused last word is filled with the (up to) 16 symbols of
 * d_text (2-bit big-endian, the text the index was built from) that precede SA[x], symbol SA[x]-1 in the two lowest bits; two-row
 * entries are packed as described at nvb_fm_index.ktab_located.  Use with nvb_fm_index.d_ktab = d_ktab16, ktab_located = 2. */
int nvb_fm_build_ktab_context(const nvb_fm_index* fmi, uint32_t k, const uint32_t* d_text, void* d_ktab16, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Seed + extend composition (the fmmap / nvBowtie hot loop: seeds -> match -> locate -> window ->
 * banded Gotoh -> best score per read; nvbio examples/fmmap/fmmap.cu:255-400)
 * ------------------------------------------------------------------------------------------- */
typedef struct nvb_seed_extend_params {
    uint32_t seed_len;        /* 20 (nvBowtie local) / 22 (fmmap)                                    */
    uint32_t seed_interval;   /* 10 for 150 bp: int(1 + 0.75*sqrtf(150)) evaluated on the host        */
    uint32_t band_len;        /* 31 */
    uint32_t type;            /* NVB_LOCAL */
    uint32_t both_strands;    /* 1: also seed/extend the reverse complement of every read           */
    uint32_t max_seed_hits;   /* ranges wider than this contribute only their first max_seed_hits rows */
    uint32_t dedup_jobs;      /* 1: hits of a read that define the same (strand, window) alignment are scored once and
                                 the result copied to each of them (bit-identical per-hit outputs, fewer cells)       */
    nvb_gotoh_scheme scheme;
    const uint8_t* d_read_quals; /* optional base qualities, one byte per read symbol: the quality of symbol p of read r is
                                    d_read_quals[offset of read r in symbols + p] (the indexing of nvb_banded_gotoh_score's
                                    d_quals); used with scheme.d_qual_table (nvBowtie's scoring); NULL = none        */
} nvb_seed_extend_params;

/* reads: n_reads strings (2- or 4-bit).  genome: 2-bit big-endian packed text of fmi->length symbols.
 * Outputs: d_best_score[n_reads] (INT_MIN when a read has no hit), d_best_pos[n_reads] = genome
 * coordinate of the best alignment's end (window begin + sink.x; 0xFFFFFFFF when none).  A read whose best job has a
 * window shorter than the read (the read runs past the genome's end: no alignment fits) keeps the DP's score for it,
 * -2^30, and gets d_best_pos 0xFFFFFFFF.
 * Optional per-hit outputs (may be NULL) of capacity hit_capacity: d_hit_read (string id = read*strands
 * + strand), d_hit_window (begin,end), d_hit_score, d_hit_sink; d_n_hits[0] receives the number of hits
 * kept (<= hit_capacity), d_n_hits[1] the number found and d_n_hits[2] the number of distinct alignment jobs
 * actually scored (device counters, no host round trip).
 * Returns NVB_E_TEMP_SIZE with the needed size when d_temp is NULL/too small. */
int nvb_seed_extend(const nvb_fm_index* fmi, const uint32_t* d_genome,
                    const nvb_string_set* reads, uint32_t n_reads,
                    const nvb_seed_extend_params* params, uint32_t hit_capacity,
                    int32_t* d_best_score, uint32_t* d_best_pos,
                    uint32_t* d_n_hits, uint32_t* d_hit_read, nvb_uint2* d_hit_window,
                    int32_t* d_hit_score, nvb_uint2* d_hit_sink,
                    void* d_temp, size_t* temp_bytes, void* stream);

/* Optional alignment of every read's best hit (what nvBowtie's banded_traceback_best produces for SAM output,
 * aligner_best_approx.h:300-500): the banded traceback of the best (strand, window) job of each read.
 *   d_ops[r*max_ops ..]  ops in END -> START order (0 M, 1 I, 2 D), d_n_ops[r] their number (0 when the read has no hit)
 *   d_begin[r]           = (genome coordinate of the alignment's first text symbol, first aligned read symbol);
 *                          (0xFFFFFFFF, 0xFFFFFFFF) with n_ops 0 when the read has no hit, or when its best job's window is
 *                          shorter than the read (no alignment: d_best_pos is 0xFFFFFFFF too)
 *   d_strand[r]          = 0 forward, 1 reverse complement (the read symbols are those of that strand's string)
 * Call with the same arguments as nvb_seed_extend plus this struct; temp size grows by the direction matrices. */
typedef struct nvb_best_alignment_out {
    uint8_t*   d_ops;
    uint32_t   max_ops;
    uint32_t*  d_n_ops;
    nvb_uint2* d_begin;
    uint8_t*   d_strand;
} nvb_best_alignment_out;

int nvb_seed_extend_traceback(const nvb_fm_index* fmi, const uint32_t* d_genome,
                    const nvb_string_set* reads, uint32_t n_reads,
                    const nvb_seed_extend_params* params, uint32_t hit_capacity,
                    int32_t* d_best_score, uint32_t* d_best_pos,
                    uint32_t* d_n_hits, uint32_t* d_hit_read, nvb_uint2* d_hit_window,
                    int32_t* d_hit_score, nvb_uint2* d_hit_sink,
                    const nvb_best_alignment_out* best_alignment,
                    void* d_temp, size_t* temp_bytes, void* stream);

/* -------------------------------------------------------------------------------------------
 * Paired-end composition (BASELINE configs[4] shape; nvBowtie best_approx paired: anchor scoring + opposite-mate full DP,
 * nvBowtie/bowtie2/cuda/aligner_best_approx_paired.h, score_opposite_inl.h:90-266, alignment_utils.h:62-95 PE_POLICY_FR).
 *
 * reads = 2*n_pairs strings: mate 1 of pair p at index p, mate 2 at index n_pairs + p.  Every mate is seeded and extended
 * on its own (nvb_seed_extend with both_strands = 1, which is required).  Per pair:
 *   - if both mates have a best alignment, on opposite strands, the forward one starting at or before the reverse one,
 *     ending at or before it, and the fragment [begin of the forward mate, end of the reverse mate) has a length in
 *     [min_frag, max_frag]: the pair is CONCORDANT as it stands (alignment begin := end - read length, clamped at 0);
 *   - otherwise every mate that has an alignment (score >= min_mate_score) acts as anchor and the OTHER mate is searched
 *     with the full-matrix Gotoh DP (nvb_gotoh_score, same type and scheme) where the FR policy puts it: anchor forward at
 *     [b, e) -> the reverse complement of the other mate in [b, min(b + max_frag, genome length)); anchor reverse ->
 *     the other mate forward in [max(e - max_frag, 0), e)  (score_opposite_inl.h:177-191 with pe_overlap).  A rescue whose
 *     score reaches min_mate_score yields a candidate pair; the candidate with the larger score sum wins (tie: mate 1 as
 *     anchor).  No candidate: the pair is UNPAIRED and each mate keeps its own best alignment.
 * A mate's alignment BEGIN is taken as (end - read length, clamped at 0), not from a traceback: with soft clips or indels the true
 * start differs by a few bases, so pairs within that distance of min_frag / max_frag may be classified differently from a
 * caller that traces every alignment (nvBowtie does); callers that need the exact extent can request the traceback
 * (nvb_seed_extend_traceback) and re-check those pairs.
 * At most rescue_capacity full-DP jobs are run per call (in pair order; d_n_rescue[1] reports how many were wanted).
 * Outputs (mate m of pair p at index m*n_pairs + p): d_pair_score (sum of the two mates' scores, INT_MIN when unpaired),
 * d_pair_flags (NVB_PAIR_*), d_mate_score (INT_MIN = unaligned), d_mate_pos (genome coordinate one past the last aligned
 * base, 0xFFFFFFFF = unaligned), d_mate_strand (0 forward, 1 reverse complement). */
typedef struct nvb_pair_params {
    uint32_t min_frag, max_frag;
    int32_t  min_mate_score;
    uint32_t rescue_capacity;
} nvb_pair_params;
typedef struct nvb_pair_out {
    int32_t*  d_pair_score;     /* [n_pairs]   */
    uint32_t* d_pair_flags;     /* [n_pairs]   */
    int32_t*  d_mate_score;     /* [2*n_pairs] */
    uint32_t* d_mate_pos;       /* [2*n_pairs] */
    uint8_t*  d_mate_strand;    /* [2*n_pairs] */
    uint32_t* d_n_rescue;       /* [2] full-DP jobs run, wanted (may be NULL) */
} nvb_pair_out;
#define NVB_PAIR_UNPAIRED       0u
#define NVB_PAIR_CONCORDANT     1u    /* the mates' independent best alignments form a proper FR pair */
#define NVB_PAIR_RESCUED_MATE1  2u    /* mate 1 was placed by the opposite-mate DP next to mate 2's alignment */
#define NVB_PAIR_RESCUED_MATE2  4u

int nvb_seed_extend_paired(const nvb_fm_index* fmi, const uint32_t* d_genome,
                    const nvb_string_set* reads, uint32_t n_pairs,
                    const nvb_seed_extend_params* params, uint32_t hit_capacity,
                    const nvb_pair_params* pair_params, const nvb_pair_out* out,
                    uint32_t* d_n_hits, void* d_temp, size_t* temp_bytes, void* stream);

/* -------------------------------------------------------------------------------------------
 * Host-buffer entry point: batches of reads in HOST memory in, per-read results in HOST memory out.
 * Replaces nvBowtie's input thread -> compute thread hand-off and its per-stage cudaDeviceSynchronize
 * (nvBowtie/bowtie2/cuda/compute_thread.cu:213-243, nvBowtie/bowtie2/cuda/defs.h:64, aligner_best_approx.h:219-241):
 * `depth` batches are in flight at once -- the host->device copy of batch i+1 and the device->host copy of batch i-1
 * overlap the kernels of batch i on separate streams.  By default all batches share ONE compute stream (their kernels run back
 * to back); the environment variable NVB_PIPELINE_COMPUTE_STREAMS=k (read at creation) spreads consecutive batches over k
 * compute streams so that kernels of neighbouring batches may share the SMs (measured: profiles/README.md).
 *
 * Reads: n_reads fixed-stride strings of `read_len` symbols, `words_per_read` 32-bit words each (big-endian packing,
 * read_bits = 2 or 4).  pair_params != NULL: paired-end (reads = mate 1 of every pair, then mate 2; n_reads even).
 * submit() takes a host pointer (pinned memory makes the copy asynchronous) that must stay valid until wait() returns for
 * that ticket; wait() blocks until that batch's results are in the pipeline's own pinned host buffers and returns pointers
 * to them (valid until `depth` further batches have been submitted).  One pipeline is used from one host thread.
 * ------------------------------------------------------------------------------------------- */
typedef struct nvb_pipeline nvb_pipeline;
typedef struct nvb_pipeline_result {
    const int32_t*  best_score;    /* [n_reads]  single end (NULL when paired) */
    const uint32_t* best_pos;      /* [n_reads]  */
    const uint32_t* n_hits;        /* [3] hits kept, found, distinct alignment jobs */
    const int32_t*  pair_score;    /* [n_pairs]   paired end (NULL when single end), as nvb_pair_out */
    const uint32_t* pair_flags;    /* [n_pairs]   */
    const int32_t*  mate_score;    /* [2*n_pairs] */
    const uint32_t* mate_pos;      /* [2*n_pairs] */
    const uint8_t*  mate_strand;   /* [2*n_pairs] */
    const uint32_t* n_rescue;      /* [2] */
    float           device_ms;     /* device time of this batch's kernels (its compute stream), for reporting */
} nvb_pipeline_result;

int  nvb_pipeline_create(const nvb_fm_index* fmi, const uint32_t* d_genome, const nvb_seed_extend_params* params,
                         const nvb_pair_params* pair_params /* NULL = single end */,
                         uint32_t n_reads, uint32_t read_len, uint32_t words_per_read, uint32_t read_bits,
                         uint32_t hit_capacity, uint32_t depth, nvb_pipeline** out);
int  nvb_pipeline_submit(nvb_pipeline* p, const uint32_t* h_read_words, uint32_t* ticket);
int  nvb_pipeline_wait(nvb_pipeline* p, uint32_t ticket, nvb_pipeline_result* out);
/* bytes moved per batch: host -> device, device -> host */
void nvb_pipeline_traffic(const nvb_pipeline* p, size_t* h2d_bytes, size_t* d2h_bytes);
void nvb_pipeline_destroy(nvb_pipeline* p);

/* Profiling aid (the reference wraps every stage in cuda::Timer, nvBowtie/bowtie2/cuda/aligner_best_approx.h:
 * 219-241): device time in ms of the seven stages of the most recent direct nvb_seed_extend, nvb_seed_extend_traceback
 * or nvb_seed_extend_paired call on the current device -- [fw,rc] strings, seed match (FM-index), hit slots, locate +
 * windows, job de-duplication, banded extension, best-per-read.  nvb_pipeline batches record no stages (see
 * nvb_pipeline_result.device_ms).  Synchronises on the call's last event. */
int nvb_seed_extend_stage_ms(float ms[7]);

#ifdef __cplusplus
}
#endif
#endif /* NVBIO_B200_H */
