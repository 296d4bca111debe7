// pipeline_core.cuh -- per-thread routines of the seed + extend composition that tests also run on the host
// (tests/host/host_harness.cu), like fm_core.cuh / gotoh_core.cuh, and the composition's entry point.
#pragma once
#include "fm_core.cuh"

namespace nvb {

__host__ __device__ __forceinline__ uint32_t nvb_clz(uint32_t x) {        // x != 0
#ifdef __CUDA_ARCH__
    return (uint32_t)__clz((int)x);
#else
    return (uint32_t)__builtin_clz(x);
#endif
}

// Hits of a seed as its hit slots count them: a range the seed match already located (y == 0xFFFFFFFF: x is the text position, see
// fm_match_locate_one) is one hit, an empty range (x > y) none, a row range its rows, clamped to max_seed_hits.
__host__ __device__ __forceinline__ uint32_t seed_range_size(const uint2 range, const uint32_t max_seed_hits)
{
    const uint32_t sz = (range.y == 0xFFFFFFFFu) ? 1u : ((range.x <= range.y) ? (range.y - range.x + 1u) : 0u);
    return sz < max_seed_hits ? sz : max_seed_hits;
}

// Genome window (begin, end) of a hit at text position `pos` of the seed at read offset `seed_begin` (fmmap.cu:190-208, genome_infixes):
// the read's diagonal diag = pos - seed_begin (0 when the seed lies nearer the text start), then [diag - band/2, + len + band),
// clamped to the text [0, genome_len).
__host__ __device__ __forceinline__ uint2 hit_window(const uint32_t pos, const uint32_t seed_begin, const uint32_t len, const uint32_t band,
                                                     const uint32_t genome_len)
{
    const uint32_t diag = pos > seed_begin ? pos - seed_begin : 0u;
    const uint32_t gb = diag > band / 2u ? diag - band / 2u : 0u;
    const uint64_t ge = (uint64_t)gb + len + band;
    return make_uint2(gb, ge < genome_len ? (uint32_t)ge : genome_len);
}

// Genome coordinate of an alignment's end (or, with a traceback's source cell, its begin): window begin + sink.x.  A job whose window is
// shorter than its read (a read running past the genome's end) has no alignment: the DP leaves its sink at the default 0xFFFFFFFF (score
// NVB_SINK_MIN), and the coordinate is 0xFFFFFFFF ("no position") instead of the wrapped sum window_begin - 1.
__host__ __device__ __forceinline__ uint32_t hit_end(const uint32_t window_begin, const uint32_t sink_x)
{
    return sink_x == 0xFFFFFFFFu ? 0xFFFFFFFFu : window_begin + sink_x;
}

// Key of the best-per-read reduction (an atomicMax over the keys of a read's hits): the higher score wins, among equal scores the
// smaller hit index.  The score's sign bit is flipped so that negative scores sort below positive ones; the hit index is stored as
// 0xFFFFFFFF - hit.  Key 0 means "no hit": it would take score INT_MIN at hit 0xFFFFFFFF, beyond every hit capacity.
__host__ __device__ __forceinline__ unsigned long long best_key(const int32_t score, const uint32_t hit)
{
    return ((unsigned long long)((uint32_t)score ^ 0x80000000u) << 32) | (unsigned long long)(0xFFFFFFFFu - hit);
}
__host__ __device__ __forceinline__ int32_t best_key_score(const unsigned long long key) { return (int32_t)((uint32_t)(key >> 32) ^ 0x80000000u); }
__host__ __device__ __forceinline__ uint32_t best_key_hit(const unsigned long long key) { return 0xFFFFFFFFu - (uint32_t)(key & 0xFFFFFFFFull); }

// one bit per differing symbol (bit 2k = symbol cnt-1-k) of read[i, i+cnt) against text[t+i, ...); both 2-bit big-endian streams
__host__ __device__ __forceinline__ uint32_t job_diff_bits(const uint32_t* __restrict__ str_words, const uint32_t* __restrict__ genome,
                                                           const uint32_t po, const uint32_t t, const uint32_t i, const uint32_t cnt)
{
    const uint32_t x = (be2_window(str_words, po + i, cnt) ^ be2_window(genome, t + i, cnt)) >> (32u - 2u * cnt);
    return (x | (x >> 1)) & 0x55555555u;
}
// number of differing symbols on the diagonal starting at text position t; counting stops once it exceeds `limit`
__host__ __device__ __forceinline__ uint32_t job_differences(const uint32_t* __restrict__ str_words, const uint32_t* __restrict__ genome,
                                                             const uint32_t po, const uint32_t M, const uint32_t t, const uint32_t limit)
{
    uint32_t mm = 0;
    for (uint32_t i = 0; i < M && mm <= limit; i += 16u) mm += nvb_popc(job_diff_bits(str_words, genome, po, t, i, M - i < 16u ? M - i : 16u));
    return mm;
}

// Exact shortcut of the LOCAL banded extension for a read that lies on its seed's diagonal with (almost) no difference -- most reads of
// a real run.  With match > 0 > mismatch, gap-open penalties < 0 and gap-extension penalties <= 0:
//   * an alignment that contains a gap scores at most  G = match * M + max(pattern_gap_open, text_gap_open)  (at most M matched
//     columns, and a gap costs at least its first base);
//   * an alignment without a gap lies on ONE band diagonal, and the best of those is the maximum-sum segment of that diagonal's
//     match / mismatch scores (H along the diagonal with only the diagonal move: h = max(0, h + s)).
// So if the best segment of the seed's own diagonal scores MORE than G, and no other band diagonal can reach it (match * its number
// of equal positions stays below), that score is the band's maximum and every cell holding it lies on this diagonal: the DP's result
// is (best, last row where h == best) -- BestSink keeps the last maximal cell in row-major order (sink_inl.h:39-65).  A read without
// any difference (score match * M, only reachable in the last row) may tie with other equal diagonals (tandem repeats): the largest
// one wins.
// The job: read = 2-bit big-endian symbols [po, po + M) of str_words (po a multiple of 16), window = text[to, to + N), the seed's
// diagonal band/2 into the window (pipe_read_jobs_kernel cuts it there; a window clamped at the text start, to == 0, has it somewhere
// below and is left to the DP), band <= 32.  Returns true and (score, sink = (text end, pattern end), both 1-based ends as BestSink
// reports them) when the result is proven; false = run the DP.  Only full windows qualify (N >= M + band - 1: no pad symbol in the band);
// a job outside the conditions above (band > 32, po not a multiple of 16) is left to the DP too.  The scheme's conditions are
// shortcut_eligible's.
__host__ __device__ inline bool gapless_job_shortcut(const uint32_t* __restrict__ str_words, const uint32_t* __restrict__ genome,
                                                     const uint32_t po, const uint32_t M, const uint32_t to, const uint32_t N, const uint32_t band,
                                                     const int32_t match, const int32_t mismatch, const int32_t max_gap_open,
                                                     int32_t& score, uint32_t& sink_x, uint32_t& sink_y)
{
    if (band > 32u || (po & 15u) || M < 1u || to == 0u || N < M + band - 1u) return false;
    const uint32_t j0 = band / 2u;
    // differences a gapless alignment may have and still beat every gapped one: match * (M - mm) > match * M + max_gap_open
    const uint32_t mm_max = (uint32_t)((-max_gap_open + match - 1) / match) - 1u;
    // one pass over the seed's diagonal: its differences (at most mm_max, else the DP) and, from the runs of equal symbols between them,
    // the maximum-sum segment with the LAST end among equals.  (mismatch < 0, so h peaks at the ends of runs; a symbol-by-symbol version
    // of this loop cost 1,500 warp instructions per job)
    int32_t h = 0, best = 0; uint32_t end = 0, prev = 0, mm0 = 0;
    for (uint32_t i = 0; i < M && mm0 <= mm_max; i += 16u) {
        const uint32_t cnt = M - i < 16u ? M - i : 16u;
        uint32_t d = job_diff_bits(str_words, genome, po, to + j0, i, cnt);
        while (d && mm0 <= mm_max) {
            const uint32_t bit = 31u - nvb_clz(d);                          // highest set bit = first differing symbol of the word
            const uint32_t p = i + (cnt - 1u - (bit >> 1));
            d &= ~(1u << bit);
            h += match * (int32_t)(p - prev);
            if (h >= best) { best = h; end = p; }
            h += mismatch; h = h > 0 ? h : 0;
            prev = p + 1u; ++mm0;
        }
    }
    if (mm0 > mm_max) return false;
    h += match * (int32_t)(M - prev);
    if (h >= best) { best = h; end = M; }
    if (best <= match * (int32_t)M + max_gap_open) return false;
    // Can another band diagonal reach `best`?  Only with at most t differences (match * equal positions bounds its score).  The first 16
    // symbols decide that for nearly every diagonal: they are compared against all band offsets from four text words held in registers
    // (a full comparison only follows for a diagonal they do not rule out).
    const bool perfect = (mm0 == 0u);
    const uint32_t t = (uint32_t)((match * (int32_t)M - best) / match);
    const uint32_t c16 = M < 16u ? M : 16u;
    const uint32_t r0 = be2_window(str_words, po, c16) >> (32u - 2u * c16);
    const uint32_t wi = to >> 4, r = to & 15u, wl = (to + N - 1u) >> 4;      // wl: last word holding a window symbol
    const uint32_t g0 = genome[wi], g1 = (wi + 1u <= wl) ? genome[wi + 1u] : 0u;
    const uint32_t g2 = (wi + 2u <= wl) ? genome[wi + 2u] : 0u, g3 = (wi + 3u <= wl) ? genome[wi + 3u] : 0u;
    uint32_t jtop = j0;                                                     // largest diagonal without a difference
    for (uint32_t jj = 0; jj < band; ++jj) {
        if (jj == j0) continue;
        const uint32_t off = r + jj, idx = off >> 4, sh = 2u * (off & 15u);  // band <= 32: idx <= 2
        const uint32_t hi = idx == 0u ? g0 : (idx == 1u ? g1 : g2), lo = idx == 0u ? g1 : (idx == 1u ? g2 : g3);
        const uint32_t win = sh ? ((hi << sh) | (lo >> (32u - sh))) : hi;
        const uint32_t x = (win >> (32u - 2u * c16)) ^ r0;
        if (nvb_popc((x | (x >> 1)) & 0x55555555u) > t) continue;
        if (job_differences(str_words, genome, po, M, to + jj, t) > t) continue;
        if (!perfect) return false;                                         // another diagonal might tie: the DP decides
        if (jj > jtop) jtop = jj;                                           // (another diagonal without a difference)
    }
    score = best;
    if (perfect) { sink_x = M + jtop; sink_y = M; }
    else         { sink_x = end + j0; sink_y = end; }
    return true;
}

// Whether a seed + extend call may take gapless_job_shortcut: a LOCAL extension of 2-bit reads in a band of at most 32 diagonals, with a
// constant scheme of match > 0 > mismatch, gap-open penalties < 0 and gap-extension penalties <= 0.
__host__ __device__ __forceinline__ bool shortcut_eligible(const uint32_t type, const uint32_t bits, const uint32_t band, const nvb_gotoh_scheme& sc)
{
    return type == NVB_LOCAL && bits == 2u && band <= 32u && !sc.d_qual_table && sc.match > 0 && sc.mismatch < 0 &&
           sc.pattern_gap_open < 0 && sc.pattern_gap_ext <= 0 && sc.text_gap_open < 0 && sc.text_gap_ext <= 0;
}

// The composition behind nvb_seed_extend, nvb_seed_extend_traceback and nvb_seed_extend_paired (pipeline.cu; BA / PP + PO select the
// traceback / paired-end stages).  record_stages: record the stage events nvb_seed_extend_stage_ms reports -- the public entry points
// do, nvb_pipeline's batches (host_pipeline.cu) do not.
int seed_extend_impl(const nvb_fm_index* fmi, const uint32_t* d_genome, const nvb_string_set* reads, uint32_t n_reads,
                     const nvb_seed_extend_params* P, uint32_t hit_capacity, int32_t* d_best_score, uint32_t* d_best_pos,
                     uint32_t* d_n_hits, uint32_t* d_hit_read, nvb_uint2* d_hit_window, int32_t* d_hit_score, nvb_uint2* d_hit_sink,
                     const nvb_best_alignment_out* BA, const nvb_pair_params* PP, const nvb_pair_out* PO,
                     void* d_temp, size_t* temp_bytes, void* stream, bool record_stages);

} // namespace nvb
