// pipeline.cu -- seed + extend composition of the two hot paths (the loop nvbio's examples/fmmap/fmmap.cu:255-400
// and nvBowtie's best_approx run per read batch):
//
//   reads -> [fw, rc] strings -> seeds every `seed_interval` -> FM-index match (SA ranges)
//         -> locate every hit row -> diagonal -> genome window [diag - B/2, + read_len + B)
//         -> banded Gotoh score of the read (or its reverse complement) against the window
//         -> best score per read.
//
// Everything stays on the device between stages; the hit count never visits the host (the extension
// kernels read it from device memory).  Window rule: fmmap.cu:190-208 (genome_infixes); best-per-read
// reduction: fmmap.cu:365-385.
#include "fm_core.cuh"
#include "gotoh_core.cuh"
#include "pipeline_core.cuh"
#include <cub/device/device_scan.cuh>
#include <atomic>
#include <mutex>

namespace nvb {

struct PipeGeom {
    uint32_t n_reads;        // input reads
    uint32_t n_strings;      // n_reads * (both_strands ? 2 : 1)
    uint32_t strands;        // 1 or 2
    uint32_t stride;         // symbols per string slot in the [fw,rc] stream (multiple of 32/bits)
    uint32_t bits;           // symbol width of the [fw,rc] stream (= input width)
    uint32_t seeds_per_string;
    uint32_t seed_len, seed_interval;
    uint32_t band;
    uint32_t max_seed_hits;
    uint32_t genome_len;
    uint32_t hit_capacity;
};

// string s = 2*read + strand (strands==2) or read: copy / reverse-complement into an aligned slot.
// One thread per output word.
template <int BITS>
__global__ void __launch_bounds__(256)
pipe_make_strings_kernel(const StrSet reads, const PipeGeom g, uint32_t* __restrict__ out_words, uint32_t* __restrict__ out_len)
{
    constexpr uint32_t SPW = 32 / BITS;
    const uint32_t words_per_string = g.stride / SPW;
    const uint64_t t = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    if (t >= (uint64_t)g.n_strings * words_per_string) return;
    const uint32_t s = (uint32_t)(t / words_per_string), w = (uint32_t)(t % words_per_string);
    const uint32_t read = s / g.strands, strand = s % g.strands;
    const uint32_t off = str_off(reads, read), len = str_len(reads, read);
    if (w == 0) out_len[s] = len;
    uint32_t word = 0;
    for (uint32_t k = 0; k < SPW; ++k) {
        const uint32_t p = w * SPW + k;
        uint32_t c = 0;
        if (p < len) {
            if (strand == 0) c = sym_at_rt(reads.words, reads.bits, reads.big_endian, off + p);
            else { c = sym_at_rt(reads.words, reads.bits, reads.big_endian, off + (len - 1u - p)); c = (c < 4u) ? 3u - c : c; }
        }
        word |= c << (32u - BITS - BITS * k);              // big-endian packing
    }
    out_words[t] = word;
}

// base qualities of the [fw, rc] strings: byte p of string s at out[s * stride + p] (the rc string's are the read's, reversed)
__global__ void __launch_bounds__(256)
pipe_make_quals_kernel(const StrSet reads, const PipeGeom g, const uint8_t* __restrict__ quals, uint8_t* __restrict__ out)
{
    const uint64_t t = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    if (t >= (uint64_t)g.n_strings * g.stride) return;
    const uint32_t s = (uint32_t)(t / g.stride), p = (uint32_t)(t % g.stride);
    const uint32_t read = s / g.strands, strand = s % g.strands;
    const uint32_t off = str_off(reads, read), len = str_len(reads, read);
    out[t] = (p < len) ? quals[off + (strand == 0 ? p : len - 1u - p)] : (uint8_t)0;
}

// 2-bit fast path of the above: whole words at a time.  16 consecutive symbols starting at any symbol offset are a
// funnel shift of two words; the reverse complement of a word is ~brev(word) with the two bits of every symbol
// swapped back.
__device__ __forceinline__ uint32_t load16_2bit_be(const uint32_t* __restrict__ words, uint32_t p /* symbol offset */, uint32_t cnt /* symbols needed */)
{
    const uint32_t w = p >> 4, sh = 2u * (p & 15u);
    const uint32_t a = words[w];
    if (sh == 0) return a;
    const uint32_t b = ((p & 15u) + cnt > 16u) ? words[w + 1] : 0u;     // never touch a word the string does not reach
    return (a << sh) | (b >> (32u - sh));
}
__device__ __forceinline__ uint32_t revcomp16_2bit(uint32_t x)
{
    uint32_t y = __brev(~x);                                  // symbols reversed, bits inside each symbol swapped
    return ((y >> 1) & 0x55555555u) | ((y & 0x55555555u) << 1);
}
__global__ void __launch_bounds__(256)
pipe_make_strings_2bit_be_kernel(const StrSet reads, const PipeGeom g, uint32_t* __restrict__ out_words, uint32_t* __restrict__ out_len)
{
    const uint32_t words_per_string = g.stride / 16u;
    const uint64_t t = (uint64_t)blockIdx.x * 256 + threadIdx.x, total = (uint64_t)g.n_strings * words_per_string;
    if (t >= total) return;
    // 32-bit index arithmetic whenever the word count allows it (measured: no difference -- the stage's 0.10 ms per million reads are the
    // first touch of the input after the L2 flush between steps and the write-back of that flush, not this kernel's instructions)
    uint32_t s, w;
    if (total <= 0xFFFFFFFFull) { s = (uint32_t)t / words_per_string; w = (uint32_t)t - s * words_per_string; }
    else                        { s = (uint32_t)(t / words_per_string); w = (uint32_t)(t % words_per_string); }
    const uint32_t read = s / g.strands, strand = s % g.strands;
    const uint32_t off = str_off(reads, read), len = str_len(reads, read);
    if (w == 0) out_len[s] = len;
    const uint32_t first = w * 16u;                           // first output symbol of this word
    uint32_t word = 0;
    if (first < len) {
        const uint32_t cnt = (len - first) < 16u ? (len - first) : 16u;
        if (strand == 0) {
            word = load16_2bit_be(reads.words, off + first, cnt);
        } else {
            // output symbols first..first+cnt-1 are the complements of input symbols len-1-first .. len-first-cnt (descending)
            const uint32_t lo = len - first - cnt;            // lowest input symbol needed
            uint32_t x = load16_2bit_be(reads.words, off + lo, cnt);   // symbols lo .. lo+15 (only the first cnt matter)
            x = revcomp16_2bit(x);                             // now symbol (lo+15-j) sits at position j
            word = x << (2u * (16u - cnt));                    // drop the 16-cnt leading junk symbols
        }
        if (cnt < 16u) word &= ~(0xFFFFFFFFu >> (2u * cnt));   // zero the padding
    }
    out_words[t] = word;
}

// one thread per (string, seed slot): SA range of the seed, and its clamped size.
// genome != NULL (the per-read path on an index with the full suffix array): single-row ranges are located on the spot --
// ranges[q] = (text position, 0xFFFFFFFF), see fm_match_locate_one -- so that neither the remaining LF steps nor the later SA
// gather of that hit are needed; wider ranges stay SA ranges.
// (2048 threads per SM = every warp slot: the kernel lives on gathers in flight, so the register budget is 32)
// CTA size: seeds finish after 1 to 6 gathers, and a CTA's warp slots are only handed on when its last warp is done -- small CTAs
// keep more of the 64 slots busy (measured, seed-match stage at C3: 512 threads 1.47 ms, 256 1.40, 128 1.35, 64 1.35)
constexpr uint32_t SEED_BLOCK = 128;
constexpr uint32_t SEED_TODO_LISTS = 64;                     // todo lists (and counters) of the two-pass seed match
constexpr uint32_t SEED_TODO_PITCH = 32;                     // words between two counters: one 128-byte line each
constexpr uint32_t SEED_ITER = 8;                            // seeds per thread in its first pass
// DEFER: a seed whose k-mer occurs three or more times needs ~6 dependent gathers where the others need 1 to 3, and a warp's slot is
// held until its slowest lane is done -- such seeds are only looked up here (ranges[q] = the k-mer's range) and appended to `todo`;
// pipe_seed_match_wide_kernel finishes them, all lanes of its warps equally deep
template <int BITS, bool DEFER>
__global__ void __launch_bounds__(SEED_BLOCK, 2048 / SEED_BLOCK)
pipe_seed_match_kernel(const FmIndex f, const PipeGeom g, const uint32_t* __restrict__ words, const uint32_t* __restrict__ slen,
                       const uint32_t* __restrict__ genome, uint2* __restrict__ ranges, uint32_t* __restrict__ sizes,
                       uint32_t* __restrict__ todo, uint32_t* __restrict__ todo_count)
{
    // DEFER: SEED_ITER consecutive chunks of seeds per CTA (its seeds are done after one or two gathers: fewer, longer-lived CTAs; on its
    // own this measured no difference -- what bounded the first version of this pass was its atomics, see below)
    constexpr uint32_t ITER = DEFER ? SEED_ITER : 1u;
#pragma unroll 1
    for (uint32_t it = 0; it < ITER; ++it) {
        const uint32_t q = (blockIdx.x * ITER + it) * SEED_BLOCK + threadIdx.x;
        const bool live = q < g.n_strings * g.seeds_per_string;
        if (!DEFER && !live) return;
        uint32_t x = 1, y = 0;
        bool deferred = false;
        if (live) {
            const uint32_t s = q / g.seeds_per_string, k = q % g.seeds_per_string;
            const uint32_t len = slen[s];
            const uint32_t pos = k * g.seed_interval;
            if (pos + g.seed_len <= len) {
                if (genome) {
                    const uint32_t st = fm_match_locate_one<BITS, true, DEFER ? FM_DEFER : FM_WHOLE>(f, genome, words, s * g.stride + pos, g.seed_len, x, y);
                    if (st == FM_EMPTY) { x = 1; y = 0; }
                    deferred = DEFER && st == FM_DEFERRED;
                } else
                    fm_match_one<BITS, true>(f, words, s * g.stride + pos, g.seed_len, 0u, x, y);
            }
            ranges[q] = make_uint2(x, y);
            if (!deferred) sizes[q] = seed_range_size(make_uint2(x, y), g.max_seed_hits);
        }
        if (DEFER) {
            // one atomic per warp, spread over SEED_TODO_LISTS counters, each in its own 128-byte line.  Measured (C3, 0.9 M atomics per
            // launch): one counter 2.1 ms for this kernel, 64 counters in adjacent words 1.5 ms, 64 counters one line apart 0.9 ms (= 0.93
            // of the gather ceiling) -- same-line atomics serialise in the L2.  List c takes the CTAs with blockIdx % LISTS == c, so its
            // capacity ceil(gridDim / LISTS) * SEED_BLOCK * SEED_ITER can never overflow
            const uint32_t m = __ballot_sync(0xFFFFFFFFu, deferred);
            if (m) {
                const uint32_t lane = threadIdx.x & 31u, list = blockIdx.x % SEED_TODO_LISTS;
                const uint32_t cap = ((gridDim.x + SEED_TODO_LISTS - 1u) / SEED_TODO_LISTS) * SEED_BLOCK * SEED_ITER;
                uint32_t base = 0;
                if (lane == 0) base = atomicAdd(todo_count + list * SEED_TODO_PITCH, (uint32_t)__popc(m));
                base = __shfl_sync(0xFFFFFFFFu, base, 0);
                if (deferred) todo[(size_t)list * cap + base + __popc(m & ((1u << lane) - 1u))] = q;
            }
        }
    }
}
// the deferred seeds: resume from the k-mer's range.  CTA b works on list b % LISTS (gridDim is a multiple of LISTS), striding over it:
// the lists' lengths live on the device.  seed_grid = gridDim of the first pass (defines the lists' capacity)
template <int BITS>
__global__ void __launch_bounds__(SEED_BLOCK, 2048 / SEED_BLOCK)
pipe_seed_match_wide_kernel(const FmIndex f, const PipeGeom g, const uint32_t* __restrict__ words,
                            const uint32_t* __restrict__ genome, uint2* __restrict__ ranges, uint32_t* __restrict__ sizes,
                            const uint32_t* __restrict__ todo, const uint32_t* __restrict__ todo_count, const uint32_t seed_grid)
{
    const uint32_t list = blockIdx.x % SEED_TODO_LISTS, per_list = gridDim.x / SEED_TODO_LISTS;
    const uint32_t cap = ((seed_grid + SEED_TODO_LISTS - 1u) / SEED_TODO_LISTS) * SEED_BLOCK * SEED_ITER;
    const uint32_t n = todo_count[list * SEED_TODO_PITCH];
    for (uint32_t t = (blockIdx.x / SEED_TODO_LISTS) * SEED_BLOCK + threadIdx.x; t < n; t += per_list * SEED_BLOCK) {
        const uint32_t q = todo[(size_t)list * cap + t];
        const uint32_t s = q / g.seeds_per_string, k = q % g.seeds_per_string;
        const uint2 r = ranges[q];
        uint32_t x = r.x, y = r.y;
        if (fm_match_locate_one<BITS, true, FM_RESUME>(f, genome, words, s * g.stride + k * g.seed_interval, g.seed_len, x, y) == FM_EMPTY) { x = 1; y = 0; }
        ranges[q] = make_uint2(x, y);
        sizes[q] = seed_range_size(make_uint2(x, y), g.max_seed_hits);
    }
}

__device__ __forceinline__ uint32_t upper_bound_u32(const uint32_t* __restrict__ a, uint32_t n, uint32_t v)
{
    uint32_t lo = 0, hi = n;
    while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (a[mid] <= v) lo = mid + 1; else hi = mid; }
    return lo;
}

// counts[0] = min(total, capacity), counts[1] = total
__global__ void pipe_count_kernel(const uint32_t* __restrict__ excl, const uint32_t* __restrict__ sizes, uint32_t n_queries, uint32_t capacity,
                                  uint32_t* __restrict__ counts)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        const uint32_t total = n_queries ? excl[n_queries - 1] + sizes[n_queries - 1] : 0u;
        counts[1] = total;
        counts[0] = total < capacity ? total : capacity;
    }
}

// one thread per QUERY (most seeds have 0 or 1 hits): locate each of its SA rows, derive the genome window and the
// alignment job.  Hit h = excl[q] + j keeps the reference's slot order (filter_inl.h:99-118) without a binary search.
__global__ void __launch_bounds__(256)
pipe_expand_hits_kernel(const FmIndex f, const PipeGeom g, const uint2* __restrict__ ranges, const uint32_t* __restrict__ sizes,
                        const uint32_t* __restrict__ excl, const uint32_t* __restrict__ slen, const uint32_t* __restrict__ counts,
                        uint32_t* __restrict__ hit_string, uint32_t* __restrict__ p_off, uint32_t* __restrict__ p_len,
                        uint32_t* __restrict__ t_off, uint32_t* __restrict__ t_len)
{
    const uint32_t q = blockIdx.x * 256 + threadIdx.x;
    if (q >= g.n_strings * g.seeds_per_string) return;
    const uint32_t sz = sizes[q];
    if (sz == 0) return;
    const uint32_t base = excl[q], kept = counts[0];
    const uint32_t x = ranges[q].x;
    const uint32_t s = q / g.seeds_per_string, k = q % g.seeds_per_string;
    const uint32_t seed_begin = k * g.seed_interval;
    const uint32_t len = slen[s];
    for (uint32_t j = 0; j < sz; ++j) {
        const uint32_t h = base + j;
        if (h >= kept) break;                                                      // beyond the caller's capacity
        const uint2 w = hit_window(fm_locate_one(f, x + j), seed_begin, len, g.band, g.genome_len);
        hit_string[h] = s;
        p_off[h] = s * g.stride; p_len[h] = len;
        t_off[h] = w.x;          t_len[h] = w.y - w.x;
    }
}

// ---------------------------------------------------------------------------------------------
// per-read path (no per-hit outputs requested): one thread per read locates its hits and keeps only the distinct (strand, window)
// alignment jobs -- no per-hit array is written at all.  Jobs are staged per CTA in shared memory and appended to the global
// job list with one atomic per CTA; their order varies from run to run, the results do not (every job carries the index of the
// first hit that produced it, and the best-per-read reduction breaks score ties by it exactly as the per-hit path does).
// ---------------------------------------------------------------------------------------------
constexpr uint32_t RJ_BLOCK = 128;          // reads per CTA
constexpr uint32_t RJ_STAGE = 640;          // staged jobs per CTA (average: ~1.2 per read)
constexpr int      RJ_LOCAL = 6;            // distinct windows remembered per read (more are still scored, just not de-duplicated)

__global__ void __launch_bounds__(RJ_BLOCK)
pipe_read_jobs_kernel(const FmIndex f, const PipeGeom g, const uint2* __restrict__ ranges, const uint32_t* __restrict__ sizes,
                      const uint32_t* __restrict__ excl, const uint32_t* __restrict__ slen, uint32_t* __restrict__ counts,
                      uint32_t* __restrict__ j_string, uint32_t* __restrict__ j_first,
                      uint32_t* __restrict__ jp_off, uint32_t* __restrict__ jp_len, uint32_t* __restrict__ jt_off, uint32_t* __restrict__ jt_len)
{
    __shared__ uint32_t st_string[RJ_STAGE], st_first[RJ_STAGE], st_toff[RJ_STAGE], st_tlen[RJ_STAGE];
    __shared__ uint32_t s_cnt, s_base;
    if (threadIdx.x == 0) s_cnt = 0u;
    __syncthreads();
    const uint32_t r = blockIdx.x * RJ_BLOCK + threadIdx.x;
    const uint32_t kept = counts[0];
    if (r < g.n_reads) {
        uint32_t lk_s[RJ_LOCAL], lk_b[RJ_LOCAL], lk_e[RJ_LOCAL];
        int n_local = 0;
        // hit slots of this read: the scan's value at its first seed plus a running sum of the (clamped) range sizes, which are
        // recomputed from the ranges exactly as the match kernel stored them -- one 8-byte load per seed instead of 16
        uint32_t run = excl[r * g.strands * g.seeds_per_string];
        for (uint32_t strand = 0; strand < g.strands; ++strand) {
            const uint32_t s = r * g.strands + strand;
            const uint32_t len = slen[s];
            for (uint32_t k = 0; k < g.seeds_per_string; ++k) {
                const uint32_t q = s * g.seeds_per_string + k;
                const uint2 rq = ranges[q];
                const uint32_t sz = seed_range_size(rq, g.max_seed_hits);
                if (sz == 0u) continue;
                const bool located = rq.y == 0xFFFFFFFFu;                              // already a text position (fm_match_locate_one)
                const uint32_t base = run, x = rq.x, seed_begin = k * g.seed_interval;
                run += sz;
                for (uint32_t j = 0; j < sz; ++j) {
                    const uint32_t h = base + j;
                    if (h >= kept) break;                                              // beyond the caller's capacity
                    const uint2 w = hit_window(located ? x : fm_locate_one(f, x + j), seed_begin, len, g.band, g.genome_len);
                    const uint32_t gb = w.x, ge = w.y;
                    bool seen = false;
#pragma unroll
                    for (int e = 0; e < RJ_LOCAL; ++e) seen |= (e < n_local) && lk_s[e] == s && lk_b[e] == gb && lk_e[e] == ge;
                    if (seen) continue;
#pragma unroll
                    for (int e = 0; e < RJ_LOCAL; ++e) if (e == n_local) { lk_s[e] = s; lk_b[e] = gb; lk_e[e] = ge; }
                    if (n_local < RJ_LOCAL) ++n_local;
                    const uint32_t slot = atomicAdd(&s_cnt, 1u);
                    if (slot < RJ_STAGE) { st_string[slot] = s; st_first[slot] = h; st_toff[slot] = gb; st_tlen[slot] = ge - gb; }
                    else {                                                             // staging full: straight to the global list
                        const uint32_t o = atomicAdd(counts + 2, 1u);
                        j_string[o] = s; j_first[o] = h; jp_off[o] = s * g.stride; jp_len[o] = len; jt_off[o] = gb; jt_len[o] = ge - gb;
                    }
                }
            }
        }
    }
    __syncthreads();
    const uint32_t n = s_cnt < RJ_STAGE ? s_cnt : RJ_STAGE;
    if (threadIdx.x == 0) s_base = n ? atomicAdd(counts + 2, n) : 0u;
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < n; i += RJ_BLOCK) {
        const uint32_t o = s_base + i, s = st_string[i];
        j_string[o] = s; j_first[o] = st_first[i]; jp_off[o] = s * g.stride; jp_len[o] = slen[s]; jt_off[o] = st_toff[i]; jt_len[o] = st_tlen[i];
    }
}

// Exact shortcut of the LOCAL extension (gapless_job_shortcut, pipeline_core.cuh): jobs whose result it proves get it here; the others
// are compacted into the list the DP kernels run over.  (Earlier versions of the check: all band diagonals for every job 0.39 ms per
// million reads, a symbol-by-symbol segment loop 0.29 ms, per-diagonal text reads 0.22 ms; now 0.14 ms.)
__global__ void __launch_bounds__(256)
pipe_perfect_jobs_kernel(const PipeGeom g, const int32_t match, const int32_t mismatch, const int32_t max_gap_open, const uint32_t* __restrict__ counts,
                         const uint32_t* __restrict__ str_words, const uint32_t* __restrict__ genome,
                         const uint32_t* __restrict__ jp_off, const uint32_t* __restrict__ jp_len,
                         const uint32_t* __restrict__ jt_off, const uint32_t* __restrict__ jt_len,
                         int32_t* __restrict__ job_score, uint2* __restrict__ job_sink,
                         uint32_t* __restrict__ dp_p_off, uint32_t* __restrict__ dp_p_len, uint32_t* __restrict__ dp_t_off, uint32_t* __restrict__ dp_t_len,
                         uint32_t* __restrict__ dp_job, uint32_t* __restrict__ dp_count)
{
    __shared__ uint32_t s_warp[8], s_base;
    const uint32_t n = counts[2];
    for (uint32_t base = blockIdx.x * 256; base < n; base += gridDim.x * 256) {       // (whole CTAs stay in the loop: barriers below)
        const uint32_t j = base + threadIdx.x;
        bool todo = false;
        uint32_t po = 0, M = 0, to = 0, N = 0;
        if (j < n) {
            po = jp_off[j]; M = jp_len[j]; to = jt_off[j]; N = jt_len[j];
            int32_t score = 0; uint32_t sx = 0, sy = 0;
            if (gapless_job_shortcut(str_words, genome, po, M, to, N, g.band, match, mismatch, max_gap_open, score, sx, sy)) {
                job_score[j] = score; job_sink[j] = make_uint2(sx, sy);
            } else todo = true;
        }
        // compaction of the others: one atomic per CTA (same-address atomics serialise, ~2.4 ns each on this part)
        const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
        const uint32_t m = __ballot_sync(0xFFFFFFFFu, todo);
        if (lane == 0) s_warp[warp] = (uint32_t)__popc(m);
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t tot = 0;
            for (int w = 0; w < 8; ++w) { const uint32_t c = s_warp[w]; s_warp[w] = tot; tot += c; }
            s_base = tot ? atomicAdd(dp_count, tot) : 0u;
        }
        __syncthreads();
        if (todo) {
            const uint32_t slot = s_base + s_warp[warp] + __popc(m & ((1u << lane) - 1u));
            dp_p_off[slot] = po; dp_p_len[slot] = M; dp_t_off[slot] = to; dp_t_len[slot] = N; dp_job[slot] = j;
        }
        __syncthreads();                                                           // s_warp / s_base are rewritten by the next round
    }
}
__global__ void __launch_bounds__(256)
pipe_scatter_dp_kernel(const uint32_t* __restrict__ dp_count, const uint32_t* __restrict__ dp_job, const int32_t* __restrict__ dp_score,
                       const uint2* __restrict__ dp_sink, int32_t* __restrict__ job_score, uint2* __restrict__ job_sink)
{
    const uint32_t n = *dp_count;
    for (uint32_t a = blockIdx.x * 256 + threadIdx.x; a < n; a += gridDim.x * 256) {
        const uint32_t j = dp_job[a];
        job_score[j] = dp_score[a]; job_sink[j] = dp_sink[a];
    }
}

// best job per read: max score, ties -> the job whose first hit comes first (the per-hit path's "smallest hit index")
__global__ void __launch_bounds__(256)
pipe_reduce_jobs_kernel(const PipeGeom g, const uint32_t* __restrict__ counts, const uint32_t* __restrict__ j_string, const uint32_t* __restrict__ j_first,
                        const int32_t* __restrict__ job_score, unsigned long long* __restrict__ best_key)
{
    const uint32_t n = counts[2];
    for (uint32_t j = blockIdx.x * 256 + threadIdx.x; j < n; j += gridDim.x * 256)
        atomicMax(best_key + j_string[j] / g.strands, nvb::best_key(job_score[j], j_first[j]));
}

__global__ void __launch_bounds__(256)
pipe_init_best_kernel(const uint32_t n_reads, int32_t* __restrict__ best_score, uint32_t* __restrict__ best_pos, uint8_t* __restrict__ best_strand)
{
    const uint32_t r = blockIdx.x * 256 + threadIdx.x;
    if (r >= n_reads) return;
    best_score[r] = INT_MIN; best_pos[r] = 0xFFFFFFFFu; best_strand[r] = 0;
}

// the winning job of every read writes the read's result (first-hit indices are unique, so exactly one job matches the key)
__global__ void __launch_bounds__(256)
pipe_finalize_jobs_kernel(const PipeGeom g, const uint32_t* __restrict__ counts, const uint32_t* __restrict__ j_string, const uint32_t* __restrict__ j_first,
                          const uint32_t* __restrict__ jt_off, const int32_t* __restrict__ job_score, const uint2* __restrict__ job_sink,
                          const unsigned long long* __restrict__ best_key,
                          int32_t* __restrict__ best_score, uint32_t* __restrict__ best_pos, uint8_t* __restrict__ best_strand)
{
    const uint32_t n = counts[2];
    for (uint32_t j = blockIdx.x * 256 + threadIdx.x; j < n; j += gridDim.x * 256) {
        const uint32_t s = j_string[j], read = s / g.strands;
        if (best_key[read] != nvb::best_key(job_score[j], j_first[j])) continue;
        best_score[read] = job_score[j]; best_pos[read] = hit_end(jt_off[j], job_sink[j].x); best_strand[read] = (uint8_t)(s % g.strands);
    }
}

// Hits of one string are contiguous (queries are ordered by string, then seed).  Several seeds of a read usually
// vote for the same diagonal, i.e. the very same (string, window) alignment job: score it once.
// leader[h] = the smallest h' <= h of the same string with the same window; flag[h] = (leader[h] == h).
// A missed duplicate (beyond the look-back) only costs a redundant alignment, never a different result.
__global__ void __launch_bounds__(256)
pipe_find_leaders_kernel(const uint32_t* __restrict__ counts, const uint32_t* __restrict__ hit_string,
                         const uint32_t* __restrict__ t_off, const uint32_t* __restrict__ t_len,
                         uint32_t* __restrict__ leader, uint32_t* __restrict__ flag)
{
    // the block's 256 hits plus the 64 before them, staged once in shared memory (the look-back re-reads them ~5x on average)
    constexpr uint32_t BACK = 64u;
    __shared__ uint32_t ss[256 + BACK], so[256 + BACK], sl[256 + BACK];
    const uint32_t n = counts[0];
    const uint32_t h0 = blockIdx.x * 256;
    if (h0 >= n) return;
    for (uint32_t i = threadIdx.x; i < 256 + BACK; i += 256) {
        const int64_t g = (int64_t)h0 - BACK + i;
        const bool in = g >= 0 && g < (int64_t)n;
        ss[i] = in ? hit_string[g] : 0xFFFFFFFFu; so[i] = in ? t_off[g] : 0u; sl[i] = in ? t_len[g] : 0u;
    }
    __syncthreads();
    const uint32_t h = h0 + threadIdx.x;
    if (h >= n) return;
    const uint32_t me = threadIdx.x + BACK;
    const uint32_t s = ss[me], o = so[me], l = sl[me];
    uint32_t lead = h;
    for (uint32_t back = 1; back <= BACK && back <= h; ++back) {
        if (ss[me - back] != s) break;
        if (so[me - back] == o && sl[me - back] == l) lead = h - back;
    }
    leader[h] = lead;
    flag[h] = (lead == h) ? 1u : 0u;
}

// counts[2] = number of unique jobs
__global__ void pipe_job_count_kernel(const uint32_t* __restrict__ job_idx, const uint32_t* __restrict__ flag, uint32_t* __restrict__ counts)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        const uint32_t n = counts[0];
        counts[2] = n ? job_idx[n - 1] + flag[n - 1] : 0u;
    }
}

__global__ void __launch_bounds__(256)
pipe_compact_jobs_kernel(const uint32_t* __restrict__ counts, const uint32_t* __restrict__ flag, const uint32_t* __restrict__ job_idx,
                         const uint32_t* __restrict__ p_off, const uint32_t* __restrict__ p_len,
                         const uint32_t* __restrict__ t_off, const uint32_t* __restrict__ t_len,
                         uint32_t* __restrict__ jp_off, uint32_t* __restrict__ jp_len, uint32_t* __restrict__ jt_off, uint32_t* __restrict__ jt_len)
{
    const uint32_t h = blockIdx.x * 256 + threadIdx.x;
    if (h >= counts[0] || !flag[h]) return;
    const uint32_t j = job_idx[h];
    jp_off[j] = p_off[h]; jp_len[j] = p_len[h]; jt_off[j] = t_off[h]; jt_len[j] = t_len[h];
}

// every hit receives its group's (score, sink); the best-per-read reduction (see pipe_reduce_kernel) rides along
__global__ void __launch_bounds__(256)
pipe_scatter_scores_kernel(const PipeGeom g, const uint32_t* __restrict__ counts, const uint32_t* __restrict__ leader, const uint32_t* __restrict__ job_idx,
                           const int32_t* __restrict__ job_score, const uint2* __restrict__ job_sink, const uint32_t* __restrict__ hit_string,
                           int32_t* __restrict__ score, uint2* __restrict__ sink, unsigned long long* __restrict__ best_key)
{
    const uint32_t h = blockIdx.x * 256 + threadIdx.x;
    if (h >= counts[0]) return;
    // leader[h] is the earliest identical job within the look-back of h; it may itself have an earlier one: follow the chain to
    // the hit that really was compacted into the job list (leader[l] == l)
    uint32_t l = leader[h];
    for (uint32_t nx = leader[l]; nx != l; nx = leader[l]) l = nx;
    const uint32_t j = job_idx[l];
    const int32_t sc = job_score[j];
    score[h] = sc;
    sink[h]  = job_sink[j];
    atomicMax(best_key + hit_string[h] / g.strands, nvb::best_key(sc, h));
}

// best hit per read: max score, ties -> smallest hit index (deterministic)
__global__ void __launch_bounds__(256)
pipe_reduce_kernel(const PipeGeom g, const uint32_t* __restrict__ counts, const uint32_t* __restrict__ hit_string,
                   const int32_t* __restrict__ score, unsigned long long* __restrict__ best_key)
{
    const uint32_t h = blockIdx.x * 256 + threadIdx.x;
    if (h >= counts[0]) return;
    atomicMax(best_key + hit_string[h] / g.strands, nvb::best_key(score[h], h));
}

__global__ void __launch_bounds__(256)
pipe_finalize_kernel(const PipeGeom g, const unsigned long long* __restrict__ best_key, const uint32_t* __restrict__ t_off,
                     const uint2* __restrict__ sink, const uint32_t* __restrict__ hit_string,
                     int32_t* __restrict__ best_score, uint32_t* __restrict__ best_pos, uint8_t* __restrict__ best_strand)
{
    const uint32_t r = blockIdx.x * 256 + threadIdx.x;
    if (r >= g.n_reads) return;
    const unsigned long long key = best_key[r];
    if (key == 0ull) { best_score[r] = INT_MIN; best_pos[r] = 0xFFFFFFFFu; if (best_strand) best_strand[r] = 0; return; }
    const uint32_t h = best_key_hit(key);
    best_score[r] = best_key_score(key);
    best_pos[r] = hit_end(t_off[h], sink[h].x);
    if (best_strand) best_strand[r] = (uint8_t)(hit_string[h] % g.strands);
}

// the best hit of every read as an alignment job for the traceback (reads without a hit get an empty job)
__global__ void __launch_bounds__(256)
pipe_best_jobs_kernel(const PipeGeom g, const unsigned long long* __restrict__ best_key, const uint32_t* __restrict__ hit_string,
                      const uint32_t* __restrict__ p_off, const uint32_t* __restrict__ p_len,
                      const uint32_t* __restrict__ t_off, const uint32_t* __restrict__ t_len,
                      uint32_t* __restrict__ bp_off, uint32_t* __restrict__ bp_len, uint32_t* __restrict__ bt_off, uint32_t* __restrict__ bt_len,
                      uint8_t* __restrict__ strand)
{
    const uint32_t r = blockIdx.x * 256 + threadIdx.x;
    if (r >= g.n_reads) return;
    const unsigned long long key = best_key[r];
    if (key == 0ull) { bp_off[r] = 0; bp_len[r] = 0; bt_off[r] = 0; bt_len[r] = 0; if (strand) strand[r] = 0; return; }
    const uint32_t h = best_key_hit(key);
    bp_off[r] = p_off[h]; bp_len[r] = p_len[h]; bt_off[r] = t_off[h]; bt_len[r] = t_len[h];
    if (strand) strand[r] = (uint8_t)(hit_string[h] % g.strands);
}

// source cell (window-relative text start, read start) -> (genome coordinate, read start); reads without a hit: n_ops 0.  A best job
// without an alignment (window shorter than the read) has n_ops 0 and source (0xFFFFFFFF, 0xFFFFFFFF) from the traceback: see hit_end
__global__ void __launch_bounds__(256)
pipe_best_begin_kernel(const PipeGeom g, const unsigned long long* __restrict__ best_key, const uint32_t* __restrict__ bt_off,
                       const uint2* __restrict__ source, uint32_t* __restrict__ n_ops, uint2* __restrict__ begin)
{
    const uint32_t r = blockIdx.x * 256 + threadIdx.x;
    if (r >= g.n_reads) return;
    if (best_key[r] == 0ull) { n_ops[r] = 0; begin[r] = make_uint2(0xFFFFFFFFu, 0xFFFFFFFFu); return; }
    const uint2 sc = source[r];
    begin[r] = make_uint2(hit_end(bt_off[r], sc.x), sc.y);
}

__global__ void __launch_bounds__(256)
pipe_export_hits_kernel(const PipeGeom g, const uint32_t* __restrict__ counts, const uint32_t* __restrict__ hit_string,
                        const uint32_t* __restrict__ t_off, const uint32_t* __restrict__ t_len,
                        uint32_t* __restrict__ out_read, uint2* __restrict__ out_window)
{
    const uint32_t h = blockIdx.x * 256 + threadIdx.x;
    if (h >= counts[0]) return;
    if (out_read)   out_read[h] = hit_string[h];              // string id = read*strands + strand
    if (out_window) out_window[h] = make_uint2(t_off[h], t_off[h] + t_len[h]);
}

// ---------------------------------------------------------------------------------------------
// paired-end stage (see nvb_seed_extend_paired in the header for the rules)
// ---------------------------------------------------------------------------------------------
struct MateBest { bool has; int32_t score; uint32_t strand, beg, end, len; };

// the best alignment of read r as the single-end stages left it: score, end (one past the last aligned base), strand
__device__ __forceinline__ MateBest mate_best(const PipeGeom& g, uint32_t r, const int32_t* best_score,
                                              const uint32_t* best_pos, const uint8_t* __restrict__ best_strand,
                                              const uint32_t* __restrict__ str_len)
{
    MateBest m; m.has = false; m.score = INT_MIN; m.strand = 0; m.beg = m.end = 0xFFFFFFFFu; m.len = 0;
    const uint32_t end = best_pos[r];
    if (end == 0xFFFFFFFFu) return m;
    m.has = true;
    m.score = best_score[r];
    m.strand = best_strand[r];
    m.len = str_len[r * g.strands];                 // both strands of a read have its length
    m.end = end;
    m.beg = m.end > m.len ? m.end - m.len : 0u;
    return m;
}

// one thread per pair: concordance of the independent best alignments, else up to two opposite-mate jobs (slot 2p + anchor)
__global__ void __launch_bounds__(256)
pair_classify_kernel(const PipeGeom g, const uint32_t n_pairs, const nvb_pair_params pp,
                     // best_score / best_pos ARE mate_score / mate_pos in the paired entry point (the single-end stage writes the per-read
                     // bests straight into the mate arrays): no __restrict__ / const on either view
                     const int32_t* best_score, const uint32_t* best_pos, const uint8_t* __restrict__ best_strand,
                     const uint32_t* __restrict__ str_len,
                     uint32_t* __restrict__ want, uint32_t* __restrict__ w_pstr, uint32_t* __restrict__ w_toff, uint32_t* __restrict__ w_tlen,
                     int32_t* __restrict__ pair_score, uint32_t* __restrict__ pair_flags,
                     int32_t* mate_score, uint32_t* mate_pos, uint8_t* __restrict__ mate_strand)
{
    const uint32_t p = blockIdx.x * 256 + threadIdx.x;
    if (p >= n_pairs) return;
    MateBest m[2];
    m[0] = mate_best(g, p, best_score, best_pos, best_strand, str_len);
    m[1] = mate_best(g, n_pairs + p, best_score, best_pos, best_strand, str_len);
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        mate_score[k * n_pairs + p] = m[k].score; mate_pos[k * n_pairs + p] = m[k].end; mate_strand[k * n_pairs + p] = (uint8_t)m[k].strand;
    }
    bool conc = m[0].has && m[1].has && (m[0].strand != m[1].strand);
    if (conc) {
        const MateBest& f = m[0].strand == 0 ? m[0] : m[1];
        const MateBest& r = m[0].strand == 0 ? m[1] : m[0];
        conc = f.beg <= r.beg && f.end <= r.end && r.end > f.beg && (r.end - f.beg) >= pp.min_frag && (r.end - f.beg) <= pp.max_frag;
    }
    if (conc) {
        pair_score[p] = m[0].score + m[1].score; pair_flags[p] = NVB_PAIR_CONCORDANT;
        want[2 * p] = want[2 * p + 1] = 0u;
        return;
    }
    pair_score[p] = INT_MIN; pair_flags[p] = NVB_PAIR_UNPAIRED;
#pragma unroll
    for (int a = 0; a < 2; ++a) {                               // a = anchor mate, 1 - a = the mate to place
        uint32_t w = 0u, ps = 0u, to = 0u, tl = 0u;
        if (m[a].has && m[a].score >= pp.min_mate_score) {
            const uint32_t o_read = (uint32_t)(1 - a) * n_pairs + p;
            if (m[a].strand == 0u) { to = m[a].beg; const uint32_t e = (g.genome_len - to) < pp.max_frag ? g.genome_len : to + pp.max_frag; tl = e - to; ps = 2u * o_read + 1u; }
            else                   { to = m[a].end > pp.max_frag ? m[a].end - pp.max_frag : 0u; tl = m[a].end - to; ps = 2u * o_read; }
            w = (tl >= 1u && str_len[ps] >= 1u) ? 1u : 0u;
        }
        want[2 * p + a] = w; w_pstr[2 * p + a] = ps; w_toff[2 * p + a] = to; w_tlen[2 * p + a] = tl;
    }
}

// counts[0] = jobs run (<= capacity), counts[1] = jobs wanted
__global__ void pair_job_count_kernel(const uint32_t* __restrict__ job_idx, const uint32_t* __restrict__ want, uint32_t n_slots, uint32_t capacity,
                                      uint32_t* __restrict__ counts)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        const uint32_t total = n_slots ? job_idx[n_slots - 1] + want[n_slots - 1] : 0u;
        counts[0] = total < capacity ? total : capacity; counts[1] = total;
    }
}

__global__ void __launch_bounds__(256)
pair_compact_kernel(const PipeGeom g, const uint32_t n_slots, const uint32_t capacity, const uint32_t* __restrict__ want, const uint32_t* __restrict__ job_idx,
                    const uint32_t* __restrict__ w_pstr, const uint32_t* __restrict__ w_toff, const uint32_t* __restrict__ w_tlen,
                    const uint32_t* __restrict__ str_len,
                    uint32_t* __restrict__ jp_off, uint32_t* __restrict__ jp_len, uint32_t* __restrict__ jt_off, uint32_t* __restrict__ jt_len)
{
    const uint32_t i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n_slots || !want[i]) return;
    const uint32_t j = job_idx[i];
    if (j >= capacity) return;
    jp_off[j] = w_pstr[i] * g.stride; jp_len[j] = str_len[w_pstr[i]]; jt_off[j] = w_toff[i]; jt_len[j] = w_tlen[i];
}

__global__ void __launch_bounds__(256)
pair_finalize_kernel(const uint32_t n_pairs, const nvb_pair_params pp, const uint32_t* __restrict__ want, const uint32_t* __restrict__ job_idx,
                     const uint32_t* __restrict__ w_toff, const int32_t* __restrict__ rs_score, const uint2* __restrict__ rs_sink,
                     int32_t* __restrict__ pair_score, uint32_t* __restrict__ pair_flags,
                     int32_t* __restrict__ mate_score, uint32_t* __restrict__ mate_pos, uint8_t* __restrict__ mate_strand)
{
    const uint32_t p = blockIdx.x * 256 + threadIdx.x;
    if (p >= n_pairs || pair_flags[p] == NVB_PAIR_CONCORDANT) return;
    int best_a = -1; int32_t best_sum = INT_MIN, best_rs = 0; uint32_t best_pos = 0;
#pragma unroll
    for (int a = 0; a < 2; ++a) {
        const uint32_t i = 2 * p + a;
        if (!want[i]) continue;
        const uint32_t j = job_idx[i];
        if (j >= pp.rescue_capacity) continue;
        const int32_t rs = rs_score[j];
        if (rs < pp.min_mate_score) continue;
        const int32_t sum = mate_score[a * n_pairs + p] + rs;
        if (sum > best_sum) { best_sum = sum; best_a = a; best_rs = rs; best_pos = w_toff[i] + rs_sink[j].x; }
    }
    if (best_a < 0) return;
    const int o = 1 - best_a;
    pair_score[p] = best_sum;
    pair_flags[p] = o == 0 ? NVB_PAIR_RESCUED_MATE1 : NVB_PAIR_RESCUED_MATE2;
    mate_score[o * n_pairs + p] = best_rs;
    mate_pos[o * n_pairs + p] = best_pos;
    mate_strand[o * n_pairs + p] = (uint8_t)(1u - mate_strand[best_a * n_pairs + p]);
}

} // namespace nvb

using namespace nvb;

#define PIPE_TRY(expr) do { const int _r = (expr); if (_r != NVB_OK) return _r; } while (0)
#define PIPE_SIZE_QUERY(expr) do { const int _r = (expr); if (_r != NVB_E_TEMP_SIZE && _r != NVB_OK) return _r; } while (0)
#define NVB_STAGE(i) do { if (c.ev) NVB_CUDA_TRY(cudaEventRecord(c.ev[i], c.s)); } while (0)

// stage boundaries of the most recent direct nvb_seed_extend* call ON EACH DEVICE (events are recorded on the caller's stream; they
// cost no synchronisation).  [0]=start, then after: strings, seed match, slots, locate+windows, job dedup, extension, reduce.
// Events belong to the device that created them, so the set is per device, created under a mutex on first use; a host that drives
// several GPUs from one process (one compute thread per device) gets one set per GPU.  nvb_pipeline's batches record none.
struct StageEvents { cudaEvent_t ev[8]; bool ready; std::atomic<bool> valid; };
static StageEvents g_stage[NVB_MAX_DEVICES];
static std::mutex  g_stage_mutex;
static int default_stage_events(StageEvents** out)
{
    int dev = 0;
    NVB_CUDA_TRY(cudaGetDevice(&dev));
    if (dev < 0 || dev >= NVB_MAX_DEVICES) return NVB_E_UNSUPPORTED;
    std::lock_guard<std::mutex> lock(g_stage_mutex);
    StageEvents& S = g_stage[dev];
    if (!S.ready) {
        for (int i = 0; i < 8; ++i) NVB_CUDA_TRY(cudaEventCreate(&S.ev[i]));
        S.ready = true;
    }
    *out = &S;
    return NVB_OK;
}

extern "C" int nvb_seed_extend_stage_ms(float ms[7])
{
    if (!ms) return NVB_E_INVALID;
    StageEvents* SE = nullptr;
    PIPE_TRY(default_stage_events(&SE));
    if (!SE->valid.load(std::memory_order_acquire)) return NVB_E_INVALID;
    NVB_CUDA_TRY(cudaEventSynchronize(SE->ev[7]));
    for (int i = 0; i < 7; ++i) NVB_CUDA_TRY(cudaEventElapsedTime(&ms[i], SE->ev[i], SE->ev[i + 1]));
    return NVB_OK;
}

// test / tuning switches (include/nvbio_b200_debug.h); a call reads each of them once
static std::atomic<int> g_perfect_shortcut{1};     // 0 = every alignment job through the DP kernels
static std::atomic<int> g_seed_split{1};           // 0 = the located seed match in one pass
static std::atomic<int> g_pipe_path{0};            // 0 = automatic, 1 = always the per-hit path
extern "C" void nvb_debug_pipeline_path(int path) { g_pipe_path.store(path, std::memory_order_relaxed); }
extern "C" void nvb_debug_seed_split(int on) { g_seed_split.store(on, std::memory_order_relaxed); }
extern "C" void nvb_debug_perfect_shortcut(int on) { g_perfect_shortcut.store(on, std::memory_order_relaxed); }

// grids of kernels striding over a job count that lives on the device: resident CTAs of the 148 SMs, not hit_capacity / 256 mostly empty ones
constexpr uint32_t SHORTCUT_GRID_CAP = 148u * 8u;
constexpr uint32_t REDUCE_GRID_CAP   = 148u * 16u;

// an alignment job list: pattern = symbols [p_off, + p_len) of the [fw,rc] strings, text = genome [t_off, + t_len)
struct JobList { uint32_t *p_off, *p_len, *t_off, *t_len; };
static JobList take_jobs(TempCarver& tc, size_t n) { return JobList{tc.take<uint32_t>(n), tc.take<uint32_t>(n), tc.take<uint32_t>(n), tc.take<uint32_t>(n)}; }

// the path of one call, decided once
struct PipePlan {
    bool dedup;        // identical (string, window) jobs of a read are scored once
    bool per_read;     // no per-hit output wanted: distinct jobs straight from a thread per read, no per-hit array at all
    bool eligible;     // the per-read jobs qualify for the gapless shortcut (its arrays are carved)
    bool shortcut;     // ... and take it
    bool locate;       // the seed match locates single-row ranges (per-read path on an index with the full suffix array)
    bool split;        // ... in two passes (a k-mer table shorter than the seed)
};

// the temp arrays of one call, in carve order; those of a path the call does not take stay null
struct PipeTemp {
    uint32_t *str_words, *str_len; uint8_t* str_quals; uint2* ranges; uint32_t *sizes, *excl, *counts, *seed_todo_n;   // counts: hits kept, found, unique jobs
    uint32_t *j_string, *j_first, *leader, *flag, *job_idx;            // per-read path: string, first hit of every job; per-hit de-duplication
    JobList jobs; int32_t* job_score; uint2* job_sink;                  // the unique jobs (de-duplication)
    JobList dp; uint32_t* dp_job; int32_t* dp_score; uint2* dp_sink; uint32_t* dp_count;    // jobs the gapless shortcut leaves to the DP
    uint32_t* hit_string; JobList hits; int32_t* h_score; uint2* h_sink;    // per-hit path
    unsigned long long* best_key; uint8_t* rb_strand; char *scan_tmp, *gotoh_tmp; size_t scan_bytes, gotoh_bytes;
    JobList best; int32_t* b_score; uint2 *b_sink, *b_source; char* tb_tmp; size_t tb_bytes;    // best-alignment traceback
    uint32_t *pw_want, *pw_idx, *pw_pstr, *pw_toff, *pw_tlen, *pcounts;                         // paired-end rescue
    JobList rescue; int32_t* rs_score; uint2* rs_sink; char *pscan_tmp, *full_tmp; size_t pscan_bytes, full_bytes;
};

struct PipeCall {
    const nvb_seed_extend_params* P; PipeGeom g; uint32_t nq, spw, hit_capacity; FmIndex f; StrSet rd; const uint32_t* genome;
    nvb_string_set pats, txts;          // job-list views: formats and maximum lengths (their pointers are placeholders, see job_views)
    PipePlan plan; PipeTemp t;
    cudaStream_t s; cudaEvent_t* ev;                    // ev: stage events to record, or null
};

static void job_views(const PipeCall& c, const JobList& j, nvb_string_set& pats, nvb_string_set& txts)
{
    pats = c.pats; pats.d_words = c.t.str_words; pats.d_offsets = j.p_off; pats.d_lengths = j.p_len;
    txts = c.txts; txts.d_words = c.genome;      txts.d_offsets = j.t_off; txts.d_lengths = j.t_len;
}

// the banded extension of a job list whose length lives on the device
static int score_jobs(const PipeCall& c, const JobList& j, const uint32_t* d_n_jobs, int32_t* score, uint2* sink)
{
    nvb_string_set pats, txts;
    job_views(c, j, pats, txts);
    size_t gb = c.t.gotoh_bytes;
    return nvb_banded_gotoh_score_indirect(c.P->band_len, c.P->type, &c.P->scheme, &pats, c.t.str_quals, &txts, d_n_jobs, c.hit_capacity,
                                           score, (nvb_uint2*)sink, c.t.gotoh_tmp, &gb, c.s);
}

// carves the temp arrays (the layout behind *temp_bytes) and queries the temp the library calls of the stages need
static int carve_temp(PipeCall& c, TempCarver& tc, int32_t* d_hit_score, nvb_uint2* d_hit_sink,
                      const nvb_best_alignment_out* BA, const nvb_pair_params* PP)
{
    const nvb_seed_extend_params* P = c.P;
    const PipeGeom& g = c.g; const PipePlan& pl = c.plan; PipeTemp& t = c.t;
    const uint32_t cap = c.hit_capacity, n_reads = g.n_reads;
    PIPE_SIZE_QUERY(nvb_banded_gotoh_score(P->band_len, P->type, &P->scheme, &c.pats, nullptr, &c.txts, cap, (int32_t*)16, (nvb_uint2*)16, nullptr,
                                           &t.gotoh_bytes, c.s));
    t.str_words = tc.take<uint32_t>((size_t)g.n_strings * (g.stride / c.spw) + 4);
    t.str_len   = tc.take<uint32_t>(g.n_strings);
    t.str_quals = P->d_read_quals ? tc.take<uint8_t>((size_t)g.n_strings * g.stride + 16) : nullptr;
    t.ranges    = tc.take<uint2>(c.nq);
    t.sizes     = tc.take<uint32_t>(c.nq);
    t.excl      = tc.take<uint32_t>((size_t)c.nq + (SEED_TODO_LISTS + 1u) * SEED_BLOCK * SEED_ITER);   // (+ slack: before the scan it holds the seed-match todo lists)
    t.counts    = tc.take<uint32_t>(4);
    t.seed_todo_n = tc.take<uint32_t>(SEED_TODO_LISTS * SEED_TODO_PITCH);
    if (pl.per_read) { t.j_string = tc.take<uint32_t>(cap); t.j_first = tc.take<uint32_t>(cap); }
    if (pl.dedup && !pl.per_read) { t.leader = tc.take<uint32_t>(cap); t.flag = tc.take<uint32_t>(cap); t.job_idx = tc.take<uint32_t>(cap); }
    if (pl.dedup) { t.jobs = take_jobs(tc, cap); t.job_score = tc.take<int32_t>(cap); t.job_sink = tc.take<uint2>(cap); }
    if (pl.eligible) {
        t.dp = take_jobs(tc, cap); t.dp_job = tc.take<uint32_t>(cap); t.dp_score = tc.take<int32_t>(cap); t.dp_sink = tc.take<uint2>(cap); t.dp_count = tc.take<uint32_t>(4);
    }
    if (!pl.per_read) {
        t.hit_string = tc.take<uint32_t>(cap); t.hits = take_jobs(tc, cap);
        t.h_score = d_hit_score ? d_hit_score : tc.take<int32_t>(cap); t.h_sink = d_hit_sink ? (uint2*)d_hit_sink : tc.take<uint2>(cap);
    }
    t.best_key = tc.take<unsigned long long>(n_reads); t.rb_strand = tc.take<uint8_t>((size_t)n_reads + 16);
    NVB_CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, t.scan_bytes, t.sizes, t.excl, (int)c.nq, c.s));
    if (pl.dedup && !pl.per_read && cap) {
        size_t scan2_bytes = 0;
        NVB_CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, scan2_bytes, t.flag, t.job_idx, (int)cap, c.s));
        if (scan2_bytes > t.scan_bytes) t.scan_bytes = scan2_bytes;
    }
    t.scan_tmp = tc.take<char>(t.scan_bytes); t.gotoh_tmp = tc.take<char>(t.gotoh_bytes);
    if (BA) {               // best-alignment traceback: per-read job arrays + the traceback's own temp (direction matrices)
        t.best = take_jobs(tc, n_reads);
        t.b_score = tc.take<int32_t>(n_reads); t.b_sink = tc.take<uint2>(n_reads); t.b_source = tc.take<uint2>(n_reads);
        PIPE_SIZE_QUERY(nvb_banded_gotoh_traceback(P->band_len, P->type, &P->scheme, &c.pats, nullptr, &c.txts, n_reads, nullptr, nullptr, nullptr, nullptr,
                                                   BA->max_ops, nullptr, nullptr, &t.tb_bytes, c.s));
        t.tb_tmp = tc.take<char>(t.tb_bytes);
    }
    if (PP) {               // paired-end stage: job slots (2 per pair), compacted full-DP jobs and the DP's own temp
        const uint32_t pcap = PP->rescue_capacity;
        t.pw_want = tc.take<uint32_t>(n_reads); t.pw_idx = tc.take<uint32_t>(n_reads); t.pw_pstr = tc.take<uint32_t>(n_reads);
        t.pw_toff = tc.take<uint32_t>(n_reads); t.pw_tlen = tc.take<uint32_t>(n_reads); t.pcounts = tc.take<uint32_t>(4);
        t.rescue = take_jobs(tc, pcap); t.rs_score = tc.take<int32_t>(pcap); t.rs_sink = tc.take<uint2>(pcap);
        NVB_CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, t.pscan_bytes, t.pw_want, t.pw_idx, (int)n_reads, c.s));
        t.pscan_tmp = tc.take<char>(t.pscan_bytes);
        nvb_string_set rtxts = c.txts; rtxts.length = PP->max_frag;
        PIPE_SIZE_QUERY(nvb_gotoh_score_indirect(P->type, &P->scheme, &c.pats, nullptr, &rtxts, (const uint32_t*)16, pcap, (int32_t*)16, (nvb_uint2*)16,
                                                 nullptr, &t.full_bytes, c.s));
        t.full_tmp = tc.take<char>(t.full_bytes);
    }
    return NVB_OK;
}

// 1. [fw, rc] strings (and their base qualities)
static int run_strings(const PipeCall& c)
{
    const PipeGeom& g = c.g; const PipeTemp& t = c.t;
    const uint64_t total_words = (uint64_t)g.n_strings * (g.stride / c.spw);
    const uint32_t grid = (uint32_t)((total_words + 255) / 256);
    if (g.bits == 2 && c.rd.big_endian) pipe_make_strings_2bit_be_kernel<<<grid, 256, 0, c.s>>>(c.rd, g, t.str_words, t.str_len);
    else if (g.bits == 2)               pipe_make_strings_kernel<2><<<grid, 256, 0, c.s>>>(c.rd, g, t.str_words, t.str_len);
    else                                pipe_make_strings_kernel<4><<<grid, 256, 0, c.s>>>(c.rd, g, t.str_words, t.str_len);
    NVB_LAUNCH_CHECK();
    if (t.str_quals) {
        const uint64_t total = (uint64_t)g.n_strings * g.stride;
        pipe_make_quals_kernel<<<(uint32_t)((total + 255) / 256), 256, 0, c.s>>>(c.rd, g, c.P->d_read_quals, t.str_quals);
        NVB_LAUNCH_CHECK();
    }
    return NVB_OK;
}

// 2. seed ranges
static int run_seed_match(const PipeCall& c)
{
    const PipeGeom& g = c.g; const PipeTemp& t = c.t;
    const uint32_t grid = (c.nq + SEED_BLOCK - 1) / SEED_BLOCK;
    const uint32_t* loc_genome = c.plan.locate ? c.genome : nullptr;
    if (c.plan.split) {
        // seeds on k-mers with >= 3 occurrences are finished by a second kernel (the lists live in `excl`, which the hit-slot scan overwrites)
        NVB_CUDA_TRY(cudaMemsetAsync(t.seed_todo_n, 0, SEED_TODO_LISTS * SEED_TODO_PITCH * sizeof(uint32_t), c.s));
        const uint32_t grid1 = (grid + SEED_ITER - 1u) / SEED_ITER;
        if (g.bits == 2) pipe_seed_match_kernel<2, true><<<grid1, SEED_BLOCK, 0, c.s>>>(c.f, g, t.str_words, t.str_len, loc_genome, t.ranges, t.sizes, t.excl, t.seed_todo_n);
        else             pipe_seed_match_kernel<4, true><<<grid1, SEED_BLOCK, 0, c.s>>>(c.f, g, t.str_words, t.str_len, loc_genome, t.ranges, t.sizes, t.excl, t.seed_todo_n);
        NVB_LAUNCH_CHECK();
        const uint32_t wgrid = SEED_TODO_LISTS * 37u;                                  // 2368 CTAs = 148 SMs x 16 resident CTAs
        if (g.bits == 2) pipe_seed_match_wide_kernel<2><<<wgrid, SEED_BLOCK, 0, c.s>>>(c.f, g, t.str_words, loc_genome, t.ranges, t.sizes, t.excl, t.seed_todo_n, grid1);
        else             pipe_seed_match_wide_kernel<4><<<wgrid, SEED_BLOCK, 0, c.s>>>(c.f, g, t.str_words, loc_genome, t.ranges, t.sizes, t.excl, t.seed_todo_n, grid1);
    } else {
        if (g.bits == 2) pipe_seed_match_kernel<2, false><<<grid, SEED_BLOCK, 0, c.s>>>(c.f, g, t.str_words, t.str_len, loc_genome, t.ranges, t.sizes, nullptr, nullptr);
        else             pipe_seed_match_kernel<4, false><<<grid, SEED_BLOCK, 0, c.s>>>(c.f, g, t.str_words, t.str_len, loc_genome, t.ranges, t.sizes, nullptr, nullptr);
    }
    NVB_LAUNCH_CHECK();
    return NVB_OK;
}

// 3. hit slots
static int run_hit_slots(const PipeCall& c)
{
    size_t sb = c.t.scan_bytes; NVB_CUDA_TRY(cub::DeviceScan::ExclusiveSum(c.t.scan_tmp, sb, c.t.sizes, c.t.excl, (int)c.nq, c.s));
    pipe_count_kernel<<<1, 32, 0, c.s>>>(c.t.excl, c.t.sizes, c.nq, c.hit_capacity, c.t.counts);
    NVB_LAUNCH_CHECK();
    return NVB_OK;
}

// 4'. per read: locate, window, distinct jobs; 5'. extension; 6'. best job per read
static int run_per_read(const PipeCall& c, int32_t* d_best_score, uint32_t* d_best_pos)
{
    const PipeGeom& g = c.g; const PipeTemp& t = c.t;
    const uint32_t cap = c.hit_capacity, hgrid = (cap + 255) / 256;
    NVB_CUDA_TRY(cudaMemsetAsync(t.counts + 2, 0, sizeof(uint32_t), c.s));
    NVB_CUDA_TRY(cudaMemsetAsync(t.best_key, 0, sizeof(unsigned long long) * g.n_reads, c.s));
    if (cap) {
        pipe_read_jobs_kernel<<<(g.n_reads + RJ_BLOCK - 1) / RJ_BLOCK, RJ_BLOCK, 0, c.s>>>(c.f, g, t.ranges, t.sizes, t.excl, t.str_len, t.counts, t.j_string,
                                                                                         t.j_first, t.jobs.p_off, t.jobs.p_len, t.jobs.t_off, t.jobs.t_len);
        NVB_LAUNCH_CHECK();
    }
    NVB_STAGE(4); NVB_STAGE(5);                         // (the jobs come out distinct: no de-duplication stage)
    if (cap && c.plan.shortcut) {
        const uint32_t jgrid = hgrid < SHORTCUT_GRID_CAP ? hgrid : SHORTCUT_GRID_CAP;
        const nvb_gotoh_scheme& SC = c.P->scheme;
        NVB_CUDA_TRY(cudaMemsetAsync(t.dp_count, 0, sizeof(uint32_t), c.s));
        pipe_perfect_jobs_kernel<<<jgrid, 256, 0, c.s>>>(g, SC.match, SC.mismatch, SC.pattern_gap_open > SC.text_gap_open ? SC.pattern_gap_open : SC.text_gap_open,
                                                         t.counts, t.str_words, c.genome, t.jobs.p_off, t.jobs.p_len, t.jobs.t_off, t.jobs.t_len,
                                                         t.job_score, t.job_sink, t.dp.p_off, t.dp.p_len, t.dp.t_off, t.dp.t_len, t.dp_job, t.dp_count);
        NVB_LAUNCH_CHECK();
        PIPE_TRY(score_jobs(c, t.dp, t.dp_count, t.dp_score, t.dp_sink));
        pipe_scatter_dp_kernel<<<jgrid, 256, 0, c.s>>>(t.dp_count, t.dp_job, t.dp_score, t.dp_sink, t.job_score, t.job_sink);
        NVB_LAUNCH_CHECK();
    } else if (cap) PIPE_TRY(score_jobs(c, t.jobs, t.counts + 2, t.job_score, t.job_sink));
    NVB_STAGE(6);
    pipe_init_best_kernel<<<(g.n_reads + 255) / 256, 256, 0, c.s>>>(g.n_reads, d_best_score, d_best_pos, t.rb_strand);
    NVB_LAUNCH_CHECK();
    if (cap) {
        const uint32_t jgrid = hgrid < REDUCE_GRID_CAP ? hgrid : REDUCE_GRID_CAP;
        pipe_reduce_jobs_kernel<<<jgrid, 256, 0, c.s>>>(g, t.counts, t.j_string, t.j_first, t.job_score, t.best_key);
        NVB_LAUNCH_CHECK();
        pipe_finalize_jobs_kernel<<<jgrid, 256, 0, c.s>>>(g, t.counts, t.j_string, t.j_first, t.jobs.t_off, t.job_score, t.job_sink, t.best_key,
                                                          d_best_score, d_best_pos, t.rb_strand);
        NVB_LAUNCH_CHECK();
    }
    return NVB_OK;
}

// 4. locate + windows per hit; 4b. collapse identical (string, window) jobs; 5. extension; 6. best hit per read; the hit arrays
static int run_per_hit(const PipeCall& c, int32_t* d_best_score, uint32_t* d_best_pos, uint32_t* d_hit_read, nvb_uint2* d_hit_window)
{
    const PipeGeom& g = c.g; const PipeTemp& t = c.t;
    const uint32_t cap = c.hit_capacity, hgrid = (cap + 255) / 256;
    const bool dedup = c.plan.dedup;
    if (cap) {
        pipe_expand_hits_kernel<<<(c.nq + 255) / 256, 256, 0, c.s>>>(c.f, g, t.ranges, t.sizes, t.excl, t.str_len, t.counts, t.hit_string, t.hits.p_off, t.hits.p_len,
                                                                     t.hits.t_off, t.hits.t_len);
        NVB_LAUNCH_CHECK();
    }
    NVB_STAGE(4);
    if (dedup && cap) {
        pipe_find_leaders_kernel<<<hgrid, 256, 0, c.s>>>(t.counts, t.hit_string, t.hits.t_off, t.hits.t_len, t.leader, t.flag);
        NVB_LAUNCH_CHECK();
        // the scan runs over the whole capacity; job_idx[h] depends only on flag[0..h), so the (unwritten) entries
        // past counts[0] cannot influence any index that is read back
        size_t sb = t.scan_bytes; NVB_CUDA_TRY(cub::DeviceScan::ExclusiveSum(t.scan_tmp, sb, t.flag, t.job_idx, (int)cap, c.s));
        pipe_job_count_kernel<<<1, 32, 0, c.s>>>(t.job_idx, t.flag, t.counts);
        NVB_LAUNCH_CHECK();
        pipe_compact_jobs_kernel<<<hgrid, 256, 0, c.s>>>(t.counts, t.flag, t.job_idx, t.hits.p_off, t.hits.p_len, t.hits.t_off, t.hits.t_len,
                                                         t.jobs.p_off, t.jobs.p_len, t.jobs.t_off, t.jobs.t_len);
        NVB_LAUNCH_CHECK();
    }
    NVB_STAGE(5);
    NVB_CUDA_TRY(cudaMemsetAsync(t.best_key, 0, sizeof(unsigned long long) * g.n_reads, c.s));
    if (cap && dedup) {
        PIPE_TRY(score_jobs(c, t.jobs, t.counts + 2, t.job_score, t.job_sink));
        pipe_scatter_scores_kernel<<<hgrid, 256, 0, c.s>>>(g, t.counts, t.leader, t.job_idx, t.job_score, t.job_sink, t.hit_string, t.h_score, t.h_sink, t.best_key);
        NVB_LAUNCH_CHECK();
    } else if (cap) PIPE_TRY(score_jobs(c, t.hits, t.counts, t.h_score, t.h_sink));
    NVB_STAGE(6);
    if (cap && !dedup) {                                // (with job de-duplication the scatter kernel did the reduction)
        pipe_reduce_kernel<<<hgrid, 256, 0, c.s>>>(g, t.counts, t.hit_string, t.h_score, t.best_key);
        NVB_LAUNCH_CHECK();
    }
    pipe_finalize_kernel<<<(g.n_reads + 255) / 256, 256, 0, c.s>>>(g, t.best_key, t.hits.t_off, t.h_sink, t.hit_string, d_best_score, d_best_pos, t.rb_strand);
    NVB_LAUNCH_CHECK();
    if (cap && (d_hit_read || d_hit_window)) {
        pipe_export_hits_kernel<<<hgrid, 256, 0, c.s>>>(g, t.counts, t.hit_string, t.hits.t_off, t.hits.t_len, d_hit_read, (uint2*)d_hit_window);
        NVB_LAUNCH_CHECK();
    }
    return NVB_OK;
}

// the alignment (ops, begin, strand) of every read's best hit (per-hit path)
static int run_traceback(const PipeCall& c, const nvb_best_alignment_out* BA)
{
    const PipeGeom& g = c.g; const PipeTemp& t = c.t;
    const uint32_t rgrid = (g.n_reads + 255) / 256;
    pipe_best_jobs_kernel<<<rgrid, 256, 0, c.s>>>(g, t.best_key, t.hit_string, t.hits.p_off, t.hits.p_len, t.hits.t_off, t.hits.t_len,
                                                  t.best.p_off, t.best.p_len, t.best.t_off, t.best.t_len, BA->d_strand);
    NVB_LAUNCH_CHECK();
    nvb_string_set pats, txts;
    job_views(c, t.best, pats, txts);
    size_t tbb = t.tb_bytes;
    PIPE_TRY(nvb_banded_gotoh_traceback(c.P->band_len, c.P->type, &c.P->scheme, &pats, t.str_quals, &txts, g.n_reads, t.b_score, (nvb_uint2*)t.b_sink,
                                        (nvb_uint2*)t.b_source, BA->d_ops, BA->max_ops, BA->d_n_ops, t.tb_tmp, &tbb, c.s));
    pipe_best_begin_kernel<<<rgrid, 256, 0, c.s>>>(g, t.best_key, t.best.t_off, t.b_source, BA->d_n_ops, (uint2*)BA->d_begin);
    NVB_LAUNCH_CHECK();
    return NVB_OK;
}

// paired-end stage: concordance of the mates' best alignments, full-DP rescue of the opposite mate for the others
static int run_paired(const PipeCall& c, const nvb_pair_params* PP, const nvb_pair_out* PO, int32_t* d_best_score, uint32_t* d_best_pos)
{
    const PipeGeom& g = c.g; const PipeTemp& t = c.t;
    const uint32_t n_reads = g.n_reads, n_pairs = n_reads / 2u, cap = PP->rescue_capacity;
    const uint32_t pgrid = (n_pairs + 255) / 256, sgrid = (n_reads + 255) / 256;
    pair_classify_kernel<<<pgrid, 256, 0, c.s>>>(g, n_pairs, *PP, d_best_score, d_best_pos, t.rb_strand, t.str_len, t.pw_want, t.pw_pstr, t.pw_toff, t.pw_tlen,
                                                 PO->d_pair_score, PO->d_pair_flags, PO->d_mate_score, PO->d_mate_pos, PO->d_mate_strand);
    NVB_LAUNCH_CHECK();
    size_t sb = t.pscan_bytes; NVB_CUDA_TRY(cub::DeviceScan::ExclusiveSum(t.pscan_tmp, sb, t.pw_want, t.pw_idx, (int)n_reads, c.s));
    pair_job_count_kernel<<<1, 32, 0, c.s>>>(t.pw_idx, t.pw_want, n_reads, cap, t.pcounts);
    NVB_LAUNCH_CHECK();
    if (cap) {
        pair_compact_kernel<<<sgrid, 256, 0, c.s>>>(g, n_reads, cap, t.pw_want, t.pw_idx, t.pw_pstr, t.pw_toff, t.pw_tlen, t.str_len,
                                                    t.rescue.p_off, t.rescue.p_len, t.rescue.t_off, t.rescue.t_len);
        NVB_LAUNCH_CHECK();
        nvb_string_set pats, txts;
        job_views(c, t.rescue, pats, txts);
        txts.length = PP->max_frag; size_t fb = t.full_bytes;
        PIPE_TRY(nvb_gotoh_score_indirect(c.P->type, &c.P->scheme, &pats, t.str_quals, &txts, t.pcounts, cap, t.rs_score, (nvb_uint2*)t.rs_sink,
                                          t.full_tmp, &fb, c.s));
    }
    pair_finalize_kernel<<<pgrid, 256, 0, c.s>>>(n_pairs, *PP, t.pw_want, t.pw_idx, t.pw_toff, t.rs_score, t.rs_sink, PO->d_pair_score, PO->d_pair_flags,
                                                 PO->d_mate_score, PO->d_mate_pos, PO->d_mate_strand);
    NVB_LAUNCH_CHECK();
    if (PO->d_n_rescue) NVB_CUDA_TRY(cudaMemcpyAsync(PO->d_n_rescue, t.pcounts, 2 * sizeof(uint32_t), cudaMemcpyDeviceToDevice, c.s));
    return NVB_OK;
}

int nvb::seed_extend_impl(const nvb_fm_index* fmi, const uint32_t* d_genome, const nvb_string_set* reads, uint32_t n_reads,
                          const nvb_seed_extend_params* P, uint32_t hit_capacity, int32_t* d_best_score, uint32_t* d_best_pos,
                          uint32_t* d_n_hits, uint32_t* d_hit_read, nvb_uint2* d_hit_window, int32_t* d_hit_score, nvb_uint2* d_hit_sink,
                          const nvb_best_alignment_out* BA, const nvb_pair_params* PP, const nvb_pair_out* PO,
                          void* d_temp, size_t* temp_bytes, void* stream, bool record_stages)
{
    if (PP) {
        if (!PO || !PO->d_pair_score || !PO->d_pair_flags || !PO->d_mate_score || !PO->d_mate_pos || !PO->d_mate_strand) return NVB_E_INVALID;
        if (!P || !P->both_strands || (n_reads & 1u) || PP->max_frag == 0 || PP->min_frag > PP->max_frag) return NVB_E_INVALID;
    }
    if (BA && (!BA->d_ops || !BA->d_n_ops || !BA->d_begin || BA->max_ops == 0)) return NVB_E_INVALID;
    if (!valid_fmindex(fmi) || !fmi->d_ssa || !d_genome || !valid_strset(reads) || !P || !temp_bytes) return NVB_E_INVALID;
    if (reads->bits == 8) return NVB_E_UNSUPPORTED;
    if (P->seed_len == 0 || P->seed_interval == 0 || P->max_seed_hits == 0) return NVB_E_INVALID;
    if (n_reads && (!d_best_score || !d_best_pos)) return NVB_E_INVALID;
    const uint32_t max_len = reads->length;                 // maximum read length (== length for fixed-length sets)
    if (max_len < P->seed_len) return NVB_E_INVALID;

    PipeCall c{};
    PipeGeom& g = c.g;
    g.n_reads = n_reads; g.strands = P->both_strands ? 2u : 1u; g.n_strings = n_reads * g.strands;
    g.bits = reads->bits; c.spw = 32u / g.bits;
    g.stride = (max_len + c.spw - 1u) / c.spw * c.spw;
    g.seeds_per_string = (max_len - P->seed_len) / P->seed_interval + 1u;
    g.seed_len = P->seed_len; g.seed_interval = P->seed_interval; g.band = P->band_len;
    g.max_seed_hits = P->max_seed_hits; g.genome_len = fmi->length; g.hit_capacity = hit_capacity;
    if ((uint64_t)g.n_strings * g.stride > 0xFFFFFFFFull) return NVB_E_UNSUPPORTED;
    const uint64_t nq64 = (uint64_t)g.n_strings * g.seeds_per_string;
    if (nq64 > 0x7FFFFFFFull) return NVB_E_UNSUPPORTED;
    // hit slots are a uint32 exclusive sum of the clamped range sizes: the worst case must fit
    if (nq64 * (uint64_t)P->max_seed_hits > 0xFFFFFFFFull) return NVB_E_UNSUPPORTED;
    c.nq = (uint32_t)nq64; c.P = P; c.hit_capacity = hit_capacity; c.f = make_fmindex(fmi); c.rd = make_strset(reads); c.genome = d_genome;
    c.s = as_stream(stream);
    c.pats = nvb_string_set{(const uint32_t*)16, g.bits, 1, nullptr, nullptr, 0, max_len};      // (placeholder words for the size queries)
    c.txts = nvb_string_set{d_genome, 2, 1, nullptr, nullptr, 0, max_len + P->band_len};
    // the path, decided once
    PipePlan& p = c.plan;
    p.dedup = P->dedup_jobs != 0;
    p.per_read = p.dedup && g_pipe_path.load(std::memory_order_relaxed) != 1 && !(d_hit_read || d_hit_window || d_hit_score || d_hit_sink || BA);
    // exact shortcut for reads that equal their window (pipe_perfect_jobs_kernel): the DP then runs over a compacted job list
    p.eligible = p.per_read && shortcut_eligible(P->type, g.bits, P->band_len, P->scheme);
    p.shortcut = p.eligible && g_perfect_shortcut.load(std::memory_order_relaxed);     // (the switch does not change the temp layout)
    p.locate = p.per_read && c.f.sa_shift == 0u;
    p.split = p.locate && c.f.ktab_k && g.seed_len > c.f.ktab_k && g_seed_split.load(std::memory_order_relaxed);
    TempCarver tc(d_temp);
    PIPE_TRY(carve_temp(c, tc, d_hit_score, d_hit_sink, BA, PP));
    const size_t need = tc.total();
    if (!d_temp || *temp_bytes < need) { *temp_bytes = need; return NVB_E_TEMP_SIZE; }
    if (n_reads == 0) return NVB_OK;
    StageEvents* SE = nullptr;
    if (record_stages) PIPE_TRY(default_stage_events(&SE));
    c.ev = SE ? SE->ev : nullptr;
    NVB_STAGE(0); PIPE_TRY(run_strings(c));
    NVB_STAGE(1); PIPE_TRY(run_seed_match(c));
    NVB_STAGE(2); PIPE_TRY(run_hit_slots(c));
    NVB_STAGE(3);
    if (c.plan.per_read) PIPE_TRY(run_per_read(c, d_best_score, d_best_pos));
    else                 PIPE_TRY(run_per_hit(c, d_best_score, d_best_pos, d_hit_read, d_hit_window));
    if (BA) PIPE_TRY(run_traceback(c, BA));
    if (PP) PIPE_TRY(run_paired(c, PP, PO, d_best_score, d_best_pos));
    if (!c.plan.dedup) NVB_CUDA_TRY(cudaMemcpyAsync(c.t.counts + 2, c.t.counts, sizeof(uint32_t), cudaMemcpyDeviceToDevice, c.s));
    if (d_n_hits) NVB_CUDA_TRY(cudaMemcpyAsync(d_n_hits, c.t.counts, 3 * sizeof(uint32_t), cudaMemcpyDeviceToDevice, c.s));
    NVB_STAGE(7);
    if (SE) SE->valid.store(true, std::memory_order_release);
    return NVB_OK;
}

extern "C" int nvb_seed_extend(const nvb_fm_index* fmi, const uint32_t* d_genome, const nvb_string_set* reads, uint32_t n_reads,
                    const nvb_seed_extend_params* P, uint32_t hit_capacity, int32_t* d_best_score, uint32_t* d_best_pos,
                    uint32_t* d_n_hits, uint32_t* d_hit_read, nvb_uint2* d_hit_window, int32_t* d_hit_score, nvb_uint2* d_hit_sink,
                    void* d_temp, size_t* temp_bytes, void* stream)
{
    return seed_extend_impl(fmi, d_genome, reads, n_reads, P, hit_capacity, d_best_score, d_best_pos, d_n_hits, d_hit_read, d_hit_window,
                            d_hit_score, d_hit_sink, nullptr, nullptr, nullptr, d_temp, temp_bytes, stream, true);
}

extern "C" int nvb_seed_extend_traceback(const nvb_fm_index* fmi, const uint32_t* d_genome, const nvb_string_set* reads, uint32_t n_reads,
                    const nvb_seed_extend_params* P, uint32_t hit_capacity, int32_t* d_best_score, uint32_t* d_best_pos,
                    uint32_t* d_n_hits, uint32_t* d_hit_read, nvb_uint2* d_hit_window, int32_t* d_hit_score, nvb_uint2* d_hit_sink,
                    const nvb_best_alignment_out* best_alignment, void* d_temp, size_t* temp_bytes, void* stream)
{
    if (!best_alignment) return NVB_E_INVALID;
    return seed_extend_impl(fmi, d_genome, reads, n_reads, P, hit_capacity, d_best_score, d_best_pos, d_n_hits, d_hit_read, d_hit_window,
                            d_hit_score, d_hit_sink, best_alignment, nullptr, nullptr, d_temp, temp_bytes, stream, true);
}

extern "C" int nvb_seed_extend_paired(const nvb_fm_index* fmi, const uint32_t* d_genome, const nvb_string_set* reads, uint32_t n_pairs,
                    const nvb_seed_extend_params* P, uint32_t hit_capacity, const nvb_pair_params* pair_params, const nvb_pair_out* out,
                    uint32_t* d_n_hits, void* d_temp, size_t* temp_bytes, void* stream)
{
    if (!pair_params || !out || n_pairs > 0x3FFFFFFFu || !temp_bytes) return NVB_E_INVALID;
    // the per-read best (score, end) of the single-end stage lands in the mate arrays first and is then refined per pair
    return seed_extend_impl(fmi, d_genome, reads, 2u * n_pairs, P, hit_capacity, out->d_mate_score, out->d_mate_pos, d_n_hits, nullptr, nullptr,
                            nullptr, nullptr, nullptr, pair_params, out, d_temp, temp_bytes, stream, true);
}
