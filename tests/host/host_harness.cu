// tests/host/host_harness.cu -- TEST INFRASTRUCTURE.
// Runs the product's per-thread __host__ __device__ routines (fm_core.cuh, gotoh_core.cuh) serially on the
// CPU so that their logic can be checked against the oracle in the GPU-less dev container.  The kernels
// proper (thread mapping, shared-memory staging, todo lists) are covered by the -m gpu tests.
#include "../../nvbio_b200/csrc/fm_core.cuh"
#include "../../nvbio_b200/csrc/gotoh_core.cuh"
#include "../../nvbio_b200/csrc/gotoh_full_core.cuh"
#include "../../nvbio_b200/csrc/pipeline_core.cuh"
#include <vector>

using namespace nvb;

static FmIndex mk(const uint32_t* bwt_occ, const uint32_t* ssa, const uint32_t* L2, uint32_t n, uint32_t primary,
                  uint32_t sa_interval = 16, const uint32_t* ktab = nullptr, uint32_t ktab_k = 0, uint32_t ktab_located = 0) {
    nvb_fm_index c; c.d_bwt_occ = bwt_occ; c.d_ssa = ssa; c.length = n; c.primary = primary;
    for (int i = 0; i < 5; ++i) c.L2[i] = L2[i];
    c.sa_interval = sa_interval; c.d_ktab = (const nvb_uint2*)ktab; c.ktab_k = ktab_k; c.ktab_located = ktab_located;
    return make_fmindex(&c);
}

extern "C" {

void hh_fm_rank(const uint32_t* bwt_occ, const uint32_t* L2, uint32_t n, uint32_t primary,
                const uint32_t* k, const uint8_t* c, uint32_t nq, uint32_t* out) {
    const FmIndex f = mk(bwt_occ, nullptr, L2, n, primary);
    for (uint32_t i = 0; i < nq; ++i) out[i] = fm_rank1(f, k[i], c[i] & 3u);
}

// mirrors fm_ktab_level_kernel level by level
void hh_fm_build_ktab(const uint32_t* bwt_occ, const uint32_t* L2, uint32_t n, uint32_t primary, uint32_t k, uint32_t* ktab) {
    const FmIndex f = mk(bwt_occ, nullptr, L2, n, primary);
    uint2* tab = (uint2*)ktab;
    tab[0] = make_uint2(0u, n);
    uint32_t prev = 1;
    for (uint32_t t = 1; t <= k; ++t, prev *= 4u)
        for (uint32_t v = 0; v < prev; ++v) {
            const uint2 r = tab[v];
            for (int c = 3; c >= 0; --c) {
                uint32_t x = r.x, y = r.y;
                if (x <= y) fm_step(f, (uint32_t)c, x, y);
                tab[(uint32_t)c * prev + v] = make_uint2(x, y);
            }
        }
}

// 8-byte entries {x, y} -> 16-byte entries {x, y, SA[x], SA[y]} (SA values for one- and two-row ranges: what nvb_fm_build_ktab_located produces)
void hh_fm_ktab_locate(const uint32_t* ktab8, const uint32_t* full_sa, uint32_t k, uint32_t* ktab16) {
    for (uint64_t v = 0; v < (1ull << (2u * k)); ++v) {
        const uint32_t x = ktab8[2 * v], y = ktab8[2 * v + 1];
        ktab16[4 * v] = x; ktab16[4 * v + 1] = y;
        ktab16[4 * v + 2] = (x == y || y == x + 1u) ? full_sa[x] : 0u; ktab16[4 * v + 3] = (y == x + 1u) ? full_sa[y] : 0u;
    }
}

// ... + the text context (what nvb_fm_build_ktab_context adds): one-row entries .w = the up to 16 symbols before SA[x]; two-row entries
// (n < 0xC0000000) .y = marker | the 7 symbols before SA[x] | those before SA[x+1] << 14
static uint32_t hh_text_before(const uint32_t* text_words, uint32_t pos, uint32_t want) {
    const uint32_t cnt = (pos == 0xFFFFFFFFu) ? 0u : (pos < want ? pos : want);
    return cnt ? (be2_window(text_words, pos - cnt, cnt) >> (32u - 2u * cnt)) : 0u;
}
void hh_fm_ktab_context(uint32_t* ktab16, uint32_t k, const uint32_t* text_words, uint32_t n) {
    for (uint64_t v = 0; v < (1ull << (2u * k)); ++v) {
        const uint32_t x = ktab16[4 * v], y = ktab16[4 * v + 1];
        if (x == y) ktab16[4 * v + 3] = hh_text_before(text_words, ktab16[4 * v + 2], 16u);
        else if (y == x + 1u && n < KTAB_TWO_ROW_MARK)
            ktab16[4 * v + 1] = KTAB_TWO_ROW_MARK | hh_text_before(text_words, ktab16[4 * v + 2], 7u) | (hh_text_before(text_words, ktab16[4 * v + 3], 7u) << 14);
    }
}

void hh_fm_match(const uint32_t* bwt_occ, const uint32_t* L2, uint32_t n, uint32_t primary,
                 const uint32_t* words, uint32_t bits, uint32_t be, const uint32_t* off, const uint32_t* len, uint32_t nq,
                 uint32_t flags, uint32_t* out_xy, const uint32_t* ktab, uint32_t ktab_k, uint32_t ktab_located) {
    const FmIndex f = mk(bwt_occ, nullptr, L2, n, primary, 16, ktab, ktab_k, ktab_located);
    for (uint32_t i = 0; i < nq; ++i) {
        uint32_t x, y;
#define CALL(B, E) fm_match_one<B, E>(f, words, off[i], len[i], flags, x, y)
        NVB_DISPATCH_STREAM(bits, be, CALL);
#undef CALL
        out_xy[2 * i] = x; out_xy[2 * i + 1] = y;
    }
}

void hh_fm_match_approx(const uint32_t* bwt_occ, const uint32_t* L2, uint32_t n, uint32_t primary,
                        const uint32_t* words, uint32_t bits, uint32_t be, const uint32_t* off, const uint32_t* len, uint32_t nq,
                        uint32_t flags, uint32_t exact_len, int find_exact, uint32_t max_out, uint32_t* out_xy, uint32_t* counts, uint32_t* sums) {
    const FmIndex f = mk(bwt_occ, nullptr, L2, n, primary);
    for (uint32_t i = 0; i < nq; ++i) {
        uint32_t sum = 0, cnt = 0;
#define CALL(B, E) cnt = fm_map_approx_one<B, E>(f, words, off[i], len[i], exact_len, flags, find_exact != 0, (uint2*)out_xy + (size_t)i * max_out, max_out, sum)
        NVB_DISPATCH_STREAM(bits, be, CALL);
#undef CALL
        counts[i] = cnt; sums[i] = sum;
    }
}

// fm_match_locate_one over an index with the full suffix array: out[3*i] = status (0 empty, 1 range, 2 located), then (x, y)
void hh_fm_match_locate(const uint32_t* bwt_occ, const uint32_t* full_sa, const uint32_t* L2, uint32_t n, uint32_t primary,
                        const uint32_t* genome, const uint32_t* words, uint32_t bits, uint32_t be, const uint32_t* off, const uint32_t* len,
                        uint32_t nq, uint32_t* out, const uint32_t* ktab, uint32_t ktab_k, uint32_t ktab_located) {
    const FmIndex f = mk(bwt_occ, full_sa, L2, n, primary, 1, ktab, ktab_k, ktab_located);
    for (uint32_t i = 0; i < nq; ++i) {
        uint32_t x = 0, y = 0, st = 0;
        if (bits == 2) st = fm_match_locate_one<2, true>(f, genome, words, off[i], len[i], x, y);
        else           st = fm_match_locate_one<4, true>(f, genome, words, off[i], len[i], x, y);
        (void)be;
        out[3 * i] = st; out[3 * i + 1] = x; out[3 * i + 2] = y;
    }
}

// the same through the two-pass form the seed-match stage uses: FM_DEFER first, FM_RESUME for the seeds it hands back; returns their number
uint32_t hh_fm_match_locate_split(const uint32_t* bwt_occ, const uint32_t* full_sa, const uint32_t* L2, uint32_t n, uint32_t primary,
                                  const uint32_t* genome, const uint32_t* words, uint32_t bits, const uint32_t* off, const uint32_t* len,
                                  uint32_t nq, uint32_t* out, const uint32_t* ktab, uint32_t ktab_k, uint32_t ktab_located) {
    const FmIndex f = mk(bwt_occ, full_sa, L2, n, primary, 1, ktab, ktab_k, ktab_located);
    uint32_t deferred = 0;
    for (uint32_t i = 0; i < nq; ++i) {
        uint32_t x = 0, y = 0, st = 0;
        if (bits == 2) st = fm_match_locate_one<2, true, FM_DEFER>(f, genome, words, off[i], len[i], x, y);
        else           st = fm_match_locate_one<4, true, FM_DEFER>(f, genome, words, off[i], len[i], x, y);
        if (st == FM_DEFERRED) {
            ++deferred;
            if (bits == 2) st = fm_match_locate_one<2, true, FM_RESUME>(f, genome, words, off[i], len[i], x, y);
            else           st = fm_match_locate_one<4, true, FM_RESUME>(f, genome, words, off[i], len[i], x, y);
            if (st == FM_EMPTY) x = y = 0;                  // (x, y) are only defined for the other two states
        }
        out[3 * i] = st; out[3 * i + 1] = x; out[3 * i + 2] = y;
    }
    return deferred;
}

// gapless_job_shortcut over n jobs: solved[a] = 1 and (score[a], sink_xy[2a..]) when the routine proves the LOCAL band result
void hh_gapless_job_shortcut(const uint32_t* str_words, const uint32_t* genome_words, const uint32_t* po, const uint32_t* M, const uint32_t* to,
                             const uint32_t* N, uint32_t n, uint32_t band, int32_t match, int32_t mismatch, int32_t max_gap_open,
                             uint8_t* solved, int32_t* score, uint32_t* sink_xy) {
    for (uint32_t a = 0; a < n; ++a) {
        int32_t sc = 0; uint32_t sx = 0, sy = 0;
        solved[a] = gapless_job_shortcut(str_words, genome_words, po[a], M[a], to[a], N[a], band, match, mismatch, max_gap_open, sc, sx, sy) ? 1 : 0;
        score[a] = sc; sink_xy[2 * a] = sx; sink_xy[2 * a + 1] = sy;
    }
}

// the per-hit rules of the seed + extend composition over n inputs
void hh_hit_window(const uint32_t* pos, const uint32_t* seed_begin, const uint32_t* len, const uint32_t* band, const uint32_t* genome_len,
                   uint32_t n, uint32_t* window) {
    for (uint32_t a = 0; a < n; ++a) {
        const uint2 w = hit_window(pos[a], seed_begin[a], len[a], band[a], genome_len[a]);
        window[2 * a] = w.x; window[2 * a + 1] = w.y;
    }
}
void hh_hit_end(const uint32_t* window_begin, const uint32_t* sink_x, uint32_t n, uint32_t* end) {
    for (uint32_t a = 0; a < n; ++a) end[a] = hit_end(window_begin[a], sink_x[a]);
}
void hh_best_key(const int32_t* score, const uint32_t* hit, uint32_t n, unsigned long long* key, int32_t* key_score, uint32_t* key_hit) {
    for (uint32_t a = 0; a < n; ++a) {
        key[a] = best_key(score[a], hit[a]); key_score[a] = best_key_score(key[a]); key_hit[a] = best_key_hit(key[a]);
    }
}
void hh_seed_range_size(const uint32_t* ranges, uint32_t n, uint32_t max_seed_hits, uint32_t* size) {
    for (uint32_t a = 0; a < n; ++a) size[a] = seed_range_size(make_uint2(ranges[2 * a], ranges[2 * a + 1]), max_seed_hits);
}

// generic rank dictionary (dict_rank<W,I>): out[q] = rank(i[q], c[q]), all as uint64
void hh_dict_rank(const void* text, uint32_t word_bits, const void* occ, uint32_t K, const uint64_t* qi, const uint8_t* qc, uint32_t nq, uint64_t* out) {
    for (uint32_t q = 0; q < nq; ++q) {
        if (word_bits == 32) out[q] = dict_rank<uint32_t, uint32_t>((const uint32_t*)text, (const uint32_t*)occ, K, qi[q] == ~0ull ? 0xFFFFFFFFu : (uint32_t)qi[q], qc[q]);
        else                 out[q] = dict_rank<uint64_t, uint64_t>((const uint64_t*)text, (const uint64_t*)occ, K, qi[q], qc[q]);
    }
}

void hh_fm_locate(const uint32_t* bwt_occ, const uint32_t* ssa, const uint32_t* L2, uint32_t n, uint32_t primary,
                  const uint32_t* rows, uint32_t nq, uint32_t* out, uint32_t sa_interval) {
    const FmIndex f = mk(bwt_occ, ssa, L2, n, primary, sa_interval);
    for (uint32_t i = 0; i < nq; ++i) out[i] = fm_locate_one(f, rows[i]);
}

} // extern "C"

template <int B, int TYPE>
static void run_generic(const GotohScheme& S, const uint32_t* pw, uint32_t pbits, uint32_t pbe, const uint32_t* poff, const uint32_t* plen,
                        const uint8_t* quals, const uint32_t* tw, uint32_t tbits, uint32_t tbe, const uint32_t* toff, const uint32_t* tlen,
                        uint32_t n, int32_t* score, uint32_t* sx, uint32_t* sy) {
    for (uint32_t i = 0; i < n; ++i) {
        const SinkResult r = gotoh_generic<B, TYPE>(S, pw, pbits, pbe, poff[i], plen[i], quals, tw, tbits, tbe, toff[i], tlen[i]);
        score[i] = r.score; sx[i] = r.x; sy[i] = r.y;
    }
}

// mirrors gotoh_window_kernel
template <int B, int TYPE>
static void run_window(const GotohScheme& S, const uint32_t* pw, uint32_t pbits, uint32_t pbe, const uint32_t* poff, const uint32_t* plen,
                       const uint8_t* quals, const uint32_t* tw, uint32_t tbits, uint32_t tbe, const uint32_t* toff, const uint32_t* tlen,
                       uint32_t n, uint32_t wb, uint32_t we, const int32_t* min_score, int16_t* ckpt, int32_t* score, uint32_t* sx, uint32_t* sy, uint8_t* alive) {
    for (uint32_t i = 0; i < n; ++i) {
        SinkResult r;
        if (wb == 0) { r.score = NVB_SINK_MIN; r.x = r.y = 0xFFFFFFFFu; score[i] = r.score; sx[i] = r.x; sy[i] = r.y; alive[i] = 1; }
        else { if (!alive[i]) continue; r.score = score[i]; r.x = sx[i]; r.y = sy[i]; }
        if (wb >= plen[i]) continue;
        const bool ok = gotoh_window<B, TYPE>(S, pw, pbits, pbe, poff[i], plen[i], quals, tw, tbits, tbe, toff[i], tlen[i],
                                              wb, we < plen[i] ? we : plen[i], min_score ? min_score[i] : INT_MIN, (short2*)(ckpt + (size_t)i * 2 * B), r);
        score[i] = r.score; sx[i] = r.x; sy[i] = r.y; alive[i] = ok ? 1 : 0;
    }
}

// mirrors gotoh_pair_kernel: precondition check -> packed pair routine, else generic
static int g_hh_rows2 = 1;

template <int B, int TYPE>
static void run_pair(const GotohScheme& S, const uint8_t* quals, const uint32_t* pw, uint32_t pbits, uint32_t pbe, const uint32_t* poff, const uint32_t* plen,
                     const uint32_t* tw, uint32_t tbe, const uint32_t* toff, const uint32_t* tlen,
                     uint32_t n, uint32_t sel_rows, int32_t* score, uint32_t* sx, uint32_t* sy, uint32_t* n_fallback) {
    std::vector<uint16_t> sel(sel_rows + 1);
    for (uint32_t a0 = 0; a0 < n; a0 += 2) {
        const bool has1 = a0 + 1 < n;
        const uint32_t a1 = has1 ? a0 + 1 : a0;
        const uint32_t M0 = plen[a0], M1 = plen[a1], N0 = tlen[a0], N1 = tlen[a1];
        const uint32_t Mmax = M0 > M1 ? M0 : M1, L = Mmax + B - 1;
        const bool ok = M0 >= 1 && M1 >= 1 && N0 >= M0 + B - 1 && N1 >= M1 + B - 1 && L <= sel_rows && (TYPE == NVB_LOCAL || M0 == M1);
        if (!ok) {
            for (uint32_t a = a0; a <= a1; ++a) {
                const SinkResult r = gotoh_generic<B, TYPE>(S, pw, pbits, pbe, poff[a], plen[a], quals, tw, 2, tbe, toff[a], tlen[a]);
                score[a] = r.score; sx[a] = r.x; sy[a] = r.y; ++*n_fallback;
            }
            continue;
        }
        SymReaderRT r0(tw, 2, tbe), r1(tw, 2, tbe);
        for (uint32_t t = 0; t < L; ++t) {
            const uint32_t g0 = t < N0 ? r0.get(toff[a0] + t) : 0u, g1 = t < N1 ? r1.get(toff[a1] + t) : 0u;
            sel[t] = (uint16_t)pair_selector(g0, g1);
        }
        SinkResult q0, q1;
        // the kernel dispatcher's rule (launch_pair): compile-time pattern format for 2- / 4-bit big-endian patterns without a quality table
#define HH_PAIR2(PF, R2) gotoh_pair<B, TYPE, PF, R2>(S, pw, pbits, pbe, poff[a0], M0, poff[a1], M1, N0, N1, sel.data(), 1, q0, q1, quals)
        // two rows in flight per loop iteration (the kernels' default), unless switched off
#define HH_PAIR(PF) do { if (g_hh_rows2) HH_PAIR2(PF, true); else HH_PAIR2(PF, false); } while (0)
        if (!S.qtab && pbe && pbits == 2)      HH_PAIR(2);
        else if (!S.qtab && pbe && pbits == 4) HH_PAIR(4);
        else                                   HH_PAIR(0);
#undef HH_PAIR
#undef HH_PAIR2
        score[a0] = q0.score; sx[a0] = q0.x; sy[a0] = q0.y;
        if (has1) { score[a1] = q1.score; sx[a1] = q1.x; sy[a1] = q1.y; }
    }
}

extern "C" {

} // extern "C"
template <int B, int TYPE>
static void run_traceback(const GotohScheme& S, const uint32_t* pw, uint32_t pbits, uint32_t pbe, const uint32_t* poff, const uint32_t* plen,
                          const uint32_t* tw, uint32_t tbits, uint32_t tbe, const uint32_t* toff, const uint32_t* tlen, uint32_t n, uint32_t max_ops,
                          int32_t* score, uint32_t* sink_xy, uint32_t* source_xy, uint8_t* ops, uint32_t* n_ops) {
    for (uint32_t a = 0; a < n; ++a) {
        std::vector<uint32_t> dirs((size_t)(plen[a] + 1) * DirWords<B>::N);
        const SinkResult r = gotoh_generic_impl<B, TYPE, true>(S, pw, pbits, pbe, poff[a], plen[a], nullptr, tw, tbits, tbe, toff[a], tlen[a], dirs.data());
        score[a] = r.score; sink_xy[2 * a] = r.x; sink_xy[2 * a + 1] = r.y;
        uint32_t sx = 0xFFFFFFFFu, sy = 0xFFFFFFFFu, cnt = 0;
        if (r.x != 0xFFFFFFFFu && r.y != 0xFFFFFFFFu) cnt = gotoh_walk<B, TYPE>(dirs.data(), r, ops + (size_t)a * max_ops, max_ops, sx, sy);
        source_xy[2 * a] = sx; source_xy[2 * a + 1] = sy; n_ops[a] = cnt;
    }
}
extern "C" {

#define TYPE_SWITCH(BAND, FN, ...) \
    switch (type) { case 0: FN<BAND, 0>(__VA_ARGS__); return 0; case 1: FN<BAND, 1>(__VA_ARGS__); return 0; case 2: FN<BAND, 2>(__VA_ARGS__); return 0; } return -1;

int hh_gotoh_generic(int band, int type, const int32_t* scheme6, const int32_t* qtab,
                     const uint32_t* pw, uint32_t pbits, uint32_t pbe, const uint32_t* poff, const uint32_t* plen, const uint8_t* quals,
                     const uint32_t* tw, uint32_t tbits, uint32_t tbe, const uint32_t* toff, const uint32_t* tlen,
                     uint32_t n, int32_t* score, uint32_t* sx, uint32_t* sy) {
    GotohScheme S; S.match = scheme6[0]; S.mismatch = scheme6[1]; S.pgo = scheme6[2]; S.pge = scheme6[3]; S.tgo = scheme6[4]; S.tge = scheme6[5]; S.qtab = qtab; S.one = 1u; S.keymul = 32u;
    switch (band) {
    case 3:  TYPE_SWITCH(3,  run_generic, S, pw, pbits, pbe, poff, plen, quals, tw, tbits, tbe, toff, tlen, n, score, sx, sy)
    case 5:  TYPE_SWITCH(5,  run_generic, S, pw, pbits, pbe, poff, plen, quals, tw, tbits, tbe, toff, tlen, n, score, sx, sy)
    case 7:  TYPE_SWITCH(7,  run_generic, S, pw, pbits, pbe, poff, plen, quals, tw, tbits, tbe, toff, tlen, n, score, sx, sy)
    case 15: TYPE_SWITCH(15, run_generic, S, pw, pbits, pbe, poff, plen, quals, tw, tbits, tbe, toff, tlen, n, score, sx, sy)
    case 31: TYPE_SWITCH(31, run_generic, S, pw, pbits, pbe, poff, plen, quals, tw, tbits, tbe, toff, tlen, n, score, sx, sy)
    case 63: TYPE_SWITCH(63, run_generic, S, pw, pbits, pbe, poff, plen, quals, tw, tbits, tbe, toff, tlen, n, score, sx, sy)
    }
    return -1;
}

int hh_gotoh_window(int band, int type, const int32_t* scheme6, const int32_t* qtab,
                    const uint32_t* pw, uint32_t pbits, uint32_t pbe, const uint32_t* poff, const uint32_t* plen, const uint8_t* quals,
                    const uint32_t* tw, uint32_t tbits, uint32_t tbe, const uint32_t* toff, const uint32_t* tlen,
                    uint32_t n, uint32_t wb, uint32_t we, const int32_t* min_score, int16_t* ckpt, int32_t* score, uint32_t* sx, uint32_t* sy, uint8_t* alive) {
    GotohScheme S; S.match = scheme6[0]; S.mismatch = scheme6[1]; S.pgo = scheme6[2]; S.pge = scheme6[3]; S.tgo = scheme6[4]; S.tge = scheme6[5]; S.qtab = qtab; S.one = 1u; S.keymul = 32u;
    switch (band) {
    case 7:  TYPE_SWITCH(7,  run_window, S, pw, pbits, pbe, poff, plen, quals, tw, tbits, tbe, toff, tlen, n, wb, we, min_score, ckpt, score, sx, sy, alive)
    case 15: TYPE_SWITCH(15, run_window, S, pw, pbits, pbe, poff, plen, quals, tw, tbits, tbe, toff, tlen, n, wb, we, min_score, ckpt, score, sx, sy, alive)
    case 31: TYPE_SWITCH(31, run_window, S, pw, pbits, pbe, poff, plen, quals, tw, tbits, tbe, toff, tlen, n, wb, we, min_score, ckpt, score, sx, sy, alive)
    }
    return -1;
}

int hh_gotoh_full_q(int type, const int32_t* scheme6, const int32_t* qtab, const uint8_t* quals,
                  const uint32_t* pw, uint32_t pbits, uint32_t pbe, const uint32_t* poff, const uint32_t* plen,
                  const uint32_t* tw, uint32_t tbits, uint32_t tbe, const uint32_t* toff, const uint32_t* tlen, uint32_t n,
                  int32_t* score, uint32_t* sx, uint32_t* sy) {
    GotohScheme S; S.match = scheme6[0]; S.mismatch = scheme6[1]; S.pgo = scheme6[2]; S.pge = scheme6[3]; S.tgo = scheme6[4]; S.tge = scheme6[5]; S.qtab = qtab; S.one = 1u; S.keymul = 32u;
    for (uint32_t a = 0; a < n; ++a) {
        std::vector<int2> col(tlen[a] + 1);
        SinkResult r;
        if (type == 0)      r = gotoh_full<0>(S, pw, pbits, pbe, poff[a], plen[a], tw, tbits, tbe, toff[a], tlen[a], col.data(), 1, quals);
        else if (type == 1) r = gotoh_full<1>(S, pw, pbits, pbe, poff[a], plen[a], tw, tbits, tbe, toff[a], tlen[a], col.data(), 1, quals);
        else                r = gotoh_full<2>(S, pw, pbits, pbe, poff[a], plen[a], tw, tbits, tbe, toff[a], tlen[a], col.data(), 1, quals);
        score[a] = r.score; sx[a] = r.x; sy[a] = r.y;
    }
    return 0;
}

int hh_gotoh_full(int type, const int32_t* scheme6,
                  const uint32_t* pw, uint32_t pbits, uint32_t pbe, const uint32_t* poff, const uint32_t* plen,
                  const uint32_t* tw, uint32_t tbits, uint32_t tbe, const uint32_t* toff, const uint32_t* tlen, uint32_t n,
                  int32_t* score, uint32_t* sx, uint32_t* sy) {
    GotohScheme S; S.match = scheme6[0]; S.mismatch = scheme6[1]; S.pgo = scheme6[2]; S.pge = scheme6[3]; S.tgo = scheme6[4]; S.tge = scheme6[5]; S.qtab = nullptr; S.one = 1u; S.keymul = 32u;
    for (uint32_t a = 0; a < n; ++a) {
        std::vector<int2> col(tlen[a] + 1);
        SinkResult r;
        if (type == 0)      r = gotoh_full<0>(S, pw, pbits, pbe, poff[a], plen[a], tw, tbits, tbe, toff[a], tlen[a], col.data(), 1);
        else if (type == 1) r = gotoh_full<1>(S, pw, pbits, pbe, poff[a], plen[a], tw, tbits, tbe, toff[a], tlen[a], col.data(), 1);
        else                r = gotoh_full<2>(S, pw, pbits, pbe, poff[a], plen[a], tw, tbits, tbe, toff[a], tlen[a], col.data(), 1);
        score[a] = r.score; sx[a] = r.x; sy[a] = r.y;
    }
    return 0;
}

// packed pair version; alignments (2p, 2p+1) are paired when their lengths agree, else scored singly with gotoh_full
// returns the number of alignments that took the packed path
// host-side admission rule of the packed full-matrix path for a batch
int hh_full_pair_path_ok(int type, const int32_t* scheme6, uint32_t max_m, uint32_t max_n) {
    nvb_gotoh_scheme cs; cs.match = scheme6[0]; cs.mismatch = scheme6[1]; cs.pattern_gap_open = scheme6[2]; cs.pattern_gap_ext = scheme6[3];
    cs.text_gap_open = scheme6[4]; cs.text_gap_ext = scheme6[5]; cs.d_qual_table = nullptr; cs.qual_table_min = cs.qual_table_max = 0;
    return full_pair_path_ok(type, &cs, max_m, max_n) ? 1 : 0;
}

int hh_gotoh_full_pair(int type, const int32_t* scheme6,
                  const uint32_t* pw, uint32_t pbits, uint32_t pbe, const uint32_t* poff, const uint32_t* plen,
                  const uint32_t* tw, uint32_t tbits, uint32_t tbe, const uint32_t* toff, const uint32_t* tlen, uint32_t n,
                  int32_t* score, uint32_t* sx, uint32_t* sy) {
    GotohScheme S; S.match = scheme6[0]; S.mismatch = scheme6[1]; S.pgo = scheme6[2]; S.pge = scheme6[3]; S.tgo = scheme6[4]; S.tge = scheme6[5]; S.qtab = nullptr; S.one = 1u; S.keymul = 32u;
    int packed = 0;
    for (uint32_t a = 0; a < n; a += 2) {
        const uint32_t a1 = (a + 1 < n) ? a + 1 : a;
        std::vector<uint2> col(tlen[a] + 1);
        uint16_t sel[FULL_W];
        SinkResult r0, r1;
        bool ok = plen[a] == plen[a1] && tlen[a] == tlen[a1] && plen[a] >= 1 && tlen[a] >= 1;
        if (ok) {
            if (type == 0)      ok = gotoh_full_pair<0>(S, pw, pbits, pbe, poff[a], poff[a1], plen[a], tw, tbits, tbe, toff[a], toff[a1], tlen[a], col.data(), 1, sel, 1, r0, r1);
            else if (type == 1) ok = gotoh_full_pair<1>(S, pw, pbits, pbe, poff[a], poff[a1], plen[a], tw, tbits, tbe, toff[a], toff[a1], tlen[a], col.data(), 1, sel, 1, r0, r1);
            else                ok = gotoh_full_pair<2>(S, pw, pbits, pbe, poff[a], poff[a1], plen[a], tw, tbits, tbe, toff[a], toff[a1], tlen[a], col.data(), 1, sel, 1, r0, r1);
        }
        if (ok) {
            packed += (a1 != a) ? 2 : 1;
            score[a] = r0.score; sx[a] = r0.x; sy[a] = r0.y;
            if (a1 != a) { score[a1] = r1.score; sx[a1] = r1.x; sy[a1] = r1.y; }
        } else {
            hh_gotoh_full(type, scheme6, pw, pbits, pbe, poff + a, plen + a, tw, tbits, tbe, toff + a, tlen + a, (a1 != a) ? 2 : 1, score + a, sx + a, sy + a);
        }
    }
    return packed;
}

// the packed full-matrix routine in its quality-table form (per-column profiles); falls back to the int32 routine pair by pair like
// the kernel's todo list; returns the number of alignments that took the packed path, -2 when the scheme is not admitted
int hh_gotoh_full_pair_qual(int type, const int32_t* scheme6, const int32_t* qtab, const uint8_t* quals,
                  const uint32_t* pw, uint32_t pbits, uint32_t pbe, const uint32_t* poff, const uint32_t* plen,
                  const uint32_t* tw, uint32_t tbits, uint32_t tbe, const uint32_t* toff, const uint32_t* tlen, uint32_t n,
                  uint32_t max_m, uint32_t max_n, int32_t* score, uint32_t* sx, uint32_t* sy) {
    GotohScheme S; S.match = scheme6[0]; S.mismatch = scheme6[1]; S.pgo = scheme6[2]; S.pge = scheme6[3]; S.tgo = scheme6[4]; S.tge = scheme6[5]; S.qtab = qtab; S.one = 1u; S.keymul = 32u;
    nvb_gotoh_scheme cs; cs.match = S.match; cs.mismatch = S.mismatch; cs.pattern_gap_open = S.pgo; cs.pattern_gap_ext = S.pge;
    cs.text_gap_open = S.tgo; cs.text_gap_ext = S.tge; cs.d_qual_table = qtab;
    int32_t lo = qtab[0], hi = qtab[0];
    for (int i = 0; i < 512; ++i) { lo = qtab[i] < lo ? qtab[i] : lo; hi = qtab[i] > hi ? qtab[i] : hi; }
    cs.qual_table_min = lo; cs.qual_table_max = hi;
    if (!full_pair_path_ok(type, &cs, max_m, max_n)) return -2;
    int packed = 0;
    for (uint32_t a = 0; a < n; a += 2) {
        const uint32_t a1 = (a + 1 < n) ? a + 1 : a;
        std::vector<uint2> col(tlen[a] + 1);
        uint32_t colp[2 * FULL_W];
        SinkResult r0, r1;
        bool ok = plen[a] == plen[a1] && tlen[a] == tlen[a1] && plen[a] >= 1 && tlen[a] >= 1;
        if (ok) {
            if (type == 0)      ok = gotoh_full_pair<0, true>(S, pw, pbits, pbe, poff[a], poff[a1], plen[a], tw, tbits, tbe, toff[a], toff[a1], tlen[a], col.data(), 1, nullptr, 1, r0, r1, nullptr, colp, quals);
            else if (type == 1) ok = gotoh_full_pair<1, true>(S, pw, pbits, pbe, poff[a], poff[a1], plen[a], tw, tbits, tbe, toff[a], toff[a1], tlen[a], col.data(), 1, nullptr, 1, r0, r1, nullptr, colp, quals);
            else                ok = gotoh_full_pair<2, true>(S, pw, pbits, pbe, poff[a], poff[a1], plen[a], tw, tbits, tbe, toff[a], toff[a1], tlen[a], col.data(), 1, nullptr, 1, r0, r1, nullptr, colp, quals);
        }
        if (ok) {
            packed += (a1 != a) ? 2 : 1;
            score[a] = r0.score; sx[a] = r0.x; sy[a] = r0.y;
            if (a1 != a) { score[a1] = r1.score; sx[a1] = r1.x; sy[a1] = r1.y; }
        } else {
            for (uint32_t k = a; k <= a1; ++k) {
                std::vector<int2> c1(tlen[k] + 1);
                SinkResult r;
                if (type == 0)      r = gotoh_full_impl<0, false>(S, pw, pbits, pbe, poff[k], plen[k], tw, tbits, tbe, toff[k], tlen[k], c1.data(), 1, nullptr, 0, quals);
                else if (type == 1) r = gotoh_full_impl<1, false>(S, pw, pbits, pbe, poff[k], plen[k], tw, tbits, tbe, toff[k], tlen[k], c1.data(), 1, nullptr, 0, quals);
                else                r = gotoh_full_impl<2, false>(S, pw, pbits, pbe, poff[k], plen[k], tw, tbits, tbe, toff[k], tlen[k], c1.data(), 1, nullptr, 0, quals);
                score[k] = r.score; sx[k] = r.x; sy[k] = r.y;
            }
        }
    }
    return packed;
}

// gapless fast path of the banded traceback: ok[a] = 1 and len[a] = number of substitutions when the alignment (score, sink) is resolved
int hh_gapless_traceback(int type, const int32_t* scheme6, const int32_t* qtab, const uint8_t* quals,
                  const uint32_t* pw, uint32_t pbits, uint32_t pbe, const uint32_t* poff, const uint32_t* plen,
                  const uint32_t* tw, uint32_t tbits, uint32_t tbe, const uint32_t* toff, const uint32_t* tlen, uint32_t n,
                  const int32_t* score, const uint32_t* sink_xy, uint32_t* len, uint8_t* ok) {
    GotohScheme S; S.match = scheme6[0]; S.mismatch = scheme6[1]; S.pgo = scheme6[2]; S.pge = scheme6[3]; S.tgo = scheme6[4]; S.tge = scheme6[5]; S.qtab = qtab; S.one = 1u; S.keymul = 32u;
    for (uint32_t a = 0; a < n; ++a) {
        uint32_t l = 0; bool r;
        if (type == 0)      r = gapless_traceback<0>(S, pw, pbits, pbe, poff[a], plen[a], quals, tw, tbits, tbe, toff[a], tlen[a], score[a], sink_xy[2 * a], sink_xy[2 * a + 1], l);
        else if (type == 1) r = gapless_traceback<1>(S, pw, pbits, pbe, poff[a], plen[a], quals, tw, tbits, tbe, toff[a], tlen[a], score[a], sink_xy[2 * a], sink_xy[2 * a + 1], l);
        else                r = gapless_traceback<2>(S, pw, pbits, pbe, poff[a], plen[a], quals, tw, tbits, tbe, toff[a], tlen[a], score[a], sink_xy[2 * a], sink_xy[2 * a + 1], l);
        len[a] = l; ok[a] = r ? 1 : 0;
    }
    return 0;
}

int hh_gotoh_full_traceback(int type, const int32_t* scheme6,
                  const uint32_t* pw, uint32_t pbits, uint32_t pbe, const uint32_t* poff, const uint32_t* plen,
                  const uint32_t* tw, uint32_t tbits, uint32_t tbe, const uint32_t* toff, const uint32_t* tlen, uint32_t n, uint32_t max_ops,
                  int32_t* score, uint32_t* sink_xy, uint32_t* source_xy, uint8_t* ops, uint32_t* n_ops) {
    GotohScheme S; S.match = scheme6[0]; S.mismatch = scheme6[1]; S.pgo = scheme6[2]; S.pge = scheme6[3]; S.tgo = scheme6[4]; S.tge = scheme6[5]; S.qtab = nullptr; S.one = 1u; S.keymul = 32u;
    for (uint32_t a = 0; a < n; ++a) {
        std::vector<int2> col(tlen[a] + 1);
        const uint32_t rw = (plen[a] + 31u) / 32u * 4u;
        std::vector<uint32_t> dirs((size_t)(tlen[a] + 1) * (rw ? rw : 4u));
        SinkResult r;
        uint32_t sx = 0xFFFFFFFFu, sy = 0xFFFFFFFFu, cnt = 0;
#define HH_FT(T) { r = gotoh_full_impl<T, true>(S, pw, pbits, pbe, poff[a], plen[a], tw, tbits, tbe, toff[a], tlen[a], col.data(), 1, dirs.data(), rw); \
                   if (r.x != 0xFFFFFFFFu && r.y != 0xFFFFFFFFu) cnt = gotoh_full_walk<T>(dirs.data(), rw, r, ops + (size_t)a * max_ops, max_ops, sx, sy); }
        if (type == 0) HH_FT(0) else if (type == 1) HH_FT(1) else HH_FT(2)
#undef HH_FT
        score[a] = r.score; sink_xy[2 * a] = r.x; sink_xy[2 * a + 1] = r.y; source_xy[2 * a] = sx; source_xy[2 * a + 1] = sy; n_ops[a] = cnt;
    }
    return 0;
}

int hh_gotoh_traceback(int band, int type, const int32_t* scheme6,
                       const uint32_t* pw, uint32_t pbits, uint32_t pbe, const uint32_t* poff, const uint32_t* plen,
                       const uint32_t* tw, uint32_t tbits, uint32_t tbe, const uint32_t* toff, const uint32_t* tlen, uint32_t n, uint32_t max_ops,
                       int32_t* score, uint32_t* sink_xy, uint32_t* source_xy, uint8_t* ops, uint32_t* n_ops) {
    GotohScheme S; S.match = scheme6[0]; S.mismatch = scheme6[1]; S.pgo = scheme6[2]; S.pge = scheme6[3]; S.tgo = scheme6[4]; S.tge = scheme6[5]; S.qtab = nullptr; S.one = 1u; S.keymul = 32u;
    switch (band) {
    case 7:  TYPE_SWITCH(7,  run_traceback, S, pw, pbits, pbe, poff, plen, tw, tbits, tbe, toff, tlen, n, max_ops, score, sink_xy, source_xy, ops, n_ops)
    case 15: TYPE_SWITCH(15, run_traceback, S, pw, pbits, pbe, poff, plen, tw, tbits, tbe, toff, tlen, n, max_ops, score, sink_xy, source_xy, ops, n_ops)
    case 31: TYPE_SWITCH(31, run_traceback, S, pw, pbits, pbe, poff, plen, tw, tbits, tbe, toff, tlen, n, max_ops, score, sink_xy, source_xy, ops, n_ops)
    }
    return -1;
}

// 1 (default): two pattern rows in flight per loop iteration, as the kernels do; 0: one row
void hh_set_pair_rows2(int on) { g_hh_rows2 = on; }

// returns -2 when the scheme is not admissible for the packed path
int hh_gotoh_pair(int band, int type, const int32_t* scheme6, const int32_t* qtab, const uint8_t* quals, uint32_t max_m,
                  const uint32_t* pw, uint32_t pbits, uint32_t pbe, const uint32_t* poff, const uint32_t* plen,
                  const uint32_t* tw, uint32_t tbe, const uint32_t* toff, const uint32_t* tlen,
                  uint32_t n, int32_t* score, uint32_t* sx, uint32_t* sy, uint32_t* n_fallback) {
    GotohScheme S; S.match = scheme6[0]; S.mismatch = scheme6[1]; S.pgo = scheme6[2]; S.pge = scheme6[3]; S.tgo = scheme6[4]; S.tge = scheme6[5]; S.qtab = qtab; S.one = 1u; S.keymul = 32u;
    nvb_gotoh_scheme cs; cs.match = S.match; cs.mismatch = S.mismatch; cs.pattern_gap_open = S.pgo; cs.pattern_gap_ext = S.pge;
    cs.text_gap_open = S.tgo; cs.text_gap_ext = S.tge; cs.d_qual_table = qtab; cs.qual_table_min = cs.qual_table_max = 0;
    if (qtab) { int32_t lo = qtab[0], hi = qtab[0]; for (int i = 0; i < 512; ++i) { lo = qtab[i] < lo ? qtab[i] : lo; hi = qtab[i] > hi ? qtab[i] : hi; }
                cs.qual_table_min = lo; cs.qual_table_max = hi; }
    if (!pair_path_ok(band, type, &cs, max_m)) return -2;
    const uint32_t sel_rows = max_m + band - 1;
    *n_fallback = 0;
    switch (band) {
    case 7:  TYPE_SWITCH(7,  run_pair, S, quals, pw, pbits, pbe, poff, plen, tw, tbe, toff, tlen, n, sel_rows, score, sx, sy, n_fallback)
    case 15: TYPE_SWITCH(15, run_pair, S, quals, pw, pbits, pbe, poff, plen, tw, tbe, toff, tlen, n, sel_rows, score, sx, sy, n_fallback)
    case 31: TYPE_SWITCH(31, run_pair, S, quals, pw, pbits, pbe, poff, plen, tw, tbe, toff, tlen, n, sel_rows, score, sx, sy, n_fallback)
    }
    return -1;
}

} // extern "C"
