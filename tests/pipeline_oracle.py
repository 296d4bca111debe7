"""Oracle composition of the seed+extend pipeline (test infrastructure): the same stages as
nvbio_b200/csrc/pipeline.cu, each stage computed by the CPU oracle / reference library."""
import numpy as np


def _scheme_args(sch):
    """(scheme tuple, qtab or None) of a SimpleGotohScheme / QualityGotohScheme"""
    if hasattr(sch, "table_host"):
        return (sch.match_bonus, int(sch.table_host[0, 1]), sch.pgo, sch.pge, sch.tgo, sch.tge), sch.table_host
    return (sch.match, sch.mismatch, sch.gap_open, sch.gap_ext), None


NO_POS = 0xFFFFFFFF


def hit_end(window_begin, sink_x):
    """genome coordinate window begin + sink.x of an alignment end (include/nvbio_b200.h, d_best_pos); NO_POS for the DP's default
    sink 0xFFFFFFFF, which a window shorter than its read gets (no alignment fits)"""
    return NO_POS if int(sink_x) == NO_POS else int(window_begin) + int(sink_x)


def seed_extend_oracle(O, idx, genome_sym, reads, params, quals=None, hit_capacity=None):
    """reads: list of uint8 arrays; quals: optional list of uint8 arrays (base qualities, with a QualityGotohScheme).
    hit_capacity: hits at index >= capacity are dropped (in hit order) and the best is taken over the kept hits only.
    Returns dict(best_score, best_pos, best_hit (-1: none), hit_string, hit_window, hit_score, hit_sink, n_hits (kept), n_found)."""
    L, I, B = params.seed_len, params.seed_interval, params.band_len
    n = idx.n
    strands = 2 if params.both_strands else 1
    strings, squals = [], []
    for i, r in enumerate(reads):
        strings.append(r)
        if quals is not None:
            squals.append(quals[i])
        if strands == 2:
            rc = np.where(r < 4, 3 - r, r)[::-1].astype(np.uint8)
            strings.append(rc)
            if quals is not None:
                squals.append(quals[i][::-1])
    max_len = max(len(r) for r in reads)
    K = (max_len - L) // I + 1
    # seeds
    q, off, ln, valid = [], [], [], []
    o = 0
    for s in strings:
        for k in range(K):
            p = k * I
            if p + L <= len(s):
                q.append(s[p:p + L]); off.append(o); ln.append(L); o += L; valid.append(True)
            else:
                off.append(o); ln.append(0); valid.append(False)
    qcat = np.concatenate(q) if q else np.zeros(1, np.uint8)
    ranges, _ = O.match(idx, qcat, np.array(off, np.uint32), np.array(ln, np.uint32))
    # hits in slot order: seed by seed (string, then seed), the first max_seed_hits rows of each range
    x, y = ranges[:, 0].astype(np.int64), ranges[:, 1].astype(np.int64)
    sz = np.where(np.array(valid, bool) & (x <= y), np.minimum(y - x + 1, params.max_seed_hits), 0)
    n_found = int(sz.sum())
    qi = np.repeat(np.arange(len(sz)), sz)
    rows = (x[qi] + np.arange(n_found) - np.repeat(np.cumsum(sz) - sz, sz))
    kept = n_found if hit_capacity is None else min(n_found, hit_capacity)
    qi, rows = qi[:kept], rows[:kept]
    hit_string, seed_begin = qi // K, (qi % K) * I
    pos = O.locate(idx, rows.astype(np.uint32)).astype(np.int64) if kept else np.zeros(0, np.int64)
    s_len = np.array([len(s) for s in strings], np.int64)
    s_off = np.cumsum(s_len) - s_len
    ln_s = s_len[hit_string]
    diag = np.where(pos > seed_begin, pos - seed_begin, 0)
    gb = np.where(diag > B // 2, diag - B // 2, 0)
    ge = np.minimum(gb + ln_s + B, n)
    wins = np.stack([gb, ge], axis=1)
    scheme, qtab = _scheme_args(params.scheme)
    score = np.zeros(kept, np.int64); sink = np.zeros((kept, 2), np.int64)
    if kept:
        # every distinct (string, window) job once; the patterns are the strings themselves
        jobs, inv = np.unique(np.stack([hit_string, gb, ge], axis=1), axis=0, return_inverse=True)
        inv = inv.reshape(-1)
        sc, sx, sy, _ = O.banded_gotoh(B, params.type, scheme, np.concatenate(strings), s_off[jobs[:, 0]].astype(np.uint32),
                                       s_len[jobs[:, 0]].astype(np.uint32), genome_sym, jobs[:, 1].astype(np.uint32),
                                       (jobs[:, 2] - jobs[:, 1]).astype(np.uint32),
                                       qual=np.concatenate(squals) if quals is not None else None, qtab=qtab)
        score = sc.astype(np.int64)[inv]
        sink = np.stack([sx.astype(np.int64), sy.astype(np.int64)], axis=1)[inv]
    # best hit per read: max score, ties -> smallest hit index
    best_score = np.full(len(reads), -2**31, np.int64)
    best_pos = np.full(len(reads), NO_POS, np.int64)
    best_hit = np.full(len(reads), -1, np.int64)
    read = hit_string // strands
    order = np.lexsort((np.arange(kept), -score, read))
    first = order[np.r_[True, read[order][1:] != read[order][:-1]]] if kept else order
    for h in first.tolist():
        r = int(read[h])
        best_hit[r] = h; best_score[r] = int(score[h]); best_pos[r] = hit_end(gb[h], sink[h, 0])
    return dict(best_score=best_score, best_pos=best_pos, best_hit=best_hit, hit_string=hit_string.astype(np.int64),
                hit_window=wins.astype(np.int64).reshape(-1, 2), hit_score=score, hit_sink=sink.reshape(-1, 2), n_hits=kept, n_found=n_found)


def seed_extend_paired_oracle(O, idx, genome_sym, reads, params, pair, n_pairs, quals=None):
    """Oracle composition of nvb_seed_extend_paired: the single-end composition above for the 2*n_pairs mates, the pairing rules of
    include/nvbio_b200.h restated in Python, and the opposite-mate rescue scored by the oracle's full-matrix Gotoh.
    reads: mate 1 of every pair, then mate 2.  Returns dict(pair_score, pair_flags, mate_score[2,n], mate_pos[2,n], mate_strand[2,n],
    n_rescue)."""
    se = seed_extend_oracle(O, idx, genome_sym, reads, params, quals=quals)
    glen = idx.n
    strands = 2
    best_h = se["best_hit"]
    INT_MIN = -2**31

    def mate(r):
        # a mate is aligned when its best hit has a position (a window shorter than the read has none: hit_end)
        h = best_h[r]
        end = NO_POS if h < 0 else hit_end(se["hit_window"][h][0], se["hit_sink"][h][0])
        if end == NO_POS:
            return dict(has=False, score=INT_MIN, strand=0, beg=0xFFFFFFFF, end=0xFFFFFFFF, len=0)
        s = int(se["hit_string"][h])
        ln = len(reads[r])
        return dict(has=True, score=int(se["hit_score"][h]), strand=s % strands, beg=max(end - ln, 0), end=end, len=ln)

    cap = 2 * n_pairs if pair.rescue_capacity is None else pair.rescue_capacity
    pair_score = np.full(n_pairs, INT_MIN, np.int64); pair_flags = np.zeros(n_pairs, np.int64)
    mate_score = np.full((2, n_pairs), INT_MIN, np.int64); mate_pos = np.full((2, n_pairs), 0xFFFFFFFF, np.int64)
    mate_strand = np.zeros((2, n_pairs), np.int64)
    jobs = []          # (pair, anchor, pattern symbols, window begin, window length)
    for p in range(n_pairs):
        m = [mate(p), mate(n_pairs + p)]
        for k in range(2):
            mate_score[k, p], mate_pos[k, p], mate_strand[k, p] = m[k]["score"], m[k]["end"], m[k]["strand"]
        conc = m[0]["has"] and m[1]["has"] and m[0]["strand"] != m[1]["strand"]
        if conc:
            f, r = (m[0], m[1]) if m[0]["strand"] == 0 else (m[1], m[0])
            frag = r["end"] - f["beg"]
            conc = f["beg"] <= r["beg"] and f["end"] <= r["end"] and r["end"] > f["beg"] and pair.min_frag <= frag <= pair.max_frag
        if conc:
            pair_score[p] = m[0]["score"] + m[1]["score"]; pair_flags[p] = 1
            continue
        for a in range(2):
            if not (m[a]["has"] and m[a]["score"] >= pair.min_mate_score):
                continue
            o = reads[(1 - a) * n_pairs + p]
            oq = quals[(1 - a) * n_pairs + p] if quals is not None else None
            if m[a]["strand"] == 0:
                to = m[a]["beg"]; te = min(to + pair.max_frag, glen)
                pat = np.where(o < 4, 3 - o, o)[::-1].astype(np.uint8)
                pq = oq[::-1] if oq is not None else None
            else:
                to = max(m[a]["end"] - pair.max_frag, 0); te = m[a]["end"]
                pat = o
                pq = oq
            if te - to >= 1 and len(pat) >= 1:
                jobs.append((p, a, pat, to, te - to, pq))
    wanted = len(jobs)
    run = jobs[:cap]
    if run:
        pats = np.concatenate([j[2] for j in run])
        p_len = np.array([len(j[2]) for j in run], np.uint32)
        p_off = (np.cumsum(p_len) - p_len).astype(np.uint32)
        t_off = np.array([j[3] for j in run], np.uint32); t_len = np.array([j[4] for j in run], np.uint32)
        scheme, qtab = _scheme_args(params.scheme)
        rs, rx, _ = O.gotoh_full(params.type, scheme, pats, p_off, p_len, genome_sym, t_off, t_len,
                                 qual=np.concatenate([j[5] for j in run]) if quals is not None else None, qtab=qtab)
        cand = {}
        for (p, a, _, to, _, _), s, x in zip(run, rs, rx):
            if int(s) < pair.min_mate_score:
                continue
            tot = int(mate_score[a, p]) + int(s)
            if p not in cand or tot > cand[p][0]:
                cand[p] = (tot, a, int(s), to + int(x))
        for p, (tot, a, s, pos) in cand.items():
            o = 1 - a
            pair_score[p] = tot; pair_flags[p] = 2 if o == 0 else 4
            mate_score[o, p] = s; mate_pos[o, p] = pos; mate_strand[o, p] = 1 - mate_strand[a, p]
    return dict(pair_score=pair_score, pair_flags=pair_flags, mate_score=mate_score, mate_pos=mate_pos, mate_strand=mate_strand,
                n_rescue=(len(run), wanted))
