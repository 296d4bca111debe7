"""Generate tests/golden/*.npz by RUNNING THE REFERENCE ITSELF (oracle/_ref/libnvbio_ref.so, i.e. the
unmodified nvbio templates compiled by oracle/Makefile from /root/reference).

Run in the dev container only (needs /root/reference to have built oracle/_ref):
    python tests/golden/make_golden.py

The fixtures pin (a) the two banded-Gotoh problems asserted by the reference's own test
(nvbio-test/alignment_test.cu:761-825), (b) seeded random banded problems for every BAND/TYPE the
reference instantiates, incl. text symbols > 3 and ragged lengths, (c) a small FM-index
(SA, BWT, occ, SSA, match ranges, locate results) incl. a repetitive text, (d) full-matrix Gotoh scores, sinks and
tracebacks (gotoh_full.npz; `--only-full` regenerates just that file), (e) the reference tree's source files and their line counts
(reference_files.json, which the documentation's citations are checked against; `--only-files DIR` writes it from the tree at DIR).
"""
import os
import sys
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import orc  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))

G1_P = "ACAACTA"
G1_T = "AAACACCCTAACACACTAAA"
G2_P = ("TTATGTAGGTGGTCTGGTTTTTGCCTTTTAAGCTTCTGCAAAAAACAACAACAAACTTGTGGTATTACACTGACTCTACAGATCAATTTGGGGACAACTTCC"
        "ATGTGTTCCACCACCAATACTGAATCTTTCAATCGACTGACGTGGTAT")
G2_T = ("ATCGGATTCTTTCTTACTTGTAGGTGGTCTGGTTTTTGCCTTTTAAGCTTCTGCAAAAAACAACAACAAACTTGTGGTATTACACTGACTCTACAGATCAA"
        "TTTGGGGACAACTTCCATGTGTTCCACCACCAATACTGAATCTTTCAATCGACTGACGTGGTATCTCTCTCTCCATCTAT")


def random_problems(rng, n, band, max_m, alphabet_text=4, ragged=True):
    """patterns sampled from their own windows with mutations, so that alignments are non-trivial"""
    pats, txts, p_off, p_len, t_off, t_len = [], [], [], [], [], []
    po = to = 0
    for _ in range(n):
        m = int(rng.integers(1, max_m + 1)) if ragged else max_m
        extra = int(rng.integers(0, band + 8))
        extra = max(extra, band - 1 - m)                       # the reference reads text[0..B-2] unchecked
        N = m + extra
        t = rng.integers(0, alphabet_text, size=N).astype(np.uint8)
        start = int(rng.integers(0, min(extra, band // 2) + 1))
        p = []
        j = start
        while len(p) < m:
            r = rng.random()
            if r < 0.05 or j >= N:
                p.append(int(rng.integers(0, 4)))           # substitution / insertion
                if r < 0.03:
                    j += 1
            elif r < 0.08:
                j += 1                                         # deletion
            else:
                p.append(int(t[j]) & 3)
                j += 1
        p = np.array(p[:m], dtype=np.uint8)
        if alphabet_text > 4 and rng.random() < 0.3:
            p[int(rng.integers(0, m))] = 4                     # an N in the read
        pats.append(p); txts.append(t)
        p_off.append(po); p_len.append(m); po += m
        t_off.append(to); t_len.append(N); to += N
    return (np.concatenate(pats), np.array(p_off, np.uint32), np.array(p_len, np.uint32),
            np.concatenate(txts), np.array(t_off, np.uint32), np.array(t_len, np.uint32))


def full_problems(rng, n, max_m, max_n, paired=False):
    """patterns drawn from a window of their own text with a few substitutions / an indel; `paired`: consecutive problems share
    their shape (the packed two-per-thread kernel admits them)"""
    pats, txts, po, pl, to, tl = [], [], [], [], [], []
    a = b = 0
    M = N = 0
    for i in range(n):
        if not paired or i % 2 == 0:
            M = int(rng.integers(1, max_m + 1)); N = int(rng.integers(1, max_n + 1))
        t = rng.integers(0, 4, N).astype(np.uint8)
        if N > M + 2 and rng.random() < 0.8:
            st = int(rng.integers(0, N - M - 1)); src = list(t[st:st + M + 2])
            if rng.random() < 0.4 and M > 4:
                k = int(rng.integers(1, M - 1))
                if rng.random() < 0.5:
                    del src[k]
                else:
                    src.insert(k, int(rng.integers(0, 4)))
            p = np.array(src[:M], np.uint8)
            for _k in range(int(rng.integers(0, 4))):
                p[int(rng.integers(0, M))] = rng.integers(0, 4)
        else:
            p = rng.integers(0, 4, M).astype(np.uint8)
        pats.append(p); txts.append(t); po.append(a); pl.append(M); a += M; to.append(b); tl.append(N); b += N
    return (np.concatenate(pats), np.array(po, np.uint32), np.array(pl, np.uint32), np.concatenate(txts), np.array(to, np.uint32), np.array(tl, np.uint32))


def make_full(ref):
    """(d) full-matrix Gotoh: scores + sinks (aln::alignment_score) and tracebacks (aln::alignment_traceback<256,512,64>) of the
    reference on its own 7 x 20 strings (alignment_test.cu:761-793) and on seeded random problems -> gotoh_full.npz"""
    rng = np.random.default_rng(20240924)
    out = {}
    p, t = orc.dna(G1_P), orc.dna(G1_T)
    for typ in (0, 1, 2):
        a = ref.gotoh_full_traceback(typ, (2, -1, -1, -1), p, [0], [len(p)], t, [0], [len(t)], max_ops=64)
        out[f"g1_t{typ}"] = np.array([a["score"][0], a["sink"][0][0], a["sink"][0][1], a["source"][0][0], a["source"][0][1]], np.int64)
        out[f"g1_t{typ}_ops"] = a["ops"][0][:a["n_ops"][0]].copy()
    cases, cid = [], 0
    for typ in (0, 1, 2):
        for scheme in ((2, -2, -5, -3), (2, -1, -2, -1), (0, -5, -8, -3), (1, -3, -2, -4)):
            for paired in (False, True):
                pr = full_problems(rng, 40, 150, 320, paired=paired)
                s, x, y = ref.gotoh_full(typ, scheme, *pr)
                tb = ref.gotoh_full_traceback(typ, scheme, *pr, max_ops=512)
                assert np.array_equal(s, tb["score"]) and np.array_equal(x, tb["sink"][:, 0]) and np.array_equal(y, tb["sink"][:, 1])
                for k, v in zip(("pat", "p_off", "p_len", "txt", "t_off", "t_len"), pr):
                    out[f"f{cid}_{k}"] = v
                out[f"f{cid}_res"] = np.stack([s.astype(np.int64), x.astype(np.int64), y.astype(np.int64),
                                               tb["source"][:, 0].astype(np.int64), tb["source"][:, 1].astype(np.int64), tb["n_ops"].astype(np.int64)])
                out[f"f{cid}_ops"] = np.concatenate([tb["ops"][i][:tb["n_ops"][i]] for i in range(len(s))])
                cases.append((cid, typ) + scheme)
                cid += 1
    out["cases"] = np.array(cases, dtype=np.int64)
    np.savez_compressed(os.path.join(OUT, "gotoh_full.npz"), **out)


def make_extras(ref):
    """(e) windowed banded scoring pass by pass (aln::banded_alignment_score<B>(..., window_begin, window_end, sink, checkpoint)) and
    (f) the quality-table scheme through the reference templates (TableGotohScheme in oracle/ref_shim.cpp) -> banded_extras.npz.
    Windowed problems have N >= M + B - 1 (the reference reads text[wb .. wb+B-2] unchecked at a window start)."""
    rng = np.random.default_rng(20240925)
    out = {}
    qtab = np.zeros((256, 2), np.int32)
    for q in range(256):
        qtab[q, 0] = 2
        qtab[q, 1] = -(2 + int(min(q, 40) / 40.0 * 4))
    out["qtab"] = qtab
    wcases, qcases = [], []
    cid = 0
    for band in (7, 15, 31):
        for typ in (0, 1, 2):
            # windowed: fixed M = 100, windows of 32 rows, with and without a min-score cut-off
            M = 100
            pr = random_problems(rng, 40, band, M, ragged=False)
            pat, p_off, p_len, txt, t_off, t_len = pr
            keep = t_len >= p_len + band - 1
            idxs = np.nonzero(keep)[0]
            pats = [pat[p_off[i]:p_off[i] + p_len[i]] for i in idxs]; txts = [txt[t_off[i]:t_off[i] + t_len[i]] for i in idxs]
            p_len2 = np.array([len(x) for x in pats], np.uint32); t_len2 = np.array([len(x) for x in txts], np.uint32)
            p_off2 = (np.cumsum(p_len2) - p_len2).astype(np.uint32); t_off2 = (np.cumsum(t_len2) - t_len2).astype(np.uint32)
            pr2 = (np.concatenate(pats), p_off2, p_len2, np.concatenate(txts), t_off2, t_len2)
            n = len(p_off2)
            for ms in (None, rng.integers(-20, 150, n).astype(np.int32)):
                st = orc.window_state(n, band)
                snaps = []
                for wb in range(0, M, 32):
                    ref.banded_gotoh_window(band, typ, (2, -2, -5, -3), *pr2, wb, wb + 32, st, min_score=ms)
                    snaps.append(np.concatenate([st["score"].astype(np.int64), st["sx"].astype(np.int64), st["sy"].astype(np.int64), st["alive"].astype(np.int64)]))
                for k, v in zip(("pat", "p_off", "p_len", "txt", "t_off", "t_len"), pr2):
                    out[f"w{cid}_{k}"] = v
                out[f"w{cid}_ms"] = ms if ms is not None else np.zeros(0, np.int32)
                out[f"w{cid}_snaps"] = np.stack(snaps)
                out[f"w{cid}_ckpt"] = st["ckpt"].copy()
                wcases.append((cid, band, typ))
                cid += 1
            # quality table, banded
            pr = random_problems(rng, 40, band, 120)
            qual = rng.integers(0, 64, len(pr[0])).astype(np.uint8)
            s, x, y, ok = ref.banded_gotoh(band, typ, (0, 0, -8, -3, -7, -2), *pr, qual=qual, qtab=qtab)
            for k, v in zip(("pat", "p_off", "p_len", "txt", "t_off", "t_len"), pr):
                out[f"q{cid}_{k}"] = v
            out[f"q{cid}_qual"] = qual
            out[f"q{cid}_res"] = np.stack([s.astype(np.int64), x.astype(np.int64), y.astype(np.int64), ok.astype(np.int64)])
            qcases.append((cid, band, typ))
            cid += 1
    for typ in (0, 1, 2):           # quality table, full matrix (band = 0 in the case list)
        pr = full_problems(rng, 40, 150, 300)
        qual = rng.integers(0, 64, len(pr[0])).astype(np.uint8)
        s, x, y = ref.gotoh_full(typ, (0, 0, -8, -3, -7, -2), *pr, qual=qual, qtab=qtab)
        for k, v in zip(("pat", "p_off", "p_len", "txt", "t_off", "t_len"), pr):
            out[f"q{cid}_{k}"] = v
        out[f"q{cid}_qual"] = qual
        out[f"q{cid}_res"] = np.stack([s.astype(np.int64), x.astype(np.int64), y.astype(np.int64), np.ones(len(s), np.int64)])
        qcases.append((cid, 0, typ))
        cid += 1
    out["wcases"] = np.array(wcases, np.int64); out["qcases"] = np.array(qcases, np.int64)
    np.savez_compressed(os.path.join(OUT, "banded_extras.npz"), **out)


def make_nvbowtie(ref, path=None):
    """(g) nvBowtie's OWN scoring scheme object (SmithWatermanScoringScheme<QualCost<int>,ConstantCost<int>>, scoring.h:86-105,203-317,
    compiled from the reference by oracle/ref_nvbowtie.cpp): the 256 x 2 substitution tables of its presets and of a few custom
    constants, and banded DP results with per-base qualities under the --local preset -> nvbowtie_scheme.npz"""
    out = {}
    cfgs = [(1, 0, 0, 0), (2, 0, 0, 0), (0, 2, 2, 6), (0, 0, 2, 6), (0, 3, 1, 30), (0, 1, 3, 3), (0, 2, 6, 2), (0, 0, 0, 255)]
    out["cfgs"] = np.array(cfgs, dtype=np.int32)
    for i, (preset, mb, lo, hi) in enumerate(cfgs):
        tab, gaps, lim = ref.nvbowtie_scheme(preset, mb, lo, hi)
        out[f"tab{i}"] = tab; out[f"gaps{i}"] = np.array(gaps, np.int32); out[f"lim{i}"] = np.array(lim, np.int32)
    rng = np.random.default_rng(97)
    cases = []
    for cid, (band, typ) in enumerate([(31, 1), (31, 2), (15, 1), (15, 2)]):
        pr = random_problems(rng, 60, band, 150)
        qual = rng.integers(0, 64, len(pr[0])).astype(np.uint8)
        s, x, y = ref.nvbowtie_banded(band, typ, pr[0], qual, pr[1], pr[2], pr[3], pr[4], pr[5], preset=1)
        for k, v in zip(("pat", "p_off", "p_len", "txt", "t_off", "t_len"), pr):
            out[f"d{cid}_{k}"] = np.asarray(v)
        out[f"d{cid}_qual"] = qual
        out[f"d{cid}_res"] = np.stack([s.astype(np.int64), x.astype(np.int64), y.astype(np.int64)])
        cases.append((cid, band, typ))
    out["dcases"] = np.array(cases, dtype=np.int32)
    np.savez_compressed(path or os.path.join(OUT, "nvbowtie_scheme.npz"), **out)


def make_generic_rank(ref):
    """(h) generic rank dictionary (SURVEY 8a row a6): packed words, occ tables and rank answers of the reference's rank_dictionary over
    plain 32- / 64-bit-word streams (the instantiations of nvbio-test/rank_test.cu:144-232, plus other K) -> generic_rank.npz"""
    out = {}
    rng = np.random.default_rng(5)
    cfgs = [(32, 64, 1000), (32, 128, 4097), (32, 16, 333), (64, 64, 2048), (64, 256, 5001)]
    out["cfgs"] = np.array(cfgs, dtype=np.int64)
    for i, (wb, K, n) in enumerate(cfgs):
        text = rng.integers(0, 4, n).astype(np.uint8)
        qi = np.concatenate([rng.integers(0, n, 500).astype(np.uint64), np.array([0, n - 1, K - 1, K, 0xFFFFFFFFFFFFFFFF], dtype=np.uint64)])
        qc = rng.integers(0, 4, len(qi)).astype(np.uint8)
        words, occ, ranks = ref.generic_rank(wb, K, text, qi, qc)
        out[f"text{i}"] = text; out[f"qi{i}"] = qi; out[f"qc{i}"] = qc
        out[f"words{i}"] = words[: (n + wb // 2 - 1) // (wb // 2)]; out[f"occ{i}"] = occ; out[f"ranks{i}"] = ranks
    np.savez_compressed(os.path.join(OUT, "generic_rank.npz"), **out)


def make_nvbwt_files():
    """(i) index FILES written by the reference's own writer code: nvBWT's save_bwt() / save_ssa() (nvBWT/nvBWT.cu:314-351, compiled by
    oracle/ref_nvbwt_writer.cu) are called with the arrays of two indices of fmindex.npz, exactly as nvBWT's build() calls them
    (nvBWT.cu:394-405, 514-515) -> nvbwt_files.npz holds the bytes of the .bwt / .sa files.  Note the reference's save_ssa() writes
    `&cumFreq` (the address of its pointer argument) where the four cumulative counts belong, so bytes 4..20 of a .sa file written
    by nvBWT are arbitrary; they are zeroed in the fixture and listed in `sa_unspecified`."""
    import ctypes as C, tempfile
    W = C.CDLL(os.path.join(OUT, "..", "..", "oracle", "_ref", "libnvbwt_writer.so"), mode=os.RTLD_LAZY)
    fm = np.load(os.path.join(OUT, "fmindex.npz"))
    out = {}
    for name in ("rand", "rep", "tiny"):
        n = len(fm[f"{name}_text"]); primary = int(fm[f"{name}_primary"][0])
        cum = np.ascontiguousarray(fm[f"{name}_L2"][1:5], dtype=np.uint32)
        words = np.ascontiguousarray(fm[f"{name}_bwt_occ"].reshape(-1, 8)[:, :4]).reshape(-1).astype(np.uint32)
        seq_words = (n + 15) // 16
        ssa = np.ascontiguousarray(fm[f"{name}_ssa"], dtype=np.uint32)
        ssa_len = (n + 16) // 16
        assert len(ssa) >= ssa_len and len(words) >= seq_words
        with tempfile.TemporaryDirectory() as d:
            b, a = os.path.join(d, "x.bwt").encode(), os.path.join(d, "x.sa").encode()
            W.ref_nvbwt_save_bwt(C.c_uint(n), C.c_uint(seq_words), C.c_uint(primary), cum.ctypes.data_as(C.c_void_p), words.ctypes.data_as(C.c_void_p), b)
            W.ref_nvbwt_save_ssa(C.c_uint(n), C.c_uint(16), C.c_uint(ssa_len), C.c_uint(primary), cum.ctypes.data_as(C.c_void_p), ssa.ctypes.data_as(C.c_void_p), a)
            bwt_bytes = np.fromfile(b.decode(), dtype=np.uint8); sa_bytes = np.fromfile(a.decode(), dtype=np.uint8)
        sa_bytes[4:20] = 0
        out[f"{name}_bwt_file"] = bwt_bytes; out[f"{name}_sa_file"] = sa_bytes
    out["sa_unspecified"] = np.array([4, 20], np.uint32)
    np.savez_compressed(os.path.join(OUT, "nvbwt_files.npz"), **out)


CITED_SUFFIXES = (".h", ".cu", ".cpp", ".cuh", ".cmake", ".md", ".txt")


def make_reference_files(tree):
    import json
    n_lines = {}
    for dp, _, files in os.walk(tree):
        for f in files:
            if f.endswith(CITED_SUFFIXES):
                p = os.path.join(dp, f)
                with open(p, errors="ignore") as fh:
                    n_lines[os.path.relpath(p, tree)] = sum(1 for _ in fh)
    with open(os.path.join(OUT, "reference_files.json"), "w") as fh:
        json.dump(n_lines, fh, indent=0, sort_keys=True)


def main():
    if "--only-files" in sys.argv:
        make_reference_files(sys.argv[sys.argv.index("--only-files") + 1]); print("wrote reference_files.json"); return
    if "--only-nvbwt" in sys.argv:
        make_nvbwt_files(); print("wrote nvbwt_files.npz"); return
    assert orc.Ref.available(), "build oracle/_ref first: make -C oracle"
    ref = orc.Ref()
    if "--only-extras" in sys.argv:
        make_extras(ref); print("wrote banded_extras.npz"); return
    make_full(ref)
    make_extras(ref)
    if "--only-full" in sys.argv:
        print("wrote gotoh_full.npz"); return
    rng = np.random.default_rng(20240917)
    out = {}

    # (a) the reference's own asserted problems
    for name, P, T, scheme, band in (("g1", G1_P, G1_T, (2, -1, -1, -1), 7),
                                     ("g2", G2_P, G2_T, (0, -5, -8, -3), 31)):
        p, t = orc.dna(P), orc.dna(T)
        for typ in (0, 1, 2):
            s, x, y, ok = ref.banded_gotoh(band, typ, scheme, p, [0], [len(p)], t, [0], [len(t)])
            out[f"{name}_t{typ}"] = np.array([s[0], x[0], y[0], ok[0]], dtype=np.int64)
    # (b) random problems
    cases = []
    cid = 0
    for band in (3, 5, 7, 15, 31, 63):
        for typ in (0, 1, 2):
            for scheme in ((2, -2, -5, -3), (2, -1, -1, -1), (0, -5, -8, -3), (1, -3, -2, -4)):
                alpha = 4 if cid % 3 else 6          # every third case has text symbols 4,5 (N-like)
                pr = random_problems(rng, 24, band, 40 if band < 31 else 160, alphabet_text=alpha)
                s, x, y, ok = ref.banded_gotoh(band, typ, scheme, *pr)
                for k, v in zip(("pat", "p_off", "p_len", "txt", "t_off", "t_len"), pr):
                    out[f"r{cid}_{k}"] = v
                out[f"r{cid}_res"] = np.stack([s.astype(np.int64), x.astype(np.int64), y.astype(np.int64),
                                               ok.astype(np.int64)])
                cases.append((cid, band, typ) + scheme)
                cid += 1
    out["cases"] = np.array(cases, dtype=np.int64)
    np.savez_compressed(os.path.join(OUT, "banded_gotoh.npz"), **out)

    # (c) FM-index fixtures
    fm = {}
    texts = {
        "rand": rng.integers(0, 4, size=5000).astype(np.uint8),
        "rep": np.tile(np.array([0, 1, 0, 1, 2, 3, 0, 0], np.uint8), 200)[:1531],
        "allA": np.zeros(257, np.uint8),
        "tiny": orc.dna("ACGTTGCA"),
    }
    for name, text in texts.items():
        idx = ref.build_index(text)
        n = len(text)
        nq = 300
        lens = rng.integers(1, 24, size=nq).astype(np.uint32)
        offs = np.zeros(nq, np.uint32)
        qs = []
        o = 0
        for i in range(nq):
            L = int(lens[i])
            if i % 4 != 3 and n > L:
                st = int(rng.integers(0, n - L + 1))
                q = text[st:st + L].copy()
            else:
                q = rng.integers(0, 4, size=L).astype(np.uint8)
            # NOTE: no N's here: nvbio::match() tests `c > 4` (fmindex_inl.h:329), so a symbol 4 indexes
            # occ/L2 out of bounds (it segfaults); the N -> (1,0) rule is nvBowtie's match_range
            # (mapping_inl.h:90) and is pinned by the oracle tests instead.
            qs.append(q); offs[i] = o; o += L
        q = np.concatenate(qs)
        ranges, _ = ref.match(idx, q, offs, lens)
        rows = rng.integers(0, n + 1, size=400).astype(np.uint32)
        rows[:3] = (0, idx.primary, n)
        pos = ref.locate(idx, rows)
        k = rng.integers(0, n + 1, size=500).astype(np.uint32)
        k[:3] = (0xFFFFFFFF, n, idx.primary)
        c = rng.integers(0, 4, size=500).astype(np.uint8)
        rk = ref.rank(idx, k, c)
        for key, v in dict(text=text, sa=idx.sa, bwt_occ=idx.bwt_occ, L2=idx.L2, ssa=idx.ssa,
                           primary=np.array([idx.primary], np.uint32), q=q, q_off=offs, q_len=lens,
                           ranges=ranges, rows=rows, pos=pos, rank_k=k, rank_c=c, rank_out=rk).items():
            fm[f"{name}_{key}"] = v
    fm["count_table"] = ref.count_table()
    np.savez_compressed(os.path.join(OUT, "fmindex.npz"), **fm)
    make_nvbowtie(ref)
    make_generic_rank(ref)
    make_nvbwt_files()
    print("wrote", os.listdir(OUT))


if __name__ == "__main__":
    main()
