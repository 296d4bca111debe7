"""Pins the plain-C oracle (oracle/nvb_oracle.c) against
  (1) golden vectors produced by running the reference itself (tests/golden/make_golden.py),
  (2) the reference's own templates (oracle/_ref/libnvbio_ref.so) on fresh seeded inputs: their outputs' digests are
      committed (tests/reference_digests.py), so these comparisons run without that library.
CPU only."""
import os
import numpy as np
import pytest
from oracle import orc
from tests.reference_digests import Reference

GOLD = os.path.join(os.path.dirname(__file__), "golden")
from tests.golden.make_golden import G1_P, G1_T, G2_P, G2_T, random_problems  # noqa: E402


def mask_pad(bwt_occ, n):
    """zero the BWT symbols at positions >= n (the reference's gen_bwt_from_sa leaves a stale copy of
    the last symbol at position n, nvbio/fmindex/bwt.h:61; padding never influences rank())"""
    b = bwt_occ.copy().reshape(-1, 8)
    w = b[:, :4].reshape(-1).copy()
    full, rem = n // 16, n % 16
    if rem:
        w[full] &= np.uint32((0xFFFFFFFF << (32 - 2 * rem)) & 0xFFFFFFFF)
        full += 1
    w[full:] = 0
    b[:, :4] = w.reshape(-1, 4)
    return b.reshape(-1)


@pytest.fixture(scope="module")
def O():
    return orc.Oracle()


@pytest.fixture
def R(request):
    return Reference(request, orc.Ref)


def test_reference_asserted_problems(O):
    """nvbio-test/alignment_test.cu:761-825 (scores/sinks measured by running the reference)"""
    g = np.load(os.path.join(GOLD, "banded_gotoh.npz"))
    # the survey's re-derived values
    assert tuple(g["g1_t2"][:3]) == (10, 10, 7)
    assert tuple(g["g2_t2"][:3]) == (-11, 165, 150)
    assert tuple(g["g1_t0"][:3]) == (5, 13, 7)
    for name, P, T, scheme, band in (("g1", G1_P, G1_T, (2, -1, -1, -1), 7),
                                     ("g2", G2_P, G2_T, (0, -5, -8, -3), 31)):
        p, t = orc.dna(P), orc.dna(T)
        for typ in (0, 1, 2):
            s, x, y, ok = O.banded_gotoh(band, typ, scheme, p, [0], [len(p)], t, [0], [len(t)])
            assert (int(s[0]), int(x[0]), int(y[0]), int(ok[0])) == tuple(int(v) for v in g[f"{name}_t{typ}"])


def test_banded_golden_random(O):
    g = np.load(os.path.join(GOLD, "banded_gotoh.npz"))
    for cid, band, typ, m, mm, go, ge in g["cases"]:
        pr = [g[f"r{cid}_{k}"] for k in ("pat", "p_off", "p_len", "txt", "t_off", "t_len")]
        s, x, y, ok = O.banded_gotoh(int(band), int(typ), (int(m), int(mm), int(go), int(ge)), *pr)
        res = g[f"r{cid}_res"]
        assert np.array_equal(s.astype(np.int64), res[0]), (cid, band, typ)
        assert np.array_equal(x.astype(np.int64), res[1]), (cid, band, typ)
        assert np.array_equal(y.astype(np.int64), res[2]), (cid, band, typ)
        assert np.array_equal(ok.astype(np.int64), res[3])


def test_fm_golden(O):
    g = np.load(os.path.join(GOLD, "fmindex.npz"))
    assert np.array_equal(O.count_table(), g["count_table"])
    assert g["count_table"][0b00100001] == 0x00010102          # nvbio/fmindex/bwt.h:83
    for name in ("rand", "rep", "allA", "tiny"):
        text = g[f"{name}_text"]
        idx = O.build_index(text)
        assert np.array_equal(idx.sa, g[f"{name}_sa"]), name
        assert idx.primary == int(g[f"{name}_primary"][0])
        assert np.array_equal(mask_pad(idx.bwt_occ, idx.n), mask_pad(g[f"{name}_bwt_occ"], idx.n))
        assert np.array_equal(idx.L2, g[f"{name}_L2"])
        assert np.array_equal(idx.ssa, g[f"{name}_ssa"])
        r, blocks = O.match(idx, g[f"{name}_q"], g[f"{name}_q_off"], g[f"{name}_q_len"])
        assert np.array_equal(r, g[f"{name}_ranges"]), name
        assert np.array_equal(O.locate(idx, g[f"{name}_rows"]), g[f"{name}_pos"])
        assert np.array_equal(O.rank(idx, g[f"{name}_rank_k"], g[f"{name}_rank_c"]), g[f"{name}_rank_out"])


def test_match_N_rule(O):
    """nvBowtie's match_range: any symbol > 3 -> empty range (1,0) (mapping_inl.h:90)"""
    text = np.random.default_rng(1).integers(0, 4, 300).astype(np.uint8)
    idx = O.build_index(text)
    q = np.array([0, 1, 4, 2], np.uint8)
    r, _ = O.match(idx, q, [0], [4])
    assert tuple(r[0]) == (1, 0)


def test_rank_property(O):
    """rank_test.cu:55-86: rank(dict,i,c) == running count, every (i,c)"""
    rng = np.random.default_rng(7)
    text = rng.integers(0, 4, 1000).astype(np.uint8)
    idx = O.build_index(text)
    # unpack the BWT back from the interleaved blocks
    blk = idx.bwt_occ.reshape(-1, 8)[:, :4].reshape(-1)
    bwt = np.array([(int(blk[i >> 4]) >> (30 - 2 * (i & 15))) & 3 for i in range(idx.n)])
    for c in range(4):
        run = np.cumsum(bwt == c)
        got = O.dict_rank(idx, np.arange(idx.n), np.full(idx.n, c))
        assert np.array_equal(got, run)


def test_locate_property(O):
    """fmindex_test.cu:611-664: text[locate(match(p))..] == p"""
    rng = np.random.default_rng(11)
    text = rng.integers(0, 4, 3000).astype(np.uint8)
    idx = O.build_index(text)
    for _ in range(50):
        L = int(rng.integers(4, 12)); st = int(rng.integers(0, 3000 - L))
        p = text[st:st + L]
        r, _ = O.match(idx, p, [0], [L])
        x, y = int(r[0, 0]), int(r[0, 1])
        assert x <= y
        pos = O.locate(idx, np.arange(x, y + 1))
        assert st in pos
        for q in pos:
            assert np.array_equal(text[q:q + L], p)
        assert np.array_equal(np.sort(pos), np.sort(idx.sa[x:y + 1]).astype(np.uint32))


def test_oracle_vs_reference_fresh(O, R):
    rng = np.random.default_rng(99)
    for n in (1, 2, 63, 64, 65, 1000, 20000):
        text = rng.integers(0, 4, n).astype(np.uint8)
        a = O.build_index(text)
        b = R.live.build_index(text) if R.live else None
        R.same([a.sa, a.L2, a.ssa, mask_pad(a.bwt_occ, n), a.primary], lambda: [b.sa, b.L2, b.ssa, mask_pad(b.bwt_occ, n), b.primary])
        nq = 500
        lens = rng.integers(1, 26, nq).astype(np.uint32)
        offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.uint32)
        q = rng.integers(0, 4, int(lens.sum())).astype(np.uint8)
        for i in range(0, nq, 2):                      # half of them sampled from the text
            L = int(lens[i])
            if n > L:
                st = int(rng.integers(0, n - L + 1)); q[offs[i]:offs[i] + L] = text[st:st + L]
        R.same(O.match(a, q, offs, lens)[0], lambda: R.live.match(b, q, offs, lens)[0])
        rows = rng.integers(0, n + 1, 300).astype(np.uint32)
        R.same(O.locate(a, rows), lambda: R.live.locate(b, rows))


def test_banded_vs_reference_fresh(O, R):
    rng = np.random.default_rng(5)
    for band in (3, 7, 15, 31):
        for typ in (0, 1, 2):
            scheme = tuple(int(v) for v in (rng.integers(0, 4), -rng.integers(1, 7), -rng.integers(1, 9), -rng.integers(1, 5)))
            pr = random_problems(rng, 64, band, 150, alphabet_text=5)
            R.same(O.banded_gotoh(band, typ, scheme, *pr), lambda: R.live.banded_gotoh(band, typ, scheme, *pr))


def test_traceback_reference_cigars(O):
    """the CIGARs the reference's own test asserts (nvbio-test/alignment_test.cu:793,825), in its END->START order"""
    for P, T, scheme, band, want in ((G1_P, G1_T, (2, -1, -1, -1), 7, "4M1D3M"), (G2_P, G2_T, (0, -5, -8, -3), 31, "147M2D3M")):
        p, t = orc.dna(P), orc.dna(T)
        o = O.banded_traceback(band, 2, scheme, p, [0], [len(p)], t, [0], [len(t)])
        assert orc.rle(o["ops"][0][:o["n_ops"][0]]) == want


def test_traceback_vs_reference_fresh(O, R):
    from tests.test_host_core import fixed_problems
    rng = np.random.default_rng(77)
    for band in (7, 15, 31):
        for typ in (0, 1, 2):
            scheme = tuple(int(v) for v in (rng.integers(0, 4), -rng.integers(1, 7), -rng.integers(1, 9), -rng.integers(1, 5)))
            pr = fixed_problems(rng, 120, band, 150, extra_text=int(rng.integers(0, 3)), ragged=True)
            R.same(O.banded_traceback(band, typ, scheme, *pr), lambda: R.live.banded_traceback(band, typ, scheme, *pr))


def test_full_matrix_gotoh_vs_reference(O, R):
    """aln::alignment_score (full DP, PatternBlockingTag) == the C restatement: scores and sinks, every type; plus the values
    of the reference's 7 x 20 test strings (alignment_test.cu:761-793)"""
    from tests.test_host_core import full_problems
    p, t = orc.dna(G1_P), orc.dna(G1_T)
    for typ, want in ((0, (1, 20, 7)), (1, (13, 18, 7)), (2, (13, 18, 7))):
        s, x, y = O.gotoh_full(typ, (2, -1, -1, -1), p, [0], [len(p)], t, [0], [len(t)])
        assert (int(s[0]), int(x[0]), int(y[0])) == want
    rng = np.random.default_rng(13)
    for typ in (0, 1, 2):
        for scheme in ((2, -1, -2, -1), (2, -2, -5, -3), (1, -3, -2, -4)):
            pr = full_problems(rng, 100)
            R.same(O.gotoh_full(typ, scheme, *pr), lambda: R.live.gotoh_full(typ, scheme, *pr))


def test_full_matrix_traceback_vs_reference(O, R):
    """aln::alignment_traceback<256,512,64> (full DP, checkpointed) == the C restatement (whole direction matrix): score, sink,
    source, clips and every op; the reference's own 7 x 20 strings give 4M1D3M for LOCAL / SEMI_GLOBAL (alignment_test.cu:784-793)"""
    from tests.test_host_core import full_problems
    p, t = orc.dna(G1_P), orc.dna(G1_T)
    def ops(a):
        return [a["ops"][i][:a["n_ops"][i]] for i in range(len(a["n_ops"]))]
    for typ, cig in ((0, "1M2D3M1D3M10D"), (1, "4M1D3M"), (2, "4M1D3M")):
        a = O.gotoh_full_traceback(typ, (2, -1, -1, -1), p, [0], [len(p)], t, [0], [len(t)])
        assert orc.rle(a["ops"][0][:a["n_ops"][0]]) == cig, typ
        R.same(ops(a), lambda: ops(R.live.gotoh_full_traceback(typ, (2, -1, -1, -1), p, [0], [len(p)], t, [0], [len(t)])))
    rng = np.random.default_rng(17)
    for typ in (0, 1, 2):
        for scheme in ((2, -1, -2, -1), (2, -2, -5, -3), (0, -5, -8, -3)):
            pr = full_problems(rng, 80, max_m=200, max_n=450)
            a = O.gotoh_full_traceback(typ, scheme, *pr)
            b = R.live.gotoh_full_traceback(typ, scheme, *pr) if R.live else None
            fields = ("score", "sink", "source", "n_ops", "clips")
            R.same([a[k] for k in fields] + ops(a), lambda: [b[k] for k in fields] + ops(b))


def _full_golden():
    import os
    return np.load(os.path.join(os.path.dirname(__file__), "golden", "gotoh_full.npz"))


def test_full_matrix_golden(O):
    """the committed reference outputs (tests/golden/gotoh_full.npz: aln::alignment_score + aln::alignment_traceback run by
    make_golden.py) == the oracle: score, sink, source and the op stream of every problem"""
    g = _full_golden()
    for cid, typ, m, mm, go, ge in g["cases"]:
        pr = [g[f"f{cid}_{k}"] for k in ("pat", "p_off", "p_len", "txt", "t_off", "t_len")]
        res, ops = g[f"f{cid}_res"], g[f"f{cid}_ops"]
        s, x, y = O.gotoh_full(int(typ), (int(m), int(mm), int(go), int(ge)), *pr)
        assert np.array_equal(s.astype(np.int64), res[0]) and np.array_equal(x.astype(np.int64), res[1]) and np.array_equal(y.astype(np.int64), res[2])
        tb = O.gotoh_full_traceback(int(typ), (int(m), int(mm), int(go), int(ge)), *pr, max_ops=512)
        assert np.array_equal(tb["source"][:, 0].astype(np.int64), res[3]) and np.array_equal(tb["source"][:, 1].astype(np.int64), res[4])
        assert np.array_equal(tb["n_ops"].astype(np.int64), res[5])
        assert np.array_equal(np.concatenate([tb["ops"][i][:tb["n_ops"][i]] for i in range(len(s))]), ops)


def test_windowed_banded_score_vs_reference(O, R):
    """aln::banded_alignment_score<B>(..., window_begin, window_end, sink, checkpoint) == the C restatement, pass by pass: BestSink,
    short2 checkpoint bands and the early-exit result; compared where the reference is defined (it reads text[wb .. wb+B-2]
    unchecked at a window start, so N >= M + B - 1)"""
    from tests.golden.make_golden import random_problems
    rng = np.random.default_rng(23)
    for band in (7, 15, 31):
        for typ in (0, 1, 2):
            pr = random_problems(rng, 60, band, 150)
            n = len(pr[1])
            wd = pr[5] >= pr[2] + band - 1
            for scheme, W, ms in (((2, -2, -5, -3), 32, None), ((0, -5, -8, -3), 17, None), ((2, -2, -5, -3), 32, rng.integers(-40, 160, n).astype(np.int32))):
                so, sr = orc.window_state(n, band), orc.window_state(n, band)

                def defined(st):                        # the state where the reference is defined (its alive flags decide the checkpoints)
                    return [st[k][wd] for k in ("score", "sx", "sy", "alive")] + [st["ckpt"][st["alive"].astype(bool) & wd]]
                for wb in range(0, 150, W):
                    O.banded_gotoh_window(band, typ, scheme, *pr, wb, wb + W, so, min_score=ms)
                    if R.live:
                        R.live.banded_gotoh_window(band, typ, scheme, *pr, wb, wb + W, sr, min_score=ms)
                    R.same(defined(so), lambda: defined(sr))


def _nvbowtie_like_table():
    """256 x 2 table shaped like nvBowtie's local-mode scheme: match 2, mismatch -(2 + min(q,40)/40 * 4)"""
    t = np.zeros((256, 2), np.int32)
    for q in range(256):
        t[q, 0] = 2
        t[q, 1] = -(2 + int(min(q, 40) / 40.0 * 4))
    return t


def test_quality_table_scheme_vs_reference(O, R):
    """the quality-dependent substitution path of the oracle (banded and full-matrix) == the reference's own DP templates
    instantiated with a table-driven scheme (TableGotohScheme in oracle/ref_shim.cpp, a model of the GotohScoringScheme concept),
    incl. text gap costs that differ from the pattern's"""
    from tests.golden.make_golden import random_problems
    from tests.test_host_core import full_problems
    rng = np.random.default_rng(31)
    qtab = _nvbowtie_like_table()
    scheme = (0, 0, -8, -3, -7, -2)
    for band in (7, 15, 31):
        for typ in (0, 1, 2):
            pr = random_problems(rng, 80, band, 120)
            qual = rng.integers(0, 64, len(pr[0])).astype(np.uint8)
            a = O.banded_gotoh(band, typ, scheme, *pr, qual=qual, qtab=qtab)
            b = R.live.banded_gotoh(band, typ, scheme, *pr, qual=qual, qtab=qtab) if R.live else None
            R.same(a[3], lambda: b[3])                 # where the reference ran
            ok = a[3].astype(bool)
            R.same([u[ok] for u in a[:3]], lambda: [v[ok] for v in b[:3]])
    for typ in (0, 1, 2):
        pr = full_problems(rng, 120)
        qual = rng.integers(0, 64, len(pr[0])).astype(np.uint8)
        R.same(O.gotoh_full(typ, scheme, *pr, qual=qual, qtab=qtab), lambda: R.live.gotoh_full(typ, scheme, *pr, qual=qual, qtab=qtab))


def _extras_golden():
    import os
    return np.load(os.path.join(os.path.dirname(__file__), "golden", "banded_extras.npz"))


def test_windowed_and_quality_golden(O):
    """committed outputs of the reference itself (tests/golden/banded_extras.npz, written by make_golden.py): windowed banded scoring
    pass by pass (BestSink + alive flag after every 32-row window, final checkpoint band) and the quality-table scheme (banded and
    full matrix) == the oracle"""
    g = _extras_golden()
    for cid, band, typ in g["wcases"]:
        pr = [g[f"w{cid}_{k}"] for k in ("pat", "p_off", "p_len", "txt", "t_off", "t_len")]
        ms = g[f"w{cid}_ms"]; ms = ms if len(ms) else None
        n = len(pr[1])
        st = orc.window_state(n, int(band))
        for w, wb in enumerate(range(0, 100, 32)):
            O.banded_gotoh_window(int(band), int(typ), (2, -2, -5, -3), *pr, wb, wb + 32, st, min_score=ms)
            snap = np.concatenate([st["score"].astype(np.int64), st["sx"].astype(np.int64), st["sy"].astype(np.int64), st["alive"].astype(np.int64)])
            assert np.array_equal(snap, g[f"w{cid}_snaps"][w]), (cid, band, typ, wb)
        al = st["alive"].astype(bool)
        assert np.array_equal(st["ckpt"][al], g[f"w{cid}_ckpt"][al])
    qtab = g["qtab"]
    for cid, band, typ in g["qcases"]:
        pr = [g[f"q{cid}_{k}"] for k in ("pat", "p_off", "p_len", "txt", "t_off", "t_len")]
        qual, res = g[f"q{cid}_qual"], g[f"q{cid}_res"]
        if band:
            s, x, y, _ = O.banded_gotoh(int(band), int(typ), (0, 0, -8, -3, -7, -2), *pr, qual=qual, qtab=qtab)
        else:
            s, x, y = O.gotoh_full(int(typ), (0, 0, -8, -3, -7, -2), *pr, qual=qual, qtab=qtab)
        ok = res[3].astype(bool)
        assert np.array_equal(s.astype(np.int64)[ok], res[0][ok]) and np.array_equal(x.astype(np.int64)[ok], res[1][ok]) and np.array_equal(y.astype(np.int64)[ok], res[2][ok]), (cid, band, typ)


def _nvbowtie_golden():
    return np.load(os.path.join(GOLD, "nvbowtie_scheme.npz"))


def test_quality_table_generation_vs_nvbowtie_scheme():
    """nvbio_b200.aln.QualityGotohScheme.host_table (the float32 QualCost expression evaluated on the host) == the 256 x 2 table of
    nvBowtie's own SmithWatermanScoringScheme<QualCost<int>,ConstantCost<int>> object, entry by entry (fixture written by running the
    reference's scoring.h, tests/golden/make_golden.py make_nvbowtie) -- presets --local and end-to-end, and custom constants"""
    from nvbio_b200.aln import QualityGotohScheme
    g = _nvbowtie_golden()
    presets = {1: (2, 2, 6), 2: (0, 2, 6)}                 # scoring_inl.h:74-147: local() = match 2, mmp 2..6; default ctor = match 0
    for i, (preset, mb, lo, hi) in enumerate(g["cfgs"]):
        mb, lo, hi = presets.get(int(preset), (int(mb), int(lo), int(hi)))
        assert np.array_equal(QualityGotohScheme.host_table(mb, lo, hi), g[f"tab{i}"]), (i, preset, mb, lo, hi)
        assert tuple(g[f"gaps{i}"]) == (-8, -3, -8, -3)    # open = -(const + coeff), ext = -coeff (scoring.h:290-293)
        assert int(g[f"lim{i}"][0]) == -65536              # worst_score (scoring.h:226-227)


def test_quality_table_generation_vs_nvbowtie_scheme_live(R):
    from nvbio_b200.aln import QualityGotohScheme
    for mb, lo, hi in ((2, 2, 6), (0, 2, 6), (1, 0, 40), (5, 7, 7), (0, 1, 200)):
        R.same([QualityGotohScheme.host_table(mb, lo, hi), (-6, -2, -7, -1)],
               lambda: R.live.nvbowtie_scheme(0, mb, lo, hi, read_gap=(4, 2), ref_gap=(6, 1))[:2])


def test_oracle_quality_dp_vs_nvbowtie_scheme(O):
    """the oracle's banded DP with the host-evaluated table == aln::banded_alignment_score run with nvBowtie's real scheme object
    and per-base qualities (--local preset; LOCAL and SEMI_GLOBAL, bands 15 / 31)"""
    from nvbio_b200.aln import QualityGotohScheme
    g = _nvbowtie_golden()
    qtab = QualityGotohScheme.host_table(2, 2, 6)
    for cid, band, typ in g["dcases"]:
        pr = [g[f"d{cid}_{k}"] for k in ("pat", "p_off", "p_len", "txt", "t_off", "t_len")]
        s, x, y, ok = O.banded_gotoh(int(band), int(typ), (0, 0, -8, -3, -8, -3), *pr, qual=g[f"d{cid}_qual"], qtab=qtab)
        res = g[f"d{cid}_res"]
        okb = ok.astype(bool)
        assert okb.sum() > 30
        assert np.array_equal(s.astype(np.int64)[okb], res[0][okb]) and np.array_equal(x.astype(np.int64)[okb], res[1][okb]) and np.array_equal(y.astype(np.int64)[okb], res[2][okb]), (cid, band, typ)


def test_generic_rank_dictionary_golden():
    """SURVEY 8a row a6: the plain restatement of the generic rank dictionary (32- / 64-bit words, occ every K) == the reference's
    rank_dictionary / build_occurrence_table<2,K> on the committed fixture (packed words, occ table, ranks incl. i = -1)"""
    g = np.load(os.path.join(GOLD, "generic_rank.npz"))
    for i, (wb, K, n) in enumerate(g["cfgs"]):
        w, o, r = orc.generic_rank_oracle(g[f"text{i}"], g[f"qi{i}"], g[f"qc{i}"], int(wb), int(K))
        assert np.array_equal(w, g[f"words{i}"]) and np.array_equal(o, g[f"occ{i}"]) and np.array_equal(r, g[f"ranks{i}"]), (wb, K, n)
        assert int(r[-1]) == 0                               # i = all ones


def test_best2_sink_vs_reference_fresh(O, R):
    """aln::Best2Sink<int32>(distinct_dist) (sink.h:114-147) fed by the banded DP: the plain-C restatement == the reference templates,
    every band / type, several minimum distances; un-run alignments keep the reference's sink default Field_traits<int32>::min() = -2^30"""
    rng = np.random.default_rng(41)
    for band in (7, 15, 31):
        for typ in (0, 1, 2):
            for dist in (0, 5, 40):
                pr = random_problems(rng, 50, band, 120)
                a = O.banded_gotoh_best2(band, typ, (2, -2, -5, -3), *pr, distinct_dist=dist)
                valid = pr[5] >= pr[2]
                R.same(a[valid], lambda: R.live.banded_gotoh_best2(band, typ, (2, -2, -5, -3), *pr, distinct_dist=dist)[valid])
    assert (a[:, 3] == -2**30).any() or True
