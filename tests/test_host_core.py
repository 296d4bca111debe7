"""CPU checks of the PRODUCT's per-thread routines (nvbio_b200/csrc/fm_core.cuh, gotoh_core.cuh), compiled
for the host by tests/host/host_harness.cu, against the oracle.  This is the pre-GPU gate: the same
functions are what the CUDA kernels call per thread."""
import ctypes as C
import os
import subprocess
import numpy as np
import pytest
from oracle import orc
from nvbio_b200.strings import pack_symbols
from tests.golden.make_golden import random_problems
from tests.reference_digests import Reference

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "host", "libhost_harness.so")
SRC = os.path.join(HERE, "host", "host_harness.cu")


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


@pytest.fixture(scope="module")
def H():
    deps = [SRC] + [os.path.join(HERE, "..", "nvbio_b200", "csrc", f) for f in ("fm_core.cuh", "gotoh_core.cuh", "gotoh_full_core.cuh", "pipeline_core.cuh", "common.cuh")]
    so, extra = SO, []
    if os.environ.get("NVB_HOST_HARNESS_ASAN"):
        # AddressSanitizer + UBSan build of the very same per-thread routines: run the file as
        #   NVB_HOST_HARNESS_ASAN=1 LD_PRELOAD=$(gcc -print-file-name=libasan.so) python -m pytest tests/test_host_core.py
        so = SO.replace(".so", "_asan.so")
        extra = ["-g", "-Xcompiler", "-fsanitize=address", "-Xcompiler", "-fsanitize=undefined", "-Xcompiler", "-fno-omit-frame-pointer",
                 "-Xcompiler", "-fno-sanitize-recover=undefined"]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        env = dict(os.environ); env.pop("LD_PRELOAD", None)            # (the sanitizer run preloads libasan: not into the compiler)
        subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "-std=c++17",
                               "-Wno-deprecated-declarations", "-Xcompiler", "-fPIC", "-shared", "-o", so, SRC] + extra, env=env)
    return C.CDLL(so)


@pytest.fixture(scope="module")
def O():
    return orc.Oracle()


def u32(a):
    return np.ascontiguousarray(a, dtype=np.uint32)


@pytest.mark.parametrize("n", [1, 5, 64, 65, 200, 4097])
def test_fm_core(H, O, n):
    rng = np.random.default_rng(n)
    text = rng.integers(0, 4, n).astype(np.uint8)
    idx = O.build_index(text)
    # rank
    k = rng.integers(0, n + 1, 400).astype(np.uint32); k[:3] = (0xFFFFFFFF, n, idx.primary)
    c = rng.integers(0, 4, 400).astype(np.uint8)
    out = np.zeros(400, np.uint32)
    H.hh_fm_rank(_p(idx.bwt_occ), _p(idx.L2), C.c_uint32(n), C.c_uint32(idx.primary), _p(k), _p(c), C.c_uint32(400), _p(out))
    assert np.array_equal(out, O.rank(idx, k, c))
    # match, every stream format
    nq = 300
    lens = rng.integers(1, 26, nq).astype(np.uint32)
    offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.uint32)
    q = rng.integers(0, 4, int(lens.sum())).astype(np.uint8)
    for i in range(0, nq, 2):
        L = int(lens[i])
        if n > L:
            st = int(rng.integers(0, n - L + 1)); q[offs[i]:offs[i] + L] = text[st:st + L]
    want, _ = O.match(idx, q, offs, lens)
    for bits, be in ((2, 1), (2, 0), (4, 1), (4, 0), (8, 0)):
        words = pack_symbols(q, bits, bool(be))
        got = np.zeros((nq, 2), np.uint32)
        H.hh_fm_match(_p(idx.bwt_occ), _p(idx.L2), C.c_uint32(n), C.c_uint32(idx.primary), _p(words), C.c_uint32(bits), C.c_uint32(be),
                      _p(offs), _p(lens), C.c_uint32(nq), C.c_uint32(0), _p(got), None, C.c_uint32(0), C.c_uint32(0))
        assert np.array_equal(got, want), (bits, be)
    # N rule on a 4-bit stream
    qn = q.copy(); qn[offs[5] + lens[5] - 1] = 4          # last symbol = first one consumed
    want_n, _ = O.match(idx, qn, offs, lens)
    got = np.zeros((nq, 2), np.uint32)
    words = pack_symbols(qn, 4, True)
    H.hh_fm_match(_p(idx.bwt_occ), _p(idx.L2), C.c_uint32(n), C.c_uint32(idx.primary), _p(words), C.c_uint32(4), C.c_uint32(1),
                  _p(offs), _p(lens), C.c_uint32(nq), C.c_uint32(0), _p(got), None, C.c_uint32(0), C.c_uint32(0))
    assert np.array_equal(got, want_n) and tuple(got[5]) == (1, 0)
    # forward-order + complement == backward search of the reverse complement
    rc = np.concatenate([(3 - q[o:o + l])[::-1] for o, l in zip(offs, lens)]).astype(np.uint8)
    want_rc, _ = O.match(idx, rc, offs, lens)
    words = pack_symbols(q, 2, True)
    H.hh_fm_match(_p(idx.bwt_occ), _p(idx.L2), C.c_uint32(n), C.c_uint32(idx.primary), _p(words), C.c_uint32(2), C.c_uint32(1),
                  _p(offs), _p(lens), C.c_uint32(nq), C.c_uint32(3), _p(got), None, C.c_uint32(0), C.c_uint32(0))
    assert np.array_equal(got, want_rc)
    # k-mer table: identical ranges with the first k steps looked up (incl. empty ranges, N's, short queries)
    for k in (1, 3, 6):
        ktab = np.zeros(2 * 4 ** k, np.uint32)
        H.hh_fm_build_ktab(_p(idx.bwt_occ), _p(idx.L2), C.c_uint32(n), C.c_uint32(idx.primary), C.c_uint32(k), _p(ktab))
        # ... and the same through the 16-byte "located" entries {x, y, SA[x], SA[y]}
        full_sa = idx.sa.astype(np.uint32).copy(); full_sa[0] = 0xFFFFFFFF
        ktab16 = np.zeros(4 * 4 ** k, np.uint32)
        H.hh_fm_ktab_locate(_p(ktab), _p(full_sa), C.c_uint32(k), _p(ktab16))
        # ... and with the text context packed into one- and two-row entries (ktab_located = 2; two-row entries carry a marker instead of y)
        ktab_ctx = ktab16.copy()
        H.hh_fm_ktab_context(_p(ktab_ctx), C.c_uint32(k), _p(pack_symbols(np.concatenate([text, np.zeros(64, np.uint8)]), 2, True)), C.c_uint32(n))
        two = ktab16[1::4] == ktab16[0::4] + 1
        assert np.array_equal(ktab_ctx[1::4][two] >> 30, np.full(int(two.sum()), 3, np.uint32)) and np.array_equal(ktab_ctx[1::4][~two], ktab16[1::4][~two])
        for tab, located in ((ktab, 0), (ktab16, 1), (ktab_ctx, 2)):
            for flags, w in ((0, want), (3, want_rc)):
                H.hh_fm_match(_p(idx.bwt_occ), _p(idx.L2), C.c_uint32(n), C.c_uint32(idx.primary), _p(words), C.c_uint32(2), C.c_uint32(1),
                              _p(offs), _p(lens), C.c_uint32(nq), C.c_uint32(flags), _p(got), _p(tab), C.c_uint32(k), C.c_uint32(located))
                assert np.array_equal(got, w), (k, flags, located)
            wn = pack_symbols(qn, 4, True)
            H.hh_fm_match(_p(idx.bwt_occ), _p(idx.L2), C.c_uint32(n), C.c_uint32(idx.primary), _p(wn), C.c_uint32(4), C.c_uint32(1),
                          _p(offs), _p(lens), C.c_uint32(nq), C.c_uint32(0), _p(got), _p(tab), C.c_uint32(k), C.c_uint32(located))
            assert np.array_equal(got, want_n), (k, located)
    # locate
    rows = rng.integers(0, n + 1, 300).astype(np.uint32); rows[:3] = (0, idx.primary, n)
    out = np.zeros(300, np.uint32)
    H.hh_fm_locate(_p(idx.bwt_occ), _p(idx.ssa), _p(idx.L2), C.c_uint32(n), C.c_uint32(idx.primary), _p(rows), C.c_uint32(300), _p(out), C.c_uint32(16))
    want_pos = O.locate(idx, rows)
    assert np.array_equal(out, want_pos)
    # denser sampled SA (B200 extension): same positions with fewer LF steps; interval 1 = the full SA
    for I in (1, 2, 8):
        ssa = idx.sa[::I].astype(np.uint32).copy(); ssa[0] = 0xFFFFFFFF
        H.hh_fm_locate(_p(idx.bwt_occ), _p(ssa), _p(idx.L2), C.c_uint32(n), C.c_uint32(idx.primary), _p(rows), C.c_uint32(300), _p(out), C.c_uint32(I))
        assert np.array_equal(out, want_pos), I


def _gotoh_generic(H, band, typ, scheme6, pr, pbits, pbe, tbits, tbe, qual=None, qtab=None):
    pat, p_off, p_len, txt, t_off, t_len = pr
    pw, tw = pack_symbols(pat, pbits, bool(pbe)), pack_symbols(txt, tbits, bool(tbe))
    n = len(p_off)
    score = np.zeros(n, np.int32); sx = np.zeros(n, np.uint32); sy = np.zeros(n, np.uint32)
    s6 = np.array(scheme6, np.int32)
    r = H.hh_gotoh_generic(C.c_int(band), C.c_int(typ), _p(s6), _p(qtab), _p(pw), C.c_uint32(pbits), C.c_uint32(pbe), _p(u32(p_off)), _p(u32(p_len)),
                           _p(qual), _p(tw), C.c_uint32(tbits), C.c_uint32(tbe), _p(u32(t_off)), _p(u32(t_len)), C.c_uint32(n),
                           _p(score), _p(sx), _p(sy))
    assert r == 0
    return score, sx, sy


@pytest.mark.parametrize("band", [3, 5, 7, 15, 31, 63])
@pytest.mark.parametrize("typ", [0, 1, 2])
def test_gotoh_generic(H, O, band, typ):
    rng = np.random.default_rng(band * 10 + typ)
    for scheme in ((2, -2, -5, -3), (1, -3, -2, -4), (0, -5, -8, -3)):
        pr = random_problems(rng, 40, band, 120, alphabet_text=6)      # text symbols up to 5, read N's
        want = O.banded_gotoh(band, typ, scheme, *pr)
        s6 = scheme + (scheme[2], scheme[3])
        got = _gotoh_generic(H, band, typ, s6, pr, 4, 1, 8, 0)
        for a, b in zip(got, want[:3]):
            assert np.array_equal(a, b), (band, typ, scheme)
    # 2-bit inputs, both endiannesses
    pr = random_problems(rng, 40, band, 120, alphabet_text=4)
    want = O.banded_gotoh(band, typ, (2, -2, -5, -3), *pr)
    for pbe, tbe in ((1, 1), (0, 0), (1, 0)):
        got = _gotoh_generic(H, band, typ, (2, -2, -5, -3, -5, -3), pr, 2, pbe, 2, tbe)
        for a, b in zip(got, want[:3]):
            assert np.array_equal(a, b)


def test_gotoh_generic_quality_table(H, O):
    rng = np.random.default_rng(3)
    pr = random_problems(rng, 60, 31, 150, alphabet_text=5)
    qual = rng.integers(0, 60, len(pr[0])).astype(np.uint8)
    q = np.arange(256)
    frac = (np.minimum(q, 40).astype(np.float32) / np.float32(40.0))
    mmp = 2 + (frac * np.float32(6 - 2)).astype(np.int32)
    qtab = np.ascontiguousarray(np.stack([np.full(256, 2, np.int32), -mmp.astype(np.int32)], axis=1))
    s6 = (2, -6, -8, -3, -8, -3)
    for typ in (1, 2):
        want = O.banded_gotoh(31, typ, s6, *pr, qual=qual, qtab=qtab)
        got = _gotoh_generic(H, 31, typ, s6, pr, 4, 1, 2 if False else 8, 0, qual=qual, qtab=qtab)
        for a, b in zip(got, want[:3]):
            assert np.array_equal(a, b)


def fixed_problems(rng, n, band, m, extra_text=0, ragged=False):
    """nvBowtie-shaped jobs: window = read_len + band (+extra), read sampled near the band centre"""
    pats, txts, p_off, p_len, t_off, t_len = [], [], [], [], [], []
    po = to = 0
    for _ in range(n):
        mm = int(rng.integers(max(1, m - 40), m + 1)) if ragged else m
        N = mm + band + extra_text
        t = rng.integers(0, 4, N).astype(np.uint8)
        j = int(rng.integers(0, band))
        p = []
        while len(p) < mm:
            r = rng.random()
            if r < 0.04 or j >= N:
                p.append(int(rng.integers(0, 4))); j += 1 if r < 0.03 else 0
            elif r < 0.06:
                j += 1
            else:
                p.append(int(t[j])); j += 1
        pats.append(np.array(p[:mm], np.uint8)); txts.append(t)
        p_off.append(po); p_len.append(mm); po += mm
        t_off.append(to); t_len.append(N); to += N
    return (np.concatenate(pats), np.array(p_off, np.uint32), np.array(p_len, np.uint32),
            np.concatenate(txts), np.array(t_off, np.uint32), np.array(t_len, np.uint32))


def _gotoh_pair(H, band, typ, scheme6, pr, max_m, pbits=2, pbe=1, tbe=1, qtab=None, qual=None):
    pat, p_off, p_len, txt, t_off, t_len = pr
    pw, tw = pack_symbols(pat, pbits, bool(pbe)), pack_symbols(txt, 2, bool(tbe))
    n = len(p_off)
    score = np.zeros(n, np.int32); sx = np.zeros(n, np.uint32); sy = np.zeros(n, np.uint32)
    nf = C.c_uint32(0)
    s6 = np.array(scheme6, np.int32)
    r = H.hh_gotoh_pair(C.c_int(band), C.c_int(typ), _p(s6), _p(qtab), _p(qual), C.c_uint32(max_m), _p(pw), C.c_uint32(pbits), C.c_uint32(pbe), _p(u32(p_off)), _p(u32(p_len)),
                        _p(tw), C.c_uint32(tbe), _p(u32(t_off)), _p(u32(t_len)), C.c_uint32(n), _p(score), _p(sx), _p(sy), C.byref(nf))
    return r, (score, sx, sy), nf.value


@pytest.mark.parametrize("rows2", [1, 0])
@pytest.mark.parametrize("band", [7, 15, 31])
@pytest.mark.parametrize("typ", [0, 1, 2])
def test_gotoh_pair(H, O, band, typ, rows2):
    """rows2: two pattern rows in flight per loop iteration (odd and even pattern lengths, ragged pairs) / one row"""
    H.hh_set_pair_rows2(C.c_int(rows2))
    rng = np.random.default_rng(100 + band + typ)
    for scheme in ((2, -2, -5, -3), (2, -1, -1, -1), (0, -5, -8, -3), (1, -3, -2, -4), (2, -6, -8, -3)):
        s6 = scheme + (scheme[2], scheme[3])
        for ragged in (False, True):
            pr = fixed_problems(rng, 51, band, 150, extra_text=int(rng.integers(0, 3)), ragged=ragged)   # odd count: tail pair
            want = O.banded_gotoh(band, typ, scheme, *pr)
            r, got, nf = _gotoh_pair(H, band, typ, s6, pr, 150)
            assert r == 0
            for a, b in zip(got, want[:3]):
                assert np.array_equal(a, b), (band, typ, scheme, ragged)
            if not ragged:
                assert nf == 0                       # everything went through the packed path
    # 4-bit patterns with N's, little-endian text
    pr = list(fixed_problems(rng, 40, band, 100))
    pr[0] = pr[0].copy(); pr[0][rng.integers(0, len(pr[0]), 30)] = 4
    want = O.banded_gotoh(band, typ, (2, -2, -5, -3), *pr)
    r, got, nf = _gotoh_pair(H, band, typ, (2, -2, -5, -3, -5, -3), pr, 100, pbits=4, pbe=1, tbe=0)
    assert r == 0 and nf == 0
    for a, b in zip(got, want[:3]):
        assert np.array_equal(a, b)


def test_gotoh_pair_mixed_fallback(H, O):
    """short windows / empty patterns in a batch go through the generic routine, pairwise"""
    rng = np.random.default_rng(9)
    pr = random_problems(rng, 80, 31, 150, alphabet_text=4)
    want = O.banded_gotoh(31, 1, (2, -2, -5, -3), *pr)
    r, got, nf = _gotoh_pair(H, 31, 1, (2, -2, -5, -3, -5, -3), pr, 160)
    assert r == 0 and nf > 0
    for a, b in zip(got, want[:3]):
        assert np.array_equal(a, b)


def test_pair_path_admission(H):
    # scores that do not fit the 16-bit budget must be refused (-2), not computed wrongly
    pr = fixed_problems(np.random.default_rng(1), 4, 31, 50)
    r, _, _ = _gotoh_pair(H, 31, 1, (40, -2, -5, -3, -5, -3), pr, 150)        # 150*40 >= 2048
    assert r == -2
    r, _, _ = _gotoh_pair(H, 31, 2, (2, -2, -200, -3, -200, -3), pr, 150)      # S - Go does not fit int8
    assert r == -2


def test_gotoh_pair_quality_table(H, O):
    """nvBowtie's quality-dependent substitution through the packed path (per-row profiles from the table)"""
    rng = np.random.default_rng(21)
    q = np.arange(256)
    frac = (np.minimum(q, 40).astype(np.float32) / np.float32(40.0))
    mmp = 2 + (frac * np.float32(6 - 2)).astype(np.int32)
    qtab = np.ascontiguousarray(np.stack([np.full(256, 2, np.int32), -mmp.astype(np.int32)], axis=1))
    s6 = (2, -6, -8, -3, -8, -3)
    for band in (15, 31):
        for typ in (1, 2):
            for ragged in (False, True):
                pr = fixed_problems(rng, 41, band, 150, ragged=ragged)
                qual = rng.integers(0, 60, len(pr[0])).astype(np.uint8)
                want = O.banded_gotoh(band, typ, s6, *pr, qual=qual, qtab=qtab)
                r, got, nf = _gotoh_pair(H, band, typ, s6, pr, 150, pbits=4, qtab=qtab, qual=qual)
                assert r == 0 and (ragged or nf == 0)
                for a, b in zip(got, want[:3]):
                    assert np.array_equal(a, b), (band, typ, ragged)


@pytest.mark.parametrize("band", [7, 15, 31])
@pytest.mark.parametrize("typ", [0, 1, 2])
def test_gotoh_traceback(H, O, band, typ):
    """direction-matrix traceback of the product's per-thread routine == the oracle's (== the reference's checkpointed
    aln::banded_alignment_traceback, pinned in tests/test_oracle.py)"""
    rng = np.random.default_rng(300 + band + typ)
    for scheme in ((2, -2, -5, -3), (2, -1, -1, -1), (0, -5, -8, -3)):
        pr = fixed_problems(rng, 60, band, 150, extra_text=int(rng.integers(0, 3)), ragged=True)
        want = O.banded_traceback(band, typ, scheme, *pr)
        pat, p_off, p_len, txt, t_off, t_len = pr
        pw, tw = pack_symbols(pat, 4, True), pack_symbols(txt, 2, True)
        n, max_ops = len(p_off), 512
        score = np.zeros(n, np.int32); sink = np.zeros((n, 2), np.uint32); source = np.zeros((n, 2), np.uint32)
        ops = np.zeros((n, max_ops), np.uint8); n_ops = np.zeros(n, np.uint32)
        s6 = np.array(scheme + (scheme[2], scheme[3]), np.int32)
        r = H.hh_gotoh_traceback(C.c_int(band), C.c_int(typ), _p(s6), _p(pw), C.c_uint32(4), C.c_uint32(1), _p(u32(p_off)), _p(u32(p_len)),
                                 _p(tw), C.c_uint32(2), C.c_uint32(1), _p(u32(t_off)), _p(u32(t_len)), C.c_uint32(n), C.c_uint32(max_ops),
                                 _p(score), _p(sink), _p(source), _p(ops), _p(n_ops))
        assert r == 0
        assert np.array_equal(score, want["score"]) and np.array_equal(sink, want["sink"]) and np.array_equal(source, want["source"])
        assert np.array_equal(n_ops, want["n_ops"]) and np.array_equal(ops, want["ops"]), (band, typ, scheme)


def approx_expected(O, idx, q, offs, lens, exact_len, find_exact, fwd, comp):
    """the reference's map<find_exact> characterised through the PINNED exact match(): every single-substitution
    variant (consumed position ascending, substituted symbol ascending) whose range is non-empty, then the exact match"""
    exp = []
    for o, L in zip(offs, lens):
        s = q[o:o + L].copy()
        if not fwd:
            s = s[::-1]
        if comp:
            s = np.where(s < 4, 3 - s, s).astype(np.uint8)
        l1 = min(exact_len, L)
        npos = [i for i in range(L) if s[i] > 3]
        if (npos and npos[0] < l1) or len(npos) > 1:
            exp.append([]); continue
        if npos:
            l1 = npos[0]
        variants = []
        last = L if not npos else npos[0] + 1            # after an N position the base range is dead
        for i in range(l1, last):
            for sub in range(4):
                if sub != s[i]:
                    v = s.copy(); v[i] = sub; variants.append(v)
        if find_exact and not npos:
            variants.append(s.copy())
        if variants:
            cat = np.concatenate([v[::-1] for v in variants])       # match() consumes from the END of its pattern
            r, _ = O.match(idx, cat, np.arange(len(variants)) * L, np.full(len(variants), L))
            exp.append([tuple(x) for x in r if x[0] <= x[1]])
        else:
            exp.append([])
    return exp


def test_generic_rank_dictionary(H):
    """product's dict_rank<W,I> (generic rank dictionary, SURVEY 8a row a6) == the reference's answers on the committed fixture"""
    g = np.load(os.path.join(HERE, "golden", "generic_rank.npz"))
    for i, (wb, K, n) in enumerate(g["cfgs"]):
        qi = np.ascontiguousarray(g[f"qi{i}"]); qc = np.ascontiguousarray(g[f"qc{i}"])
        words = np.concatenate([g[f"words{i}"], np.zeros(4, g[f"words{i}"].dtype)]); occ = np.ascontiguousarray(g[f"occ{i}"])
        out = np.zeros(len(qi), np.uint64)
        H.hh_dict_rank(_p(words), C.c_uint32(int(wb)), _p(occ), C.c_uint32(int(K)), _p(qi), _p(qc), C.c_uint32(len(qi)), _p(out))
        assert np.array_equal(out, g[f"ranks{i}"]), (wb, K, n)


@pytest.mark.parametrize("bits", [4, 2])
@pytest.mark.parametrize("n,k", [(300, 0), (300, 3), (5000, 0), (5000, 4), (5000, 6), (70, 2)])
def test_fm_match_locate_shortcut(H, O, n, k, bits):
    """fm_match_locate_one (single-row ranges located through the full SA + a text comparison instead of the remaining LF steps)
    == match() followed by locate(): same emptiness, same range when it stays wider than one row, and for single-row results the
    very position locate(match(p)) returns -- incl. repeats, N's, seeds running off the text start, queries shorter than k.
    bits = 2: the 2-bit big-endian fast path (table index and text comparison as bit patterns; no N's in a 2-bit stream); query
    lengths up to 40 so that the comparison spans more than one 16-symbol chunk"""
    rng = np.random.default_rng(n * 7 + k)
    unit = rng.integers(0, 4, 37).astype(np.uint8)
    text = np.concatenate([rng.integers(0, 4, n // 2), np.tile(unit, n)[: n - n // 2]]).astype(np.uint8)    # second half: a tandem repeat
    idx = O.build_index(text)
    nq = 600
    lens = rng.integers(1, 41 if bits == 2 else 24, nq).astype(np.uint32)
    offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.uint32)
    q = rng.integers(0, 4, int(lens.sum())).astype(np.uint8)
    for i in range(nq):
        L = int(lens[i])
        if i % 3 and n > L:
            st = int(rng.integers(0, n - L + 1)) if i % 5 else 0            # some seeds start at text position 0
            q[offs[i]:offs[i] + L] = text[st:st + L]
            if i % 7 == 0:
                q[offs[i] + int(rng.integers(0, L))] ^= 1                    # one substitution
            if i % 11 == 0 and bits == 4:
                q[offs[i] + int(rng.integers(0, L))] = 4                     # an N
    want, _ = O.match(idx, q, offs, lens)
    full_sa = idx.sa.astype(np.uint32).copy(); full_sa[0] = 0xFFFFFFFF
    gw = pack_symbols(np.concatenate([text, np.zeros(64, np.uint8)]), 2, True)
    ktab = None
    if k:
        ktab = np.zeros(2 * 4 ** k, np.uint32)
        H.hh_fm_build_ktab(_p(idx.bwt_occ), _p(idx.L2), C.c_uint32(n), C.c_uint32(idx.primary), C.c_uint32(k), _p(ktab))
    words = np.concatenate([pack_symbols(q, bits, True), np.zeros(2, np.uint32)])
    out = np.zeros((nq, 3), np.uint32)
    H.hh_fm_match_locate(_p(idx.bwt_occ), _p(full_sa), _p(idx.L2), C.c_uint32(n), C.c_uint32(idx.primary), _p(gw), _p(words), C.c_uint32(bits), C.c_uint32(1),
                         _p(offs), _p(lens), C.c_uint32(nq), _p(out), _p(ktab), C.c_uint32(k), C.c_uint32(0))
    if k:
        # the 16-byte located table answers the same (status, x, y) without the SA gather for single-row k-mers
        ktab16 = np.zeros(4 * 4 ** k, np.uint32)
        H.hh_fm_ktab_locate(_p(ktab), _p(full_sa), C.c_uint32(k), _p(ktab16))
        out16 = np.zeros((nq, 3), np.uint32)
        H.hh_fm_match_locate(_p(idx.bwt_occ), _p(full_sa), _p(idx.L2), C.c_uint32(n), C.c_uint32(idx.primary), _p(gw), _p(words), C.c_uint32(bits),
                             C.c_uint32(1), _p(offs), _p(lens), C.c_uint32(nq), _p(out16), _p(ktab16), C.c_uint32(k), C.c_uint32(1))
        # same answers; a single row may come back as FM_RANGE (x, x) on one path and FM_LOCATED (its position) on the other (a k-mer
        # with two occurrences is resolved by two text comparisons when the table carries both SA values): compare by meaning
        def norm(o):
            o = o.copy()
            one = (o[:, 0] == 1) & (o[:, 1] == o[:, 2])
            if one.any():
                o[one, 1] = O.locate(idx, o[one, 1].astype(np.uint32)); o[one, 2] = 0xFFFFFFFF; o[one, 0] = 2
            return o
        assert np.array_equal(norm(out16), norm(out))
        assert (out16[:, 0] == 2).sum() >= (out[:, 0] == 2).sum()
        # ... and with the text context in one-row entries (ktab_located = 2): the same answers as the located table, field by field
        # (seeds longer than k + 16 still compare against the text)
        ktab_ctx = ktab16.copy()
        H.hh_fm_ktab_context(_p(ktab_ctx), C.c_uint32(k), _p(gw), C.c_uint32(n))
        out_ctx = np.zeros((nq, 3), np.uint32)
        H.hh_fm_match_locate(_p(idx.bwt_occ), _p(full_sa), _p(idx.L2), C.c_uint32(n), C.c_uint32(idx.primary), _p(gw), _p(words), C.c_uint32(bits),
                             C.c_uint32(1), _p(offs), _p(lens), C.c_uint32(nq), _p(out_ctx), _p(ktab_ctx), C.c_uint32(k), C.c_uint32(2))
        assert np.array_equal(out_ctx, out16)
    # the two-pass form of the seed-match stage (FM_DEFER, then FM_RESUME for what it hands back) == the single call, for every table
    # format (without a table every multi-row query is handed back at step 0)
    tabs = [(None, 0, 0)] if not k else [(ktab, k, 0), (ktab16, k, 1), (ktab_ctx, k, 2)]
    for tab, kk, loc in tabs:
        whole, split = np.zeros((nq, 3), np.uint32), np.zeros((nq, 3), np.uint32)
        H.hh_fm_match_locate(_p(idx.bwt_occ), _p(full_sa), _p(idx.L2), C.c_uint32(n), C.c_uint32(idx.primary), _p(gw), _p(words), C.c_uint32(bits),
                             C.c_uint32(1), _p(offs), _p(lens), C.c_uint32(nq), _p(whole), _p(tab), C.c_uint32(kk), C.c_uint32(loc))
        H.hh_fm_match_locate_split.restype = C.c_uint32
        nd = H.hh_fm_match_locate_split(_p(idx.bwt_occ), _p(full_sa), _p(idx.L2), C.c_uint32(n), C.c_uint32(idx.primary), _p(gw), _p(words),
                                        C.c_uint32(bits), _p(offs), _p(lens), C.c_uint32(nq), _p(split), _p(tab), C.c_uint32(kk), C.c_uint32(loc))
        assert np.array_equal(split, whole), (kk, loc)
        assert 0 < nd <= nq and (nd < nq or not kk)
    n_loc = 0
    for i in range(nq):
        x, y = int(want[i, 0]), int(want[i, 1])
        st, ox, oy = (int(v) for v in out[i])
        if x > y:
            assert st == 0, (i, want[i], out[i])
        elif st == 2:
            assert x == y and ox == int(O.locate(idx, np.array([x], np.uint32))[0]) and oy == 0xFFFFFFFF, (i, want[i], out[i])
            n_loc += 1
        else:
            assert st == 1 and (ox, oy) == (x, y), (i, want[i], out[i])
            assert x < y or int(lens[i]) <= k or True
    assert n_loc > 50


@pytest.mark.parametrize("fwd,comp", [(True, False), (False, True), (True, True)])
def test_fm_match_approx(H, O, fwd, comp):
    rng = np.random.default_rng(5 + fwd + 2 * comp)
    n = 3000
    text = rng.integers(0, 4, n).astype(np.uint8)
    idx = O.build_index(text)
    nq = 200
    lens = rng.integers(8, 16, nq).astype(np.uint32)
    offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.uint32)
    q = rng.integers(0, 4, int(lens.sum())).astype(np.uint8)
    for i in range(nq):                                   # seeds from the text with one planted substitution
        L = int(lens[i]); st = int(rng.integers(0, n - L))
        seg = text[st:st + L].copy()
        if comp:
            seg = (3 - seg)
        if not fwd:
            pass
        # put it in the stream so that the CONSUMED order spells the reversed text segment (match() is a backward search)
        cons = seg[::-1].copy() if not comp else seg[::-1].copy()
        if i % 3:
            cons[int(rng.integers(L // 2, L))] ^= 1
        if i % 17 == 0:
            cons[int(rng.integers(0, L))] = 4
        q[offs[i]:offs[i] + L] = cons if fwd else cons[::-1]
    flags = (1 if fwd else 0) | (2 if comp else 0)
    for exact_len, find_exact in ((5, 1), (0, 0), (8, 1)):
        want = approx_expected(O, idx, q, offs, lens, exact_len, bool(find_exact), fwd, comp)
        max_out = 48
        words = pack_symbols(q, 4, True)
        out = np.zeros((nq, max_out, 2), np.uint32); counts = np.zeros(nq, np.uint32); sums = np.zeros(nq, np.uint32)
        H.hh_fm_match_approx(_p(idx.bwt_occ), _p(idx.L2), C.c_uint32(n), C.c_uint32(idx.primary), _p(words), C.c_uint32(4), C.c_uint32(1),
                             _p(offs), _p(lens), C.c_uint32(nq), C.c_uint32(flags), C.c_uint32(exact_len), C.c_int(find_exact),
                             C.c_uint32(max_out), _p(out), _p(counts), _p(sums))
        nonempty = 0
        for i in range(nq):
            got = [tuple(x) for x in out[i, :counts[i]]]
            assert counts[i] <= max_out
            assert got == want[i], (i, exact_len, find_exact, got, want[i])
            assert sums[i] == sum(y - x + 1 for x, y in want[i])
            nonempty += len(got) > 0
        assert nonempty > nq // 3


def full_problems(rng, n, max_m=130, max_n=400):
    pats, txts, po, pl, to, tl = [], [], [], [], [], []
    a = b = 0
    for _ in range(n):
        M = int(rng.integers(1, max_m + 1)); N = int(rng.integers(1, max_n + 1))
        t = rng.integers(0, 4, N).astype(np.uint8)
        if N > M and rng.random() < 0.7:
            st = int(rng.integers(0, N - M + 1)); p = t[st:st + M].copy()
            for _k in range(int(rng.integers(0, 5))):
                p[int(rng.integers(0, M))] = rng.integers(0, 4)
        else:
            p = rng.integers(0, 4, M).astype(np.uint8)
        pats.append(p); txts.append(t); po.append(a); pl.append(M); a += M; to.append(b); tl.append(N); b += N
    return (np.concatenate(pats), np.array(po, np.uint32), np.array(pl, np.uint32), np.concatenate(txts), np.array(to, np.uint32), np.array(tl, np.uint32))


@pytest.mark.parametrize("typ", [0, 1, 2])
def test_gotoh_full(H, O, typ):
    """full-matrix Gotoh per-thread routine (32-column stripes, four 8-column LOCAL trackers) == the oracle (== the reference's
    aln::alignment_score, pinned in tests/test_oracle.py), scores and sinks incl. LOCAL tie order"""
    rng = np.random.default_rng(500 + typ)
    for scheme in ((2, -1, -2, -1), (2, -2, -5, -3), (0, -5, -8, -3), (2, -1, -1, -1)):
        pr = full_problems(rng, 120)
        want = O.gotoh_full(typ, scheme, *pr)
        pat, p_off, p_len, txt, t_off, t_len = pr
        for pbits, tbits, tbe in ((4, 2, 0), (2, 2, 1)):
            pw, tw = pack_symbols(pat, pbits, True), pack_symbols(txt, tbits, bool(tbe))
            n = len(p_off)
            score = np.zeros(n, np.int32); sx = np.zeros(n, np.uint32); sy = np.zeros(n, np.uint32)
            s6 = np.array(scheme + (scheme[2], scheme[3]), np.int32)
            H.hh_gotoh_full(C.c_int(typ), _p(s6), _p(pw), C.c_uint32(pbits), C.c_uint32(1), _p(p_off), _p(p_len),
                            _p(tw), C.c_uint32(tbits), C.c_uint32(tbe), _p(t_off), _p(t_len), C.c_uint32(n), _p(score), _p(sx), _p(sy))
            assert np.array_equal(score, want[0]) and np.array_equal(sx, want[1]) and np.array_equal(sy, want[2]), (typ, scheme)


def paired_full_problems(rng, n_pairs, max_m=130, max_n=300, n_frac=0.0):
    """consecutive alignments share (M, N) so that the packed pair path admits them"""
    pats, txts, po, pl, to, tl = [], [], [], [], [], []
    a = b = 0
    for _ in range(n_pairs):
        M = int(rng.integers(1, max_m + 1)); N = int(rng.integers(1, max_n + 1))
        for _k in range(2):
            t = rng.integers(0, 4, N).astype(np.uint8)
            if N > M and rng.random() < 0.7:
                st = int(rng.integers(0, N - M + 1)); p = t[st:st + M].copy()
                for _j in range(int(rng.integers(0, 5))):
                    p[int(rng.integers(0, M))] = rng.integers(0, 4)
            else:
                p = rng.integers(0, 4, M).astype(np.uint8)
            if n_frac and rng.random() < n_frac:
                p[int(rng.integers(0, M))] = 4
            pats.append(p); txts.append(t); po.append(a); pl.append(M); a += M; to.append(b); tl.append(N); b += N
    return (np.concatenate(pats), np.array(po, np.uint32), np.array(pl, np.uint32), np.concatenate(txts), np.array(to, np.uint32), np.array(tl, np.uint32))


@pytest.mark.parametrize("typ", [0, 1, 2])
def test_gotoh_full_pair(H, O, typ):
    """packed s16x2 full-matrix routine (two alignments per thread) == the oracle: scores, sinks, LOCAL tie order; lengths that
    are and are not multiples of the 32-column stripe; N's in the pattern fall back to the int32 routine"""
    rng = np.random.default_rng(600 + typ)
    for scheme in ((2, -1, -2, -1), (2, -2, -5, -3), (0, -5, -8, -3), (2, -1, -1, -1)):
        for n_frac in (0.0, 0.2):
            pr = paired_full_problems(rng, 70, n_frac=n_frac)
            want = O.gotoh_full(typ, scheme, *pr)
            pat, p_off, p_len, txt, t_off, t_len = pr
            for pbits, tbits, tbe in ((4, 2, 1), (4, 4, 1), (2, 8, 0)):
                if pbits == 2 and n_frac:
                    continue
                pw, tw = pack_symbols(pat, pbits, True), pack_symbols(txt, tbits, bool(tbe))
                n = len(p_off)
                score = np.zeros(n, np.int32); sx = np.zeros(n, np.uint32); sy = np.zeros(n, np.uint32)
                s6 = np.array(scheme + (scheme[2], scheme[3]), np.int32)
                packed = H.hh_gotoh_full_pair(C.c_int(typ), _p(s6), _p(pw), C.c_uint32(pbits), C.c_uint32(1), _p(p_off), _p(p_len),
                                              _p(tw), C.c_uint32(tbits), C.c_uint32(tbe), _p(t_off), _p(t_len), C.c_uint32(n), _p(score), _p(sx), _p(sy))
                assert packed > 0 and (n_frac or packed == n)
                assert np.array_equal(score, want[0]) and np.array_equal(sx, want[1]) and np.array_equal(sy, want[2]), (typ, scheme, pbits, tbits)


@pytest.mark.parametrize("typ", [0, 1, 2])
def test_gotoh_full_traceback(H, O, typ):
    """full-matrix traceback (direction nibbles per 32-column stripe + state-machine walk) == the oracle (== the reference's
    aln::alignment_traceback, pinned in tests/test_oracle.py): score, sink, source and every op"""
    rng = np.random.default_rng(700 + typ)
    for scheme in ((2, -1, -2, -1), (2, -2, -5, -3), (0, -5, -8, -3)):
        pr = full_problems(rng, 100, max_m=140, max_n=300)
        want = O.gotoh_full_traceback(typ, scheme, *pr, max_ops=512)
        pat, p_off, p_len, txt, t_off, t_len = pr
        pw, tw = pack_symbols(pat, 4, True), pack_symbols(txt, 2, True)
        n = len(p_off)
        score = np.zeros(n, np.int32); sink = np.zeros((n, 2), np.uint32); source = np.zeros((n, 2), np.uint32)
        ops = np.zeros((n, 512), np.uint8); n_ops = np.zeros(n, np.uint32)
        s6 = np.array(scheme + (scheme[2], scheme[3]), np.int32)
        H.hh_gotoh_full_traceback(C.c_int(typ), _p(s6), _p(pw), C.c_uint32(4), C.c_uint32(1), _p(p_off), _p(p_len),
                                  _p(tw), C.c_uint32(2), C.c_uint32(1), _p(t_off), _p(t_len), C.c_uint32(n), C.c_uint32(512),
                                  _p(score), _p(sink), _p(source), _p(ops), _p(n_ops))
        assert np.array_equal(score, want["score"]) and np.array_equal(sink, want["sink"]) and np.array_equal(source, want["source"])
        assert np.array_equal(n_ops, want["n_ops"])
        for i in range(n):
            assert np.array_equal(ops[i, :n_ops[i]], want["ops"][i, :n_ops[i]]), (typ, scheme, i)


@pytest.mark.parametrize("band", [7, 15, 31])
def test_gotoh_window(H, O, band):
    """windowed banded scoring (checkpoint bands carried between passes, early exit on min_score) == the oracle pass by pass
    (== aln::banded_alignment_score(..., window_begin, window_end, sink, checkpoint), pinned in tests/test_oracle.py), and the
    last pass == the whole-pattern score"""
    from tests.golden.make_golden import random_problems
    rng = np.random.default_rng(800 + band)
    for typ in (0, 1, 2):
        for scheme in ((2, -2, -5, -3), (0, -5, -8, -3)):
            pr = random_problems(rng, 50, band, 120, alphabet_text=6)
            pat, p_off, p_len, txt, t_off, t_len = pr
            n = len(p_off)
            whole = O.banded_gotoh(band, typ, scheme, *pr)
            pw, tw = pack_symbols(pat, 4, True), pack_symbols(txt, 8, False)
            s6 = np.array(scheme + (scheme[2], scheme[3]), np.int32)
            for W, ms in ((32, None), (13, None), (32, rng.integers(-60, 120, n).astype(np.int32))):
                so = orc.window_state(n, band); sh = orc.window_state(n, band)
                for wb in range(0, 120, W):
                    O.banded_gotoh_window(band, typ, scheme, *pr, wb, wb + W, so, min_score=ms)
                    H.hh_gotoh_window(C.c_int(band), C.c_int(typ), _p(s6), None, _p(pw), C.c_uint32(4), C.c_uint32(1), _p(p_off), _p(p_len), None,
                                      _p(tw), C.c_uint32(8), C.c_uint32(0), _p(t_off), _p(t_len), C.c_uint32(n), C.c_uint32(wb), C.c_uint32(wb + W),
                                      _p(ms) if ms is not None else None, _p(sh["ckpt"]), _p(sh["score"]), _p(sh["sx"]), _p(sh["sy"]), _p(sh["alive"]))
                    for k in ("score", "sx", "sy", "alive"):
                        assert np.array_equal(so[k], sh[k]), (band, typ, scheme, W, wb, k)
                    al = so["alive"].astype(bool)
                    assert np.array_equal(so["ckpt"][al], sh["ckpt"][al]), (band, typ, scheme, W, wb)
                if ms is None:
                    ok = whole[3].astype(bool)
                    assert np.array_equal(sh["score"][ok], whole[0][ok]) and np.array_equal(sh["sx"][ok], whole[1][ok]) and np.array_equal(sh["sy"][ok], whole[2][ok])
                    assert not sh["alive"][~ok].any()
                else:
                    assert 0.1 < sh["alive"].mean() < 0.98


@pytest.mark.parametrize("typ", [0, 1, 2])
def test_gotoh_full_quality_table(H, O, typ):
    """full-matrix int32 routine with per-base qualities and a 256 x 2 score table == the oracle (pinned against the reference
    templates with a table-driven scheme in tests/test_oracle.py)"""
    from tests.test_oracle import _nvbowtie_like_table
    rng = np.random.default_rng(880 + typ)
    qtab = _nvbowtie_like_table()
    scheme = (0, 0, -8, -3, -7, -2)
    pr = full_problems(rng, 120)
    pat, p_off, p_len, txt, t_off, t_len = pr
    qual = rng.integers(0, 64, len(pat)).astype(np.uint8)
    want = O.gotoh_full(typ, scheme, *pr, qual=qual, qtab=qtab)
    pw, tw = pack_symbols(pat, 4, True), pack_symbols(txt, 2, True)
    n = len(p_off)
    score = np.zeros(n, np.int32); sx = np.zeros(n, np.uint32); sy = np.zeros(n, np.uint32)
    s6 = np.array(scheme, np.int32)
    qt = np.ascontiguousarray(qtab.reshape(-1))
    H.hh_gotoh_full_q(C.c_int(typ), _p(s6), _p(qt), _p(qual), _p(pw), C.c_uint32(4), C.c_uint32(1), _p(p_off), _p(p_len),
                      _p(tw), C.c_uint32(2), C.c_uint32(1), _p(t_off), _p(t_len), C.c_uint32(n), _p(score), _p(sx), _p(sy))
    assert np.array_equal(score, want[0]) and np.array_equal(sx, want[1]) and np.array_equal(sy, want[2])


def test_packed_paths_hold_their_16bit_bounds(H, O):
    """random schemes up to the edge of the admission rules (large gap / mismatch costs, long texts): whenever the host-side rule
    admits a batch to a packed s16x2 path, the packed routine is bit-identical to the int32 oracle -- the bound leaves no room for a
    wrap-around; schemes the rule rejects are counted, not tested"""
    rng = np.random.default_rng(4242)
    admitted_full = admitted_band = 0
    for trial in range(60):
        scheme = (int(rng.integers(0, 21)), -int(rng.integers(0, 41)), -int(rng.integers(1, 61)), -int(rng.integers(1, 31)))
        s6 = np.array(scheme + (scheme[2], scheme[3]), np.int32)
        typ = int(rng.integers(0, 3))
        # full matrix
        pr = paired_full_problems(rng, 20, max_m=120, max_n=200)
        pat, p_off, p_len, txt, t_off, t_len = pr
        if H.hh_full_pair_path_ok(C.c_int(typ), _p(s6), C.c_uint32(int(p_len.max())), C.c_uint32(int(t_len.max()))):
            admitted_full += 1
            want = O.gotoh_full(typ, scheme, *pr)
            pw, tw = pack_symbols(pat, 2, True), pack_symbols(txt, 2, True)
            n = len(p_off)
            score = np.zeros(n, np.int32); sx = np.zeros(n, np.uint32); sy = np.zeros(n, np.uint32)
            packed = H.hh_gotoh_full_pair(C.c_int(typ), _p(s6), _p(pw), C.c_uint32(2), C.c_uint32(1), _p(p_off), _p(p_len),
                                          _p(tw), C.c_uint32(2), C.c_uint32(1), _p(t_off), _p(t_len), C.c_uint32(n), _p(score), _p(sx), _p(sy))
            assert packed == n
            assert np.array_equal(score, want[0]) and np.array_equal(sx, want[1]) and np.array_equal(sy, want[2]), ("full", typ, scheme)
        # banded
        band = int(rng.choice([7, 15, 31]))
        prb = fixed_problems(rng, 40, band, 150, ragged=(typ == 1))
        pat, p_off, p_len, txt, t_off, t_len = prb
        n = len(p_off)
        pw, tw = pack_symbols(pat, 4, True), pack_symbols(txt, 2, True)
        score = np.zeros(n, np.int32); sx = np.zeros(n, np.uint32); sy = np.zeros(n, np.uint32); nf = np.zeros(1, np.uint32)
        r = H.hh_gotoh_pair(C.c_int(band), C.c_int(typ), _p(s6), None, None, C.c_uint32(150), _p(pw), C.c_uint32(4), C.c_uint32(1), _p(p_off), _p(p_len),
                            _p(tw), C.c_uint32(1), _p(t_off), _p(t_len), C.c_uint32(n), _p(score), _p(sx), _p(sy), _p(nf))
        if r == 0:
            admitted_band += 1
            want = O.banded_gotoh(band, typ, scheme, *prb)
            assert np.array_equal(score, want[0]) and np.array_equal(sx, want[1]) and np.array_equal(sy, want[2]), ("banded", band, typ, scheme)
    assert admitted_full >= 20 and admitted_band >= 10


@pytest.mark.parametrize("pbits,pbe", [(2, 1), (2, 0), (4, 1), (4, 0), (8, 0), (8, 1)])
def test_gotoh_pair_pattern_stream_formats(H, O, pbits, pbe):
    """the packed banded routine reads its pattern through PatStream (words normalised to big-endian symbol order at refill):
    every packing the ABI admits -- 2 / 4 / 8 bits, either endianness, patterns starting at arbitrary (unaligned) offsets"""
    rng = np.random.default_rng(70 + pbits * 2 + pbe)
    for band, typ in ((31, 1), (15, 2), (7, 0)):
        pr = fixed_problems(rng, 61, band, 97, ragged=(typ == 1))        # 97-symbol patterns: offsets are not word multiples
        r, got, nf = _gotoh_pair(H, band, typ, (2, -2, -5, -3, -5, -3), pr, 97, pbits=pbits, pbe=pbe)
        assert r == 0
        want = O.banded_gotoh(band, typ, (2, -2, -5, -3), *pr)
        assert all(np.array_equal(a, b) for a, b in zip(got, want[:3])), (pbits, pbe, band, typ)


@pytest.mark.parametrize("pbits,pbe,tbits,tbe", [(2, 0, 2, 0), (4, 0, 4, 0), (2, 1, 4, 0), (8, 0, 2, 0), (4, 1, 2, 1)])
def test_gotoh_full_pair_stream_formats(H, O, pbits, pbe, tbits, tbe):
    """the packed full-matrix routine reads pattern and text through SymSeq: little-endian and mixed packings, unaligned offsets"""
    rng = np.random.default_rng(90 + pbits + 3 * tbits + pbe + tbe)
    for typ in (0, 1, 2):
        pr = paired_full_problems(rng, 40, max_m=90, max_n=170)
        want = O.gotoh_full(typ, (2, -2, -5, -3), *pr)
        pat, p_off, p_len, txt, t_off, t_len = pr
        pw, tw = pack_symbols(pat, pbits, bool(pbe)), pack_symbols(txt, tbits, bool(tbe))
        n = len(p_off)
        score = np.zeros(n, np.int32); sx = np.zeros(n, np.uint32); sy = np.zeros(n, np.uint32)
        s6 = np.array((2, -2, -5, -3, -5, -3), np.int32)
        packed = H.hh_gotoh_full_pair(C.c_int(typ), _p(s6), _p(pw), C.c_uint32(pbits), C.c_uint32(pbe), _p(p_off), _p(p_len),
                                      _p(tw), C.c_uint32(tbits), C.c_uint32(tbe), _p(t_off), _p(t_len), C.c_uint32(n), _p(score), _p(sx), _p(sy))
        assert packed == n
        assert np.array_equal(score, want[0]) and np.array_equal(sx, want[1]) and np.array_equal(sy, want[2]), (typ, pbits, pbe, tbits, tbe)


@pytest.mark.parametrize("typ", [0, 1, 2])
@pytest.mark.parametrize("band", [7, 15, 31])
def test_gapless_traceback_fast_path(H, O, band, typ):
    """gapless_traceback (the fast path of nvb_banded_gotoh_traceback): whenever it claims an alignment from (score, sink) alone, the
    oracle's traceback (pinned to the reference's) is exactly that all-substitution suffix of the sink's diagonal -- reads with and
    without indels, N's in pattern and text (never claimed through), every scheme; GLOBAL is never claimed"""
    rng = np.random.default_rng(band * 11 + typ)
    claimed = 0
    for scheme in ((2, -2, -5, -3), (2, -6, -8, -3), (1, -1, -1, -1), (0, -5, -8, -3)):
        for with_n in (False, True):
            pr = list(fixed_problems(rng, 120, band, 90, ragged=(typ == 1)))
            if with_n:
                pr[0] = pr[0].copy(); pr[0][rng.random(len(pr[0])) < 0.01] = 4
                pr[3] = pr[3].copy(); pr[3][rng.random(len(pr[3])) < 0.01] = 4
            pat, p_off, p_len, txt, t_off, t_len = pr
            want = O.banded_traceback(band, typ, scheme, *pr, max_ops=256)
            n = len(p_off)
            pw, tw = pack_symbols(pat, 4, True), pack_symbols(txt, 4, True)
            s6 = np.array(scheme + (scheme[2], scheme[3]), np.int32)
            ln = np.zeros(n, np.uint32); ok = np.zeros(n, np.uint8)
            sink = np.ascontiguousarray(want["sink"].astype(np.uint32))
            H.hh_gapless_traceback(C.c_int(typ), _p(s6), None, None, _p(pw), C.c_uint32(4), C.c_uint32(1), _p(p_off), _p(p_len),
                                   _p(tw), C.c_uint32(4), C.c_uint32(1), _p(t_off), _p(t_len), C.c_uint32(n),
                                   _p(np.ascontiguousarray(want["score"].astype(np.int32))), _p(sink), _p(ln), _p(ok))
            if typ == 0:
                assert not ok.any()
            for a in np.nonzero(ok)[0]:
                L = int(ln[a])
                assert int(want["n_ops"][a]) == L and not want["ops"][a][:L].any(), (band, typ, scheme, a)
                assert tuple(int(v) for v in want["source"][a]) == (int(sink[a, 0]) - L, int(sink[a, 1]) - L), (band, typ, scheme, a)
            claimed += int(ok.sum())
    assert typ == 0 or claimed > 20


@pytest.mark.parametrize("typ", [0, 1, 2])
def test_gotoh_full_pair_quality_table(H, O, typ):
    """the packed full-matrix routine with quality-dependent substitution scores (per-column profiles indexed by the text symbol, the row's
    selector from the two text symbols) == the oracle's table-driven full DP: pairs of equal shape take the packed path (patterns with N
    included: an N column is an all-mismatch profile), pairs of different shape and texts with N the int32 routine"""
    from tests.test_oracle import _nvbowtie_like_table
    rng = np.random.default_rng(4400 + typ)
    qtab = _nvbowtie_like_table(); qt = np.ascontiguousarray(qtab.reshape(-1).astype(np.int32))
    scheme = (int(qtab[0, 0]), int(qtab[0, 1]), -8, -3, -7, -2); s6 = np.array(scheme, np.int32)
    most = 0
    for n_frac, text_n in ((0.0, False), (0.02, False), (0.0, True)):
        for pr_i, pr in enumerate((paired_full_problems(rng, 60, max_m=150, max_n=300), full_problems(rng, 60, max_m=100, max_n=200))):
            pat, p_off, p_len, txt, t_off, t_len = pr
            pat = pat.copy(); txt = txt.copy()
            if n_frac:
                pat[rng.random(len(pat)) < n_frac] = 4
            if text_n:
                txt[rng.random(len(txt)) < 0.002] = 4
            qual = rng.integers(0, 60, len(pat)).astype(np.uint8)
            want = O.gotoh_full(typ, scheme, pat, p_off, p_len, txt, t_off, t_len, qual=qual, qtab=qtab)
            pw, tw = pack_symbols(pat, 4, True), pack_symbols(txt, 4, True)
            n = len(p_off)
            score = np.zeros(n, np.int32); sx = np.zeros(n, np.uint32); sy = np.zeros(n, np.uint32)
            packed = H.hh_gotoh_full_pair_qual(C.c_int(typ), _p(s6), _p(qt), _p(qual), _p(pw), C.c_uint32(4), C.c_uint32(1), _p(p_off), _p(p_len),
                                               _p(tw), C.c_uint32(4), C.c_uint32(1), _p(t_off), _p(t_len), C.c_uint32(n),
                                               C.c_uint32(int(max(p_len))), C.c_uint32(int(max(t_len))), _p(score), _p(sx), _p(sy))
            assert packed >= 0
            assert np.array_equal(score, want[0]) and np.array_equal(sx, want[1]) and np.array_equal(sy, want[2]), (typ, n_frac, text_n, packed)
            most = max(most, packed)
            if not text_n and pr_i == 0:
                assert packed == n                    # equal-shape pairs, no N in the text: everything through the packed routine
    assert most > 0


def test_gotoh_window_quality_table(H, O):
    """windowed banded scoring with per-base qualities and a score table (the early-exit threshold then uses table[0] as the
    reference's scoring.match(0) does): pass-by-pass == the oracle, last pass == the whole-pattern score"""
    from tests.golden.make_golden import random_problems
    from tests.test_oracle import _nvbowtie_like_table
    rng = np.random.default_rng(901)
    qtab = _nvbowtie_like_table(); qt = np.ascontiguousarray(qtab.reshape(-1))
    scheme = (0, 0, -8, -3, -7, -2); s6 = np.array(scheme, np.int32)
    for band, typ in ((31, 1), (15, 2), (7, 0)):
        pr = random_problems(rng, 50, band, 110)
        pat, p_off, p_len, txt, t_off, t_len = pr
        n = len(p_off)
        qual = rng.integers(0, 64, len(pat)).astype(np.uint8)
        whole = O.banded_gotoh(band, typ, scheme, *pr, qual=qual, qtab=qtab)
        pw, tw = pack_symbols(pat, 4, True), pack_symbols(txt, 8, False)
        for ms in (None, rng.integers(-60, 120, n).astype(np.int32)):
            so = orc.window_state(n, band); sh = orc.window_state(n, band)
            for wb in range(0, 110, 32):
                O.banded_gotoh_window(band, typ, scheme, *pr, wb, wb + 32, so, min_score=ms, qual=qual, qtab=qtab)
                H.hh_gotoh_window(C.c_int(band), C.c_int(typ), _p(s6), _p(qt), _p(pw), C.c_uint32(4), C.c_uint32(1), _p(p_off), _p(p_len), _p(qual),
                                  _p(tw), C.c_uint32(8), C.c_uint32(0), _p(t_off), _p(t_len), C.c_uint32(n), C.c_uint32(wb), C.c_uint32(wb + 32),
                                  _p(ms) if ms is not None else None, _p(sh["ckpt"]), _p(sh["score"]), _p(sh["sx"]), _p(sh["sy"]), _p(sh["alive"]))
                for k in ("score", "sx", "sy", "alive"):
                    assert np.array_equal(so[k], sh[k]), (band, typ, wb, k)
            if ms is None:
                ok = whole[3].astype(bool)
                assert np.array_equal(sh["score"][ok], whole[0][ok]) and np.array_equal(sh["sx"][ok], whole[1][ok])

@pytest.mark.parametrize("band", [31, 15, 8, 63])
def test_gapless_job_shortcut(H, O, band, request):
    """gapless_job_shortcut (the exact shortcut of the LOCAL extension in nvb_seed_extend): whenever it claims a job, (score, sink) are
    exactly what the oracle's banded DP and the reference's own aln::banded_alignment_score<BAND> (oracle/_ref, bands 31 and 15) return -- reads with 0..4 substitutions at random and at chosen
    places (the ends, next to the ends, adjacent), reads with an indel (never provable), tandem repeats of period 1, 2, 3, 7 and 40 (other
    band diagonals as good as the seed's), short and ragged reads, windows longer than the band needs, four schemes.  Jobs outside the
    routine's preconditions are never claimed: band 63, and reads whose offset in their stream is not a multiple of 16"""
    rng = np.random.default_rng(900 + band)
    n_txt = 60_000
    text = rng.integers(0, 4, n_txt).astype(np.uint8)
    for st, period in ((5_000, 1), (8_000, 2), (11_000, 3), (14_000, 7), (20_000, 40)):
        text[st:st + 2_500] = np.tile(text[st:st + period], 2_500 // period + 1)[:2_500]
    n = 3_000
    stride = 160
    M = np.full(n, 150, np.uint32); M[:600] = rng.integers(1, 151, 600)
    pos = rng.integers(100, n_txt - 400, n)
    pos[600:1500] = rng.integers(5_000, 22_000, 900)                    # inside / across the repeats
    reads = np.zeros((n, stride), np.uint8)
    places = [(0,), (1,), (-1,), (-2,), (0, 1), (-2, -1), (0, -1), (1, -2), (2, 3), (70,), (70, 71), (10, -10), (0, 1, 2), (-3, -2, -1), (3, 70)]
    for a in range(n):
        m = int(M[a]); r = text[pos[a]:pos[a] + m].copy()
        kind = a % 7
        if kind in (1, 2, 3):                                           # 1..4 random substitutions
            for q in rng.integers(0, m, rng.integers(1, 5)):
                r[q] = (r[q] + 1 + rng.integers(0, 3)) % 4
        elif kind == 4:                                                 # chosen places
            for q in places[(a // 7) % len(places)]:
                if -m <= q < m:
                    r[q] = (r[q] + 1 + (a % 3)) % 4
        elif kind == 5 and m > 20:                                      # an indel
            cut = int(rng.integers(5, m - 5))
            r = np.concatenate([r[:cut], r[cut + 1:], text[pos[a] + m:pos[a] + m + 1]]) if a % 2 else np.concatenate([r[:cut], [(r[cut] + 1) % 4], r[cut:m - 1]])
        reads[a, :m] = r
    to = (pos - band // 2).astype(np.uint32)
    N = (M + band - 1 + (np.arange(n) % 3) * 5).astype(np.uint32)       # some windows longer than needed
    N[5::50] = M[5::50] + band - 2                                      # ... and a few too short: never claimed
    po = (np.arange(n) * stride).astype(np.uint32)
    sw = np.concatenate([pack_symbols(reads.reshape(-1), 2, True), np.zeros(2, np.uint32)])
    gw = np.concatenate([pack_symbols(np.concatenate([text, np.zeros(64, np.uint8)]), 2, True), np.zeros(2, np.uint32)])
    sw5 = np.concatenate([pack_symbols(np.concatenate([np.zeros(5, np.uint8), reads.reshape(-1)]), 2, True), np.zeros(2, np.uint32)])
    po5 = po + np.uint32(5)                                             # the same reads 5 symbols further into their stream
    R = Reference(request, orc.Ref)
    total = 0
    for scheme in ((2, -2, -5, -3), (1, -4, -6, -1), (2, -6, -8, -3), (3, -1, -2, -2)):
        solved = np.zeros(n, np.uint8); score = np.zeros(n, np.int32); sink = np.zeros((n, 2), np.uint32)
        H.hh_gapless_job_shortcut(_p(sw5), _p(gw), _p(po5), _p(M), _p(to), _p(N), C.c_uint32(n), C.c_uint32(band), C.c_int32(scheme[0]), C.c_int32(scheme[1]),
                                  C.c_int32(scheme[2]), _p(solved), _p(score), _p(sink))
        assert not solved.any(), (band, scheme)
        H.hh_gapless_job_shortcut(_p(sw), _p(gw), _p(po), _p(M), _p(to), _p(N), C.c_uint32(n), C.c_uint32(band), C.c_int32(scheme[0]), C.c_int32(scheme[1]),
                                  C.c_int32(scheme[2]), _p(solved), _p(score), _p(sink))
        ok = solved.astype(bool)
        if band > 32:
            assert not ok.any(), (band, scheme)
            continue
        ws, wx, wy, _ = O.banded_gotoh(band, 1, scheme, reads.reshape(-1), po, M, text, to, N)
        if band in (31, 15):
            # ... and the reference's own aln::banded_alignment_score<BAND> (oracle/_ref) says the same as the restatement
            full = N >= M + band - 1                                    # (shorter windows: the reference reads past the text, undefined)
            R.same([ws[full], wx[full], wy[full]],
                   lambda: [r[full] for r in R.live.banded_gotoh(band, 1, scheme, reads.reshape(-1), po, M, text, to, N)[:3]])
        assert np.array_equal(score[ok], ws[ok]) and np.array_equal(sink[ok, 0], wx[ok]) and np.array_equal(sink[ok, 1], wy[ok]), (band, scheme)
        assert not ok[N < M + band - 1].any()
        exact = (np.arange(n) % 7 == 0) | (np.arange(n) % 7 == 6)
        assert ok[exact & (N >= M + band - 1)].all()                     # a read without a difference is always resolved
        total += int(ok.sum())
        print("gapless_job_shortcut band %d scheme %s: %d of %d jobs claimed" % (band, scheme, int(ok.sum()), n))
    assert band > 32 or total > 4 * n // 4


def test_hit_window(H):
    """hit_window (the genome window of a hit on both extension paths) == the window rule of tests/pipeline_oracle.py clamped to the
    text: seeds nearer the text start than their read offset, diagonals within band/2 of the text start, windows running past the
    text's end, and the largest uint32 positions"""
    rng = np.random.default_rng(41)
    n = 3000
    glen = rng.integers(1, 2**32, n, dtype=np.uint64)
    pos = (rng.random(n) * glen).astype(np.uint64)
    sb = rng.integers(0, 300, n, dtype=np.uint64); ln = rng.integers(1, 300, n, dtype=np.uint64); band = rng.integers(2, 64, n, dtype=np.uint64)
    pos[:500] = sb[:500] // 2                                           # seed nearer the text start than its read offset
    pos[500:1000] = sb[500:1000] + band[500:1000] // 2 - 1              # diagonal within band/2 of the text start
    pos[1000:1500] = rng.integers(0, 10**6, 500, dtype=np.uint64); sb[1000:1500] = 0
    glen[1000:1500] = pos[1000:1500] + 1 + ln[1000:1500] // 2           # window past the text's end
    pos[1500:1600] = 0xFFFFFFFF; glen[1500:1600] = 0xFFFFFFFF           # the largest positions
    ln[1550:1600] = 0xFFFFFFFF; band[1580:1600] = 0xFFFFFFFF
    args = [u32(a) for a in (pos, sb, ln, band, glen)]
    got = np.zeros((n, 2), np.uint32)
    H.hh_hit_window(*[_p(a) for a in args], C.c_uint32(n), _p(got))
    for a in range(n):
        p, s, L, B, G = (int(v[a]) for v in (pos, sb, ln, band, glen))
        diag = p - s if p > s else 0
        gb = diag - B // 2 if diag > B // 2 else 0
        assert (int(got[a, 0]), int(got[a, 1])) == (gb, min(gb + L + B, G)), (a, p, s, L, B, G)
    assert (got[1000:1500, 1] == u32(glen[1000:1500])).all()


def test_hit_end(H):
    """hit_end (a read's best_pos and its traceback's begin): window begin + sink.x for a sink the DP reported, 0xFFFFFFFF ("no position")
    for the default sink of a window shorter than its read -- never the wrapped window_begin - 1 -- including windows that begin at 0"""
    rng = np.random.default_rng(44)
    wb = np.concatenate([[0, 0, 0, 1, 5, 199_885, 0xFFFFFFFE, 0xFFFFFFFF], rng.integers(0, 2**31, 500)]).astype(np.uint32)
    sx = np.concatenate([[0, 7, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 1, 0xFFFFFFFF], rng.integers(0, 400, 500)]).astype(np.uint32)
    sx[100:200] = 0xFFFFFFFF
    got = np.zeros(len(wb), np.uint32)
    H.hh_hit_end(_p(wb), _p(sx), C.c_uint32(len(wb)), _p(got))
    want = [0xFFFFFFFF if x == 0xFFFFFFFF else b + x for b, x in zip(wb.tolist(), sx.tolist())]
    assert got.tolist() == want
    assert got[:8].tolist() == [0, 7, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF]
    assert (got[100:200] == 0xFFFFFFFF).all() and (got[8:100] != 0xFFFFFFFF).all()


def test_best_key(H):
    """best_key orders the hits of a read as the best-per-read reduction needs: a higher score wins, an equal score goes to the smaller hit
    index, negative scores sort below positive ones; score / hit <-> key round-trips and no hit packs to key 0 ("no hit")"""
    rng = np.random.default_rng(43)
    score = np.concatenate([[-2**31, -1, 0, 1, 2**31 - 1, -5, -5, 7, 7], rng.integers(-2**31, 2**31, 1000), rng.integers(-3, 4, 1000)]).astype(np.int32)
    hit = np.concatenate([[0, 5, 5, 5, 0, 3, 4, 0, 0xFFFFFFFE], rng.integers(0, 0xFFFFFFFF, 1000), rng.integers(0, 20, 1000)]).astype(np.uint32)
    n = len(score)
    key = np.zeros(n, np.uint64); ks = np.zeros(n, np.int32); kh = np.zeros(n, np.uint32)
    H.hh_best_key(_p(score), _p(hit), C.c_uint32(n), _p(key), _p(ks), _p(kh))
    assert np.array_equal(ks, score) and np.array_equal(kh, hit) and (key != 0).all()
    s, h = score.astype(np.int64), hit.astype(np.int64)
    wins = (s[:, None] > s[None, :]) | ((s[:, None] == s[None, :]) & (h[:, None] < h[None, :]))
    assert np.array_equal(key[:, None] > key[None, :], wins)
    assert key[1] < key[3] and key[0] < key[2] and key[5] > key[6] and key[7] > key[8]


def test_seed_range_size(H):
    """seed_range_size (the hits a seed contributes, both extension paths and the seed match): an empty range contributes none, a range the
    seed match already located (y = 0xFFFFFFFF) one, a row range its rows up to max_seed_hits"""
    ranges = np.array([(1, 0), (9, 4), (0xFFFFFFFF, 0), (7, 7), (3, 12), (0, 0xFFFFFFFE), (123456, 0xFFFFFFFF), (0, 0xFFFFFFFF)], np.uint32)
    for max_hits in (1, 5, 100, 0xFFFFFFFF):
        got = np.zeros(len(ranges), np.uint32)
        H.hh_seed_range_size(_p(np.ascontiguousarray(ranges)), C.c_uint32(len(ranges)), C.c_uint32(max_hits), _p(got))
        want = [min(1 if y == 0xFFFFFFFF else (y - x + 1 if x <= y else 0), max_hits) for x, y in ranges.tolist()]
        assert got.tolist() == want, max_hits
