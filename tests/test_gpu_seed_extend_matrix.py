"""-m gpu: nvb_seed_extend against the oracle composition (tests/pipeline_oracle.py) across its parameter space.

The inputs are generated here with numpy from fixed seeds (not with nvbio_b200.synth), so they do not depend on the code under test:
a random genome of 200,003 symbols and a copy with a 500-bp unit repeated 40 times and a period-7 tandem repeat; per genome reads at
their true locus (both strands, substitutions and indels), reads on the genome's first and last positions (windows clamped at 0 or n),
reads that run past the genome's end (genome[n-k:] + a random tail, and their reverse complements), and random reads; ragged and
4-bit variants (N anywhere, N as first / last symbol, N in a seed's k-mer, a read of N only).

Every parameter row runs the per-read path (the default call) on six index variants -- the reference format (SA every 16 symbols), the
full SA (single-row fold), and the full SA with a k = 8 table (plain, located, context) and a k = 12 context table, the tables with the
two-pass seed match on and off -- with the exact shortcut on and off and with a hit capacity that truncates; and once the per-hit path
with every hit array.  The oracle does not depend on the index: it is computed once per row."""
import ctypes as C
import numpy as np
import pytest
import torch
from oracle import orc
import nvbio_b200 as nb
from nvbio_b200 import aln
from nvbio_b200.strings import PackedStringSet, pack_symbols
from tests.gpu_util import require_gpu, dev_u32, host_u32
from tests.pipeline_oracle import seed_extend_oracle, seed_extend_paired_oracle, NO_POS

pytestmark = pytest.mark.gpu

G_LEN = 200_003                      # not a multiple of 16
L = 150
INT_MIN = -2**31
A = (2, -2, -5, -3)
B = (1, -4, -6, -1)
Z = (0, -5, -8, -3)                  # every LOCAL score is 0: ties decide the result
BIG = (40, -2, -5, -3)               # beyond the packed kernels' range: the int32 kernel carries the pipeline
Q = "quality"                        # QualityGotohScheme with read_quals
OVERHANG_K = (10, 12, 20, 22, 32, 60, 100, L - 1)
INDEXES = ("ref", "fold", "k8", "k8loc", "k8ctx", "k12ctx")


def revcomp(r):
    return np.where(r < 4, 3 - r, r)[::-1].astype(np.uint8)


def make_genomes():
    rng = np.random.default_rng(2024)
    g = rng.integers(0, 4, G_LEN).astype(np.uint8)
    rep = g.copy()
    rep[60_000:80_000] = np.tile(g[1000:1500], 40)                    # multi-row ranges, more than RJ_LOCAL windows per read
    rep[120_000:126_000] = np.tile(g[3000:3007], 6000 // 7 + 1)[:6000]  # period 7: diagonals that tie inside one band
    return {"rand": g, "rep": rep}


def mutate(rng, seg, sub, indel):
    seg = seg.copy()
    m = rng.random(len(seg)) < sub
    seg[m] = (seg[m] + rng.integers(1, 4, int(m.sum()))) % 4
    u = rng.random(len(seg))
    keep = u >= indel / 2                                              # deletions
    ins = (u >= indel / 2) & (u < indel)                                # insertions after these positions
    out = []
    for s, k, i in zip(seg.tolist(), keep.tolist(), ins.tolist()):
        if k:
            out.append(s)
        if i:
            out.append(int(rng.integers(0, 4)))
    return np.array(out, np.uint8)


def make_reads(gsym, seed, read_len, ragged=False, bits=2):
    """~690 reads: true-locus (both strands, 1 % substitutions, 0.2 % indels; every 8th in the 500-bp repeat, every 8th in the period-7
    repeat), the genome's first / last 40 positions, overhanging the end (k in OVERHANG_K, 3 tails each, and reverse complements), random"""
    rng = np.random.default_rng(seed)
    n = len(gsym)
    reads = []
    for i in range(560):
        if i % 8 == 0:
            p = int(rng.integers(60_000, 80_000 - read_len - 20))
        elif i % 8 == 1:
            p = int(rng.integers(120_000, 126_000 - read_len - 20))
        else:
            p = int(rng.integers(0, n - read_len - 20))
        r = mutate(rng, gsym[p:p + read_len + 20], 0.01, 0.002)[:read_len]
        reads.append(revcomp(r) if i & 1 else r)
    for j, p in enumerate(list(range(0, 40, 2)) + list(range(n - read_len - 39, n - read_len + 1, 2))):
        r = gsym[p:p + read_len].copy()
        reads.append(revcomp(r) if j % 3 == 2 else r)
    overhang = []
    for k in OVERHANG_K:
        if k >= read_len:
            continue
        for t in range(3):
            r = np.concatenate([gsym[n - k:], rng.integers(0, 4, read_len - k).astype(np.uint8)])
            overhang += [len(reads), len(reads) + 1]
            reads += [r, revcomp(r)]
    for _ in range(40):
        reads.append(rng.integers(0, 4, read_len).astype(np.uint8))
    if ragged:
        lens = rng.integers(4, read_len + 1, len(reads))
        lens[10:39] = [10, 12, 20, 22, 32, 64] * 4 + [9, 11, 19, 21, 31]         # exactly a seed length, and one below
        lens[:10] = read_len
        lens[overhang] = read_len
        reads = [r[:int(l)] for r, l in zip(reads, lens)]
    if bits == 4:
        for r in reads:
            r[rng.random(len(r)) < 0.003] = 4
        reads[0][0] = 4                                                          # N first
        reads[1][-1] = 4                                                         # N last
        for i, q in zip(range(2, 8), (19, 11, 9, 21, 31, 15)):                   # N in the last k symbols of the first seed
            reads[i][q] = 4
            reads[i][min(q + 40, len(reads[i]) - 1)] = 4
        reads[8][:] = 4                                                          # N only
    return reads, overhang


def string_set(reads, bits, read_len):
    spw = 32 // bits
    stride = (read_len + spw - 1) // spw * spw
    n = len(reads)
    buf = np.zeros((n, stride), np.uint8)
    lens = np.array([len(r) for r in reads], np.uint32)
    for i, r in enumerate(reads):
        buf[i, :len(r)] = r
    words = torch.from_numpy(pack_symbols(buf.reshape(-1), bits, True).view(np.int32)).cuda()
    if (lens == read_len).all():
        return PackedStringSet.fixed(words, n, read_len, stride=stride, bits=bits), stride
    return PackedStringSet(words=words, bits=bits, big_endian=True, offsets=dev_u32(np.arange(n, dtype=np.uint32) * stride),
                           lengths=dev_u32(lens), stride=0, length=read_len, count=n), stride


def scheme_of(sc):
    if sc == Q:
        return aln.QualityGotohScheme(match_bonus=2, mm_min=2, mm_max=6, read_gap_const=5, read_gap_coeff=3, ref_gap_const=5, ref_gap_coeff=3)
    return aln.SimpleGotohScheme(*sc)


class World:
    """genomes, oracle indexes and device index variants, built on first use and shared by the module"""

    def __init__(self):
        self.O = orc.Oracle()
        self.gsym = make_genomes()
        self.gw = {k: torch.from_numpy(pack_symbols(g, 2, True).view(np.int32)).cuda() for k, g in self.gsym.items()}
        self._idx, self._fmi, self._reads = {}, {}, {}

    def idx(self, gname):
        if gname not in self._idx:
            self._idx[gname] = self.O.build_index(self.gsym[gname])
        return self._idx[gname]

    def fmi(self, gname, variant):
        key = (gname, variant)
        if key not in self._fmi:
            gw = self.gw[gname]
            if variant == "ref":
                i = self.idx(gname)
                f = nb.FMIndexDevice.from_host(i.bwt_occ, i.ssa, i.L2, i.n, i.primary)
            else:
                f, _ = nb.FMIndexDevice.from_text(gw, G_LEN, sa_interval=1)
                if variant != "fold":
                    k = 12 if variant == "k12ctx" else 8
                    f.build_ktab(k, located=variant != "k8", text=gw if variant.endswith("ctx") else None)
            torch.cuda.synchronize()
            self._fmi[key] = f
        return self._fmi[key]

    def reads(self, gname, bits, ragged, read_len):
        key = (gname, bits, ragged, read_len)
        if key not in self._reads:
            seed = {"rand": 1, "rep": 2}[gname] * 100 + bits * 10 + int(ragged) + read_len
            reads, overhang = make_reads(self.gsym[gname], seed, read_len, ragged, bits)
            rs, stride = string_set(reads, bits, read_len)
            qual = np.random.default_rng(seed + 7).integers(0, 50, (len(reads), stride)).astype(np.uint8)
            self._reads[key] = dict(reads=reads, overhang=overhang, rs=rs, stride=stride, qual=qual,
                                    quals=[qual[i, :len(r)] for i, r in enumerate(reads)], d_qual=torch.from_numpy(qual.reshape(-1)).cuda())
        return self._reads[key]


@pytest.fixture(scope="module")
def world():
    require_gpu()
    return World()


# genome, bits, ragged, read length, type, band, seed length, seed interval, both strands, max seed hits, scheme
ROWS = [
    ("rand", 2, False, L, aln.LOCAL, 3, 20, 10, True, 100, A),
    ("rand", 4, False, L, aln.LOCAL, 5, 12, 6, True, 100, B),
    ("rep", 2, False, L, aln.LOCAL, 7, 10, 5, True, 3, A),
    ("rand", 2, True, L, aln.LOCAL, 15, 22, 25, True, 100, A),
    ("rep", 2, False, L, aln.LOCAL, 31, 20, 10, True, 1, Z),
    ("rand", 2, False, L, aln.LOCAL, 63, 32, 8, True, 100, A),
    ("rand", 2, False, L, aln.LOCAL, 31, 20, 10, False, 100, B),
    ("rand", 2, False, L, aln.LOCAL, 31, 20, 10, True, 100, BIG),
    ("rand", 2, False, L, aln.LOCAL, 31, 20, 10, True, 100, Q),
    ("rep", 4, False, L, aln.LOCAL, 31, 20, 10, True, 100, A),
    ("rand", 2, False, 64, aln.LOCAL, 15, 64, 10, True, 100, A),
    ("rand", 4, True, L, aln.LOCAL, 63, 22, 25, True, 100, B),
    ("rand", 2, False, L, aln.GLOBAL, 3, 20, 10, True, 100, A),
    ("rand", 4, False, L, aln.GLOBAL, 7, 12, 6, True, 100, B),
    ("rand", 2, False, L, aln.GLOBAL, 31, 20, 10, False, 100, A),
    ("rep", 2, False, L, aln.GLOBAL, 31, 10, 5, True, 3, BIG),
    ("rand", 2, False, 64, aln.GLOBAL, 15, 64, 64, True, 100, B),
    ("rep", 4, True, L, aln.GLOBAL, 63, 32, 8, True, 100, Z),
    ("rand", 2, False, L, aln.SEMI_GLOBAL, 5, 22, 25, True, 100, A),
    ("rand", 2, False, L, aln.SEMI_GLOBAL, 15, 20, 10, True, 100, Q),
    ("rand", 4, True, L, aln.SEMI_GLOBAL, 63, 32, 8, True, 100, B),
    ("rep", 2, False, L, aln.SEMI_GLOBAL, 31, 20, 10, True, 1, Z),
    ("rep", 4, False, L, aln.SEMI_GLOBAL, 15, 12, 6, True, 100, A),
    ("rep", 2, True, L, aln.SEMI_GLOBAL, 7, 10, 5, False, 100, B),
]
TYPE_NAME = {aln.GLOBAL: "global", aln.LOCAL: "local", aln.SEMI_GLOBAL: "semi"}


def row_id(r):
    g, bits, ragged, rl, typ, band, sl, si, both, mh, sc = r
    sn = {A: "A", B: "B", Z: "Z", BIG: "BIG", Q: "Q"}[sc]
    return "%s-%db%s%s-%s-b%d-s%d.%d%s-h%d-%s" % (g, bits, "r" if ragged else "", "" if rl == L else "L%d" % rl, TYPE_NAME[typ], band, sl, si,
                                                  "" if both else "-fw", mh, sn)


def params_of(world, r):
    g, bits, ragged, rl, typ, band, sl, si, both, mh, sc = r
    d = world.reads(g, bits, ragged, rl)
    p = nb.SeedExtendParams(seed_len=sl, seed_interval=si, band_len=band, type=typ, both_strands=both, max_seed_hits=mh,
                            scheme=scheme_of(sc), read_quals=d["d_qual"] if sc == Q else None)
    return p, d


_ORACLE = {}


def oracle_of(world, r, hit_capacity=None):
    """the oracle composition of a row (module cache: once per row and capacity)"""
    key = (r, hit_capacity)
    if key not in _ORACLE:
        p, d = params_of(world, r)
        _ORACLE[key] = seed_extend_oracle(world.O, world.idx(r[0]), world.gsym[r[0]], d["reads"], p,
                                          quals=d["quals"] if r[10] == Q else None, hit_capacity=hit_capacity)
    return _ORACLE[key]


def unique_jobs(want):
    return len(set(zip(want["hit_string"].tolist(), want["hit_window"][:, 0].tolist(), want["hit_window"][:, 1].tolist())))


def first_diff(a, b):
    d = np.nonzero(a != b)[0]
    return "%d differ, first reads %s: got %s want %s" % (len(d), d[:6].tolist(), a[d[:6]].tolist(), b[d[:6]].tolist())


def check_best(ws, want, what):
    got_s = ws.best_score.cpu().numpy().astype(np.int64)
    got_p = host_u32(ws.best_pos).astype(np.int64)
    assert np.array_equal(got_s, want["best_score"]), (what, "best_score", first_diff(got_s, want["best_score"]))
    assert np.array_equal(got_p, want["best_pos"]), (what, "best_pos", first_diff(got_p, want["best_pos"]))


class Switch:
    """a debug switch of include/nvbio_b200_debug.h set for the duration of a with block"""

    def __init__(self, name, value, default):
        self.f, self.value, self.default = getattr(nb.lib(), name), value, default

    def __enter__(self):
        self.f(C.c_int(self.value))

    def __exit__(self, *exc):
        self.f(C.c_int(self.default))


@pytest.mark.parametrize("row", ROWS, ids=[row_id(r) for r in ROWS])
def test_seed_extend_matrix_vs_oracle(world, row):
    """per index variant: the default call (per-read path), the same without the exact shortcut and with a truncating hit capacity ==
    the oracle; once the per-hit path, hit by hit"""
    gname = row[0]
    params, d = params_of(world, row)
    rs, gw = d["rs"], world.gw[gname]
    want = oracle_of(world, row)
    total = want["n_found"]
    assert total > 0
    cap = total + 1024
    cap3 = total // 3
    want3 = oracle_of(world, row, cap3)
    uniq = unique_jobs(want)
    # the overhanging reads whose best job has no alignment report no position (and the input really contains such reads)
    ov = np.array(d["overhang"])
    no_aln = ov[(want["best_hit"][ov] >= 0) & (want["best_pos"][ov] == NO_POS)]
    assert (want["best_score"][no_aln] == -2**30).all()
    if row[6] >= 20 and row[3] == L:
        assert len(no_aln) > 0
    for variant in INDEXES:
        fmi = world.fmi(gname, variant)
        splits = (1, 0) if variant.startswith("k") else (1,)
        for split in splits:
            what = (variant, "split" if split else "one pass")
            with Switch("nvb_debug_seed_split", split, 1):
                ws = nb.seed_extend(fmi, gw, rs, params, hit_capacity=cap)
                torch.cuda.synchronize()
                kept, found, jobs = [int(v) for v in ws.n_hits.cpu()]
                assert (kept, found) == (total, total), what
                assert uniq <= jobs <= kept, (what, uniq, jobs, kept)
                check_best(ws, want, what)
                with Switch("nvb_debug_perfect_shortcut", 0, 1):
                    ws = nb.seed_extend(fmi, gw, rs, params, hit_capacity=cap)
                    torch.cuda.synchronize()
                assert [int(v) for v in ws.n_hits.cpu()[:2]] == [total, total], what
                check_best(ws, want, what + ("no shortcut",))
                if cap3:
                    ws = nb.seed_extend(fmi, gw, rs, params, hit_capacity=cap3)
                    torch.cuda.synchronize()
                    kept, found, jobs = [int(v) for v in ws.n_hits.cpu()]
                    assert (kept, found) == (cap3, total) and jobs <= kept, what
                    check_best(ws, want3, what + ("capacity %d" % cap3,))
    # the per-hit path, every hit array (one index per row, in turn)
    variant = INDEXES[ROWS.index(row) % len(INDEXES)]
    ws = nb.seed_extend(world.fmi(gname, variant), gw, rs, params, hit_capacity=cap, keep_hits=True)
    torch.cuda.synchronize()
    kept = int(ws.n_hits[0])
    assert kept == total and uniq <= int(ws.n_hits[2]) <= kept
    assert np.array_equal(ws.hit_read.cpu().numpy()[:kept].astype(np.int64), want["hit_string"]), variant
    assert np.array_equal(host_u32(ws.hit_window)[:kept].astype(np.int64), want["hit_window"]), variant
    assert np.array_equal(ws.hit_score.cpu().numpy()[:kept].astype(np.int64), want["hit_score"]), variant
    assert np.array_equal(host_u32(ws.hit_sink)[:kept].astype(np.int64), want["hit_sink"]), variant
    check_best(ws, want, (variant, "per hit"))


def test_rejected_arguments_leave_the_library_usable(world):
    """a band the DP does not accept (8) and an alignment type of 3 raise NvbError; a valid call afterwards gives the oracle's results"""
    row = ROWS[6]
    params, d = params_of(world, row)
    fmi, gw = world.fmi(row[0], "k8ctx"), world.gw[row[0]]
    want = oracle_of(world, row)
    for field, bad in (("band_len", 8), ("type", 3)):
        p2, _ = params_of(world, row)
        setattr(p2, field, bad)
        with pytest.raises(nb.NvbError):
            nb.seed_extend(fmi, gw, d["rs"], p2, hit_capacity=want["n_found"] + 1024)
        torch.cuda.synchronize()
        ws = nb.seed_extend(fmi, gw, d["rs"], params, hit_capacity=want["n_found"] + 1024)
        torch.cuda.synchronize()
        check_best(ws, want, field)


def test_traceback_vs_oracle(world):
    """nvb_seed_extend_traceback: for every read the oracle's winning (string, window) job, traced back by the oracle -- n_ops, ops, begin
    (window begin + source.x, source.y) and strand -- for LOCAL, SEMI_GLOBAL and GLOBAL with bands 5, 15 and 31, reads overhanging the
    genome's end included (their best job has no alignment: no ops, begin (0xFFFFFFFF, 0xFFFFFFFF)).  Band 63 is refused."""
    gname = "rand"
    d = world.reads(gname, 2, False, L)
    reads, rs, gw, gsym = d["reads"], d["rs"], world.gw[gname], world.gsym[gname]
    fmi = world.fmi(gname, "fold")
    strings = []
    for r in reads:
        strings += [r, revcomp(r)]
    s_len = np.array([len(s) for s in strings], np.uint32)
    s_off = (np.cumsum(s_len) - s_len).astype(np.uint32)
    scat = np.concatenate(strings)
    no_aln_seen = 0
    for typ in (aln.LOCAL, aln.SEMI_GLOBAL, aln.GLOBAL):
        for band in (5, 15, 31):
            params = nb.SeedExtendParams(seed_len=20, seed_interval=10, band_len=band, type=typ, both_strands=True, max_seed_hits=100,
                                         scheme=aln.SimpleGotohScheme(*A))
            want = seed_extend_oracle(world.O, world.idx(gname), gsym, reads, params)
            ws = nb.seed_extend(fmi, gw, rs, params, hit_capacity=want["n_found"] + 1024, traceback=True)
            torch.cuda.synchronize()
            what = (TYPE_NAME[typ], band)
            check_best(ws, want, what)
            bh = want["best_hit"]
            has = bh >= 0
            hs = want["hit_string"][bh[has]]
            win = want["hit_window"][bh[has]]
            o = world.O.banded_traceback(band, typ, A, scat, s_off[hs], s_len[hs], gsym, win[:, 0].astype(np.uint32),
                                         (win[:, 1] - win[:, 0]).astype(np.uint32), max_ops=ws.max_ops)
            n_ops = np.zeros(len(reads), np.int64); begin = np.full((len(reads), 2), NO_POS, np.int64); strand = np.zeros(len(reads), np.int64)
            ops = np.zeros((len(reads), ws.max_ops), np.uint8)
            n_ops[has] = o["n_ops"]; ops[has] = o["ops"]; strand[has] = hs % 2
            src = o["source"].astype(np.int64)
            ok = src[:, 0] != NO_POS
            begin[np.nonzero(has)[0][ok]] = np.stack([win[ok, 0] + src[ok, 0], src[ok, 1]], axis=1)
            assert (o["score"] == want["hit_score"][bh[has]]).all(), what
            no_aln_seen += int((~ok).sum())
            got_n = ws.best_n_ops.cpu().numpy().astype(np.int64)
            assert np.array_equal(got_n, n_ops), (what, "n_ops", first_diff(got_n, n_ops))
            got_ops = ws.best_ops.cpu().numpy()
            for r in range(len(reads)):
                assert np.array_equal(got_ops[r, :n_ops[r]], ops[r, :n_ops[r]]), (what, "ops", r)
            got_b = host_u32(ws.best_begin).astype(np.int64)
            assert np.array_equal(got_b, begin), (what, "begin", first_diff(got_b[:, 0], begin[:, 0]), first_diff(got_b[:, 1], begin[:, 1]))
            got_st = ws.best_strand.cpu().numpy().astype(np.int64)
            assert np.array_equal(got_st[has], strand[has]), what
    assert no_aln_seen > 0                                                 # the overhanging reads reached the no-alignment case
    params = nb.SeedExtendParams(band_len=63)
    with pytest.raises(nb.NvbError):
        nb.seed_extend(fmi, gw, rs, params, traceback=True)
    torch.cuda.synchronize()


def test_streaming_4bit_semi_global_vs_direct_and_oracle(world):
    """StreamingSeedExtend single-end, 4-bit reads, SEMI_GLOBAL band 15, one strand, depth 2: three batches with overhanging reads, each ==
    the direct call and the oracle"""
    gname = "rand"
    gsym, gw = world.gsym[gname], world.gw[gname]
    fmi = world.fmi(gname, "k8ctx")
    params = nb.SeedExtendParams(seed_len=20, seed_interval=10, band_len=15, type=aln.SEMI_GLOBAL, both_strands=False, max_seed_hits=100,
                                 scheme=aln.SimpleGotohScheme(*B))
    batches = []
    for b in range(3):
        reads, _ = make_reads(gsym, 900 + b, L, bits=4)
        batches.append(reads)
    n_reads = len(batches[0])
    assert all(len(r) == n_reads for r in batches)
    wpr = (L + 7) // 8
    cap = 100 * n_reads
    st = nb.StreamingSeedExtend(fmi, gw, params, n_reads, L, wpr, hit_capacity=cap, depth=2, bits=4)
    try:
        hosts, directs, wants = [], [], []
        for reads in batches:
            rs, stride = string_set(reads, 4, L)
            assert stride == wpr * 8
            hosts.append(rs.words[:n_reads * wpr].reshape(n_reads, wpr).cpu().pin_memory())
            ws = nb.seed_extend(fmi, gw, rs, params, hit_capacity=cap)
            torch.cuda.synchronize()
            directs.append((ws.best_score.cpu().clone(), ws.best_pos.cpu().clone(), ws.n_hits.cpu().clone()))
            wants.append(seed_extend_oracle(world.O, world.idx(gname), gsym, reads, params, hit_capacity=cap))
        # (the results are views of the pipeline's host buffers, reused `depth` submissions later: keep copies)
        tickets = [st.submit(hosts[0]), st.submit(hosts[1])]
        got = [tuple(v.clone() for v in st.result(tickets[0]))]
        tickets.append(st.submit(hosts[2]))
        got += [tuple(v.clone() for v in st.result(t)) for t in tickets[1:]]
        for b in range(3):
            sc, ps, nh = got[b]
            assert torch.equal(sc, directs[b][0]) and torch.equal(ps, directs[b][1]) and torch.equal(nh, directs[b][2]), b
            assert np.array_equal(sc.numpy().astype(np.int64), wants[b]["best_score"]), (b, first_diff(sc.numpy().astype(np.int64), wants[b]["best_score"]))
            gp = ps.numpy().view(np.uint32).astype(np.int64)
            assert np.array_equal(gp, wants[b]["best_pos"]), (b, first_diff(gp, wants[b]["best_pos"]))
            assert int(nh[0]) == wants[b]["n_hits"] and int(nh[1]) == wants[b]["n_found"], b
    finally:
        st.close()


def test_paired_with_mates_at_the_genome_ends_vs_oracle(world):
    """nvb_seed_extend_paired, LOCAL band 31: pairs inside the genome, pairs whose mates lie at its start, and pairs with a mate that runs
    past its end (no alignment: that mate is unaligned, the other one anchors a rescue) == seed_extend_paired_oracle"""
    gname = "rand"
    gsym, gw = world.gsym[gname], world.gw[gname]
    n = len(gsym)
    fmi = world.fmi(gname, "k8loc")
    rng = np.random.default_rng(77)
    m1, m2 = [], []
    for i in range(300):
        p = int(rng.integers(0, n - 600)); frag = int(rng.integers(250, 400))
        m1.append(mutate(rng, gsym[p:p + L + 10], 0.01, 0.002)[:L])
        m2.append(revcomp(mutate(rng, gsym[p + frag - L - 10:p + frag], 0.01, 0.002)[-L:]))
    for p in range(0, 40, 4):                                                # at the genome's start
        m1.append(gsym[p:p + L].copy()); m2.append(revcomp(gsym[p + 200:p + 200 + L]))
        m1.append(revcomp(gsym[p + 200:p + 200 + L])); m2.append(gsym[p:p + L].copy())
    for k in (20, 60, 100, L - 1):                                           # a mate past the genome's end
        for t in range(3):
            tail = rng.integers(0, 4, L - k).astype(np.uint8)
            over = np.concatenate([gsym[n - k:], tail])
            m1.append(gsym[n - k - 250:n - k - 250 + L].copy()); m2.append(revcomp(over))
            m1.append(over); m2.append(revcomp(gsym[n - 300:n - 300 + L]))
    n_pairs = len(m1)
    reads = m1 + m2
    rs, _ = string_set(reads, 2, L)
    params = nb.SeedExtendParams(seed_len=20, seed_interval=10, band_len=31, type=aln.LOCAL, both_strands=True, max_seed_hits=100,
                                 scheme=aln.SimpleGotohScheme(*A))
    for pair in (nb.PairParams(min_frag=0, max_frag=500, min_mate_score=50), nb.PairParams(min_frag=100, max_frag=420, min_mate_score=80)):
        ws = nb.seed_extend_paired(fmi, gw, rs, params, pair, hit_capacity=100 * len(reads))
        torch.cuda.synchronize()
        want = seed_extend_paired_oracle(world.O, world.idx(gname), gsym, reads, params, pair, n_pairs)
        assert tuple(int(v) for v in ws.n_rescue.cpu()) == want["n_rescue"]
        for k in ("pair_flags", "pair_score", "mate_score", "mate_strand"):
            got = getattr(ws, k).cpu().numpy().astype(np.int64)
            assert np.array_equal(got, want[k]), (k, first_diff(got.reshape(-1), want[k].reshape(-1)))
        got = host_u32(ws.mate_pos).astype(np.int64)
        assert np.array_equal(got, want["mate_pos"]), ("mate_pos", first_diff(got.reshape(-1), want["mate_pos"].reshape(-1)))
        fl = want["pair_flags"]
        assert (fl == 1).sum() > 200 and ((fl == 2) | (fl == 4)).sum() > 0
