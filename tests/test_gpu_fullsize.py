"""-m gpu: parity at BASELINE.json's FULL sizes against the reference's own templates (oracle/_ref, OpenMP over all host cores):
their outputs' digests are committed (tests/reference_digests.py), so these comparisons run without that library."""
import os

import numpy as np
import pytest
import torch
from oracle import orc
from oracle.cpu_pipeline import cpu_seed_extend
import nvbio_b200 as nb
from nvbio_b200 import aln, synth
from nvbio_b200.strings import PackedStringSet
from tests.gpu_util import require_gpu, host_u32
from tests.reference_digests import Reference

pytestmark = pytest.mark.gpu


def _unpack_rows(words, L):
    i = np.arange(L)
    sh = (30 - 2 * (i & 15)).astype(np.uint32)
    return ((words[:, i >> 4] >> sh) & 3).astype(np.uint8)


def live_reference():
    r = orc.Ref()
    r.set_num_threads(len(os.sched_getaffinity(0)))
    return r


@pytest.fixture
def R(request):
    require_gpu()
    return Reference(request, live_reference)


@pytest.fixture(scope="module")
def genome100():
    require_gpu()
    n = 100_000_000
    gw = synth.random_genome_words(n)
    fmi, _ = nb.FMIndexDevice.from_text(gw, n)            # reference format (SA every 16)
    host = fmi.to_host()
    idx = orc._Index(n=n, primary=host["primary"], bwt_occ=host["bwt_occ"], ssa=host["ssa"], L2=host["L2"])
    return n, gw, fmi, idx


def test_c2_full_1M_seeds_100Mbp(R, genome100):
    """configs[1]: every one of the 1M x 22 bp SA ranges and every located hit position bit-identical to nvbio::match /
    nvbio::locate; also with the k-mer table and the full suffix array switched on"""
    n, gw, fmi, idx = genome100
    nq, L = 1_000_000, 22
    sw, pos = synth.sample_seeds(gw, n, nq, L, random_frac=0.1)          # 10% random seeds: mostly empty ranges
    q = PackedStringSet.fixed(sw.reshape(-1), nq, L, stride=32)
    sym = _unpack_rows(host_u32(sw), L).reshape(-1)
    ranges = host_u32(nb.match(fmi, q))
    R.same(ranges, lambda: R.live.match(idx, sym, (np.arange(nq, dtype=np.uint32) * L), np.full(nq, L, np.uint32))[0])
    flt = nb.FMIndexFilterDevice()
    n_hits = flt.rank(fmi, q)
    sizes = np.where(ranges[:, 0] <= ranges[:, 1], ranges[:, 1].astype(np.int64) - ranges[:, 0] + 1, 0)
    assert n_hits == int(sizes.sum())
    hits = host_u32(flt.locate(0, n_hits))
    rows = np.repeat(ranges[:, 0].astype(np.int64), sizes) + (np.arange(n_hits) - np.repeat(np.cumsum(sizes) - sizes, sizes))
    R.same(hits[:, 0], lambda: R.live.locate(idx, rows.astype(np.uint32)))
    assert np.array_equal(hits[:, 1].astype(np.int64), np.repeat(np.arange(nq), sizes))
    # B200 extensions leave every range / position unchanged
    ext, _ = nb.FMIndexDevice.from_text(gw, n, sa_interval=1)
    ext.build_ktab(12)
    assert np.array_equal(host_u32(nb.match(ext, q)), ranges)
    flt2 = nb.FMIndexFilterDevice()
    assert flt2.rank(ext, q) == n_hits
    assert np.array_equal(host_u32(flt2.locate(0, n_hits)), hits)


def test_c4_slice_1M_alignments(R, genome100):
    """configs[3] shape (151 bp reads vs 300 bp windows, LOCAL (2,-2,-5,-3)), 1M alignments per band: (score, sink) of every
    alignment bit-identical to aln::banded_alignment_score<B> run by the reference on the host"""
    n, gw, fmi, idx = genome100
    n_al, M, W = 1_000_000, 151, 300
    rw, pos, _ = synth.sample_reads(gw, n, n_al, M, rc_half=False)
    begin = synth.windows_for_reads(n, pos, M, W)
    P = PackedStringSet.fixed(rw.reshape(-1), n_al, M, stride=rw.shape[1] * 16)
    T = PackedStringSet(words=gw, bits=2, big_endian=True, offsets=begin.to(torch.int32), lengths=None, stride=0, length=W, count=n_al)
    pat = _unpack_rows(host_u32(rw), M).reshape(-1)
    gwh = host_u32(gw)
    wpos = begin.cpu().numpy()[:, None] + np.arange(W)[None, :]
    txt = (((gwh[wpos >> 4] >> (30 - 2 * (wpos & 15)).astype(np.uint32)) & 3).astype(np.uint8)).reshape(-1)
    p_off = np.arange(n_al, dtype=np.uint32) * M; p_len = np.full(n_al, M, np.uint32)
    t_off = np.arange(n_al, dtype=np.uint32) * W; t_len = np.full(n_al, W, np.uint32)
    for band in (15, 31):
        s, k = aln.batch_banded_alignment_score(band, aln.make_gotoh_aligner(aln.LOCAL, aln.SimpleGotohScheme(2, -2, -5, -3)), P, T)
        kk = host_u32(k)
        R.same([s.cpu().numpy(), kk[:, 0], kk[:, 1]], lambda: R.live.banded_gotoh(band, 1, (2, -2, -5, -3), pat, p_off, p_len, txt, t_off, t_len)[:3])


def test_c1_sw_benchmark_10k(R):
    """configs[0] (sw-benchmark's CPU-runnable case): 10K x 100 bp reads vs 1 Kbp references, Gotoh GLOBAL (2,-1,-2,-1) as
    sw-benchmark sets it (sw-benchmark.cu:592-641) -- the full-matrix DP of every read against its whole reference and the
    band-15 DP, each (score, sink) bit-identical to the reference's own templates run on the host; LOCAL and SEMI_GLOBAL too"""
    rng = np.random.default_rng(77)
    n_al, M, N = 10_000, 100, 1000
    txt = rng.integers(0, 4, (n_al, N)).astype(np.uint8)
    st = rng.integers(0, N - M, n_al)
    pat = np.stack([txt[i, st[i]:st[i] + M] for i in range(n_al)])
    pat = np.where(rng.random(pat.shape) < 0.04, rng.integers(0, 4, pat.shape), pat).astype(np.uint8)
    p_off = np.arange(n_al, dtype=np.uint32) * M; p_len = np.full(n_al, M, np.uint32)
    t_off = np.arange(n_al, dtype=np.uint32) * N; t_len = np.full(n_al, N, np.uint32)
    P = PackedStringSet.from_symbols(pat.reshape(-1), p_off, p_len, bits=2, big_endian=True)
    T = PackedStringSet.from_symbols(txt.reshape(-1), t_off, t_len, bits=2, big_endian=True)
    scheme = (2, -1, -2, -1)
    for typ in (0, 1, 2):
        s, k = aln.batch_alignment_score(aln.make_gotoh_aligner(typ, aln.SimpleGotohScheme(*scheme)), P, T)
        kk = host_u32(k)
        R.same([s.cpu().numpy(), kk[:, 0], kk[:, 1]], lambda: R.live.gotoh_full(typ, scheme, pat.reshape(-1), p_off, p_len, txt.reshape(-1), t_off, t_len))
    s, k = aln.batch_banded_alignment_score(15, aln.make_gotoh_aligner(aln.GLOBAL, aln.SimpleGotohScheme(*scheme)), P, T)
    kk = host_u32(k)
    R.same([s.cpu().numpy(), kk[:, 0], kk[:, 1]], lambda: R.live.banded_gotoh(15, 0, scheme, pat.reshape(-1), p_off, p_len, txt.reshape(-1), t_off, t_len)[:3])


def test_c3_100k_reads_pipeline(R, genome100):
    """configs[2] shape (150 bp reads, 20 bp seeds every 10 bp, both strands, band 31 LOCAL) on 100K reads: best score per
    read and the number of hits identical to the reference composition (match -> locate -> banded score -> max)"""
    n, gw, fmi, idx = genome100
    n_reads = 100_000
    rw, pos, strand = synth.sample_reads(gw, n, n_reads, 150, seed=11, mut_seed=12)
    rs = PackedStringSet.fixed(rw.reshape(-1), n_reads, 150, stride=rw.shape[1] * 16)
    ext, _ = nb.FMIndexDevice.from_text(gw, n, sa_interval=1)
    ext.build_ktab(12)
    for index in (fmi, ext):
        ws = nb.seed_extend(index, gw, rs, nb.SeedExtendParams(), hit_capacity=40 * n_reads)
        torch.cuda.synchronize()
        kept, total, jobs = [int(v) for v in ws.n_hits.cpu()]
        assert kept == total
        want = (lambda w: [w["n_hits"], w["best_score"]])
        R.same([total, ws.best_score.cpu().numpy()], lambda: want(cpu_seed_extend(R.live, idx, host_u32(gw), _unpack_rows(host_u32(rw), 150))))
