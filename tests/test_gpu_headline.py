"""-m gpu: parity and index verification ON THE EXACT HEADLINE CONFIGURATION that bench.py times (BASELINE.json configs[2]):
3,000,000,000 bp synthetic genome, device suffix sort, FULL suffix array (sa_interval = 1) and the 16-mer range table
(ktab_k = 16) -- n > 2^31, the sizes where 32-bit index arithmetic breaks.

  * the 3 Gbp index itself (reference's own property tests, nvbio-test/fmindex_test.cu:582-664, 230-239, rank_test.cu:55-86):
    sampled adjacent-suffix order, BWT == text[SA-1], occ counters vs the BWT blocks, L2 == symbol counts,
    text[locate(match(p)) ..] == p;
  * seed + extend on bench.py's own CPU-leg reads: best score per read, every per-hit score / sink and the hit count equal
    the reference's own templates (oracle/_ref, OpenMP) run over the SAME index, through both pipeline paths (their outputs'
    digests are committed, tests/reference_digests.py)."""
import os

import numpy as np
import pytest
import torch

import nvbio_b200 as nb
from nvbio_b200 import aln, synth
from nvbio_b200.strings import PackedStringSet
from oracle import orc
from oracle.cpu_pipeline import cpu_seed_extend, gather_2bit
from tests.gpu_util import require_gpu, host_u32
from tests.reference_digests import Reference
from tests.test_gpu_fullsize import live_reference

pytestmark = pytest.mark.gpu

N = 3_000_000_000
KTAB_K, SA_INTERVAL = 16, 1
READ_LEN, SEED_LEN, SEED_INTERVAL, BAND = 150, 20, 10, 31
SCHEME = (2, -2, -5, -3)


def keys(gwh, pos, nsym):
    """the nsym <= 32 symbols of a 2-bit big-endian stream starting at int64 positions `pos`, as uint64 keys (first symbol most significant)"""
    pos = np.asarray(pos, dtype=np.int64)
    w = pos >> 4
    sh = (2 * (pos & 15)).astype(np.uint64)
    a, b, c = (gwh[w + i].astype(np.uint64) for i in range(3))
    hi = (a << np.uint64(32)) | b                       # symbols 0..31 of the word pair
    lo = c << np.uint64(32)
    k = np.where(sh > 0, (hi << sh) | (lo >> (np.uint64(64) - np.where(sh > 0, sh, np.uint64(1)))), hi)
    return k >> np.uint64(64 - 2 * nsym)


@pytest.fixture(scope="module")
def H():
    require_gpu()
    free, total = torch.cuda.mem_get_info()
    if total < 150e9:
        pytest.skip("needs a 180 GB part")
    genome = synth.random_genome_words(N)
    fmi, _ = nb.FMIndexDevice.from_text(genome, N, sa_interval=SA_INTERVAL)
    torch.cuda.empty_cache()
    fmi.build_ktab(KTAB_K, located=True, text=genome)   # bench.py's default: 16-byte entries {x, y, SA[x], SA[y] | text context}
    torch.cuda.synchronize()
    gwh = host_u32(genome)
    return dict(genome=genome, fmi=fmi, gwh=gwh)


def test_3gbp_suffix_array_sampled_order(H):
    """2M random pairs of adjacent SA rows: suffix SA[r] < suffix SA[r+1] (64-symbol prefixes decide; ties would fail)"""
    fmi, gwh = H["fmi"], H["gwh"]
    g = torch.Generator(device="cuda"); g.manual_seed(1)
    rows = torch.unique(torch.randint(1, N, (2_000_000,), generator=g, device="cuda", dtype=torch.int64))   # SA rows 1 .. n-1 (row 0 is `$`)
    sa = fmi.ssa                                                                              # full SA: ssa[r] = SA[r], ssa[0] = -1
    assert sa.numel() == N + 1
    p0 = (sa[rows].to(torch.int64) & 0xFFFFFFFF).cpu().numpy()
    p1 = (sa[rows + 1].to(torch.int64) & 0xFFFFFFFF).cpu().numpy()
    ok = (p0 < N - 64) & (p1 < N - 64)
    assert ok.mean() > 0.999
    p0, p1 = p0[ok], p1[ok]
    a1, b1 = keys(gwh, p0, 32), keys(gwh, p1, 32)
    a2, b2 = keys(gwh, p0 + 32, 32), keys(gwh, p1 + 32, 32)
    assert np.all((a1 < b1) | ((a1 == b1) & (a2 < b2)))
    # the suffix array is a permutation at this size: distinct positions in the sample, all < n
    assert p0.max() < N and len(np.unique(p0)) == len(p0) > 1_900_000
    assert (int(sa[0].item()) & 0xFFFFFFFF) == 0xFFFFFFFF


def test_3gbp_bwt_occ_L2(H):
    fmi, gwh = H["fmi"], H["gwh"]
    primary = fmi.primary
    g = torch.Generator(device="cuda"); g.manual_seed(2)
    rows = torch.randint(1, N + 1, (2_000_000,), generator=g, device="cuda", dtype=torch.int64)
    rows = rows[rows != primary]
    sa = (fmi.ssa[rows].to(torch.int64) & 0xFFFFFFFF)
    k = torch.where(rows < primary, rows, rows - 1)                                           # BWT index of row r (`$` row removed)
    blk = fmi.bwt_occ.view(-1, 8)
    word = blk[k >> 6, (k & 63) >> 4].to(torch.int64) & 0xFFFFFFFF
    sym = ((word >> (30 - 2 * (k & 15))) & 3).cpu().numpy()
    sa = sa.cpu().numpy()
    assert (sa > 0).all()                                                                     # SA[r] = 0 only at r = primary
    assert np.array_equal(sym, gather_2bit(gwh, sa - 1))                                      # bwt[r] = text[SA[r] - 1]
    # occ counters: occ[k+1] - occ[k] = symbol counts of block k, on 1M sampled blocks; occ[0] = 0; totals = L2
    n_blocks = (N + 63) // 64
    kb = torch.randint(0, n_blocks - 1, (1_000_000,), generator=g, device="cuda", dtype=torch.int64)
    b0 = blk[kb].cpu().numpy().view(np.uint32); b1 = blk[kb + 1].cpu().numpy().view(np.uint32)
    sh = (30 - 2 * np.arange(16)).astype(np.uint32)
    syms = ((b0[:, :4, None] >> sh[None, None, :]) & 3).reshape(len(b0), 64)
    for c in range(4):
        assert np.array_equal((syms == c).sum(1).astype(np.uint32), b1[:, 4 + c] - b0[:, 4 + c]), c
    assert not blk[0, 4:].any()
    # L2 = exclusive symbol counts of the whole text (counted independently on the device, 16 symbols per word)
    gw = H["genome"][: (N + 15) // 16].to(torch.int64) & 0xFFFFFFFF
    assert N % 16 == 0
    cnt = [0, 0, 0, 0]
    for s in range(16):
        v = (gw >> (30 - 2 * s)) & 3
        for c in range(4):
            cnt[c] += int((v == c).sum().item())
    assert list(fmi.L2) == [0, cnt[0], cnt[0] + cnt[1], cnt[0] + cnt[1] + cnt[2], N]


def test_3gbp_locate_of_match_is_the_pattern(H):
    """nvbio-test/fmindex_test.cu:582-664 shaped: 1M 20-mers sampled from the text -- every located hit of match(p) spells p,
    and the position it was sampled from is among the hits; with and without the 16-mer table, full SA and SA every 16"""
    fmi, genome, gwh = H["fmi"], H["genome"], H["gwh"]
    nq, L = 1_000_000, 20
    sw, spos = synth.sample_seeds(genome, N, nq, L)
    q = PackedStringSet.fixed(sw.reshape(-1), nq, L, stride=32)
    flt = nb.FMIndexFilterDevice()
    n_hits = flt.rank(fmi, q)
    ranges = host_u32(flt.ranges())
    assert (ranges[:, 0] <= ranges[:, 1]).all() and n_hits >= nq
    hits = host_u32(flt.locate(0, n_hits))
    want = keys(gwh, spos.cpu().numpy().astype(np.int64), L)
    got = keys(gwh, hits[:, 0].astype(np.int64), L)
    assert np.array_equal(got, want[hits[:, 1]])
    found = np.zeros(nq, bool)
    found[hits[hits[:, 0].astype(np.int64) == spos.cpu().numpy().astype(np.int64)[hits[:, 1]], 1]] = True
    assert found.all()
    # the same ranges and positions from the reference-format view of this index (no table, SA every 16)
    plain = nb.FMIndexDevice(fmi.bwt_occ, fmi.ssa[::16].contiguous(), fmi.L2, N, fmi.primary, sa_interval=16)
    flt2 = nb.FMIndexFilterDevice()
    assert flt2.rank(plain, q) == n_hits
    assert np.array_equal(host_u32(flt2.ranges()), ranges)
    assert np.array_equal(host_u32(flt2.locate(0, n_hits)), hits)


def _unpack_rows(words, L):
    i = np.arange(L)
    sh = (30 - 2 * (i & 15)).astype(np.uint32)
    return ((words[:, i >> 4] >> sh) & 3).astype(np.uint8)


def test_headline_seed_extend_equals_reference(H, request):
    """bench.py's CPU-leg read sample (20,000 x 150 bp, 1% substitutions, 0.1% indels, both strands) over the headline index:
    hit count, every per-hit (score, sink) in the reference's slot order and the best score per read == the reference's own
    templates (nvbio::match -> locate -> aln::banded_alignment_score<31> -> max) over the same index in the reference's format"""
    R = Reference(request, live_reference)
    fmi, genome, gwh = H["fmi"], H["genome"], H["gwh"]
    n_reads = 20_000
    rw, pos, strand = synth.sample_reads(genome, N, n_reads, READ_LEN, sub_rate=0.01, indel_rate=0.001,
                                         seed=synth.SEED_QUERIES + 7919 * 1000, mut_seed=synth.SEED_MUT + 104729 * 1000)
    rw = rw.contiguous()
    want = None
    if R.live:
        idx = orc._Index(n=N, primary=fmi.primary, bwt_occ=host_u32(fmi.bwt_occ), ssa=host_u32(fmi.ssa[::16].contiguous()), L2=np.array(fmi.L2, np.uint32))
        want = cpu_seed_extend(R.live, idx, gwh, _unpack_rows(host_u32(rw), READ_LEN), SEED_LEN, SEED_INTERVAL, BAND, 1, SCHEME, True, 100)
    rs = PackedStringSet.fixed(rw.reshape(-1), n_reads, READ_LEN, stride=rw.shape[1] * 16)
    params = nb.SeedExtendParams(seed_len=SEED_LEN, seed_interval=SEED_INTERVAL, band_len=BAND, type=aln.LOCAL, both_strands=True,
                                 max_seed_hits=100, dedup_jobs=True, scheme=aln.SimpleGotohScheme(*SCHEME))
    # the path the benchmark times (per read, no per-hit arrays)
    ws = nb.seed_extend(fmi, genome, rs, params, hit_capacity=24 * n_reads)
    torch.cuda.synchronize()
    kept, total, jobs = [int(v) for v in ws.n_hits.cpu()]
    assert kept == total and 0 < jobs <= total
    best = ws.best_score.cpu().numpy().astype(np.int64)
    R.same([total, best], lambda: [want["n_hits"], want["best_score"]])
    assert (best > READ_LEN).mean() > 0.99
    # the per-hit path: every hit's score in the reference's slot order
    ws2 = nb.seed_extend(fmi, genome, rs, params, hit_capacity=24 * n_reads, keep_hits=True)
    torch.cuda.synchronize()
    assert [int(v) for v in ws2.n_hits.cpu()][:2] == [total, total]
    R.same([ws2.hit_score[:total].cpu().numpy(), ws2.hit_read[:total].cpu().numpy() // 2], lambda: [want["hit_score"], want["hit_read"]])
    assert np.array_equal(ws2.best_score.cpu().numpy().astype(np.int64), best)
    assert np.array_equal(ws2.best_pos.cpu().numpy(), ws.best_pos.cpu().numpy())
