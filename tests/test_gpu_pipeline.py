"""-m gpu: the seed+extend composition (seeds -> match -> locate -> window -> banded Gotoh -> best per read)
against the oracle composition, hit by hit."""
import numpy as np
import pytest
import torch
from oracle import orc
import nvbio_b200 as nb
from nvbio_b200 import aln, synth
from nvbio_b200.strings import PackedStringSet, pack_symbols, unpack_symbols
from tests.gpu_util import require_gpu, dev_u32, host_u32
from tests.pipeline_oracle import seed_extend_oracle

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("both,read_len,ragged", [(True, 150, False), (False, 100, False), (True, 120, True)])
def test_seed_extend_vs_oracle(both, read_len, ragged):
    require_gpu()
    O = orc.Oracle()
    n = 200_000
    gw = synth.random_genome_words(n, seed=77)
    gsym = unpack_symbols(host_u32(gw), n)
    idx = O.build_index(gsym)
    fmi = nb.FMIndexDevice.from_host(idx.bwt_occ, idx.ssa, idx.L2, idx.n, idx.primary)
    n_reads = 600
    rw, pos, strand = synth.sample_reads(gw, n, n_reads, read_len, sub_rate=0.02, indel_rate=0.004, seed=5, mut_seed=6)
    wpr = rw.shape[1]
    reads_sym = [unpack_symbols(host_u32(rw[i]), read_len) for i in range(n_reads)]
    if ragged:
        rng = np.random.default_rng(3)
        lens = rng.integers(read_len - 50, read_len + 1, n_reads).astype(np.uint32)
        reads_sym = [r[:l] for r, l in zip(reads_sym, lens)]
        rs = PackedStringSet(words=rw.reshape(-1), bits=2, big_endian=True,
                             offsets=(torch.arange(n_reads, device="cuda", dtype=torch.int32) * (wpr * 16)),
                             lengths=dev_u32(lens), stride=0, length=read_len, count=n_reads)
    else:
        rs = PackedStringSet.fixed(rw.reshape(-1), n_reads, read_len, stride=wpr * 16)
    params = nb.SeedExtendParams(seed_len=20, seed_interval=10, band_len=31, type=aln.LOCAL, both_strands=both,
                                 max_seed_hits=50, scheme=aln.SimpleGotohScheme(2, -2, -5, -3))
    ws = nb.seed_extend(fmi, gw, rs, params, hit_capacity=64 * n_reads, keep_hits=True)
    torch.cuda.synchronize()
    want = seed_extend_oracle(O, idx, gsym, reads_sym, params)
    kept, total, jobs = [int(v) for v in ws.n_hits.cpu()]
    assert kept == total == want["n_hits"]
    uniq = len(set(zip(want["hit_string"].tolist(), want["hit_window"][:, 0].tolist(), want["hit_window"][:, 1].tolist())))
    assert jobs == uniq < kept              # identical (strand, window) jobs are scored once
    assert np.array_equal(ws.hit_read.cpu().numpy()[:kept].astype(np.int64), want["hit_string"])
    assert np.array_equal(host_u32(ws.hit_window)[:kept].astype(np.int64), want["hit_window"])
    assert np.array_equal(ws.hit_score.cpu().numpy()[:kept].astype(np.int64), want["hit_score"])
    assert np.array_equal(host_u32(ws.hit_sink)[:kept].astype(np.int64), want["hit_sink"])
    assert np.array_equal(ws.best_score.cpu().numpy().astype(np.int64), want["best_score"])
    assert np.array_equal(host_u32(ws.best_pos).astype(np.int64), want["best_pos"])
    # without job de-duplication: same outputs, every hit scored separately
    params.dedup_jobs = False
    ws2 = nb.seed_extend(fmi, gw, rs, params, hit_capacity=64 * n_reads, keep_hits=True)
    torch.cuda.synchronize()
    assert int(ws2.n_hits[2]) == kept
    assert torch.equal(ws2.hit_score[:kept], ws.hit_score[:kept]) and torch.equal(ws2.hit_sink[:kept], ws.hit_sink[:kept])
    assert torch.equal(ws2.best_score, ws.best_score) and torch.equal(ws2.best_pos, ws.best_pos)
    # most reads are found at their true locus (every other read is reverse-complemented: single-strand
    # runs can only find the forward half)
    found = (ws.best_score.cpu().numpy() > read_len)   # > half of the perfect score 2*len
    if ragged:
        found = (ws.best_score.cpu().numpy() > np.array([len(r) for r in reads_sym]))
    assert found.mean() > (0.9 if both else 0.45)


def test_seed_extend_4bit_reads_with_N():
    require_gpu()
    O = orc.Oracle()
    n = 50_000
    gw = synth.random_genome_words(n, seed=9)
    gsym = unpack_symbols(host_u32(gw), n)
    idx = O.build_index(gsym)
    fmi = nb.FMIndexDevice.from_host(idx.bwt_occ, idx.ssa, idx.L2, idx.n, idx.primary)
    rng = np.random.default_rng(0)
    reads = []
    for i in range(200):
        p = int(rng.integers(0, n - 100)); r = gsym[p:p + 100].copy()
        r[rng.integers(0, 100, 3)] = 4
        reads.append(r)
    sym = np.concatenate(reads)
    rs = PackedStringSet.from_symbols(sym, np.arange(200) * 100, np.full(200, 100), bits=4, big_endian=True)
    params = nb.SeedExtendParams(seed_len=20, seed_interval=10, band_len=31, both_strands=True, max_seed_hits=10)
    ws = nb.seed_extend(fmi, gw, rs, params, hit_capacity=20000, keep_hits=True)
    torch.cuda.synchronize()
    want = seed_extend_oracle(O, idx, gsym, reads, params)
    kept = int(ws.n_hits[0])
    assert kept == want["n_hits"]
    assert np.array_equal(ws.hit_score.cpu().numpy()[:kept].astype(np.int64), want["hit_score"])
    assert np.array_equal(ws.best_score.cpu().numpy().astype(np.int64), want["best_score"])


def test_hit_capacity_is_respected():
    require_gpu()
    n = 100_000
    gw = synth.random_genome_words(n, seed=1)
    fmi, _ = nb.FMIndexDevice.from_text(gw, n)
    rw, pos, strand = synth.sample_reads(gw, n, 500, 150, sub_rate=0.0, indel_rate=0.0)
    rs = PackedStringSet.fixed(rw.reshape(-1), 500, 150, stride=rw.shape[1] * 16)
    ws = nb.seed_extend(fmi, gw, rs, nb.SeedExtendParams(), hit_capacity=1000, keep_hits=True)
    kept, total, jobs = [int(v) for v in ws.n_hits.cpu()]
    assert kept == 1000 and total > 1000 and jobs <= kept


def test_unaligned_2bit_reads_and_streaming_api():
    """2-bit reads of odd lengths packed back to back (offsets not word aligned) through the word-wise [fw,rc]
    materialisation, and the host-to-host StreamingSeedExtend API against the plain call."""
    require_gpu()
    O = orc.Oracle()
    n = 120_000
    gw = synth.random_genome_words(n, seed=31)
    gsym = unpack_symbols(host_u32(gw), n)
    idx = O.build_index(gsym)
    fmi = nb.FMIndexDevice.from_host(idx.bwt_occ, idx.ssa, idx.L2, idx.n, idx.primary)
    rng = np.random.default_rng(12)
    reads, offs, lens, o = [], [], [], 0
    for i in range(400):
        L = int(rng.integers(61, 151)); p = int(rng.integers(0, n - L))
        r = gsym[p:p + L].copy()
        if i & 1:
            r = (3 - r)[::-1].copy()
        reads.append(r); offs.append(o); lens.append(L); o += L
    rs = PackedStringSet.from_symbols(np.concatenate(reads), offs, lens, bits=2, big_endian=True)
    rs.length = 150
    params = nb.SeedExtendParams(max_seed_hits=20)
    ws = nb.seed_extend(fmi, gw, rs, params, hit_capacity=40000, keep_hits=True)
    torch.cuda.synchronize()
    want = seed_extend_oracle(O, idx, gsym, reads, params)
    kept = int(ws.n_hits[0])
    assert kept == want["n_hits"]
    assert np.array_equal(ws.hit_score.cpu().numpy()[:kept].astype(np.int64), want["hit_score"])
    assert np.array_equal(host_u32(ws.hit_window)[:kept].astype(np.int64), want["hit_window"])
    assert np.array_equal(ws.best_score.cpu().numpy().astype(np.int64), want["best_score"])
    # streaming API on fixed-length batches
    rw, pos, strand = synth.sample_reads(gw, n, 1000, 150, seed=3, mut_seed=4)
    plain = nb.seed_extend(fmi, gw, PackedStringSet.fixed(rw.reshape(-1), 1000, 150, stride=rw.shape[1] * 16), nb.SeedExtendParams(), hit_capacity=64000)
    torch.cuda.synchronize()
    st = nb.StreamingSeedExtend(fmi, gw, nb.SeedExtendParams(), 1000, 150, rw.shape[1], hit_capacity=64000, depth=2)
    host = rw.cpu().pin_memory()
    tickets = [st.submit(host) for _ in range(2)]
    for t in tickets + [st.submit(host)]:
        sc, ps, nh = st.result(t)
        assert torch.equal(sc, plain.best_score.cpu()) and torch.equal(ps, plain.best_pos.cpu())
        assert torch.equal(nh, plain.n_hits.cpu())


def test_stage_times_belong_to_the_last_direct_call(monkeypatch):
    """last_stage_ms() reports the most recent direct seed_extend call: StreamingSeedExtend batches in flight on two compute streams
    record no stage events and leave the reported times as they were"""
    from nvbio_b200.pipeline import last_stage_ms
    require_gpu()
    n = 120_000
    gw = synth.random_genome_words(n, seed=31)
    fmi, _ = nb.FMIndexDevice.from_text(gw, n)
    rw, _, _ = synth.sample_reads(gw, n, 1000, 150, seed=3, mut_seed=4)
    nb.seed_extend(fmi, gw, PackedStringSet.fixed(rw.reshape(-1), 1000, 150, stride=rw.shape[1] * 16), nb.SeedExtendParams(), hit_capacity=64000)
    before = last_stage_ms()
    monkeypatch.setenv("NVB_PIPELINE_COMPUTE_STREAMS", "2")
    st = nb.StreamingSeedExtend(fmi, gw, nb.SeedExtendParams(), 1000, 150, rw.shape[1], hit_capacity=64000, depth=2)
    host = rw.cpu().pin_memory()
    for _ in range(3):
        for t in [st.submit(host) for _ in range(2)]:
            st.result(t)
    st.close()
    torch.cuda.synchronize()
    assert last_stage_ms() == before


def test_best_alignment_traceback():
    """CIGAR of every read's best hit: re-applying the ops to the genome reproduces the read (up to its substitutions) and
    the score; equals the oracle traceback of the same (strand, window) job"""
    require_gpu()
    O = orc.Oracle()
    n = 150_000
    gw = synth.random_genome_words(n, seed=41)
    gsym = unpack_symbols(host_u32(gw), n)
    fmi, _ = nb.FMIndexDevice.from_text(gw, n, sa_interval=1)
    n_reads = 500
    rw, pos, strand = synth.sample_reads(gw, n, n_reads, 150, sub_rate=0.02, indel_rate=0.01, seed=8, mut_seed=9)
    rs = PackedStringSet.fixed(rw.reshape(-1), n_reads, 150, stride=rw.shape[1] * 16)
    ws = nb.seed_extend(fmi, gw, rs, nb.SeedExtendParams(), hit_capacity=64 * n_reads, keep_hits=True, traceback=True)
    torch.cuda.synchronize()
    score = ws.best_score.cpu().numpy(); n_ops = ws.best_n_ops.cpu().numpy(); ops = ws.best_ops.cpu().numpy()
    begin = host_u32(ws.best_begin); st = ws.best_strand.cpu().numpy(); bpos = host_u32(ws.best_pos)
    checked = 0
    for r in range(n_reads):
        if score[r] == -2**31:
            assert n_ops[r] == 0
            continue
        read = unpack_symbols(host_u32(rw[r]), 150)
        if st[r]:
            read = (3 - read)[::-1]
        j, i = int(begin[r, 0]), int(begin[r, 1])
        s, prev = 0, -1
        for op in ops[r, :n_ops[r]][::-1]:
            if op == 0:
                s += 2 if read[i] == gsym[j] else -2; i += 1; j += 1
            elif op == 1:
                s += -3 if prev == 1 else -5; i += 1
            else:
                s += -3 if prev == 2 else -5; j += 1
            prev = op
        assert s == score[r] and j == int(bpos[r]), (r, s, score[r], j, bpos[r])
        checked += 1
    assert checked > 0.9 * n_reads
    # indel-carrying reads produce I/D ops
    assert (ops == 1).any() and (ops == 2).any()


def test_paired_end_vs_oracle():
    """nvb_seed_extend_paired == the oracle composition (single-end stages + pairing rules + opposite-mate full-matrix Gotoh):
    concordant pairs, rescued mates (heavily mutated second mates), unpaired (mates from different loci, too-far fragments),
    every output array; plus a capacity-limited run"""
    from tests.pipeline_oracle import seed_extend_paired_oracle
    require_gpu()
    O = orc.Oracle()
    n = 300_000
    gw = synth.random_genome_words(n, seed=78)
    gsym = unpack_symbols(host_u32(gw), n)
    idx = O.build_index(gsym)
    fmi = nb.FMIndexDevice.from_host(idx.bwt_occ, idx.ssa, idx.L2, idx.n, idx.primary)
    n_pairs, L = 500, 100
    rw, left, frag = synth.sample_pairs(gw, n, n_pairs, L, frag_mean=300, frag_sd=40, sub_rate=0.02, hard_frac=0.3, hard_sub_rate=0.2, seed=11, mut_seed=12)
    rw = rw.clone()
    # discordant cases: second mates of a few pairs taken from another pair (different locus), a few fragments beyond max_frag
    rw[n_pairs + 5:n_pairs + 25] = rw[n_pairs + 105:n_pairs + 125].clone()
    wpr = rw.shape[1]
    reads_sym = [unpack_symbols(host_u32(rw[i]), L) for i in range(2 * n_pairs)]
    rs = PackedStringSet.fixed(rw.reshape(-1), 2 * n_pairs, L, stride=wpr * 16)
    params = nb.SeedExtendParams(seed_len=20, seed_interval=10, band_len=31, type=aln.LOCAL, both_strands=True,
                                 max_seed_hits=50, scheme=aln.SimpleGotohScheme(2, -2, -5, -3))
    for pair in (nb.PairParams(min_frag=0, max_frag=420, min_mate_score=50), nb.PairParams(min_frag=250, max_frag=330, min_mate_score=80),
                 nb.PairParams(min_frag=0, max_frag=420, min_mate_score=50, rescue_capacity=37)):
        ws = nb.seed_extend_paired(fmi, gw, rs, params, pair, hit_capacity=64 * 2 * n_pairs)
        torch.cuda.synchronize()
        want = seed_extend_paired_oracle(O, idx, gsym, reads_sym, params, pair, n_pairs)
        assert tuple(int(v) for v in ws.n_rescue.cpu()) == want["n_rescue"]
        assert np.array_equal(ws.pair_flags.cpu().numpy().astype(np.int64), want["pair_flags"])
        assert np.array_equal(ws.pair_score.cpu().numpy().astype(np.int64), want["pair_score"])
        assert np.array_equal(ws.mate_score.cpu().numpy().astype(np.int64), want["mate_score"])
        assert np.array_equal(host_u32(ws.mate_pos).astype(np.int64), want["mate_pos"])
        assert np.array_equal(ws.mate_strand.cpu().numpy().astype(np.int64), want["mate_strand"])
        fl = want["pair_flags"]
        if pair.rescue_capacity is None and pair.min_frag == 0:
            assert (fl == 1).sum() > 0.5 * n_pairs and ((fl == 2) | (fl == 4)).sum() > 0.1 * n_pairs and (fl == 0).sum() >= 10


def test_streaming_paired_host_api():
    """nvb_pipeline (host buffers in / out, several batches in flight on different compute streams) in paired-end mode ==
    nvb_seed_extend_paired on the same batches, batch by batch, incl. the slot reuse after `depth` submissions"""
    require_gpu()
    n = 400_000
    gw = synth.random_genome_words(n, seed=91)
    fmi, _ = nb.FMIndexDevice.from_text(gw, n, sa_interval=1)
    fmi.build_ktab(8)
    n_pairs, L = 3000, 150
    params = nb.SeedExtendParams()
    pair = nb.PairParams(min_frag=0, max_frag=500, min_mate_score=80, rescue_capacity=1024)
    batches, want = [], []
    for b in range(5):
        rw, _, _ = synth.sample_pairs(gw, n, n_pairs, L, frag_mean=350.0, frag_sd=30.0, sub_rate=0.01, hard_frac=0.1, hard_sub_rate=0.2,
                                      seed=100 + b, mut_seed=200 + b)
        rw = rw.contiguous()
        rs = PackedStringSet.fixed(rw.reshape(-1), 2 * n_pairs, L, stride=rw.shape[1] * 16)
        ws = nb.seed_extend_paired(fmi, gw, rs, params, pair, hit_capacity=24 * 2 * n_pairs)
        torch.cuda.synchronize()
        want.append({k: getattr(ws, k).cpu().clone() for k in ("pair_score", "pair_flags", "mate_score", "mate_pos", "mate_strand", "n_rescue")})
        batches.append(rw.cpu().pin_memory())
    for depth in (1, 2, 3):
        st = nb.StreamingSeedExtend(fmi, gw, params, 2 * n_pairs, L, batches[0].shape[1], hit_capacity=24 * 2 * n_pairs, depth=depth, pair=pair)
        assert st.h2d_bytes == batches[0].numel() * 4 and st.d2h_bytes >= n_pairs * (4 + 4 + 8 + 8 + 2)
        inflight = []
        for b in range(5):
            inflight.append((b, st.submit(batches[b])))
            if len(inflight) == depth:
                bb, t = inflight.pop(0)
                got = st.result(t)
                for k, v in want[bb].items():
                    assert torch.equal(got[k].reshape(v.shape), v), (depth, bb, k)
        for bb, t in inflight:
            got = st.result(t)
            for k, v in want[bb].items():
                assert torch.equal(got[k].reshape(v.shape), v), (depth, bb, k)
        assert st.last_device_ms > 0
        st.close()


def test_seed_extend_with_base_qualities():
    """nvBowtie's quality-dependent scoring through the composition: per-read qualities (reversed for the rc strings) reach the
    banded extension and the opposite-mate DP; single-end and paired outputs == the oracle composition"""
    from tests.pipeline_oracle import seed_extend_paired_oracle
    require_gpu()
    O = orc.Oracle()
    n = 200_000
    gw = synth.random_genome_words(n, seed=79)
    gsym = unpack_symbols(host_u32(gw), n)
    idx = O.build_index(gsym)
    fmi = nb.FMIndexDevice.from_host(idx.bwt_occ, idx.ssa, idx.L2, idx.n, idx.primary)
    n_pairs, L = 300, 100
    rw, left, frag = synth.sample_pairs(gw, n, n_pairs, L, frag_mean=300, frag_sd=40, sub_rate=0.03, hard_frac=0.3, hard_sub_rate=0.2, seed=21, mut_seed=22)
    wpr = rw.shape[1]
    n_reads = 2 * n_pairs
    reads_sym = [unpack_symbols(host_u32(rw[i]), L) for i in range(n_reads)]
    rng = np.random.default_rng(8)
    qual = rng.integers(0, 50, (n_reads, wpr * 16)).astype(np.uint8)          # laid out like the read stream (stride wpr*16 symbols)
    quals = [qual[i, :L] for i in range(n_reads)]
    rs = PackedStringSet.fixed(rw.reshape(-1), n_reads, L, stride=wpr * 16)
    sch = aln.QualityGotohScheme(match_bonus=2, mm_min=2, mm_max=6, read_gap_const=5, read_gap_coeff=3, ref_gap_const=5, ref_gap_coeff=3)
    params = nb.SeedExtendParams(seed_len=20, seed_interval=10, band_len=31, type=aln.LOCAL, both_strands=True, max_seed_hits=50, scheme=sch,
                                 read_quals=torch.from_numpy(qual.reshape(-1)).cuda())
    ws = nb.seed_extend(fmi, gw, rs, params, hit_capacity=64 * n_reads, keep_hits=True)
    torch.cuda.synchronize()
    want = seed_extend_oracle(O, idx, gsym, reads_sym, params, quals=quals)
    kept = int(ws.n_hits[0])
    assert kept == want["n_hits"]
    assert np.array_equal(ws.hit_score.cpu().numpy()[:kept].astype(np.int64), want["hit_score"])
    assert np.array_equal(host_u32(ws.hit_sink)[:kept].astype(np.int64), want["hit_sink"])
    assert np.array_equal(ws.best_score.cpu().numpy().astype(np.int64), want["best_score"])
    # the qualities matter: the same batch without them scores differently somewhere
    plain = nb.seed_extend(fmi, gw, rs, nb.SeedExtendParams(seed_len=20, seed_interval=10, band_len=31, type=aln.LOCAL, both_strands=True,
                                                           max_seed_hits=50, scheme=sch), hit_capacity=64 * n_reads, keep_hits=True)
    assert not torch.equal(plain.hit_score[:kept], ws.hit_score[:kept])
    pair = nb.PairParams(min_frag=0, max_frag=420, min_mate_score=40)
    wp = nb.seed_extend_paired(fmi, gw, rs, params, pair, hit_capacity=64 * n_reads)
    torch.cuda.synchronize()
    wantp = seed_extend_paired_oracle(O, idx, gsym, reads_sym, params, pair, n_pairs, quals=quals)
    assert tuple(int(v) for v in wp.n_rescue.cpu()) == wantp["n_rescue"] and wantp["n_rescue"][0] > 10
    assert np.array_equal(wp.pair_flags.cpu().numpy().astype(np.int64), wantp["pair_flags"])
    assert np.array_equal(wp.pair_score.cpu().numpy().astype(np.int64), wantp["pair_score"])
    assert np.array_equal(wp.mate_score.cpu().numpy().astype(np.int64), wantp["mate_score"])
    assert np.array_equal(host_u32(wp.mate_pos).astype(np.int64), wantp["mate_pos"])


def test_single_row_fold_and_located_table():
    """full suffix array: the per-read path locates single-row ranges inside the match kernel (SA gather + text compare instead of the
    remaining LF steps), with the 16-byte located k-mer table the SA gather of a single-row k-mer comes with the table entry, and
    with its text context the comparison needs no read of the text either;
    every combination gives the per-hit path's results on a genome with a repeat family (multi-row ranges) and reads with N"""
    import ctypes as C
    require_gpu()
    n = 300_000
    gw = synth.random_genome_words(n, seed=77)
    gsym = unpack_symbols(host_u32(gw), n).copy()
    gsym[100_000:130_000] = np.tile(gsym[2000:2300], 100)
    gw = torch.from_numpy(pack_symbols(gsym, 2, True).view(np.int32)).cuda()
    n_reads, L = 4000, 150
    rw, pos, strand = synth.sample_reads(gw, n, n_reads, L, sub_rate=0.01, indel_rate=0.001, seed=21, mut_seed=22)
    sym = np.stack([unpack_symbols(host_u32(rw[i]), L) for i in range(n_reads)])
    sym[np.random.default_rng(8).random(sym.shape) < 0.002] = 4
    stride = ((L + 7) // 8) * 8
    buf = np.zeros((n_reads, stride), np.uint8); buf[:, :L] = sym
    words = torch.from_numpy(pack_symbols(buf.reshape(-1), 4, True).view(np.int32)).cuda()
    rs = PackedStringSet.fixed(words, n_reads, L, stride=stride, bits=4)
    params = nb.SeedExtendParams(seed_len=20, seed_interval=10, band_len=31, type=aln.LOCAL, both_strands=True, max_seed_hits=40,
                                 scheme=aln.SimpleGotohScheme(2, -2, -5, -3))
    L_ = nb.lib()
    results = {}
    for name, k, located in (("plain", 0, 0), ("ktab", 8, 0), ("located", 8, 1), ("located5", 5, 1), ("context", 8, 2), ("context3", 3, 2)):
        fmi, _ = nb.FMIndexDevice.from_text(gw, n, sa_interval=1)
        if k:
            fmi.build_ktab(k, located=bool(located), text=gw if located == 2 else None)      # context3: 17 symbols left > the 16 of context
        fast = nb.seed_extend(fmi, gw, rs, params, hit_capacity=100 * n_reads)
        torch.cuda.synchronize()
        L_.nvb_debug_pipeline_path(C.c_int(1))
        try:
            slow = nb.seed_extend(fmi, gw, rs, params, hit_capacity=100 * n_reads)
            torch.cuda.synchronize()
        finally:
            L_.nvb_debug_pipeline_path(C.c_int(0))
        assert torch.equal(fast.n_hits[:2], slow.n_hits[:2]), name
        assert torch.equal(fast.best_score, slow.best_score) and torch.equal(fast.best_pos, slow.best_pos), name
        if k:
            # the seed-match stage in one pass instead of two (seeds on repeated k-mers finished by a second kernel): same results
            L_.nvb_debug_seed_split(C.c_int(0))
            try:
                one = nb.seed_extend(fmi, gw, rs, params, hit_capacity=100 * n_reads)
                torch.cuda.synchronize()
            finally:
                L_.nvb_debug_seed_split(C.c_int(1))
            assert torch.equal(fast.n_hits[:2], one.n_hits[:2]) and torch.equal(fast.best_score, one.best_score) and torch.equal(fast.best_pos, one.best_pos), name
        results[name] = (fast.best_score.clone(), fast.best_pos.clone(), fast.n_hits[:2].clone())
    for name in ("ktab", "located", "located5", "context", "context3"):
        assert all(torch.equal(a, b) for a, b in zip(results[name], results["plain"])), name
    assert int((results["plain"][0] > 200).sum()) > n_reads // 2


@pytest.mark.parametrize("sub_rate", [0.0, 0.004, 0.02])
def test_perfect_match_shortcut(sub_rate):
    """a read that equals its window on a band diagonal gets score = match * len and the sink of the LARGEST such diagonal without running
    the DP (pipe_perfect_jobs_kernel): same best score / position per read and the same counts as with every job through the
    DP kernels, and as the per-hit path -- on a genome with a period-7 tandem repeat (several perfect diagonals inside one band), a
    period-300 repeat family, reads at the genome's ends (clamped and truncated windows) and ragged read lengths"""
    import ctypes as C
    require_gpu()
    n = 200_000
    gw = synth.random_genome_words(n, seed=123)
    gsym = unpack_symbols(host_u32(gw), n).copy()
    gsym[50_000:70_000] = np.tile(gsym[1000:1007], 20_000 // 7 + 1)[:20_000]
    gsym[120_000:150_000] = np.tile(gsym[2000:2300], 100)
    gw = torch.from_numpy(pack_symbols(np.concatenate([gsym, np.zeros(128, np.uint8)]), 2, True).view(np.int32)).cuda()
    n_reads, L = 6000, 150
    rw, pos, strand = synth.sample_reads(gw, n, n_reads, L, sub_rate=sub_rate, indel_rate=0.0005 if sub_rate else 0.0, seed=31, mut_seed=32)
    sym = np.stack([unpack_symbols(host_u32(rw[i]), L) for i in range(n_reads)])
    # reads hanging on the genome's two ends
    for i, st in enumerate((0, 3, 9, n - L, n - L - 2, n - L - 20)):
        sym[i] = gsym[st:st + L]
    lens = np.full(n_reads, L, np.uint32); lens[10:400] = np.random.default_rng(4).integers(60, L + 1, 390)
    # reads with one, two or three substitutions at chosen places (the ends, next to the ends, adjacent, spread out): the few-difference
    # branch of the shortcut (maximum-sum segment of the diagonal, last end among equals) incl. its boundary cases; some of them inside
    # the period-7 repeat, where other diagonals are as good and the DP has to decide
    places = [(0,), (1,), (L - 1,), (L - 2,), (0, 1), (L - 2, L - 1), (0, L - 1), (1, L - 2), (2, 3), (74,), (74, 75), (10, 140), (0, 1, 2),
              (L - 3, L - 2, L - 1), (3, 70), (5,), (L - 6,), (2,), (L - 3,), (37, 111)]
    rng_c = np.random.default_rng(17)
    for k, pl in enumerate(places * 3):
        i = 400 + k
        st = int(rng_c.integers(52_000, 68_000)) if k % 3 == 2 else int(rng_c.integers(80_000, 110_000))
        sym[i] = gsym[st:st + L]
        for q in pl:
            sym[i, q] = (sym[i, q] + 1 + (k % 3)) % 4
        lens[i] = L
    stride = ((L + 15) // 16) * 16
    buf = np.zeros((n_reads, stride), np.uint8); buf[:, :L] = sym
    words = torch.from_numpy(pack_symbols(buf.reshape(-1), 2, True).view(np.int32)).cuda()
    rs = PackedStringSet(words=words, bits=2, big_endian=True, offsets=torch.arange(n_reads, dtype=torch.int32, device="cuda") * stride,
                         lengths=torch.from_numpy(lens.view(np.int32)).cuda(), stride=0, length=L, count=n_reads)
    fmi, _ = nb.FMIndexDevice.from_text(gw, n, sa_interval=1)
    fmi.build_ktab(8, located=True, text=gw)
    L_ = nb.lib()
    for scheme in (aln.SimpleGotohScheme(2, -2, -5, -3), aln.SimpleGotohScheme(1, -4, -6, -1)):
        params = nb.SeedExtendParams(seed_len=20, seed_interval=10, band_len=31, type=aln.LOCAL, both_strands=True, max_seed_hits=30, scheme=scheme)
        fast = nb.seed_extend(fmi, gw, rs, params, hit_capacity=200 * n_reads)
        torch.cuda.synchronize()
        L_.nvb_debug_perfect_shortcut(C.c_int(0))
        try:
            full = nb.seed_extend(fmi, gw, rs, params, hit_capacity=200 * n_reads)
            torch.cuda.synchronize()
        finally:
            L_.nvb_debug_perfect_shortcut(C.c_int(1))
        L_.nvb_debug_pipeline_path(C.c_int(1))
        try:
            slow = nb.seed_extend(fmi, gw, rs, params, hit_capacity=200 * n_reads)
            torch.cuda.synchronize()
        finally:
            L_.nvb_debug_pipeline_path(C.c_int(0))
        for other in (full, slow):
            assert torch.equal(fast.best_score, other.best_score) and torch.equal(fast.best_pos, other.best_pos)
            assert torch.equal(fast.n_hits[:2], other.n_hits[:2])
        assert torch.equal(fast.n_hits, full.n_hits)
        if sub_rate == 0.0:
            assert int((fast.best_score == scheme.match * torch.from_numpy(lens.astype(np.int32)).cuda()).sum()) > 0.95 * n_reads


@pytest.mark.parametrize("bits,ragged,cap_div", [(2, False, 0), (4, True, 0), (2, False, 3)])
def test_per_read_path_equals_per_hit_path(bits, ragged, cap_div):
    """the per-read path of nvb_seed_extend (taken when no per-hit output is requested: distinct jobs straight from a thread per
    read, no per-hit arrays) gives the same best score / position per read and the same hit counts as the per-hit path, incl.
    4-bit reads with N, ragged lengths, a repetitive genome (many hits per read) and a hit capacity that truncates"""
    import ctypes as C
    require_gpu()
    n = 150_000
    gw = synth.random_genome_words(n, seed=91)
    gsym = unpack_symbols(host_u32(gw), n).copy()
    gsym[60_000:90_000] = np.tile(gsym[1000:1500], 60)                 # a 500 bp unit repeated 60 times: reads there have many hits
    gw = torch.from_numpy(pack_symbols(gsym, 2, True).view(np.int32)).cuda()
    fmi, _ = nb.FMIndexDevice.from_text(gw, n)
    n_reads, L = 3000, 120
    rw, pos, strand = synth.sample_reads(gw, n, n_reads, L, sub_rate=0.02, indel_rate=0.003, seed=15, mut_seed=16)
    wpr = rw.shape[1]
    sym = np.stack([unpack_symbols(host_u32(rw[i]), L) for i in range(n_reads)])
    if bits == 4:
        rng = np.random.default_rng(5)
        sym[rng.random(sym.shape) < 0.004] = 4
    lens = np.full(n_reads, L, np.uint32)
    if ragged:
        lens = np.random.default_rng(6).integers(L - 60, L + 1, n_reads).astype(np.uint32)
    spw = 32 // bits
    stride = ((L + spw - 1) // spw) * spw
    buf = np.zeros((n_reads, stride), np.uint8); buf[:, :L] = sym
    words = torch.from_numpy(pack_symbols(buf.reshape(-1), bits, True).view(np.int32)).cuda()
    rs = PackedStringSet(words=words, bits=bits, big_endian=True, offsets=(torch.arange(n_reads, device="cuda", dtype=torch.int32) * stride),
                         lengths=dev_u32(lens), stride=0, length=L, count=n_reads)
    params = nb.SeedExtendParams(seed_len=20, seed_interval=10, band_len=31, type=aln.LOCAL, both_strands=True, max_seed_hits=40,
                                 scheme=aln.SimpleGotohScheme(2, -2, -5, -3))
    probe = nb.seed_extend(fmi, gw, rs, params, hit_capacity=400 * n_reads)
    total = int(probe.n_hits[1])
    assert total > 20 * n_reads                                         # the repeat region really produces many hits
    cap = 400 * n_reads if not cap_div else total // cap_div
    L_ = nb.lib()
    fast = nb.seed_extend(fmi, gw, rs, params, hit_capacity=cap)
    torch.cuda.synchronize()
    L_.nvb_debug_pipeline_path(C.c_int(1))
    try:
        slow = nb.seed_extend(fmi, gw, rs, params, hit_capacity=cap)
        torch.cuda.synchronize()
    finally:
        L_.nvb_debug_pipeline_path(C.c_int(0))
    assert torch.equal(fast.n_hits[:2], slow.n_hits[:2])
    assert torch.equal(fast.best_score, slow.best_score) and torch.equal(fast.best_pos, slow.best_pos)
    # ground truth without any de-duplication logic: every hit scored on its own (chains of identical jobs longer than the
    # per-hit path's look-back occur in the repeat region and must resolve to the job that was really scored)
    params.dedup_jobs = False
    truth = nb.seed_extend(fmi, gw, rs, params, hit_capacity=cap, keep_hits=True)
    params.dedup_jobs = True
    L_.nvb_debug_pipeline_path(C.c_int(1))
    try:
        slow_hits = nb.seed_extend(fmi, gw, rs, params, hit_capacity=cap, keep_hits=True)
        torch.cuda.synchronize()
    finally:
        L_.nvb_debug_pipeline_path(C.c_int(0))
    k = int(truth.n_hits[0])
    assert torch.equal(truth.hit_score[:k], slow_hits.hit_score[:k]) and torch.equal(truth.hit_sink[:k], slow_hits.hit_sink[:k])
    assert torch.equal(truth.best_score, fast.best_score) and torch.equal(truth.best_pos, fast.best_pos)
    assert int(fast.n_hits[2]) <= int(slow.n_hits[0]) and int(fast.n_hits[2]) > 0
    if cap_div:
        assert int(fast.n_hits[0]) == cap < total
