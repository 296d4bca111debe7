#!/usr/bin/env python
"""bench.py -- the driver's benchmark contract for nvbio_b200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--genome-mbp 3000] [--reads 1000000] [--workload seed_extend|fm_match|banded_gotoh] [--dump-outputs DIR]

Default workload = BASELINE.json configs[2] "nvBowtie seed-and-extend: 1M x 150bp single-end, 20bp seeds,
band=31, synthetic 3Gbp index" -- the configuration the headline metric (Mreads/s, 150 bp, seed+extend) is
quoted on; it fits one B200.  One step = one pass of the seed+extend hot path (seeds -> FM-index match ->
locate -> windows -> banded Gotoh LOCAL -> best per read) over one batch of synthetic reads.
value      : whole-job Mreads/s with the reads already resident in HBM (device events, max over ranks)
e2e        : the same through the public API with HOST buffers (pinned H2D of the packed reads + D2H of the
             per-read results inside the timed region)
roofline   : the FM-index seed-match kernel (HBM-bound random 32-byte gathers), algorithmic bytes / live
             CUDA-event kernel time vs MEASURED_PEAKS.json
cpu_baseline: the reference's own templates (oracle/_ref, OpenMP, all host cores) on a bounded read sample
--impl reference : the reference CPU path alone, same metric/config (rank 0 only)
Multi-GPU: one process per GPU (torchrun), rank 0 builds the index and NCCL-broadcasts it once; reads are
sharded (weak scaling: every rank processes its own --reads batch); no collective in the steady state.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SCHEME = (2, -2, -5, -3)      # SimpleGotohScheme(2,-2,-5,-3), LOCAL (fmmap.cu:358 precedent; SURVEY 8d C3/C4)
SEED_LEN, SEED_INTERVAL, BAND, READ_LEN = 20, 10, 31, 150


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps of the headline seed+extend measurement and of its host-to-host (e2e) leg; the secondary measurements "
                         "keep their own sizes (paired end: the --c5-total-pairs job; reference-format fm_match and other_configs: best of 5; CPU baseline: one step)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="seed_extend", choices=["seed_extend", "fm_match", "banded_gotoh"])
    ap.add_argument("--genome-mbp", type=float, default=3000.0)
    ap.add_argument("--reads", type=int, default=1_000_000, help="reads per GPU per step")
    ap.add_argument("--cpu-sample", type=int, default=20000, help="reads in the bounded CPU-baseline sample")
    ap.add_argument("--sa-interval", type=int, default=1, help="sampled-SA interval of the device index (16 = reference format, 1 = full SA)")
    ap.add_argument("--ktab-k", type=int, default=16, help="k of the k-mer range table (0 = none)")
    ap.add_argument("--ktab-located", type=int, default=2, help="0: 8-byte table entries {x, y}; 1: 16-byte entries {x, y, SA[x], SA[y]} (needs --sa-interval 1; 69 GB at k = 16); "
                    "2: the same, one-row entries also hold the 16 text symbols before SA[x] (nvb_fm_build_ktab_context)")
    ap.add_argument("--depth", type=int, default=3, help="batches in flight in the host-to-host (e2e) pipeline")
    ap.add_argument("--e2e-sweep", action="store_true", help="also time the host-to-host pipeline with other (depth, compute streams) shapes")
    ap.add_argument("--no-dedup", action="store_true", help="score every hit separately (no job de-duplication)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the C2 / C4 kernel-level measurements")
    ap.add_argument("--pairs", type=int, default=500_000, help="read pairs per GPU per step of the paired-end (C5-shaped) measurement; 0 = skip")
    ap.add_argument("--c5-total-pairs", type=int, default=100_000_000,
                    help="total pairs of the paired-end job (BASELINE configs[4]: 100M), processed as ceil(total / (gpus x pairs)) steps per GPU")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (rank 0) as DIR/<name>.npy: per-read best score and position, and the hit "
                         "counts; the inputs are the same from run to run, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of this project's timed path: not with --impl reference")
    return args


DUMP_MAX_READS = 2_000_000      # 3 float64 arrays of at most 2M entries: 48 MB


def dump_outputs(out_dir, ws):
    """the per-read results of the timed seed+extend step (float64: exact for int32 scores and uint32 positions); above DUMP_MAX_READS reads
    a fixed, seeded sample of them, identified by read_index"""
    n = ws.best_score.numel()
    sel = np.arange(n) if n <= DUMP_MAX_READS else np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_READS, replace=False))
    out = {"read_index": sel,
           "best_score": ws.best_score.cpu().numpy()[sel],
           "best_pos": ws.best_pos.cpu().numpy().view(np.uint32)[sel],
           "n_hits": ws.n_hits.cpu().numpy()}          # kept, found, distinct alignment jobs
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_traffic(kernel, field="dram_bytes_per_launch", **cfg):
    """a per-launch counter of `kernel` (default: DRAM bytes) from the committed `ncu --set full` captures (profiles/traffic.json),
    when one exists for exactly this configuration; else None"""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        for e in json.load(open(p)):
            if e["kernel"] == kernel and all(e.get(k) == v for k, v in cfg.items()):
                return e.get(field)
    except Exception:
        pass
    return None


def gather_rate(ms, **cfg):
    """second denominator for the seed-match kernel: its L2 read requests per launch (ncu capture of exactly this configuration)
    over the live launch time, against the measured rate of dependent random 16-byte gathers on this part"""
    req = measured_traffic("pipe_seed_match_kernel", "l2_read_requests_per_launch", **cfg)
    ceil = measured_traffic("pipe_seed_match_kernel", "gather_ceiling_G_per_s", **cfg)
    if not req or not ceil:
        return None
    ach = req / (ms * 1e-3) / 1e9
    return {"l2_read_requests_per_launch": req, "achieved_G_per_s": ach, "ceiling_G_per_s": ceil, "frac": ach / ceil,
            "source": measured_traffic("pipe_seed_match_kernel", "gather_ceiling_source", **cfg)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------
def setup_dist(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(0)
        local = 0
    return rank, local, world


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def build_index(args, rank, world, device):
    """rank 0 builds (genome, FM-index) on its GPU; the others receive replicas over NCCL"""
    import nvbio_b200 as nb
    from nvbio_b200 import synth, dist as nd
    n = int(args.genome_mbp * 1e6)
    t_build = t_bcast = 0.0
    fmi = genome = None
    if rank == 0:
        torch.cuda.synchronize(); t0 = time.perf_counter()
        genome = synth.random_genome_words(n, device=device)
        fmi, _ = nb.FMIndexDevice.from_text(genome, n, sa_interval=args.sa_interval)
        torch.cuda.synchronize(); t_build = time.perf_counter() - t0
        torch.cuda.empty_cache()
    if world > 1:
        barrier(world); t0 = time.perf_counter()
        fmi, genome = nd.broadcast_index(fmi, genome, device, src=0)
        barrier(world); t_bcast = time.perf_counter() - t0
    if args.ktab_k > 0 and args.impl == "ours":
        torch.cuda.synchronize(); t0 = time.perf_counter()
        fmi.build_ktab(args.ktab_k, located=bool(args.ktab_located) and args.sa_interval == 1,    # every rank derives the table from its replica
                       text=genome if args.ktab_located == 2 else None)
        torch.cuda.synchronize(); t_build += time.perf_counter() - t0
    return n, genome, fmi, t_build, t_bcast


def make_reads(genome, n, n_reads, rank, device):
    from nvbio_b200 import synth
    rw, pos, strand = synth.sample_reads(genome, n, n_reads, READ_LEN, sub_rate=0.01, indel_rate=0.001, device=device,
                                         seed=synth.SEED_QUERIES + 7919 * rank, mut_seed=synth.SEED_MUT + 104729 * rank)
    return rw.contiguous()


# ------------------------------------------------------------------------------------------------
def host_reference_index(fmi, with_ssa=True):
    """the device index as host arrays in the REFERENCE'S format (SA sampled every 16 rows, no table), for the CPU checkers"""
    from oracle import orc
    ssa16 = None
    if with_ssa:
        step = 16 // fmi.sa_interval
        ssa16 = np.ascontiguousarray(fmi.ssa[::step].contiguous().cpu().numpy().view(np.uint32))   # slice on the device: a full SA is 12 GB
    return orc._Index(n=fmi.length, primary=fmi.primary, bwt_occ=fmi.bwt_occ.cpu().numpy().view(np.uint32), ssa=ssa16,
                      L2=np.array(fmi.L2, dtype=np.uint32))


def cpu_reference_leg(args, n, genome, fmi, steps, warmup, want_blocks=True, parity_with=None):
    """the reference's CPU path (oracle/_ref if present, else the C port) on a bounded sample per step.
    parity_with = (nb, params): afterwards (untimed) the last sample's reads also go through nvb_seed_extend over THIS run's device
    index and every per-hit score, the hit count and the best score per read are compared with the reference's"""
    from oracle import orc
    from oracle.cpu_pipeline import cpu_seed_extend
    from nvbio_b200 import synth
    E = orc.Ref() if orc.Ref.available() else orc.Oracle()
    thread_options = [1]
    if E.kind == "reference":
        # all the host threads the box offers (torchrun exports OMP_NUM_THREADS=1 to its workers: override it).  The
        # path is latency bound, so SMT siblings can hurt: the warm-up tries both "every hardware thread" and "half of
        # them" and the timed steps use whichever was faster for the reference.
        try:
            n_thr = len(os.sched_getaffinity(0))
        except AttributeError:
            n_thr = os.cpu_count() or 1
        thread_options = [n_thr] + ([n_thr // 2] if n_thr >= 4 else [])
        E.set_num_threads(thread_options[0])
    cores = thread_options[0] if E.kind == "reference" else 1
    idx = host_reference_index(fmi)
    gw = genome.cpu().numpy().view(np.uint32)
    nsample = args.cpu_sample
    times, res = [], None
    O = orc.Oracle() if want_blocks else None
    trial = {}
    for it in range(max(warmup, len(thread_options)) + steps):
        if E.kind == "reference":
            if it < len(thread_options):
                E.set_num_threads(thread_options[it])
            elif it == len(thread_options) and len(trial) > 1:
                cores = min(trial, key=trial.get)
                E.set_num_threads(cores)
        rw = make_reads(genome, n, nsample, 1000 + it, genome.device)
        words = rw.cpu().numpy().view(np.uint32)
        sym = _unpack_rows(words, READ_LEN)
        res = cpu_seed_extend(E, idx, gw, sym, SEED_LEN, SEED_INTERVAL, BAND, 1, SCHEME, True, 100,
                              count_blocks_with=(O if (want_blocks and it == 0) else None), blocks_from_step=args.ktab_k)
        if it == 0 and want_blocks:
            blocks_per_seed = res["blocks"] / res["n_seeds"]
            tail_blocks_per_seed = (res["blocks_tail"] / res["n_seeds"]) if res["blocks_tail"] is not None else blocks_per_seed
        if E.kind == "reference" and it < len(thread_options):
            trial[thread_options[it]] = res["t_total"]
        if it >= max(warmup, len(thread_options)):
            times.append(res["t_total"])
    t = float(np.mean(times)) if times else float("nan")
    out = dict(kind=E.kind, cores=cores, sample="%d reads x %d bp per step (%d seeds, %d extensions), C calls only" %
               (nsample, READ_LEN, res["n_seeds"], res["n_hits"]), value=nsample / t / 1e6, unit="Mreads/s",
               ms_per_step=t * 1e3, t_match_ms=res["t_match"] * 1e3, t_locate_ms=res["t_locate"] * 1e3, t_dp_ms=res["t_dp"] * 1e3,
               gcups=res["cells"] / res["t_dp"] / 1e9 if res["t_dp"] > 0 else None,
               mseeds_per_s=res["n_seeds"] / res["t_match"] / 1e6 if res["t_match"] > 0 else None)
    if want_blocks:
        out["blocks_per_seed"] = blocks_per_seed
        out["tail_blocks_per_seed"] = tail_blocks_per_seed
    if parity_with is not None:
        nb, params = parity_with
        from nvbio_b200.strings import PackedStringSet
        rs = PackedStringSet.fixed(rw.reshape(-1), nsample, READ_LEN, stride=rw.shape[1] * 16)
        a = nb.seed_extend(fmi, genome, rs, params, hit_capacity=24 * nsample)                    # the path the benchmark times
        b = nb.seed_extend(fmi, genome, rs, params, hit_capacity=24 * nsample, keep_hits=True)    # per-hit outputs
        torch.cuda.synchronize()
        kept, total, jobs = [int(v) for v in a.n_hits.cpu()]
        best_ok = bool(np.array_equal(a.best_score.cpu().numpy().astype(np.int64), res["best_score"]) and
                       np.array_equal(b.best_score.cpu().numpy().astype(np.int64), res["best_score"]))
        hits_ok = bool(kept == total == res["n_hits"] and np.array_equal(b.hit_score[:total].cpu().numpy(), res["hit_score"]))
        out["parity"] = {"ok": bool(best_ok and hits_ok), "reads": nsample, "hits": res["n_hits"], "best_score_per_read_identical": best_ok,
                         "per_hit_scores_and_hit_count_identical": hits_ok,
                         "against": "%s (nvbio::match -> locate -> aln::banded_alignment_score<31> -> max per read) over the same %d bp index in the "
                                    "reference's format; device index: sa_interval=%d, ktab_k=%d" % (E.kind, n, fmi.sa_interval, fmi.ktab_k)}
    return out


def _unpack_rows(words, L):
    i = np.arange(L)
    sh = (30 - 2 * (i & 15)).astype(np.uint32)
    return ((words[:, i >> 4] >> sh) & 3).astype(np.uint8)


# ------------------------------------------------------------------------------------------------
def run_reference(args):
    # under torchrun only rank 0 works; the other ranks exit 0 at once (no process group is needed)
    if int(os.environ.get("RANK", "0")) != 0:
        return
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    # the index is built on the device as untimed set-up (a 3 Gbp suffix sort on the host takes ~1 h); the
    # timed path is the reference's CPU code only
    n, genome, fmi, t_build, _ = build_index(args, 0, 1, device)
    r = cpu_reference_leg(args, n, genome, fmi, args.steps, args.warmup, want_blocks=False)
    line = {
        "impl": "reference", "metric": "Mreads/s (150bp) seed+extend", "value": r["value"], "unit": "Mreads/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": workload_config(args, n, args.reads, world=args.gpus),
        "index": index_description(16, 0, n),
        "cpu_baseline": {"value": r["value"], "unit": "Mreads/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"],
                         "fm_match_Mseeds_s": r["mseeds_per_s"], "banded_gotoh_GCUPS": r["gcups"]},
        "e2e": {"value": r["value"], "unit": "Mreads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "index_build": "device suffix sort (set-up, untimed): %.1f s" % t_build,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, n, reads_per_gpu, world, index=None):
    """`workload` names the job (the same for both arms); `index` says how THIS arm holds the FM-index"""
    cfg = {"workload": "nvBowtie seed-and-extend: %d x %dbp single-end reads per GPU, %dbp seeds every %dbp on both strands, "
                       "band=%d Gotoh LOCAL (2,-2,-5,-3), synthetic %.0f Mbp 2-bit genome, FM-index = 32-byte {bwt,occ} blocks (occ every 64)"
                       % (reads_per_gpu, READ_LEN, SEED_LEN, SEED_INTERVAL, BAND, n / 1e6),
           "reads_per_gpu_per_step": reads_per_gpu, "genome_bp": n, "parallelism": "dp%d (index replicated by one NCCL broadcast)" % world,
           "l2": "index (%.2f GB of blocks alone) exceeds L2; a 512 MiB buffer is overwritten between timed steps" % (n / 64 * 32 / 1e9)}
    if index is not None:
        cfg["index"] = index
    return cfg


def index_description(sa_interval, ktab_k, n, nbytes=None, located=False):
    eb = 16 if located else 8
    d = {"sa_interval": sa_interval, "ktab_k": ktab_k, "ktab_located": int(located) if ktab_k else 0,
         "layout": "%s + %s" % ("full suffix array (4 B per base)" if sa_interval == 1 else "SA sampled every %d rows" % sa_interval,
                                ("%d-mer SA-range table (4^%d x %d B = %.1f GB%s)" % (ktab_k, ktab_k, eb, 4 ** ktab_k * eb / 1e9,
                                                                                     ("; entries {x, y, SA[x], SA[y]}" + (", one-row entries {x, x, SA[x], 16 text symbols before SA[x]}" if int(located) == 2 else "")) if located else "")) if ktab_k else "no k-mer table (the reference's format)")}
    if nbytes is not None:
        d["bytes_per_gpu"] = int(nbytes)
    return d


def c1_config(device, best_ms):
    """BASELINE configs[0]: 10K x 100 bp reads, each against its own 1 Kbp reference, SimpleGotohScheme(2,-1,-2,-1) as sw-benchmark
    sets it (sw-benchmark.cu:592-641): (i) what sw-benchmark runs -- the full-matrix DP, every type; (ii) the band-15 GLOBAL variant
    the config name mentions (100 bp vs the 114 bp window of the read).  The reference's own host path (aln::alignment_score /
    banded_alignment_score over OpenMP) is timed beside it on the same inputs and its results compared."""
    import nvbio_b200 as nb
    from nvbio_b200 import aln
    from nvbio_b200.strings import PackedStringSet, pack_symbols
    from oracle import orc
    rng = np.random.default_rng(77)
    n_al, M, N = 10_000, 100, 1000
    txt = rng.integers(0, 4, (n_al, N)).astype(np.uint8)
    st = rng.integers(0, N - M - 14, n_al)
    pat = np.stack([txt[i, st[i]:st[i] + M] for i in range(n_al)])
    pat = np.where(rng.random(pat.shape) < 0.02, rng.integers(0, 4, pat.shape), pat).astype(np.uint8)
    p_off = np.arange(n_al, dtype=np.uint32) * M; p_len = np.full(n_al, M, np.uint32)
    t_off = np.arange(n_al, dtype=np.uint32) * N; t_len = np.full(n_al, N, np.uint32)
    P = PackedStringSet.from_symbols(pat.reshape(-1), p_off, p_len, bits=2, big_endian=True)
    T = PackedStringSet.from_symbols(txt.reshape(-1), t_off, t_len, bits=2, big_endian=True)
    w_off = (t_off + st).astype(np.uint32); w_len = np.full(n_al, M + 14, np.uint32)
    Tw = PackedStringSet.from_symbols(txt.reshape(-1), w_off, w_len, bits=2, big_endian=True)
    scheme = (2, -1, -2, -1)
    R = orc.Ref() if orc.Ref.available() else None
    if R is not None:
        R.set_num_threads(len(os.sched_getaffinity(0)))
    res = {"scheme": "SimpleGotohScheme(2,-1,-2,-1)", "cells_full": n_al * M * N, "cells_band15": n_al * M * 15}
    for typ, name in ((0, "global"), (1, "local"), (2, "semi_global")):
        al = aln.make_gotoh_aligner(typ, aln.SimpleGotohScheme(*scheme))
        out = [None]

        def go():
            out[0] = aln.batch_alignment_score(al, P, T)
        ms = best_ms(go, reps=3)
        e = {"GCUPS": n_al * M * N / (ms * 1e-3) / 1e9, "ms": ms}
        if R is not None:
            t0 = time.perf_counter()
            ws, wx, wy = R.gotoh_full(typ, scheme, pat.reshape(-1), p_off, p_len, txt.reshape(-1), t_off, t_len)
            cpu_s = time.perf_counter() - t0
            k = out[0][1].cpu().numpy().view(np.uint32)
            e["reference_cpu_GCUPS"] = n_al * M * N / cpu_s / 1e9
            e["bit_identical_to_reference"] = bool(np.array_equal(out[0][0].cpu().numpy(), ws) and np.array_equal(k[:, 0], wx) and np.array_equal(k[:, 1], wy))
        res["full_matrix_" + name] = e
    al = aln.make_gotoh_aligner(aln.GLOBAL, aln.SimpleGotohScheme(*scheme))
    out = [None]

    def go_b():
        out[0] = aln.batch_banded_alignment_score(15, al, P, Tw)
    ms = best_ms(go_b, reps=3)
    e = {"GCUPS": n_al * M * 15 / (ms * 1e-3) / 1e9, "ms": ms}
    if R is not None:
        t0 = time.perf_counter()
        ws, wx, wy, _ = R.banded_gotoh(15, 0, scheme, pat.reshape(-1), p_off, p_len, txt.reshape(-1), w_off, w_len)
        cpu_s = time.perf_counter() - t0
        k = out[0][1].cpu().numpy().view(np.uint32)
        e["reference_cpu_GCUPS"] = n_al * M * 15 / cpu_s / 1e9
        e["bit_identical_to_reference"] = bool(np.array_equal(out[0][0].cpu().numpy(), ws) and np.array_equal(k[:, 0], wx) and np.array_equal(k[:, 1], wy))
        res["reference_cpu_cores"] = R.num_threads() if hasattr(R, "num_threads") else len(os.sched_getaffinity(0))
    res["banded_15_global"] = e
    res["note"] = "10K alignments = 5K two-per-thread DP threads: launch/occupancy-bound on 148 SMs, not a throughput figure (see C4 and the full-matrix sweep in profiles/)"
    return res


def other_configs(device):
    """BASELINE.json configs[1] (FM-index exact match, 1M x 22 bp seeds, 100 Mbp) and configs[3] (banded Gotoh LOCAL,
    10M x 151 bp vs 300 bp windows, (2,2,5,3), band sweep) -- the two kernel-level metrics of the headline string,
    measured in the same run, each through the public API (device events, best of 5 after a warm-up)."""
    import nvbio_b200 as nb
    from nvbio_b200 import aln, synth
    from nvbio_b200.strings import PackedStringSet
    from oracle import orc

    def best_ms(fn, reps=5):
        fn(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        best = 1e30
        for _ in range(reps):
            e0.record(); fn(); e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return best
    out = {}
    peak, _ = measured_peaks()
    # ---- C1: sw-benchmark's case (BASELINE configs[0]) ----
    try:
        out["sw_benchmark_10Kx100bp_vs_1Kbp"] = c1_config(device, best_ms)
    except Exception as e:
        out["sw_benchmark_10Kx100bp_vs_1Kbp"] = {"error": repr(e)[:300]}
    # ---- C2 ----
    n = 100_000_000
    gw = synth.random_genome_words(n, device=device)
    fmi, _ = nb.FMIndexDevice.from_text(gw, n)                       # reference format: SA_INT 16, no k-mer table
    nq, L = 1_000_000, 22
    sw, _ = synth.sample_seeds(gw, n, nq, L, device=device)
    q = PackedStringSet.fixed(sw.reshape(-1), nq, L, stride=32)
    ranges = torch.empty((nq, 2), dtype=torch.int32, device=device)
    ms_plain = best_ms(lambda: nb.match(fmi, q, out=ranges))
    # exact block count of the reference algorithm on a 50K-seed sample (oracle)
    O = orc.Oracle()
    host = fmi.to_host()
    idx = orc._Index(n=n, primary=host["primary"], bwt_occ=host["bwt_occ"], ssa=host["ssa"], L2=host["L2"])
    samp = _unpack_rows(sw[:50000].cpu().numpy().view(np.uint32), L)
    want, blocks = O.match(idx, samp.reshape(-1), np.arange(50000) * L, np.full(50000, L))
    parity = bool(np.array_equal(ranges[:50000].cpu().numpy().view(np.uint32), want))
    bps = 32.0 * blocks / 50000 + L * 2 / 8.0 + 8.0
    fmi.build_ktab(10)
    ms_ktab = best_ms(lambda: nb.match(fmi, q, out=ranges))
    out["fm_index_exact_match_1Mx22bp_100Mbp"] = {
        "Mseeds_per_s": nq / (ms_plain * 1e-3) / 1e6, "ms": ms_plain, "algorithmic_bytes_per_seed": bps,
        "algorithmic_GBs": nq * bps / (ms_plain * 1e-3) / 1e9, "frac_of_measured_hbm_peak": nq * bps / (ms_plain * 1e-3) / 1e9 / peak,
        "note": "reference-format index (no k-mer table); the 50 MB index is L2-resident on B200, so this is L2, not HBM, traffic",
        "with_10mer_table_Mseeds_per_s": nq / (ms_ktab * 1e-3) / 1e6, "ranges_bit_identical_to_oracle_on_50k_sample": parity}
    # ---- C4 ----
    n_al, M, W = 10_000_000, 151, 300
    rw, pos, _ = synth.sample_reads(gw, n, n_al, M, device=device, rc_half=False)
    begin = synth.windows_for_reads(n, pos, M, W, device=device)
    P = PackedStringSet.fixed(rw.reshape(-1), n_al, M, stride=rw.shape[1] * 16)
    T = PackedStringSet(words=gw, bits=2, big_endian=True, offsets=begin.to(torch.int32), lengths=None, stride=0, length=W, count=n_al)
    al = aln.make_gotoh_aligner(aln.LOCAL, aln.SimpleGotohScheme(*SCHEME))
    res = (torch.empty(n_al, dtype=torch.int32, device=device), torch.empty((n_al, 2), dtype=torch.int32, device=device))
    sweep = {}
    for band in (7, 15, 31):
        temp = torch.empty(aln.banded_temp_bytes(band, al, P, T) + 256, dtype=torch.uint8, device=device)
        ms = best_ms(lambda: aln.batch_banded_alignment_score(band, al, P, T, out=res, temp=temp), reps=3)
        sweep["band_%d" % band] = {"GCUPS": n_al * M * band / (ms * 1e-3) / 1e9, "ms": ms}
    out["banded_gotoh_local_10Mx151bp_300bp_windows"] = dict(sweep, scheme="SimpleGotohScheme(2,-2,-5,-3)",
                                                             note="cells = n x 151 x BAND_LEN; integer-issue bound")
    # ---- the reference's own CUDA kernels recompiled for sm_100a, same inputs, same run (BASELINE.md section 3) ----
    del P, T, res, rw, pos, begin
    torch.cuda.empty_cache()
    try:
        import importlib.util
        spec = importlib.util.spec_from_file_location("compare_ref_cuda", os.path.join(ROOT, "tools", "compare_ref_cuda.py"))
        crc = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(crc)
        if os.path.exists(crc.BIN):
            fmi2, _ = nb.FMIndexDevice.from_text(gw, n)
            out["vs_reference_cuda_sm100a"] = {
                "banded_gotoh_1Mx150bp_band31": crc.banded_compare(gw, n, 1_000_000, 150),
                "fm_index_filter_rank_locate_1Mx22bp": crc.fm_compare(fmi2, gw, n, 1_000_000, 22),
                "note": "oracle/_ref/ref_cuda_bench = nvbio's batched_banded_alignment_score_kernel / FMIndexFilterDevice compiled from the "
                        "reference's headers for sm_100a; speedup = reference ms / nvbio_b200 ms on identical inputs, results bit-compared"}
        else:
            out["vs_reference_cuda_sm100a"] = {"unavailable": "oracle/_ref/ref_cuda_bench not built"}
    except Exception as e:
        out["vs_reference_cuda_sm100a"] = {"error": repr(e)[:300]}
    return out


def paired_end_config(args, nb, fmi, genome, n, params, device, world, nd):
    """BASELINE configs[4] shape at per-GPU scale: `--pairs` FR pairs of 2 x 150 bp per GPU per step through
    nvb_seed_extend_paired (both mates seeded + extended, concordance check, opposite-mate full-matrix Gotoh rescue).
    Device-resident timing, L2 flushed between steps, max over ranks."""
    from nvbio_b200.pipeline import PairedWorkspace
    from nvbio_b200.strings import PackedStringSet
    from nvbio_b200 import synth
    n_pairs = args.pairs
    rank = int(os.environ.get("RANK", "0"))
    words, left, frag = synth.sample_pairs(genome, n, n_pairs, READ_LEN, frag_mean=350.0, frag_sd=30.0, sub_rate=0.01, hard_frac=0.05,
                                           hard_sub_rate=0.2, device=device, seed=0x51ED + rank, mut_seed=0xC0FFEE + rank)
    wpr = words.shape[1]
    rs = PackedStringSet.fixed(words.reshape(-1), 2 * n_pairs, READ_LEN, stride=wpr * 16)
    pair = nb.PairParams(min_frag=0, max_frag=500, min_mate_score=80, rescue_capacity=max(n_pairs // 4, 1024))
    ws = PairedWorkspace(fmi, genome, rs, params, pair, 24 * 2 * n_pairs)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=device)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # a second batch so that consecutive steps do not see the same reads
    words2, _, _ = synth.sample_pairs(genome, n, n_pairs, READ_LEN, frag_mean=350.0, frag_sd=30.0, sub_rate=0.01, hard_frac=0.05,
                                      hard_sub_rate=0.2, device=device, seed=0x61ED + rank, mut_seed=0xD0FFEE + rank)
    rs2 = PackedStringSet.fixed(words2.reshape(-1), 2 * n_pairs, READ_LEN, stride=wpr * 16)
    for _ in range(2):
        flush.zero_(); nb.seed_extend_paired(fmi, genome, rs2, params, pair, workspace=ws)
    barrier(world)
    # the whole configs[4] job: total pairs / (gpus x pairs per step) steps on every GPU, every step timed on the device
    k = max(1, -(-args.c5_total_pairs // (world * n_pairs)))
    total = 0.0
    for i in range(k):
        flush.zero_()
        ev0.record(); nb.seed_extend_paired(fmi, genome, rs2 if (i & 1) else rs, params, pair, workspace=ws); ev1.record()
        torch.cuda.synchronize()
        total += ev0.elapsed_time(ev1)
    if k & 1 == 0:                                        # leave batch 0's results in the workspace for the checks below
        nb.seed_extend_paired(fmi, genome, rs, params, pair, workspace=ws); torch.cuda.synchronize()
    barrier(world)
    total = nd.max_over_ranks(total, device)
    ms = total / k
    flags = ws.pair_flags.cpu().numpy()
    run, wanted = [int(v) for v in ws.n_rescue.cpu()]
    kept, hits, _ = [int(v) for v in ws.n_hits.cpu()]
    # placement check against the generator's truth: the forward mate must end at left + 150, the reverse one at left + frag
    pos = ws.mate_pos.cpu().numpy().view(np.uint32).astype(np.int64)
    strand = ws.mate_strand.cpu().numpy()
    l, f = left.cpu().numpy(), frag.cpu().numpy()
    truth = np.where(strand == 0, l[None, :] + READ_LEN, (l + f)[None, :])
    placed = np.abs(pos - truth) <= 8
    paired = flags != 0
    # ---- the same job host to host: packed pairs from pinned host memory in, per-pair results in host memory out (C ABI nvb_pipeline) ----
    e2e = None
    try:
        host = [words.cpu().pin_memory(), words2.cpu().pin_memory()]
        st = nb.StreamingSeedExtend(fmi, genome, params, 2 * n_pairs, READ_LEN, wpr, hit_capacity=24 * 2 * n_pairs, depth=args.depth, pair=pair)

        def run_stream(k_steps):
            q, chk = [], 0
            for i in range(k_steps):
                q.append(st.submit(host[i & 1]))
                if len(q) == args.depth:
                    chk += int(st.result(q.pop(0))["pair_flags"][0])
            while q:
                last = st.result(q.pop(0)); chk += int(last["pair_flags"][0])
            return last
        run_stream(max(3, args.depth))
        barrier(world)
        k2 = min(k, 40)
        t0 = time.perf_counter()
        last = run_stream(k2)
        torch.cuda.synchronize()
        e_ms = (time.perf_counter() - t0) * 1e3
        barrier(world)
        e_ms = nd.max_over_ranks(e_ms, device) / k2
        e2e = {"Mreads_per_s": world * 2 * n_pairs / (e_ms * 1e-3) / 1e6, "Mpairs_per_s": world * n_pairs / (e_ms * 1e-3) / 1e6, "ms_per_step": e_ms,
               "steps": k2, "h2d_bytes_per_step": st.h2d_bytes, "d2h_bytes_per_step": st.d2h_bytes, "depth": args.depth,
               "job_seconds_at_this_rate": k * e_ms * 1e-3,
               "api": "C ABI nvb_pipeline (paired mode) via nvbio_b200.StreamingSeedExtend, wall clock over the steps, max over ranks"}
        st.close()
    except Exception as e:
        if world > 1:
            raise
        e2e = {"error": repr(e)[:300]}
    return {"e2e": e2e,"workload": "%d FR pairs (2 x %d bp) per GPU per step, fragments ~N(350,30), 1%% substitutions, 5%% of the second mates with 20%% "
                        "substitutions; both mates seeded+extended (band %d LOCAL), opposite-mate rescue by full-matrix Gotoh LOCAL in the "
                        "500 bp fragment window" % (n_pairs, READ_LEN, BAND),
            "Mreads_per_s": world * 2 * n_pairs / (ms * 1e-3) / 1e6, "Mpairs_per_s": world * n_pairs / (ms * 1e-3) / 1e6, "ms_per_step": ms, "n_gpus": world,
            "job": {"total_pairs": k * world * n_pairs, "steps_per_gpu": k, "device_seconds": total * 1e-3,
                    "note": "BASELINE configs[4] size (100M pairs of 2 x 150 bp) as steps of two alternating synthetic batches per GPU; device time = sum of "
                            "the per-step CUDA-event times, max over ranks (L2 flushed between steps, input generation untimed)"},
            "pairs_concordant_frac": float((flags == 1).mean()), "pairs_rescued_frac": float(((flags == 2) | (flags == 4)).mean()),
            "pairs_unpaired_frac": float((flags == 0).mean()), "rescue_jobs_run": run, "rescue_jobs_wanted": wanted,
            "rescue_cells": run * READ_LEN * 500, "hits_truncated": bool(kept != hits),
            "paired_and_both_mates_at_true_locus_frac": float((paired & placed[0] & placed[1]).mean()),
            "rank0_counts_only": True}


def count_blocks(args, n, genome, fmi):
    """algorithmic 32-byte blocks per seed of the reference algorithm (every LF step: its distinct {bwt,occ} blocks, SURVEY 8d) and of
    the steps left after the k-mer table look-up, counted exactly by the plain-C oracle on a sample of this workload's reads
    (checker use: it counts, it is not timed).  The same count at every world size."""
    from oracle import orc
    nsample = min(args.cpu_sample, 5000)
    O = orc.Oracle()
    rw = make_reads(genome, n, nsample, 999, genome.device)
    sym = _unpack_rows(rw.cpu().numpy().view(np.uint32), READ_LEN)
    idx = host_reference_index(fmi, with_ssa=False)
    strings = np.empty((2 * nsample, READ_LEN), np.uint8)
    strings[0::2] = sym
    strings[1::2] = (3 - sym)[:, ::-1]
    K = (READ_LEN - SEED_LEN) // SEED_INTERVAL + 1
    cols = (np.arange(K) * SEED_INTERVAL)[:, None] + np.arange(SEED_LEN)[None, :]
    q = np.ascontiguousarray(strings[:, cols].reshape(-1))
    nq = 2 * nsample * K
    off = (np.arange(nq, dtype=np.uint32) * SEED_LEN).astype(np.uint32)
    ln = np.full(nq, SEED_LEN, np.uint32)
    _, blocks = O.match(idx, q, off, ln)
    tail = blocks
    if args.ktab_k:
        _, tail = O.match(idx, q, off, ln, blocks_from_step=args.ktab_k)
    return blocks / nq, tail / nq, nq


def reference_format_fm_match(args, nb, fmi, n, genome, device, blocks_per_seed, peak):
    """The kernel the north-star's HBM-roofline target names: backward search over the REFERENCE-FORMAT index (no k-mer table, HBM
    resident: the 3 Gbp index's 1.5 GB of blocks), one launch of nvb_fm_match over this workload's 28 M 20-mers; algorithmic bytes =
    32 B x distinct blocks per LF step (oracle count) + query + 8 B out."""
    from nvbio_b200.strings import PackedStringSet
    plain = nb.FMIndexDevice(fmi.bwt_occ, None, fmi.L2, n, fmi.primary, sa_interval=16)
    n_reads = args.reads
    rw = make_reads(genome, n, n_reads, 4242, device)
    wpr = rw.shape[1]
    K = (READ_LEN - SEED_LEN) // SEED_INTERVAL + 1
    # seed k of read r = symbols [k*10, k*10+20) of the read's slot: an infix set over the packed reads
    r = torch.arange(n_reads, device=device, dtype=torch.int64)[:, None] * (wpr * 16)
    off = (r + torch.arange(K, device=device, dtype=torch.int64)[None, :] * SEED_INTERVAL).reshape(-1).to(torch.int32)
    nq = n_reads * K
    q = PackedStringSet(words=rw.reshape(-1), bits=2, big_endian=True, offsets=off, lengths=None, stride=0, length=SEED_LEN, count=nq)
    ranges = torch.empty((nq, 2), dtype=torch.int32, device=device)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(2):
        nb.match(plain, q, out=ranges)
    best = 1e30
    for _ in range(5):
        flush.zero_()
        e0.record(); nb.match(plain, q, out=ranges); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    bps = 32.0 * blocks_per_seed + SEED_LEN * 2 / 8.0 + 8.0
    gbs = nq * bps / (best * 1e-3) / 1e9
    found = float((ranges[:, 0].to(torch.int64) & 0xFFFFFFFF <= (ranges[:, 1].to(torch.int64) & 0xFFFFFFFF)).float().mean())
    return {"kernel": "fm_match_kernel (nvb_fm_match, reference-format index: no k-mer table)", "seeds": nq, "ms": best,
            "Mseeds_per_s": nq / (best * 1e-3) / 1e6, "algorithmic_bytes_per_seed": bps, "blocks_per_seed": blocks_per_seed,
            "achieved_GBs": gbs, "peak_GBs": peak, "frac": gbs / peak, "index_bytes": int(fmi.bwt_occ.numel() * 4),
            "seeds_found_frac": found,
            "note": "forward-strand 20-mers of %d reads (every one occurs in the genome up to the reads' 1%% substitutions); L2 flushed before every launch" % n_reads}


def e2e_single(args, nb, fmi, genome, params, batches, n_reads, wpr, hit_capacity, world, nd, device, depth):
    """host-to-host through the C ABI's nvb_pipeline (nvbio_b200.StreamingSeedExtend): every step copies ITS packed reads from pinned
    host memory, runs the hot path and copies the per-read (score, position) back; `depth` batches in flight"""
    host_reads = [b.cpu().pin_memory() for b in batches]
    stream = nb.StreamingSeedExtend(fmi, genome, params, n_reads, READ_LEN, wpr, hit_capacity=hit_capacity, depth=depth)
    last = {}

    def run(k_steps):
        q, chk = [], 0
        for i in range(k_steps):
            q.append(stream.submit(host_reads[i % 2]))
            if len(q) == depth:
                sc, _, nh = stream.result(q.pop(0)); chk += int(sc[0]) + int(nh[0])      # the host really reads the results
        while q:
            sc, _, nh = stream.result(q.pop(0)); chk += int(sc[0]) + int(nh[0])
        last["score"] = sc.clone()
        return chk
    # the timed region starts with an empty pipeline and ends when the last result has been read on the host (fill and drain
    # included: about one and a half batches, so a run of few steps understates the steady rate)
    k_steps = args.steps
    run(max(args.warmup, depth))
    barrier(world)
    t0 = time.perf_counter()
    run(k_steps)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3
    barrier(world)
    ms = nd.max_over_ranks(ms, device) / k_steps
    e2e_single.steps = k_steps
    found = float((last["score"] > READ_LEN).float().mean())
    h2d, d2h = stream.h2d_bytes, stream.d2h_bytes
    stream.close()
    return ms, h2d, d2h, found


def run_ours(args):
    import nvbio_b200 as nb
    from nvbio_b200 import aln
    from nvbio_b200.strings import PackedStringSet
    from nvbio_b200.pipeline import SeedExtendWorkspace, last_stage_ms
    from nvbio_b200 import dist as nd

    rank, local, world = setup_dist(args)
    device = torch.device("cuda", local)
    nb.lib()                                            # fail loudly if the CUDA library is missing
    n, genome, fmi, t_build, t_bcast = build_index(args, rank, world, device)
    n_reads = args.reads
    params = nb.SeedExtendParams(seed_len=SEED_LEN, seed_interval=SEED_INTERVAL, band_len=BAND, type=aln.LOCAL,
                                 both_strands=True, max_seed_hits=100, dedup_jobs=not args.no_dedup,
                                 scheme=aln.SimpleGotohScheme(*SCHEME))
    batches = [make_reads(genome, n, n_reads, rank * 16 + b, device) for b in range(2)]
    wpr = batches[0].shape[1]

    def as_set(words):
        return PackedStringSet.fixed(words.reshape(-1), n_reads, READ_LEN, stride=wpr * 16)
    hit_capacity = 24 * n_reads
    ws = SeedExtendWorkspace(fmi, genome, as_set(batches[0]), params, hit_capacity, keep_hits=False)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=device)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def step(words):
        nb.seed_extend(fmi, genome, as_set(words), params, workspace=ws)

    # ---- device-resident timing ------------------------------------------------------------
    sampler = ClockSampler(local); sampler.start()      # nvidia-smi needs ~0.5 s to deliver its first sample
    for i in range(args.warmup):
        flush.zero_(); step(batches[i % 2])
    barrier(world)
    total_ms, stage_acc, hits = 0.0, None, 0
    for i in range(args.steps):
        flush.zero_()
        ev0.record(); step(batches[i % 2]); ev1.record()
        torch.cuda.synchronize()
        total_ms += ev0.elapsed_time(ev1)
        st = last_stage_ms()
        stage_acc = st if stage_acc is None else {k: stage_acc[k] + st[k] for k in st}
        kept, hits, jobs = [int(v) for v in ws.n_hits.cpu()]
        if kept != hits:
            raise SystemExit("bench: hit capacity %d exceeded (%d hits): results would be truncated" % (hit_capacity, hits))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ws)             # before the untimed steps below overwrite the workspace
    barrier(world)
    # a K-step region of a few ms per step can end before nvidia-smi has sampled it: keep the same load running
    # (untimed) until the sampler holds a handful of in-load samples
    t_load = time.perf_counter()
    n_before = len(sampler.rows)
    while len(sampler.rows) < n_before + 5 and time.perf_counter() - t_load < 3.0:
        step(batches[0]); torch.cuda.synchronize()
    sampler.rows = sampler.rows[max(n_before - 1, 0):]
    clocks = sampler.stop()
    clocks["note"] = "sampled while the timed step kept running back to back (the K-step region alone is shorter than one nvidia-smi period)"
    total_ms = nd.max_over_ranks(total_ms, device)
    ms_per_step = total_ms / args.steps
    value = world * n_reads / (ms_per_step * 1e-3) / 1e6
    stage_ms = {k: v / args.steps for k, v in stage_acc.items()}

    # ---- end to end through the C ABI with host buffers ------------------------------------------
    # Inputs arrive from the host every step and the index (+SA +table) is far larger than L2, so no flush is needed here.
    del ws
    torch.cuda.empty_cache()
    e2e_ms, h2d, d2h, found = e2e_single(args, nb, fmi, genome, params, batches, n_reads, wpr, hit_capacity, world, nd, device, args.depth)
    e2e_value = world * n_reads / (e2e_ms * 1e-3) / 1e6
    e2e_alt = None
    if world == 1 and args.e2e_sweep:                   # other pipeline shapes, for the record: (batches in flight, compute streams)
        e2e_alt = []
        for dep, streams in ((1, 1), (2, 1), (3, 1), (2, 2), (3, 3)):
            os.environ["NVB_PIPELINE_COMPUTE_STREAMS"] = str(streams)
            ms1, _, _, _ = e2e_single(args, nb, fmi, genome, params, batches, n_reads, wpr, hit_capacity, world, nd, device, dep)
            e2e_alt.append({"depth": dep, "compute_streams": streams, "ms_per_step": ms1, "value": n_reads / (ms1 * 1e-3) / 1e6})
        os.environ.pop("NVB_PIPELINE_COMPUTE_STREAMS", None)

    # ---- paired-end composition (C5 shape), every world size --------------------------------------
    paired = None
    if args.pairs > 0:
        try:
            paired = paired_end_config(args, nb, fmi, genome, n, params, device, world, nd)
        except SystemExit:
            raise
        except Exception as e:
            if world > 1:
                raise                                    # a rank that skips the collectives would hang the others
            paired = {"error": repr(e)[:300]}
    if rank != 0:
        return
    # ---- algorithmic bytes (rank 0, every N: the same oracle count), CPU baseline + parity on this very configuration (N=1) ----
    n_seeds = 2 * n_reads * ((READ_LEN - SEED_LEN) // SEED_INTERVAL + 1)
    blocks_per_seed, tail_blocks, _ = count_blocks(args, n, genome, fmi)
    cpu = parity = None
    if world == 1 and not args.no_cpu_baseline:
        r = cpu_reference_leg(args, n, genome, fmi, steps=1, warmup=1, want_blocks=False, parity_with=(nb, params))
        cpu = {"value": r["value"], "unit": "Mreads/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"],
               "fm_match_Mseeds_s": r["mseeds_per_s"], "banded_gotoh_GCUPS": r["gcups"]}
        parity = r.get("parity")
    peak, peak_src = measured_peaks()
    # reference algorithm: every LF step fetches its distinct 32-byte blocks (SURVEY 8d).  This kernel replaces the first
    # k steps by one 8-byte table entry (one 32-byte sector), so ITS necessary traffic is the tail blocks + that sector.
    ref_bytes_per_seed = 32.0 * blocks_per_seed + SEED_LEN * 2 / 8.0 + 8.0
    bytes_per_seed = 32.0 * tail_blocks + (32.0 if args.ktab_k else 0.0) + SEED_LEN * 2 / 8.0 + 8.0
    fm_ms = stage_ms["seed_match"]
    achieved = n_seeds * bytes_per_seed / (fm_ms * 1e-3) / 1e9
    cells = jobs * READ_LEN * BAND
    idx_desc = index_description(fmi.sa_interval, fmi.ktab_k, n, fmi.nbytes() + genome.numel() * 4, located=fmi.ktab_located)
    line = {
        "metric": "Mreads/s (150bp) seed+extend", "value": value, "unit": "Mreads/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int32", "data": "synthetic", "config": workload_config(args, n, n_reads, world),
        "index": idx_desc,
        "e2e": {"value": e2e_value, "unit": "Mreads/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms,
                "api": "C ABI nvb_pipeline_submit / nvb_pipeline_wait via nvbio_b200.StreamingSeedExtend (pinned host in/out, %d batches in flight: copy-in, "
                       "compute and copy-out streams; wall clock from an empty pipeline to the last result read on the host)" % args.depth,
                "steps": args.steps, "depth": args.depth, "compute_streams": int(os.environ.get("NVB_PIPELINE_COMPUTE_STREAMS", "1")), "sweep": e2e_alt},
        # own kernels per step on the per-read path (the cub scan not counted): strings, seed match (+ its second pass when a k-mer table and
        # the full SA are present), count, read jobs, (shortcut check, scatter: LOCAL with a constant scheme), DP pair kernel, DP generic
        # kernel, init, reduce, finalize
        "gpu_launches": ((9 + 2 + (1 if (fmi.ktab_k and fmi.sa_interval == 1 and SEED_LEN > fmi.ktab_k) else 0)) if params.dedup_jobs else 8) * args.steps,
        "clocks": clocks,
        "roofline": {"kernel": "pipe_seed_match_kernel (FM-index backward search, %d seeds x %d LF steps)" % (n_seeds, SEED_LEN),
                     "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": measured_traffic("pipe_seed_match_kernel", ktab_k=args.ktab_k, genome_bp=n, reads=n_reads, ktab_located=int(fmi.ktab_located), single_row_fold=(fmi.sa_interval == 1)),
                     "peak_source": peak_src, "ms_per_launch": fm_ms,
                     "gather_rate": gather_rate(fm_ms, ktab_k=args.ktab_k, genome_bp=n, reads=n_reads, ktab_located=int(fmi.ktab_located),
                                                single_row_fold=(fmi.sa_interval == 1)),
                     "algorithmic_bytes_per_seed": bytes_per_seed, "blocks_per_seed": tail_blocks,
                     "reference_algorithm_bytes_per_seed": ref_bytes_per_seed, "reference_algorithm_blocks_per_seed": blocks_per_seed,
                     "reference_algorithm_equiv_GBs": n_seeds * ref_bytes_per_seed / (fm_ms * 1e-3) / 1e9,
                     "note": "32 B x distinct {bwt,occ} blocks per LF step after the %d-mer table look-up (plain-C oracle count on a read sample of this "
                             "workload, the same at every N) + one 32 B table sector + query + 8 B out; the reference algorithm (no table) needs "
                             "reference_algorithm_bytes_per_seed" % args.ktab_k},
        "stage_ms": stage_ms,
        "fm_match_Mseeds_s": n_seeds / (fm_ms * 1e-3) / 1e6,
        "banded_gotoh": {"alignments_per_step": hits, "distinct_jobs_scored": jobs, "effective_GCUPS": cells / (stage_ms["extend"] * 1e-3) / 1e9,
                         "band": BAND, "note": "cells = distinct jobs x 150 x 31 over the extension stage's time.  EFFECTIVE rate: jobs whose read lies on the "
                                               "seed's diagonal with 0-1 substitutions get their (bit-identical) result from the exact shortcut without "
                                               "running the DP (DESIGN.md 3.7; 42 % of the jobs at this error rate); the DP kernel's own rate is "
                                               "other_configs' C4 line (integer-issue bound, DPX s16x2)"},
        "reads_found_frac": found,
        "index_build": {"build_s": t_build, "broadcast_s": t_bcast},
    }
    if parity is not None:
        line["parity_on_headline_config"] = parity["ok"]
        line["parity"] = parity
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if paired is not None:
        line["paired_end"] = paired
    if world == 1 and not args.no_other_configs:
        del batches, flush
        torch.cuda.empty_cache()
        try:
            line["fm_match_reference_format"] = reference_format_fm_match(args, nb, fmi, n, genome, device, blocks_per_seed, peak)
        except Exception as e:
            line["fm_match_reference_format"] = {"error": repr(e)[:300]}
        del fmi, genome
        torch.cuda.empty_cache()
        try:
            line["other_configs"] = other_configs(device)
        except Exception as e:                       # never lose the headline line to a secondary measurement
            line["other_configs"] = {"error": repr(e)[:300]}
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: nvbio_b200 has no CPU fallback")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
