#!/usr/bin/env python
"""bench.py -- frameshift Forward throughput (GCUPS) of the translated-search hot path on B200.

Workload (BASELINE.json configs[2]): a Pfam-sized profile (tutorial tRNA-synthetases.bhmm, model 1,
M=192) against a 100 Mbp synthetic genome (iid ACGT, a frameshifted back-translated homolog planted
every 50 kbp, seed 42 + rank), tiled into 1200-nt DNA windows; one step = the frameshift Forward parser
(p7_ForwardParser_Frameshift_3Codons semantics) over every window of the genome.  Cells = sum Lw * M, the
reference's own Mc/s definition (src/impl_sse/fwdback_fs.c:3115).

  value  : device-timed (CUDA events on the launching stream), genome and descriptors resident in HBM
  e2e    : same step through the C ABI with HOST buffers: H2D of the block + window descriptors, 4-bit
           packing, Forward, D2H of scores/status -- wall clock around the calls
  roofline: FP32 pipe (the recursion is FMA work, SURVEY 8d): 20 FLOP/cell vs an FFMA probe measured in
           the same process; an HBM line is given too to show the kernel is nowhere near memory bound
  cpu_baseline / --impl reference: the restated CPU oracle (the reference itself needs Easel, which is not
           vendored, so it cannot be compiled) on all host cores, on a bounded sample of the same windows

N > 1: one process per GPU (torchrun), each rank owns its own 100 Mbp shard (weak scaling, no collective
on the DP path); the only communication is the barrier and the max-over-ranks of the timings.

Second metric, "search" (BASELINE.json configs[3] as written): bathsearch --fs Mbp/s of the three profiles of
tRNA-synthetases.bhmm against ONE synthetic genome in contigs of 1-10 Mbp with planted homologs of all three, sharded by
blocks over the N devices by ONE process (rank 0; bathhost_search_create_multi over 12-24 device contexts, the three profiles
searched at the same time by bathhost_search_finish_many) with one merged hit list per profile: strong scaling on a fixed target;
the one-profile-at-a-time order of the reference's query loop is timed beside it and must give the same tables.  At N > 1 the same search is also run on one device and the two
tables compared byte for byte (search.checks.hits_identical_to_1gpu); at N = 1 the GPU search of the CPU-baseline prefix
is compared with the CPU-oracle pipeline's table field by field (search.checks.hits_identical_to_cpu_prefix, rule in
search.checks.cpu_prefix_rule; byte identity per profile beside it).

--steps sets the timed steps of the Forward legs and the timed passes of the search.  --dump-outputs DIR writes what the last of
them computed: fs_fwd_scores / fs_fwd_status (one value per window) and search_hits_<profile> (one row per hit of the merged list,
columns SEARCH_HIT_FIELDS).  Every input is generated from a fixed seed, so two builds run with the same arguments can be compared
output for output.
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True    # the benchmark writes nothing in the tree it runs from (no __pycache__ either)

HMM_FILE = os.path.join(ROOT, "tests", "golden", "tRNA-synthetases.bhmm")
HMM_INDEX = 1
FLOP_PER_CELL = 20.0          # SURVEY 8d: 3-codon Forward parser, mul and add counted separately


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mbp", type=float, default=100.0, help="genome size per GPU, Mbp")
    ap.add_argument("--window", type=int, default=1200, help="DNA window length Lw")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="target CPU time of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--search-cpu-mbp", type=float, default=200.0, help="size of the CPU-baseline sample of the search leg, Mbp")
    ap.add_argument("--search-mbp", type=float, default=1000.0,
                    help="also run the whole stage-batched bathsearch --fs pipeline (3 profiles) over a genome of this many Mbp (0 = skip)")
    ap.add_argument("--no-filters-leg", action="store_true", help="skip the integer-filter roofline leg")
    ap.add_argument("--contexts-per-gpu", type=int, default=0,
                    help="device contexts per profile and GPU in the search leg (0: 4 on one or two GPUs, 2 on four, 1 on eight -- the three "
                         "profiles run at the same time and every context has a host thread of its own: 12-24 of them in all)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (Forward scores and status per window, the search's hit lists) to "
                         "DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's outputs: use it with --impl ours")
    return args


# ------------------------------------------------------------------------------------------------
DUMP_BYTES = 60 << 20             # all files of --dump-outputs together stay under 64 MB, .npy headers included
SEARCH_HIT_FIELDS = ("seqidx", "strand", "ali_from", "ali_to", "env_from", "env_to", "sq_len", "hmm_from", "hmm_to", "evalue", "lnP",
                     "score", "bias", "pre_score", "envsc", "oasc", "pid", "shifts", "stops", "trace_len")


def dump_arrays(outdir, arrays, budget):
    """Writes each array of {name: array} as outdir/<name>.npy (float32 stays float32, everything else becomes float64, exact for the
    integers written here).  An array larger than `budget` bytes is cut to a sample of its rows -- the same rows for arrays of the same
    length, drawn from a fixed seed -- whose row numbers go to <name>_rows.npy."""
    os.makedirs(outdir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        a = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
        row_bytes = a.itemsize * (a.size // max(len(a), 1))
        if a.nbytes > budget:
            keep = budget // (row_bytes + 8)
            rows = np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))
            a = a[rows]
            np.save(os.path.join(outdir, name + "_rows.npy"), rows.astype(np.float64))
        np.save(os.path.join(outdir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
            atexit.register(self._kill)            # a run that fails before stop() leaves no sampler running
        except Exception:
            self.proc = None

    def _kill(self):
        if self.proc is not None and self.proc.poll() is None:
            self.proc.kill()

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.path)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


# ------------------------------------------------------------------------------------------------
def make_workload(rank, mbp, window):
    from bath_b200 import hostapi, synth
    model = hostapi.QueryModel(HMM_FILE, HMM_INDEX)
    n = int(mbp * 1e6)
    rng = np.random.default_rng(42 + rank)
    dsq, plants = synth.planted_genome(rng, n, model.mat(), every=50000, fs_rate=model.fsprob)
    starts, lengths = synth.tile_windows(n, window)
    return model, dsq, starts, lengths, plants


def cpu_model_name():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def cpu_sample(model_M, dsq, starts, lengths, seconds, nthreads):
    """Times the CPU port (native build, all host threads) on a bounded prefix of the windows: the AVX2 + FMA build of the parser
    (oracle/fwd3_avx2.c) where the host has it -- the reference's production build is SIMD too -- and the scalar restatement, which is
    the checker, beside it.  The only place besides tests/ and smoke() where oracle/ is executed -- as the thing compared against.
    Returns (SIMD or scalar GCUPS, its description, windows checked, scalar scores of those windows, scalar GCUPS)."""
    from oracle import pyoracle as po
    po.lib(native=True)
    omodel = po.Model(HMM_FILE, HMM_INDEX)
    assert omodel.M == model_M

    def timed(simd, budget):
        probe = min(len(starts), 64 * nthreads)
        t0 = time.perf_counter()
        po.batch_forward_parser(omodel, dsq, starts[:probe], lengths[:probe], nthreads, simd=simd)
        dt = max(time.perf_counter() - t0, 1e-6)
        n = int(min(len(starts), max(probe, probe * budget / dt)))
        t0 = time.perf_counter()
        sc, st = po.batch_forward_parser(omodel, dsq, starts[:n], lengths[:n], nthreads, simd=simd)
        dt = time.perf_counter() - t0
        return float(lengths[:n].astype(np.int64).sum()) * model_M / dt / 1e9, n, dt, sc

    v_sc, n_sc, dt_sc, sc = timed(False, seconds * 0.5)
    if po.simd_supported():
        v, n, dt, ssc = timed(True, seconds * 0.5)
        m = min(n, n_sc)
        what = (f"first {n} of {len(starts)} windows ({dt:.1f} s, {nthreads} threads, AVX2+FMA port of the parser, -O3 -march=native, "
                f"{cpu_model_name()}; max |simd - scalar oracle| = {float(np.max(np.abs(ssc[:m] - sc[:m]))):.1e} nat on {m} windows)")
        return v, what, n_sc, sc, v_sc, "avx2+fma"
    what = f"first {n_sc} of {len(starts)} windows ({dt_sc:.1f} s, {nthreads} threads, scalar C oracle -O3 -march=native, {cpu_model_name()})"
    return v_sc, what, n_sc, sc, v_sc, "scalar"


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path on the host cores.  The reference
    binary cannot be built (Easel not vendored), so this is the restated oracle: kind = "port"."""
    if rank != 0:
        return
    model, dsq, starts, lengths, _ = make_workload(0, args.mbp, args.window)
    ncpu = os.cpu_count() or 1
    per_step = max(2.0, min(20.0, 120.0 / max(1, args.steps + args.warmup)))
    from oracle import pyoracle as po
    po.lib(native=True)
    omodel = po.Model(HMM_FILE, HMM_INDEX)
    simd = po.simd_supported()                      # the reference's production build is SIMD: so is this arm where the host allows
    probe = min(len(starts), 64 * ncpu)
    t0 = time.perf_counter()
    po.batch_forward_parser(omodel, dsq, starts[:probe], lengths[:probe], ncpu, simd=simd)
    dt = max(time.perf_counter() - t0, 1e-6)
    n = int(min(len(starts), max(probe, probe * per_step / dt)))
    for _ in range(args.warmup):
        po.batch_forward_parser(omodel, dsq, starts[:n], lengths[:n], ncpu, simd=simd)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        po.batch_forward_parser(omodel, dsq, starts[:n], lengths[:n], ncpu, simd=simd)
    dt = time.perf_counter() - t0
    cells = float(lengths[:n].astype(np.int64).sum()) * model.M
    value = cells * args.steps / dt / 1e9
    sample = (f"{n} of {len(starts)} windows of {args.window} nt per step ({cells / 1e9:.3f} Gcells), {ncpu} threads, "
              f"{'AVX2+FMA port of the parser (oracle/fwd3_avx2.c)' if simd else 'scalar C oracle'}, {cpu_model_name()}")
    search = search_leg_cpu(args.search_cpu_mbp, ncpu, args.search_mbp) if args.search_mbp > 0 else None
    emit_json_line({
        "impl": "reference", "metric": "frameshift Forward GCUPS", "value": value, "unit": "GCUPS",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, model.M, len(starts)),
        "cpu_baseline": {"value": value, "unit": "GCUPS", "cores": ncpu, "kind": "port", "simd": "avx2+fma" if simd else "scalar", "sample": sample},
        "e2e": {"value": value, "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "search": ({"metric": "bathsearch --fs Mbp/s", **search} if search else None),
        "note": "restated CPU port (AVX2+FMA build of the parser where the host has it, else scalar C; -O3 -march=native, pthreads over "
                "windows, FTZ/DAZ per thread as impl_Init sets them); the reference binary needs Easel, which is not vendored, so it "
                "cannot be compiled here",
    })


STD_CODE = "KNKNTTTTRSRSIIMIQHQHPPPPRRRRLLLLEDEDAAAAGGGGVVVV*Y*YSSSS*CWCLFLF"      # NCBI table 1, codon index 16 a + 4 b + c over ACGT


def filters_leg(ctx, model, n_nt, hbm_peak, hbm_src):
    """north_star's second roofline: the integer filters "against integer-ALU issue rate and HBM GB/s".  The Forward leg's genome is
    resident on the device (slot 0): six-frame translation + MSV over every ORF of the top strand in the pipeline's own call
    (bathgpu_orfs_msv_screen, blocks of 262144 nt with 3 x max_length of context), kernel groups timed with CUDA events, then the
    Viterbi filter over every ORF of the first blocks.  Algorithmic operation counts per DP cell as SURVEY 8(a) gives them
    (src/impl_sse/msvfilter.c:145-148: 4 byte operations per MSV cell; src/impl_sse/vitfilter.c:145-171: 14 16-bit operations per
    Viterbi cell) against the 16-bit lane-operation rate an in-process probe sustains (bathgpu_measure_int16_peak)."""
    from bath_b200 import capi
    M = model.M
    rbv, rwv, twv = model.filter_tables()
    ctx.load_filter_profile(model.filter_params(), rbv, rwv, twv)
    W, Cx = 262144, 3 * model.max_length
    blocks, pos = [], 1
    while pos <= n_nt:
        c = 0 if pos == 1 else min(Cx, pos - 1)
        b1 = min(n_nt, pos + W - 1)
        blocks.append((pos - c - 1, b1 - (pos - c) + 1, c))
        pos = b1 + 1
    bl = np.zeros(len(blocks), capi.block_dtype)
    bl["goff"], bl["n"], bl["C"] = [b[0] for b in blocks], [b[1] for b in blocks], [b[2] for b in blocks]
    maxlen = int(bl["n"].max()) // 3 + 2
    Ls = np.arange(maxlen + 1)
    tjb = np.zeros(maxlen + 1, np.uint8)
    xwm = np.zeros(maxlen + 1, np.int16)
    for L in range(1, maxlen + 1):
        tjb[L], xwm[L] = model.orf_length_params(L)
    tjb[0] = tjb[1]
    p1 = (Ls.astype(np.float32) / (Ls + 1).astype(np.float32)).astype(np.float64)
    null = np.zeros(maxlen + 1, np.float32)
    null[1:] = (Ls[1:] * np.log(p1[1:]) + np.log(1.0 - p1[1:])).astype(np.float32)
    aa = "ACDEFGHIKLMNPQRSTVWY"
    gcode = np.array([27 if ch == "*" else aa.index(ch) for ch in STD_CODE], np.uint8)
    ctx.select_slot(0)
    best = None
    for rep in range(4):                                         # first call allocates; best of the next three
        per, hits, res = ctx.orfs_msv_screen(bl, 0, gcode, 20, tjb, null, 8.0)
        ms, norf, nres = ctx.orfs_stage_breakdown()
        if rep >= 1 and (best is None or float(ms.sum()) < float(best[0].sum())):
            best = (ms.copy(), norf, nres)
    ms, norf, nres = [float(v) for v in best[0]], int(best[1]), int(best[2])
    int_peak = float(ctx.measure_int16_peak())
    msv_cells_s = nres * M / (ms[3] * 1e-3)
    finder_ms = float(ms[0] + ms[1] + ms[2] + ms[4])
    finder_bytes = float(n_nt / 2 + 4.0 * n_nt + nres)                  # packed strand read, classes written once and read by the two passes and by MSV, residues of survivors aside
    out = {"int16_peak_tera_ops": int_peak, "peak_source": "VIADDMNMX.S16x2 + VIMNMX.S16x2 probe in this process, one operation per instruction and 16-bit half (bathgpu_measure_int16_peak)",
           "strand_nt": int(n_nt), "orfs": norf, "residues_scored": nres, "survivors": int(len(hits)),
           "stage_ms": {"codon_classes": float(ms[0]), "orf_count_pass": float(ms[1]), "orf_emit_pass": float(ms[2]), "msv": float(ms[3]),
                        "screen_gather": float(ms[4])},
           "msv": {"cells_per_s": msv_cells_s, "ops_per_cell": 4, "achieved_tera_ops": msv_cells_s * 4 / 1e12,
                   "frac_of_int16_peak": msv_cells_s * 4 / 1e12 / int_peak,
                   "hbm": {"achieved": nres / (ms[3] * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s", "peak_source": hbm_src,
                           "note": "1 B per residue read from the class stream (stride 3) + 24 B of descriptor per ORF"}},
           "orf_finder": {"nt_per_s": n_nt / (finder_ms * 1e-3), "hbm": {"achieved": finder_bytes / (finder_ms * 1e-3) / 1e9, "peak": hbm_peak,
                          "unit": "GB/s", "frac": finder_bytes / (finder_ms * 1e-3) / 1e9 / hbm_peak, "algorithmic_bytes": finder_bytes}}}
    # Viterbi filter over every ORF of the first blocks (the pipeline runs it on the ~1 % that pass MSV + bias: too few to time)
    nb = min(len(bl), 40)
    per, hits, res = ctx.orfs_msv_screen(bl[:nb], 0, gcode, 20, tjb, null, -1e30)
    d = np.zeros(len(hits), capi.orf_dtype)
    d["offset"], d["L"] = hits["offset"], hits["n"]
    d["tjb_b"], d["xw_move"] = tjb[np.minimum(hits["n"], maxlen)], xwm[np.minimum(hits["n"], maxlen)]
    ctx.vit_orfs(d, max_wins=64)
    tv = float(min((ctx.vit_orfs(d, max_wins=64), ctx.last_stage_timing()[0])[1] for _ in range(3)))
    vit_cells_s = float(hits["n"].astype(np.int64).sum()) * M / (tv * 1e-3)
    out["viterbi"] = {"orfs": int(len(hits)), "ms": float(tv), "cells_per_s": vit_cells_s, "ops_per_cell": 14,
                      "achieved_tera_ops": vit_cells_s * 14 / 1e12, "frac_of_int16_peak": vit_cells_s * 14 / 1e12 / int_peak}
    return out


SEARCH_MODELS = (0, 1, 2)        # tRNA-synthetases.bhmm: M = 185, 192, 247


def search_target(mbp):
    """BASELINE configs[3]'s target: contigs of 1-10 Mbp, a homolog every 50 kbp taken in turn from the three profiles (seed 42)"""
    from bath_b200 import hostapi, synth
    models = [hostapi.QueryModel(HMM_FILE, i) for i in SEARCH_MODELS]
    rng = np.random.default_rng(42)
    total = int(mbp * 1e6)
    contigs, plants = synth.planted_contigs(rng, total, [m.mat() for m in models], every=50000, fs_rates=[m.fsprob for m in models],
                                            min_len=min(1_000_000, total), max_len=min(10_000_000, total))
    return models, contigs, plants


def compare_tables(a, b):
    from bath_b200 import hostapi
    return hostapi.compare_tables(a, b)


def run_search(models, contigs, gpu_ctxs=None, backends=None, **options):
    """every profile against the whole target, one profile after the other: (seconds per profile, tables, stats, hit lists)"""
    from bath_b200 import hostapi
    secs, tables, stats, hits = [], [], [], []
    for model in models:
        search = hostapi.Search(model, gpu_ctx=gpu_ctxs, backend=backends, **options)
        t0 = time.perf_counter()
        for name, dsq in contigs:
            search.queue_sequence(name, dsq)
        search.finish(fetch=False)                 # the C call returns with the merged, thresholded hit list in host memory
        secs.append(time.perf_counter() - t0)
        h = search.hits()                          # ctypes structs -> Python dicts: harness work, not timed
        tables.append(search.tblout(header=False))
        stats.append(search.stats())
        hits.append(h)
        search.close()
    return secs, tables, stats, hits


def run_search_together(models, contigs, ctx_sets):
    """the profiles of the query file searched at the same time, each over its own device contexts (bathhost_search_finish_many):
    (seconds for all of them, tables, stats, hit lists)"""
    from bath_b200 import hostapi
    searches = [hostapi.Search(m, gpu_ctx=cs) for m, cs in zip(models, ctx_sets)]
    t0 = time.perf_counter()
    for s in searches:
        for name, dsq in contigs:
            s.queue_sequence(name, dsq)
    hostapi.Search.finish_many(searches)
    dt = time.perf_counter() - t0
    hits = [s.hits() for s in searches]
    tables = [s.tblout(header=False) for s in searches]
    stats = [s.stats() for s in searches]
    for s in searches:
        s.close()
    return dt, tables, stats, hits


def recovered(hits_per_model, contigs, plants):
    """planted homologs overlapped by a hit of their own profile on their own contig"""
    names = [n for n, _ in contigs]
    by = {}
    for k, hits in enumerate(hits_per_model):
        for h in hits:
            by.setdefault((k, h["name"]), []).append((min(h["ali_from"], h["ali_to"]), max(h["ali_from"], h["ali_to"])))
    found = 0
    for c, a, b, strand, k in plants:
        if any(lo <= b and hi >= a for lo, hi in by.get((k, names[c]), ())):
            found += 1
    return found


def search_leg(devices, per_gpu, mbp, cpu_mbp, with_cpu, steps):
    """BASELINE.json's second metric on rank 0: bathsearch --fs end to end (ORF translation, MSV/bias/Viterbi/Forward filters, DNA
    windows, frameshift Forward/Backward, domain definition, rescoring, merged hit list) through the host pipeline
    (bath_b200/host/pipeline.cpp) and the C ABI, host buffers in, hit records out, for each of the three profiles.  Mbp/s = target
    nucleotides x profiles (one strand counted, both searched) / wall seconds of one of `steps` timed passes.  Returns the JSON
    record and the hit lists of the last timed pass, one per profile."""
    from bath_b200 import capi, hostapi
    models, contigs, plants = search_target(mbp)
    pinned = []
    for name, dsq in contigs:                                  # the target sits in page-locked host memory, as the e2e leg's inputs do
        buf = capi.pinned_array(dsq.shape, np.uint8)
        buf[:] = dsq
        pinned.append((name, buf))
    total_nt = sum(len(d) - 2 for _, d in contigs)
    # the three profiles run at the same time, each over per_gpu contexts of its own on every device
    sets = [[capi.Context(d) for d in devices for _ in range(per_gpu)] for _ in models]
    # untimed passes of the three profiles first (device buffers and page-locked host buffers reach their working sizes, kernels of
    # every model size get loaded: the steady state of a multi-query search); the first one's time is reported as first_pass_seconds
    t0 = time.perf_counter()
    run_search_together(models, pinned, sets)
    cold = time.perf_counter() - t0
    run_search_together(models, pinned, sets)                  # second untimed pass: with the searches running at the same time, buffers change hands between passes
    passes = []
    for _ in range(steps):                                     # --steps timed passes; the metric is the target searched that often / their total time
        dt_k, tables, stats, hits = run_search_together(models, pinned, sets)
        passes.append(dt_k)
    dt = sum(passes) / len(passes)
    # the reference's own order beside it: one profile after the other, every context of the first set + second set on each
    ctxs = sets[0] + sets[1]
    run_search(models, pinned, gpu_ctxs=ctxs)
    secs, tables_serial, _, _ = run_search(models, pinned, gpu_ctxs=ctxs)
    out = {"metric": "bathsearch --fs Mbp/s", "value": total_nt * len(models) / dt / 1e6, "unit": "Mbp/s", "seconds": dt, "seconds_per_pass": passes,
           "one_profile_at_a_time": {"value": total_nt * len(models) / sum(secs) / 1e6, "seconds_per_profile": secs, "contexts_per_gpu": 2 * per_gpu},
           "first_pass_seconds": cold, "target_mbp": total_nt / 1e6, "contigs": len(contigs), "profiles": [m.M for m in models],
           "n_gpus": len(devices), "contexts_per_gpu": per_gpu * len(models), "contexts_per_profile_per_gpu": per_gpu, "scaling": "strong",
           "hits": [len(h) for h in hits], "planted": len(plants), "planted_recovered": recovered(hits, contigs, plants),
           "stats": stats[1], "stats_per_profile": stats, "checks": {"tables_identical_to_one_profile_at_a_time": bool(tables == tables_serial)},
           "note": "one process drives every device: the three profiles are searched at the same time (bathhost_search_finish_many, one "
                   "search per profile over device contexts of its own on every GPU; bathhost_search_create_multi deals the blocks of the "
                   "one target to a search's contexts); the hit-window list / length-model chain / residue counts are kept in the "
                   "reference's serial order on the host, one merged hit list per profile; stage times in stats are summed over contexts"}
    if len(devices) > 1:                                        # the same search on one device: the tables must agree byte for byte
        one = [[capi.Context(devices[0]) for _ in range(4)] for _ in models]     # the 1-GPU configuration of this bench
        run_search_together(models, pinned, one)
        dt1, tables1, _, _ = run_search_together(models, pinned, one)
        out["one_gpu"] = {"value": total_nt * len(models) / dt1 / 1e6, "seconds": dt1, "contexts_per_profile_per_gpu": 4}
        out["checks"]["hits_identical_to_1gpu"] = bool(tables1 == tables)
        for cs in one:
            for c in cs:
                c.close()
    if with_cpu:
        # CPU baseline of this metric: the same pipeline over the CPU oracle's stage calls on a bounded prefix of the target; the GPU
        # search of the same prefix must write the same table
        from oracle import pyoracle as po
        po.lib(native=True)
        ncpu = os.cpu_count() or 1
        sub, n = cpu_sample_contigs(contigs, cpu_mbp)
        be, keep = po.cpu_backend(ncpu, simd=True)
        run_search(models[:1], sub[:1], backends=be)              # thread pool and tables warm, as the GPU arm's untimed first pass
        t0 = time.perf_counter()
        csecs, ctables, _, chits = run_search(models, sub, backends=be)
        cdt = time.perf_counter() - t0
        del keep
        _, gtables, _, _ = run_search(models, sub, gpu_ctxs=ctxs)
        out["cpu_baseline"] = {"value": n * len(models) / cdt / 1e6, "unit": "Mbp/s", "cores": ncpu, "kind": "port", "hits": [len(h) for h in chits],
                               "seconds_per_profile": csecs,
                               "sample": f"first {n / 1e6:g} Mbp of the target ({len(sub)} contigs), 3 profiles ({cdt:.1f} s, {ncpu} threads, C oracle behind the same host pipeline, its MSV / SSV screen on the AVX2 build where the host has AVX2)"}
        cmp = [compare_tables(g, c) for g, c in zip(gtables, ctables)]
        out["checks"]["hits_identical_to_cpu_prefix"] = bool(all(c[1] for c in cmp))
        out["checks"]["cpu_prefix_tables_byte_identical"] = [bool(c[0]) for c in cmp]
        out["checks"]["cpu_prefix_lines_that_differ"] = [int(c[2]) for c in cmp]
        out["checks"]["cpu_prefix_rule"] = ("hits_identical_to_cpu_prefix (hostapi.compare_tables): the same hit set -- hits matched by target, query, "
                                            "model and target coordinates, frameshift/stop counts and CIGAR string; E-value, score, bias and identity of a "
                                            "hit equal to within one unit of the last printed digit; rank changes only among hits whose printed E-values agree")
    for cs in sets:
        for c in cs:
            c.close()
    return out, hits


def search_leg_cpu(mbp, nthreads, target_mbp):
    """--impl reference: the same pipeline with the CPU oracle behind the stage calls (oracle/cpu_backend.c) on all host threads, on a
    bounded prefix of the target.  Oracle code is the thing timed here, never part of the product path."""
    from oracle import pyoracle as po
    po.lib(native=True)
    models, contigs, plants = search_target(target_mbp)
    sub, n = cpu_sample_contigs(contigs, mbp)
    be, keep = po.cpu_backend(nthreads, simd=True)
    run_search(models[:1], sub[:1], backends=be)
    t0 = time.perf_counter()
    secs, tables, stats, hits = run_search(models, sub, backends=be)
    dt = time.perf_counter() - t0
    del keep
    return {"value": n * len(models) / dt / 1e6, "unit": "Mbp/s", "cores": nthreads, "kind": "port", "hits": [len(h) for h in hits],
            "seconds_per_profile": secs,
            "sample": f"first {n / 1e6:g} Mbp of the target ({len(sub)} contigs), 3 profiles ({dt:.1f} s, {nthreads} threads, C oracle behind the same host pipeline, its MSV / SSV screen on the AVX2 build where the host has AVX2)"}


def cpu_sample_contigs(contigs, mbp):
    """the CPU arm's bounded sample of the search target: whole contigs in order until <mbp> Mbp, the last one cut"""
    want, sub, got = int(mbp * 1e6), [], 0
    for name, dsq in contigs:
        if got >= want:
            break
        n = min(len(dsq) - 2, want - got)
        if n == len(dsq) - 2:
            sub.append((name, dsq))
        else:
            cut = np.full(n + 2, 255, np.uint8)
            cut[1:-1] = dsq[1:n + 1]
            sub.append((name, cut))
        got += n
    return sub, got


def workload_config(args, M, nwin):
    return {"workload": f"tRNA-synthetases.bhmm[{HMM_INDEX}] (M={M}) frameshift Forward parser vs {args.mbp:g} Mbp synthetic genome "
                        f"per GPU, planted frameshifted homologs every 50 kbp, tiled into {args.window}-nt windows",
            "profile_M": M, "genome_mbp_per_gpu": args.mbp, "window_nt": args.window, "windows_per_gpu": nwin,
            "l2": "flushed between timed steps (512 MiB device write, untimed)", "sharding": "genome windows per GPU, profile replicated"}


# ------------------------------------------------------------------------------------------------
# Rank 0 prints exactly ONE line on stdout.  Libraries write there too (NCCL's version banner appears on some boxes whatever
# NCCL_DEBUG says), so file descriptor 1 is pointed at stderr for the whole run and the JSON line goes to the saved descriptor.
_JSON_FD = None


def capture_stdout():
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit_json_line(obj):
    data = (json.dumps(obj) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_JSON_FD, data)


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    capture_stdout()

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from bath_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"       # keep NCCL's version banner out of stdout: rank 0 prints exactly one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    # the ranks that wait while rank 0 runs the sharded search wait on the CPU (an NCCL barrier would spin on their GPUs, which rank 0 is using)
    cpu_group = dist.new_group(backend="gloo") if world > 1 else None

    def cpu_barrier():
        if world > 1:
            dist.barrier(group=cpu_group)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    from bath_b200 import ranks

    def max_over_ranks(x):
        return ranks.reduce_scalar(x, "max", device="cuda")

    def sum_over_ranks(x):
        return ranks.reduce_scalar(x, "sum", device="cuda")

    model, dsq_np, starts, lengths, plants = make_workload(rank, args.mbp, args.window)
    nplants = len(plants)
    M, nwin = model.M, len(starts)
    cells_local = float(lengths.astype(np.int64).sum()) * M

    ctx = capi.Context(local_rank)
    ctx.load_fs_profile(3, model.rfv(3), model.tfv(3))
    fp32_peak, eff_mhz = ctx.measure_fp32_peak()

    # host buffers of the e2e leg: pinned, filled once (the copies are what is timed, not the generation)
    dsq = capi.pinned_array(dsq_np.shape, np.uint8)
    dsq[:] = dsq_np
    wins = capi.pinned_array((nwin,), capi.window_dtype)
    wins[:] = capi.Context.make_windows(starts, lengths, nj=1.0)
    xfE = (0.5, 0.5)

    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")

    # ---- device-resident timing -------------------------------------------------------------
    ctx.upload_block(dsq)
    ctx.stage_windows(wins)
    for _ in range(max(args.warmup, 3)):
        ctx.fs_fwd_staged(xfE)
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    dev_ms, launches = 0.0, 0
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        flush.zero_()
        torch.cuda.synchronize()
        ctx.fs_fwd_staged(xfE)
        ms, nl = ctx.last_stage_timing()
        dev_ms += ms
        launches += nl
    barrier()
    wall_ms = (time.perf_counter() - t_wall0) * 1e3
    dev_ms = max_over_ranks(dev_ms)
    sc_dev, st_dev = ctx.fetch_scores(nwin)
    dump_budget = DUMP_BYTES // (2 * world + len(SEARCH_MODELS))          # per file: every rank's two, rank 0's hit lists
    if args.dump_outputs:
        sfx = f"_rank{rank}" if world > 1 else ""
        dump_arrays(args.dump_outputs, {"fs_fwd_scores" + sfx: sc_dev, "fs_fwd_status" + sfx: st_dev.astype(np.float32)}, dump_budget)

    # ---- end to end through the C ABI with host buffers -------------------------------------
    sc = capi.pinned_array((nwin,), np.float32)
    st = capi.pinned_array((nwin,), np.int32)
    for _ in range(2):
        ctx.fs_fwd_block_into(dsq, wins, xfE, sc, st)          # upload + score in one C-ABI call (the upload rides behind the kernel)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ctx.fs_fwd_block_into(dsq, wins, xfE, sc, st)
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    clocks = sampler.stop() if rank == 0 else None
    if not np.array_equal(sc, sc_dev) or not np.array_equal(st, st_dev):
        raise SystemExit("e2e and device-resident runs disagree")
    # the same call on a host-packed block (two nucleotides per byte, packed once outside the timed region as a sequence reader
    # would hand it over): half the H2D bytes, no packing kernel -- reported beside the headline e2e, which stays on ESL_DSQ bytes
    packed = capi.pinned_array(((len(dsq) - 2 + 1) // 2,), np.uint8)
    capi.pack_dna4(dsq, out=packed)
    sc4 = capi.pinned_array((nwin,), np.float32)
    st4 = capi.pinned_array((nwin,), np.int32)
    for _ in range(2):
        ctx.fs_fwd_block_packed4_into(packed, len(dsq) - 2, wins, xfE, sc4, st4)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ctx.fs_fwd_block_packed4_into(packed, len(dsq) - 2, wins, xfE, sc4, st4)
    barrier()
    e2e4_s = max_over_ranks(time.perf_counter() - t0)
    if not np.array_equal(sc4, sc_dev) or not np.array_equal(st4, st_dev):
        raise SystemExit("packed e2e and device-resident runs disagree")
    n_ok = int((st == 0).sum())

    cells_total = sum_over_ranks(cells_local)
    value = cells_total * args.steps / (dev_ms * 1e-3) / 1e9
    e2e_value = cells_total * args.steps / e2e_s / 1e9
    h2d = int(dsq.nbytes + wins.nbytes)
    d2h = int(sc.nbytes + st.nbytes)

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"

    # ---- the integer filters' roofline (rank 0; the strand is still resident on the device)
    filters = None
    if rank == 0 and not args.no_filters_leg:
        filters = filters_leg(ctx, model, len(dsq_np) - 2, hbm_peak, hbm_src)

    # ---- second metric: the whole search, config 4 as written: ONE target, three profiles, blocks dealt to the N devices by one process
    # (rank 0 drives every device; the other ranks wait at the barrier with their devices idle)
    search = None
    if args.search_mbp > 0:
        ctx.close()
        del flush
        torch.cuda.empty_cache()
        barrier()
        devices = ranks.search_devices(rank, world, torch.cuda.device_count())
        if devices:
            per_gpu = args.contexts_per_gpu if args.contexts_per_gpu > 0 else max(1, min(4, 8 // len(devices)))
            search, hits = search_leg(devices, per_gpu, args.search_mbp, args.search_cpu_mbp, world == 1 and not args.no_cpu_baseline,
                                      args.steps)
            if args.dump_outputs:                                 # one row per hit in the merged list, columns SEARCH_HIT_FIELDS
                dump_arrays(args.dump_outputs, {f"search_hits_{k}": np.array([[h[f] for f in SEARCH_HIT_FIELDS] for h in hk], np.float64)
                                                .reshape(-1, len(SEARCH_HIT_FIELDS)) for k, hk in zip(SEARCH_MODELS, hits)}, dump_budget)
        cpu_barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    per_gpu_cells_s = cells_local * args.steps / (dev_ms * 1e-3)
    achieved_tf = FLOP_PER_CELL * per_gpu_cells_s / 1e12
    # DRAM traffic of one launch of the dominant kernel from the committed ncu --set full capture of this same workload
    traffic = None
    try:
        tr = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "forward_traffic.json")))
        if tr.get("profile_M") == M and tr.get("windows") == nwin:
            traffic = {"bytes_per_launch": tr["dram_bytes_read"] + tr["dram_bytes_write"], "dram_bytes_read": tr["dram_bytes_read"],
                       "dram_bytes_write": tr["dram_bytes_write"], "source": tr["source"]}
    except (OSError, ValueError, KeyError):
        pass
    alg_bytes = float(lengths.astype(np.int64).sum()) / 2 + nwin * (24 + 8)      # packed DNA in, descriptors in, score+status out
    out = {
        "metric": "frameshift Forward GCUPS", "value": value, "unit": "GCUPS", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, M, nwin),
        "e2e": {"value": e2e_value, "unit": "GCUPS", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_s / args.steps * 1e3,
                "host_packed_4bit": {"value": cells_total * args.steps / e2e4_s / 1e9, "unit": "GCUPS", "ms_per_step": e2e4_s / args.steps * 1e3,
                                     "h2d_bytes_per_step": int(packed.nbytes + wins.nbytes), "d2h_bytes_per_step": d2h,
                                     "note": "bathgpu_fs_fwd_block_packed4: the block handed over two nucleotides per byte (packed outside the timed region)"}},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": {"bound": "fp32", "achieved": achieved_tf, "peak": fp32_peak, "unit": "TFLOP/s",
                     "frac": achieved_tf / fp32_peak, "traffic": traffic,
                     "kernel": "fs3_forward_parser_kernel", "flop_per_cell": FLOP_PER_CELL,
                     "peak_source": f"FFMA probe in this process ({eff_mhz:.0f} MHz effective x 148 SM x 128 lanes x 2)",
                     "hbm": {"achieved": alg_bytes * args.steps / (dev_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                             "frac": alg_bytes * args.steps / (dev_ms * 1e-3) / 1e9 / hbm_peak, "peak_source": hbm_src,
                             "algorithmic_bytes_per_step": alg_bytes}},
        "checks": {"windows": nwin, "status_ok": n_ok, "planted_homologs": nplants, "max_score_nats": float(np.max(sc)),
                   "wall_ms_timed_loop_incl_flush": wall_ms},
    }
    if filters is not None:
        out["roofline_filters"] = filters
    if search is not None:
        out["search"] = search
    if world == 1 and not args.no_cpu_baseline:
        ncpu = os.cpu_count() or 1
        v, what, n, osc, v_scalar, simd = cpu_sample(M, dsq_np, starts, lengths, args.cpu_seconds, ncpu)
        out["cpu_baseline"] = {"value": v, "unit": "GCUPS", "cores": ncpu, "kind": "port", "simd": simd, "sample": what,
                               "scalar_oracle_value": v_scalar}
        out["checks"]["max_abs_diff_vs_oracle_nats"] = float(np.max(np.abs(osc - sc[:n])))
        out["checks"]["windows_checked_against_oracle"] = int(n)
    emit_json_line(out)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
