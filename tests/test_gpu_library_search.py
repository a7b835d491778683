"""GPU: the ORF screen over a profile set (bathgpu_orfs_msv_screen_set) against one bathgpu_orfs_msv_screen per profile, and the library
search (hostapi.LibrarySearch) against standalone GPU searches and against the CPU-backend library search."""
import ctypes as C

import numpy as np
import pytest

import common

pytestmark = pytest.mark.gpu

SHIPPED = ["2OG-FeII_Oxy_3.bhmm", "AMP_N.bhmm", "MET-ct4.bhmm", "PTH2.bhmm", "PTHR37536.bhmm", "tRNA-proteins.bhmm", "tRNA-synthetases.bhmm"]
LONG = {"M1280": common.SYNTHETIC["synthetic_M903.bhmm"] + [("tRNA-synthetases.bhmm", 0), ("tRNA-synthetases.bhmm", 1)],
        "M2014": common.SYNTHETIC["synthetic_M903.bhmm"] * 2 + common.SYNTHETIC["synthetic_M208.bhmm"]}


def _models(oracle, paths):
    out = []
    for p in paths:
        n = oracle.lib().bo_hmmfile_count(p.encode())
        out += [oracle.Model(p, i) for i in range(n)]
    return out


def _screen_matches_single(oracle, ctx, models, seed):
    from bath_b200 import capi
    from test_gpu_orf_filters import host_params
    from test_gpu_orf_finder import tables
    lib = oracle.lib()
    rng = np.random.default_rng(seed)
    n = 60000
    dsq = common.random_dna(rng, n, p_degenerate=0.002)
    for z, at in enumerate((2000, 20000, 41000)):                     # homologs of a few of the profiles: high scores, overflows
        ins = common.sample_homolog(rng, common.hmm_mat(models[(7 * z) % len(models)]), fs_rate=0.0, stop_rate=0.0)[: 9000]
        dsq[at: at + len(ins)] = ins
    ctx.select_slot(0)
    ctx.upload_block(dsq)
    ctx.revcomp_slot(0, 1)
    profiles = []
    for m in models:
        rbv, rwv, twv, _, _ = m.om_tables()
        profiles.append((host_params(oracle, m, 16, 8), rbv, rwv, twv))
    ctx.load_filter_profile_set([(p[0], p[1]) for p in profiles])
    gcode = np.frombuffer(C.string_at(lib.bo_gencode_basic(1), 64), np.uint8)
    tjb, null = tables(oracle, models[0], 14000 // 3 + 2)
    jobs = []
    for p in range(len(models)):                                       # blocks of 12 kb; the context differs from profile to profile
        C_ = 150 + 90 * (p % 7)
        bl = np.zeros(5, capi.block_dtype)
        for b in range(5):
            ctxn = 0 if b == 0 else C_
            bl[b]["goff"], bl[b]["n"], bl[b]["C"] = 12000 * b - ctxn, min(12000 + ctxn, n - 12000 * b + ctxn), ctxn
        jobs.append((p, bl, -1e30 if p % 2 == 0 else 2.0))
    nsurv = 0
    for slot in (0, 1):
        ctx.select_slot(slot)
        got = ctx.orfs_msv_screen_set(jobs, slot, gcode, 20, tjb, null)
        got = [(per.copy(), hits.copy(), res.copy()) for per, hits, res in got]
        for (p, bl, mb), (per, hits, res) in zip(jobs, got):
            ctx.load_filter_profile(*profiles[p])
            per1, hits1, res1 = ctx.orfs_msv_screen(bl, slot, gcode, 20, tjb, null, mb)
            assert np.array_equal(per, per1), (slot, p)
            assert len(hits) == len(hits1), (slot, p)
            for f in ("block", "index", "start", "end", "n", "frame", "status"):
                assert np.array_equal(hits[f], hits1[f]), (slot, p, f)
            assert np.array_equal(hits["usc"].view(np.uint32), hits1["usc"].view(np.uint32)), (slot, p)
            for h, h1 in zip(hits, hits1):
                assert np.array_equal(res[h["offset"]: h["offset"] + h["n"]], res1[h1["offset"]: h1["offset"] + h1["n"]])
            nsurv += len(hits)
    ms, norf, scored = ctx.orfs_stage_breakdown()
    assert norf > 0 and scored > 0 and ms[3] > 0
    assert nsurv > 1000


def test_screen_set_matches_single_profile_screens(oracle, gpu_ctx):
    """every shipped model plus the 624- and 903-node ones in one set (every MSV width up to 16 words per lane), both strands"""
    models = _models(oracle, [common.golden(p) for p in SHIPPED] + [common.golden("synthetic_M624.bhmm"), common.golden("synthetic_M903.bhmm")])
    assert len(models) <= 64
    _screen_matches_single(oracle, gpu_ctx, models, 5)


def test_screen_set_with_long_models(oracle, tmp_path):
    """the 1280- and 2014-node models (24 and 32 words per lane) in a set with short ones, on a long-model context"""
    from bath_b200 import capi
    paths = []
    for name, parts in LONG.items():
        path = str(tmp_path / f"synthetic_{name}.bhmm")
        common.concat_models(parts, path, f"synthetic_{name}")
        paths.append(path)
    models = _models(oracle, paths + [common.golden("AMP_N.bhmm"), common.golden("tRNA-synthetases.bhmm")])
    ctx = capi.Context(0, long_models=True)
    try:
        _screen_matches_single(oracle, ctx, models, 6)
    finally:
        ctx.close()


def _target(path, seed, n=250_000, ncontigs=2):
    from bath_b200 import hostapi, synth
    model = hostapi.QueryModel(common.golden(path), 0)
    rng = np.random.default_rng(seed)
    return [(f"contig{c + 1}", synth.planted_genome(rng, n, model.mat(), every=20_000, fs_rate=model.fsprob)[0]) for c in range(ncontigs)]


def _standalone(path, ctxs, targets, **opt):
    from bath_b200 import hostapi
    out = []
    for i in range(hostapi.load().bathhost_model_count(path.encode())):
        s = hostapi.Search(hostapi.QueryModel(path, i), ctxs, **opt)
        for name, dsq in targets:
            s.queue_sequence(name, dsq)
        s.finish(fetch=False)
        out.append((s.tblout(), {k: s.stats()[k] for k in COUNTERS}))
        s.close()
    return out


COUNTERS = ("nseqs", "nres", "pos_past_msv", "pos_past_bias", "pos_past_vit", "pos_past_fwd", "n_orfs", "n_windows", "n_std_windows",
            "n_regions", "n_multidomain_regions", "n_envelopes", "n_hits_reported")


def _library(path, targets, ctxs=None, backend=None, **opt):
    from bath_b200 import hostapi
    lib = hostapi.LibrarySearch(path, gpu_ctx=ctxs, backend=backend, **opt)
    for name, dsq in targets:
        lib.queue_sequence(name, dsq)
    lib.finish()
    out = [(s.tblout(), {k: s.stats()[k] for k in COUNTERS}) for s in lib.searches], lib.tblout()
    lib.close()
    return out


@pytest.mark.parametrize("std_only", [0, 1])
def test_library_search_equals_standalone_gpu_searches(oracle, gpu_ctx, std_only):
    from bath_b200 import capi
    path = common.golden("tRNA-proteins.bhmm")
    targets = _target("tRNA-proteins.bhmm", 11)
    extra = capi.Context(0)
    try:
        for ctxs in ([gpu_ctx], [gpu_ctx, extra]):
            ref = _standalone(path, ctxs, targets, std_only=std_only, block_length=60_000)
            assert sum(r[1]["n_hits_reported"] for r in ref) > 0
            per, table = _library(path, targets, ctxs=ctxs, std_only=std_only, block_length=60_000)
            assert per == ref
        be, keep = oracle.cpu_backend(8)
        cpu_per, cpu_table = _library(path, targets, backend=be, std_only=std_only, block_length=60_000)
        assert cpu_table == table
    finally:
        extra.close()


def test_library_larger_than_one_set_call(gpu_ctx, tmp_path):
    """78 models (tRNA-proteins six and a half times over): more than one set call holds, so the library is screened in groups; every
    copy of a model gives the table of that model's standalone search"""
    text = open(common.golden("tRNA-proteins.bhmm")).read()
    first = text.split("//\n")[0] + "//\n"
    path = str(tmp_path / "library.bhmm")
    with open(path, "w") as f:
        f.write(text * 6 + first * 6)
    targets = _target("tRNA-proteins.bhmm", 12, n=120_000, ncontigs=1)
    ref = _standalone(common.golden("tRNA-proteins.bhmm"), [gpu_ctx], targets)
    per, _ = _library(path, targets, ctxs=[gpu_ctx])
    assert len(per) == 78
    for i, (a, b) in enumerate(per):
        r = ref[i % 12] if i < 72 else ref[0]
        assert a == r[0] and b == r[1], i
