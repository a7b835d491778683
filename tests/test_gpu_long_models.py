"""Profiles of 1025 to 2048 nodes: every stage against the CPU oracle, the multi-warp envelope sweeps against the one-warp ones, whole
searches against the CPU backend, library conversion, and the 2048-node limit.

The long models are built here from node blocks of shipped models (common.concat_models): M = 1280 (48 nodes per lane, 6 warps per
window or envelope) and M = 2014 (64 nodes per lane, 8 warps).  The stage checks are the existing per-stage tests, run on these models
with their tolerances: MSV / SSV / Viterbi bit-exact, parsers within 1e-3 nat, posteriors within 1e-4, traces identical.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import common

M903 = common.SYNTHETIC["synthetic_M903.bhmm"]
M208 = common.SYNTHETIC["synthetic_M208.bhmm"]
LONG = {
    "M1280": M903 + [("tRNA-synthetases.bhmm", 0), ("tRNA-synthetases.bhmm", 1)],
    "M2014": M903 + M903 + M208,
}
LENGTHS = {"M1280": 1280, "M2014": 2014}
LONG_NAMES = sorted(LONG)


@pytest.fixture(scope="module")
def long_models(tmp_path_factory):
    d = tmp_path_factory.mktemp("long_models")
    out = {}
    for name, parts in LONG.items():
        path = str(d / f"synthetic_{name}.bhmm")
        common.concat_models(parts, path, f"synthetic_{name}")
        out[name] = path
    return out


@pytest.fixture(scope="module")
def long_ctx():
    """a device context that takes profiles of up to 2048 nodes (the session's context keeps the default 1024)"""
    from bath_b200 import capi
    ctx = capi.Context(0, long_models=True)
    yield ctx
    ctx.close()


# ---------------------------------------------------------------- CPU

@pytest.mark.parametrize("name", LONG_NAMES)
def test_long_models_load_on_the_host(oracle, long_models, name):
    """the host model set-up and the oracle take the long models whole (nothing on the host side stops at 1024 nodes)"""
    from bath_b200 import hostapi
    model = hostapi.QueryModel(long_models[name])
    assert model.M == LENGTHS[name]
    assert oracle.Model(long_models[name]).M == LENGTHS[name]


# ---------------------------------------------------------------- GPU: every stage against the oracle

@pytest.mark.gpu
@pytest.mark.parametrize("name", LONG_NAMES)
@pytest.mark.parametrize("lanes", [(16, 8), (32, 16)])
def test_filters_bit_exact_long(oracle, long_ctx, long_models, name, lanes):
    from test_gpu_orf_filters import test_filters_bit_exact
    test_filters_bit_exact(oracle, long_ctx, long_models[name], 0, lanes)


@pytest.mark.gpu
@pytest.mark.parametrize("name", LONG_NAMES)
def test_protein_forward_parser_long(oracle, long_ctx, long_models, name):
    from test_gpu_orf_filters import test_protein_forward_parser
    test_protein_forward_parser(oracle, long_ctx, long_models[name], 0)


@pytest.mark.gpu
@pytest.mark.parametrize("name", LONG_NAMES)
def test_forward_parser_long(oracle, long_ctx, long_models, name):
    from test_gpu_fs_forward import test_forward_parser_matches_oracle
    test_forward_parser_matches_oracle(oracle, long_ctx, long_models[name], 0)


@pytest.mark.gpu
@pytest.mark.parametrize("name", LONG_NAMES)
def test_backward_parser_long(oracle, long_ctx, long_models, name):
    from test_gpu_fs_backward import test_backward_and_domain_decoding_match_oracle
    test_backward_and_domain_decoding_match_oracle(oracle, long_ctx, long_models[name], 0)


def fewer(module, name, n_homolog, n_random):
    """module.name(rng, model, n_homolog, n_random) with fewer items: the matrices the checks fetch are those of the stage call's last
    chunk, so the envelopes of one check must fit the matrix budget together (2 GiB: 26 000 rows of a 2048-node envelope)"""
    orig = getattr(module, name)
    return lambda rng, model, *_, **__: orig(rng, model, n_homolog, n_random)


@pytest.mark.gpu
@pytest.mark.parametrize("name", LONG_NAMES)
def test_envelope_stage_long(oracle, long_ctx, long_models, name, monkeypatch):
    """the multi-warp Forward, Backward + decoding + null2 and optimal-accuracy sweeps, then the traceback"""
    import test_gpu_fs_domains as m
    monkeypatch.setattr(m, "make_envelopes", fewer(m, "make_envelopes", n_homolog=3, n_random=2))
    m.test_domain_stage_matches_oracle(oracle, long_ctx, long_models[name], 0)


@pytest.mark.gpu
def test_envelope_stage_long_chunks(oracle, long_ctx, long_models):
    """more 2014-node envelopes than the matrix budget holds at once: the call cuts them into chunks, and every envelope's scores,
    null2 and trace equal those of a call with that envelope alone"""
    from bath_b200 import capi
    from test_gpu_fs_domains import make_envelopes
    model = oracle.Model(long_models["M2014"])
    dsq, envs = make_envelopes(np.random.default_rng(3), model, n_homolog=8, n_random=3)
    assert sum(L + 1 for _, L in envs) > 26_214, "the envelopes must overflow one chunk"
    long_ctx.load_fs_profile(5, model.rfv(5), model.tfv(5))
    long_ctx.upload_block(dsq)
    res, tr = long_ctx.fs_domains(capi.Context.make_windows([s for s, _ in envs], [L for _, L in envs], nj=0.0), xfE5=(1.0, 0.0))
    for t, (s, L) in enumerate(envs):
        r1, t1 = long_ctx.fs_domains(capi.Context.make_windows([s], [L], nj=0.0), xfE5=(1.0, 0.0))
        for f in ("status", "envsc", "bcksc", "oasc", "null2", "trace_len"):
            assert res[f][t].tobytes() == r1[f][0].tobytes(), (t, f, res[f][t], r1[f][0])
        o = res["trace_offset"][t]
        assert tr[o: o + res["trace_len"][t]].tobytes() == t1[: r1["trace_len"][0]].tobytes(), t


@pytest.mark.gpu
@pytest.mark.parametrize("name", LONG_NAMES)
def test_forward_matrices_long(oracle, long_ctx, long_models, name):
    """bathgpu_fs_forward_matrices (D cells kept) on a tandem pair of homologs against the oracle's multihit Forward: cells within 2e-4
    of their row's largest entry.  A row is rescaled when its E value passes 1e4; at 2000 nodes the device's and the oracle's sums can
    fall on the two sides of that line, so the comparison undoes the scale factors, and rows whose factors differ must be such rows."""
    from bath_b200 import capi, hostapi
    from test_multidomain_cpu import tandem_target, multihit_forward
    model = oracle.Model(long_models[name])
    rng = np.random.default_rng(3)
    dsq, parts = tandem_target(oracle, model, rng, spacer=0, flank=150)
    n = len(dsq) - 2
    regions = [(101, n - 90), (140, 140 + parts[0] // 2)]
    long_ctx.load_fs_profile(5, model.rfv(5), model.tfv(5))
    long_ctx.upload_block(dsq)
    pm, pl = hostapi.length_model(100, nj=1.0)
    regs = capi.Context.make_windows([i for i, _ in regions], [j - i + 1 for i, j in regions], nj=1.0)
    regs["pmove"] = pm; regs["ploop"] = pl
    mx, xr, off, sc, st = long_ctx.fs_forward_matrices(regs, model.M, xfE5=(0.5, 0.5))
    for r, (i, j) in enumerate(regions):
        fwd, want_sc = multihit_forward(oracle, model, dsq, i, j)
        assert st[r] == 0 and abs(sc[r] - want_sc) <= 1e-3, (r, sc[r], want_sc)
        L = j - i + 1
        g_mx, g_xr = mx[off[r]: off[r] + L + 1], xr[off[r]: off[r] + L + 1]
        w_mx, w_xr = oracle.mx_dp(fwd), oracle.mx_xmx(fwd)
        gs, ws = g_xr[:, 5].astype(np.float64), w_xr[:, 5].astype(np.float64)
        assert np.allclose(gs[(gs > 1) & (ws > 1)], ws[(gs > 1) & (ws > 1)], rtol=1e-4), "scale factors of rows both sides rescaled"
        differ = np.nonzero((gs > 1) != (ws > 1))[0]
        for z in differ:                    # one side rescaled a row whose E the other kept just under the threshold
            lo, hi = (g_xr, w_xr) if g_xr[z, 5] == 1.0 else (w_xr, g_xr)
            assert abs(lo[z, 0] / 1e4 - 1) <= 1e-3 and abs(hi[z, 5] / 1e4 - 1) <= 1e-3, (r, z, g_xr[z], w_xr[z])
        fac = np.exp(np.cumsum(np.log(ws)) - np.cumsum(np.log(gs)))
        w_mx = w_mx.reshape(L + 1, -1) * fac[:, None]
        w_x = w_xr[:, :5] * fac[:, None]
        ref = np.maximum(np.maximum(w_mx.max(axis=1), w_x.max(axis=1)), 1e-30)[:, None]
        d = max(float(np.max(np.abs(g_mx.reshape(L + 1, -1) - w_mx) / ref)), float(np.max(np.abs(g_xr[:, :5] - w_x) / ref)))
        assert d <= 2e-4, (name, r, d)
        print(f"{name} region {r}: {len(differ)} rows rescaled on one side only, worst relative cell error {d:.2e}")
        oracle.lib().bo_mx_destroy(fwd)
    oracle.lib().bo_fs_oprofile_ReconfigUnihit(model.om_fs5, 100)


@pytest.mark.gpu
@pytest.mark.parametrize("name", LONG_NAMES)
def test_standard_branch_long(oracle, long_ctx, long_models, name, monkeypatch):
    import test_gpu_orf_domains as m
    m.test_orf_parsers_xrows_match_oracle(oracle, long_ctx, long_models[name], 0)
    monkeypatch.setattr(m, "make_orfs", fewer(m, "make_orfs", n_homolog=5, n_random=2))
    m.test_orf_domain_stage_matches_oracle(oracle, long_ctx, long_models[name], 0)


@pytest.mark.gpu
@pytest.mark.parametrize("which", [3, 5])
def test_set_scores_mixing_long_and_short_models(long_ctx, long_models, which):
    """bathgpu_fs_set_scores over a set of long and short models: bit-identical to loading each profile alone"""
    from bath_b200 import capi, hostapi
    models = [hostapi.QueryModel(long_models[n]) for n in LONG_NAMES]
    models += [hostapi.QueryModel(common.golden("AMP_N.bhmm")), hostapi.QueryModel(common.golden("synthetic_M903.bhmm")),
               hostapi.QueryModel(common.golden("tRNA-synthetases.bhmm"), 1)]
    rng = np.random.default_rng(23 + which)
    dsq = common.random_dna(rng, 300_000, p_degenerate=0.002)
    long_ctx.select_slot(0)
    long_ctx.upload_block(dsq)
    prof = rng.permutation(np.repeat(np.arange(len(models)), 4))
    lengths = rng.integers(6, 1500, len(prof))
    starts = rng.integers(1, 300_000 - lengths + 2)
    xfE = np.array([(0.5, 0.5) if p % 2 == 0 else (1.0, 0.0) for p in range(len(models))], np.float32)
    long_ctx.load_fs_profile_set(which, [(m.rfv(which), m.tfv(which)) for m in models])
    wins = capi.Context.make_set_windows(starts, lengths, prof)
    sc, st = long_ctx.fs_set_scores(which, wins, xfE)
    for p, m in enumerate(models):
        idx = np.nonzero(prof == p)[0]
        long_ctx.load_fs_profile(which, m.rfv(which), m.tfv(which))
        one = capi.Context.make_windows(starts[idx], lengths[idx])
        if which == 3:
            s1, t1 = long_ctx.fs_fwd_windows(one, tuple(xfE[p]))
        else:
            s1, t1 = np.empty(len(idx), np.float32), np.empty(len(idx), np.int32)
            xf = np.ascontiguousarray(xfE[p])
            fp = C.POINTER(C.c_float)
            long_ctx._check(long_ctx.lib.bathgpu_fs_forward_matrices(long_ctx.h, one.ctypes.data, len(idx), xf.ctypes.data_as(fp), None, None, 0,
                                                                    s1.ctypes.data_as(fp), t1.ctypes.data_as(C.POINTER(C.c_int32))))
        assert np.array_equal(st[idx], t1), (m.name, st[idx], t1)
        ok = t1 == 0
        assert np.array_equal(sc[idx][ok].view(np.uint32), s1[ok].view(np.uint32)), (m.name, which, sc[idx], s1)


# ---------------------------------------------------------------- GPU: multi-warp against one-warp envelope sweeps

_SWEEP = r"""
import sys, numpy as np
sys.path.insert(0, sys.argv[1])
import common
from bath_b200 import capi
from oracle import pyoracle
from test_gpu_fs_domains import make_envelopes
model = pyoracle.Model(common.golden(sys.argv[2]), 0)
dsq, envs = make_envelopes(np.random.default_rng(5), model, n_homolog=9, n_random=4)
ctx = capi.Context(0)
ctx.load_fs_profile(5, model.rfv(5), model.tfv(5))
ctx.upload_block(dsq)
e = capi.Context.make_windows([s for s, _ in envs], [l for _, l in envs], nj=0.0)
res, tr = ctx.fs_domains(e, xfE5=(1.0, 0.0))
out = {"status": res["status"], "envsc": res["envsc"], "null2": res["null2"], "trace_len": res["trace_len"],
       "trace_offset": res["trace_offset"]}
for f in ("st", "k", "i", "c", "pp"):
    out["tr_" + f] = np.array(tr[f][: int(res["trace_offset"][-1] + res["trace_len"][-1])])
for t, (s, L) in enumerate(envs):
    if res["status"][t] == 0:
        pp, oa, ppx, oax = ctx.fs_fetch_domain_matrices(t, model.M, L)
        out[f"pp{t}"] = pp
        out[f"oa{t}"] = oa
np.savez(sys.argv[3], **out)
ctx.close()
"""


def _sweep(tmp_path, hmm, mode):
    out = str(tmp_path / f"{hmm}_{mode}.npz")
    env = dict(os.environ, BATHGPU_FS5_MW=str(mode))
    here = os.path.dirname(os.path.abspath(__file__))
    env["PYTHONPATH"] = os.pathsep.join([os.path.dirname(here), here] + ([env["PYTHONPATH"]] if env.get("PYTHONPATH") else []))
    subprocess.run([sys.executable, "-c", _SWEEP, here, hmm, out], check=True, env=env, cwd=os.path.dirname(here))
    return np.load(out)


@pytest.mark.gpu
@pytest.mark.parametrize("hmm", ["synthetic_M624.bhmm", "synthetic_M903.bhmm"])
def test_forced_multi_warp_sweeps_match_one_warp(tmp_path, hmm):
    """BATHGPU_FS5_MW=2 runs the multi-warp envelope sweeps at 24 and 32 nodes per lane: the same posteriors within 1e-4 and the
    same traces as the one-warp sweeps (each in a process of its own, which reads the variable fresh)"""
    common.golden(hmm)
    one, mw = _sweep(tmp_path, hmm, 0), _sweep(tmp_path, hmm, 2)
    assert np.array_equal(one["status"], mw["status"])
    ok = one["status"] == 0
    assert ok.any()
    assert float(np.max(np.abs(one["envsc"][ok] - mw["envsc"][ok]))) <= 1e-3
    np.testing.assert_allclose(one["null2"][ok], mw["null2"][ok], rtol=1e-4, atol=1e-6)
    assert np.array_equal(one["trace_len"], mw["trace_len"])
    for f in ("st", "k", "i", "c"):
        assert np.array_equal(one["tr_" + f], mw["tr_" + f]), f
    assert float(np.max(np.abs(one["tr_pp"] - mw["tr_pp"]))) <= 1e-4
    for t in np.nonzero(ok)[0]:
        assert float(np.max(np.abs(one[f"pp{t}"] - mw[f"pp{t}"]))) <= 1e-4, t
        fa, fb = np.isfinite(one[f"oa{t}"]), np.isfinite(mw[f"oa{t}"])
        assert np.array_equal(fa, fb), t
        assert float(np.max(np.abs(one[f"oa{t}"][fa] - mw[f"oa{t}"][fa]))) <= 1e-3, t


# ---------------------------------------------------------------- GPU: whole searches, conversion, the limit

def planted_target(long_models, rng):
    """homologs of both long models (and a partial one) between random flanks, two sequences"""
    from bath_b200 import hostapi
    seqs = []
    for z, name in enumerate(LONG_NAMES):
        model = hostapi.QueryModel(long_models[name])
        from oracle import pyoracle
        mat = common.hmm_mat(pyoracle.Model(long_models[name]))
        ins = common.sample_homolog(rng, mat, fs_rate=0.005, stop_rate=0.001)
        part = common.sample_homolog(rng, mat, fs_rate=0.005, stop_rate=0.001)[: 3 * model.M // 2]
        body = np.concatenate([rng.integers(0, 4, 3000), ins, rng.integers(0, 4, 5000), part, rng.integers(0, 4, 2000)]).astype(np.uint8)
        seqs.append((f"target{z}", body))
    return seqs


@pytest.mark.gpu
@pytest.mark.parametrize("std_only", [0, 1])
@pytest.mark.parametrize("name", LONG_NAMES)
def test_search_long_model_matches_cpu_backend(oracle, long_ctx, long_models, name, std_only):
    """a search with a long model: the GPU search and the CPU-backend search write byte-identical tables"""
    from bath_b200 import hostapi
    seqs = planted_target(long_models, np.random.default_rng(41))
    tables = []
    for device in (True, False):
        model = hostapi.QueryModel(long_models[name])
        if device:
            search = hostapi.Search(model, long_ctx, std_only=std_only)
        else:
            be, keep = oracle.cpu_backend(4)
            search = hostapi.Search(model, backend=be, std_only=std_only)
        for sname, body in seqs:
            d = np.full(len(body) + 2, 255, np.uint8)
            d[1:-1] = body
            search.add_sequence(sname, d)
        hits = search.finish()
        tables.append((search.tblout(), len(hits)))
    assert tables[0][1] >= 1, "the planted homolog must be found"
    assert tables[0][0] == tables[1][0]


@pytest.mark.gpu
def test_convert_library_with_a_long_model(long_ctx, long_models, tmp_path):
    """a HMMER3/f library holding a 2014-node model converts, with the taus of the per-model calibration chain"""
    from bath_b200 import hostapi
    from test_convert import hmmer3_text, fs_lines
    parts = [(common.golden("AMP_N.bhmm"), 0), (long_models["M2014"], 0), (long_models["M1280"], 0)]
    src, dst = tmp_path / "lib.hmm", str(tmp_path / "lib.bhmm")
    src.write_text("".join(hmmer3_text(p) for p, _ in parts))
    assert hostapi.convert(str(src), dst, gpu_ctx=long_ctx) == len(parts)
    want, x = [], 0
    for p, i in parts:
        ev, x = hostapi.calibrate(hostapi.QueryModel(p, i), gpu_ctx=long_ctx, convert_flow=True, rng_state=x, which=24)
        want.append(f"STATS LOCAL FS3 FORWARD {np.float32(ev[6]):8.4f} {np.float32(ev[5]):8.5f}")
        want.append(f"STATS LOCAL FS5 FORWARD {np.float32(ev[7]):8.4f} {np.float32(ev[5]):8.5f}")
    assert fs_lines(open(dst).read()) == want


@pytest.mark.gpu
def test_profile_length_limits(gpu_ctx, long_ctx, long_models, tmp_path):
    """A context without long models refuses the 1280-node model with EINVAL and a message naming 1024; a context with them refuses
    M = 2148 with a message naming 2048, from the frameshift and filter loaders and from search creation.  Both keep working."""
    from bath_b200 import capi, hostapi
    path = str(tmp_path / "synthetic_M2148.bhmm")              # the 2014-node model and AMP_N's 134 nodes
    common.concat_models(LONG["M2014"] + [("AMP_N.bhmm", 0)], path, "synthetic_M2148")
    for ctx, model, limit in ((gpu_ctx, hostapi.QueryModel(long_models["M1280"]), "1024"), (long_ctx, hostapi.QueryModel(path), "2048")):
        assert model.M > int(limit)
        for which in (3, 5):
            with pytest.raises(capi.BathGpuError) as ei:
                ctx.load_fs_profile(which, model.rfv(which), model.tfv(which))
            assert ei.value.code == capi.EINVAL and limit in str(ei.value)
        with pytest.raises(capi.BathGpuError) as ei:
            ctx.load_filter_profile(model.filter_params(), *model.filter_tables())
        assert ei.value.code == capi.EINVAL and limit in str(ei.value)
        with pytest.raises(RuntimeError, match=f"status {capi.EINVAL}"):
            hostapi.Search(model, ctx)
        small = hostapi.QueryModel(common.golden("AMP_N.bhmm"))
        ctx.load_fs_profile(5, small.rfv(5), small.tfv(5))
    # switching long models off again brings the 1024-node limit back
    long_ctx.lib.bathgpu_set_long_models(long_ctx.h, 0)
    try:
        m1280 = hostapi.QueryModel(long_models["M1280"])
        with pytest.raises(capi.BathGpuError, match="1024"):
            long_ctx.load_fs_profile(3, m1280.rfv(3), m1280.tfv(3))
    finally:
        long_ctx.lib.bathgpu_set_long_models(long_ctx.h, 1)
