"""HMMER3/f -> BATH3/f conversion (bathhost_convert, hostapi.convert) and the profile-set calls it batches the frameshift calibration
with (bathgpu_load_fs_profile_set, bathgpu_fs_set_scores).

The HMMER3/f inputs are derived from shipped bathconvert outputs: header "HMMER3/f [3.3 | Nov 2019]", the FS3 / FS5 STATS,
FRAMESHIFT PROB and CODON TABLE lines deleted.  Converting them back must give the shipped file, the two FS STATS values within the
2.5e-4 test_calibration.py holds the calibration to, and exactly the values of the per-model calibration loop."""
import ctypes as C
import os

import numpy as np
import pytest

import common

TOL = 2.5e-4
FS_TAGS = ("STATS LOCAL FS3", "STATS LOCAL FS5", "FRAMESHIFT PROB", "CODON TABLE")
CONVERTED = [("tRNA-proteins.bhmm", 12, 1), ("MET-ct4.bhmm", 2, 4), ("PTHR37536.bhmm", 1, 1)]


def hmmer3_text(name):
    out = []
    for line in open(common.golden(name)):
        if line.startswith("BATH3/f"):
            out.append("HMMER3/f [3.3 | Nov 2019]\n")
        elif not line.startswith(FS_TAGS):
            out.append(line)
    return "".join(out)


def write_hmmer3(tmp_path, name):
    p = tmp_path / (name.replace(".bhmm", ".hmm"))
    p.write_text(hmmer3_text(name))
    return str(p)


def fs_lines(text):
    return [l for l in text.splitlines() if l.startswith(("STATS LOCAL FS3", "STATS LOCAL FS5"))]


def loop_lines(name, count, **kw):
    """the FS STATS lines the per-model calibration loop gives (generator carried from model to model), printed as the writer prints"""
    from bath_b200 import hostapi
    out, x = [], 0
    for i in range(count):
        ev, x = hostapi.calibrate(hostapi.QueryModel(common.golden(name), i), convert_flow=True, rng_state=x, which=24, **kw)
        out.append(f"STATS LOCAL FS3 FORWARD {np.float32(ev[6]):8.4f} {np.float32(ev[5]):8.5f}")
        out.append(f"STATS LOCAL FS5 FORWARD {np.float32(ev[7]):8.4f} {np.float32(ev[5]):8.5f}")
    return out


def check_against_shipped(name, got, want_fs):
    shipped = open(common.golden(name)).read()
    other = lambda t: [l for l in t.splitlines() if not l.startswith(("STATS LOCAL FS3", "STATS LOCAL FS5"))]
    assert other(got) == other(shipped)                               # every other byte as the shipped file
    assert got.endswith("\n") and len(got.splitlines()) == len(shipped.splitlines())
    g, s = fs_lines(got), fs_lines(shipped)
    assert g == want_fs                                               # the per-model loop, value for value
    assert len(g) == len(s)
    identical = 0
    for a, b in zip(g, s):
        fa, fb = a.split(), b.split()
        assert fa[:4] == fb[:4] and fa[5] == fb[5]
        assert abs(float(fa[4]) - float(fb[4])) <= TOL, (a, b)
        identical += a == b
    print(f"{name}: {identical} of {len(s)} FS STATS lines byte-identical to the shipped file")
    return identical


# ---------------------------------------------------------------- CPU: the per-model path over the oracle's stage calls

@pytest.mark.parametrize("name,count,ct", CONVERTED)
def test_convert_reproduces_shipped_files_cpu(oracle, tmp_path, name, count, ct):
    from bath_b200 import hostapi
    be, keep = oracle.cpu_backend(4)
    src, dst = write_hmmer3(tmp_path, name), str(tmp_path / "out.bhmm")
    assert hostapi.convert(src, dst, backend=be, ct=ct) == count
    check_against_shipped(name, open(dst).read(), loop_lines(name, count, backend=be))
    del keep


def test_convert_rejects_other_formats_and_bad_arguments(oracle, tmp_path):
    from bath_b200 import hostapi
    be, keep = oracle.cpu_backend(1)
    dst = tmp_path / "out.bhmm"
    text = hmmer3_text("PTHR37536.bhmm")
    cases = [(common.golden("PTHR37536.bhmm"), {}, 7),                                 # already BATH3/f
             (text.replace("HMMER3/f [3.3 | Nov 2019]", "HMMER2.0  [2.3.2]"), {}, 7),   # another format's header
             (text.replace("HMMER3/f", "HMMER3/e"), {}, 7),                             # an older HMMER3 letter
             (text + "garbage\n", {}, 7),                                               # a bad header after a good model
             (text, {"ct": 7}, 11),                                                     # no codon table 7
             (text, {"fsprob": 0.3}, 11)]
    for k, (src, kw, code) in enumerate(cases):
        if not os.path.exists(src):
            p = tmp_path / f"in{k}.hmm"
            p.write_text(src)
            src = str(p)
        with pytest.raises(hostapi.ConvertError) as e:
            hostapi.convert(src, str(dst), backend=be, **kw)
        assert e.value.code == code, (k, e.value)
        assert not dst.exists() and not os.path.exists(str(dst) + ".partial")
    del keep


# ---------------------------------------------------------------- CPU: the batched path, with an overflow where we want one

class SetBackend:
    """The oracle's stage calls plus load_fs_profile_set / fs_set_scores as a CPU loop over them (one profile at a time).  The
    sequence of the chosen window of the chosen model (its content, whoever scores it later) is reported as overflowing in the
    3-codon simulation: by fs_set_scores and by fs_fwd_windows alike, so that bathhost_calibrate sees the same overflow."""
    SetLoad = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.POINTER(C.c_float)),
                          C.POINTER(C.POINTER(C.c_float)))
    SetScores = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_int32))
    Upload = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_uint8), C.c_int64)
    FwdWindows = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_int32))
    LoadFs = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float))
    FwdMatrices = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float),
                              C.c_int64, C.POINTER(C.c_float), C.POINTER(C.c_int32))

    def __init__(self, oracle, inject=None):
        from bath_b200 import capi
        self.capi = capi
        self.be, self.keep = oracle.cpu_backend(4)
        self.inject = inject                       # (model, window) of a batch's 3-codon simulation, or None
        self.target = None                         # the nucleotides of that window once seen
        self.block = None
        self.sets = {}
        self.orig_upload = self.Upload(self.be.upload_block)
        self.orig_fwd = self.FwdWindows(self.be.fs_fwd_windows)
        self.orig_load = self.LoadFs(self.be.load_fs_profile)
        self.orig_mx = self.FwdMatrices(self.be.fs_forward_matrices)
        self.cb = [self.Upload(self._upload), self.FwdWindows(self._fwd), self.SetLoad(self._set_load), self.SetScores(self._set_scores)]
        for name, f in zip(("upload_block", "fs_fwd_windows", "load_fs_profile_set", "fs_set_scores"), self.cb):
            setattr(self.be, name, C.cast(f, C.c_void_p))

    def _upload(self, ctx, dsq, n):
        self.block = np.ctypeslib.as_array(dsq, shape=(n + 2,)).copy()
        return self.orig_upload(ctx, dsq, n)

    def _seq(self, start, L):
        return self.block[start:start + L].tobytes()

    def _fwd(self, ctx, wins, n, xfE, sc, st):
        r = self.orig_fwd(ctx, wins, n, xfE, sc, st)
        w = np.ctypeslib.as_array(C.cast(wins, C.POINTER(C.c_uint8)), shape=(n * self.capi.window_dtype.itemsize,)).view(self.capi.window_dtype)
        for z in range(n):
            if self.target is not None and self._seq(int(w["start"][z]), int(w["L"][z])) == self.target:
                st[z] = 16
        return r

    def _set_load(self, ctx, which, n, M, nrows, rfv, tfv):
        self.sets[which] = [(np.ctypeslib.as_array(rfv[p], shape=(nrows[p] * (M[p] + 1),)).copy(),
                             np.ctypeslib.as_array(tfv[p], shape=(8 * (M[p] + 1),)).copy(), M[p], nrows[p]) for p in range(n)]
        return 0

    def _set_scores(self, ctx, which, wins, n, xfE, sc, st):
        capi = self.capi
        w = np.ctypeslib.as_array(C.cast(wins, C.POINTER(C.c_uint8)), shape=(n * capi.set_window_dtype.itemsize,)).view(capi.set_window_dtype)
        fp = C.POINTER(C.c_float)
        for p in np.unique(w["profile"]):
            rfv, tfv, M, nrows = self.sets[which][p]
            if self.orig_load(ctx, which, M, nrows, rfv.ctypes.data_as(fp), tfv.ctypes.data_as(fp)) != 0:
                return 11
            idx = np.nonzero(w["profile"] == p)[0]
            sub = np.zeros(len(idx), capi.window_dtype)
            for f in ("start", "L", "pmove", "ploop"):
                sub[f] = w[f][idx]
            s_, t_ = np.zeros(len(idx), np.float32), np.zeros(len(idx), np.int32)
            xf = np.array([xfE[2 * p], xfE[2 * p + 1]], np.float32)
            if which == 3:
                r = self.orig_fwd(ctx, sub.ctypes.data, len(idx), xf.ctypes.data_as(fp), s_.ctypes.data_as(fp), t_.ctypes.data_as(C.POINTER(C.c_int32)))
            else:
                r = self.orig_mx(ctx, sub.ctypes.data, len(idx), xf.ctypes.data_as(fp), None, None, 0, s_.ctypes.data_as(fp),
                                 t_.ctypes.data_as(C.POINTER(C.c_int32)))
            if r != 0:
                return r
            if which == 3 and self.inject is not None and self.target is None and p == self.inject[0]:
                z = idx[self.inject[1]]
                self.target = self._seq(int(w["start"][z]), int(w["L"][z]))
            for k, z in enumerate(idx):
                sc[z], st[z] = s_[k], t_[k]
                if which == 3 and self.target is not None and self._seq(int(w["start"][z]), int(w["L"][z])) == self.target:
                    st[z] = 16
        return 0


def test_convert_batched_path_falls_back_at_an_overflow_cpu(oracle, tmp_path):
    from bath_b200 import hostapi
    name, count = "tRNA-proteins.bhmm", 12
    src = write_hmmer3(tmp_path, name)

    plain = SetBackend(oracle)
    assert hostapi.convert(src, str(tmp_path / "plain.bhmm"), backend=plain.be) == count
    got_plain = open(tmp_path / "plain.bhmm").read()
    ref, keep = oracle.cpu_backend(4)
    check_against_shipped(name, got_plain, loop_lines(name, count, backend=ref))
    del keep

    hit = SetBackend(oracle, inject=(5, 17))
    assert hostapi.convert(src, str(tmp_path / "hit.bhmm"), backend=hit.be) == count
    assert hit.target is not None
    got = open(tmp_path / "hit.bhmm").read()
    # the serial chain over the same stage calls: bathhost_calibrate sees the overflow of that sequence and draws one more
    serial = SetBackend(oracle)
    serial.target = hit.target
    assert fs_lines(got) == loop_lines(name, count, backend=serial.be)
    # models before 5 are untouched; model 5 and the models after it (whose draws moved on by one sequence) are not
    a, b = fs_lines(got), fs_lines(got_plain)
    assert a[:10] == b[:10]
    assert a[10:12] != b[10:12]
    assert all(a[2 * m:2 * m + 2] != b[2 * m:2 * m + 2] for m in range(6, 12)), "the overflow must shift the draws of every later model"


# ---------------------------------------------------------------- GPU: the set calls against the single-profile calls

def all_models():
    from bath_b200 import hostapi
    out = []
    for f in sorted(os.listdir(common.GOLDEN)):
        if f.endswith(".bhmm") and not f.startswith("synthetic_"):
            out += [hostapi.QueryModel(common.golden(f), i) for i in range(hostapi.load().bathhost_model_count(os.fsencode(common.golden(f))))]
    out += [hostapi.QueryModel(common.golden(f)) for f in ("synthetic_M624.bhmm", "synthetic_M903.bhmm")]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("which", [3, 5])
def test_fs_set_scores_match_single_profile_calls(gpu_ctx, which):
    from bath_b200 import capi
    models = all_models()
    rng = np.random.default_rng(11 + which)
    dsq = common.random_dna(rng, 400_000, p_degenerate=0.002)
    gpu_ctx.select_slot(0)
    gpu_ctx.upload_block(dsq)
    nper = rng.integers(2, 7, len(models))
    prof = rng.permutation(np.repeat(np.arange(len(models)), nper))               # profiles interleaved
    lengths = rng.integers(6, 1500, len(prof))
    lengths[::7] = rng.integers(6, 40, len(lengths[::7]))                          # ragged, some very short
    starts = rng.integers(1, 400_000 - lengths + 2)
    xfE = np.array([(0.5, 0.5) if p % 2 == 0 else (1.0, 0.0) for p in range(len(models))], np.float32)
    gpu_ctx.load_fs_profile_set(which, [(m.rfv(which), m.tfv(which)) for m in models])
    wins = capi.Context.make_set_windows(starts, lengths, prof)
    sc, st = gpu_ctx.fs_set_scores(which, wins, xfE)
    for p, m in enumerate(models):
        idx = np.nonzero(prof == p)[0]
        gpu_ctx.load_fs_profile(which, m.rfv(which), m.tfv(which))
        one = capi.Context.make_windows(starts[idx], lengths[idx])
        if which == 3:
            s1, t1 = gpu_ctx.fs_fwd_windows(one, tuple(xfE[p]))
        else:
            s1, t1 = np.empty(len(idx), np.float32), np.empty(len(idx), np.int32)
            xf = np.ascontiguousarray(xfE[p])
            fp = C.POINTER(C.c_float)
            gpu_ctx._check(gpu_ctx.lib.bathgpu_fs_forward_matrices(gpu_ctx.h, one.ctypes.data, len(idx), xf.ctypes.data_as(fp), None, None, 0,
                                                                    s1.ctypes.data_as(fp), t1.ctypes.data_as(C.POINTER(C.c_int32))))
        assert np.array_equal(st[idx], t1), (m.name, st[idx], t1)
        ok = t1 == 0
        assert np.array_equal(sc[idx][ok].view(np.uint32), s1[ok].view(np.uint32)), (m.name, which, sc[idx], s1)


@pytest.mark.gpu
@pytest.mark.parametrize("name,count,ct", CONVERTED)
def test_convert_reproduces_shipped_files_gpu(gpu_ctx, tmp_path, name, count, ct):
    from bath_b200 import hostapi
    src, dst = write_hmmer3(tmp_path, name), str(tmp_path / "out.bhmm")
    assert hostapi.convert(src, dst, gpu_ctx=gpu_ctx, ct=ct) == count
    check_against_shipped(name, open(dst).read(), loop_lines(name, count, gpu_ctx=gpu_ctx))
