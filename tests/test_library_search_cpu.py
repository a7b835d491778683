"""A profile library against one target (bathhost_search_create_library, hostapi.LibrarySearch) on the CPU stage calls: every model's
table, counters and output must be those of a standalone Search of that model, whether the ORF screen runs model by model (the
backend's set entries NULL) or as one set call per unit (the oracle's stand-in, a loop over the single-profile screen), on one
context or several, and with chunks small enough to hold several blocks whose contexts differ from model to model."""
import ctypes as C

import numpy as np
import pytest

import common

COUNTERS = ("nseqs", "nres", "pos_past_msv", "pos_past_bias", "pos_past_vit", "pos_past_fwd", "n_orfs", "n_windows", "n_std_windows",
            "n_regions", "n_multidomain_regions", "n_envelopes", "n_hits_reported")


def _genome(path, seed):
    from bath_b200 import hostapi, synth
    model = hostapi.QueryModel(common.golden(path), 0)
    rng = np.random.default_rng(seed)
    out = []
    for c in range(2):
        dsq, _ = synth.planted_genome(rng, 90_000, model.mat(), every=15_000, fs_rate=model.fsprob)
        out.append((f"contig{c + 1}", dsq))
    return out


def _standalone(oracle, path, targets, **opt):
    from bath_b200 import hostapi
    out = []
    for i in range(hostapi.load().bathhost_model_count(common.golden(path).encode())):
        be, keep = oracle.cpu_backend(2)
        s = hostapi.Search(hostapi.QueryModel(common.golden(path), i), backend=be, **opt)
        for name, dsq in targets:
            s.queue_sequence(name, dsq)
        s.finish(fetch=False)
        out.append((s.tblout(), {k: s.stats()[k] for k in COUNTERS}, s.output()))
        s.close()
        del keep
    return out


class SetScreenStandIn:
    """The backend's set trio (load_filter_profile_set, orfs_msv_screen_set, orfs_fetch_set) on the CPU oracle, as a loop over its
    single-profile screen: job j loads its model's profiles into the oracle context and runs bo_backend_orfs_msv_screen; the survivors of
    all jobs are concatenated (offsets shifted by the residues of the jobs before) and their residues uploaded as the slot's buffer, which
    is the layout the device call leaves.  The set loader's rbv pointers name the models (they are the models' own tables)."""

    _load_t = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_void_p))
    _screen_t = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                            C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64))
    _fetch_t = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p)

    class Job(C.Structure):
        _fields_ = [("profile", C.c_int32), ("nblocks", C.c_int32), ("blocks", C.c_void_p), ("min_bits", C.c_double)]

    def __init__(self, oracle, models):
        from bath_b200 import capi, hostapi
        self.H = hostapi.load()
        # the oracle's entry points with prototypes of their own (other tests may set argtypes on the shared library's functions)
        L, vp = oracle.lib(), C.c_void_p
        proto = {"load_fs_profile": (C.c_int, vp, C.c_int, C.c_int, C.c_int, vp, vp), "load_filter_profile": (C.c_int, vp, vp, vp, vp, vp),
                 "orfs_msv_screen": (C.c_int, vp, vp, C.c_int, C.c_int, vp, C.c_int, vp, vp, C.c_int, C.c_double, vp, vp, vp),
                 "orfs_fetch": (C.c_int, vp, vp, vp), "upload_orfs": (C.c_int, vp, vp, C.c_int64)}
        self.bo = {n: C.CFUNCTYPE(*t)(C.cast(getattr(L, "bo_backend_" + n), vp).value) for n, t in proto.items()}
        self.hit_dtype = capi.orf_hit_dtype
        self.by_rbv = {C.cast(self.H.bathhost_model_rbv(m.h), C.c_void_p).value: m for m in models}
        self.sets, self.out, self.calls = {}, {}, 0
        self.cb = (self._load_t(self.load), self._screen_t(self.screen), self._fetch_t(self.fetch))

    def install(self, be):
        be.load_filter_profile_set, be.orfs_msv_screen_set, be.orfs_fetch_set = [C.cast(f, C.c_void_p) for f in self.cb]

    def load(self, ctx, n, prm, rbv):
        size = C.sizeof(C.c_int32) * 13
        self.sets[ctx] = [(self.by_rbv[rbv[k]], prm + k * size) for k in range(n)]
        return 0

    def screen(self, ctx, jobs, njobs, complement, gcode, min_len, tjb, null, max_len, norfs, nhits, nres):
        H, bo, vp = self.H, self.bo, C.c_void_p
        self.calls += 1
        jobs = C.cast(jobs, C.POINTER(self.Job))
        hits, res, ob = [], [], 0
        for j in range(njobs):
            m, prm = self.sets[ctx][jobs[j].profile]
            for which in (3, 5):
                st = bo["load_fs_profile"](ctx, which, m.M, H.bathhost_model_nrows(m.h, which), C.cast(H.bathhost_model_rfv(m.h, which), vp),
                                           C.cast(H.bathhost_model_tfv(m.h, which), vp))
                assert st == 0
            assert bo["load_filter_profile"](ctx, prm, C.cast(H.bathhost_model_rbv(m.h), vp), C.cast(H.bathhost_model_rwv(m.h), vp),
                                             C.cast(H.bathhost_model_twv(m.h), vp)) == 0
            h, r = C.c_int64(0), C.c_int64(0)
            st = bo["orfs_msv_screen"](ctx, jobs[j].blocks, jobs[j].nblocks, complement, gcode, min_len, tjb, null, max_len, jobs[j].min_bits,
                                       C.addressof(norfs.contents) + 8 * ob, C.addressof(h), C.addressof(r))
            if st != 0:
                return st
            hj, rj = np.zeros(max(h.value, 1), self.hit_dtype), np.zeros(max(r.value, 1), np.uint8)
            bo["orfs_fetch"](ctx, hj.ctypes.data, rj.ctypes.data)
            hj, rj = hj[: h.value], rj[: r.value]
            hj["offset"] += sum(len(x) for x in res)
            hits.append(hj); res.append(rj)
            nhits[j], nres[j] = h.value, r.value
            ob += jobs[j].nblocks
        all_h, all_r = np.concatenate(hits), np.concatenate(res)
        if len(all_r):
            bo["upload_orfs"](ctx, all_r.ctypes.data, len(all_r))
        self.out[ctx] = (all_h, all_r)
        return 0

    def fetch(self, ctx, hits, residues):
        h, r = self.out[ctx]
        if len(h):
            C.memmove(hits, h.ctypes.data, h.nbytes)
            C.memmove(residues, r.ctypes.data, r.nbytes)
        return 0


def _library(oracle, path, targets, nbackends, set_screen, **opt):
    from bath_b200 import hostapi
    pairs = [oracle.cpu_backend(2) for _ in range(nbackends)]
    models = [hostapi.QueryModel(common.golden(path), i) for i in range(hostapi.load().bathhost_model_count(common.golden(path).encode()))]
    standin = SetScreenStandIn(oracle, models)
    if set_screen:
        for be, _ in pairs:
            standin.install(be)
    lib = hostapi.LibrarySearch(models, backend=[p[0] for p in pairs], **opt)
    for name, dsq in targets:
        lib.queue_sequence(name, dsq)
    lib.finish()
    per = [(s.tblout(), {k: s.stats()[k] for k in COUNTERS}, s.output()) for s in lib.searches]
    whole = (lib.tblout(), lib.output())
    lib.close()
    assert (standin.calls > 0) == set_screen
    del pairs
    return per, whole


@pytest.mark.parametrize("path", ["tRNA-proteins.bhmm", "tRNA-synthetases.bhmm"])
@pytest.mark.parametrize("opt", [{}, {"std_only": 1}])
def test_library_equals_standalone_searches(oracle, path, opt):
    targets = _genome(path, 7)
    opt = dict(opt, block_length=20_000)
    ref = _standalone(oracle, path, targets, **opt)
    assert sum(r[1]["n_hits_reported"] for r in ref) > 0
    for nbackends, chunk_nt, set_screen in ((1, 0, False), (1, 0, True), (3, 45_000, False), (3, 45_000, True)):
        per, whole = _library(oracle, path, targets, nbackends, set_screen, chunk_nt=chunk_nt, **opt)
        assert len(per) == len(ref)
        for i, (a, b) in enumerate(zip(per, ref)):
            assert a[0] == b[0], (nbackends, set_screen, i)
            assert a[1] == b[1], (nbackends, set_screen, i)
            assert a[2] == b[2], (nbackends, set_screen, i)
        head = ref[0][0].splitlines(keepends=True)
        header = "".join(l for l in head if l.startswith("#"))
        rows = "".join("".join(l for l in r[0].splitlines(keepends=True) if not l.startswith("#")) for r in ref)
        assert whole[0] == header + rows
        assert whole[1] == "".join(r[2] + "//\n" for r in ref)


def test_library_refuses_a_model_longer_than_the_contexts_accept(oracle):
    """a backend whose profile loader refuses one model's length: creation fails with that status and a message naming the model, and
    no target is ever uploaded"""
    from bath_b200 import hostapi
    be, keep = oracle.cpu_backend(1)
    L = oracle.lib()
    lengths = [hostapi.QueryModel(common.golden("tRNA-proteins.bhmm"), i).M for i in range(12)]
    limit = sorted(lengths)[-1] - 1                       # the longest model is "too long"
    longest = lengths.index(max(lengths))
    load_t = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p)
    upload_t = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int64)
    real_load = load_t(C.cast(getattr(L, "bo_backend_load_fs_profile"), C.c_void_p).value)
    uploads = []

    def load(ctx, which, M, nrows, rfv, tfv):
        return 11 if M > limit else real_load(ctx, which, M, nrows, rfv, tfv)

    def upload(ctx, dsq, n):
        uploads.append(n)
        return 11

    cb_load, cb_upload = load_t(load), upload_t(upload)
    be.load_fs_profile = C.cast(cb_load, C.c_void_p)
    be.upload_block = C.cast(cb_upload, C.c_void_p)
    with pytest.raises(hostapi.LibraryError) as e:
        hostapi.LibrarySearch(common.golden("tRNA-proteins.bhmm"), backend=be)
    assert e.value.code == 11
    assert f"model {longest} " in str(e.value)
    assert uploads == []
    del keep
