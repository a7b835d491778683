"""ctypes binding of libbathhost.so (include/bathhost.h): the host side of the path."""
import ctypes as C
import os

import numpy as np

from .build import host_library_path

OK = 0
EXPORTS = [
    "bathhost_model_read", "bathhost_model_count", "bathhost_model_destroy", "bathhost_model_get_info",
    "bathhost_model_nrows", "bathhost_model_rfv", "bathhost_model_tfv", "bathhost_model_codons",
    "bathhost_model_indel_pos", "bathhost_model_mat", "bathhost_model_consensus", "bathhost_length_model",
    "bathhost_model_filter_params", "bathhost_model_rbv", "bathhost_model_rwv", "bathhost_model_twv",
    "bathhost_orf_length_params", "bathhost_model_computed_max_length",
    "bathhost_search_create", "bathhost_search_create_multi", "bathhost_search_queue", "bathhost_search_run", "bathhost_search_destroy", "bathhost_search_last_error", "bathhost_search_sequence",
    "bathhost_search_finish", "bathhost_search_finish_many", "bathhost_search_nhits", "bathhost_search_get_hit", "bathhost_search_get_stats",
    "bathhost_sample_region_segments", "bathhost_cluster_region_segments", "bathhost_sample_region_segments_protein",
    "bathhost_cluster_region_segments_protein", "bathhost_search_format_tblout",
    "bathhost_calibrate", "bathhost_model_lambda", "bathhost_search_format_report", "bathhost_search_format_output", "bathhost_search_format_fstblout",
    "bathhost_convert", "bathhost_convert_last_error",
]


class ModelInfo(C.Structure):
    _fields_ = [("M", C.c_int32), ("max_length", C.c_int32), ("codon_table", C.c_int32), ("fsprob", C.c_float),
                ("evparam", C.c_float * 8), ("has_fs3_stats", C.c_int32), ("has_fs5_stats", C.c_int32),
                ("name", C.c_char * 128), ("acc", C.c_char * 64)]


class FilterParams(C.Structure):
    _fields_ = [("M", C.c_int32), ("tbm_b", C.c_int32), ("tec_b", C.c_int32), ("base_b", C.c_int32), ("bias_b", C.c_int32),
                ("scale_b", C.c_float), ("base_w", C.c_int32), ("ddbound_w", C.c_int32), ("xw_E_move", C.c_int32),
                ("xw_E_loop", C.c_int32), ("scale_w", C.c_float)]


class Backend(C.Structure):
    """bathhost_backend: the device library as a table of function pointers (include/bathhost.h)"""
    _names = ["last_error", "load_fs_profile", "load_filter_profile", "select_slot", "upload_block", "upload_orfs", "msv_orfs", "ssv_windows",
              "vit_orfs", "fwd_orfs", "fs_fwd_windows", "fs_fwd_bck_xrows", "fs_bck_decode", "fs_domains", "fs_forward_matrices", "orf_fwd_bck_xrows", "orf_domains", "orfs_msv_screen", "orfs_fetch", "revcomp_slot", "host_alloc", "host_free", "bias_forward", "orf_forward_matrices", "upload_block_segments"]
    # the optional pair at the end of the table: left NULL by a table that fills _names only (bathhost_convert then calibrates
    # model by model)
    _set_names = ["load_fs_profile_set", "fs_set_scores"]
    _fields_ = [("ctx", C.c_void_p)] + [(n, C.c_void_p) for n in _names + _set_names]


class Options(C.Structure):
    _fields_ = [("F1", C.c_double), ("F2", C.c_double), ("F3", C.c_double), ("F4", C.c_double), ("E", C.c_double),
                ("min_orf_len", C.c_int32), ("block_length", C.c_int32), ("cpu_lanes_u8", C.c_int32), ("cpu_lanes_i16", C.c_int32),
                ("no_bias", C.c_int32), ("no_null2", C.c_int32), ("top_only", C.c_int32), ("bottom_only", C.c_int32), ("std_only", C.c_int32),
                ("show_frameline", C.c_int32), ("reserved0", C.c_int32), ("chunk_nt", C.c_int64)]


class Hit(C.Structure):
    _fields_ = [("seqidx", C.c_int64), ("name", C.c_char * 64), ("strand", C.c_int32),
                ("ali_from", C.c_int64), ("ali_to", C.c_int64), ("env_from", C.c_int64), ("env_to", C.c_int64), ("sq_len", C.c_int64),
                ("hmm_from", C.c_int32), ("hmm_to", C.c_int32), ("evalue", C.c_double), ("lnP", C.c_double),
                ("score", C.c_float), ("bias", C.c_float), ("pre_score", C.c_float), ("envsc", C.c_float), ("oasc", C.c_float),
                ("pid", C.c_float), ("shifts", C.c_int32), ("stops", C.c_int32), ("trace_len", C.c_int32), ("cigar", C.c_char * 1024)]


class Stats(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("nseqs", "nres", "pos_past_msv", "pos_past_bias", "pos_past_vit", "pos_past_fwd", "n_orfs",
                                         "n_windows", "n_std_windows", "n_regions", "n_multidomain_regions", "n_envelopes",
                                         "n_hits_reported", "us_orfs", "us_upload", "us_msv", "us_bias", "us_vit", "us_fwd",
                                         "us_windows", "us_fs_fwd", "us_fs_domains", "us_std", "us_xrows", "us_decode", "us_score")]


class Segment(C.Structure):
    _fields_ = [("idx", C.c_int32), ("i", C.c_int32), ("j", C.c_int32), ("k", C.c_int32), ("m", C.c_int32), ("prob", C.c_float)]


_lib = None


class Calibration(C.Structure):
    """bathhost_calibration (include/bathhost.h)"""
    _fields_ = [("seed", C.c_uint32), ("rng_state", C.c_uint32), ("convert_flow", C.c_int32), ("which_mask", C.c_int32),
                ("lambda_", C.c_double)]


def load():
    global _lib
    if _lib is not None:
        return _lib
    path = host_library_path()
    if not os.path.exists(path):
        raise ImportError(f"{path} is missing: build it with `python -m bath_b200.build`")
    L = C.CDLL(path)
    vp, fp, u8p = C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_uint8)
    L.bathhost_model_read.restype = C.c_int
    L.bathhost_model_read.argtypes = [C.c_char_p, C.c_int, C.c_int, C.POINTER(vp)]
    L.bathhost_sample_region_segments.restype = C.c_int
    L.bathhost_sample_region_segments.argtypes = [fp, fp, C.c_int, C.c_int, fp, fp, C.c_uint32, C.c_int, C.c_int, C.POINTER(Segment), C.c_int,
                                                  C.POINTER(C.c_int)]
    L.bathhost_cluster_region_segments.restype = C.c_int
    L.bathhost_cluster_region_segments.argtypes = [C.POINTER(Segment), C.c_int, C.c_int, C.POINTER(Segment), C.c_int, C.POINTER(C.c_int)]
    L.bathhost_model_count.restype = C.c_int
    L.bathhost_model_count.argtypes = [C.c_char_p]
    L.bathhost_model_destroy.restype = None
    L.bathhost_model_destroy.argtypes = [vp]
    L.bathhost_model_get_info.restype = C.c_int
    L.bathhost_model_get_info.argtypes = [vp, C.POINTER(ModelInfo)]
    L.bathhost_model_nrows.restype = C.c_int
    L.bathhost_model_nrows.argtypes = [vp, C.c_int]
    for name, res in (("bathhost_model_rfv", fp), ("bathhost_model_tfv", fp), ("bathhost_model_codons", u8p),
                      ("bathhost_model_indel_pos", u8p)):
        f = getattr(L, name)
        f.restype, f.argtypes = res, [vp, C.c_int]
    L.bathhost_model_mat.restype = fp
    L.bathhost_model_mat.argtypes = [vp]
    L.bathhost_model_consensus.restype = C.c_char_p
    L.bathhost_model_consensus.argtypes = [vp]
    L.bathhost_model_filter_params.restype = C.c_int
    L.bathhost_model_filter_params.argtypes = [vp, C.POINTER(FilterParams)]
    L.bathhost_model_rbv.restype = u8p
    L.bathhost_model_rbv.argtypes = [vp]
    L.bathhost_model_rwv.restype = C.POINTER(C.c_int16)
    L.bathhost_model_rwv.argtypes = [vp]
    L.bathhost_model_twv.restype = C.POINTER(C.c_int16)
    L.bathhost_model_twv.argtypes = [vp]
    L.bathhost_orf_length_params.restype = None
    L.bathhost_orf_length_params.argtypes = [vp, C.c_int, C.POINTER(C.c_uint8), C.POINTER(C.c_int16)]
    L.bathhost_search_create.restype = C.c_int
    L.bathhost_search_create.argtypes = [vp, C.POINTER(Backend), C.POINTER(Options), C.POINTER(vp)]
    L.bathhost_search_create_multi.restype = C.c_int
    L.bathhost_search_create_multi.argtypes = [vp, C.POINTER(Backend), C.c_int, C.POINTER(Options), C.POINTER(vp)]
    L.bathhost_search_queue.restype = C.c_int
    L.bathhost_search_queue.argtypes = [vp, C.c_char_p, u8p, C.c_int64]
    L.bathhost_search_run.restype = C.c_int
    L.bathhost_search_run.argtypes = [vp]
    L.bathhost_search_destroy.restype = None
    L.bathhost_search_destroy.argtypes = [vp]
    L.bathhost_search_last_error.restype = C.c_char_p
    L.bathhost_search_last_error.argtypes = [vp]
    L.bathhost_search_sequence.restype = C.c_int
    L.bathhost_search_sequence.argtypes = [vp, C.c_char_p, u8p, C.c_int64]
    L.bathhost_search_finish.restype = C.c_int
    L.bathhost_search_finish.argtypes = [vp]
    L.bathhost_search_finish_many.restype = C.c_int
    L.bathhost_search_finish_many.argtypes = [C.POINTER(C.c_void_p), C.c_int]
    L.bathhost_search_nhits.restype = C.c_int
    L.bathhost_search_nhits.argtypes = [vp]
    L.bathhost_search_get_hit.restype = C.c_int
    L.bathhost_search_get_hit.argtypes = [vp, C.c_int, C.POINTER(Hit)]
    L.bathhost_search_get_stats.restype = C.c_int
    L.bathhost_search_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.bathhost_model_computed_max_length.restype = C.c_int
    L.bathhost_model_computed_max_length.argtypes = [vp]
    L.bathhost_calibrate.restype = C.c_int
    L.bathhost_calibrate.argtypes = [vp, C.POINTER(Backend), C.POINTER(Calibration), C.POINTER(C.c_double)]
    L.bathhost_model_lambda.restype = C.c_double
    L.bathhost_model_lambda.argtypes = [vp]
    L.bathhost_convert.restype = C.c_int
    L.bathhost_convert.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_float, C.c_uint32, C.POINTER(Backend), C.POINTER(C.c_int)]
    L.bathhost_convert_last_error.restype = C.c_char_p
    L.bathhost_convert_last_error.argtypes = []
    L.bathhost_length_model.restype = None
    L.bathhost_length_model.argtypes = [C.c_int, C.c_float, fp, fp]
    _lib = L
    return L


class QueryModel:
    """One query profile set up as bathsearch does (src/bathsearch.c:794-801): local mode,
    3- and 5-codon-length frameshift profiles in odds-ratio form."""

    def __init__(self, path, index=0, ct=0):
        self.lib = load()
        h = C.c_void_p()
        st = self.lib.bathhost_model_read(os.fsencode(path), index, ct, C.byref(h))
        if st != OK:
            raise IOError(f"cannot read model {index} of {path}: status {st}")
        self.h = h
        info = ModelInfo()
        self.lib.bathhost_model_get_info(h, C.byref(info))
        self.M = info.M
        self.max_length = info.max_length
        self.fsprob = info.fsprob
        self.codon_table = info.codon_table
        self.evparam = list(info.evparam)
        self.name = info.name.decode()

    def close(self):
        if getattr(self, "h", None):
            self.lib.bathhost_model_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def nrows(self, which=3):
        return self.lib.bathhost_model_nrows(self.h, which)

    def rfv(self, which=3):
        return np.ctypeslib.as_array(self.lib.bathhost_model_rfv(self.h, which), shape=(self.nrows(which), self.M + 1))

    def tfv(self, which=3):
        return np.ctypeslib.as_array(self.lib.bathhost_model_tfv(self.h, which), shape=(8, self.M + 1))

    def codons(self, which=3):
        mc = self.nrows(which) - 29
        flat = np.ctypeslib.as_array(self.lib.bathhost_model_codons(self.h, which), shape=((self.M + 1) * (mc + 1),))
        return flat[: (self.M + 1) * mc].reshape(self.M + 1, mc)

    def indel_pos(self, which=3):
        mc = self.nrows(which) - 29
        flat = np.ctypeslib.as_array(self.lib.bathhost_model_indel_pos(self.h, which), shape=((self.M + 1) * (mc + 1),))
        return flat[: (self.M + 1) * mc].reshape(self.M + 1, mc)

    def filter_params(self, cpu_lanes_u8=16, cpu_lanes_i16=8):
        """dict in the shape capi.Context.load_filter_profile takes"""
        p = FilterParams()
        self.lib.bathhost_model_filter_params(self.h, C.byref(p))
        d = {name: getattr(p, name) for name, _ in FilterParams._fields_}
        d.update(cpu_lanes_u8=cpu_lanes_u8, cpu_lanes_i16=cpu_lanes_i16)
        return d

    def filter_tables(self):
        M = self.M
        return (np.ctypeslib.as_array(self.lib.bathhost_model_rbv(self.h), shape=(29, M + 1)),
                np.ctypeslib.as_array(self.lib.bathhost_model_rwv(self.h), shape=(29, M + 1)),
                np.ctypeslib.as_array(self.lib.bathhost_model_twv(self.h), shape=(8, M + 1)))

    def orf_length_params(self, L):
        a, b = C.c_uint8(), C.c_int16()
        self.lib.bathhost_orf_length_params(self.h, int(L), C.byref(a), C.byref(b))
        return a.value, b.value

    def mat(self):
        return np.ctypeslib.as_array(self.lib.bathhost_model_mat(self.h), shape=(self.M + 1, 20))


def length_model(L_amino, nj=1.0):
    pm, pl = C.c_float(), C.c_float()
    load().bathhost_length_model(int(L_amino), float(nj), C.byref(pm), C.byref(pl))
    return pm.value, pl.value


_DNA = {c: i for i, c in enumerate("ACGT-RYMKSWHBVDN*~")}


def digitize_dna(seq):
    """Easel digital DNA: codes at [1..L], sentinel 255 at [0] and [L+1]"""
    s = seq.upper().replace("U", "T").replace("X", "N")
    a = np.full(len(s) + 2, 255, dtype=np.uint8)
    a[1:-1] = [_DNA[c] for c in s]
    return a


def read_fasta(path):
    out, name, buf = [], None, []
    with open(path) as fh:
        for line in fh:
            line = line.rstrip("\n")
            if line.startswith(">"):
                if name is not None:
                    out.append((name, "".join(buf)))
                name, buf = line[1:].split(None, 1)[0], []
            else:
                buf.append(line.strip())
    if name is not None:
        out.append((name, "".join(buf)))
    return out


def backend_from(gpu_lib, ctx_handle):
    """bathhost_backend over a loaded libbathgpu.so (ctypes CDLL) and a bathgpu_ctx handle"""
    be = Backend()
    be.ctx = ctx_handle
    for n in Backend._names + Backend._set_names:
        setattr(be, n, C.cast(getattr(gpu_lib, "bathgpu_" + n), C.c_void_p))
    return be


def calibrate(model, gpu_ctx=None, backend=None, seed=42, lam=0.0, which=31, convert_flow=False, rng_state=0):
    """E-value parameters of a model by simulation on the device (p7_Calibrate with the frameshift branch, or bathconvert's
    frameshift-only flow): returns (evparam[8], generator state).  See bathhost_calibrate in include/bathhost.h."""
    lib = load()
    if backend is None:
        if gpu_ctx is None:
            raise ValueError("a device context is required: the product has no CPU path")
        backend = backend_from(gpu_ctx.lib, gpu_ctx.h)
    cal = Calibration(seed, rng_state, int(convert_flow), which, float(lam))
    out = (C.c_double * 8)()
    st = lib.bathhost_calibrate(model.h, C.byref(backend), C.byref(cal), out)
    if st != OK:
        raise RuntimeError(f"bathhost_calibrate: status {st}")
    return [float(v) for v in out], int(cal.rng_state)


class ConvertError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"bathhost_convert: status {code}: {msg}")
        self.code = code


def convert(in_path, out_path, gpu_ctx=None, backend=None, ct=1, fsprob=0.01, seed=42):
    """A HMMER3/f profile library (hmmbuild output, any number of models) as a BATH3/f one that bathsearch reads: each model's
    text with the FS3 / FS5 Forward taus bathconvert's calibration gives, FRAMESHIFT PROB and CODON TABLE added (see bathhost_convert
    in include/bathhost.h).  Returns the number of models; raises ConvertError (code EFORMAT = 7 for input that is not HMMER3/f,
    EINVAL = 11 for ct / fsprob) and leaves out_path unwritten on failure."""
    lib = load()
    if backend is None:
        if gpu_ctx is None:
            raise ValueError("a device context is required: the product has no CPU path")
        backend = backend_from(gpu_ctx.lib, gpu_ctx.h)
    n = C.c_int(0)
    st = lib.bathhost_convert(os.fsencode(in_path), os.fsencode(out_path), int(ct), float(fsprob), int(seed), C.byref(backend), C.byref(n))
    if st != OK:
        raise ConvertError(st, lib.bathhost_convert_last_error().decode())
    return int(n.value)


class Search:
    """One query against target sequences: the stage-batched pipeline of bathsearch --fs (pipeline.cpp)."""

    def __init__(self, model, gpu_ctx=None, backend=None, **options):
        """gpu_ctx: a capi.Context, or a list of them (several GPUs, or several contexts per GPU): the product path.
        backend: a ready bathhost_backend table (or a list of them) instead -- used by the tests and the CPU-baseline legs
        of bench.py to put the CPU oracle behind the same pipeline."""
        self.lib = load()
        self.model = model
        self.gpu_ctx = gpu_ctx                       # keeps the device context(s) alive
        if backend is None:
            if gpu_ctx is None:
                raise ValueError("a device context is required: the product has no CPU path")
            ctxs = gpu_ctx if isinstance(gpu_ctx, (list, tuple)) else [gpu_ctx]
            backend = [backend_from(c.lib, c.h) for c in ctxs]
        backends = list(backend) if isinstance(backend, (list, tuple)) else [backend]
        self.backend = (Backend * len(backends))(*backends)
        self._keep = []                              # queued target arrays: they must outlive bathhost_search_run
        opt = Options(**options)
        h = C.c_void_p()
        st = self.lib.bathhost_search_create_multi(model.h, self.backend, len(backends), C.byref(opt), C.byref(h))
        if st != OK:
            raise RuntimeError(f"bathhost_search_create_multi: status {st}")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.bathhost_search_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def add_sequence(self, name, dsq):
        dsq = np.ascontiguousarray(dsq, np.uint8)
        st = self.lib.bathhost_search_sequence(self.h, name.encode(), dsq.ctypes.data_as(C.POINTER(C.c_uint8)), len(dsq) - 2)
        if st != OK:
            raise RuntimeError(f"bathhost_search_sequence: status {st}: {self.lib.bathhost_search_last_error(self.h).decode()}")

    def queue_sequence(self, name, dsq):
        """one more target for the next run(): all queued sequences are searched in one stage-batched pass"""
        dsq = np.ascontiguousarray(dsq, np.uint8)
        self._keep.append(dsq)
        st = self.lib.bathhost_search_queue(self.h, name.encode(), dsq.ctypes.data_as(C.POINTER(C.c_uint8)), len(dsq) - 2)
        if st != OK:
            raise RuntimeError(f"bathhost_search_queue: status {st}")

    def run(self):
        st = self.lib.bathhost_search_run(self.h)
        self._keep = []
        if st != OK:
            raise RuntimeError(f"bathhost_search_run: status {st}: {self.lib.bathhost_search_last_error(self.h).decode()}")

    def finish(self, fetch=True):
        """bathhost_search_finish: everything still queued is searched, E-values, duplicate removal, ordering, thresholds.
        fetch=False returns the number of hits and leaves their conversion into Python dicts to hits() (a harness cost, ~10 us per hit)."""
        if self._keep:
            self.run()
        st = self.lib.bathhost_search_finish(self.h)
        if st != OK:
            raise RuntimeError(f"bathhost_search_finish: status {st}")
        return self.hits() if fetch else int(self.lib.bathhost_search_nhits(self.h))

    @staticmethod
    def finish_many(searches):
        """bathhost_search_finish_many: the searches (different profiles, device contexts of their own, targets already queued) run at
        the same time, one host thread each; every search ends up as after its own finish(fetch=False)"""
        if not searches:
            return
        arr = (C.c_void_p * len(searches))(*[s.h for s in searches])
        st = searches[0].lib.bathhost_search_finish_many(arr, len(searches))
        for s in searches:
            s._keep = []
        if st != OK:
            msgs = "; ".join(s.lib.bathhost_search_last_error(s.h).decode() for s in searches)
            raise RuntimeError(f"bathhost_search_finish_many: status {st}: {msgs}")

    def hits(self):
        hits = []
        for i in range(self.lib.bathhost_search_nhits(self.h)):
            h = Hit()
            self.lib.bathhost_search_get_hit(self.h, i, C.byref(h))
            hits.append({n: (getattr(h, n).decode() if isinstance(getattr(h, n), bytes) else getattr(h, n)) for n, _ in Hit._fields_})
        return hits

    def tblout(self, header=True):
        """the --tblout --cigar table of the reported hits (header + hit lines, no trailer), as bathsearch writes it"""
        need = C.c_size_t(0)
        self.lib.bathhost_search_format_tblout.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t)]
        self.lib.bathhost_search_format_tblout(self.h, int(header), None, 0, C.byref(need))
        buf = C.create_string_buffer(need.value)
        st = self.lib.bathhost_search_format_tblout(self.h, int(header), buf, need.value, C.byref(need))
        if st != OK:
            raise RuntimeError(f"bathhost_search_format_tblout: status {st}")
        return buf.value.decode()

    def fstblout(self, header=True):
        """the --fstblout table: one line per frameshift / stop codon of the reported frameshift-branch hits"""
        return self._format(self.lib.bathhost_search_format_fstblout, int(header))

    def output(self, textw=150):
        """one query's section of bathsearch's output from "Query:" to "Total number of hits:" (no banner, no timings)"""
        return self._format(self.lib.bathhost_search_format_output, textw)

    def report(self, textw=150):
        """the hit-dependent part of bathsearch's main output: "Scores for complete hits" table and the per-hit annotation with
        alignments (everything between the "Query:" block and the pipeline statistics), as bathsearch writes it"""
        return self._format(self.lib.bathhost_search_format_report, textw)

    def _format(self, f, textw):
        need = C.c_size_t(0)
        f.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t)]
        f(self.h, int(textw), None, 0, C.byref(need))
        buf = C.create_string_buffer(need.value)
        st = f(self.h, int(textw), buf, need.value, C.byref(need))
        if st != OK:
            raise RuntimeError(f"{f.__name__}: status {st}")
        return buf.value.decode()

    def stats(self):
        s = Stats()
        self.lib.bathhost_search_get_stats(self.h, C.byref(s))
        return {n: getattr(s, n) for n, _ in Stats._fields_}


def sample_region_segments(mx, xrows, tfv, odds, ireg, seed=42, nsamples=200):
    """bathhost_sample_region_segments on one region's Forward matrix mx [(L+1)][(M+1)][8], xrows [(L+1)][6]:
    list of (idx, i, j, k, m, prob), one per sampled domain"""
    import numpy as np
    L = load()
    mx = np.ascontiguousarray(mx, np.float32); xr = np.ascontiguousarray(xrows, np.float32)
    tf = np.ascontiguousarray(tfv, np.float32); od = np.ascontiguousarray(odds, np.float32)
    fp = C.POINTER(C.c_float)
    cap = nsamples * 64
    out = (Segment * cap)()
    n = C.c_int(0)
    st = L.bathhost_sample_region_segments(mx.ctypes.data_as(fp), xr.ctypes.data_as(fp), mx.shape[1] - 1, mx.shape[0] - 1, tf.ctypes.data_as(fp),
                                           od.ctypes.data_as(fp), seed, nsamples, ireg, out, cap, C.byref(n))
    if st != 0:
        raise RuntimeError(f"bathhost_sample_region_segments: status {st}")
    return [(g.idx, g.i, g.j, g.k, g.m, g.prob) for g in out[:n.value]]


def sample_region_segments_protein(mx, xrows, tfv, rf, odds, ireg, res, seed=42, nsamples=200):
    """bathhost_sample_region_segments_protein: (segments, n2sc[0..L]) for one region's protein Forward matrix mx [(L+1)][(M+1)][4]
    {M, D, I, 0}; res = the region's residues (length L); rf = amino-acid emission odds [29][M+1]"""
    import numpy as np
    L = load()
    mx = np.ascontiguousarray(mx, np.float32); xr = np.ascontiguousarray(xrows, np.float32)
    tf = np.ascontiguousarray(tfv, np.float32); od = np.ascontiguousarray(odds, np.float32); rfa = np.ascontiguousarray(rf, np.float32)
    r1 = np.concatenate([[255], np.asarray(res, np.uint8), [255]]).astype(np.uint8)
    fp = C.POINTER(C.c_float)
    cap = nsamples * 64
    out = (Segment * cap)()
    n = C.c_int(0)
    Lr = mx.shape[0] - 1
    n2 = np.zeros(Lr + 1, np.float32)
    f = L.bathhost_sample_region_segments_protein
    f.restype = C.c_int
    f.argtypes = [fp, fp, C.c_int, C.c_int, fp, fp, fp, C.c_uint32, C.c_int, C.c_int, C.POINTER(C.c_uint8), C.POINTER(Segment), C.c_int,
                  C.POINTER(C.c_int), fp]
    st = f(mx.ctypes.data_as(fp), xr.ctypes.data_as(fp), mx.shape[1] - 1, Lr, tf.ctypes.data_as(fp), rfa.ctypes.data_as(fp),
           od.ctypes.data_as(fp), seed, nsamples, ireg, r1.ctypes.data_as(C.POINTER(C.c_uint8)), out, cap, C.byref(n), n2.ctypes.data_as(fp))
    if st != 0:
        raise RuntimeError(f"bathhost_sample_region_segments_protein: status {st}")
    return [(g.idx, g.i, g.j, g.k, g.m, g.prob) for g in out[:n.value]], n2


def cluster_region_segments(segments, nsamples=200, protein=False):
    L = load()
    if protein:
        L.bathhost_cluster_region_segments_protein.restype = C.c_int
        L.bathhost_cluster_region_segments_protein.argtypes = L.bathhost_cluster_region_segments.argtypes
        sp = (Segment * max(1, len(segments)))(*[Segment(*g) for g in segments])
        out = (Segment * 64)()
        n = C.c_int(0)
        st = L.bathhost_cluster_region_segments_protein(sp, len(segments), nsamples, out, 64, C.byref(n))
        if st != 0:
            raise RuntimeError(f"bathhost_cluster_region_segments_protein: status {st}")
        return [(g.idx, g.i, g.j, g.k, g.m, g.prob) for g in out[:n.value]]
    sp = (Segment * max(1, len(segments)))(*[Segment(*g) for g in segments])
    out = (Segment * 64)()
    n = C.c_int(0)
    st = L.bathhost_cluster_region_segments(sp, len(segments), nsamples, out, 64, C.byref(n))
    if st != 0:
        raise RuntimeError(f"bathhost_cluster_region_segments: status {st}")
    return [(g.idx, g.i, g.j, g.k, g.m, g.prob) for g in out[:n.value]]


def compare_tables(a, b):
    """--tblout tables hit by hit.  Hits are matched by target, query, model and target coordinates, frameshift / stop counts and
    CIGAR string: the two tables must hold the same hits.  The four printed floats of a hit (E-value, score, bias, percent identity)
    may differ by one unit of their last printed digit -- the device and the CPU oracle sum the same FP32 terms in different orders,
    and a value on a rounding boundary of %.1f prints either way -- and, the table being sorted by E-value, hits whose E-values agree
    to that precision may change places (the E-values read down the two tables must agree rank by rank).
    Returns (byte_identical, equivalent, lines_that_differ)."""
    if a == b:
        return True, True, 0
    la = [x for x in a.splitlines() if x and not x.startswith("#")]
    lb = [x for x in b.splitlines() if x and not x.startswith("#")]
    if len(la) != len(lb):
        return False, False, -1

    def close(i, u, v):
        fu, fv = float(u), float(v)
        if i == 11:
            return abs(fu - fv) <= 0.11 * max(abs(fu), abs(fv))            # two significant digits printed
        return abs(fu - fv) <= (0.0101 if i == 14 else 0.101)

    def parse(lines):
        out = {}
        for x in lines:
            f = x.split()
            if len(f) < 16:                                                    # 18 columns with --fs (shifts, stops), 16 without
                return None
            key = tuple(f[1:11]) + tuple(f[15:])
            if key in out:
                return None
            out[key] = f
        return out

    da, db = parse(la), parse(lb)
    if da is None or db is None or da.keys() != db.keys():
        return False, False, -1
    for key, fa in da.items():
        fb = db[key]
        if not all(close(i, fa[i], fb[i]) for i in (11, 12, 13, 14)):
            return False, False, -1
    ndiff = 0
    for x, y in zip(la, lb):
        fx, fy = x.split(), y.split()
        if fx[1:] != fy[1:]:
            ndiff += 1
            if not close(11, fx[11], fy[11]):                                 # another hit at this rank: only among equal E-values
                return False, False, -1
    return False, True, ndiff
