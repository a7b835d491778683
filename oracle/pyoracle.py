"""ctypes binding of the CPU oracle (oracle/liboracle.so).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and the
cpu_baseline / --impl reference legs of bench.py.  The product never imports it.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

K, KP = 20, 29
NXCELLS, NSCELLS, NSCELLS_FS = 6, 3, 8
XC_E, XC_N, XC_J, XC_B, XC_C, XC_SCALE = range(6)
OK, ERANGE = 0, 16
ST_NAMES = {1: "M", 2: "D", 3: "I", 4: "S", 5: "N", 6: "B", 7: "E", 8: "C", 9: "T", 10: "J", 11: "X"}
LOCAL, UNILOCAL = 1, 3


class HMM(C.Structure):
    _fields_ = [("M", C.c_int), ("max_length", C.c_int), ("name", C.c_char * 128), ("acc", C.c_char * 64),
                ("evparam", C.c_float * 8), ("has_stats_fs3", C.c_int), ("has_stats_fs5", C.c_int),
                ("fsprob", C.c_float), ("ct", C.c_int), ("compo", C.c_float * K), ("has_compo", C.c_int),
                ("t", C.POINTER(C.c_float)), ("mat", C.POINTER(C.c_float)), ("ins", C.POINTER(C.c_float)),
                ("consensus", C.c_char_p)]


class BG(C.Structure):
    _fields_ = [("f", C.c_float * K), ("p1", C.c_float), ("omega", C.c_float),
                ("fh_t", (C.c_float * 3) * 2), ("fh_e", (C.c_float * K) * 2),
                ("fh_eo", (C.c_float * KP) * 2), ("fh_pi", C.c_float * 3)]


class PROFILE(C.Structure):
    _fields_ = [("M", C.c_int), ("L", C.c_int), ("mode", C.c_int), ("max_length", C.c_int), ("nj", C.c_float),
                ("tsc", C.POINTER(C.c_float)), ("rsc", C.POINTER(C.c_float)), ("xsc", (C.c_float * 2) * 4),
                ("evparam", C.c_float * 8), ("compo", C.c_float * K)]


class FS_PROFILE(C.Structure):
    _fields_ = [("M", C.c_int), ("L", C.c_int), ("mode", C.c_int), ("max_length", C.c_int),
                ("codon_lengths", C.c_int), ("maxcodons", C.c_int), ("nj", C.c_float), ("fsprob", C.c_float),
                ("tsc", C.POINTER(C.c_float)), ("rsc", C.POINTER(C.c_float)), ("xsc", (C.c_float * 2) * 4),
                ("codons", C.POINTER(C.c_uint8)), ("indel_pos", C.POINTER(C.c_uint8)), ("evparam", C.c_float * 8)]


class FS_OPROFILE(C.Structure):
    _fields_ = [("M", C.c_int), ("L", C.c_int), ("mode", C.c_int), ("codon_lengths", C.c_int),
                ("maxcodons", C.c_int), ("nrows", C.c_int), ("nj", C.c_float),
                ("rfv", C.POINTER(C.c_float)), ("tfv", C.POINTER(C.c_float)), ("xf", (C.c_float * 2) * 4),
                ("evparam", C.c_float * 8)]


class OPROFILE(C.Structure):
    _fields_ = [("M", C.c_int), ("L", C.c_int), ("mode", C.c_int), ("max_length", C.c_int), ("nj", C.c_float),
                ("rbv", C.POINTER(C.c_uint8)), ("tbm_b", C.c_uint8), ("tec_b", C.c_uint8), ("tjb_b", C.c_uint8),
                ("base_b", C.c_uint8), ("bias_b", C.c_uint8), ("scale_b", C.c_float),
                ("rwv", C.POINTER(C.c_int16)), ("twv", C.POINTER(C.c_int16)), ("xw", (C.c_int16 * 2) * 4),
                ("base_w", C.c_int16), ("ddbound_w", C.c_int16), ("scale_w", C.c_float),
                ("rfv", C.POINTER(C.c_float)), ("tfv", C.POINTER(C.c_float)), ("xf", (C.c_float * 2) * 4),
                ("evparam", C.c_float * 8), ("compo", C.c_float * K)]


class WINDOW(C.Structure):
    _fields_ = [("n", C.c_int), ("k", C.c_int), ("length", C.c_int), ("target_len", C.c_int), ("id", C.c_int),
                ("score", C.c_float)]


class WINDOWLIST(C.Structure):
    _fields_ = [("w", C.POINTER(WINDOW)), ("count", C.c_int), ("nalloc", C.c_int)]


class ORF(C.Structure):
    _fields_ = [("start", C.c_int), ("end", C.c_int), ("frame", C.c_int), ("n", C.c_int), ("offset", C.c_int64)]


class MX(C.Structure):
    _fields_ = [("M", C.c_int), ("L", C.c_int), ("allocL", C.c_int), ("nscells", C.c_int),
                ("dp", C.POINTER(C.c_float)), ("xmx", C.POINTER(C.c_float)), ("totscale", C.c_float),
                ("has_own_scales", C.c_int)]


class SEGMENT(C.Structure):
    _fields_ = [("idx", C.c_int), ("i", C.c_int), ("j", C.c_int), ("k", C.c_int), ("m", C.c_int), ("prob", C.c_float)]


class TRACE(C.Structure):
    _fields_ = [("N", C.c_int), ("nalloc", C.c_int), ("M", C.c_int), ("L", C.c_int),
                ("st", C.POINTER(C.c_char)), ("k", C.POINTER(C.c_int)), ("i", C.POINTER(C.c_int)),
                ("c", C.POINTER(C.c_int)), ("pp", C.POINTER(C.c_float))]


def build(force=False):
    """Compile oracle/*.c into liboracle.so (gcc).  Building the checker is not using it."""
    so = os.path.join(_HERE, "liboracle.so")
    srcs = [os.path.join(_HERE, f) for f in os.listdir(_HERE) if f.endswith((".c", ".h"))]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["make", "-s", "-C", _HERE])
    return so


def build_native(outdir):
    """Host-tuned build (-O3 -march=native) for the CPU-baseline legs of bench.py; built on the box that runs it, into outdir
    (bench.py writes nothing in the source tree, which may be read-only)."""
    so = os.path.join(outdir, "liboracle_native.so")
    subprocess.check_call(["make", "-s", "-B", "-C", _HERE, "native", f"NATIVE={so}"])   # -B: never trust a copy built on another host
    return so


def lib(native=False):
    global _LIB
    if _LIB is not None:
        return _LIB
    if native:
        with tempfile.TemporaryDirectory(prefix="bath_oracle_native_") as d:
            L = C.CDLL(build_native(d))          # the loaded mapping outlives the file
    else:
        L = C.CDLL(build())
    P = C.POINTER
    u8p, fp = P(C.c_uint8), P(C.c_float)
    sig = {
        "bo_hmmfile_read": (C.c_int, [C.c_char_p, C.c_int, P(P(HMM))]),
        "bo_hmmfile_count": (C.c_int, [C.c_char_p]),
        "bo_hmm_destroy": (None, [P(HMM)]),
        "bo_bg_create": (P(BG), []),
        "bo_bg_destroy": (None, [P(BG)]),
        "bo_bg_SetLength": (None, [P(BG), C.c_int]),
        "bo_bg_NullOne": (C.c_float, [P(BG), C.c_int]),
        "bo_bg_fs_NullOne": (C.c_float, [P(BG), C.c_int]),
        "bo_profile_config": (P(PROFILE), [P(HMM), P(BG), C.c_int, C.c_int]),
        "bo_profile_destroy": (None, [P(PROFILE)]),
        "bo_fs_profile_config": (P(FS_PROFILE), [P(HMM), P(BG), C.c_int, C.c_int, C.c_int, C.c_int]),
        "bo_fs_profile_destroy": (None, [P(FS_PROFILE)]),
        "bo_fs_ReconfigLength": (None, [P(FS_PROFILE), C.c_int]),
        "bo_fs_ReconfigUnihit": (None, [P(FS_PROFILE), C.c_int]),
        "bo_fs_ReconfigMultihit": (None, [P(FS_PROFILE), C.c_int]),
        "bo_fs_oprofile_convert": (P(FS_OPROFILE), [P(FS_PROFILE)]),
        "bo_fs_oprofile_destroy": (None, [P(FS_OPROFILE)]),
        "bo_fs_oprofile_ReconfigLength": (None, [P(FS_OPROFILE), C.c_int]),
        "bo_fs_oprofile_ReconfigUnihit": (None, [P(FS_OPROFILE), C.c_int]),
        "bo_fs_oprofile_ReconfigMultihit": (None, [P(FS_OPROFILE), C.c_int]),
        "bo_mx_create": (P(MX), [C.c_int, C.c_int, C.c_int]),
        "bo_mx_destroy": (None, [P(MX)]),
        "bo_trace_create": (P(TRACE), []),
        "bo_trace_reuse": (None, [P(TRACE)]),
        "bo_trace_destroy": (None, [P(TRACE)]),
        "bo_ForwardParser_Frameshift_3Codons": (C.c_int, [u8p, C.c_int, P(FS_OPROFILE), P(MX), fp]),
        "bo_BackwardParser_Frameshift_3Codons": (C.c_int, [u8p, C.c_int, P(FS_OPROFILE), P(MX), P(MX), fp]),
        "bo_Forward_Frameshift": (C.c_int, [u8p, C.c_int, P(FS_OPROFILE), P(MX), fp]),
        "bo_Backward_Frameshift": (C.c_int, [u8p, C.c_int, P(FS_OPROFILE), P(MX), P(MX), fp]),
        "bo_Decoding_Frameshift": (C.c_int, [P(FS_OPROFILE), P(MX), P(MX)]),
        "bo_DomainDecoding_Frameshift": (C.c_int, [fp, P(MX), P(MX), fp, fp, fp]),
        "bo_OptimalAccuracy_Frameshift": (C.c_int, [P(FS_OPROFILE), P(MX), P(MX), fp]),
        "bo_OATrace_Frameshift": (C.c_int, [P(FS_OPROFILE), P(MX), P(MX), P(TRACE)]),
        "bo_Null2_fs_ByExpectation": (C.c_int, [P(FS_OPROFILE), P(MX), fp]),
        "bo_oprofile_convert": (P(OPROFILE), [P(PROFILE)]),
        "bo_oprofile_destroy": (None, [P(OPROFILE)]),
        "bo_oprofile_ReconfigLength": (None, [P(OPROFILE), C.c_int]),
        "bo_oprofile_ssv_scores": (None, [P(OPROFILE), u8p]),
        "bo_SSVFilter": (C.c_int, [u8p, C.c_int, P(OPROFILE), fp]),
        "bo_MSVFilter": (C.c_int, [u8p, C.c_int, P(OPROFILE), fp]),
        "bo_MSVFilter_opt": (C.c_int, [u8p, C.c_int, P(OPROFILE), C.c_int, fp]),
        "bo_SSVFilter_BATH": (C.c_int, [u8p, C.c_int, P(OPROFILE), u8p, C.c_float, C.c_double, C.c_int, P(WINDOWLIST)]),
        "bo_ViterbiFilter": (C.c_int, [u8p, C.c_int, P(OPROFILE), fp]),
        "bo_ViterbiFilter_BATH": (C.c_int, [u8p, C.c_int, P(OPROFILE), u8p, C.c_float, C.c_double, C.c_int,
                                            P(WINDOWLIST), fp]),
        "bo_ForwardParser": (C.c_int, [u8p, C.c_int, P(OPROFILE), fp]),
        "bo_find_orfs": (C.c_int, [u8p, C.c_int, u8p, C.c_int, P(P(ORF)), P(C.c_int), P(u8p), P(C.c_int64)]),
        "bo_oprofile_ReconfigMultihit": (None, [P(OPROFILE), C.c_int]),
        "bo_oprofile_ReconfigUnihit": (None, [P(OPROFILE), C.c_int]),
        "bo_Forward": (C.c_int, [u8p, C.c_int, P(OPROFILE), P(MX), fp]),
        "bo_Backward": (C.c_int, [u8p, C.c_int, P(OPROFILE), P(MX), P(MX), fp]),
        "bo_Decoding": (C.c_int, [P(OPROFILE), P(MX), P(MX), P(MX)]),
        "bo_DomainDecoding": (C.c_int, [fp, P(MX), P(MX), C.c_int, fp, fp, fp]),
        "bo_OptimalAccuracy": (C.c_int, [P(OPROFILE), P(MX), P(MX), fp]),
        "bo_OATrace": (C.c_int, [P(OPROFILE), P(MX), P(MX), C.c_int, P(TRACE)]),
        "bo_Null2_ByExpectation": (C.c_int, [P(OPROFILE), P(MX), fp]),
        "bo_windowlist_reset": (None, [P(WINDOWLIST)]),
        "bo_windowlist_free": (None, [P(WINDOWLIST)]),
        "bo_gumbel_invsurv": (C.c_double, [C.c_double, C.c_double, C.c_double]),
        "bo_gumbel_surv": (C.c_double, [C.c_double, C.c_double, C.c_double]),
        "bo_exp_surv": (C.c_double, [C.c_double, C.c_double, C.c_double]),
        "bo_exp_logsurv": (C.c_double, [C.c_double, C.c_double, C.c_double]),
        "bo_profile_ReconfigLength": (None, [P(PROFILE), C.c_int]),
        "bo_batch_ForwardParser_3Codons": (C.c_int, [u8p, P(C.c_int64), P(C.c_int32), C.c_int, P(FS_OPROFILE),
                                                     C.c_int, fp, P(C.c_int32)]),
        "bo_FLogsum": (C.c_float, [C.c_float, C.c_float]),
        "bo_FLogsumInit": (None, []),
        "bo_cephes_expf": (C.c_float, [C.c_float]),
        "bo_nt_digitize": (C.c_int, [C.c_char]),
        "bo_aa_digitize": (C.c_int, [C.c_char]),
        "bo_dna_revcomp": (None, [u8p, C.c_int64]),
        "bo_gencode_basic": (u8p, [C.c_int]),
        "bo_Lambda": (C.c_double, [P(HMM), P(BG)]),
        "bo_Calibrate": (C.c_int, [P(HMM), P(BG), P(OPROFILE), P(FS_OPROFILE), P(FS_OPROFILE), C.c_int, C.c_uint32, C.c_double,
                                   C.c_int, C.c_int, P(C.c_uint32), P(C.c_double)]),
        "bo_region_trace_ensemble_frameshift": (C.c_int, [P(FS_OPROFILE), P(MX), C.c_int, C.c_int, C.c_uint32, C.c_int,
                                                          P(SEGMENT), C.c_int, P(C.c_int), P(SEGMENT), C.c_int]),
    }
    for name, (res, args) in sig.items():
        f = getattr(L, name)
        f.restype, f.argtypes = res, args
    L.bo_FLogsumInit()
    _LIB = L
    return L


# ------------------------------------------------------------------ helpers

def u8ptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint8))


def fptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def read_fasta(path):
    """-> list of (name, desc, sequence string)"""
    out, name, desc, buf = [], None, "", []
    with open(path) as fh:
        for line in fh:
            line = line.rstrip("\n")
            if line.startswith(">"):
                if name is not None:
                    out.append((name, desc, "".join(buf)))
                hdr = line[1:].split(None, 1)
                name, desc, buf = hdr[0], (hdr[1] if len(hdr) > 1 else ""), []
            else:
                buf.append(line.strip())
    if name is not None:
        out.append((name, desc, "".join(buf)))
    return out


_NT = {c: i for i, c in enumerate("ACGT-RYMKSWHBVDN*~")}


def digitize_dna(seq):
    """-> uint8 array, 1-based with sentinels 255 at [0] and [L+1] (ESL_DSQ)"""
    s = seq.upper().replace("U", "T").replace("X", "N")
    a = np.full(len(s) + 2, 255, dtype=np.uint8)
    a[1:-1] = [_NT[c] for c in s]
    return a


def revcomp_dsq(dsq):
    d = dsq.copy()
    lib().bo_dna_revcomp(u8ptr(d), len(d) - 2)
    return d


class Model:
    """One query profile: HMM + bg + gm_fs5/gm_fs3 + om_fs5/om_fs3, as bathsearch
    sets them up (src/bathsearch.c:794-801: dummy L=100, p7_LOCAL)."""

    def __init__(self, path, index=0, ct=None):
        L = lib()
        self.path, self.index = path, index
        hp = C.POINTER(HMM)()
        st = L.bo_hmmfile_read(path.encode(), index, C.byref(hp))
        if st != OK:
            raise IOError(f"cannot read model {index} of {path}: status {st}")
        self.hmm = hp
        self.M = hp.contents.M
        self.max_length = hp.contents.max_length
        self.evparam = list(hp.contents.evparam)
        self.ct = ct if ct is not None else (hp.contents.ct if hp.contents.ct > 0 else 1)
        self.bg = L.bo_bg_create()
        self.gm_fs5 = L.bo_fs_profile_config(self.hmm, self.bg, self.ct, 5, 100, LOCAL)
        self.gm_fs3 = L.bo_fs_profile_config(self.hmm, self.bg, self.ct, 3, 100, LOCAL)
        self.om_fs5 = L.bo_fs_oprofile_convert(self.gm_fs5)
        self.om_fs3 = L.bo_fs_oprofile_convert(self.gm_fs3)
        # protein profile for the ORF filters (src/bathsearch.c:794-796: p7_ProfileConfig(L=100, p7_LOCAL), p7_oprofile_Convert)
        self.gm = L.bo_profile_config(self.hmm, self.bg, 100, LOCAL)
        self.om = L.bo_oprofile_convert(self.gm)
        self._ssv_scores = np.zeros((self.M + 1) * KP, np.uint8)
        L.bo_oprofile_ssv_scores(self.om, u8ptr(self._ssv_scores))

    def rfv(self, which=3):
        om = (self.om_fs3 if which == 3 else self.om_fs5).contents
        return np.ctypeslib.as_array(om.rfv, shape=(om.nrows, om.M + 1))

    def tfv(self, which=3):
        om = (self.om_fs3 if which == 3 else self.om_fs5).contents
        return np.ctypeslib.as_array(om.tfv, shape=(8, om.M + 1))

    def ssv_scores(self):
        return self._ssv_scores

    def om_tables(self):
        """un-striped integer/float tables of the protein profile: rbv [Kp][M+1] u8, rwv [Kp][M+1] i16, twv [8][M+1] i16"""
        o = self.om.contents
        M = self.M
        return (np.ctypeslib.as_array(o.rbv, shape=(KP, M + 1)), np.ctypeslib.as_array(o.rwv, shape=(KP, M + 1)),
                np.ctypeslib.as_array(o.twv, shape=(8, M + 1)), np.ctypeslib.as_array(o.rfv, shape=(KP, M + 1)),
                np.ctypeslib.as_array(o.tfv, shape=(8, M + 1)))

    def xf(self, which=3):
        om = (self.om_fs3 if which == 3 else self.om_fs5).contents
        return np.array([[om.xf[s][t] for t in range(2)] for s in range(4)], dtype=np.float32)


def calibrate(model, seed=42, lam=None, which=31, convert_flow=False, rng_x=0):
    """p7_Calibrate with the frameshift branch (src/evalues.c:64-183) on a FRESH copy of the model's profiles (the simulations
    reconfigure the length models): evparam[8].  lam=None: the model file's lambda, as bathconvert passes it
    (src/bathconvert.c:157); lam <= 0: p7_Lambda.  convert_flow: bathconvert's frameshift-only
    calibration on a generator that runs on from model to model (rng_x = state left by the previous model, 0 = fresh).
    Returns (evparam, generator state)."""
    m = Model.__new__(Model)
    Model.__init__(m, model.path, model.index, model.ct)
    out = (C.c_double * 8)()
    if lam is None:
        lam = float(model.evparam[5])
    x = C.c_uint32(rng_x)
    st = lib().bo_Calibrate(m.hmm, m.bg, m.om, m.om_fs3, m.om_fs5, m.ct, seed, float(lam), which, int(convert_flow), C.byref(x), out)
    if st != OK:
        raise RuntimeError(f"bo_Calibrate: status {st}")
    return [float(v) for v in out], x.value


def simd_supported():
    L = lib()
    L.bo_fwd3_simd_supported.restype = C.c_int
    return bool(L.bo_fwd3_simd_supported())


def batch_forward_parser(model, dsq, starts, lengths, nthreads=1, simd=False):
    """Forward parser (3 codon lengths) over windows dsq[start .. start+L-1] with a thread pool.  simd: the AVX2 + FMA build
    (fwd3_avx2.c) instead of the scalar restatement."""
    n = len(starts)
    st64 = np.ascontiguousarray(starts, np.int64)
    l32 = np.ascontiguousarray(lengths, np.int32)
    sc = np.empty(n, np.float32)
    status = np.empty(n, np.int32)
    fn = lib().bo_batch_ForwardParser_3Codons_simd if simd else lib().bo_batch_ForwardParser_3Codons
    if simd:
        fn.restype, fn.argtypes = lib().bo_batch_ForwardParser_3Codons.restype, lib().bo_batch_ForwardParser_3Codons.argtypes
    rc = fn(u8ptr(dsq), st64.ctypes.data_as(C.POINTER(C.c_int64)), l32.ctypes.data_as(C.POINTER(C.c_int32)), n, model.om_fs3,
            int(nthreads), fptr(sc), status.ctypes.data_as(C.POINTER(C.c_int32)))
    if rc != OK:
        raise RuntimeError(f"bo_batch_ForwardParser_3Codons: status {rc}")
    return sc, status


_AA = {c: i for i, c in enumerate("ACDEFGHIKLMNPQRSTVWY-BJZOUX*~")}


def digitize_amino(seq):
    a = np.full(len(seq) + 2, 255, dtype=np.uint8)
    a[1:-1] = [_AA[c] for c in seq.upper()]
    return a


def find_orfs(dsq, n, gcode, min_len):
    """bo_find_orfs: list of (start, end, frame, residues array) in the reference's order"""
    L = lib()
    orfs, norf, res, nres = C.POINTER(ORF)(), C.c_int(), C.POINTER(C.c_uint8)(), C.c_int64()
    g = np.ascontiguousarray(gcode, np.uint8)
    d = np.ascontiguousarray(dsq, np.uint8)
    assert L.bo_find_orfs(u8ptr(d), int(n), u8ptr(g), int(min_len), C.byref(orfs), C.byref(norf), C.byref(res), C.byref(nres)) == 0
    r = np.ctypeslib.as_array(res, shape=(max(nres.value, 1),))[: nres.value].copy()
    out = [(orfs[i].start, orfs[i].end, orfs[i].frame, r[orfs[i].offset: orfs[i].offset + orfs[i].n]) for i in range(norf.value)]
    libc = C.CDLL(None)
    libc.free(orfs); libc.free(res)
    return out


def windows(wl):
    return [(wl.w[z].n, wl.w[z].k, wl.w[z].length, wl.w[z].score) for z in range(wl.count)]


def cpu_backend(nthreads=1, simd=False):
    """The batched stage calls of include/bathgpu.h on the CPU (oracle/cpu_backend.c), as a bathhost_backend table for the
    host pipeline.  TESTS AND BENCH ONLY.  Returns (backend struct, keep-alive handle).  simd=True: the MSV + SSV screen of every ORF on
    the AVX2 build of the same byte arithmetic (msv_avx2.c), for bench.py's CPU arm; the scalar restatement is the checker."""
    from bath_b200 import hostapi
    L = lib()
    L.bo_backend_create.restype = C.c_void_p
    L.bo_backend_create.argtypes = [C.c_int]
    L.bo_backend_destroy.argtypes = [C.c_void_p]
    h = L.bo_backend_create(int(nthreads))
    if simd:
        L.bo_backend_set_simd.argtypes = [C.c_void_p, C.c_int]
        L.bo_backend_set_simd(h, 1)
    be = hostapi.Backend()
    be.ctx = h
    for n in hostapi.Backend._names:
        setattr(be, n, C.cast(getattr(L, "bo_backend_" + n), C.c_void_p))

    class _Handle:
        def __init__(self, ptr):
            self.ptr = ptr

        def __del__(self):
            try:
                L.bo_backend_destroy(self.ptr)
            except Exception:
                pass

    return be, _Handle(h)


def region_trace_ensemble(om_fs5, fwd, ireg, jreg, seed=42, nsamples=200):
    """region_trace_ensemble_frameshift on a filled multihit Forward matrix: (sampled segments, consensus envelopes), each a list
    of (idx, i, j, k, m, prob)"""
    cap = nsamples * 64
    sp, out = (SEGMENT * cap)(), (SEGMENT * 64)()
    nsp = C.c_int(0)
    nc = lib().bo_region_trace_ensemble_frameshift(om_fs5, fwd, ireg, jreg, seed, nsamples, sp, cap, C.byref(nsp), out, 64)
    if nc < 0:
        raise RuntimeError("stochastic traceback failed")
    as_t = lambda g: (g.idx, g.i, g.j, g.k, g.m, g.prob)
    return [as_t(sp[z]) for z in range(nsp.value)], [as_t(out[z]) for z in range(nc)]


def mx_xmx(mx):
    m = mx.contents
    return np.ctypeslib.as_array(m.xmx, shape=(m.allocL + 2, NXCELLS))[: m.L + 1]


def mx_dp(mx):
    m = mx.contents
    return np.ctypeslib.as_array(m.dp, shape=(m.allocL + 1, m.M + 1, m.nscells))[: m.L + 1]


def trace_list(tr):
    t = tr.contents
    return [(ST_NAMES[ord(t.st[z])], t.k[z], t.i[z], t.c[z], t.pp[z]) for z in range(t.N)]
