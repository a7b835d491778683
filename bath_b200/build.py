"""Build libbathgpu.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "csrc")
_SO = os.path.join(_HERE, "libbathgpu.so")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-ftz=true", "-shared", "-Xcompiler", "-fPIC"]


def library_path():
    """Path of the built library (BATHGPU_LIB overrides it, for A/B builds while tuning)."""
    return os.environ.get("BATHGPU_LIB", _SO)


def _sources():
    out = []
    for root, _, files in os.walk(_CSRC):
        out += [os.path.join(root, f) for f in files if f.endswith((".cu", ".cuh", ".h", ".cpp", ".hpp"))]
    out.append(os.path.join(_HERE, "..", "include", "bathgpu.h"))
    return out


_HOST = os.path.join(_HERE, "host")
_HOST_SO = os.path.join(_HERE, "libbathhost.so")
GXX_FLAGS = ["-O2", "-g", "-std=c++17", "-fPIC", "-shared", "-Wall", "-ffp-contract=off", "-fno-fast-math", "-pthread"]


def host_library_path():
    return _HOST_SO


def build_host_library(force=False):
    """libbathhost.so: the host side of the path (model set-up, length models, pipeline logic), g++ only."""
    srcs = [os.path.join(_HOST, f) for f in sorted(os.listdir(_HOST)) if f.endswith((".cpp", ".h"))]
    srcs.append(os.path.join(_HERE, "..", "include", "bathhost.h"))
    if not force and os.path.exists(_HOST_SO) and all(os.path.getmtime(s) <= os.path.getmtime(_HOST_SO) for s in srcs):
        return _HOST_SO
    cmd = [os.environ.get("CXX", "g++")] + GXX_FLAGS + ["-o", _HOST_SO] + [s for s in srcs if s.endswith(".cpp")]
    subprocess.check_call(cmd)
    return _HOST_SO


_INTEG = os.path.join(_HERE, "..", "integration")
_SHIM_SO = os.path.join(_INTEG, "libbathshim.so")


def shim_library_path():
    return _SHIM_SO


def build_shim_library(force=False):
    """integration/libbathshim.so: the reference's impl-layer parser prototypes implemented on libbathgpu.so (impl_cuda_shim.c), compiled
    against the stand-in for impl_sse.h, plus the test helper that stripes profiles the SSE way.  gcc only; needs libbathgpu.so to link."""
    srcs = [os.path.join(_INTEG, f) for f in ("impl_cuda_shim.c", "shim_test_helper.c", "bath_impl_standin.h")]
    srcs.append(os.path.join(_HERE, "..", "include", "bathgpu.h"))
    if not force and os.path.exists(_SHIM_SO) and all(os.path.getmtime(s) <= os.path.getmtime(_SHIM_SO) for s in srcs + [_SO]):
        return _SHIM_SO
    cmd = [os.environ.get("CC", "gcc"), "-O2", "-g", "-std=gnu11", "-msse2", "-fPIC", "-shared", "-Wall", "-Wextra",
           "-I", _INTEG, "-I", os.path.join(_HERE, "..", "include"), "-o", _SHIM_SO] + [s for s in srcs if s.endswith(".c")] + \
          ["-L", _HERE, "-lbathgpu", "-Wl,-rpath,$ORIGIN/../bath_b200", "-lm"]
    subprocess.check_call(cmd)
    return _SHIM_SO


_OBJ = os.path.join(_HERE, "_obj")

# kernels_tu.cu is compiled once per (family, node-count set): see csrc/launch.h
_FAMILIES = {"fwd": 1, "bck": 2, "fs5": 3, "orf": 4}
_SETS = {"a": 0, "b": 1, "c": 2, "d": 3, "e": 4, "f": 5, "g": 6, "h": 7}
_FILTERS = {"msv": 5, "vit_lo": 6, "vit_hi": 7}


def _units():
    """(object name, source, extra -D flags) of every translation unit of libbathgpu.so"""
    units = [("bathgpu", os.path.join(_CSRC, "bathgpu.cu"), [])]
    tu = os.path.join(_CSRC, "kernels_tu.cu")
    for fam, fid in _FAMILIES.items():
        for sname, sid in _SETS.items():
            units.append((f"k_{fam}_{sname}", tu, [f"-DBATHGPU_FAMILY={fid}", f"-DBATHGPU_SET={sid}"]))
    for fam, fid in _FILTERS.items():
        units.append((f"k_{fam}", tu, [f"-DBATHGPU_FAMILY={fid}", "-DBATHGPU_SET=0"]))
    return units


def build_library(force=False, verbose=False, jobs=None, variant=None, extra_flags=()):
    """variant / extra_flags: an A/B build while tuning (libbathgpu_<variant>.so, its own object directory); load it with BATHGPU_LIB."""
    srcs = _sources()
    newest = max(os.path.getmtime(s) for s in srcs + [os.path.abspath(__file__)])
    _SO = os.path.join(_HERE, f"libbathgpu_{variant}.so") if variant else globals()["_SO"]
    _OBJ = globals()["_OBJ"] + (f"_{variant}" if variant else "")
    if not force and os.path.exists(_SO) and newest <= os.path.getmtime(_SO):
        return _SO
    from concurrent.futures import ThreadPoolExecutor
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    os.makedirs(_OBJ, exist_ok=True)
    flags = [f for f in NVCC_FLAGS if f != "-shared"] + (["-Xptxas", "-v"] if verbose else []) + list(extra_flags)

    def compile_one(unit):
        name, src, defs = unit
        obj = os.path.join(_OBJ, name + ".o")
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < newest:
            subprocess.check_call([nvcc] + flags + defs + ["-c", src, "-o", obj])
        return obj

    units = _units()
    if variant and os.environ.get("BATHGPU_VARIANT_UNITS"):      # rebuild only these units, take the rest from the main build
        only = set(os.environ["BATHGPU_VARIANT_UNITS"].split(","))
        main_obj = globals()["_OBJ"]
        keep = [os.path.join(main_obj, u[0] + ".o") for u in units if u[0] not in only]
        units = [u for u in units if u[0] in only]
    else:
        keep = []
    # longest first: the node-count sets with the most (or the largest) instantiations
    units.sort(key=lambda u: (u[0].endswith(("_h", "_g", "_f", "_e", "_c", "_b")), u[0]), reverse=True)
    with ThreadPoolExecutor(max_workers=jobs or os.cpu_count() or 4) as pool:
        objs = list(pool.map(compile_one, units)) + keep
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-Xcompiler", "-fPIC", "-o", _SO] + objs)
    return _SO


if __name__ == "__main__":
    import sys
    print(build_host_library(force="--force" in sys.argv))
    var = next((a.split("=", 1)[1] for a in sys.argv if a.startswith("--variant=")), None)
    extra = [a for a in sys.argv[1:] if a.startswith("-D")]
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv, variant=var, extra_flags=extra))
    if not var:
        print(build_shim_library(force="--force" in sys.argv))
