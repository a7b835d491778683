"""Models per second of the HMMER3/f -> BATH3/f conversion on one GPU: the batched driver (hostapi.convert: the frameshift simulations
of up to 128 models per device call) against the per-model paths it replaces.

The library is ~1000 models: every shipped model, turned back into HMMER3/f (header, FS STATS / FRAMESHIFT / CODON lines removed),
repeated with the NAME suffixed.  Timed, each after an untimed pass over a 40-model library and repeated --repeats times:
  batched     hostapi.convert with the device set calls
  per_model   hostapi.convert through a backend without them: bathhost_calibrate model by model (host set-up still threaded)
  loop        hostapi.QueryModel + hostapi.calibrate per model from Python, the generator carried: the per-model loop, all serial
  setup       hostapi.QueryModel alone for every model: the host's share of the loop (profile construction)
The batched output is checked against the loop's values line by line.  Prints one JSON line (and writes it to --out)."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

FS_TAGS = ("STATS LOCAL FS3", "STATS LOCAL FS5", "FRAMESHIFT PROB", "CODON TABLE")


def records(path):
    out, cur = [], []
    for line in open(path):
        cur.append(line)
        if line.startswith("//"):
            out.append(cur)
            cur = []
    return out


def library(path, n_models):
    """(models written, their source records): shipped codon-table-1 models as HMMER3/f, repeated, names suffixed"""
    import common
    src = []
    for f in sorted(os.listdir(common.GOLDEN)):
        if f.endswith(".bhmm") and not f.startswith("synthetic_") and f != "MET-ct4.bhmm":
            src += [(f, i, r) for i, r in enumerate(records(common.golden(f)))]
    out = []
    with open(path, "w") as fh:
        for k in range(n_models):
            f, i, rec = src[k % len(src)]
            for line in rec:
                if line.startswith("BATH3/f"):
                    fh.write("HMMER3/f [3.3 | Nov 2019]\n")
                elif line.startswith("NAME"):
                    fh.write(line.rstrip("\n") + f"_r{k // len(src)}\n")
                elif not line.startswith(FS_TAGS):
                    fh.write(line)
            out.append((f, i))
    return out


def fs_lines(text):
    return [l for l in text.splitlines() if l.startswith(("STATS LOCAL FS3", "STATS LOCAL FS5"))]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--models", type=int, default=1000)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    from bath_b200 import capi, hostapi
    import common

    gpu = {"name": None, "power_limit": None}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        gpu["name"], gpu["power_limit"] = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    except Exception as e:                      # the measurement stands without it; say so
        gpu["error"] = repr(e)

    ctx = capi.Context(0)
    be_set = hostapi.backend_from(ctx.lib, ctx.h)
    be_one = hostapi.backend_from(ctx.lib, ctx.h)
    be_one.load_fs_profile_set = None
    be_one.fs_set_scores = None

    tmp = tempfile.mkdtemp()
    lib_path, warm_path = os.path.join(tmp, "lib.hmm"), os.path.join(tmp, "warm.hmm")
    src = library(lib_path, args.models)
    library(warm_path, 40)
    sizes = [hostapi.QueryModel(common.golden(f), i).M for f, i in src]

    def run_convert(be, path, out):
        t0 = time.perf_counter()
        n = hostapi.convert(path, out, backend=be)
        return n, time.perf_counter() - t0

    def run_loop(models):
        t0 = time.perf_counter()
        x, lines = 0, []
        for f, i in models:
            ev, x = hostapi.calibrate(hostapi.QueryModel(common.golden(f), i), backend=be_set, convert_flow=True, rng_state=x, which=24)
            lines.append(f"STATS LOCAL FS3 FORWARD {np.float32(ev[6]):8.4f} {np.float32(ev[5]):8.5f}")
            lines.append(f"STATS LOCAL FS5 FORWARD {np.float32(ev[7]):8.4f} {np.float32(ev[5]):8.5f}")
        return lines, time.perf_counter() - t0

    def run_setup(models):
        t0 = time.perf_counter()
        for f, i in models:
            hostapi.QueryModel(common.golden(f), i).close()
        return time.perf_counter() - t0

    run_convert(be_set, warm_path, os.path.join(tmp, "w1.bhmm"))
    run_convert(be_one, warm_path, os.path.join(tmp, "w2.bhmm"))
    run_loop(src[:40])

    res = {"batched": [], "per_model": [], "loop": [], "setup": []}
    out_b, out_p = os.path.join(tmp, "b.bhmm"), os.path.join(tmp, "p.bhmm")
    loop_lines = None
    for _ in range(args.repeats):               # the three paths alternate, so that drift of the shared host hits all of them
        n, t = run_convert(be_set, lib_path, out_b)
        res["batched"].append(t)
        n2, t = run_convert(be_one, lib_path, out_p)
        res["per_model"].append(t)
        loop_lines, t = run_loop(src)
        res["loop"].append(t)
        res["setup"].append(run_setup(src))
    assert n == n2 == len(src)
    same_b = fs_lines(open(out_b).read()) == loop_lines
    same_p = fs_lines(open(out_p).read()) == loop_lines
    result = {"gpu": gpu, "models": len(src), "M_min": int(min(sizes)), "M_max": int(max(sizes)), "M_mean": float(np.mean(sizes)),
              "host_cores": os.cpu_count(), "repeats": args.repeats,
              "seconds": {k: [round(v, 3) for v in vs] for k, vs in res.items()},
              "models_per_s": {k: round(len(src) / min(vs), 1) for k, vs in res.items()},
              "batched_equals_loop": same_b, "per_model_equals_loop": same_p}
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    ctx.close()
    if not (same_b and same_p):
        sys.exit(1)


if __name__ == "__main__":
    main()
