"""Time a profile library against one planted genome on one GPU, three ways, alternating (best of --repeats):
  (a) library: hostapi.LibrarySearch -- the target uploaded once per context, the ORF screen of many profiles in one device call;
  (b) loop:    one hostapi.Search per model over the same contexts, one after the other;
  (c) many:    hostapi.Search.finish_many over groups of models, one device context per search of a group.
The library holds the shipped BATH3/f models repeated to --models (mixed M and MAXL).  Reports wall seconds, profiles x Gbp / s, the
set screen's kernel-group times of the library's last call, whether every model's table is the same on the three paths, and the card's
name and power limit read in the same run.  Usage: python scripts/library_search_time.py [--models 100] [--mbp 100] [--out f.json]"""
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

SHIPPED = ["tRNA-proteins.bhmm", "tRNA-synthetases.bhmm", "AMP_N.bhmm", "2OG-FeII_Oxy_3.bhmm", "PTH2.bhmm", "PTHR37536.bhmm"]


def library(path, n_models):
    import common
    texts = []
    for f in SHIPPED:
        texts += [t + "//\n" for t in open(common.golden(f)).read().split("//\n") if t.strip()]
    with open(path, "w") as fh:
        for z in range(n_models):
            fh.write(texts[z % len(texts)])
    return n_models


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--models", type=int, default=100)
    ap.add_argument("--mbp", type=float, default=100.0)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--group", type=int, default=4, help="searches per finish_many call in path (c), each on a context of its own")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    from bath_b200 import capi, hostapi, synth
    import common

    gpu = {"name": None, "power_limit": None}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        gpu["name"], gpu["power_limit"] = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    except Exception as e:
        gpu["error"] = repr(e)

    tmp = tempfile.mkdtemp()
    path = os.path.join(tmp, "library.bhmm")
    n = library(path, args.models)
    models = [hostapi.QueryModel(path, i) for i in range(n)]
    rng = np.random.default_rng(2026)
    nt = int(args.mbp * 1e6)
    dsq, _ = synth.planted_genome(rng, nt, models[0].mat(), every=200_000, fs_rate=models[0].fsprob)
    ctxs = [capi.Context(0) for _ in range(args.group)]

    def run_library():
        lib = hostapi.LibrarySearch(models, gpu_ctx=ctxs[0])
        lib.queue_sequence("genome", dsq)
        t0 = time.perf_counter()
        lib.finish()
        t = time.perf_counter() - t0
        ms, norf, scored = ctxs[0].orfs_stage_breakdown()
        tabs = [s.tblout() for s in lib.searches]
        lib.close()
        return t, tabs, [round(float(x), 3) for x in ms]

    def run_loop():
        t, tabs = 0.0, []
        for m in models:
            s = hostapi.Search(m, ctxs[0])
            s.queue_sequence("genome", dsq)
            t0 = time.perf_counter()
            s.finish(fetch=False)
            t += time.perf_counter() - t0
            tabs.append(s.tblout())
            s.close()
        return t, tabs

    def run_many():
        t, tabs = 0.0, []
        for g0 in range(0, n, args.group):
            ss = [hostapi.Search(m, ctxs[k]) for k, m in enumerate(models[g0: g0 + args.group])]
            for s in ss:
                s.queue_sequence("genome", dsq)
            t0 = time.perf_counter()
            hostapi.Search.finish_many(ss)
            t += time.perf_counter() - t0
            tabs += [s.tblout() for s in ss]
            for s in ss:
                s.close()
        return t, tabs

    secs = {"library": [], "loop": [], "many": []}
    screen_ms = None
    same = True
    for _ in range(args.repeats):                # the paths alternate, so that drift of the shared host hits all of them
        t, ta, screen_ms = run_library()
        secs["library"].append(t)
        t, tb = run_loop()
        secs["loop"].append(t)
        t, tc = run_many()
        secs["many"].append(t)
        same = same and ta == tb == tc
    gbp = nt / 1e9
    result = {"gpu": gpu, "models": n, "M": [int(min(m.M for m in models)), int(max(m.M for m in models))],
              "max_length": [int(min(m.max_length for m in models)), int(max(m.max_length for m in models))],
              "target_mbp": args.mbp, "repeats": args.repeats, "group": args.group,
              "seconds": {k: [round(v, 3) for v in vs] for k, vs in secs.items()},
              "profile_gbp_per_s": {k: round(n * gbp / min(vs), 2) for k, vs in secs.items()},
              "library_set_screen_ms_last_call": {"classes": screen_ms[0], "count": screen_ms[1], "emit": screen_ms[2], "msv": screen_ms[3],
                                                  "screen": screen_ms[4]},
              "tables_identical": same}
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    for c in ctxs:
        c.close()
    if not same:
        sys.exit(1)


if __name__ == "__main__":
    main()
