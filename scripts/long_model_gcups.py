"""Long models (M = 1280 and 2014, the models of tests/test_gpu_long_models.py) on one device: Forward parser, Forward + Backward and
envelope-stage GCUPS, and the search rate of one long model over a >= 100 Mbp random target.  Kernel times are CUDA-event times of
the stage calls (bathgpu_last_stage_timing); the search rate is host wall time around whole searches that end in a device wait.
The card's name, power limit and maximum SM clock are read in the same run.

    python scripts/long_model_gcups.py OUT.json [target_mbp]
"""
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, '.'); sys.path.insert(0, 'tests')
import common
from oracle import pyoracle as po          # only to read the profile files into the load calls' tables
from bath_b200 import capi, hostapi

LONG = {"M1280": common.SYNTHETIC["synthetic_M903.bhmm"] + [("tRNA-synthetases.bhmm", 0), ("tRNA-synthetases.bhmm", 1)],
        "M2014": common.SYNTHETIC["synthetic_M903.bhmm"] * 2 + common.SYNTHETIC["synthetic_M208.bhmm"]}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    out_path = sys.argv[1]
    target_mbp = float(sys.argv[2]) if len(sys.argv) > 2 else 100.0
    tmp = tempfile.mkdtemp()
    paths = {}
    for name, parts in LONG.items():
        paths[name] = os.path.join(tmp, f"synthetic_{name}.bhmm")
        common.concat_models(parts, paths[name], f"synthetic_{name}")
    ctx = capi.Context(0, long_models=True)
    rng = np.random.default_rng(42)
    result = {"device": card(), "points": []}
    for name in sorted(LONG):
        model = po.Model(paths[name])
        M = model.M
        # Forward parser and Forward + Backward (3 codon lengths), windows of 2400 nt
        ctx.load_fs_profile(3, model.rfv(3), model.tfv(3))
        Lw, nwin = 2400, 2048
        ctx.upload_block(common.random_dna(rng, nwin * Lw))
        w = capi.Context.make_windows(1 + np.arange(nwin) * Lw, np.full(nwin, Lw))
        ctx.stage_windows(w)
        for _ in range(2): ctx.fs_fwd_staged()
        t = min((ctx.fs_fwd_staged(), ctx.last_stage_timing()[0])[1] for _ in range(3))
        nb = 1024
        ctx.fs_fwd_bck_xrows(w[:nb])
        tb = min((ctx.fs_fwd_bck_xrows(w[:nb]), ctx.last_stage_timing()[0])[1] for _ in range(2))
        # envelope stage (5 codon lengths): Forward, Backward + decoding + null2, optimal accuracy, traceback; envelopes of 3 M + 300 nt
        ctx.load_fs_profile(5, model.rfv(5), model.tfv(5))
        Le, nenv = 3 * M + 300, 32
        ctx.upload_block(common.random_dna(rng, nenv * Le))
        e = capi.Context.make_windows(1 + np.arange(nenv) * Le, np.full(nenv, Le), nj=0.0)
        steps = nenv * (Le + M + 8)
        ctx.fs_domains(e, xfE5=(1.0, 0.0), max_steps=steps)
        te = min((ctx.fs_domains(e, xfE5=(1.0, 0.0), max_steps=steps), ctx.last_stage_timing()[0])[1] for _ in range(2))
        pt = {"model": name, "M": M,
              "forward_gcups": nwin * Lw * M / t / 1e6, "forward_windows": nwin, "window_nt": Lw,
              "forward_backward_gcups": 2 * nb * Lw * M / tb / 1e6, "forward_backward_windows": nb,
              "envelope_stage_gcups": nenv * Le * M / te / 1e6, "envelopes": nenv, "envelope_nt": Le}
        print(json.dumps(pt), flush=True)
        result["points"].append(pt)
    # search rate: the 2014-node model over target_mbp of iid ACGT, 10 Mbp sequences, both branches of the default (--fs) pipeline
    qm = hostapi.QueryModel(paths["M2014"])
    seqs = [common.random_dna(rng, 10_000_000) for _ in range(int(np.ceil(target_mbp / 10)))]
    warm = hostapi.Search(qm, ctx)
    warm.add_sequence("warm", common.random_dna(rng, 1_000_000))
    warm.finish()
    t0 = time.perf_counter()
    search = hostapi.Search(qm, ctx)
    for z, d in enumerate(seqs):
        search.add_sequence(f"seq{z}", d)
    hits = search.finish()
    dt = time.perf_counter() - t0
    nt = sum(len(d) - 2 for d in seqs)
    result["search"] = {"model": "M2014", "target_mbp": nt / 1e6, "seconds": dt, "mbp_per_s": nt / 1e6 / dt, "hits": len(hits),
                        "stats": {k: (v if isinstance(v, (int, float)) else str(v)) for k, v in search.stats().items()}}
    print(json.dumps(result["search"]), flush=True)
    ctx.close()
    with open(out_path, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
