"""Batched ICM training against a loop of single-model training, on one GPU.

Workload: M seeded synthetic gene sets (tools/workloads.py `coding`, 1500 stop-free strings x 999 bp = 1.5 Mbp each, codon
table re-weighted by `reweight_gc` to GC fractions linspace(0.30, 0.70, M)), the shape of glimmer-mg's per-cluster gene
models.  Sets this small take the direct counting path; the saving batching can bring is in level round trips and
flagged-node synchronisations, so it is measured over the number of models.

Library timing: one process, the sets uploaded once; per repeat, a loop of ICMTraining.Train_Model over the sets and one
Train_Models call over the same sets, alternating, both warmed up first.  Every model's bytes are compared between the
two.  "counted Gbp/s" = training bases x (depth + 1) tree levels / wall time (every level walks every window once).
Command-line timing (--cli-max): M separate `build-icm -r` processes against one `build-icm -r -B list`, wall clock.
The card's name and power limit are read in the same run and printed with the numbers, one JSON line per measurement.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import workloads as W  # noqa: E402

SEED = 9100


def gene_sets(m):
    out = []
    for k, gc in enumerate(np.linspace(0.30, 0.70, m)):
        ts, toff = W.coding(1500, 333, seed=SEED + k, freq=W.reweight_gc(W.codon_freq(), float(gc)))
        out.append((ts, toff))
    return out


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def library(g, ctx, sets, shape, repeats):
    ss = [g.SeqSet(ctx, ascii=a, offsets=o) for a, o in sets]
    tr = g.ICMTraining(ctx, *shape)
    bases = sum(s.total for s in ss)

    def loop():
        return [tr.Train_Model(s, reverse=True) for s in ss]

    def batch():
        return tr.Train_Models(ss, reverse=True)

    loop(), batch()  # warm-up: modules, pools, pinned staging
    t_loop, t_batch, l_loop, l_batch = [], [], [], []
    for _ in range(repeats):
        for fn, ts, ls in ((loop, t_loop, l_loop), (batch, t_batch, l_batch)):
            ctx.sync()
            l0 = ctx.launches
            t0 = time.perf_counter()
            models = fn()
            ctx.sync()
            ts.append(time.perf_counter() - t0)
            ls.append(ctx.launches - l0)
            if fn is loop:
                want = [m.image() for m in models]
            else:
                got = [m.image() for m in models]
            del models
        assert got == want, "a batched model differs from its single-model training"
    m = len(sets)
    row = {"models": m, "shape": "/".join(map(str, shape)), "bases": bases}
    for name, ts, ls in (("loop", t_loop, l_loop), ("batch", t_batch, l_batch)):
        med = float(np.median(ts))
        row[name] = {"ms_per_model": 1e3 * med / m, "ms_per_call": 1e3 * med, "counted_gbps": bases * (shape[1] + 1) / med / 1e9,
                     "launches_per_call": ls[-1], "spread_pct": 100.0 * (max(ts) - min(ts)) / med, "times_s": ts}
    row["speedup"] = float(np.median(t_loop) / np.median(t_batch))
    row["bytes_identical"] = True
    return row


def cli(sets, shape, tmp):
    exe = os.path.join(ROOT, "glimmer_mg_b200", "host", "bin", "build-icm")
    opts = ["-r", "-w", str(shape[0]), "-d", str(shape[1]), "-p", str(shape[2])]
    files = []
    for k, (a, o) in enumerate(sets):
        f = os.path.join(tmp, f"in{k}.fa")
        W.write_fasta(f, a, o, prefix="g")
        files.append(f)
    t0 = time.perf_counter()
    for k, f in enumerate(files):
        with open(f, "rb") as fin:
            subprocess.run([exe, *opts, os.path.join(tmp, f"single{k}.icm")], stdin=fin, check=True)
    t_single = time.perf_counter() - t0
    with open(os.path.join(tmp, "list"), "w") as fp:
        for k, f in enumerate(files):
            fp.write(f"{f} {os.path.join(tmp, f'batch{k}.icm')}\n")
    t0 = time.perf_counter()
    subprocess.run([exe, *opts, "-B", os.path.join(tmp, "list")], check=True, stdin=subprocess.DEVNULL)
    t_batch = time.perf_counter() - t0
    same = all(open(os.path.join(tmp, f"single{k}.icm"), "rb").read() == open(os.path.join(tmp, f"batch{k}.icm"), "rb").read()
               for k in range(len(files)))
    assert same, "build-icm -B wrote a model that differs from the single run's"
    return {"models": len(sets), "shape": "/".join(map(str, shape)), "processes_s": t_single, "batch_s": t_batch,
            "speedup": t_single / t_batch, "bytes_identical": same}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--models", default="16,128,512")
    ap.add_argument("--shapes", default="12/7/3,12/7/1")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--cli-max", type=int, default=128, help="command-line timing for M up to this (0: none)")
    args = ap.parse_args()
    import glimmer_mg_b200 as g
    ctx = g.Context(0)
    gpu = card()
    shapes = [tuple(int(x) for x in s.split("/")) for s in args.shapes.split(",")]
    for m in [int(x) for x in args.models.split(",")]:
        sets = gene_sets(m)
        for shape in shapes:
            print(json.dumps({"kind": "library", "gpu": gpu, **library(g, ctx, sets, shape, args.repeats)}), flush=True)
        if m <= args.cli_max:
            with tempfile.TemporaryDirectory() as tmp:
                print(json.dumps({"kind": "cli", "gpu": gpu, **cli(sets, shapes[0], tmp)}), flush=True)


if __name__ == "__main__":
    main()
