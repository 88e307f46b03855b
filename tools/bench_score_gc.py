"""Time glimmer-mg scoring with a per-read independent model (gmg_score_orfs_mg_gc, what glimmer-mg -c needs) against the
single-model call and against the per-read loop of the existing API that -c has to use without it.

Input: seeded reads of the reads100 shape (312 500 x 100 bp, lower-case acgt), one gene ICM trained on the device from the
golden cluster-4 gene set (12/7/3, build-icm -r), ORFs found on the device.  Per mode (plain, -i):
  (a) single_ms        gmg_score_orfs_mg with the set's GC fraction
  (b) same_gc_ms       gmg_score_orfs_mg_gc with that GC value for every read
  (c) distinct_gc_ms   gmg_score_orfs_mg_gc with a distinct seeded GC value (and ignore length) for every read
  (d) loop_ms_per_read the per-read loop of the existing API (create, set_orfs, Build_Indep_WO_Stops, score_orfs_mg,
                       get_starts, free) over the first --loop reads, per read; loop_ms_312500 scales it to the batch
Times are host-clock medians over --reps calls after one warm-up call; every call returns synchronised (the start count
comes back).  Prints the card's name, power limit and SM clocks first, then one JSON line per mode."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import glimmer_mg_b200 as g  # noqa: E402
import oracle_lib as O  # noqa: E402  (golden file reader)
from test_gpu_score_gc import seeded_reads  # noqa: E402  (the tests' read generator)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip().replace("\n", " | ")


def median_ms(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=312_500)
    ap.add_argument("--len", type=int, default=100)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--loop", type=int, default=2000)
    ap.add_argument("--out", default=None, help="also append the lines to this file")
    a = ap.parse_args()
    lines = [f"# card: {card()}"]
    print(lines[0], flush=True)
    ctx = g.Context(0)
    genes = [s for _, s in O.read_fasta(os.path.join(ROOT, "tests", "golden", "seqs.cluster-4.run1.filt.gene.fasta.gz"))]
    gene = g.ICMTraining(ctx).Train_Model(genes, reverse=True)
    reads, _ = seeded_reads(a.reads, a.len, 2026)
    ss = g.SeqSet(ctx, seqs=reads)
    gc = ss.gc_fraction()
    gcs = np.random.default_rng(5).uniform(0.25, 0.75, a.reads)
    for name, flags in (("plain", {}), ("indels", {"allow_indels": 1})):
        p = g.Params(True, **flags)
        p.set_ignore_score_len(gc)
        isl = np.array([g.lib().gmg_ignore_score_len(float(x), p.c) for x in gcs], np.int32)
        ss.find_orfs(p)
        orfs, ooff = ss.get_orfs()
        indep = g.ICM.Build_Indep_WO_Stops(ctx, gc)
        same = np.full(a.reads, gc)
        t_a = median_ms(lambda: ss.score_orfs_mg(gene, indep, p), a.reps)
        t_b = median_ms(lambda: ss.score_orfs_mg_gc(gene, same, p), a.reps)
        t_c = median_ms(lambda: ss.score_orfs_mg_gc(gene, gcs, p, isl), a.reps)
        flagged = ctx.indep_flagged
        launches = ctx.launches
        ss.score_orfs_mg_gc(gene, gcs, p, isl)
        launches = ctx.launches - launches
        n = min(a.loop, a.reads)

        def loop():
            for i in range(n):
                one = g.SeqSet(ctx, seqs=[reads[i]])
                one.set_orfs(orfs[ooff[i]:ooff[i + 1]], np.array([0, ooff[i + 1] - ooff[i]], np.int64))
                m = g.ICM.Build_Indep_WO_Stops(ctx, float(gcs[i]))
                p.c.ignore_score_len = int(isl[i])
                one.score_orfs_mg(gene, m, p)
                one.get_starts()
                m.close()
                one.close()
        t_d = median_ms(loop, 1) / n
        p.set_ignore_score_len(gc)
        rec = {"mode": name, "reads": a.reads, "len": a.len, "orfs": int(ooff[-1]), "single_ms": round(t_a, 3),
               "same_gc_ms": round(t_b, 3), "distinct_gc_ms": round(t_c, 3), "distinct_over_single": round(t_c / t_a, 2),
               "distinct_gc_launches": launches, "flagged_entries": flagged, "loop_reads": n,
               "loop_ms_per_read": round(t_d, 4), "loop_ms_312500": round(t_d * a.reads, 1),
               "distinct_Gbps": round(a.reads * a.len / (t_c * 1e-3) / 1e9, 2)}
        line = json.dumps(rec)
        print(line, flush=True)
        lines.append(line)
    if a.out:
        with open(a.out, "a") as f:
            f.write("\n".join(lines) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
