"""Time gmg_seqset_extract (SeqSet.extract) against the host route a caller had before it: unpack the set, cut and
reverse-complement the regions in numpy, gmg_seqset_create the result.  Device events on the context's stream bracket
every call (both routes end in a stream synchronisation).  Two inputs:

  genes   the 1161 .train regions of NC_000915 (1.67 Mbp genome, 1.0 Mbp of genes)
  large   about 10^6 regions of about 1 kbp, both strands, from a seeded 600 Mbp set (150 MB packed: larger than the
          126 MB L2, so the source is read from HBM)

Prints the card's name and power limit, then one JSON line per input.  The host route's numbers are for one call; the
device route's are the median of --reps calls after one warm-up call."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import glimmer_mg_b200 as g  # noqa: E402
import oracle_lib as O  # noqa: E402  (golden-file reader only)

COMP = bytes.maketrans(b"acgt", b"tgca")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def host_route(ctx, src, reg):
    """unpack -> numpy / bytes -> gmg_seqset_create"""
    raw = src.unpack()
    out = []
    for s, a, n, d in zip(*(x.tolist() for x in reg)):
        x = raw[src.off[s] + a:src.off[s] + a + n]
        out.append(x if d > 0 else x.translate(COMP)[::-1])
    return g.SeqSet(ctx, seqs=out)


def timed(stream, fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    a.record(stream)
    r = fn()
    b.record(stream)
    b.synchronize()
    return r, a.elapsed_time(b), (time.perf_counter() - t0) * 1e3


def run(name, ctx, stream, src, reg, reps):
    out_bases = int(reg[2].astype(np.int64).sum())
    ext, _, _ = timed(stream, lambda: src.extract(*reg))  # warm-up
    ext.close()
    dev = []
    for _ in range(reps):
        ext, ms, _ = timed(stream, lambda: src.extract(*reg))
        dev.append(ms)
        ext.close()
    host, host_ms, host_wall = timed(stream, lambda: host_route(ctx, src, reg))
    ext = src.extract(*reg)
    # the host route complements after Filter: it differs where a minus region holds a non-acgt byte
    differ = int(np.count_nonzero(np.frombuffer(ext.unpack(), np.uint8) != np.frombuffer(host.unpack(), np.uint8)))
    ext.close()
    host.close()
    med = float(np.median(dev))
    # bytes the kernels must move at least: the source's packed words of every output base, the output words
    moved = 2 * out_bases / 4
    print(json.dumps({"input": name, "regions": len(reg[0]), "out_bases": out_bases, "source_bases": src.total,
                      "extract_ms_median": round(med, 4), "extract_ms_min": round(min(dev), 4), "reps": reps,
                      "extract_GBps_min_traffic": round(moved / med / 1e6, 1),
                      "host_route_ms": round(host_ms, 2), "host_route_wall_ms": round(host_wall, 2),
                      "speedup": round(host_ms / med, 1), "bases_differing_from_host_route": differ}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--large-mbp", type=int, default=600)
    ap.add_argument("--regions", type=int, default=1000000)
    args = ap.parse_args()
    print("card:", card(), flush=True)
    stream = torch.cuda.Stream()
    ctx = g.Context(0, stream.cuda_stream)

    genome = O.read_fasta(os.path.join(O.GOLDEN, "NC_000915.fna.gz"))[0][1]
    src = g.SeqSet(ctx, seqs=[genome])
    reg = g.regions_from_coords([h for h, _ in O.read_fasta(os.path.join(O.GOLDEN, "NC_000915.train.gz"))])
    run("genes", ctx, stream, src, reg, args.reps)
    src.close()

    rng = np.random.default_rng(2026)
    n_seq = 64
    total = args.large_mbp * 1000000
    off = np.linspace(0, total, n_seq + 1).astype(np.int64)
    ascii = np.frombuffer(b"acgt", np.uint8)[rng.integers(0, 4, total, dtype=np.uint8)]
    ascii[rng.integers(0, total, total // 10000)] = ord("n")  # one IUPAC code per 10 kbp
    src = g.SeqSet(ctx, ascii=ascii, offsets=off)
    del ascii
    n = args.regions
    seq = rng.integers(0, n_seq, n).astype(np.int32)
    length = rng.integers(500, 1500, n).astype(np.int32)
    lo = (rng.random(n) * (np.diff(off)[seq] - length)).astype(np.int32)
    strand = rng.choice(np.array([-1, 1], np.int8), n)
    run("large", ctx, stream, src, (seq, lo, length, strand), max(3, args.reps // 4))
    src.close()
    ctx.close()


if __name__ == "__main__":
    main()
