"""Time gmg_seqset_from_fastq (SeqSet.from_fastq) against the host route a caller had before it: split the FASTQ image on
the host into a FASTA image and a quality-file image (numpy; tests/test_gpu_fastq.host_images), then gmg_seqset_from_fasta
and gmg_seqset_quality_from_fasta.  Every image lives in page-locked memory (gmg_host_alloc).  Two shapes of seeded reads
(Phred 0-40, offset 33): 312 500 x 100 bp (the size of bench.py's reads100 set) and 10^6 x 150 bp.

Reported per shape, as medians over --reps calls after one warm-up call:
  call_ms        host clock around the C-ABI call (it returns synchronised): what a caller waits for
  device_ms      CUDA events on the context's stream around the same call
  h2d_ms         host clock around a plain H2D copy of the same pinned image (cudaMemcpyAsync + synchronise)
  *_GBps         image bytes over those times
  python_ms      SeqSet.from_fastq, which also decodes every header into a Python string (one call)
  host route     conversion, from_fasta and quality_from_fasta (host clock), and their sum
Prints the card's name, power limit and SM clocks first, then one JSON line per shape."""
import argparse
import ctypes as C
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
from test_gpu_fastq import host_images, seeded_fastq  # noqa: E402  (the tests' host route and read generator)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip().replace("\n", " | ")


def pinned_copy(ctx, name, data):
    buf = ctx.pinned(name, len(data), np.uint8)
    buf[:] = np.frombuffer(data, np.uint8)
    return buf


def timed(stream, fn):
    """-> (result, host ms, device ms) of a call that ends synchronised"""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    t0 = time.perf_counter()
    r = fn()
    t1 = time.perf_counter()
    b.record(stream)
    b.synchronize()
    return r, (t1 - t0) * 1e3, a.elapsed_time(b)


def from_fastq(ctx, buf):
    h, n = C.c_void_p(), C.c_int64()
    if g.lib().gmg_seqset_from_fastq(ctx.h, buf.ctypes.data, len(buf), 33, C.byref(h), C.byref(n)):
        raise g.GmgError(g.lib().gmg_last_error().decode())
    return h


def from_fasta(ctx, fasta):
    h, n = C.c_void_p(), C.c_int64()
    if g.lib().gmg_seqset_from_fasta(ctx.h, fasta.ctypes.data, len(fasta), C.byref(h), C.byref(n)):
        raise g.GmgError(g.lib().gmg_last_error().decode())
    return h


def set_quality(ctx, h, qual):
    if g.lib().gmg_seqset_quality_from_fasta(ctx.h, h, qual.ctypes.data, len(qual)):
        raise g.GmgError(g.lib().gmg_last_error().decode())


def run(name, ctx, stream, n_reads, length, reps):
    image = seeded_fastq(n_reads, length, 2026)
    buf = pinned_copy(ctx, "fastq", image)
    dev = torch.empty(len(buf), dtype=torch.uint8, device="cuda")
    n = len(buf)

    def h2d():
        if g.lib().gmg_ctx_memcpy_h2d(ctx.h, C.c_void_p(dev.data_ptr()), buf.ctypes.data, n):
            raise g.GmgError(g.lib().gmg_last_error().decode())

    call, call_dev, copy = [], [], []
    for k in range(reps + 1):  # alternate the two so that both see the same conditions; call 0 warms up
        h, ms, dms = timed(stream, lambda: from_fastq(ctx, buf))
        g.lib().gmg_seqset_free(h)
        _, cms, _ = timed(stream, h2d)
        if k:
            call.append(ms)
            call_dev.append(dms)
            copy.append(cms)
    t0 = time.perf_counter()
    got = g.SeqSet.from_fastq(ctx, buf)
    python_ms = (time.perf_counter() - t0) * 1e3

    t0 = time.perf_counter()
    fasta_img, qual_img, _ = host_images(image)
    convert_ms = (time.perf_counter() - t0) * 1e3
    fasta, qual = pinned_copy(ctx, "fasta", fasta_img), pinned_copy(ctx, "qual", qual_img)
    hf, hq, h = [], [], None
    for k in range(max(1, reps // 4) + 1):  # call 0 warms up
        if h is not None:
            g.lib().gmg_seqset_free(h)
        h, fms, _ = timed(stream, lambda: from_fasta(ctx, fasta))
        _, qms, _ = timed(stream, lambda: set_quality(ctx, h, qual))
        if k:
            hf.append(fms)
            hq.append(qms)
    want = g.SeqSet._adopt(ctx, h)
    identical = bool((got.off == want.off).all() and got.unpack() == want.unpack()
                     and (got.qualities() == want.qualities()).all())
    got.close()
    want.close()
    med = lambda x: float(np.median(x))  # noqa: E731
    call_ms, dev_ms, h2d_ms = med(call), med(call_dev), med(copy)
    host_ms = convert_ms + med(hf) + med(hq)
    print(json.dumps({
        "input": name, "records": n_reads, "bases": n_reads * length, "image_bytes": n,
        "fasta_image_bytes": len(fasta_img), "quality_image_bytes": len(qual_img), "reps": reps,
        "call_ms": round(call_ms, 3), "call_ms_min": round(min(call), 3), "device_ms": round(dev_ms, 3),
        "h2d_ms": round(h2d_ms, 3), "call_GBps": round(n / call_ms / 1e6, 2), "h2d_GBps": round(n / h2d_ms / 1e6, 2),
        "call_over_h2d": round(call_ms / h2d_ms, 2), "python_ms": round(python_ms, 1),
        "host_convert_ms": round(convert_ms, 1), "host_from_fasta_ms": round(med(hf), 3),
        "host_quality_ms": round(med(hq), 3), "host_route_ms": round(host_ms, 1),
        "speedup_vs_host_route": round(host_ms / call_ms, 1), "identical_to_host_route": identical}), flush=True)
    del dev


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    print("card:", card(), flush=True)
    stream = torch.cuda.Stream()
    ctx = g.Context(0, stream.cuda_stream)
    run("reads100_size", ctx, stream, 312500, 100, args.reps)
    run("1M_x_150bp", ctx, stream, 1000000, 150, args.reps)
    print("card after:", card(), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
