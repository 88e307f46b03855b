#!/usr/bin/env python
"""bench.py -- ICM-scored Gbp/s of the B200 hot path, next to the CPU reference.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload NAME] [--dump-outputs DIR]

Default workload ``reads100`` = BASELINE.json configs[4], the sharded read set north_star's scaling target names
(SURVEY.md section 8(d) config 5): 16 synthetic genomes (GC 0.30..0.70) with their own ICMs trained on the device,
625 000 error-free 100 bp reads each (seed 5); a "step" is one half-cluster batch of 312 500 reads (31.25 Mbp)
through the glimmer-mg scoring half (K1 six-frame walks, K2 prefix sums / stop tables, K3 start enumeration) with
its cluster's ICM; rank r takes batches r, r+N, ... (no collective: reads never interact).  It fits one GPU, so the
N=1 line and the 1/2/4/8 scaling lines measure the same thing.  A default run (no --workload) also runs the other
BASELINE configs with fewer steps and nests their lines under "extra": contig5m (configs[1], glimmer3 whole-genome
half), train500m (configs[3], build-icm with the per-level count exchange) and reads400 (configs[2], glimmer-mg -i).

  value  whole-job Gbp/s with the packed batch and its ORF table already resident in HBM, CUDA events on the
         launching stream, L2 flushed (256 MB write) before every step, max over ranks.
  e2e    the same metric through the C-ABI call sequence a host makes with HOST buffers: pinned ASCII ->
         gmg_seqset_create (H2D + Filter / 2-bit pack) -> gmg_find_orfs -> gmg_score_orfs_* -> gmg_get_orfs +
         gmg_get_starts (D2H), copies inside the timed region.
  roofline   the dominant streaming kernel of the workload: algorithmic HBM bytes per launch (DESIGN.md section 3)
         divided by its CUDA-event duration measured live in the timed region (gmg_ctx_profile).
  parity_checked / parity   the results of the last end-to-end step compared with the oracle port (tests/config_parity.py)
         OUTSIDE the timed region: ORF tables, start lists incl. FP64 score bits, model files.  A difference aborts
         the run -- a number without parity is not printed.
  cpu_baseline   the unmodified reference binary (oracle/_ref, built from /root/reference by oracle/Makefile) on a
         bounded sample of the same workload on one host core (it is single-threaded).
  e2e_app    whole-application wall time: the reference's own driver compiled over the C-ABI
         (glimmer_mg_b200/host/bin/glimmer3-gmg, glimmer-mg-gmg, build-icm) against the unmodified binary on the same
         input file, outputs compared byte for byte.

``--impl reference`` times the reference's own CPU implementation with every host core: one process per core, each
on its own bounded slice of the workload (the reference's only parallelism is process-per-sequence-set,
scripts/train_all.py:58).
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

METRIC = "ICM-scored Gbp/s"
UNIT = "Gbp/s"
CONTIG_LEN = 5_000_000
K1_BYTES_PER_BASE = 0.25 + 6 * 4  # packed read + six float planes written (DESIGN.md, K1)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)  # a 0.25 ms step: 100 of them average out host jitter
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=None, choices=["contig5m", "reads400", "reads100", "train500m", "simplescore"],
                    help="default: reads100 (BASELINE.json configs[4], the sharded read set north_star's scaling target names), "
                         "with the contig5m / train500m / reads400 lines of the same run nested under \"extra\"")
    ap.add_argument("--no-extra", action="store_true", help="default workload only, no nested lines")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle check of the results (profiling runs)")
    ap.add_argument("--no-pipeline", action="store_true", help="end to end with one batch at a time only")
    ap.add_argument("--scale", type=float, default=1.0,
                    help="shrink a non-default workload (fraction of its reads / training strings); 1.0 = BASELINE size")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="b200 arm only: after the timed steps, write what the last timed step of the workload computed "
                         "(rank 0) as DIR/<name>.npy, float32 / float64, at most 64 MB in all, so that two builds can be "
                         "compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm; the reference arm keeps none")
    return args


DUMP_BYTES = 64 << 20
DUMP_SEED = 20261020


def dump_outputs(dirname, arrays):
    """{name: array} -> dirname/<name>.npy; float32 stays float32, everything else is widened to float64 (exact for the
    int16 / int32 / int64 fields written here)."""
    import numpy as np
    arrays = {name: np.ascontiguousarray(a) for name, a in arrays.items()}
    arrays = {name: a if a.dtype == np.float32 else a.astype(np.float64) for name, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:  # the whole-call tables are not sampled: only a workload far beyond BASELINE size gets here
        raise SystemExit(f"bench.py: --dump-outputs: {total} bytes exceed the {DUMP_BYTES}-byte limit")
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


def seeded_sample(n, fits):
    """Indices of a fixed, seeded sample of n items: all of them if fits(all), else the first half, quarter, ... of one
    seeded permutation until fits(sample), down to none -- the same sample on every run with the same n."""
    import numpy as np
    idx = np.arange(n)
    if fits(idx):
        return idx
    perm = np.random.default_rng(DUMP_SEED).permutation(n)
    m = n // 2
    while m > 0 and not fits(np.sort(perm[:m])):
        m //= 2
    return np.sort(perm[:m])


def scoring_outputs(orfs, ooff, starts, soff):
    """What a caller of the scoring half receives (ORF table + per-ORF start lists) as float64 tables: every ORF and
    start when they fit DUMP_BYTES, else a seeded sample of ORFs with their complete start lists.
      counts        [sequences, ORFs, starts] of the whole call
      orf_counts    ORFs per sequence; start_counts  starts per ORF (whole call)
      orfs          sampled ORFs: index, sequence, frame, stop_position, orf_len, gene_len
      starts        their starts: ORF index, j, pos, score, which, truncated, first, n_err, err_pos[2], err_type[2]"""
    import numpy as np
    ooff, soff = np.asarray(ooff, np.int64), np.asarray(soff, np.int64)
    n_orfs = len(orfs)
    per_orf = np.diff(soff)
    fixed = 8 * (3 + len(ooff) - 1 + n_orfs)
    pick = seeded_sample(n_orfs, lambda ids: fixed + 8 * (6 * len(ids) + 12 * int(per_orf[ids].sum())) <= DUMP_BYTES)
    seq = np.searchsorted(ooff, pick, side="right") - 1
    o = orfs[pick]
    orf_tab = np.stack([pick, seq, o["frame"], o["stop_position"], o["orf_len"], o["gene_len"]], axis=1).astype(np.float64)
    lens = per_orf[pick]
    owner = np.repeat(pick, lens)
    rows = np.repeat(soff[pick], lens) + np.arange(int(lens.sum())) - np.repeat(np.cumsum(lens) - lens, lens)
    s = starts[rows]
    start_tab = np.column_stack([owner, s["j"], s["pos"], s["score"], s["which"], s["truncated"], s["first"], s["n_err"],
                                 s["err_pos"], s["err_type"]]).astype(np.float64)
    return {"counts": np.array([len(ooff) - 1, n_orfs, len(starts)], np.float64), "orf_counts": np.diff(ooff),
            "start_counts": per_orf, "orfs": orf_tab, "starts": start_tab}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fp:
            return float(json.load(fp)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(kernel, units):
    """DRAM bytes per launch of `kernel` from the committed ncu capture, scaled to this launch's units."""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as fp:
            t = json.load(fp)[kernel]
        return t["dram_bytes_per_unit"] * units
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons of one GPU during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 - 0.05 <= t <= t1 + 0.15] or [r for _, r in self.rows]
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except Exception:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


class Env:
    """Per-process CUDA / torch.distributed state shared by every workload of one bench.py run."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)  # > 126 MB L2

    def barrier(self):
        import torch
        import torch.distributed as dist
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def close(self):
        import torch.distributed as dist
        if self.world > 1:
            dist.destroy_process_group()


def parity_mod():
    """The checker (tests/config_parity.py over the oracle port); only ever called outside timed regions."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import config_parity as CP
    return CP


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def ref_bin(name):
    """oracle/_ref/bin: the unmodified reference; glimmer_mg_b200/host/bin: its drivers compiled over the C-ABI (*-gmg)."""
    d = os.path.join(ROOT, "glimmer_mg_b200", "host", "bin") if name.endswith("-gmg") else os.path.join(ROOT, "oracle", "_ref", "bin")
    p = os.path.join(d, name)
    return p if os.path.exists(p) else None


def run_glimmer3_procs(fastas, workdir):
    """Run one reference glimmer3 per FASTA concurrently; returns wall seconds."""
    import workloads as W
    exe = ref_bin("glimmer3")
    t0 = time.perf_counter()
    procs = [subprocess.Popen([exe, "-u", "-12", "-m", W.gene_model_path(), fa, os.path.join(workdir, f"out{i}")],
                              stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, cwd=workdir)
             for i, fa in enumerate(fastas)]
    for p in procs:
        if p.wait() != 0:
            raise RuntimeError("reference glimmer3 failed")
    return time.perf_counter() - t0


def port_scoring_seconds(contig_bytes):
    """The oracle port (oracle/icm_oracle.c): Find_Orfs + Score_Orfs start enumeration only, 1 thread."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    import workloads as W
    og = O.lib().orc_icm_read(W.gene_model_path().encode())
    s = bytes(contig_bytes)
    gc = (s.count(b"c") + s.count(b"g")) / len(s)
    oi = O.build_indep(gc)
    op = O.params(False)
    t0 = time.perf_counter()
    orfs = O.find_orfs(s, op)
    O.g3_score_orfs(og, oi, s, op, orfs)
    return time.perf_counter() - t0


def cpu_baseline(contig_arr):
    """cpu_baseline leg of the b200 arm: the whole contig, one reference process (single-threaded binary)."""
    import workloads as W
    tmp = tempfile.mkdtemp(prefix="gmg_bench_")
    try:
        if ref_bin("glimmer3"):
            fa = os.path.join(tmp, "contig.fa")
            W.write_fasta(fa, contig_arr, prefix="contig")
            sec = run_glimmer3_procs([fa], tmp)
            out = {"value": len(contig_arr) / sec / 1e9, "unit": UNIT, "cores": 1, "kind": "reference",
                   "sample": f"the full {len(contig_arr)} bp contig through the unmodified glimmer3 binary "
                             f"(-u -12 -m; FASTA read + Find_Orfs + Score_Orfs + event DP + .predict), {sec:.2f} s"}
            n = min(len(contig_arr), 1_000_000)
            psec = port_scoring_seconds(contig_arr[:n].tobytes())
            out["port_scoring_only"] = {"value": n / psec / 1e9, "unit": UNIT, "cores": 1,
                                        "sample": f"oracle port, Find_Orfs + Score_Orfs start lists only, first {n} bp"}
            return out
        n = min(len(contig_arr), 2_000_000)
        sec = port_scoring_seconds(contig_arr[:n].tobytes())
        return {"value": n / sec / 1e9, "unit": UNIT, "cores": 1, "kind": "port",
                "sample": f"oracle port (Find_Orfs + Score_Orfs start lists), first {n} bp of the contig, {sec:.2f} s"}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def _timed(cmd, stdin_path=None, cwd=None):
    fin = open(stdin_path, "rb") if stdin_path else None
    t0 = time.perf_counter()
    try:
        rc = subprocess.run(cmd, stdin=fin, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, cwd=cwd).returncode
    finally:
        if fin:
            fin.close()
    if rc != 0:
        raise RuntimeError(f"{cmd[0]} failed (exit {rc})")
    return time.perf_counter() - t0


def _app_pair(ref_exe, gmg_exe, args_of, files, what, bases, stdin_path=None):
    """Wall time of the whole APPLICATION: the unmodified reference binary against the same driver compiled over
    the C-ABI (process start, CUDA context creation, file I/O, host DP and output included), same input file,
    output files compared byte for byte.  `args_of(tag)` -> argument list writing output files `files(tag)`."""
    if not (ref_exe and gmg_exe and os.path.exists(ref_exe) and os.path.exists(gmg_exe)):
        return {"unavailable": "drop-in or reference binary not built (needs the reference checkout at build time)"}
    _timed([gmg_exe, *args_of("warm")], stdin_path)  # first CUDA context of this process tree: driver / module load
    t_ref = _timed([ref_exe, *args_of("ref")], stdin_path)
    t_gmg = min(_timed([gmg_exe, *args_of("gmg")], stdin_path) for _ in range(2))
    same = all(open(a, "rb").read() == open(b, "rb").read() for a, b in zip(files("ref"), files("gmg")))
    return {"what": what, "reference_s": t_ref, "b200_s": t_gmg, "speedup": t_ref / t_gmg, "bases": int(bases),
            "reference_gbps": bases / t_ref / 1e9, "b200_gbps": bases / t_gmg / 1e9, "outputs_identical": bool(same)}


def app_glimmer3(contig_arr):
    import workloads as W
    tmp = tempfile.mkdtemp(prefix="gmg_app_")
    try:
        fa = os.path.join(tmp, "contig.fa")
        W.write_fasta(fa, contig_arr, prefix="contig")
        return _app_pair(ref_bin("glimmer3"), ref_bin("glimmer3-gmg"),
                         lambda tag: ["-u", "-12", "-m", W.gene_model_path(), fa, os.path.join(tmp, tag)],
                         lambda tag: [os.path.join(tmp, tag + ".predict")],
                         "glimmer3 -u -12 -m NC_000915.icm on the contig's FASTA file -> .predict, whole process wall time; "
                         "b200 = the reference's own driver with Score_Orfs bound to gmg_score_orfs_g3", len(contig_arr))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def app_glimmer_mg(ascii_arr, off, n_reads, flags, model_path):
    import workloads as W
    tmp = tempfile.mkdtemp(prefix="gmg_app_")
    try:
        fa = os.path.join(tmp, "reads.fa")
        W.write_fasta(fa, ascii_arr[:off[n_reads]], off[:n_reads + 1], prefix="r")
        return _app_pair(ref_bin("glimmer-mg"), ref_bin("glimmer-mg-gmg"),
                         lambda tag: ["-u", "1.0", *flags, "-m", model_path, fa, os.path.join(tmp, tag)],
                         lambda tag: [os.path.join(tmp, tag + ".predict")],
                         f"glimmer-mg -u 1.0 {' '.join(flags)} -m <icm> on the first {n_reads} reads of the batch (FASTA file) -> "
                         f".predict, whole process wall time", int(off[n_reads]))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def app_build_icm(ascii_arr, off):
    import workloads as W
    tmp = tempfile.mkdtemp(prefix="gmg_app_")
    try:
        fa = os.path.join(tmp, "train.fa")
        W.write_fasta(fa, ascii_arr, off, prefix="g")
        ours = os.path.join(ROOT, "glimmer_mg_b200", "host", "bin", "build-icm")
        return _app_pair(ref_bin("build-icm"), ours, lambda tag: ["-r", os.path.join(tmp, tag + ".icm")],
                         lambda tag: [os.path.join(tmp, tag + ".icm")],
                         f"build-icm -r < {len(off) - 1} training strings (FASTA on stdin) -> model file, whole process wall "
                         f"time; b200 = glimmer_mg_b200/host/bin/build-icm", int(off[-1]), stdin_path=fa)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


# ---------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import workloads as W
    cores = host_cores()
    # bounded sample per step: the whole --steps K --warmup W run stays around a minute (0.8 us per base and core)
    slice_len = max(50_000, min(500_000, int(75e6 / max(1, args.steps + args.warmup))))
    tmp = tempfile.mkdtemp(prefix="gmg_ref_")
    try:
        kind = "reference" if ref_bin("glimmer3") else "port"
        n_contigs = max(1, args.gpus)
        contigs = [W.contig(W.CONTIG_SEED + r, CONTIG_LEN) for r in range(n_contigs)]
        slices = []
        for i in range(cores):  # distinct slices, round-robin over the job's contigs
            c = contigs[i % n_contigs]
            a = ((i // n_contigs) * slice_len) % (len(c) - slice_len)
            slices.append(c[a:a + slice_len])
        times = []
        if kind == "reference":
            fastas = []
            for i, s in enumerate(slices):
                fa = os.path.join(tmp, f"slice{i}.fa")
                W.write_fasta(fa, s, prefix="slice")
                fastas.append(fa)
            for k in range(args.warmup + args.steps):
                sec = run_glimmer3_procs(fastas, tmp)
                if k >= args.warmup:
                    times.append(sec)
        else:
            cores = 1
            for k in range(args.warmup + args.steps):
                sec = port_scoring_seconds(slices[0].tobytes())
                if k >= args.warmup:
                    times.append(sec)
        bases = slice_len * (len(slices) if kind == "reference" else 1)
        total = sum(times)
        value = bases * len(times) / total / 1e9
        sample = (f"each step: {cores} concurrent glimmer3 processes (one per host core), each on its own "
                  f"{slice_len} bp slice of the workload contig(s)" if kind == "reference" else
                  f"each step: oracle port on one {slice_len} bp slice, 1 thread")
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "impl": "reference",
                "config": {"workload": "contig5m: synthetic 5 Mbp bacterial contig per GPU, glimmer3 whole-genome "
                                       "scoring (BASELINE.json configs[1])", "model": "tests/golden/NC_000915.icm"},
                "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
                "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line), flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


# ---------------------------------------------------------------------------------------------------
def run_b200(args, env):
    import numpy as np
    import torch
    import torch.distributed as dist
    import glimmer_mg_b200 as g
    import workloads as W

    rank, world, local, dev, barrier = env.rank, env.world, env.local, env.dev, env.barrier

    stream = torch.cuda.Stream(device=dev)
    K, Wu = args.steps, max(args.warmup, 3)
    with torch.cuda.stream(stream):
        ctx = g.Context(local, stream.cuda_stream)
        contig = W.contig(W.CONTIG_SEED + rank, CONTIG_LEN)
        n = len(contig)
        h_ascii = torch.empty(n, dtype=torch.uint8).pin_memory()
        h_ascii.numpy()[:] = contig
        off = np.array([0, n], np.int64)
        gene = g.ICM.Read(ctx, W.gene_model_path())
        flush = env.flush

        # ---- resident phase: packed contig + ORF table live in HBM ----
        ss = g.SeqSet(ctx, ascii=h_ascii.numpy(), offsets=off)
        gc = ss.gc_fraction()
        p = g.Params(False)
        p.set_ignore_score_len(gc)
        indep = g.ICM.Build_Indep_WO_Stops(ctx, gc, p.stop_codons)
        n_orfs = ss.find_orfs(p)
        for _ in range(Wu):
            ss.score_orfs_g3(gene, indep, p)
        ctx.sync()
        ctx.profile(True)
        for k in ("k1", "k3", "orf", "pack"):
            ctx.profile_read(k)
        e0 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
        e1 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
        clocks = ClockSampler(local) if rank == 0 else None
        barrier()
        launches0 = ctx.launches
        t_wall0 = time.time()
        for k in range(K):
            flush.zero_()
            e0[k].record(stream)
            n_starts = ss.score_orfs_g3(gene, indep, p)
            e1[k].record(stream)
        barrier()
        t_wall1 = time.time()
        launches = ctx.launches - launches0
        ms = sum(a.elapsed_time(b) for a, b in zip(e0, e1))
        k1_ms, k1_n = ctx.profile_read("k1")
        k3_ms, k3_n = ctx.profile_read("k3")
        clk = clocks.stop(t_wall0, t_wall1) if clocks else None
        if rank == 0 and args.dump_outputs:
            dump_outputs(args.dump_outputs, scoring_outputs(*ss.get_orfs(), *ss.get_starts()))

        # ---- end to end: host ASCII in, ORFs + start lists out ----
        e2e_ms = 0.0
        d2h = 0
        for k in range(Wu + K):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record(stream)
            s2 = g.SeqSet(ctx, ascii=h_ascii.numpy(), offsets=off)
            s2.find_orfs(p)
            s2.score_orfs_g3(gene, indep, p)
            orfs, ooff = s2.get_orfs(pinned=True)
            starts, soff = s2.get_starts(pinned=True)
            b.record(stream)
            torch.cuda.synchronize()
            if k >= Wu:
                e2e_ms += a.elapsed_time(b)
                d2h = orfs.nbytes + ooff.nbytes + starts.nbytes + soff.nbytes
            if k + 1 < Wu + K:
                s2.close()
        ctx.profile(False)
        # ---- parity (outside the timed region): the last end-to-end step's ORF table and start lists of the WHOLE
        # contig against the oracle port, bit for bit (BASELINE.md section 3)
        parity = None
        if rank == 0 and not args.no_parity:
            CP = parity_mod()
            st = CP.check_scoring("g3", contig, off, [0], orfs, ooff, starts, soff, CP.oracle_model(path=W.gene_model_path()),
                                  gc, p.stop_codons, ignore_score_len=p.ignore_score_len)
            parity = {"checked": "ORF table + start lists (order, j, pos, which, flags, FP64 score bits) of the whole contig "
                                 "identical to the oracle port", **st, "ordered_fallback_orfs": int(s2.ordered_fallbacks)}
        s2.close()

    t = torch.tensor([ms, e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max, e2e_max = t.tolist()
    if rank == 0:
        total_bases = n * world
        value = total_bases * K / (ms_max / 1e3) / 1e9
        e2e = total_bases * K / (e2e_max / 1e3) / 1e9
        peak, peak_src = measured_peak()
        k1_bytes = n * K1_BYTES_PER_BASE
        achieved = k1_bytes / (k1_ms / max(k1_n, 1) / 1e3) / 1e9
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wu,
                "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": "contig5m: synthetic 5 Mbp bacterial contig per GPU (seed 20261017+rank), "
                                       "glimmer3 whole-genome scoring half: K1 six-frame walks + per-ORF start "
                                       "enumeration (BASELINE.json configs[1])",
                           "model": "tests/golden/NC_000915.icm (12/7/3)", "bases_per_gpu": n, "orfs": int(n_orfs),
                           "starts": int(n_starts), "l2": "256 MB flush write before every timed step",
                           "sharding": "one contig per GPU, no collective"},
                "roofline": {"bound": "hbm", "kernel": "k1_planes", "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": achieved / peak, "traffic": ncu_traffic("k1_planes", n),
                             "peak_source": peak_src, "algorithmic_bytes_per_launch": k1_bytes,
                             "kernel_ms": k1_ms / max(k1_n, 1), "kernel_share_of_step": k1_ms / ms,
                             "k3_ms_per_step": k3_ms / K},
                "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(n + off.nbytes),
                        "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_max / K},
                "gpu_launches": int(launches), "clocks": clk,
                "parity_checked": parity is not None, "parity": parity}
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(contig)
            line["e2e_app"] = app_glimmer3(contig)
        return line
    return None


# ===================================================================================================
# The other BASELINE.json configs (parity-test cases at N=1 per the bench contract; selectable with
# --workload so that every SURVEY.md section 8(d) config has a measured line under profiles/).
#   reads400   configs[2]: 1M x 400 bp 454-like reads (seed 42), glimmer-mg -i scoring half; step = one batch
#              of 25 000 reads (10 Mbp); rank r takes batches r, r+N, ...
#   reads100   configs[4]: 16 synthetic genomes (GC 0.30..0.70) with their own device-trained ICMs, 625 000
#              error-free 100 bp reads each (seed 5); step = one half-cluster batch of 312 500 reads
#              (31.25 Mbp) scored with its cluster's ICM; rank r takes batches r, r+N, ...
#   train500m  configs[3]: build-icm -r on 500 500 x 999 bp stop-free coding strings (seed 7), strings dealt
#              round-robin to ranks, every level's count slab all-reduced (NCCL) -- "strong" scaling;
#              step = one full Train_Model.
K2_BYTES_PER_BASE = 24 + 48 + 8 + 1   # planes read; cum doubles, stop tables, quality written (DESIGN.md, K2)
READS400_BATCH, READS400_TOTAL, READS400_LEN = 25_000, 1_000_000, 400
READS100_BATCH, READS100_PER_CLUSTER, READS100_LEN, READS100_CLUSTERS = 312_500, 625_000, 100, 16
TRAIN_SEQS, TRAIN_CODONS = 500_500, 333
MAX_RESIDENT_BATCHES = 8


# Job order of the reads100 workload: batch b (two per cluster) belongs to cluster PERM[(b + 4 (b // 16)) % 16].  The ORF
# density follows the GC content (0.30 .. 0.70 over the clusters; fewer stop codons at high GC), so a job list in GC order
# gives the ranks of a multi-GPU run unlike work -- and the first few batches, all a single GPU keeps resident, are the
# cheapest ones.  With this order the batches a rank is dealt (b = rank + world * i) have the same mean GC at every world
# size: PERM[m] + PERM[m + 8] = 15, every stride-4 quadruple sums to 30, the first eight entries to 60.
READS100_PERM = (0, 14, 2, 12, 11, 5, 9, 7, 15, 1, 13, 3, 4, 10, 6, 8)


def reads100_cluster_of_batch(b):
    return READS100_PERM[(b + 4 * (b // READS100_CLUSTERS)) % READS100_CLUSTERS]


def reads_batches(kind, rank, world, scale, n_wanted):
    """Host data of the batches this rank processes -> list of (ascii, off, model id), plus a description."""
    import numpy as np
    import workloads as W
    out = []
    if kind == "reads400":
        contig = W.contig(W.CONTIG_SEED, CONTIG_LEN)
        per = max(64, int(READS400_BATCH * scale))
        n_batches = READS400_TOTAL // READS400_BATCH
        for i in range(min(n_wanted, MAX_RESIDENT_BATCHES)):
            b = (rank + world * i) % n_batches
            a, off = W.reads(contig, per, READS400_LEN, W.READS400_SEED + 7919 * b, indel=True)
            out.append((a, off, 0))
        desc = (f"reads400: {per} reads x {READS400_LEN} bp per step, 454-like homopolymer indels, drawn from the config-2 "
                f"contig (seed 42 + batch), glimmer-mg -i scoring half: K1 + K2 prefix/stops/quality + K3 indel "
                f"start recursion (BASELINE.json configs[2])")
        return out, desc
    freq = W.codon_freq()
    per = max(64, int(READS100_BATCH * scale))
    n_batches = READS100_CLUSTERS * (READS100_PER_CLUSTER // READS100_BATCH)
    genomes = {}
    for i in range(min(n_wanted, MAX_RESIDENT_BATCHES)):
        b = (rank + world * i) % n_batches
        k = reads100_cluster_of_batch(b)
        if k not in genomes:
            gc = float(np.linspace(0.30, 0.70, READS100_CLUSTERS)[k])
            genomes[k] = W.contig(W.READS100_SEED * 1000 + k, 2_000_000, freq=W.reweight_gc(freq, gc), gc=gc)
        a, off = W.reads(genomes[k], per, READS100_LEN, W.READS100_SEED + 7919 * b, indel=False)
        out.append((a, off, k))
    desc = (f"reads100: {per} error-free reads x {READS100_LEN} bp per step from one of {READS100_CLUSTERS} synthetic genomes "
            f"(GC 0.30..0.70), each scored with its own cluster ICM trained on the device, glimmer-mg scoring half "
            f"(BASELINE.json configs[4])")
    return out, desc


def cluster_training_strings(k):
    """Training genes of cluster k: stop-free coding strings from the genome's re-weighted codon table."""
    import numpy as np
    import workloads as W
    gc = float(np.linspace(0.30, 0.70, READS100_CLUSTERS)[k])
    return W.coding(1500, 333, seed=W.READS100_SEED * 1000 + 500 + k, freq=W.reweight_gc(W.codon_freq(), gc))


def ref_glimmer_mg_seconds(fastas, workdir, flags, models):
    """One reference glimmer-mg per FASTA concurrently; wall seconds of the slowest."""
    exe = ref_bin("glimmer-mg")
    t0 = time.perf_counter()
    procs = [subprocess.Popen([exe, "-u", "1.0", *flags, "-m", models[i], fa, os.path.join(workdir, f"out{i}")],
                              stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, cwd=workdir)
             for i, fa in enumerate(fastas)]
    for p in procs:
        if p.wait() != 0:
            raise RuntimeError("reference glimmer-mg failed")
    return time.perf_counter() - t0


def port_mg_seconds(ascii_arr, off, indels):
    """Oracle port of the glimmer-mg scoring half on a few reads, 1 thread (used when oracle/_ref is absent)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    import workloads as W
    og = O.lib().orc_icm_read(W.gene_model_path().encode())
    s_all = ascii_arr.tobytes()
    gc = (s_all.count(b"c") + s_all.count(b"g")) / max(1, len(s_all))
    oi = O.build_indep(gc)
    op = O.params(True, allow_indels=1 if indels else 0)
    t0 = time.perf_counter()
    for i in range(len(off) - 1):
        s = s_all[off[i]:off[i + 1]]
        O.mg_score_orfs(og, oi, s, op, O.find_orfs(s, op))
    return time.perf_counter() - t0


def reads_cpu_sample(kind, ascii_arr, off, n_reads, tmp, model_path, tag=0):
    import workloads as W
    fa = os.path.join(tmp, f"sample{tag}.fa")
    W.write_fasta(fa, ascii_arr[:off[n_reads]], off[:n_reads + 1], prefix="r")
    return fa


def run_reference_reads(args, kind):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import numpy as np
    import workloads as W
    cores = host_cores()
    n_sample = 1500 if kind == "reads400" else 15000
    n_sample = max(n_sample // 15, min(n_sample, n_sample * 47 // max(1, args.steps + args.warmup)))  # ~ a minute in total
    flags = ["-i"] if kind == "reads400" else []
    tmp = tempfile.mkdtemp(prefix="gmg_ref_")
    try:
        batches, desc = reads_batches(kind, 0, 1, max(args.scale, 1e-9), 1)
        a, off, _ = batches[0]
        have = ref_bin("glimmer-mg") is not None
        fastas, bases = [], 0
        n_avail = len(off) - 1
        n_sample = min(n_sample, n_avail)
        for i in range(cores if have else 1):
            lo = (i * n_sample) % max(1, n_avail - n_sample + 1)
            sa, so = a[off[lo]:off[lo + n_sample]], off[lo:lo + n_sample + 1] - off[lo]
            bases += int(so[-1])
            if have:
                fa = os.path.join(tmp, f"s{i}.fa")
                W.write_fasta(fa, sa, so, prefix="r")
                fastas.append(fa)
            else:
                port_in = (sa, so)
        model_path = W.gene_model_path()
        if have and kind == "reads100" and ref_bin("build-icm"):
            # the cluster's own ICM, trained by the reference's build-icm on the cluster's genes (not timed)
            ts, toff = cluster_training_strings(batches[0][2])
            tfa = os.path.join(tmp, "train.fa")
            W.write_fasta(tfa, ts, toff, prefix="g")
            model_path = os.path.join(tmp, "cluster.icm")
            with open(tfa, "rb") as fin:
                subprocess.run([ref_bin("build-icm"), "-r", model_path], stdin=fin, check=True, stdout=subprocess.DEVNULL,
                               stderr=subprocess.DEVNULL)
        times = []
        for k in range(args.warmup + args.steps):
            sec = (ref_glimmer_mg_seconds(fastas, tmp, flags, [model_path] * len(fastas)) if have
                   else port_mg_seconds(port_in[0], port_in[1], kind == "reads400"))
            if k >= args.warmup:
                times.append(sec)
        value = bases * len(times) / sum(times) / 1e9
        used = cores if have else 1
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "impl": "reference",
                "config": {"workload": desc, "model": "tests/golden/NC_000915.icm" if model_path == W.gene_model_path() else
                           "the cluster's 12/7/3 ICM trained by the reference build-icm -r"},
                "cpu_baseline": {"value": value, "unit": UNIT, "cores": used, "kind": "reference" if have else "port",
                                 "sample": f"each step: {used} concurrent glimmer-mg {' '.join(flags)} processes, each on its own "
                                           f"{n_sample} reads of the workload (FASTA read + scoring + event DP + .predict)"},
                "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line), flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def run_b200_reads(args, env, kind):
    import numpy as np
    import torch
    import torch.distributed as dist
    import glimmer_mg_b200 as g
    import workloads as W

    rank, world, local, dev, barrier = env.rank, env.world, env.local, env.dev, env.barrier

    stream = torch.cuda.Stream(device=dev)
    K, Wu = args.steps, max(args.warmup, 3)
    indels = kind == "reads400"
    with torch.cuda.stream(stream):
        ctx = g.Context(local, stream.cuda_stream)
        batches, desc = reads_batches(kind, rank, world, args.scale, K + Wu)
        nb = len(batches)
        flush = env.flush
        # models: the sample genome's ICM (reads400) or one device-trained ICM per cluster (reads100)
        genes = {}
        for _, _, k in batches:
            if k in genes:
                continue
            if kind == "reads400":
                genes[k] = g.ICM.Read(ctx, W.gene_model_path())
            else:
                ts, toff = cluster_training_strings(k)
                genes[k] = g.ICMTraining(ctx, 12, 7, 3).Train_Model(g.SeqSet(ctx, ascii=ts, offsets=toff), reverse=True)
        pinned, pinned_off, sets, indeps, params, gcs = [], [], [], [], [], []
        for a, off, k in batches:
            h = torch.empty(len(a), dtype=torch.uint8).pin_memory()
            h.numpy()[:] = a
            pinned.append(h)
            ho = torch.empty(len(off), dtype=torch.int64).pin_memory()  # the sequence offsets travel with the bases
            ho.numpy()[:] = off
            pinned_off.append(ho)
            ss = g.SeqSet(ctx, ascii=h.numpy(), offsets=off)
            gc = ss.gc_fraction()
            gcs.append(gc)
            p = g.Params(True, allow_indels=1 if indels else 0)
            p.set_ignore_score_len(gc)
            indeps.append(g.ICM.Build_Indep_WO_Stops(ctx, gc, p.stop_codons))
            params.append(p)
            ss.find_orfs(p)
            sets.append(ss)
        bases = [int(b[1][-1]) for b in batches]
        n_starts = 0
        for i in range(max(Wu, nb)):  # every resident batch once: its start-list buffers exist before the timed steps
            j = i % nb
            n_starts = sets[j].score_orfs_mg(genes[batches[j][2]], indeps[j], params[j])
        ctx.sync()
        ctx.profile(True)
        for k in ("k1", "k2", "k3", "orf", "pack"):
            ctx.profile_read(k)
        e0 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
        e1 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
        clocks = ClockSampler(local) if rank == 0 else None
        barrier()
        launches0 = ctx.launches
        t_wall0 = time.time()
        done_bases = 0
        for k in range(K):
            j = (Wu + k) % nb
            flush.zero_()
            e0[k].record(stream)
            n_starts = sets[j].score_orfs_mg(genes[batches[j][2]], indeps[j], params[j])
            e1[k].record(stream)
            done_bases += bases[j]
        barrier()
        t_wall1 = time.time()
        launches = ctx.launches - launches0
        ms = sum(a.elapsed_time(b) for a, b in zip(e0, e1))
        kms = {k: ctx.profile_read(k) for k in ("k1", "k2", "k3")}
        clk = clocks.stop(t_wall0, t_wall1) if clocks else None
        n_orfs_last, uncert = sets[(Wu + K - 1) % nb].n_orfs, sets[(Wu + K - 1) % nb].uncertified
        if rank == 0 and args.dump_outputs:
            last = sets[(Wu + K - 1) % nb]
            dump_outputs(args.dump_outputs, scoring_outputs(*last.get_orfs(), *last.get_starts()))

        # ---- end to end: pinned host ASCII in, ORF table + start lists out (pinned) ----
        for s in sets:
            s.close()
        e2e_ms, d2h, h2d, e2e_bases = 0.0, 0, 0, 0
        # glimmer-mg -u 1.0 without a feature file: prior -1 + 1, default start-codon log-odds, length log-odds 0
        event_model = g.EventModel(prior=0.0, len_lo=np.zeros((1, 2, 2, (READS400_LEN if indels else READS100_LEN) // 3 + 64)))
        We = max(Wu, nb)  # every resident batch once before timing (pinned staging and pool blocks sized)
        for k in range(We + K):
            j = k % nb
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record(stream)
            # the call sequence of the chunk-level glimmer-mg binding (host/mg_score_orfs_dropin.inc): ORF table and the
            # REDUCED start lists (one candidate per ORF and start position, row a11b) come back to the host
            s2 = g.SeqSet(ctx, ascii=pinned[j].numpy(), offsets=pinned_off[j].numpy())
            s2.find_orfs(params[j])
            orfs, ooff = s2.get_orfs(pinned=True)
            s2.score_orfs_mg(genes[batches[j][2]], indeps[j], params[j])
            s2.reduce_starts_mg(params[j], event_model)
            red, rfirst, rcnt, rstatus = s2.get_reduced_starts(pinned=True)
            b.record(stream)
            torch.cuda.synchronize()
            if k >= We:
                e2e_ms += a.elapsed_time(b)
                e2e_bases += bases[j]
                d2h = orfs.nbytes + ooff.nbytes + red.nbytes + rfirst.nbytes + rcnt.nbytes + rstatus.nbytes
                h2d = len(batches[j][0]) + batches[j][1].nbytes + event_model.len_lo.nbytes
            if k + 1 < We + K:
                s2.close()
        ctx.profile(False)
        # ---- parity (outside the timed region): a sample of the last end-to-end batch against the oracle port
        parity = None
        if rank == 0 and not args.no_parity:
            CP = parity_mod()
            ba, boff, bk = batches[j]
            ids = CP.sample_ids(len(boff) - 1, 600 if indels else 3000)
            og = CP.oracle_model(path=W.gene_model_path()) if indels else CP.oracle_model(genes[bk])
            starts, soff = s2.get_starts()  # the raw lists stay on the device; fetched here only for the check
            st = CP.check_scoring("mg", ba, boff, ids, orfs, ooff, starts, soff, og, s2.gc_fraction(),
                                  params[j].stop_codons, allow_indels=1 if indels else 0,
                                  ignore_score_len=params[j].ignore_score_len)
            orf_ids = [o for i in ids[:200] for o in range(int(ooff[i]), int(ooff[i + 1]))]
            rs = CP.check_reduction(orfs, ooff, np.diff(boff), starts, soff, red, rfirst, rcnt, rstatus, params[j].min_gene_len,
                                    event_model, orf_ids=orf_ids)
            parity = {"checked": f"ORF tables + raw start lists (order, j, pos, which, flags, error lists, FP64 score bits) of "
                                 f"{len(ids)} reads of the last end-to-end batch ({int(s2.n_starts)} raw starts in the batch) "
                                 f"identical to the oracle port; the device-side reduction of {len(orf_ids)} ORFs identical to the "
                                 f"reference's filter + per-position arg-max restated on the raw lists", **st,
                      "reduction": rs, "raw_starts": int(s2.n_starts), "surviving_starts": int(len(red)),
                      "uncertified_reads": int(s2.uncertified)}
        s2.close()
        # ---- end to end with N_LANES batches in flight: the same call sequence from N_LANES host threads, each with its own
        # context and stream, so that one batch's H2D / D2H copies overlap the other's kernels (what a streaming
        # integration does with consecutive chunks).  Every step still copies its inputs from pinned host memory and its
        # results back inside the timed region.
        pipe_ms = None
        if not args.no_pipeline:
            import threading
            lanes = [(ctx, genes, indeps, stream)]
            extra_ctx = []
            for _ in range(N_LANES - 1):
                stream_b = torch.cuda.Stream(device=dev)
                ctx_b = g.Context(local, stream_b.cuda_stream)
                genes_b = {k: g.ICM.from_tables(ctx_b, *m.dims()[:3], *m.tables()) for k, m in genes.items()}
                indeps_b = [g.ICM.Build_Indep_WO_Stops(ctx_b, gcs[i], params[i].stop_codons) for i in range(nb)]
                lanes.append((ctx_b, genes_b, indeps_b, stream_b))
                extra_ctx.append(ctx_b)

            def one(lane, jb):
                c, gs, ins, _ = lanes[lane]
                s3 = g.SeqSet(c, ascii=pinned[jb].numpy(), offsets=pinned_off[jb].numpy())
                s3.find_orfs(params[jb])
                s3.get_orfs(pinned=True)
                s3.score_orfs_mg(gs[batches[jb][2]], ins[jb], params[jb])
                s3.reduce_starts_mg(params[jb], event_model)
                s3.get_reduced_starts(pinned=True)
                s3.close()

            for lane in range(N_LANES):
                for k in range(We):
                    one(lane, k % nb)
            barrier()
            ev0 = torch.cuda.Event(enable_timing=True)
            ends = [torch.cuda.Event(enable_timing=True) for _ in range(N_LANES)]
            ev0.record(stream)  # both streams are idle here
            errs = []

            def worker(lane):
                try:
                    torch.cuda.set_device(local)
                    for k in range(lane, K, N_LANES):
                        one(lane, (We + k) % nb)
                    ends[lane].record(lanes[lane][3])
                except Exception as exc:  # pragma: no cover
                    errs.append(exc)

            th = [threading.Thread(target=worker, args=(lane,)) for lane in range(N_LANES)]
            for t_ in th:
                t_.start()
            for t_ in th:
                t_.join()
            torch.cuda.synchronize()
            if errs:
                raise errs[0]
            pipe_ms = max(ev0.elapsed_time(e) for e in ends)
            pipe_bases = sum(bases[(We + k) % nb] for k in range(K))
            for c_ in extra_ctx:
                c_.close()

    t = torch.tensor([ms, e2e_ms, pipe_ms or 0.0], dtype=torch.float64, device=dev)
    tb = torch.tensor([done_bases, e2e_bases, pipe_bases if pipe_ms else 0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tb, op=dist.ReduceOp.SUM)
    ms_max, e2e_max, pipe_max = t.tolist()
    all_bases, all_e2e_bases, all_pipe_bases = tb.tolist()
    # per-rank view (diagnostic): step, kernel and end-to-end times of every rank -- batches differ between ranks (GC
    # 0.30 .. 0.70: the ORF density varies) and the headline takes the slowest
    mine = torch.tensor([ms / K, kms["k1"][0] / K, kms["k2"][0] / K, kms["k3"][0] / K, e2e_ms / K, (pipe_ms or 0.0) / K],
                        dtype=torch.float64, device=dev)
    per_rank = [mine]
    if world > 1:
        per_rank = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(per_rank, mine)
    per_rank = [[round(x, 4) for x in r.tolist()] for r in per_rank]
    if rank == 0:
        value = all_bases / (ms_max / 1e3) / 1e9
        e2e = all_e2e_bases / (e2e_max / 1e3) / 1e9
        peak, peak_src = measured_peak()
        per_base = {"k1": K1_BYTES_PER_BASE, "k2": K2_BYTES_PER_BASE}
        dom = max(("k1", "k2"), key=lambda k: kms[k][0])
        nb_avg = done_bases / K
        dom_ms = kms[dom][0] / max(kms[dom][1], 1)
        achieved = nb_avg * per_base[dom] / (dom_ms / 1e3) / 1e9
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wu,
                "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": desc, "model": "tests/golden/NC_000915.icm (12/7/3)" if indels else
                           "one 12/7/3 ICM per cluster, trained on the device (build-icm -r) from 1500 x 999 bp genes",
                           "bases_per_step_per_gpu": int(nb_avg), "orfs_last_step": int(n_orfs_last),
                           "starts_last_step": int(n_starts), "uncertified_reads": int(uncert),
                           "l2": "256 MB flush write before every timed step",
                           "sharding": "batches dealt to ranks, no collective"},
                "roofline": {"bound": "hbm", "kernel": {"k1": "k1_planes", "k2": "k2_prefix"}[dom], "achieved": achieved,
                             "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": ncu_traffic({"k1": "k1_planes_reads100", "k2": "k2_prefix_reads400"}[dom], nb_avg),
                             "peak_source": peak_src, "algorithmic_bytes_per_launch": nb_avg * per_base[dom],
                             "kernel_ms": dom_ms, "kernel_share_of_step": kms[dom][0] / ms,
                             "ms_per_step_by_kernel": {k: v[0] / K for k, v in kms.items()},
                             "note": ("k3 = the flat start enumeration of -i (one thread per candidate call, L2-latency / issue "
                                      "bound): no HBM roofline; its time is listed beside the two streaming kernels") if indels else
                                     ("k1 = the bucketed walk kernel + the partial-window fix kernel (shared-memory gather wavefronts "
                                      "at 77 % of the pipe, not HBM, bind it); k3 = the fused K2 + K3 pass (k3_mg_plain_lanes: DRAM "
                                      "sector gathers through the bucket index, latency bound): its time is listed beside K1")},
                "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                        "ms_per_step": e2e_max / K, "in_flight": 1},
                "gpu_launches": int(launches), "clocks": clk,
                "parity_checked": parity is not None, "parity": parity,
                "per_rank_ms": {"columns": ["step", "k1", "k2", "k3", "e2e_one_batch", "e2e_in_flight"], "rows": per_rank}}
        if pipe_max > 0:
            # headline e2e = the streaming form (N_LANES batches in flight); the one-batch-at-a-time figure stays beside it
            line["e2e"].update({"value": all_pipe_bases / (pipe_max / 1e3) / 1e9, "ms_per_step": pipe_max / K, "in_flight": N_LANES,
                                "how": f"{N_LANES} host threads, each with its own context / stream, take batches in turn: copies of "
                                       "one batch overlap the kernels of the others; every step copies its input from pinned host "
                                       "memory and its ORF table + reduced start lists back",
                                "one_batch_at_a_time": {"value": e2e, "ms_per_step": e2e_max / K}})
        if world == 1 and not args.no_cpu_baseline:
            tmp = tempfile.mkdtemp(prefix="gmg_bench_")
            try:
                a, off, _ = batches[0]
                n_s = min(len(off) - 1, 4000 if indels else 40000)
                if ref_bin("glimmer-mg"):
                    fa = reads_cpu_sample(kind, a, off, n_s, tmp, W.gene_model_path())
                    sec = ref_glimmer_mg_seconds([fa], tmp, ["-i"] if indels else [], [W.gene_model_path()])
                    kindname = "reference"
                else:
                    sec = port_mg_seconds(a[:off[n_s]], off[:n_s + 1], indels)
                    kindname = "port"
                line["cpu_baseline"] = {"value": int(off[n_s]) / sec / 1e9, "unit": UNIT, "cores": 1, "kind": kindname,
                                        "sample": f"first {n_s} reads of the first batch through glimmer-mg -u 1.0"
                                                  f"{' -i' if indels else ''} on one core (single-threaded binary; "
                                                  f"sample-genome ICM), {sec:.2f} s"}
                mp = W.gene_model_path()
                if not indels:  # the cluster's own ICM, as the pipeline would use it
                    mp = os.path.join(tmp, "cluster.icm")
                    genes[batches[0][2]].Output(mp)
                line["e2e_app"] = app_glimmer_mg(a, off, n_s, ["-i"] if indels else [], mp)
            finally:
                shutil.rmtree(tmp, ignore_errors=True)
        return line
    return None


# ---------------------------------------------------------------------------------------------------
TRAIN_METRIC = "counted Gbp/s"


def ref_build_icm_seconds(ascii_arr, off, tmp):
    import workloads as W
    fa = os.path.join(tmp, "train.fa")
    W.write_fasta(fa, ascii_arr, off, prefix="g")
    exe = ref_bin("build-icm")
    t0 = time.perf_counter()
    with open(fa, "rb") as fin:
        rc = subprocess.run([exe, "-r", os.path.join(tmp, "m.icm")], stdin=fin, stdout=subprocess.DEVNULL,
                            stderr=subprocess.DEVNULL).returncode
    if rc != 0:
        raise RuntimeError("reference build-icm failed")
    return time.perf_counter() - t0


def port_train_seconds(ascii_arr, off):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    s_all = ascii_arr.tobytes()
    rev = [s_all[off[i]:off[i + 1]][::-1] for i in range(len(off) - 1)]
    arr = O.cstr_array(rev)
    t0 = time.perf_counter()
    O.lib().orc_icm_train(arr, len(rev), 12, 7, 3)
    return time.perf_counter() - t0


def train_cpu(n_seqs):
    import workloads as W
    a, off = W.coding(n_seqs, TRAIN_CODONS, W.TRAIN_SEED)
    tmp = tempfile.mkdtemp(prefix="gmg_bench_")
    try:
        if ref_bin("build-icm"):
            return int(off[-1]), ref_build_icm_seconds(a, off, tmp), "reference"
        return int(off[-1]), port_train_seconds(a, off), "port"
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def train_reference_sha(n_seqs):
    """sha256 of the model file the reference writes for the first n_seqs training strings -> (digest, how)."""
    import hashlib
    import workloads as W
    if n_seqs == TRAIN_SEQS:
        try:
            with open(os.path.join(ROOT, "tests", "golden", "train500m.sha256.json")) as fp:
                rec = json.load(fp)
            if rec["n_seqs"] == n_seqs and rec["seed"] == W.TRAIN_SEED:
                return rec["model_file_sha256"], ("the unmodified reference build-icm -r on the same 500 Mbp (committed digest, "
                                                  "tests/golden/train500m.sha256.json)")
        except Exception:
            return None, None
        return None, None
    if n_seqs > 6000:
        return None, None
    a, off = W.coding(n_seqs, TRAIN_CODONS, W.TRAIN_SEED)
    tmp = tempfile.mkdtemp(prefix="gmg_bench_")
    try:
        out = os.path.join(tmp, "m.icm")
        if ref_bin("build-icm"):
            ref_build_icm_seconds(a, off, tmp)
            how = "the unmodified reference build-icm -r run on the same strings"
        else:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import oracle_lib as O
            raw = a.tobytes()
            rev = [raw[off[i]:off[i + 1]][::-1] for i in range(len(off) - 1)]
            O.lib().orc_icm_write(O.lib().orc_icm_train(O.cstr_array(rev), len(rev), 12, 7, 3), out.encode())
            how = "the oracle port's Train_Model on the same strings"
        return hashlib.sha256(open(out, "rb").read()).hexdigest(), how
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def train_desc(n_seqs):
    return (f"train500m: build-icm -r (Train_Model, 12/7/3) on {n_seqs} stop-free coding strings x {3 * TRAIN_CODONS} bp "
            f"(seed 7), strings dealt round-robin to ranks, one int32 count-slab all-reduce per tree level "
            f"(BASELINE.json configs[3])")


def run_reference_train(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    n_seqs = max(16, int(TRAIN_SEQS * args.scale))
    n_sample = min(n_seqs, max(100, min(2500, 2500 * 20 // max(1, args.steps + args.warmup))))  # ~ a minute in total
    times = []
    for k in range(args.warmup + args.steps):
        bases, sec, kind = train_cpu(n_sample)
        if k >= args.warmup:
            times.append(sec)
    value = bases * len(times) / sum(times) / 1e9
    line = {"metric": TRAIN_METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic", "impl": "reference",
            "config": {"workload": train_desc(n_seqs)},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": kind,
                             "sample": f"each step: build-icm -r on the first {n_sample} training strings ({bases} bp), one "
                                       f"core -- one model cannot be split over processes (SURVEY.md 8(d))"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_b200_train(args, env):
    import numpy as np
    import torch
    import torch.distributed as dist
    import glimmer_mg_b200 as g
    from glimmer_mg_b200 import shard
    import workloads as W

    rank, world, local, dev, barrier = env.rank, env.world, env.local, env.dev, env.barrier

    stream = torch.cuda.Stream(device=dev)
    K, Wu = args.steps, max(args.warmup, 3)
    n_seqs = max(16, int(TRAIN_SEQS * args.scale))
    with torch.cuda.stream(stream):
        ctx = g.Context(local, stream.cuda_stream)
        a_all, off_all = W.coding(n_seqs, TRAIN_CODONS, W.TRAIN_SEED)
        if world > 1:
            a, off = shard.take_sequences(a_all, off_all, shard.round_robin(n_seqs, rank, world))
        else:
            a, off = a_all, off_all
        total_bases = int(off_all[-1])
        del a_all
        h = torch.empty(len(a), dtype=torch.uint8).pin_memory()
        h.numpy()[:] = a
        ar = shard.torch_allreduce(local) if world > 1 else None
        flush = env.flush
        ss = g.SeqSet(ctx, ascii=h.numpy(), offsets=off)
        trainer = g.ICMTraining(ctx, 12, 7, 3)
        model = None
        for _ in range(Wu):
            model = trainer.Train_Model(ss, reverse=True, allreduce=ar, rank=rank, world=world, global_bases=total_bases)
        ctx.sync()
        ctx.profile(True)
        ctx.profile_read("k4")
        e0 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
        e1 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
        clocks = ClockSampler(local) if rank == 0 else None
        barrier()
        launches0 = ctx.launches
        t_wall0 = time.time()
        for k in range(K):
            flush.zero_()
            e0[k].record(stream)
            tw = time.perf_counter()
            model = trainer.Train_Model(ss, reverse=True, allreduce=ar, rank=rank, world=world, global_bases=total_bases)
            e1[k].record(stream)
            if os.environ.get("GMG_BENCH_DEBUG"):
                print(f"train step {k}: host wall {1e3 * (time.perf_counter() - tw):.1f} ms", file=sys.stderr)
        barrier()
        t_wall1 = time.time()
        launches = ctx.launches - launches0
        ms = sum(x.elapsed_time(y) for x, y in zip(e0, e1))
        k4_ms, k4_n = ctx.profile_read("k4")
        clk = clocks.stop(t_wall0, t_wall1) if clocks else None
        if rank == 0 and args.dump_outputs:
            mip, prob = model.tables()
            dump_outputs(args.dump_outputs, {"model_mip": mip.astype(np.float32), "model_prob": prob})
        ss.close()
        # ---- end to end: pinned host strings in, model tables out ----
        e2e_ms, d2h = 0.0, 0
        for k in range(Wu + K):
            flush.zero_()
            x, y = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            x.record(stream)
            s2 = g.SeqSet(ctx, ascii=h.numpy(), offsets=off)
            m2 = trainer.Train_Model(s2, reverse=True, allreduce=ar, rank=rank, world=world, global_bases=total_bases)
            mip, prob = m2.tables()
            y.record(stream)
            torch.cuda.synchronize()
            if k >= Wu:
                e2e_ms += x.elapsed_time(y)
                d2h = mip.nbytes + prob.nbytes
            s2.close()
            if k + 1 < Wu + K:
                m2.close()
        ctx.profile(False)
        import hashlib
        digest = hashlib.sha256(mip.tobytes() + prob.tobytes()).hexdigest()[:16]
        # ---- parity (outside the timed region): the model FILE of the last end-to-end step against the unmodified
        # reference build-icm's -- the committed digest of its 25-minute run at full size
        # (tests/golden/train500m.sha256.json, tools/make_train500m_golden.py), a live run below 6 000 strings
        tmpd = tempfile.mkdtemp(prefix="gmg_bench_")
        try:
            mfile = os.path.join(tmpd, "dev.icm")
            m2.Output(mfile)
            file_sha = hashlib.sha256(open(mfile, "rb").read()).hexdigest()
        finally:
            shutil.rmtree(tmpd, ignore_errors=True)
        m2.close()
        all_sha = [file_sha]
        if world > 1:
            all_sha = [None] * world
            dist.all_gather_object(all_sha, file_sha)
        parity = None
        if rank == 0 and not args.no_parity:
            want, how = train_reference_sha(n_seqs)
            if want is not None:
                if any(x != want for x in all_sha):
                    raise SystemExit(f"bench.py: PARITY FAILURE: trained model file sha256 {all_sha} != reference {want} ({how})")
                parity = {"checked": f"model file written from every rank's trained model byte-identical (sha256) to {how}",
                          "model_file_sha256": file_sha, "ranks": world}
            elif len(set(all_sha)) != 1:
                raise SystemExit(f"bench.py: PARITY FAILURE: ranks hold different models {all_sha}")

    t = torch.tensor([ms, e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max, e2e_max = t.tolist()
    if rank == 0:
        value = total_bases * K / (ms_max / 1e3) / 1e9
        e2e = total_bases * K / (e2e_max / 1e3) / 1e9
        peak, peak_src = measured_peak()
        my_bases = int(off[-1])
        alg = my_bases * 8 * 0.25  # eight level passes over the packed strings
        k4_step_ms = k4_ms / K
        achieved = alg / (k4_step_ms / 1e3) / 1e9
        line = {"metric": TRAIN_METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wu,
                "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "int32", "data": "synthetic",
                "config": {"workload": train_desc(n_seqs), "training_bases": total_bases, "bases_per_gpu": my_bases,
                           "model_sha256_16": digest, "l2": "256 MB flush write before every timed step",
                           "host_recomputed_nodes": int(getattr(trainer, "flagged_nodes", 0)),
                           "sharding": "round-robin strings; window histogram all-reduced once (NCCL), every rank walks 1/N of "
                                       "its cells per level, each level's count slab all-reduced" if world > 1
                           else "single GPU, no exchange"},
                "roofline": {"bound": "hbm", "kernel": "k4_count", "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": alg / 8, "kernel_ms": k4_ms / max(k4_n, 1),
                             "kernel_share_of_step": k4_ms / ms,
                             "atomic_payload_gbs": my_bases * 352 / (k4_step_ms / 1e3) / 1e9,
                             "note": "K4 is bound by the shared/L2 atomic rate (88 int32 increments per base per model, "
                                     "352 B/base of RMW payload), not by HBM: the HBM figure is the packed-string "
                                     "re-read (8 x 0.25 B/base) and is expected to be a small fraction of peak"},
                "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(len(a) + off.nbytes),
                        "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_max / K},
                "gpu_launches": int(launches), "clocks": clk,
                "parity_checked": parity is not None, "parity": parity}
        if world == 1 and not args.no_cpu_baseline:
            an, offn = W.coding(min(n_seqs, 5000), TRAIN_CODONS, W.TRAIN_SEED)
            line["e2e_app"] = app_build_icm(an, offn)
            bases, sec, kind = train_cpu(min(n_seqs, 5000))
            line["cpu_baseline"] = {"value": bases / sec / 1e9, "unit": UNIT, "cores": 1, "kind": kind,
                                    "sample": f"build-icm -r on the first {min(n_seqs, 5000)} training strings ({bases} bp) on "
                                              f"one core (one model cannot be split over processes), {sec:.2f} s"}
        return line
    return None


# ---------------------------------------------------------------------------------------------------
# simplescore: the many-model read scoring that precedes glimmer-mg in the full pipeline (SURVEY.md section 8(f) row 4;
# Phymm / Scimm `simple-score`, scripts/scoreReadsGlim.pl:450,482): Score_String of every read under every
# classification ICM.  16 period-1 ICMs (12/7/1) trained from the 16 synthetic genomes' coding strings, 250 000 reads x
# 400 bp drawn from the config-2 contig; a step scores all reads against all models in one call.  The metric counts
# read bases x models ("model-bases").
SIMPLE_MODELS, SIMPLE_READS, SIMPLE_LEN, SIMPLE_TRAIN_SEQS = 16, 250_000, 400, 300
SIMPLE_METRIC = "ICM-scored Gbp/s"


def simple_reads(rank, scale):
    import workloads as W
    contig = W.contig(W.CONTIG_SEED, CONTIG_LEN)
    n = max(64, int(SIMPLE_READS * scale))
    return W.reads(contig, n, SIMPLE_LEN, 11 + rank, indel=False)


def simple_training(k):
    import numpy as np
    import workloads as W
    gc = float(np.linspace(0.30, 0.70, SIMPLE_MODELS)[k])
    return W.coding(SIMPLE_TRAIN_SEQS, 333, seed=W.READS100_SEED * 1000 + 700 + k, freq=W.reweight_gc(W.codon_freq(), gc))


def simple_desc(n_reads):
    return (f"simplescore: Score_String of {n_reads} reads x {SIMPLE_LEN} bp under {SIMPLE_MODELS} period-1 ICMs (12/7/1, "
            f"trained from {SIMPLE_TRAIN_SEQS} x 999 bp coding strings of 16 synthetic genomes) in one call; Gbp/s counts "
            f"read bases x models (SURVEY.md section 8(f) row 4)")


def _simple_ref_worker(job):
    """One reference process: Score_String (the unmodified ICM library through oracle/_ref's ctypes shim, or the oracle
    port where oracle/_ref is absent) of a slice of reads under every model; returns seconds."""
    model_paths, seqs, use_ref = job
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    if use_ref:
        R = O.ref()
        read, score = R.ref_icm_read, R.ref_score_string
    else:
        read, score = O.lib().orc_icm_read, O.lib().orc_score_string
    hs = [read(p.encode()) for p in model_paths]
    t0 = time.perf_counter()
    acc = 0.0
    for h in hs:
        for s in seqs:
            acc += score(h, s, len(s), 0)
    return time.perf_counter() - t0


def run_reference_simple(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from concurrent.futures import ProcessPoolExecutor
    import workloads as W
    cores = host_cores()
    n_sample = max(50, min(1500, 1500 * 40 // max(1, args.steps + args.warmup)))
    a, off = simple_reads(0, min(1.0, max(args.scale, 1e-9)))
    n_avail = len(off) - 1
    n_sample = min(n_sample, n_avail)
    tmp = tempfile.mkdtemp(prefix="gmg_ref_")
    try:
        exe = ref_bin("build-icm")
        have = exe is not None and os.path.exists(os.path.join(ROOT, "oracle", "_ref", "lib", "libref_icm.so"))
        if not have:
            cores = 1
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import oracle_lib as O
        paths = []
        for k in range(SIMPLE_MODELS):  # the reference's own build-icm (or the oracle port) trains the models (not timed)
            ts, toff = simple_training(k)
            mp = os.path.join(tmp, f"m{k}.icm")
            if have:
                fa = os.path.join(tmp, f"train{k}.fa")
                W.write_fasta(fa, ts, toff, prefix="g")
                with open(fa, "rb") as fin:
                    subprocess.run([exe, "-d", "7", "-w", "12", "-p", "1", mp], stdin=fin, check=True,
                                   stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            else:
                raw_t = ts.tobytes()
                strs = O.cstr_array([raw_t[toff[i]:toff[i + 1]] for i in range(len(toff) - 1)])
                O.lib().orc_icm_write(O.lib().orc_icm_train(strs, len(toff) - 1, 12, 7, 1), mp.encode())
            paths.append(mp)
        raw = a.tobytes()
        jobs = []
        for i in range(cores):
            lo = (i * n_sample) % max(1, n_avail - n_sample + 1)
            jobs.append((paths, [raw[off[j]:off[j + 1]] for j in range(lo, lo + n_sample)], have))
        times = []
        with ProcessPoolExecutor(max_workers=cores) as ex:
            for k in range(args.warmup + args.steps):
                t0 = time.perf_counter()
                list(ex.map(_simple_ref_worker, jobs))
                if k >= args.warmup:
                    times.append(time.perf_counter() - t0)
        bases = cores * n_sample * SIMPLE_LEN * SIMPLE_MODELS
        value = bases * len(times) / sum(times) / 1e9
        line = {"metric": SIMPLE_METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "impl": "reference",
                "config": {"workload": simple_desc(n_avail)},
                "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference" if have else "port",
                                 "sample": f"each step: {cores} processes, each ICM_t::Score_String of its own {n_sample} reads "
                                           f"under all {SIMPLE_MODELS} models (" +
                                           ("the unmodified ICM library through a ctypes shim)" if have else
                                            "the oracle port, models trained by its Train_Model)")},
                "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line), flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def run_b200_simple(args, env):
    import numpy as np
    import torch
    import torch.distributed as dist
    import glimmer_mg_b200 as g

    rank, world, local, dev, barrier = env.rank, env.world, env.local, env.dev, env.barrier

    stream = torch.cuda.Stream(device=dev)
    K, Wu = args.steps, max(args.warmup, 3)
    with torch.cuda.stream(stream):
        ctx = g.Context(local, stream.cuda_stream)
        models = []
        for k in range(SIMPLE_MODELS):
            ts, toff = simple_training(k)
            models.append(g.ICMTraining(ctx, 12, 7, 1).Train_Model(g.SeqSet(ctx, ascii=ts, offsets=toff), reverse=False))
        a, off = simple_reads(rank, args.scale)
        h = torch.empty(len(a), dtype=torch.uint8).pin_memory()
        h.numpy()[:] = a
        flush = env.flush
        ss = g.SeqSet(ctx, ascii=h.numpy(), offsets=off)
        n_reads, n_bases = ss.n, ss.total
        for _ in range(Wu):
            out = g.score_strings_many(ctx, models, ss, 0, pinned=True)
        ctx.sync()
        ctx.profile(True)
        ctx.profile_read("fs")
        e0 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
        e1 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
        clocks = ClockSampler(local) if rank == 0 else None
        barrier()
        launches0 = ctx.launches
        t_wall0 = time.time()
        for k in range(K):
            flush.zero_()
            e0[k].record(stream)
            out = g.score_strings_many(ctx, models, ss, 0, pinned=True)  # includes the D2H of the score matrix
            e1[k].record(stream)
        barrier()
        t_wall1 = time.time()
        launches = ctx.launches - launches0
        ms = sum(x.elapsed_time(y) for x, y in zip(e0, e1))
        k_ms, k_n = ctx.profile_read("fs")
        clk = clocks.stop(t_wall0, t_wall1) if clocks else None
        if rank == 0 and args.dump_outputs:  # reads (columns) sampled only when the matrix exceeds DUMP_BYTES
            cols = seeded_sample(out.shape[1], lambda ids: out.shape[0] * len(ids) * 8 <= DUMP_BYTES)
            dump_outputs(args.dump_outputs, {"scores": out[:, cols], "score_reads": cols})
        ss.close()
        e2e_ms = 0.0
        for k in range(Wu + K):
            flush.zero_()
            x, y = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            x.record(stream)
            s2 = g.SeqSet(ctx, ascii=h.numpy(), offsets=off)
            out = g.score_strings_many(ctx, models, s2, 0, pinned=True)
            y.record(stream)
            torch.cuda.synchronize()
            if k >= Wu:
                e2e_ms += x.elapsed_time(y)
            s2.close()
        ctx.profile(False)
        parity = None
        if rank == 0 and not args.no_parity:  # 200 reads x every model against the oracle port's Score_String, bit for bit
            CP = parity_mod()
            import oracle_lib as O
            raw = a.tobytes()
            ids = CP.sample_ids(n_reads, 200)
            for km, m in enumerate(models):
                om = CP.oracle_model(m)
                for i in ids:
                    sq = raw[off[i]:off[i + 1]]
                    want = O.lib().orc_score_string(om, sq, len(sq), 0)
                    if np.float64(out[km, i]).view(np.uint64) != np.float64(want).view(np.uint64):
                        raise SystemExit(f"bench.py: PARITY FAILURE: Score_String model {km} read {i}: {out[km, i]!r} != {want!r}")
            parity = {"checked": f"Score_String of {len(ids)} reads under each of the {len(models)} models bit-identical to the "
                                 f"oracle port"}
    t = torch.tensor([ms, e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max, e2e_max = t.tolist()
    if rank == 0:
        mb = n_bases * SIMPLE_MODELS * world
        peak, peak_src = measured_peak()
        kern_ms = k_ms / max(k_n, 1)
        # algorithmic HBM bytes of the kernel: the packed reads once per model (L2 keeps them) + one double per (model, read)
        alg = n_bases * 0.25 + n_reads * SIMPLE_MODELS * 8
        line = {"metric": SIMPLE_METRIC, "value": mb * K / (ms_max / 1e3) / 1e9, "unit": UNIT, "n_gpus": world, "steps": K,
                "warmup": Wu, "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": simple_desc(n_reads), "reads_per_gpu": int(n_reads), "models": SIMPLE_MODELS,
                           "l2": "256 MB flush write before every timed step", "sharding": "reads dealt to ranks, no collective"},
                "roofline": {"bound": "hbm", "kernel": "k_score_many", "achieved": alg / (kern_ms / 1e3) / 1e9, "peak": peak,
                             "unit": "GB/s", "frac": alg / (kern_ms / 1e3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": alg, "kernel_ms": kern_ms, "kernel_share_of_step": k_ms / ms,
                             "note": "gather-bound: 8 shared-memory byte lookups and one L2 leaf gather per (model, base); "
                                     "HBM only carries 0.25 B/base in and 8 B per (model, read) out"},
                "e2e": {"value": mb * K / (e2e_max / 1e3) / 1e9, "unit": UNIT, "h2d_bytes_per_step": int(len(a) + off.nbytes),
                        "d2h_bytes_per_step": int(out.nbytes), "ms_per_step": e2e_max / K},
                "gpu_launches": int(launches), "clocks": clk, "parity_checked": parity is not None, "parity": parity}
        return line
    return None


def _default_lanes():
    """Batches in flight of the streaming end-to-end measurement: 4, fewer when the ranks of a node would otherwise hold
    more synchronising host threads than the node has cores."""
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        cores = os.cpu_count() or 4
    world = int(os.environ.get("WORLD_SIZE", "1"))
    return max(2, min(4, cores // max(world, 1) - 1))


N_LANES = int(os.environ.get("GMG_BENCH_LANES", "0")) or _default_lanes()


def main():
    # the bench contract is ONE JSON line on stdout.  With NCCL_DEBUG=VERSION (set on the GPU boxes) NCCL prints its
    # version banner to stdout and ignores NCCL_DEBUG_FILE; at WARN and above the file is honoured: keep the banner,
    # send it to stderr
    if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"
    if os.environ.get("NCCL_DEBUG"):
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    args = parse_args()
    default_run = args.workload is None
    if default_run:
        args.workload = "reads100"
    if args.impl == "reference":
        if args.workload in ("reads400", "reads100"):
            run_reference_reads(args, args.workload)
        elif args.workload == "train500m":
            run_reference_train(args)
        elif args.workload == "simplescore":
            run_reference_simple(args)
        else:
            run_reference(args)
        return
    runners = {"contig5m": run_b200, "reads400": lambda a, e: run_b200_reads(a, e, "reads400"),
               "reads100": lambda a, e: run_b200_reads(a, e, "reads100"), "train500m": run_b200_train,
               "simplescore": run_b200_simple}
    env = Env()
    try:
        line = runners[args.workload](args, env)
        if default_run and not args.no_extra:
            # the other BASELINE configs in the same run (fewer steps each: the whole default run stays within minutes)
            import copy
            extra = {}
            for wl, steps in (("contig5m", 50), ("train500m", 8), ("reads400", 10)):
                sub = copy.copy(args)
                sub.workload = wl
                sub.steps = min(args.steps, steps)
                sub.warmup = min(max(args.warmup, 3), 5)
                sub.dump_outputs = None  # the dump holds the headline workload's outputs only
                sub_line = runners[wl](sub, env)
                if sub_line is not None:
                    extra[wl] = sub_line
            if line is not None:
                line["extra"] = extra
        if line is not None:
            print(json.dumps(line), flush=True)
    finally:
        env.close()


if __name__ == "__main__":
    main()
