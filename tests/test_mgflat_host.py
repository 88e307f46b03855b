"""The flat glimmer-mg start enumeration (glimmer_mg_b200/csrc/gmg_mg_flat.cuh: the __host__ __device__ bodies of the
K3 kernels) compiled for the HOST by tests/mgflat_host_check.cu and run against the oracle port on the reference's
sample reads.  A logic check that needs no GPU; the same functions run inside the kernels on the device, where
tests/test_gpu_parity.py holds them to the same lists."""
import gzip
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "tests", "_build")
EXE = os.path.join(BUILD, "mgflat_check")
SRC = [os.path.join(ROOT, "tests", "mgflat_host_check.cu"), os.path.join(ROOT, "oracle", "icm_oracle.c"),
       os.path.join(ROOT, "glimmer_mg_b200", "csrc", "gmg_mg_flat.cuh")]


@pytest.fixture(scope="module")
def harness():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    os.makedirs(BUILD, exist_ok=True)
    if not os.path.exists(EXE) or any(os.path.getmtime(EXE) < os.path.getmtime(f) for f in SRC):
        subprocess.run([nvcc, "-O2", "-std=c++17", "-x", "cu", "-w", "--fmad=false", "-Xcompiler", "-fno-fast-math",
                        "-o", EXE, SRC[0], SRC[1], "-lm"], check=True, cwd=BUILD)
    fa = os.path.join(BUILD, "seqs.fa")
    if not os.path.exists(fa):
        with gzip.open(os.path.join(ROOT, "tests", "golden", "seqs.fa.gz"), "rb") as f, open(fa, "wb") as g:
            g.write(f.read())
    return fa


# (reads, allow_indels, allow_subs, indel_max, truncate_len)
@pytest.mark.parametrize("args", [(400, 1, 0, 2, 0), (400, 0, 1, 2, 0), (300, 1, 1, 2, 0), (400, 1, 0, 1, 0), (400, 0, 0, 2, 0),
                                  (999, 1, 0, 2, 100), (300, 1, 1, 2, 76), (200, 1, 1, 2, 13),
                                  (999, 0, 0, 2, 100), (999, 0, 0, 2, 99), (999, 0, 0, 2, 98), (600, 0, 0, 2, 77),
                                  (300, 0, 0, 2, 13)])
def test_flat_enumeration_equals_oracle_on_the_host(harness, args):
    run(harness, *args)


def run(harness, *args):
    r = subprocess.run([EXE, os.path.join(ROOT, "tests", "golden", "NC_000915.icm"), harness] + [str(a) for a in args],
                       capture_output=True, text=True, timeout=600)
    last = r.stdout.strip().splitlines()[-1] if r.stdout.strip() else ""
    assert r.returncode == 0 and last.startswith("OK:"), r.stdout[-3000:] + r.stderr[-2000:]
    return {k: int(v) for k, v in re.findall(r"(qualities 0|>= 163|\+inf|-inf): (\d+)", last)}


# seeded Phred values as from a quality file, half of them at the table edges (0, 17-20, 162, 163, 255): the oracle gets
# them as read, the flat passes the plane glimmer-mg builds (Clean_Quality_454 under -i only) and Pass_Stop_Penalty per root
# (reads, allow_indels, allow_subs, indel_max, truncate_len, quality seed)
@pytest.mark.parametrize("args", [(400, 0, 1, 2, 0, 11), (300, 1, 0, 2, 0, 12), (300, 1, 1, 2, 0, 13), (400, 1, 0, 1, 0, 14),
                                  (400, 0, 0, 2, 0, 15), (200, 1, 1, 2, 76, 16), (999, 0, 1, 2, 100, 17)])
def test_flat_enumeration_with_quality_file_equals_oracle_on_the_host(harness, args):
    n, ai, asub = args[:3]
    seen = run(harness, *args)
    assert seen[">= 163"] > 0
    if ai:  # cleaned: no zero survives, so no stop probability of 0
        assert seen["qualities 0"] == 0 and seen["+inf"] == 0
    else:
        assert seen["qualities 0"] > 0
    if asub and not ai:  # a 0 on a stop base: p_stop = 0, an infinite substitution penalty reaches the start scores
        assert seen["+inf"] > 0
