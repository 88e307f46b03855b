"""Drop-in boundary, end to end on the GPU: the C++ hosts over the C-ABI.

* glimmer_mg_b200/host/bin/glimmer3-gmg and glimmer-mg-gmg are the reference's own drivers compiled
  (glimmer_mg_b200/host/Makefile, `dropin`) against glimmer_mg_b200/host/icm.hh and linked to libgmgicm.so instead of the reference's ICM
  library, with the scoring half redirected to host/*_dropin.inc.  Their .predict output must equal, byte for
  byte, the reference's golden NC_000915.run1.predict (sample-run config, BASELINE.json configs[0]) and the
  .predict files the unmodified reference wrote for the committed read sets (plain / -i / -s).
* glimmer_mg_b200/host/bin/build-icm is our own C++ build-icm over the ICM_Training_t facade: its model files
  must equal the unmodified reference build-icm's, byte for byte, binary and text form.
"""
import gzip
import hashlib
import json
import os
import subprocess

import pytest

import oracle_lib as O

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
G = os.path.join(HERE, "golden")
REFBIN = os.path.join(ROOT, "oracle", "_ref", "bin")
HOSTBIN = os.path.join(ROOT, "glimmer_mg_b200", "host", "bin")
ICM = os.path.join(G, "NC_000915.icm")

pytestmark = pytest.mark.gpu


def _need(path):
    if not os.path.exists(path):
        pytest.skip(f"{os.path.relpath(path, ROOT)} not built (needs the reference checkout at build time)")
    return path


def _gunzip(name, dst):
    with gzip.open(os.path.join(G, name), "rb") as f, open(dst, "wb") as g:
        g.write(f.read())
    return dst


def _run(cmd, **kw):
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, **kw)
    assert r.returncode == 0, f"{cmd}\n{r.stdout[-2000:]}\n{r.stderr[-2000:]}"
    return r


def test_glimmer3_dropin_reproduces_golden_predict(tmp_path):
    exe = _need(os.path.join(HOSTBIN, "glimmer3-gmg"))
    fna = _gunzip("NC_000915.fna.gz", str(tmp_path / "NC_000915.fna"))
    _run([exe, "-u", "-12", "-m", ICM, fna, str(tmp_path / "run")])
    got = open(tmp_path / "run.predict", "rb").read()
    want = gzip.open(os.path.join(G, "NC_000915.run1.predict.gz"), "rb").read()
    assert got.count(b"\n") == want.count(b"\n") and got == want, "glimmer3 over the GPU path differs from the golden .predict"
    assert want.count(b"orf") >= 1500


def test_glimmer3_dropin_option_variants(tmp_path):
    """Option variants (-X truncated ORFs, -g/-A, -z translation table, -l) on a 300 kbp prefix: equal the
    unmodified reference binary's .predict."""
    exe = _need(os.path.join(HOSTBIN, "glimmer3-gmg"))
    ref = _need(os.path.join(REFBIN, "glimmer3"))
    lines = gzip.open(os.path.join(G, "NC_000915.fna.gz"), "rt").readlines()
    fna = tmp_path / "p.fna"
    fna.write_text(lines[0] + "".join(lines[1:1 + 300000 // 70]))
    # the last two: start / stop codon PATTERNS with IUPAC ambiguity codes (Codon_t masks, Common/gene.cc:39-161)
    for flags in (["-u", "-12"], ["-u", "-12", "-X"], ["-u", "-12", "-g", "90", "-A", "atg,gtg"], ["-u", "-8", "-z", "4", "-l"],
                  ["-u", "-12", "-Z", "tar,tga"], ["-u", "-12", "-A", "atg,ktg", "-P", "0.6,0.4", "-Z", "trr"]):
        _run([exe, *flags, "-m", ICM, str(fna), str(tmp_path / "a")])
        _run([ref, *flags, "-m", ICM, str(fna), str(tmp_path / "b")])
        assert open(tmp_path / "a.predict", "rb").read() == open(tmp_path / "b.predict", "rb").read(), flags
    want = gzip.open(os.path.join(G, "g3_300k.predict.gz"), "rb").read()
    _run([exe, "-u", "-12", "-m", ICM, str(fna), str(tmp_path / "c")])
    assert open(tmp_path / "c.predict", "rb").read() == want


def test_glimmer3_dropin_detail_log_opt_in(tmp_path):
    """The `.detail` log (compiled off in the reference: `bool Detail_Log = false`, glimmer_base.cc:20) behind GMG_DETAIL=1:
    every line -- ORF coordinates, gene scores and the six integerised All_Frame_Score columns, computed for all ORFs
    in one device call -- equals what the reference writes when built with the flag on (oracle/_ref/bin/glimmer3-detail)."""
    exe = _need(os.path.join(HOSTBIN, "glimmer3-gmg"))
    ref = _need(os.path.join(REFBIN, "glimmer3-detail"))
    lines = gzip.open(os.path.join(G, "NC_000915.fna.gz"), "rt").readlines()
    fna = tmp_path / "p.fna"
    fna.write_text(lines[0] + "".join(lines[1:1 + 200000 // 70]))
    for flags in (["-u", "-12"], ["-u", "-12", "-X"]):
        _run([ref, *flags, "-m", ICM, str(fna), str(tmp_path / "r")])
        _run([exe, *flags, "-m", ICM, str(fna), str(tmp_path / "g")], env=dict(os.environ, GMG_DETAIL="1"))
        want = [l for l in open(tmp_path / "r.detail") if not l.startswith("Command:")]
        got = [l for l in open(tmp_path / "g.detail") if not l.startswith("Command:")]
        assert len(want) > 1000 and got == want, flags
        assert open(tmp_path / "g.predict", "rb").read() == open(tmp_path / "r.predict", "rb").read()
    _run([exe, "-u", "-12", "-m", ICM, str(fna), str(tmp_path / "off")])
    assert not os.path.exists(tmp_path / "off.detail")   # off by default, like the shipped reference binaries


@pytest.mark.parametrize("tag,n,flags", [("plain", 120, []), ("indel", 40, ["-i"]), ("sub", 80, ["-s"])])
def test_glimmer_mg_dropin_reproduces_reference_predict(tmp_path, tag, n, flags):
    exe = _need(os.path.join(HOSTBIN, "glimmer-mg-gmg"))
    recs = O.read_fasta(os.path.join(G, "seqs.fa.gz"))[:n]
    fa = tmp_path / "reads.fa"
    with open(fa, "wb") as f:
        for h, s in recs:
            f.write(b">" + h.encode() + b"\n" + s + b"\n")
    _run([exe, "-u", "1.0", "-m", ICM, *flags, str(fa), str(tmp_path / "mg")])
    got = open(tmp_path / "mg.predict", "rb").read()
    want = gzip.open(os.path.join(G, f"mg_{tag}_{n}.predict.gz"), "rb").read()
    assert got == want, f"glimmer-mg {flags} over the GPU path differs from the reference's .predict"


@pytest.mark.parametrize("opts", [["-r"], [], ["-r", "-d", "5", "-w", "10", "-p", "1"], ["-r", "-F"], ["-r", "-t"],
                                  ["-t", "-p", "2", "-d", "3"]])
def test_build_icm_host_cli_matches_reference_binary(tmp_path, opts):
    """Model files of our build-icm equal the unmodified reference build-icm's, byte for byte, live where oracle/_ref was
    built.  Always: against golden/build_icm_cluster5.sha256.json, the sha256 of the files this build-icm wrote at a
    commit where this comparison with the reference binary passed.  For "-r", "" and "-r -d 5 -w 10 -p 1" the oracle
    port's Train_Model writes the same files, which confirms those three independently; for "-r -F", "-r -t" and
    "-t -p 2 -d 3" nothing independent confirms them here, so without oracle/_ref these three are regression checks."""
    exe = os.path.join(ROOT, "glimmer_mg_b200", "host", "bin", "build-icm")
    assert os.path.exists(exe), "glimmer_mg_b200/host/bin/build-icm missing: run __graft_entry__.build()"
    train = _gunzip("seqs.cluster-5.run1.filt.gene.fasta.gz", str(tmp_path / "train.fa"))
    with open(train, "rb") as fin:
        _run([exe, *opts, str(tmp_path / "a.icm")], stdin=fin)
    a = open(tmp_path / "a.icm", "rb").read()
    with open(os.path.join(G, "build_icm_cluster5.sha256.json")) as fp:
        want = json.load(fp)[" ".join(opts)]
    assert (hashlib.sha256(a).hexdigest(), len(a)) == (want["sha256"], want["bytes"]), \
        f"build-icm {opts}: model file differs from the reference binary's ({len(a)} vs {want['bytes']} bytes)"
    ref = os.path.join(REFBIN, "build-icm")
    if os.path.exists(ref):
        with open(train, "rb") as fin:
            _run([ref, *opts, str(tmp_path / "b.icm")], stdin=fin)
        assert a == open(tmp_path / "b.icm", "rb").read(), f"build-icm {opts}: model file differs from the reference binary's"


def test_build_icm_host_cli_errors_like_the_reference(tmp_path):
    exe = os.path.join(ROOT, "glimmer_mg_b200", "host", "bin", "build-icm")
    r = subprocess.run([exe, "-r", str(tmp_path / "x.icm")], input=b"", capture_output=True)
    assert r.returncode != 0 and b"no input data" in r.stderr
    r = subprocess.run([exe, "-d", "0", str(tmp_path / "x.icm")], input=b">a\nacgt\n", capture_output=True)
    assert r.returncode != 0 and b"Bad model depth" in r.stderr
