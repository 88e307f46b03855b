"""CPU tests that PIN the oracle (oracle/icm_oracle.c):

 * against the reference's own golden vectors (Score_String known answers, trained
   models) committed under tests/golden/ (copied verbatim from the reference's
   sample-run/ by tests/golden/make_golden.py);
 * against outputs of the unmodified reference (raw start-list dumps, committed; and
   live calls into oracle/_ref/lib/libref_icm.so where that was built).
"""
import ctypes as C
import gzip
import hashlib
import json
import os

import numpy as np
import pytest

import oracle_lib as O
from dumps import boost, parse_dump, starts_as_tuples

L = O.lib()
G = O.GOLDEN


def _reference_golden(name):
    """What the unmodified reference library returned for the committed inputs of the tests below
    (golden/reference_library.json; its "about" entry says how it was recorded)."""
    with open(os.path.join(G, "reference_library.json")) as fp:
        return json.load(fp)[name]


def _digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def _reads(n=None):
    recs = O.read_fasta(os.path.join(G, "seqs.fa.gz"))
    return recs if n is None else recs[:n]


def _gc(seqs):
    return L.orc_gc_fraction(O.cstr_array(seqs), (C.c_int * len(seqs))(*[len(s) for s in seqs]), len(seqs))


@pytest.mark.parametrize("k", [4, 5])
def test_score_string_known_answers(k):
    """sample-run/glimmer-mg/results/icm-k.scores.tmp: Score_String(read, len, 0) of every read under
    cluster-k.icm (period-1 Scimm models), printed with 4 decimals."""
    m = L.orc_icm_read(os.path.join(G, f"cluster-{k}.icm").encode())
    assert m
    gold = [l.split() for l in open(os.path.join(G, f"icm-{k}.scores.tmp"))]
    reads = _reads()
    assert len(gold) == len(reads) == 999
    for (h, s), (gh, gv) in zip(reads, gold):
        assert h == gh
        assert "%.4f" % L.orc_score_string(m, s, len(s), 0) == "%.4f" % float(gv)
    L.orc_icm_free(m)


def test_score_string_all_six_models_from_reference_tree():
    if not os.path.exists(O.REF_SAMPLE):
        pytest.skip("reference checkout not present")
    reads = _reads()
    n = 0
    for k in range(6):
        m = L.orc_icm_read(f"{O.REF_SAMPLE}/glimmer-mg/results/cluster-{k}.icm".encode())
        gold = [l.split() for l in open(f"{O.REF_SAMPLE}/glimmer-mg/results/icm-{k}.scores.tmp")]
        for (h, s), (gh, gv) in zip(reads, gold):
            assert "%.4f" % L.orc_score_string(m, s, len(s), 0) == "%.4f" % float(gv)
            n += 1
        L.orc_icm_free(m)
    assert n == 5994


def test_model_io_roundtrip(tmp_path):
    src = os.path.join(G, "NC_000915.icm")
    m = L.orc_icm_read(src.encode())
    out = str(tmp_path / "rt.icm")
    assert L.orc_icm_write(m, out.encode()) == 0
    assert open(src, "rb").read() == open(out, "rb").read()
    mip, prob = O.icm_tables(m)
    assert mip.shape == (3, 21845) and (mip >= -2).all() and (mip <= 10).all()
    assert int((mip >= -1).sum()) == 62743  # SURVEY section 4: nodes written in the golden model


def _scalar_ops(read, frame_score, cumulative_score, score_string, build_indep, tables):
    """sha256 of what one ICM implementation returns for the scalar operations on the committed inputs."""
    path = os.path.join(G, "NC_000915.icm").encode()
    m = read(path)
    out = {"tables NC_000915.icm": _digest(*tables(m))}
    fs, cs, ss = hashlib.sha256(), hashlib.sha256(), hashlib.sha256()
    for h, s in _reads(40):
        s = O.filter_lower(s)
        for f in range(3):
            a = np.zeros(len(s))
            frame_score(m, s, len(s), f, a.ctypes.data)
            fs.update(a.tobytes())
            cumulative_score(m, s, len(s), f, a.ctypes.data)
            cs.update(a.tobytes())
            ss.update(np.float64(score_string(m, s, len(s), f)).tobytes())
        for n in (0, 1, 5, 11, 12, 13):  # short / ragged strings
            ss.update(np.float64(score_string(m, s, n, 1)).tobytes())
    out.update({"Frame_Score": fs.hexdigest(), "Cumulative_Score": cs.hexdigest(), "Score_String": ss.hexdigest()})
    for gc in (0.25, 0.3887516210824964, 0.5, 0.7):
        out[f"Build_Indep_WO_Stops {gc!r}"] = _digest(*tables(build_indep(gc, ("taa", "tag", "tga"))))
    out["Build_Indep_WO_Stops 0.4 taa,tag prob"] = _digest(tables(build_indep(0.4, ("taa", "tag")))[1])  # table 4
    return out


def test_scalar_ops_match_reference_library():
    """Model tables, Frame_Score, Cumulative_Score, Score_String (incl. short / ragged strings) and Build_Indep_WO_Stops
    of the oracle bit-identical to the unmodified reference library: against its recorded results always, and live
    where oracle/_ref was built."""
    mine = _scalar_ops(L.orc_icm_read, L.orc_frame_score, L.orc_cumulative_score, L.orc_score_string,
                       lambda gc, stops: O.build_indep(gc, stops), O.icm_tables)
    assert mine == _reference_golden("scalar_ops")
    if O.have_ref():
        R = O.ref()
        theirs = _scalar_ops(R.ref_icm_read, R.ref_frame_score, R.ref_cumulative_score, R.ref_score_string,
                             lambda gc, stops: R.ref_icm_build_indep(gc, O.cstr_array(list(stops)), len(stops)), O.ref_tables)
        assert theirs == mine


@pytest.mark.parametrize("tag,n,flags", [("plain", 120, {}), ("indel", 40, dict(allow_indels=1)),
                                         ("sub", 80, dict(allow_subs=1))])
def test_mg_scoring_half_matches_reference_dump(tag, n, flags):
    """Frame_Scores, Find_Orfs and the raw per-ORF start_list (order, j, pos, which, flags, error lists and
    FP64 score bits) against the instrumented reference glimmer-mg (-u 1.0 -m NC_000915.icm [-i|-s])."""
    recs = parse_dump(os.path.join(G, f"mg_{tag}_{n}.dump.gz"))
    reads = _reads(n)
    gene = L.orc_icm_read(os.path.join(G, "NC_000915.icm").encode())
    gc = _gc([s for _, s in reads])
    indep = O.build_indep(gc)
    p = O.params(True, **flags)
    p.ignore_score_len = L.orc_ignore_score_len(gc, C.byref(p))
    byhdr = {r["hdr"]: r for r in recs}
    n_fs = n_starts = 0
    for h, s0 in reads:
        s = O.filter_lower(s0)
        orfs = O.find_orfs(s, p)
        r = byhdr.get(h)
        if r is None:
            assert len(orfs) == 0
            continue
        if r["fs"]:
            fs = O.score_all_frames(gene, indep, s)
            for f in range(6):
                assert (fs[f].view(np.uint64) == r["fs"][f]).all()
            n_fs += 1
        assert [o["o"] for o in r["orfs"]] == [tuple(int(x) for x in o.tolist()) for o in orfs]
        off, st = O.mg_score_orfs(gene, indep, s, p, orfs)
        for i, o in enumerate(r["orfs"]):
            assert starts_as_tuples(st[off[i]:off[i + 1]]) == boost(o["starts"], p.ignore_score_len)
            n_starts += len(o["starts"])
    assert n_starts > 1000
    if tag == "plain":
        assert n_fs == 25


def test_g3_scoring_half_matches_reference_dump():
    recs = parse_dump(os.path.join(G, "g3_300k.dump.gz"))
    fna = O.read_fasta(os.path.join(G, "NC_000915.fna.gz"))[0][1][:(300000 // 70) * 70]
    s = O.filter_lower(fna)
    gene = L.orc_icm_read(os.path.join(G, "NC_000915.icm").encode())
    gc = _gc([fna])
    indep = O.build_indep(gc)
    p = O.params(False)
    p.ignore_score_len = L.orc_ignore_score_len(gc, C.byref(p))
    orfs = O.find_orfs(s, p)
    off, st = O.g3_score_orfs(gene, indep, s, p, orfs)
    mine = {tuple(int(x) for x in o.tolist()): starts_as_tuples(st[off[i]:off[i + 1]]) for i, o in enumerate(orfs)}
    assert len(recs) == 1 and len(recs[0]["orfs"]) > 2000
    seen = set()
    for o in recs[0]["orfs"]:
        assert mine[o["o"]] == o["starts"]  # dump is taken after the boost in glimmer3
        seen.add(o["o"])
    # ORFs the reference skipped before the hook have first_j + 1 < Min_Gene_Len (glimmer3.cc:1432)
    for k, v in mine.items():
        if k not in seen:
            assert not v or v[0][0] + 1 < 75


def _train_strings(name):
    return [s.lower()[::-1] for _, s in O.read_fasta(os.path.join(G, name))]  # build-icm -r


@pytest.mark.parametrize("fasta,model", [
    ("seqs.cluster-4.run1.filt.gene.fasta.gz", "seqs.cluster-4.run1.filt.gicm"),
    ("seqs.cluster-5.run1.filt.gene.fasta.gz", "seqs.cluster-5.run1.filt.gicm")])
def test_training_matches_golden_models(fasta, model):
    """Tree topology identical to the authors' golden model; probabilities within 1 float ulp (the goldens
    were produced with another platform's logf -- SURVEY section 7)."""
    strs = _train_strings(fasta)
    m = L.orc_icm_train(O.cstr_array(strs), len(strs), 12, 7, 3)
    g = L.orc_icm_read(os.path.join(G, model).encode())
    ma, pa = O.icm_tables(m)
    mg, pg = O.icm_tables(g)
    assert (ma == mg).all()
    live = ma >= -1
    ulp = np.abs(pa.view(np.int32).astype(np.int64) - pg.view(np.int32).astype(np.int64))[live]
    assert ulp.max() <= 1


@pytest.mark.slow
def test_training_bit_identical_to_reference_library(tmp_path):
    """Model files trained by the oracle byte-identical to the unmodified reference library's: against the recorded
    sha256 of the reference's files always, and live where oracle/_ref was built."""
    want = _reference_golden("training")
    for fasta in ("seqs.cluster-5.run1.filt.gene.fasta.gz", "NC_000915.train.gz"):
        strs = _train_strings(fasta)
        arr = O.cstr_array(strs)
        m = L.orc_icm_train(arr, len(strs), 12, 7, 3)
        a = str(tmp_path / "a.icm")
        L.orc_icm_write(m, a.encode())
        assert hashlib.sha256(open(a, "rb").read()).hexdigest() == want[fasta], fasta
        if O.have_ref():
            R = O.ref()
            r = R.ref_icm_train(arr, len(strs), 12, 7, 3)
            b = str(tmp_path / "b.icm")
            R.ref_icm_write(r, b.encode())
            assert open(a, "rb").read() == open(b, "rb").read()
            R.ref_icm_train_free(r)
        if fasta.startswith("NC_"):
            g = L.orc_icm_read(os.path.join(G, "NC_000915.icm").encode())
            assert (O.icm_tables(m)[0] == O.icm_tables(g)[0]).all()


@pytest.mark.skipif(not O.have_ref(), reason="oracle/_ref not built")
def test_reference_build_reproduces_golden_predict(tmp_path):
    """The unmodified reference compiled by oracle/Makefile reproduces the repository's own golden .predict
    (sample-run/glimmer3, 1 549 gene lines) -- this is what makes oracle/_ref a valid parity anchor."""
    import gzip
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "oracle", "_ref", "bin", "glimmer3")
    if not os.path.exists(exe):
        pytest.skip("reference glimmer3 not built")
    g = os.path.join(root, "tests", "golden")
    fna = tmp_path / "g.fna"
    fna.write_bytes(gzip.open(os.path.join(g, "NC_000915.fna.gz"), "rb").read())
    r = subprocess.run([exe, "-u", "-12", "-m", os.path.join(g, "NC_000915.icm"), str(fna), str(tmp_path / "out")],
                       capture_output=True, timeout=300)
    assert r.returncode == 0
    assert open(tmp_path / "out.predict", "rb").read() == gzip.open(os.path.join(g, "NC_000915.run1.predict.gz"), "rb").read()


@pytest.mark.parametrize("case", sorted(O.QUAL_EDGE_IMAGES))
def test_quality_reader_restatement_equals_reference(case, tmp_path):
    """The restated quality-file reader the GPU tests check gmg_quality_parse_fasta against (py_qual_records) sees what the
    UNMODIFIED Fasta_Qual_Vec_Read (Common/fasta.cc:115-170) sees, on malformed input too: against the reference's
    recorded records always, and live through oracle/_ref's shim where that was built."""
    mine = O.py_qual_records(O.QUAL_EDGE_IMAGES[case])
    assert [[h.decode("latin-1"), v] for h, v in mine] == _reference_golden("quality_records")[case]
    if O.have_ref() and hasattr(O.ref(), "ref_fasta_qual_read_file"):
        path = tmp_path / "in.qual"
        path.write_bytes(O.QUAL_EDGE_IMAGES[case])
        assert O.ref_qual_records(str(path)) == mine
