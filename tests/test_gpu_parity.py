"""GPU parity tests: the CUDA path (through the C-ABI of libgmgicm.so) against the oracle
(oracle/icm_oracle.c), the reference's golden vectors and dumps of the unmodified reference.

Bar: bit-exact for every integer / index output AND for every FP64 score (the sums are formed in
the reference's order, or certified exact -- DESIGN.md); trained models byte-identical.
"""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib as O
from dumps import boost, parse_dump, starts_as_tuples

pytestmark = pytest.mark.gpu
G = O.GOLDEN


@pytest.fixture(scope="module")
def gm():
    import glimmer_mg_b200 as g
    return g


@pytest.fixture(scope="module")
def ctx(gm):
    c = gm.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def reads():
    return O.read_fasta(os.path.join(G, "seqs.fa.gz"))


@pytest.fixture(scope="module")
def genome():
    return O.read_fasta(os.path.join(G, "NC_000915.fna.gz"))[0][1]


def _gc_oracle(seqs):
    return O.lib().orc_gc_fraction(O.cstr_array(seqs), (C.c_int * len(seqs))(*[len(s) for s in seqs]), len(seqs))


def _bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def test_model_io_and_tables(gm, ctx, tmp_path):
    for name in ("NC_000915.icm", "cluster-4.icm", "seqs.cluster-4.run1.filt.gicm"):
        path = os.path.join(G, name)
        m = gm.ICM.Read(ctx, path)
        o = O.lib().orc_icm_read(path.encode())
        mip, prob = m.tables()
        omip, oprob = O.icm_tables(o)
        assert (mip == omip).all() and (prob.view(np.uint32) == oprob.view(np.uint32)).all()
        out = str(tmp_path / "w.icm")
        m.Output(out)
        assert open(out, "rb").read() == open(path, "rb").read()
        assert m.image() == open(path, "rb").read()                      # buffer forms (no file)
        m2 = gm.ICM.Input(ctx, open(path, "rb").read())
        mip2, prob2 = m2.tables()
        assert (mip2 == mip).all() and (prob2.view(np.uint32) == prob.view(np.uint32)).all()
        with pytest.raises(gm.GmgError, match="ERROR reading"):
            gm.ICM.Input(ctx, open(path, "rb").read()[:1000])
    with pytest.raises(gm.GmgError):
        gm.ICM.Read(ctx, str(tmp_path / "missing.icm"))
    bad = tmp_path / "bad.icm"
    bad.write_bytes(b"x" * 100)
    with pytest.raises(gm.GmgError, match="ERROR reading ICM header"):
        gm.ICM.Read(ctx, str(bad))


def test_build_indep_wo_stops(gm, ctx):
    for gc, stops in ((0.3887516210824964, ("taa", "tag", "tga")), (0.5, ("taa", "tag", "tga")),
                      (0.66, ("taa", "tag"))):
        m = gm.ICM.Build_Indep_WO_Stops(ctx, gc, stops)
        mip, prob = m.tables()
        omip, oprob = O.icm_tables(O.build_indep(gc, stops))
        assert (mip == omip).all() and (prob.view(np.uint32) == oprob.view(np.uint32)).all()


def test_filter_pack_gc(gm, ctx):
    rng = np.random.default_rng(1)
    alphabet = np.frombuffer(b"acgtACGTnNrRyYsSwWmMkKbBdDhHvVxX*-", np.uint8)
    seqs = [alphabet[rng.integers(0, len(alphabet), n)].tobytes() for n in (0, 1, 31, 32, 33, 64, 1000, 5, 0, 777)]
    ss = gm.SeqSet(ctx, seqs=seqs)
    assert ss.unpack() == b"".join(O.filter_lower(s) for s in seqs)
    assert ss.gc_fraction() == _gc_oracle(seqs)


def _py_fasta(image):
    """Fasta_Read (Common/fasta.cc:236-283) restated: [(header text, sequence bytes)] -- used only where the reference
    build (oracle/_ref) is absent; the test below pins the device parser to the reference's own reader."""
    recs, i, n = [], image.find(b">"), len(image)
    while i != -1:
        h = i + 1
        while h < n and image[h:h + 1] == b" ":
            h += 1
        if h == n:
            break  # '>' followed by blanks and the end of the file: no record (fasta.cc:251-255)
        e = image.find(b"\n", h)
        e = n if e == -1 else e
        nxt = image.find(b">", e)
        body = image[e:(n if nxt == -1 else nxt)]
        recs.append((image[h:e], bytes(c for c in body if c not in b" \t\n\v\f\r")))
        i = nxt
    return recs


@pytest.mark.parametrize("case", ["reads", "genome", "edge", "edge2", "blank_tail", "empty", "norecord"])
def test_fasta_ingest_on_device(gm, ctx, case, tmp_path):
    """gmg_seqset_from_fasta: records, headers, offsets and packed bases equal what the UNMODIFIED reference reader
    (Fasta_Read through oracle/_ref's shim) makes of the same bytes, incl. malformed input."""
    import gzip
    if case == "reads":
        image = gzip.open(os.path.join(G, "seqs.fa.gz"), "rb").read()
    elif case == "genome":
        image = gzip.open(os.path.join(G, "NC_000915.fna.gz"), "rb").read()
    elif case == "edge":
        image = (b"junk before\nthe first record\n>r1 first  \r\nACGTNNacgt\r\n\r\nGG TT\tAA\n>empty\n>r3 > odd header\n"
                 b"acgRYKM>r4 starts mid line\nttt\n\n>last header without newline")
    elif case == "edge2":
        image = b">   leading blanks\nac gt\n>\nnoheader\n> \n\n>x\rcarriage\ronly\nGATTACA\n>tab\there\nN\n"
    elif case == "blank_tail":
        image = b">a\nacgt\n>   "
    elif case == "empty":
        image = b""
    else:
        image = b"no records here\nacgt\n"
    want = _py_fasta(image)
    if O.have_ref() and hasattr(O.ref(), "ref_fasta_read_file"):
        path = tmp_path / "in.fa"
        path.write_bytes(image)
        assert O.ref_fasta_records(str(path)) == want, "the restated reader disagrees with the reference's Fasta_Read"
    ss = gm.SeqSet.from_fasta(ctx, image)
    assert ss.n == len(want)
    assert [h.encode() for h in ss.headers] == [h for h, _ in want]
    lens = [len(s) for _, s in want]
    assert ss.off.tolist() == [0] + np.cumsum(lens).tolist() if lens else ss.off.tolist() == [0]
    if ss.total:
        assert ss.unpack() == b"".join(O.filter_lower(s) for _, s in want)
        ref = gm.SeqSet(ctx, seqs=[s for _, s in want])
        assert abs(ss.gc_fraction() - ref.gc_fraction()) == 0.0


@pytest.mark.parametrize("case", ["reads", "edge", "edge2", "empty", "norecord"])
def test_quality_ingest_on_device(gm, ctx, reads, case, tmp_path):
    """gmg_quality_parse_fasta: records and values equal what the UNMODIFIED reference reader (Fasta_Qual_Vec_Read through
    oracle/_ref's shim) makes of the same bytes, incl. malformed input; gmg_seqset_quality_from_fasta attaches them to a set
    exactly as a host-supplied quality array."""
    rng = np.random.default_rng(3)
    if case == "reads":
        sub = reads[:200]
        qs = [rng.integers(0, 41, len(s)) for _, s in sub]
        image = b"".join(b">" + h.encode() + b"\n" + b"\n".join(b" ".join(b"%d" % v for v in q[k:k + 17]) for k in range(0, len(q), 17))
                         + b"\n" for (h, _), q in zip(sub, qs))
    else:
        image = O.QUAL_EDGE_IMAGES[case]
    want = O.py_qual_records(image)
    if O.have_ref() and hasattr(O.ref(), "ref_fasta_qual_read_file"):
        path = tmp_path / "in.qual"
        path.write_bytes(image)
        assert O.ref_qual_records(str(path)) == want, "the restated reader disagrees with the reference's Fasta_Qual_Vec_Read"
    off, vals = gm.parse_quality_fasta(ctx, image)
    assert len(off) - 1 == len(want)
    assert np.diff(off).tolist() == [len(q) for _, q in want]
    assert vals.tolist() == [v for _, q in want for v in q]
    if case == "reads":
        p = gm.Params(True, allow_indels=1, have_quality_file=1)
        gene = gm.ICM.Read(ctx, os.path.join(G, "NC_000915.icm"))

        def run(ss):
            gc = ss.gc_fraction()
            p.set_ignore_score_len(gc)
            indep = gm.ICM.Build_Indep_WO_Stops(ctx, gc)
            ss.find_orfs(p)
            ss.score_orfs_mg(gene, indep, p)
            st, so = ss.get_starts()
            return st.tobytes(), so.tolist()

        a = gm.SeqSet(ctx, seqs=[s for _, s in sub], qual=np.concatenate(qs).astype(np.uint8))
        b = gm.SeqSet(ctx, seqs=[s for _, s in sub])
        b.set_quality_fasta(image)
        assert run(a) == run(b)
        c = gm.SeqSet(ctx, seqs=[s for _, s in sub[:-1]])
        with pytest.raises(gm.GmgError):
            c.set_quality_fasta(image)


@pytest.mark.parametrize("k", [4, 5])
def test_score_string_known_answers(gm, ctx, reads, k):
    m = gm.ICM.Read(ctx, os.path.join(G, f"cluster-{k}.icm"))
    gold = [l.split() for l in open(os.path.join(G, f"icm-{k}.scores.tmp"))]
    got = m.score_strings([s for _, s in reads], 0)
    om = O.lib().orc_icm_read(os.path.join(G, f"cluster-{k}.icm").encode())
    for (h, s), (gh, gv), v in zip(reads, gold, got):
        assert "%.4f" % v == "%.4f" % float(gv)
        assert v == O.lib().orc_score_string(om, s, len(s), 0)


def test_score_strings_many_models(gm, ctx, reads):
    """Every read against every model in one launch (models of different periodicity mixed): the reference's golden
    Score_String values (4 decimals), and bit-identical to the per-model call and to the oracle.  frame 1 exercises
    the period cycling of the period-3 model."""
    names = ["cluster-4.icm", "NC_000915.icm", "cluster-5.icm", "seqs.cluster-5.run1.filt.gicm"]
    models = [gm.ICM.Read(ctx, os.path.join(G, nm)) for nm in names]
    seqs = [s for _, s in reads] + [b"", b"acg", b"acgtacgtacgtac"]
    ss = gm.SeqSet(ctx, seqs=seqs)
    for frame in (0, 1):
        got = gm.score_strings_many(ctx, models, ss, frame)
        assert got.shape == (len(models), len(seqs))
        for k, (nm, m) in enumerate(zip(names, models)):
            one = m.score_strings(ss, frame)
            assert (got[k].view(np.uint64) == one.view(np.uint64)).all(), nm
            om = O.lib().orc_icm_read(os.path.join(G, nm).encode())
            P = m.Get_Periodicity()
            for i in range(0, len(seqs), 7):
                assert got[k, i] == O.lib().orc_score_string(om, seqs[i], len(seqs[i]), frame if P > 1 else 0), (nm, i)
    for k, kk in ((0, 4), (2, 5)):
        gold = [l.split() for l in open(os.path.join(G, f"icm-{kk}.scores.tmp"))]
        got = gm.score_strings_many(ctx, models, ss, 0)
        for (gh, gv), v in zip(gold, got[k]):
            assert "%.4f" % v == "%.4f" % float(gv)


def test_score_strings_many_redo_path(gm, ctx, reads, monkeypatch):
    """(model, read) pairs whose exactness certificate fails are repeated in the reference's serial order: forced for
    every pair here, the matrix must keep its bits."""
    names = ["cluster-4.icm", "NC_000915.icm"]
    models = [gm.ICM.Read(ctx, os.path.join(G, nm)) for nm in names]
    ss = gm.SeqSet(ctx, seqs=[s for _, s in reads[:300]] + [b"", b"ac"])
    want = gm.score_strings_many(ctx, models, ss, 1).copy()
    monkeypatch.setenv("GMG_MANY_FORCE_REDO", "1")
    got = gm.score_strings_many(ctx, models, ss, 1)
    assert (got.view(np.uint64) == want.view(np.uint64)).all()
    for k, m in enumerate(models):
        assert (got[k].view(np.uint64) == m.score_strings(ss, 1).view(np.uint64)).all()


def test_scalar_surface_matches_oracle(gm, ctx, reads):
    path = os.path.join(G, "NC_000915.icm")
    m = gm.ICM.Read(ctx, path)
    om = O.lib().orc_icm_read(path.encode())
    L = O.lib()
    for _, s0 in reads[:6]:
        s = O.filter_lower(s0)
        for f in range(3):
            a = np.zeros(len(s))
            L.orc_frame_score(om, s, len(s), f, a.ctypes.data)
            assert (_bits(m.Frame_Score(s0, f)) == _bits(a)).all()
            L.orc_cumulative_score(om, s, len(s), f, a.ctypes.data)
            assert (_bits(m.Cumulative_Score(s0, f)) == _bits(a)).all()
        for n in (1, 5, 11, 12, 13, 40):
            assert m.Score_String(s0, 1, n) == L.orc_score_string(om, s, n, 1)
        assert m.Full_Window_Prob(s[20:32], 2) == L.orc_full_window_prob(om, s[20:32], 2)
        assert m.Partial_Window_Prob(7, s, 1) == L.orc_partial_window_prob(om, 7, s, 1)
    assert len(m.score_strings([b""], 0)) == 1 and m.score_strings([b""], 0)[0] == 0.0


def test_all_frame_scores_match_oracle_score_string(gm, ctx, genome):
    """gmg_all_frame_scores (All_Frame_Score glimmer3.cc:328-359, the `.detail` columns): for random regions the six
    sums equal Score_String of the reversed region / its reverse complement under the oracle, bit for bit."""
    path = os.path.join(G, "NC_000915.icm")
    gene = gm.ICM.Read(ctx, path)
    og = O.lib().orc_icm_read(path.encode())
    seqs = [genome[:60000], genome[100000:100500], genome[7:40]]
    ss = gm.SeqSet(ctx, seqs=seqs)
    rng = np.random.default_rng(3)
    items = [(0, 0, 60000), (0, 59990, 10), (1, 0, 500), (2, 0, 33), (2, 5, 0), (1, 17, 1)]
    for _ in range(60):
        lo = int(rng.integers(0, 59000))
        items.append((0, lo, int(rng.integers(1, 900))))
    got = ss.all_frame_scores(gene, [i[0] for i in items], [i[1] for i in items], [i[2] for i in items])
    comp = bytes.maketrans(b"acgt", b"tgca")
    for (sq, lo, ln), row in zip(items, got):
        region = O.filter_lower(seqs[sq])[lo:lo + ln]
        down, up = region[::-1], region.translate(comp)
        for f0 in range(3):
            assert row[f0] == O.lib().orc_score_string(og, down, ln, f0), (sq, lo, ln, f0)
            assert row[3 + f0] == O.lib().orc_score_string(og, up, ln, f0), (sq, lo, ln, f0)


def test_score_all_frames_bit_exact(gm, ctx, reads, monkeypatch):
    path = os.path.join(G, "NC_000915.icm")
    gene = gm.ICM.Read(ctx, path)
    og = O.lib().orc_icm_read(path.encode())
    seqs = [s for _, s in reads[:60]]
    seqs += [b"", b"a", b"acgtacgtacg", b"acgtacgtacgt", seqs[0][:13], seqs[1][:100], b"n" * 40]  # ragged / short
    gc = _gc_oracle(seqs)
    indep = gm.ICM.Build_Indep_WO_Stops(ctx, gc)
    oi = O.build_indep(gc)
    ss = gm.SeqSet(ctx, seqs=seqs)
    fs = ss.score_all_frames(gene, indep)
    for s0, got in zip(seqs, fs):
        want = O.score_all_frames(og, oi, O.filter_lower(s0))
        assert got.shape == want.shape
        assert (_bits(got) == _bits(want)).all()
    # the other route for partial windows on read sets: tested in the walk loop, as for long sequences
    monkeypatch.setenv("GMG_K1_FIX", "0")
    fs2 = gm.SeqSet(ctx, seqs=seqs).score_all_frames(gene, indep)
    monkeypatch.delenv("GMG_K1_FIX")
    for a, b in zip(fs, fs2):
        assert (_bits(a) == _bits(b)).all()
    # golden Frame_Scores of the unmodified reference (first 25 reads)
    recs = parse_dump(os.path.join(G, "mg_plain_120.dump.gz"))
    gc = _gc_oracle([s for _, s in reads[:120]])
    indep = gm.ICM.Build_Indep_WO_Stops(ctx, gc)
    fs = gm.SeqSet(ctx, seqs=[s for _, s in reads[:25]]).score_all_frames(gene, indep)
    byhdr = {r["hdr"]: r for r in recs}
    n = 0
    for (h, _), got in zip(reads[:25], fs):
        if h in byhdr and byhdr[h]["fs"]:
            for f in range(6):
                assert (_bits(got[f]) == byhdr[h]["fs"][f]).all()
            n += 1
    assert n >= 20


@pytest.mark.parametrize("w,d", [(12, 5), (12, 2), (16, 8), (18, 4), (9, 7)])
def test_score_all_frames_other_model_shapes(gm, ctx, reads, w, d):
    """K1 beyond the build-icm defaults: runtime-depth fast path (w <= 16, d <= 8) and the generic kernel (w > 16)."""
    strs = [s[::-1] for s in _train_strings("seqs.cluster-5.run1.filt.gene.fasta.gz")]
    om = O.lib().orc_icm_train(O.cstr_array(strs), len(strs), w, d, 3)
    omip, oprob = O.icm_tables(om)
    gene = gm.ICM.from_tables(ctx, w, d, 3, omip, oprob)
    seqs = [s for _, s in reads[100:130]] + [b"acgtacgtacgtacgtacgt"[:n] for n in (1, 8, 9, 15, 16, 17, 18, 19, 20)]
    gc = _gc_oracle(seqs)
    indep = gm.ICM.Build_Indep_WO_Stops(ctx, gc)
    oi = O.build_indep(gc)
    fs = gm.SeqSet(ctx, seqs=seqs).score_all_frames(gene, indep)
    for s0, got in zip(seqs, fs):
        want = O.score_all_frames(om, oi, O.filter_lower(s0))
        assert (_bits(got) == _bits(want)).all()


@pytest.mark.parametrize("flags", [dict(), dict(allow_indels=1), dict(allow_subs=1), dict(allow_truncated=0)])
def test_find_orfs_reads(gm, ctx, reads, flags):
    seqs = [s for _, s in reads[:150]] + [b"", b"acgt" * 10, b"atg" + b"aaa" * 30 + b"taa"]
    p = gm.Params(True, **flags)
    op = O.params(True, **flags)
    ss = gm.SeqSet(ctx, seqs=seqs)
    n = ss.find_orfs(p)
    orfs, off = ss.get_orfs()
    assert off[-1] == n
    for i, s0 in enumerate(seqs):
        want = O.find_orfs(O.filter_lower(s0), op)
        got = orfs[off[i]:off[i + 1]]
        assert got.tolist() == want.tolist(), i


@pytest.mark.parametrize("flags", [dict(min_gene_len=6), dict(min_gene_len=9, allow_indels=1, min_indel_orf_len=6),
                                   dict(min_gene_len=12, allow_truncated=0)])
def test_find_orfs_tiny_and_ragged_sequences(gm, ctx, genome, flags):
    """The tiled ORF finder on what its staging does not cover: thousands of sequences of 0 .. 12 bases (more than 128
    sequence bounds inside a 1 024-base tile: the per-base lookup path), sequences that straddle tiles, a long one whose
    look-backs leave the staged bitmap words, and ORFs that close exactly at tile edges -- each table equal to the
    checker's for that sequence alone."""
    rng = np.random.default_rng(17)
    g = O.filter_lower(genome[:300000])
    seqs, pos = [], 0
    for _ in range(6000):  # tiny: the bounds of a tile overflow the staged list
        n = int(rng.integers(0, 13))
        seqs.append(g[pos:pos + n])
        pos += n
    for n in (1024, 1023, 1025, 2048, 3, 0, 1, 2, 5000, 7, 1024 * 3 - 1):  # tile-sized and straddling
        seqs.append(g[pos:pos + n])
        pos += n
    seqs.append(b"atg" + b"gcc" * 900 + b"taa" + b"a" * 50)  # one ORF of 2.7 kbp: look-backs far beyond the halo
    for _ in range(300):  # read-like
        n = int(rng.integers(30, 400))
        seqs.append(g[pos:pos + n])
        pos += n
    p = gm.Params(True, **flags)
    op = O.params(True, **flags)
    ss = gm.SeqSet(ctx, seqs=seqs)
    n = ss.find_orfs(p)
    orfs, off = ss.get_orfs()
    assert off[-1] == n and n > 1000
    for i, s0 in enumerate(seqs):
        want = O.find_orfs(s0, op)
        assert orfs[off[i]:off[i + 1]].tolist() == want.tolist(), (i, len(s0))


@pytest.mark.parametrize("truncated", [0, 1])
def test_find_orfs_genome(gm, ctx, genome, truncated):
    s0 = genome[:400000]
    p = gm.Params(False, allow_truncated=truncated)
    op = O.params(False, allow_truncated=truncated)
    ss = gm.SeqSet(ctx, seqs=[s0])
    ss.find_orfs(p)
    orfs, off = ss.get_orfs()
    want = O.find_orfs(O.filter_lower(s0), op)
    assert orfs.tolist() == want.tolist()


@pytest.mark.parametrize("tag,n,flags", [("plain", 120, {}), ("indel", 40, dict(allow_indels=1)),
                                         ("sub", 80, dict(allow_subs=1))])
def test_mg_start_lists_match_reference_dump(gm, ctx, reads, tag, n, flags):
    """glimmer-mg -u 1.0 -m NC_000915.icm [-i|-s]: ORFs and raw start_list of every ORF identical to the
    unmodified reference (order, j, pos, which, flags, error lists and FP64 score BITS)."""
    recs = parse_dump(os.path.join(G, f"mg_{tag}_{n}.dump.gz"))
    sub = reads[:n]
    gene = gm.ICM.Read(ctx, os.path.join(G, "NC_000915.icm"))
    ss = gm.SeqSet(ctx, seqs=[s for _, s in sub])
    gc = ss.gc_fraction()
    assert gc == _gc_oracle([s for _, s in sub])
    p = gm.Params(True, **flags)
    p.set_ignore_score_len(gc)
    indep = gm.ICM.Build_Indep_WO_Stops(ctx, gc, p.stop_codons)
    ss.find_orfs(p)
    ss.score_orfs_mg(gene, indep, p)
    assert ss.uncertified == 0
    orfs, ooff = ss.get_orfs()
    starts, soff = ss.get_starts()
    byhdr = {r["hdr"]: r for r in recs}
    total = 0
    for i, (h, _) in enumerate(sub):
        r = byhdr.get(h)
        mine = orfs[ooff[i]:ooff[i + 1]]
        if r is None:
            assert len(mine) == 0
            continue
        assert [o["o"] for o in r["orfs"]] == [tuple(x) for x in mine.tolist()]
        for k, o in enumerate(r["orfs"]):
            oi = ooff[i] + k
            got = starts_as_tuples(starts[soff[oi]:soff[oi + 1]])
            assert got == boost(o["starts"], p.ignore_score_len), (h, o["o"])
            total += len(got)
    assert total > 1000


def test_mg_start_lists_match_oracle_more_reads(gm, ctx, reads):
    """A larger differential run against the oracle, indel mode with a quality 'file'."""
    rng = np.random.default_rng(7)
    sub = [s for _, s in reads[300:380]] + [b"", b"acg"]
    quals = [rng.integers(1, 41, len(s)).astype(np.uint8) for s in sub]
    gene_path = os.path.join(G, "seqs.cluster-5.run1.filt.gicm")
    gene = gm.ICM.Read(ctx, gene_path)
    og = O.lib().orc_icm_read(gene_path.encode())
    ss = gm.SeqSet(ctx, seqs=sub, qual=np.concatenate(quals))
    gc = ss.gc_fraction()
    for flags in (dict(allow_indels=1, have_quality_file=1), dict(allow_indels=1, allow_subs=1)):
        p = gm.Params(True, **flags)
        p.set_ignore_score_len(gc)
        op = O.params(True, **flags)
        op.ignore_score_len = p.ignore_score_len
        indep = gm.ICM.Build_Indep_WO_Stops(ctx, gc)
        oi = O.build_indep(gc)
        ss.find_orfs(p)
        ss.score_orfs_mg(gene, indep, p)
        orfs, ooff = ss.get_orfs()
        starts, soff = ss.get_starts()
        for i, s0 in enumerate(sub):
            s = O.filter_lower(s0)
            want_orfs = O.find_orfs(s, op)
            assert orfs[ooff[i]:ooff[i + 1]].tolist() == want_orfs.tolist()
            q = quals[i].astype(np.int32) if flags.get("have_quality_file") else None
            woff, wst = O.mg_score_orfs(og, oi, s, op, want_orfs, q)
            for k in range(len(want_orfs)):
                o = ooff[i] + k
                assert starts_as_tuples(starts[soff[o]:soff[o + 1]]) == starts_as_tuples(wst[woff[k]:woff[k + 1]])


@pytest.mark.parametrize("flags", [dict(allow_indels=1), dict(allow_subs=1), dict(allow_indels=1, allow_subs=1),
                                   dict(allow_indels=1, indel_max=1)])
def test_mg_flat_thread_and_ordered_paths_agree(gm, ctx, reads, monkeypatch, flags):
    """-i / -s start lists come from the flat level-by-level enumeration (gmg_mg_flat.cuh).  The thread-per-ORF
    recursion (GMG_K3MG_MODE=1) and the ordered path of sequences without an exactness certificate (forced for
    every / every third sequence) must give the identical CSR, and all of them the oracle's lists."""
    rs = [s for _, s in reads[:150]]
    gene_path = os.path.join(G, "NC_000915.icm")
    gene = gm.ICM.Read(ctx, gene_path)
    indep = gm.ICM.Build_Indep_WO_Stops(ctx, 0.39)
    p = gm.Params(True, **flags)
    p.set_ignore_score_len(0.39)

    def run():
        ss = gm.SeqSet(ctx, seqs=rs)
        ss.find_orfs(p)
        ss.score_orfs_mg(gene, indep, p)
        st, off = ss.get_starts()
        return st.tobytes(), off.tolist(), ss.uncertified

    want = run()                                   # flat
    assert want[2] == 0
    monkeypatch.setenv("GMG_K3MG_MODE", "1")
    assert run()[:2] == want[:2]                   # one thread per ORF, explicit stack
    monkeypatch.delenv("GMG_K3MG_MODE")
    monkeypatch.setenv("GMG_MG_FORCE_UNCERT", "1")
    got = run()
    assert got[:2] == want[:2] and got[2] == len(rs)   # every sequence re-summed in the reference's order
    monkeypatch.setenv("GMG_MG_FORCE_UNCERT", "3")
    got = run()
    assert got[:2] == want[:2] and got[2] == (len(rs) + 2) // 3   # both paths in one batch
    monkeypatch.delenv("GMG_MG_FORCE_UNCERT")
    assert len(want[0]) > 48 * 3000
    # and the oracle
    og = O.lib().orc_icm_read(gene_path.encode())
    oi = O.build_indep(0.39)
    op = O.params(True, **flags)
    op.ignore_score_len = p.ignore_score_len
    starts = np.frombuffer(want[0], gm.START_DTYPE)
    k = 0
    for s0 in rs[:40]:
        s = O.filter_lower(s0)
        worfs = O.find_orfs(s, op)
        woff, wst = O.mg_score_orfs(og, oi, s, op, worfs)
        a, b = want[1][k], want[1][k + len(worfs)]
        assert starts[a:b].tobytes() == wst.tobytes()
        k += len(worfs)


def test_mg_plain_fused_scan_matches_thread_path_and_oracle(gm, ctx, reads, monkeypatch):
    """Plain glimmer-mg (no -i / -s): K2 + K3 fused into one per-ORF scan over the K1 planes (k3_mg_plain_lanes, k3_mg_plain).  Same CSR as
    K2 + one thread per ORF (GMG_K3MG_MODE=1), also when every ORF longer than 30 bases is summed in the reference's
    serial order (forced), for ragged / empty / tiny sequences, and equal to the oracle's lists."""
    rs = [s for _, s in reads[:300]] + [b"", b"acgtacgtacgt", reads[5][1][:75], reads[6][1][:76], reads[7][1][:100]]
    gene_path = os.path.join(G, "NC_000915.icm")
    gene = gm.ICM.Read(ctx, gene_path)
    p = gm.Params(True)
    ss0 = gm.SeqSet(ctx, seqs=rs)
    gc = ss0.gc_fraction()
    p.set_ignore_score_len(gc)
    indep = gm.ICM.Build_Indep_WO_Stops(ctx, gc)

    def run():
        ss = gm.SeqSet(ctx, seqs=rs)
        ss.find_orfs(p)
        ss.score_orfs_mg(gene, indep, p)
        st, off = ss.get_starts()
        orfs, ooff = ss.get_orfs()
        return st.tobytes(), off.tolist(), ss.uncertified, orfs, ooff

    want = run()  # fused, one codon per lane, two ORFs per warp up to 192 scored bases (parallel scan under the per-ORF certificate)
    assert want[2] == 0
    for mode in ("0", "1"):  # a scan per 32 bases (ORFs beyond 384 scored bases) / one codon per lane, one ORF per warp
        monkeypatch.setenv("GMG_PLAIN_LANES", mode)
        got = run()
        assert got[:2] == want[:2] and got[2] == 0, mode
        monkeypatch.delenv("GMG_PLAIN_LANES")
    monkeypatch.setenv("GMG_K3MG_MODE", "1")
    assert run()[:2] == want[:2]
    monkeypatch.delenv("GMG_K3MG_MODE")
    monkeypatch.setenv("GMG_MG_FORCE_UNCERT", "1")
    got = run()
    assert got[:2] == want[:2] and got[2] > 100   # ORFs re-summed serially by one lane
    monkeypatch.delenv("GMG_MG_FORCE_UNCERT")
    import config_parity as CP
    a = np.frombuffer(b"".join(rs), np.uint8)
    off = np.concatenate([[0], np.cumsum([len(r) for r in rs])]).astype(np.int64)
    st = CP.check_scoring("mg", a, off, range(len(rs)), want[3], want[4], np.frombuffer(want[0], gm.START_DTYPE),
                          np.asarray(want[1]), CP.oracle_model(path=gene_path), gc, ("taa", "tag", "tga"),
                          ignore_score_len=p.ignore_score_len)
    assert st["starts"] > 5000


@pytest.mark.parametrize("flags,table", [(dict(allow_indels=1), "default"), (dict(allow_indels=1), "random"),
                                         (dict(allow_indels=1, allow_subs=1), "random"), (dict(), "default")])
def test_mg_start_list_reduction(gm, ctx, reads, monkeypatch, flags, table):
    """Row a11b: the per-(ORF, start position) arg-max of Add_Events and Score_Orfs_Errors' two gates on the device
    (gmg_reduce_starts_mg) against a restatement of the reference's filter run on the raw lists."""
    import config_parity as CP
    rs = [s for _, s in reads[:200]] + [b"", b"acgtacgt"]
    gene = gm.ICM.Read(ctx, os.path.join(G, "NC_000915.icm"))
    ss = gm.SeqSet(ctx, seqs=rs)
    gc = ss.gc_fraction()
    indep = gm.ICM.Build_Indep_WO_Stops(ctx, gc)
    p = gm.Params(True, **flags)
    p.set_ignore_score_len(gc)
    ss.find_orfs(p)
    ss.score_orfs_mg(gene, indep, p)
    orfs, ooff = ss.get_orfs()
    raw, soff = ss.get_starts()
    if table == "default":
        model = gm.EventModel(prior=0.0)  # glimmer-mg -u 1.0: LogOdds_Prior = -1 + 1
    else:
        rng = np.random.default_rng(11)
        model = gm.EventModel(prior=-0.25, start_lo=[0.3, -0.4, -1.1], len_lo=rng.normal(0.0, 1.5, (1, 2, 2, 200)))
    monkeypatch.setenv("GMG_RED_SMALL", "0")  # every ORF through the warp-per-ORF kernel
    n_kept_w = ss.reduce_starts_mg(p, model)
    red_w, first_w, cnt_w, status_w = ss.get_reduced_starts()
    monkeypatch.delenv("GMG_RED_SMALL")
    n_kept = ss.reduce_starts_mg(p, model)  # lists of up to eight records: one thread per ORF
    red, first, cnt, status = ss.get_reduced_starts()
    assert n_kept == len(red) == int(cnt.sum())
    assert n_kept_w == n_kept and (cnt_w == cnt).all() and (status_w == status).all()
    for o in np.flatnonzero(cnt):  # same survivors (their order within an ORF is free: one per start position)
        a = red[first[o]:first[o] + cnt[o]]
        b = red_w[first_w[o]:first_w[o] + cnt_w[o]]
        assert sorted(x.tobytes() for x in a) == sorted(x.tobytes() for x in b), o
    st = CP.check_reduction(orfs, ooff, [len(s) for s in rs], raw, soff, red, first, cnt, status, p.min_gene_len, model)
    assert st["kept_orfs"] > 50 and st["handed_back"] <= st["orfs"] // 20, st
    assert n_kept < len(raw)
    if flags.get("allow_indels"):
        assert n_kept * 4 < len(raw), (n_kept, len(raw))   # the point of the exercise
    # the raw list of a single ORF (what the host fetches for status 2)
    o = int(np.argmax(np.diff(soff)))
    assert ss.get_orf_starts(o).tobytes() == raw[soff[o]:soff[o + 1]].tobytes()


def test_g3_start_lists_match_reference_dump(gm, ctx, genome):
    recs = parse_dump(os.path.join(G, "g3_300k.dump.gz"))
    s0 = genome[:(300000 // 70) * 70]
    gene = gm.ICM.Read(ctx, os.path.join(G, "NC_000915.icm"))
    ss = gm.SeqSet(ctx, seqs=[s0])
    gc = ss.gc_fraction()
    p = gm.Params(False)
    p.set_ignore_score_len(gc)
    indep = gm.ICM.Build_Indep_WO_Stops(ctx, gc)
    ss.find_orfs(p)
    ss.score_orfs_g3(gene, indep, p)
    orfs, _ = ss.get_orfs()
    starts, soff = ss.get_starts()
    mine = {tuple(o): starts_as_tuples(starts[soff[i]:soff[i + 1]]) for i, o in enumerate(orfs.tolist())}
    assert len(recs[0]["orfs"]) > 2000
    for o in recs[0]["orfs"]:
        assert mine[o["o"]] == o["starts"], o["o"]


def test_find_orfs_two_pass_path_gives_the_same_table(gm, ctx, reads, monkeypatch):
    """The single-pass finder stages at most 256 ORFs per 1 024-base tile; the overflow path (two passes) must give the
    identical table."""
    p = gm.Params(True, allow_indels=1)
    rs = [s for _, s in reads[:300]]
    ss = gm.SeqSet(ctx, seqs=rs)
    ss.find_orfs(p)
    a, aoff = ss.get_orfs()
    monkeypatch.setenv("GMG_ORF_TWO_PASS", "1")
    ss2 = gm.SeqSet(ctx, seqs=rs)
    ss2.find_orfs(p)
    b, boff = ss2.get_orfs()
    assert len(a) > 5000 and a.tobytes() == b.tobytes() and aoff.tolist() == boff.tolist()


@pytest.mark.parametrize("truncated", [0, 1])
def test_g3_full_genome_matches_oracle(gm, ctx, genome, truncated):
    path = os.path.join(G, "NC_000915.icm")
    gene = gm.ICM.Read(ctx, path)
    og = O.lib().orc_icm_read(path.encode())
    ss = gm.SeqSet(ctx, seqs=[genome])
    gc = ss.gc_fraction()
    p = gm.Params(False, allow_truncated=truncated)
    p.set_ignore_score_len(gc)
    op = O.params(False, allow_truncated=truncated)
    op.ignore_score_len = p.ignore_score_len
    indep = gm.ICM.Build_Indep_WO_Stops(ctx, gc)
    oi = O.build_indep(gc)
    ss.find_orfs(p)
    ss.score_orfs_g3(gene, indep, p)
    orfs, _ = ss.get_orfs()
    starts, soff = ss.get_starts()
    s = O.filter_lower(genome)
    want_orfs = O.find_orfs(s, op)
    assert orfs.tolist() == want_orfs.tolist()
    woff, wst = O.g3_score_orfs(og, oi, s, op, want_orfs)
    assert (soff == woff).all()
    for f in ("j", "pos", "which", "truncated", "first"):
        assert (starts[f] == wst[f]).all(), f
    assert (_bits(starts["score"]) == _bits(wst["score"])).all()
    # the warp-parallel (certified exact) sums must be the common case, the ordered re-run the exception
    assert ss.ordered_fallbacks <= len(orfs) // 20


def _g3_check(gm, ctx, seqs, gene, og, **pkw):
    """glimmer3 scoring half of a batch of sequences against the oracle, sequence by sequence."""
    ss = gm.SeqSet(ctx, seqs=seqs)
    gc = ss.gc_fraction()
    p = gm.Params(False, **pkw)
    p.set_ignore_score_len(gc)
    op = O.params(False, **pkw)
    op.ignore_score_len = p.ignore_score_len
    indep = gm.ICM.Build_Indep_WO_Stops(ctx, gc)
    oi = O.build_indep(gc)
    ss.find_orfs(p)
    ss.score_orfs_g3(gene, indep, p)
    orfs, ooff = ss.get_orfs()
    starts, soff = ss.get_starts()
    n_starts = 0
    for i, s0 in enumerate(seqs):
        s = O.filter_lower(s0)
        want_orfs = O.find_orfs(s, op)
        assert orfs[ooff[i]:ooff[i + 1]].tolist() == want_orfs.tolist(), i
        woff, wst = O.g3_score_orfs(og, oi, s, op, want_orfs)
        lo, hi = soff[ooff[i]], soff[ooff[i + 1]]
        assert ((soff[ooff[i]:ooff[i + 1] + 1] - lo) == woff).all(), i
        got = starts[lo:hi]
        for f in ("j", "pos", "which", "truncated", "first"):
            assert (got[f] == wst[f]).all(), (i, f)
        assert (_bits(got["score"]) == _bits(wst["score"])).all(), i
        n_starts += len(wst)
    return ss, n_starts


def test_g3_ordered_path_gives_the_same_bits(gm, ctx, genome, monkeypatch):
    """The reference-order accumulation (taken when the exactness bound fails) and the scan-based path agree."""
    path = os.path.join(G, "NC_000915.icm")
    gene = gm.ICM.Read(ctx, path)
    og = O.lib().orc_icm_read(path.encode())
    seqs = [genome[:200000]]
    ss, n = _g3_check(gm, ctx, seqs, gene, og)
    assert n > 1000 and ss.ordered_fallbacks == 0
    monkeypatch.setenv("GMG_G3_ORDERED", "1")
    ss, n2 = _g3_check(gm, ctx, seqs, gene, og)
    assert n2 == n and ss.ordered_fallbacks == ss.n_orfs > 0


@pytest.mark.parametrize("pkw", [dict(), dict(allow_truncated=1), dict(min_gene_len=9), dict(min_gene_len=30, allow_truncated=1)])
def test_g3_many_contigs_ragged(gm, ctx, genome, pkw):
    """Several contigs in one batch (offsets not multiples of 3 or of the scan tiles, very short and empty
    sequences, ORFs that cross tile boundaries) and small Min_Gene_Len values (starts inside the partial-window
    head of the ORF string)."""
    path = os.path.join(G, "NC_000915.icm")
    gene = gm.ICM.Read(ctx, path)
    og = O.lib().orc_icm_read(path.encode())
    cuts = [0, 1537, 1537, 1600, 4673, 4680, 30001, 30013, 90000, 90100, 150001]
    seqs = [genome[a:b] for a, b in zip(cuts[:-1], cuts[1:])] + [b"", b"atg", genome[200000:200011]]
    ss, n = _g3_check(gm, ctx, seqs, gene, og, **pkw)
    assert n > 300


def _train_strings(name):
    return [s.lower() for _, s in O.read_fasta(os.path.join(G, name))]


@pytest.mark.parametrize("fasta,depth,period", [("seqs.cluster-4.run1.filt.gene.fasta.gz", 7, 3),
                                                ("seqs.cluster-5.run1.filt.gene.fasta.gz", 7, 3),
                                                ("seqs.cluster-5.run1.filt.gene.fasta.gz", 3, 1),
                                                ("NC_000915.train.gz", 7, 3)])
def test_training_byte_identical_to_oracle(gm, ctx, tmp_path, fasta, depth, period):
    """build-icm -r: the model file written from the device-counted tree equals the oracle's (and therefore,
    by tests/test_oracle.py, the reference's) byte for byte."""
    strs = _train_strings(fasta)
    m = gm.ICMTraining(ctx, 12, depth, period).Train_Model(strs, reverse=True)
    rev = [s[::-1] for s in strs]
    o = O.lib().orc_icm_train(O.cstr_array(rev), len(rev), 12, depth, period)
    a, b = str(tmp_path / "a.icm"), str(tmp_path / "b.icm")
    m.Output(a)
    O.lib().orc_icm_write(o, b.encode())
    assert open(a, "rb").read() == open(b, "rb").read()
    # not reversed, strings pre-reversed on the host: same model
    m2 = gm.ICMTraining(ctx, 12, depth, period).Train_Model(rev, reverse=False)
    m2.Output(a)
    assert open(a, "rb").read() == open(b, "rb").read()


@pytest.mark.parametrize("period,width", [(3, 12), (1, 10)])
def test_training_histogram_path_gives_the_same_model(gm, ctx, tmp_path, monkeypatch, period, width):
    """Large training sets count through the (frame, window) histogram; forced on here, it must give the byte-identical
    model file (and the same count slabs) as the direct per-window path."""
    strs = _train_strings("seqs.cluster-5.run1.filt.gene.fasta.gz")
    a, b = str(tmp_path / "a.icm"), str(tmp_path / "b.icm")
    monkeypatch.setenv("GMG_K4_HIST", "0")
    gm.ICMTraining(ctx, width, 7, period).Train_Model(strs, reverse=True).Output(a)
    tr = gm.ICMTraining(ctx, width, 7, period).levels(strs, reverse=True)
    ptr, n = tr.count_level(0)
    direct0 = ctx.d2h(ptr, n, np.int32).copy()
    tr.close()
    monkeypatch.setenv("GMG_K4_HIST", "1")
    gm.ICMTraining(ctx, width, 7, period).Train_Model(strs, reverse=True).Output(b)
    tr = gm.ICMTraining(ctx, width, 7, period).levels(strs, reverse=True)
    ptr, n = tr.count_level(0)
    assert (ctx.d2h(ptr, n, np.int32) == direct0).all() and direct0.sum() > 0
    tr.close()
    assert open(a, "rb").read() == open(b, "rb").read()


def tr_nodes(args):
    w, d, p = args
    return p * (4 ** (d + 1) - 1) // 3


@pytest.mark.parametrize("mode", ["0", "2"])
def test_training_level_finish_device_and_host_paths_agree(gm, ctx, tmp_path, monkeypatch, mode):
    """Position choice + interpolation run on the device with error bounds on every mutual-information decision
    (k4_finish_level); GMG_K4_MI=0 keeps every node on the host (glibc), GMG_K4_MI=2 flags every node so that the
    host redoes all of them after the device pass.  Same model bytes on all three routes, for three training sets."""
    for name, args in (("seqs.cluster-5.run1.filt.gene.fasta.gz", (12, 7, 3)), ("seqs.cluster-4.run1.filt.gene.fasta.gz", (12, 7, 3)),
                       ("NC_000915.train.gz", (10, 5, 1))):
        strs = [s.lower() for _, s in O.read_fasta(os.path.join(G, name))]
        tr = gm.ICMTraining(ctx, *args)
        want = tr.Train_Model(strs, reverse=True).image()
        few = tr.flagged_nodes
        monkeypatch.setenv("GMG_K4_MI", mode)
        got = gm.ICMTraining(ctx, *args).Train_Model(strs, reverse=True).image()
        monkeypatch.delenv("GMG_K4_MI")
        assert got == want, (name, mode)
        # small training sets have many exactly tied positions (equal count tables): those go to the host by design
        assert few < tr_nodes(args) // 2, f"{name}: {few} nodes within the error bound -- the bound is too loose"


def test_count_level_matches_oracle(gm, ctx):
    """K4 in isolation: the count slab of every level equals Count_Char_Pairs(_Restricted) of the oracle."""
    strs = [s[::-1] for s in _train_strings("seqs.cluster-5.run1.filt.gene.fasta.gz")]
    arr = O.cstr_array(strs)
    omip, _ = O.icm_tables(O.lib().orc_icm_train(arr, len(strs), 12, 7, 3))  # the finished tree
    om = O.lib().orc_icm_new(12, 7, 3)
    tr = gm.ICMTraining(ctx, 12, 7, 3).levels(strs, reverse=False)
    for level in range(0, 8):
        ptr, n = tr.count_level(level)
        nl = 4 ** level
        first = (nl - 1) // 3
        assert n == 3 * nl * 11 * 16
        got = ctx.d2h(ptr, n, np.int32).reshape(3, nl, 11, 16)
        full = np.zeros(3 * 21845 * 11 * 16, np.int32)
        O.lib().orc_count_level(om, arr, len(strs), level, full.ctypes.data)
        assert (got == full.reshape(3, 21845, 11, 16)[:, first:first + nl]).all(), level
        tr.finish_level(level)
        for f in range(3):  # give the oracle's walk this level's branch positions
            for i in range(first, first + nl):
                om.contents.mip[f * 21845 + i] = int(omip[f, i])
    m = tr.finish()
    assert (m.tables()[0] == omip).all()
