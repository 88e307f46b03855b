"""FASTQ ingest on the device (gmg_seqset_from_fastq, SeqSet.from_fastq, SeqSet.qualities).  The oracle is the host route:
the FASTQ image split on the host into a FASTA image and a quality-file image, then from_fasta + set_quality_fasta.  Offsets,
headers, bases, GC, qualities, the non-acgt list (through minus-strand extraction) and glimmer-mg's raw start lists must
be equal; malformed images are rejected with the record, the line and the reason."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib as O
from dumps import starts_as_tuples

G = O.GOLDEN
_WS = np.array([9, 10, 11, 12, 13, 32], np.uint8)


def host_images(image, phred_offset=33):
    """A well-formed FASTQ image -> (FASTA image, quality-file image, qualities uint8).  The FASTA record is the header line
    with '>' for '@' (header bytes verbatim) and the sequence line as is; the quality record is an empty '>' line and one
    two-digit value per quality byte.  Records end at the line of the last non-white-space byte, as in the device parser."""
    a = np.frombuffer(image, np.uint8)
    n = len(a)
    isnl = a == 10
    lid = np.cumsum(isnl, dtype=np.int32) - isnl  # line of every byte
    nl = np.flatnonzero(isnl)
    starts = np.concatenate([[0], nl + 1]).astype(np.int64)  # the text after the last '\n' is a (maybe empty) line
    ends = np.concatenate([nl, [n]]).astype(np.int64)
    nonblank = ~np.isin(a, _WS)
    n_rec = int(lid[nonblank].max()) // 4 + 1 if nonblank.any() else 0
    rec = lid // 4
    inside = rec < n_rec
    fa = a.copy()
    fa[starts[4 * np.arange(n_rec)]] = ord(">")
    fasta = fa[inside & (lid % 4 < 2)].tobytes()
    qmask = inside & (lid % 4 == 3) & ~isnl
    qs, qe = starts[4 * np.arange(n_rec) + 3], ends[4 * np.arange(n_rec) + 3]
    cr = (qe > qs) & (a[np.maximum(qe - 1, 0)] == 13) if n else np.zeros(0, bool)
    qmask[qe[cr] - 1] = False
    qual = (a[qmask] - phred_offset).astype(np.uint8)
    lens = np.bincount(rec[qmask], minlength=n_rec).astype(np.int64)
    base = np.concatenate([[0], np.cumsum(3 * lens + 3)]).astype(np.int64)
    img = np.full(int(base[-1]), ord(" "), np.uint8)
    img[base[:-1]] = ord(">")
    img[base[:-1] + 1] = ord("\n")
    img[base[1:] - 1] = ord("\n")
    rv = np.repeat(np.arange(n_rec), lens)
    k = np.arange(len(qual)) - np.repeat(np.cumsum(lens) - lens, lens)  # place of each value in its record
    p = base[rv] + 2 + 3 * k
    img[p] = ord("0") + qual // 10
    img[p + 1] = ord("0") + qual % 10
    return fasta, img.tobytes(), qual


def fastq_of(records, phred_offset=33, eol=b"\n"):
    """[(header, sequence bytes, Phred values)] -> FASTQ image"""
    return b"".join(b"@" + h.encode() + eol + s + eol + b"+" + eol + (np.asarray(q, np.uint8) + phred_offset).tobytes() + eol
                    for h, s, q in records)


def seeded_fastq(n, length, seed, phred_offset=33):
    """n seeded reads of `length` bases (acgt in upper case, about one N per 10 kbp, at least one), headers r00000000 ..,
    Phred values 0-40."""
    rng = np.random.default_rng(seed)
    w = 11 + 2 * length + 4  # "@r" + 8 digits + '\n', sequence + '\n', "+\n", qualities + '\n'
    rec = np.empty((n, w), np.uint8)
    rec[:, 0], rec[:, 1], rec[:, 10] = ord("@"), ord("r"), ord("\n")
    d = np.arange(n)
    for k in range(8):
        rec[:, 9 - k] = ord("0") + (d // 10 ** k) % 10
    seq = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, (n, length), dtype=np.uint8)]
    seq[rng.random((n, length)) < 1e-4] = ord("N")
    seq[0, 0] = ord("N")
    rec[:, 11:11 + length] = seq
    rec[:, 11 + length], rec[:, 12 + length], rec[:, 13 + length] = ord("\n"), ord("+"), ord("\n")
    rec[:, 14 + length:14 + 2 * length] = phred_offset + rng.integers(0, 41, (n, length), dtype=np.uint8)
    rec[:, -1] = ord("\n")
    return rec.tobytes()


# ---- the host-route helper (no GPU) -------------------------------------------------------------------------------
def test_host_images():
    image = b"@  r1 x\r\nAC gT\r\n+\r\n!+@I\r\n@r2\n\n+r2\n\n\n \n"
    fasta, qimg, q = host_images(image)
    assert fasta == b">  r1 x\r\nAC gT\r\n>r2\n\n"
    assert O.py_qual_records(qimg) == [(b"", [0, 10, 31, 40]), (b"", [])]
    assert q.tolist() == [0, 10, 31, 40]
    fasta, qimg, q = host_images(b"@a\nAC\n+\nhh", 64)
    assert fasta == b">a\nAC\n" and q.tolist() == [40, 40] and O.py_qual_records(qimg) == [(b"", [40, 40])]
    for blank in (b"", b" \n\n"):
        fasta, qimg, q = host_images(blank)
        assert fasta == b"" and qimg == b"" and len(q) == 0


# ---- device -------------------------------------------------------------------------------------------------------
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
def gene(gm, ctx):
    return gm.ICM.Read(ctx, os.path.join(G, "NC_000915.icm"))


def host_route(gm, ctx, image, phred_offset=33):
    fasta, qimg, _ = host_images(image, phred_offset)
    s = gm.SeqSet.from_fasta(ctx, fasta)
    s.set_quality_fasta(qimg)
    return s


def assert_same_set(a, b):
    """Offsets, headers, bases, GC, qualities and the non-acgt list (every sequence extracted on the minus strand)."""
    assert a.n == b.n and (a.off == b.off).all() and a.total == b.total
    assert a.headers == b.headers
    assert a.unpack() == b.unpack()
    if a.total:
        assert np.float64(a.gc_fraction()).view(np.uint64) == np.float64(b.gc_fraction()).view(np.uint64)
    qa, qb = a.qualities(), b.qualities()
    assert (qa is None) == (qb is None) and (qa is None or (qa == qb).all())
    if a.n:
        reg = (np.arange(a.n, dtype=np.int32), np.zeros(a.n, np.int32), np.diff(a.off).astype(np.int32),
               np.full(a.n, -1, np.int8))
        assert a.extract(*reg).unpack() == b.extract(*reg).unpack()


MODES = [{}, {"allow_indels": 1}, {"allow_subs": 1}]


def raw_starts(gm, ss, gene, flags):
    p = gm.Params(True, have_quality_file=1, **flags)
    gc = ss.gc_fraction()
    p.set_ignore_score_len(gc)
    ss.find_orfs(p)
    ss.score_orfs_mg(gene, gm.ICM.Build_Indep_WO_Stops(ss.ctx, gc), p)
    return ss.get_orfs(), ss.get_starts(), p.ignore_score_len, gc


@pytest.mark.gpu
@pytest.mark.parametrize("phred_offset", [33, 64])
@pytest.mark.parametrize("eol", ["lf", "crlf"])
def test_golden_reads(gm, ctx, gene, phred_offset, eol):
    reads = O.read_fasta(os.path.join(G, "seqs.fa.gz"))
    rng = np.random.default_rng(phred_offset)
    quals = [rng.integers(0, 41, len(s)).astype(np.uint8) for _, s in reads]
    image = fastq_of([(h, s, q) for (h, s), q in zip(reads, quals)], phred_offset, b"\r\n" if eol == "crlf" else b"\n")
    got = gm.SeqSet.from_fastq(ctx, image, phred_offset)
    want = host_route(gm, ctx, image, phred_offset)
    assert got.n == len(reads)
    assert_same_set(got, want)
    assert (got.qualities() == np.concatenate(quals)).all()
    assert [h.rstrip("\r") for h in got.headers] == [h for h, _ in reads]
    og = O.lib().orc_icm_read(os.path.join(G, "NC_000915.icm").encode())
    for flags in MODES:
        (orfs, ooff), (st, so), isl, gc = raw_starts(gm, got, gene, flags)
        (w_orfs, w_ooff), (w_st, w_so), _, _ = raw_starts(gm, want, gene, flags)
        assert orfs.tobytes() == w_orfs.tobytes() and (ooff == w_ooff).all()
        assert st.tobytes() == w_st.tobytes() and (so == w_so).all()
        # the first 200 reads against the oracle port, with the parsed qualities
        op = O.params(True, have_quality_file=1, **flags)
        op.ignore_score_len = isl
        oi = O.build_indep(gc)
        n_cmp = 0
        for i in range(200):
            s = O.filter_lower(reads[i][1])
            w_orfs = O.find_orfs(s, op)
            assert orfs[ooff[i]:ooff[i + 1]].tolist() == w_orfs.tolist()
            woff, wst = O.mg_score_orfs(og, oi, s, op, w_orfs, quals[i].astype(np.int32))
            for k in range(len(w_orfs)):
                o = ooff[i] + k
                assert starts_as_tuples(st[so[o]:so[o + 1]]) == starts_as_tuples(wst[woff[k]:woff[k + 1]])
                n_cmp += 1
        assert n_cmp > 200


EDGE = {
    "empty": b"",
    "zero_length_record": b"@a\nACGT\n+\nIIII\n@empty\n\n+\n\n@c\nGG\n+\nII\n",
    "zero_length_last_record": b"@a\nAC\n+\nII\n@b\n\n+\n",
    "at_and_plus_first_quality": b"@a\nACGT\n+\n@III\n@b\nAC\n+\n+I\n@c\nA\n+\n@\n",
    "plus_repeats_header": b"@r1 desc\nACGT\n+r1 desc\nIIII\n@r2\nA\n+  r2\nI\n@r3\r\nAC\r\n+r3\r\nII\r\n",
    "header_blanks_tabs_markers": b"@  lead\tx >y @z\nACGT\n+\nIIII\n@\ttab >\nA\n+\ttab >\nI\n@\nC\n+\nI\n@ \t\nGA\n+\nII\n",
    "iupac_both_cases": (b"@iupac\nacgtrymkswbdhvnACGTRYMKSWBDHVNuUx*-\n+\n" + b"!" * 35 + b"\n"
                         b"@minus\nNNNNrykmRYKMacgt\n+minus\n" + b"~" * 16 + b"\n"),
    "white_space_in_sequence": b"@a\r\nAC gT\tA\r\n+\r\nIIIII\r\n@b\nG G\n+\nII\n",
    "last_line_without_newline": b"@a\nACGT\n+\nIIII\n@b\nGG\n+\nII",
    "trailing_blank_lines": b"@a\nACGT\n+\nIIII\n\n\n\n \t\n\r\n\n",
    "one_record": b"@only\nACGTN\n+only\nIIII#\n",
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(EDGE))
def test_edge_cases(gm, ctx, case):
    image = EDGE[case]
    got = gm.SeqSet.from_fastq(ctx, image)
    assert_same_set(got, host_route(gm, ctx, image))
    expect = {"empty": 0, "zero_length_record": 3, "zero_length_last_record": 2, "one_record": 1,
              "trailing_blank_lines": 1, "header_blanks_tabs_markers": 4}
    if case in expect:
        assert got.n == expect[case]
    if case == "header_blanks_tabs_markers":
        assert got.headers == ["lead\tx >y @z", "\ttab >", "", "\t"]
    if case == "zero_length_record":
        assert got.off.tolist() == [0, 4, 4, 6] and got.qualities().tolist() == [40] * 6
    if case == "at_and_plus_first_quality":
        assert got.qualities().tolist() == [31, 40, 40, 40, 10, 40, 31]
    if case == "empty":
        assert got.total == 0 and got.qualities() is None


@pytest.fixture(scope="module")
def big_image():
    return seeded_fastq(1000000, 150, 2026)


@pytest.mark.gpu
def test_scale_million_reads(gm, ctx, big_image):
    got = gm.SeqSet.from_fastq(ctx, big_image)
    assert got.n == 1000000 and got.total == 150000000
    want = host_route(gm, ctx, big_image)
    assert_same_set(got, want)
    got.close()
    want.close()


@pytest.mark.gpu
def test_launches_do_not_grow_with_records(gm, ctx, big_image):
    counts = []
    for image in (seeded_fastq(10, 150, 7), big_image):
        before = ctx.launches
        s = gm.SeqSet.from_fastq(ctx, image)
        counts.append(ctx.launches - before)
        s.close()
    assert counts[0] == counts[1], counts


BAD = [
    (b"@a\nAC\n+\nII\nb\nAC\n+\nII\n", 33, r"record 2 \(line 5\): the header line does not start with '@' \(multi-line"),
    (b"@a\nACGT\nACGT\n+\nIIIIIIII\n", 33, r"record 1 \(line 3\): the separator line does not start with '\+' \(multi-line"),
    (b"@a\nAC\n+\nII\n\n@b\nAC\n+\nII\n", 33, r"record 2 \(line 5\): the header line does not start with '@'"),
    (b"@a\nAC\n-\nII\n", 33, r"record 1 \(line 3\): the separator line does not start with '\+'"),
    (b"@a\nAC\n+b\nII\n", 33, r"record 1 \(line 3\): the text after '\+' differs from the header"),
    (b"@ab\nAC\n+a\nII\n", 33, r"record 1 \(line 3\): the text after '\+' differs from the header"),
    (b"@a\nAC\n+\nIII\n", 33, r"record 1 \(line 4\): the quality line holds 3 characters, the sequence 2"),
    (b"@a\nA C\n+\nII\r\n@b\nAC\n+\nI\n", 33, r"record 2 \(line 8\): the quality line holds 1 characters, the sequence 2"),
    (b"@a\nAC\n+\nI \n", 33, r"record 1 \(line 4\): quality byte 32 at column 2 is outside \[33, 126\]"),
    (b"@a\nAC\n+\nI\x7f\n", 33, r"record 1 \(line 4\): quality byte 127 at column 2 is outside \[33, 126\]"),
    (b"@a\nAC\n+\nI?\n", 64, r"record 1 \(line 4\): quality byte 63 at column 2 is outside \[64, 126\] \(phred offset 64\)"),
    (b"@a\nAC\n+\nII\n@b\nAC\n+\nIII\n@c\nAC\n+\nI \n", 33, r"record 2 \(line 8\): the quality line holds 3"),
    (b"@a\nAC\n+\nII\n@b", 33, r"record 2 \(line 6\): truncated last record: the image ends before its sequence line"),
    (b"@a\nAC\n+\nII\n@b\nAC", 33, r"record 2 \(line 7\): truncated last record: the image ends before its '\+' line"),
    (b"@a\nAC\n+\nII\n@b\nAC\n+", 33, r"record 2 \(line 8\): truncated last record: the image ends before its quality line"),
    (b"@a\nAC\n+\nII\n", 0, r"phred_offset must be 33 or 64 \(got 0\)"),
    (b"@a\nAC\n+\nII\n", 50, r"phred_offset must be 33 or 64 \(got 50\)"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("k", range(len(BAD)))
def test_rejected(gm, ctx, k):
    image, phred_offset, msg = BAD[k]
    with pytest.raises(gm.GmgError, match=msg):
        gm.SeqSet.from_fastq(ctx, image, phred_offset)
    # no set comes back through the C-ABI either
    h, n = C.c_void_p(12345), C.c_int64(7)
    assert gm.lib().gmg_seqset_from_fastq(ctx.h, image, len(image), phred_offset, C.byref(h), C.byref(n)) != 0
    assert h.value is None and n.value == 0
    ok = gm.SeqSet.from_fastq(ctx, b"@x\nACGT\n+\nIIII\n")
    assert ok.n == 1 and ok.unpack() == b"acgt" and ok.qualities().tolist() == [40] * 4


@pytest.mark.gpu
def test_rejected_image_of_one_gib(gm, ctx):
    """A size check only: the call refuses before it reads the (small) buffer."""
    buf = np.zeros(16, np.uint8)
    h, n = C.c_void_p(), C.c_int64()
    assert gm.lib().gmg_seqset_from_fastq(ctx.h, buf.ctypes.data, 1 << 30, 33, C.byref(h), C.byref(n)) != 0
    assert h.value is None
    err = gm.lib().gmg_last_error().decode()
    assert "images of 1 GiB or more must be split at record boundaries (got 1073741824 bytes)" in err
    assert gm.SeqSet.from_fastq(ctx, b"@x\nA\n+\nI\n").n == 1


@pytest.mark.gpu
def test_qualities_of_other_routes(gm, ctx):
    q = np.arange(7, dtype=np.uint8) * 30
    assert (gm.SeqSet(ctx, seqs=[b"acg", b"tacg"], qual=q).qualities() == q).all()
    assert gm.SeqSet(ctx, seqs=[b"acg"]).qualities() is None
