"""Gene extraction on the device (gmg_seqset_extract, SeqSet.extract, regions_from_coords): regions of a resident set equal
gmg_seqset_create on the strings extract (Util/extract.cc) forms on the host, raw IUPAC codes complemented before Filter;
the NC_000915 genome plus the .train coordinates trains the reference library's model file byte for byte."""
import gzip
import hashlib
import json
import os

import numpy as np
import pytest

import oracle_lib as O

G = O.GOLDEN

# Complement (Common/delcher.cc) of the IUPAC codes, case kept; every other byte becomes n
COMP = np.full(256, ord("n"), np.uint8)
for _a, _b in zip("acgtrymkswbdhvn", "tgcayrkmswvhdbn"):
    COMP[ord(_a)], COMP[ord(_a.upper())] = ord(_b), ord(_b.upper())


def host_extract(seqs, seq, lo, length, strand):
    """The strings extract writes for the regions (the host route)."""
    out = []
    for s, a, n, d in zip(seq.tolist(), lo.tolist(), length.tolist(), strand.tolist()):
        x = seqs[s][a:a + n]
        out.append(x if d > 0 else COMP[np.frombuffer(x, np.uint8)][::-1].tobytes())
    return out


def _genome():
    return O.read_fasta(os.path.join(G, "NC_000915.fna.gz"))


def _train_records():
    return O.read_fasta(os.path.join(G, "NC_000915.train.gz"))


def _predict_lines():
    return gzip.open(os.path.join(G, "NC_000915.run1.predict.gz")).read().decode().splitlines()


# ---- coordinate parser (no GPU) ---------------------------------------------------------------------------------
def test_regions_from_coords():
    import glimmer_mg_b200 as g
    genome = _genome()
    raw = genome[0][1]
    recs = _train_records()
    seq, lo, length, strand = g.regions_from_coords([h for h, _ in recs])
    assert len(seq) == 1161 and (seq == 0).all()
    assert seq.dtype == np.int32 and lo.dtype == np.int32 and length.dtype == np.int32 and strand.dtype == np.int8
    # every record is its header's span with the stop dropped, IUPAC codes complemented before Filter on the minus strand
    strings = host_extract([raw], seq, lo, length, strand)
    assert [s.lower() for s in strings] == [r.lower() for _, r in recs]
    minus_iupac = {h.split()[0] for (h, r), d in zip(recs, strand.tolist()) if d < 0 and set(r.lower()) - set(b"acgt")}
    assert minus_iupac >= {"00082", "00277", "00321", "00684", "01087"}

    r = g.regions_from_coords(_predict_lines(), headers=[genome[0][0]], trim_stop=False)
    assert len(r[0]) == 1549 and (r[0] == 0).all() and int((r[1] + r[2]).max()) <= len(raw)

    # header selection by whole header or first word; text input; forward and minus coordinates
    seq, lo, length, strand = g.regions_from_coords(">b x\no1 10 21 +1\n\n>a\no2 30 19 -2\n", headers=["a", "b x y"],
                                                    trim_stop=False)
    assert seq.tolist() == [1, 0] and lo.tolist() == [9, 18] and length.tolist() == [12, 12]
    assert strand.tolist() == [1, -1]
    _, lo, length, _ = g.regions_from_coords(["o1 10 21", "o2 30 19"])
    assert lo.tolist() == [9, 21] and length.tolist() == [9, 9]
    for bad, kw, msg in [(["o1 100 10 +1"], {}, "wraps around"),
                         (["o1 10 100 -3"], {}, "wraps around"),
                         ([">x", "o1 1 9"], {}, "headers="),
                         ([">z", "o1 1 9"], {"headers": ["x"]}, "no sequence"),
                         (["o1 1 9"], {"headers": ["x"]}, "before the first"),
                         (["o1 1 2"], {}, "shorter than its stop"),
                         (["o1 1"], {}, "expected")]:
        with pytest.raises(g.GmgError, match=msg):
            g.regions_from_coords(bad, **kw)


# ---- device ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gm():
    import glimmer_mg_b200 as g
    return g


@pytest.fixture(scope="module")
def ctx(gm):
    c = gm.Context(0)
    yield c
    c.close()


def _same_set(a, b):
    """Offsets, bases and GC count of two sets are equal."""
    assert a.n == b.n and (a.off == b.off).all()
    assert a.unpack() == b.unpack()
    if a.total:
        assert np.float64(a.gc_fraction()).view(np.uint64) == np.float64(b.gc_fraction()).view(np.uint64)


def _synthetic(seed=11):
    """Seeded sequences of 1 base to 100 kbp, about 2 % of their bytes IUPAC codes (and a few other bytes) in both
    cases."""
    rng = np.random.default_rng(seed)
    lens = [1, 2, 3, 31, 32, 33, 63, 64, 65, 100, 997, 4096, 100000, 65537] + rng.integers(1, 20000, 20).tolist()
    odd = np.frombuffer(b"rymkswbdhvnRYMKSWBDHVNuUx-*", np.uint8)
    seqs = []
    for n in lens:
        s = np.frombuffer(b"acgtACGT", np.uint8)[rng.integers(0, 8, n)]
        m = rng.random(n) < 0.02
        s[m] = odd[rng.integers(0, len(odd), int(m.sum()))]
        seqs.append(s.tobytes())
    return seqs


def _regions(seqs, seed=12):
    """Thousands of regions on both strands: all 32 x 32 (start, end) word phases, sub-word regions, whole sequences,
    length 0 (also at a sequence end) and duplicates."""
    rng = np.random.default_rng(seed)
    lens = np.array([len(s) for s in seqs])
    big = int(np.argmax(lens))
    R = []
    for sp in range(32):
        for ep in range(32):
            a = 32 * int(rng.integers(0, 3000)) + sp
            b = 32 * int(rng.integers(a // 32 + 1, lens[big] // 32 - 1)) + ep
            R.append((big, a, b - a, 1 if (sp + ep) % 2 else -1))
            R.append((big, a, b - a, -1 if (sp + ep) % 2 else 1))
    for _ in range(3000):  # sub-word and short
        s = int(rng.integers(0, len(seqs)))
        n = int(rng.integers(0, min(lens[s], 70) + 1))
        a = int(rng.integers(0, lens[s] - n + 1))
        R.append((s, a, n, int(rng.choice([-1, 1]))))
    for s in range(len(seqs)):  # whole sequences, empty regions at both ends
        R += [(s, 0, int(lens[s]), 1), (s, 0, int(lens[s]), -1), (s, 0, 0, -1), (s, int(lens[s]), 0, 1)]
    for _ in range(1000):  # long
        s = int(rng.integers(0, len(seqs)))
        a, b = sorted(rng.integers(0, lens[s] + 1, 2).tolist())
        R.append((s, a, b - a, int(rng.choice([-1, 1]))))
    R += R[:50] + R[2048:2100]  # duplicates
    order = rng.permutation(len(R))
    R = [R[i] for i in order]
    cols = list(zip(*R))
    return (np.array(cols[0], np.int32), np.array(cols[1], np.int32), np.array(cols[2], np.int32),
            np.array(cols[3], np.int8))


def _reference_training_digest():
    return json.load(open(os.path.join(G, "reference_library.json")))["training"]["NC_000915.train.gz"]


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["from_fasta", "create"])
def test_golden_training_set(gm, ctx, route):
    """The genome on the device plus the .train coordinates = the .train records, and trains the reference's model
    file (build-icm -r, 12/7/3)."""
    genome = _genome()
    if route == "from_fasta":
        src = gm.SeqSet.from_fasta(ctx, gzip.open(os.path.join(G, "NC_000915.fna.gz")).read())
    else:
        src = gm.SeqSet(ctx, seqs=[genome[0][1]])
    recs = _train_records()
    ext = src.extract(*gm.regions_from_coords([h for h, _ in recs]))
    assert ext.n == 1161
    got = ext.unpack()
    for i, (_, r) in enumerate(recs):
        assert got[ext.off[i]:ext.off[i + 1]] == O.filter_lower(r), recs[i][0]
    tr = gm.ICMTraining(ctx, 12, 7, 3)
    img = tr.Train_Model(ext, reverse=True).image()
    assert hashlib.sha256(img).hexdigest() == _reference_training_digest()
    assert img == tr.Train_Model([r for _, r in recs], reverse=True).image()
    mip, _ = gm.ICM.Input(ctx, img).tables()
    want, _ = gm.ICM.Read(ctx, os.path.join(G, "NC_000915.icm")).tables()
    assert (mip == want).all()


@pytest.mark.gpu
def test_against_host_route(gm, ctx):
    seqs = _synthetic()
    src = gm.SeqSet(ctx, seqs=seqs)
    reg = _regions(seqs)
    assert len(reg[0]) > 5000 and (reg[3] < 0).sum() > 2000 and (reg[2] == 0).sum() > 20
    ext = src.extract(*reg)
    host = gm.SeqSet(ctx, seqs=host_extract(seqs, *reg))
    _same_set(ext, host)
    gene = gm.ICM.Read(ctx, os.path.join(G, "NC_000915.icm"))
    for frame in (0, 2):
        assert (gene.score_strings(ext, frame).view(np.uint64) == gene.score_strings(host, frame).view(np.uint64)).all()
    # several training sets: forward only, minus only, mixed
    keep = np.flatnonzero(reg[2] >= 200)
    groups = [keep[reg[3][keep] > 0], keep[reg[3][keep] < 0], keep[::3]]
    ext_sets = [src.extract(*(x[k] for x in reg)) for k in groups]
    host_sets = [gm.SeqSet(ctx, seqs=host_extract(seqs, *(x[k] for x in reg))) for k in groups]
    for a, b in zip(ext_sets, host_sets):
        _same_set(a, b)
    tr = gm.ICMTraining(ctx, 12, 7, 3)
    got = [m.image() for m in tr.Train_Models(ext_sets, reverse=True)]
    want = [m.image() for m in tr.Train_Models(host_sets, reverse=True)]
    assert got == want


@pytest.mark.gpu
def test_extract_from_extracted(gm, ctx):
    """Regions of an extracted set equal the composed regions of the source: the minus strand's output keeps the
    complemented raw codes."""
    seqs = _synthetic(21)
    src = gm.SeqSet(ctx, seqs=seqs)
    s1, a1, n1, d1 = _regions(seqs, 22)
    mid = gm.SeqSet(ctx, seqs=host_extract(seqs, s1, a1, n1, d1))
    ext1 = src.extract(s1, a1, n1, d1)
    _same_set(ext1, mid)
    rng = np.random.default_rng(23)
    k = rng.integers(0, len(s1), 4000).astype(np.int32)
    n2 = np.array([rng.integers(0, n1[j] + 1) for j in k], np.int32)
    a2 = np.array([rng.integers(0, n1[j] - n2[i] + 1) for i, j in enumerate(k)], np.int32)
    d2 = rng.choice(np.array([-1, 1], np.int8), len(k))
    twice = ext1.extract(k, a2, n2, d2)
    # the same bases straight from the source
    fwd = d1[k] > 0
    a = np.where(fwd, a1[k] + a2, a1[k] + n1[k] - a2 - n2).astype(np.int32)
    once = src.extract(s1[k], a, n2, (d1[k] * d2).astype(np.int8))
    _same_set(twice, once)
    _same_set(twice, gm.SeqSet(ctx, seqs=host_extract(host_extract(seqs, s1, a1, n1, d1), k, a2, n2, d2)))


@pytest.mark.gpu
def test_predict_regions(gm, ctx):
    genome = _genome()
    src = gm.SeqSet.from_fasta(ctx, gzip.open(os.path.join(G, "NC_000915.fna.gz")).read())
    reg = gm.regions_from_coords(_predict_lines(), headers=src.headers, trim_stop=False)
    assert len(reg[0]) == 1549
    _same_set(src.extract(*reg), gm.SeqSet(ctx, seqs=host_extract([genome[0][1]], *reg)))


@pytest.mark.gpu
def test_launches_do_not_grow_with_regions(gm, ctx):
    genome = _genome()
    src = gm.SeqSet(ctx, seqs=[genome[0][1]])
    L = len(genome[0][1])
    rng = np.random.default_rng(5)
    counts = []
    for n in (10, 100000):
        lo = rng.integers(0, L - 2000, n).astype(np.int32)
        length = rng.integers(0, 2000, n).astype(np.int32)
        if n == 10:  # whole-genome regions: both calls carry non-acgt bytes into the output
            lo[:], length[:] = 0, L
        strand = rng.choice(np.array([-1, 1], np.int8), n)
        before = ctx.launches
        s = src.extract(np.zeros(n, np.int32), lo, length, strand)
        counts.append(ctx.launches - before)
        s.close()
    assert counts[0] == counts[1], counts


@pytest.mark.gpu
def test_bad_regions(gm, ctx):
    src = gm.SeqSet(ctx, seqs=[b"acgtnacgtacgt", b"acg"])
    ok = (np.array([0, 1], np.int32), np.array([2, 0], np.int32), np.array([5, 3], np.int32), np.array([1, -1], np.int8))
    for col, val, msg in [(0, 2, "region 1: sequence 2 out of range"),
                          (0, -1, "region 1: sequence -1 out of range"),
                          (1, -1, "region 1: start -1 is negative"),
                          (2, 4, r"region 1: \[0, 4\) is not inside its 3 bp sequence"),
                          (1, 1, r"region 1: \[1, 4\) is not inside"),
                          (2, -1, "region 1: "),
                          (3, 0, "region 1: strand 0 is not"),
                          (3, 2, "region 1: strand 2 is not")]:
        bad = [x.copy() for x in ok]
        bad[col][1] = val
        with pytest.raises(gm.GmgError, match=msg):
            src.extract(*bad)
    with pytest.raises(gm.GmgError, match="strands given"):
        src.extract(*ok[:3], ok[3][:1])
    good = src.extract(*ok)
    assert good.unpack() == b"gtcac" + b"cgt"
    empty = src.extract(*(x[:0] for x in ok))
    assert empty.n == 0 and empty.total == 0
    good.close()
    empty.close()
    src.close()
