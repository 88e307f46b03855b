"""glimmer-mg scoring with a per-read independent model (gmg_score_orfs_mg_gc, SeqSet.score_orfs_mg_gc): glimmer-mg -c
builds Build_Indep_WO_Stops from every read's own GC fraction.  The batched call must give, read by read, the bits of the
existing call on that read alone with that model (and the read's own Ignore_Score_Len), and of the oracle port."""
import os

import numpy as np
import pytest

import oracle_lib as O

G = O.GOLDEN
MODES = [{}, {"allow_indels": 1}, {"allow_subs": 1}]
ROUTES = [("GMG_K3MG_MODE", "0"), ("GMG_K3MG_MODE", "1"), ("GMG_PLAIN_LANES", "0"), ("GMG_PLAIN_LANES", "1"),
          ("GMG_MG_FORCE_UNCERT", "1"), ("GMG_MG_FORCE_UNCERT", "3"), ("GMG_INDEP_FORCE_HOST", "1")]


def seeded_reads(n, length, seed):
    """n seeded reads (lower-case acgt, a few n) and Phred values 0-40"""
    rng = np.random.default_rng(seed)
    seq = np.frombuffer(b"acgt", np.uint8)[rng.integers(0, 4, (n, length), dtype=np.uint8)]
    seq[rng.random((n, length)) < 1e-3] = ord("n")
    qual = rng.integers(0, 41, (n, length), dtype=np.uint8)
    return [r.tobytes() for r in seq], qual


def distinct_gc(n, seed):
    """seeded values in [0, 1] with 0, 1, 0.5 and pairs one ulp apart among them"""
    gc = np.random.default_rng(seed).random(n)
    special = [0.0, 1.0, 0.5, 0.3, np.nextafter(0.3, 1.0), 0.61, np.nextafter(0.61, 0.0), np.nextafter(0.5, 1.0)]
    gc[:min(n, len(special))] = special[:n]
    return gc


def fastq_image(reads, qual):
    return b"".join(b"@r%d\n%s\n+\n%s\n" % (i, r, (q + 33).tobytes()) for i, (r, q) in enumerate(zip(reads, qual)))


# ---- no GPU --------------------------------------------------------------------------------------------------------
def test_distinct_gc_values():
    gc = distinct_gc(100, 1)
    assert ((gc >= 0.0) & (gc <= 1.0)).all()
    assert gc[4] != gc[3] and np.nextafter(gc[3], 1.0) == gc[4]
    assert len(np.unique(gc.view(np.uint64))) == 100


# ---- device --------------------------------------------------------------------------------------------------------
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


@pytest.fixture(scope="module")
def ogene():
    return O.lib().orc_icm_read(os.path.join(G, "NC_000915.icm").encode())


def golden_reads():
    reads = [s for _, s in O.read_fasta(os.path.join(G, "seqs.fa.gz"))]
    qual = [np.random.default_rng(7 + i).integers(0, 41, len(s)).astype(np.uint8) for i, s in enumerate(reads)]
    return reads, qual


@pytest.fixture(scope="module")
def golden():
    return golden_reads()


def make_set(gm, ctx, reads, qual, with_qual):
    q = np.concatenate([np.asarray(x, np.uint8) for x in qual]) if with_qual else None
    return gm.SeqSet(ctx, seqs=reads, qual=q)


def params(gm, flags, with_qual, isl):
    p = gm.Params(True, have_quality_file=1 if with_qual else 0, **flags)
    p.c.ignore_score_len = isl
    return p


def isl_of(gm, gc):
    """Set_Ignore_Score_Len of every GC value; near GC 0 or 1 its int conversion overflows (a negative length, which the
    call rejects), and such reads get the boost switched off (INT32_MAX) as a caller would"""
    p = gm.Params(True)
    isl = np.array([p.set_ignore_score_len(float(x)) for x in gc], np.int64)
    return np.where(isl < 0, np.iinfo(np.int32).max, isl).astype(np.int32)


def starts_per_orf(starts, off):
    return [starts[off[o]:off[o + 1]].tobytes() for o in range(len(off) - 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("flags", MODES, ids=["plain", "indels", "subs"])
@pytest.mark.parametrize("with_qual", [False, True], ids=["noqual", "qual"])
@pytest.mark.parametrize("source", ["golden", "seeded", "fastq"])
def test_same_gc_equals_single_model(gm, ctx, gene, golden, flags, with_qual, source):
    """One GC value for every read: the whole start list and its offsets equal score_orfs_mg with Build_Indep_WO_Stops(gc)."""
    if source == "golden":
        reads, qual = golden
        ss = make_set(gm, ctx, reads, qual, with_qual)
    elif source == "seeded":
        reads, qual = seeded_reads(100_000, 100, 11)
        ss = make_set(gm, ctx, reads, qual, with_qual)
    else:
        if not with_qual:
            pytest.skip("a FASTQ set always carries qualities")
        reads, qual = seeded_reads(3000, 150, 12)
        ss = gm.SeqSet.from_fastq(ctx, fastq_image(reads, qual))
    gc = ss.gc_fraction()
    p = params(gm, flags, with_qual, 0)
    p.set_ignore_score_len(gc)
    ss.find_orfs(p)
    n1 = ss.score_orfs_mg(gene, gm.ICM.Build_Indep_WO_Stops(ctx, gc), p)
    want, woff = ss.get_starts()
    n2 = ss.score_orfs_mg_gc(gene, np.full(ss.n, gc), p)
    got, goff = ss.get_starts()
    assert n1 == n2 and (woff == goff).all() and got.tobytes() == want.tobytes()


def check_against_oracle(gm, ctx, gene, ogene, reads, qual, gc, flags, with_qual, per_read_isl, n_api=0):
    """score_orfs_mg_gc on the whole set against the oracle read by read, and against the existing call on one-read sets
    for the first n_api reads; returns the context's flagged count"""
    ss = make_set(gm, ctx, reads, qual, with_qual)
    isl = isl_of(gm, gc)
    p = params(gm, flags, with_qual, 1000)
    ss.find_orfs(p)
    orfs, ooff = ss.get_orfs()
    ss.score_orfs_mg_gc(gene, gc, p, isl if per_read_isl else None)
    starts, soff = ss.get_starts()
    got = starts_per_orf(starts, soff)
    flagged = ctx.indep_flagged
    cache = {}
    for i, r in enumerate(reads):
        s = O.filter_lower(r)
        key = np.float64(gc[i]).view(np.uint64).item()
        if key not in cache:
            cache[key] = O.build_indep(float(gc[i]))
        op = O.params(True, have_quality_file=1 if with_qual else 0, **flags)
        op.ignore_score_len = int(isl[i]) if per_read_isl else 1000
        o0, o1 = ooff[i], ooff[i + 1]
        woff, wst = O.mg_score_orfs(ogene, cache[key], s, op, orfs[o0:o1], qual[i] if with_qual else None)
        for k in range(o1 - o0):
            assert got[o0 + k] == wst[woff[k]:woff[k + 1]].tobytes(), f"read {i} ORF {k} (gc {gc[i]!r})"
    for i in range(n_api):
        one = make_set(gm, ctx, [reads[i]], [qual[i]], with_qual)
        p1 = params(gm, flags, with_qual, int(isl[i]) if per_read_isl else 1000)
        one.set_orfs(orfs[ooff[i]:ooff[i + 1]], np.array([0, ooff[i + 1] - ooff[i]], np.int64))
        one.score_orfs_mg(gene, gm.ICM.Build_Indep_WO_Stops(ctx, float(gc[i])), p1)
        st, off = one.get_starts()
        assert starts_per_orf(st, off) == got[ooff[i]:ooff[i + 1]], f"read {i}: one-read set differs"
    for m in cache.values():
        O.lib().orc_icm_free(m)
    return flagged


ORACLE_CASES = [({}, False), ({}, True), ({"allow_indels": 1}, False), ({"allow_indels": 1}, True), ({"allow_subs": 1}, False),
                ({"allow_subs": 1}, True)]
ORACLE_IDS = ["plain", "plain-qual", "indels", "indels-qual", "subs", "subs-qual"]
ROUTE_CASES = [({}, False), ({"allow_indels": 1}, True), ({"allow_subs": 1}, False), ({"allow_subs": 1}, True)]
ROUTE_IDS = ["plain", "indels-qual", "subs", "subs-qual"]


@pytest.mark.gpu
@pytest.mark.parametrize("flags,with_qual", ORACLE_CASES, ids=ORACLE_IDS)
@pytest.mark.parametrize("per_read_isl", [True, False], ids=["isl", "no-isl"])
def test_distinct_gc_golden(gm, ctx, gene, ogene, golden, flags, with_qual, per_read_isl):
    reads, qual = golden
    check_against_oracle(gm, ctx, gene, ogene, reads, qual, distinct_gc(len(reads), 3), flags, with_qual, per_read_isl,
                         n_api=100)


@pytest.mark.gpu
@pytest.mark.parametrize("flags,with_qual", ORACLE_CASES, ids=ORACLE_IDS)
def test_distinct_gc_seeded(gm, ctx, gene, ogene, flags, with_qual):
    reads, qual = seeded_reads(4000, 100, 21)
    check_against_oracle(gm, ctx, gene, ogene, reads, qual, distinct_gc(len(reads), 5), flags, with_qual, True, n_api=300)


@pytest.mark.gpu
@pytest.mark.parametrize("var,val", ROUTES, ids=[f"{k}={v}" for k, v in ROUTES])
@pytest.mark.parametrize("flags,with_qual", ORACLE_CASES, ids=ORACLE_IDS)
def test_routes(gm, ctx, gene, ogene, golden, monkeypatch, var, val, flags, with_qual):
    """every route in every mode, with and without a quality file (-i without one: the qualities K2 synthesises open
    the gates)"""
    reads, qual = golden
    monkeypatch.setenv(var, val)
    flagged = check_against_oracle(gm, ctx, gene, ogene, reads[:200], qual[:200], distinct_gc(200, 9), flags, with_qual, True)
    print(f"{var}={val}: {flagged} model entries recomputed on the host")
    if var == "GMG_INDEP_FORCE_HOST":
        assert flagged > 0


@pytest.mark.gpu
@pytest.mark.parametrize("flags,with_qual", ROUTE_CASES, ids=ROUTE_IDS)
def test_reduction_after_call(gm, ctx, gene, golden, flags, with_qual):
    """reduce_starts_mg after the batched call equals the reduction after per-read calls of the existing API"""
    reads, qual = golden
    reads, qual = reads[:150], qual[:150]
    gc = distinct_gc(len(reads), 13)
    isl = isl_of(gm, gc)
    em = gm.EventModel(prior=-0.25, start_lo=[0.3, -0.4, -1.1], len_lo=np.random.default_rng(2).normal(0.0, 1.5, (1, 2, 2, 200)))
    ss = make_set(gm, ctx, reads, qual, with_qual)
    p = params(gm, flags, with_qual, 1000)
    ss.find_orfs(p)
    orfs, ooff = ss.get_orfs()
    ss.score_orfs_mg_gc(gene, gc, p, isl)
    ss.reduce_starts_mg(p, em)
    st, first, cnt, status = ss.get_reduced_starts()
    for i in range(len(reads)):
        one = make_set(gm, ctx, [reads[i]], [qual[i]], with_qual)
        one.set_orfs(orfs[ooff[i]:ooff[i + 1]], np.array([0, ooff[i + 1] - ooff[i]], np.int64))
        p1 = params(gm, flags, with_qual, int(isl[i]))
        one.score_orfs_mg(gene, gm.ICM.Build_Indep_WO_Stops(ctx, float(gc[i])), p1)
        one.reduce_starts_mg(p1, em)
        st1, first1, cnt1, status1 = one.get_reduced_starts()
        for k in range(ooff[i + 1] - ooff[i]):
            o = ooff[i] + k
            assert status[o] == status1[k] and cnt[o] == cnt1[k], f"read {i} ORF {k}"
            assert st[first[o]:first[o] + cnt[o]].tobytes() == st1[first1[k]:first1[k] + cnt1[k]].tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [{}, {"allow_indels": 1}], ids=["plain", "indels"])
def test_launches_do_not_grow(gm, ctx, gene, flags):
    """Building the models adds two launches to what score_orfs_mg launches on the same set, for 10 reads as for 10^5
    reads with 10^5 distinct GC values.  Plain glimmer-mg launches the same number in all; with -i the flat enumeration
    skips its level passes when a level has no candidate call, in either call."""
    counts = []
    for n in (10, 100_000):
        reads, qual = seeded_reads(n, 100, 31)
        ss = make_set(gm, ctx, reads, qual, False)
        p = params(gm, flags, False, 1000)
        ss.find_orfs(p)
        gc = distinct_gc(n, 33)
        isl = isl_of(gm, gc)
        indep = gm.ICM.Build_Indep_WO_Stops(ctx, 0.5)
        if flags:  # the same model for both calls, so that the flat passes see the same candidates
            gc, isl = np.full(n, 0.5), None
        ss.score_orfs_mg_gc(gene, gc, p, isl)  # warm: scratch sizes, topology
        ss.score_orfs_mg(gene, indep, p)
        before = ctx.launches
        ss.score_orfs_mg_gc(gene, gc, p, isl)
        mid = ctx.launches
        ss.score_orfs_mg(gene, indep, p)
        counts.append((mid - before, ctx.launches - mid))
    assert all(new == single + 2 for new, single in counts), counts
    if not flags:
        assert counts[0] == counts[1], counts


@pytest.mark.gpu
@pytest.mark.parametrize("bad", ["nan", "neg", "big", "isl"])
def test_rejected(gm, ctx, gene, golden, bad):
    reads, qual = golden
    ss = make_set(gm, ctx, reads[:20], qual[:20], False)
    p = params(gm, {}, False, 1000)
    ss.find_orfs(p)
    gc = np.full(20, 0.4)
    isl = np.full(20, 500, np.int32)
    if bad == "isl":
        isl[13] = -1
    else:
        gc[13] = {"nan": np.nan, "neg": -0.1, "big": 1.5}[bad]
    with pytest.raises(gm.GmgError, match="sequence 13"):
        ss.score_orfs_mg_gc(gene, gc, p, isl)
    with pytest.raises(gm.GmgError):
        ss.score_orfs_mg_gc(gene, gc[:5], p)
    gc[13], isl[13] = 0.4, 500
    n = ss.score_orfs_mg_gc(gene, gc, p, isl)
    got, off = ss.get_starts()
    p.c.ignore_score_len = 500
    assert n == ss.score_orfs_mg(gene, gm.ICM.Build_Indep_WO_Stops(ctx, 0.4), p)
    assert ss.get_starts()[0].tobytes() == got.tobytes()
