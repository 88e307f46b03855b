"""glimmer-mg scoring with per-base qualities against the oracle port (oracle/icm_oracle.c), bit for bit, in every error
mode: plain, -i, -s, -i -s and -i with indel_max 1, each with and without a quality file.  glimmer-mg cleans the file's
values (Clean_Quality_454: 0 -> 1, non-final homopolymer bases raised to threshold + 1) under -i only; under -s alone
they reach Pass_Stop_Penalty as read, so a 0 on a stop base gives p_stop = 0 and +inf scores, and three stop bases of
163 or more (1 - 10^(-q/10) rounds to 1.0) give -inf penalties.

The reads are seeded to hit the edges: qualities at the ends of the tables on stop codons and homopolymer runs, runs of
1-8 bases at every phase of the 32-base chunks and 128-base tiles of K2, neighbouring reads where one ends and the next
starts with a run of the same base, stops at the first and last bases of a read (the substitution range test at its
limit), empty and very short reads.  Every test asserts that its edge case occurred."""
import math
import os

import numpy as np
import pytest

import oracle_lib as O

G = O.GOLDEN
GENE = os.path.join(G, "NC_000915.icm")
EDGE_Q = np.array([0, 1, 2, 17, 18, 19, 20, 40, 93, 162, 163, 255])
FILE_BIG = 999999  # what the quality file holds where the host array holds 255 (the device clamps it to 255)
GC_ONE = 0.41
MODES = {"plain": {}, "indels": {"allow_indels": 1}, "subs": {"allow_subs": 1},
         "indels-subs": {"allow_indels": 1, "allow_subs": 1}, "indels-max1": {"allow_indels": 1, "indel_max": 1}}
FWD_STOPS = (b"taa", b"tag", b"tga")
REV_STOPS = (b"tta", b"cta", b"tca")  # their reverse complements, read on the forward strand


def test_float_edge_of_the_stop_probability():
    """1 - 10^(-q/10) is 1.0 from q = 163 on and below 1.0 at 162: where the -inf penalties start"""
    assert 1.0 - math.pow(10.0, -163 / 10.0) == 1.0 and 1.0 - math.pow(10.0, -162 / 10.0) < 1.0


# ---- seeded inputs -------------------------------------------------------------------------------------------------
def make_inputs(seed=2026):
    """-> dict(reads, qual (uint8 per read), stats).  Reads 4k, 4k+1 are neighbours joined by a run of one base;
    reads 4k+2 start with a forward stop and 4k+3 end with a reverse one; short and empty reads in between."""
    rng = np.random.default_rng(seed)
    acgt = np.frombuffer(b"acgt", np.uint8)
    lens = [int(x) for x in rng.integers(1000, 3001, 32)] + [0, 1, 2, 3, 15, 74, 75, 76, 77, 0] + \
           [int(x) for x in rng.integers(1000, 3001, 32)]
    reads = []
    for i, L in enumerate(lens):
        s = acgt[rng.integers(0, 4, L)]
        p = 0
        while L and p < L:  # homopolymer runs of 1-8 bases, every ~30 bases
            r = int(rng.integers(1, 9))
            s[p:p + r] = acgt[rng.integers(0, 4)]
            p += r + int(rng.integers(5, 50))
        reads.append(s)
    for i in range(len(reads) - 1):
        a, b = reads[i], reads[i + 1]
        if len(a) < 100 or len(b) < 100:
            continue
        if i % 4 == 0:  # a run at the end of read i and the same base at the start of read i + 1
            base = acgt[rng.integers(0, 4)]
            a[len(a) - int(rng.integers(1, 9)):] = base
            b[:int(rng.integers(1, 9))] = base
        elif i % 4 == 2:  # a forward stop on bases 0..2 (lo - 3 = 0), a reverse one on L-3..L-1 (hi + 1 = L - 1)
            a[:3] = np.frombuffer(FWD_STOPS[i % 3], np.uint8)
            b[len(b) - 3:] = np.frombuffer(REV_STOPS[i % 3], np.uint8)
    quals = []
    st = dict(stop_zero=0, stop_high=0, run_q18=0, run_q19=0, neighbours=0)
    for s in reads:
        L = len(s)
        q = np.where(rng.random(L) < 0.5, EDGE_Q[rng.integers(0, len(EDGE_Q), L)], rng.integers(0, 41, L))
        txt = s.tobytes()
        for k in range(L - 2):  # stop codons of either strand: all three bases >= 163, or one of them 0
            if txt[k:k + 3] in FWD_STOPS or txt[k:k + 3] in REV_STOPS:
                u = rng.random()
                if u < 0.25:
                    q[k:k + 3] = rng.choice([163, 200, 255], 3)
                elif u < 0.5:
                    q[k + int(rng.integers(0, 3))] = 0
                st["stop_high"] += int((q[k:k + 3] >= 163).all())
                st["stop_zero"] += int((q[k:k + 3] == 0).any())
        # last bases of runs (cleaning leaves them alone): -i gates open at 18, not at 19
        last = np.ones(L, bool)
        if L > 1:
            last[:-1] = s[:-1] != s[1:]
        st["run_q18"] += int(((q == 18) & last).sum())
        st["run_q19"] += int(((q == 19) & last).sum())
        quals.append(q.astype(np.uint8))
    st["neighbours"] = sum(1 for i in range(len(reads) - 1) if len(reads[i]) and len(reads[i + 1])
                           and reads[i][-1] == reads[i + 1][0])
    reads = [s.tobytes() for s in reads]
    # run ends at every phase of the 32-base chunks and 128-base tiles (batch offsets, so read boundaries move them)
    off = np.concatenate([[0], np.cumsum([len(r) for r in reads])])
    phases = set()
    for i, r in enumerate(reads):
        a = np.frombuffer(r, np.uint8)
        if len(a) > 1:
            ends = np.flatnonzero((a[:-1] == a[1:]) & np.append(a[1:-1] != a[2:], True)) + 1
            phases.update(((off[i] + ends) % 128).tolist())
    st["run_end_phases"] = len(phases)
    return dict(reads=reads, qual=quals, stats=st)


@pytest.fixture(scope="module")
def inputs():
    return make_inputs()


def test_inputs_hit_the_edges(inputs):
    st = inputs["stats"]
    assert st["stop_zero"] > 50 and st["stop_high"] > 50 and st["run_q18"] > 50 and st["run_q19"] > 50, st
    assert st["neighbours"] >= 8 and st["run_end_phases"] == 128, st
    lens = [len(r) for r in inputs["reads"]]
    assert 0 in lens and 1 in lens and 2 in lens and 15 in lens and max(lens) > 2500


def source_quals(inputs, source):
    """the values the oracle sees for a source: the host array as is, the file with 999999 for 255, FASTQ capped at 93"""
    if source == "host":
        return [q.astype(np.int32) for q in inputs["qual"]]
    if source == "file":
        return [np.where(q == 255, FILE_BIG, q.astype(np.int32)) for q in inputs["qual"]]
    return [np.minimum(q, 93).astype(np.int32) for q in inputs["qual"]]


def make_set(gm, ctx, inputs, source):
    reads = inputs["reads"]
    if source == "host":
        return gm.SeqSet(ctx, seqs=reads, qual=np.concatenate(inputs["qual"]))
    q = source_quals(inputs, source)
    if source == "file":
        s = gm.SeqSet(ctx, seqs=reads)
        s.set_quality_fasta(b"".join(b">r%d\n%s\n" % (i, b" ".join(b"%d" % v for v in x)) for i, x in enumerate(q)))
        return s
    return gm.SeqSet.from_fastq(ctx, b"".join(b"@r%d\n%s\n+\n%s\n" % (i, r, (x + 33).astype(np.uint8).tobytes())
                                               for i, (r, x) in enumerate(zip(reads, q))))


def per_read_gc(n):
    gc = np.random.default_rng(5).uniform(0.25, 0.75, n)
    gc[:4] = [0.3, np.nextafter(0.3, 1.0), 0.5, np.nextafter(0.5, 0.0)]
    return gc


def isl_of(gm, gc):
    p = gm.Params(True)
    return np.array([p.set_ignore_score_len(float(x)) for x in gc], np.int32)


# ---- the oracle, cached per (mode, quality file, source, call) -------------------------------------------------------
_ORACLE = {}


def oracle(gm, inputs, mode, hqf, source, call):
    key = (mode, hqf, source if hqf else None, call)
    if key in _ORACLE:
        return _ORACLE[key]
    og = O.lib().orc_icm_read(GENE.encode())
    quals = source_quals(inputs, source) if hqf else None
    n = len(inputs["reads"])
    gcs = np.full(n, GC_ONE) if call == "mg" else per_read_gc(n)
    isl = isl_of(gm, gcs)
    orfs, ooff, starts, soff = [], [0], [], [0]
    models = {}
    for i, r in enumerate(inputs["reads"]):
        s = O.filter_lower(r)
        op = O.params(True, have_quality_file=hqf, **MODES[mode])
        op.ignore_score_len = int(isl[i])
        if gcs[i] not in models:
            models[gcs[i]] = O.build_indep(float(gcs[i]))
        w = O.find_orfs(s, op)
        woff, wst = O.mg_score_orfs(og, models[gcs[i]], s, op, w, None if quals is None else quals[i])
        orfs.append(w)
        ooff.append(ooff[-1] + len(w))
        starts.append(wst)
        soff.extend((soff[-1] + np.asarray(woff[1:], np.int64)).tolist())
    for m in models.values():
        O.lib().orc_icm_free(m)
    O.lib().orc_icm_free(og)
    res = (np.concatenate(orfs), np.array(ooff, np.int64), np.concatenate(starts), np.array(soff, np.int64))
    _ORACLE[key] = res
    return res


def device(gm, ctx, gene, inputs, mode, hqf, source, call, threshold=None):
    ss = make_set(gm, ctx, inputs, source)
    p = gm.Params(True, have_quality_file=hqf, **MODES[mode])
    if threshold is not None:
        p.c.indel_quality_threshold = threshold
    ss.find_orfs(p)
    if call == "mg":
        p.set_ignore_score_len(GC_ONE)
        ss.score_orfs_mg(gene, gm.ICM.Build_Indep_WO_Stops(ctx, GC_ONE), p)
    else:
        gc = per_read_gc(ss.n)
        ss.score_orfs_mg_gc(gene, gc, p, isl_of(gm, gc))
    orfs, ooff = ss.get_orfs()
    starts, soff = ss.get_starts()
    return ss, (orfs, ooff, starts, soff)


def assert_same(got, want, what):
    """ORF tables and raw start lists byte for byte; the message counts the ORFs whose lists differ"""
    orfs, ooff, st, so = got
    w_orfs, w_ooff, w_st, w_so = want
    assert orfs.tobytes() == w_orfs.tobytes() and (ooff == w_ooff).all(), f"{what}: ORF tables differ"
    if (so == w_so).all() and st.tobytes() == w_st.tobytes():
        return
    n = len(so) - 1
    bad = [o for o in range(n) if st[so[o]:so[o + 1]].tobytes() != w_st[w_so[o]:w_so[o + 1]].tobytes()]
    raise AssertionError(f"{what}: start lists of {len(bad)} of {n} ORFs differ from the oracle (first: ORF {bad[:5]})")


def count_scores(starts):
    sc = starts["score"]
    return int(np.isposinf(sc).sum()), int(np.isneginf(sc).sum()), int((starts["n_err"] > 0).sum())


# ---- device ---------------------------------------------------------------------------------------------------------
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
    return gm.ICM.Read(ctx, GENE)


CASES = [(m, 0, "host") for m in MODES] + [(m, 1, s) for m in MODES for s in ("host", "file", "fastq")]


@pytest.mark.gpu
@pytest.mark.parametrize("call", ["mg", "gc"])
@pytest.mark.parametrize("mode,hqf,source", CASES, ids=[f"{m}-{'qual' if h else 'noqual'}-{s}" for m, h, s in CASES])
def test_matches_oracle(gm, ctx, gene, inputs, mode, hqf, source, call):
    _, got = device(gm, ctx, gene, inputs, mode, hqf, source, call)
    want = oracle(gm, inputs, mode, hqf, source, call)
    assert_same(got, want, f"{mode} quality file {hqf} {source} {call}")
    pinf, ninf, n_err = count_scores(want[2])
    assert len(want[2]) > 1000
    if MODES[mode].get("allow_subs") and hqf and not MODES[mode].get("allow_indels"):
        assert pinf > 0, pinf  # a 0 on a stop base
        assert ninf > 0 or source == "fastq", ninf  # three stop bases >= 163 (FASTQ carries at most 93)
    if MODES[mode].get("allow_indels"):
        assert pinf == 0 and n_err > 0  # cleaned: no 0 left; gates opened
    if mode == "plain" and hqf:  # qualities are unused without -i / -s
        _, without = device(gm, ctx, gene, inputs, mode, 0, source, call)
        assert got[2].tobytes() == without[2].tobytes() and (got[3] == without[3]).all()


ROUTES = [("GMG_K3MG_MODE", "1"), ("GMG_MG_FORCE_UNCERT", "1"), ("GMG_MG_FORCE_UNCERT", "3")]


@pytest.mark.gpu
@pytest.mark.parametrize("var,val", ROUTES, ids=[f"{k}={v}" for k, v in ROUTES])
@pytest.mark.parametrize("call", ["mg", "gc"])
@pytest.mark.parametrize("mode", ["subs", "indels", "indels-subs", "indels-max1"])
def test_routes_match_oracle(gm, ctx, gene, inputs, monkeypatch, var, val, call, mode):
    """the thread-per-ORF recursion and the ordered path of uncertified sequences, with a quality file holding 999999"""
    monkeypatch.setenv(var, val)
    ss, got = device(gm, ctx, gene, inputs, mode, 1, "file", call)
    if var == "GMG_MG_FORCE_UNCERT":
        assert ss.uncertified > 0
    assert_same(got, oracle(gm, inputs, mode, 1, "file", call), f"{var}={val} {mode} {call}")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["subs", "indels-subs"])
def test_reduction(gm, ctx, gene, inputs, mode):
    """reduce_starts_mg on start lists with infinite scores: exact ties must come back as status 2"""
    import config_parity as CP
    ss, (orfs, ooff, raw, soff) = device(gm, ctx, gene, inputs, mode, 1, "file", "mg")
    p = gm.Params(True, have_quality_file=1, **MODES[mode])
    n_len = max(len(r) for r in inputs["reads"]) // 3 + 8
    for model in (gm.EventModel(prior=0.0),
                  gm.EventModel(prior=-0.25, start_lo=[0.3, -0.4, -1.1],
                                len_lo=np.random.default_rng(2).normal(0.0, 1.5, (1, 2, 2, n_len)))):
        ss.reduce_starts_mg(p, model)
        red, first, cnt, status = ss.get_reduced_starts()
        ids = None if mode == "subs" else range(int(ooff[20]))  # -i -s: the ORFs of the first 20 reads (10^5 records)
        st = CP.check_reduction(orfs, ooff, [len(r) for r in inputs["reads"]], raw, soff, red, first, cnt, status,
                                p.min_gene_len, model, ids)
        assert st["kept_orfs"] > 50, st
    if mode == "subs":
        inf_orfs = sum(1 for o in range(len(orfs)) if np.isinf(raw["score"][soff[o]:soff[o + 1]]).any())
        assert inf_orfs > 0


@pytest.mark.gpu
def test_threshold_255_rejected(gm, ctx, gene, inputs):
    """threshold + 1 must fit the uint8 quality plane: 255 is refused with a message, the context stays usable, and 254
    (every base a gate but those the clamp brought to 255) still matches the oracle"""
    sub = dict(reads=inputs["reads"][32:44], qual=inputs["qual"][32:44])
    with pytest.raises(gm.GmgError, match=r"indel_quality_threshold 255 unsupported \(at most 254\)"):
        device(gm, ctx, gene, sub, "indels-max1", 1, "file", "mg", threshold=255)
    _, got = device(gm, ctx, gene, sub, "indels-max1", 1, "file", "mg", threshold=254)
    og = O.lib().orc_icm_read(GENE.encode())
    oi = O.build_indep(GC_ONE)
    op = O.params(True, have_quality_file=1, indel_quality_threshold=254, **MODES["indels-max1"])
    op.ignore_score_len = gm.Params(True).set_ignore_score_len(GC_ONE)
    orfs, ooff, st, so = got
    n = 0
    for i, (r, q) in enumerate(zip(sub["reads"], source_quals(sub, "file"))):
        s = O.filter_lower(r)
        w = O.find_orfs(s, op)
        assert orfs[ooff[i]:ooff[i + 1]].tobytes() == w.tobytes()
        woff, wst = O.mg_score_orfs(og, oi, s, op, w, q)
        a, b = so[ooff[i]], so[ooff[i + 1]]
        assert st[a:b].tobytes() == wst.tobytes() and ((so[ooff[i]:ooff[i + 1] + 1] - a) == woff).all(), f"read {i}"
        n += len(wst)
    assert n > 1000
    O.lib().orc_icm_free(oi)
    O.lib().orc_icm_free(og)
