"""Plain glimmer-mg on read sets takes the gene values of partial windows (the W-1 first positions of the reverse strand,
the W-1 last of the forward strand) from a dense per-read table (k1_partial_side) instead of from the K1 planes.  The raw
start lists, FP64 score bits included, must equal those of the routes that keep complete planes -- the tested K1 loop
(GMG_K1_FIX=0) and K2 + one thread per ORF (GMG_K3MG_MODE=1) -- and the oracle's, for reads of every length around the
window, reads with non-acgt bytes, several gene model windows, per-read independent models and the serial sums."""
import os

import numpy as np
import pytest

import config_parity as CP
import oracle_lib as O

pytestmark = pytest.mark.gpu
G = O.GOLDEN
# (window, depth): depth 7 takes the bucketed K1 kernel and the table (W <= 14); depth 5 the generic kernel, no table
MODELS = [(9, 7), (12, 7), (14, 7), (12, 5)]
ROUTES = [None, ("GMG_K1_FIX", "0"), ("GMG_K3MG_MODE", "1")]
IUPAC = b"nrykmswbdhvNRY"


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
def genome():
    return O.filter_lower(O.read_fasta(os.path.join(G, "NC_000915.fna.gz"))[0][1][:600000])


@pytest.fixture(scope="module", params=MODELS, ids=[f"w{w}d{d}" for w, d in MODELS])
def model(request, gm, ctx):
    w, d = request.param
    strs = [s.lower()[::-1] for _, s in O.read_fasta(os.path.join(G, "seqs.cluster-5.run1.filt.gene.fasta.gz"))]
    om = O.lib().orc_icm_train(O.cstr_array(strs), len(strs), w, d, 3)
    omip, oprob = O.icm_tables(om)
    yield w, gm.ICM.from_tables(ctx, w, d, 3, omip, oprob), om
    O.lib().orc_icm_free(om)


def read_set(genome, w, seed):
    """seeded genome slices of every length 0 .. 2W+2 (twenty of each) and of 99, 100, 101 bases (a hundred of each),
    every fifth one with one to three non-acgt bytes"""
    rng = np.random.default_rng(seed)
    lengths = [n for n in range(2 * w + 3) for _ in range(20)] + [n for n in (99, 100, 101) for _ in range(100)]
    reads = []
    for i, n in enumerate(lengths):
        a = int(rng.integers(0, len(genome) - n))
        r = bytearray(genome[a:a + n])
        if i % 5 == 0 and n:
            for _ in range(int(rng.integers(1, 4))):
                r[int(rng.integers(0, n))] = IUPAC[int(rng.integers(0, len(IUPAC)))]
        reads.append(bytes(r))
    return reads


def run_routes(gm, ctx, monkeypatch, reads, score):
    """score(ss) on a fresh set of `reads` under every route and with every certificate withdrawn; all raw start lists
    byte-identical -> (ORF table, ORF offsets, starts, start offsets) of the first run"""
    want = None
    for route in ROUTES:
        for uncert in (False, True):
            with monkeypatch.context() as m:
                if route:
                    m.setenv(*route)
                if uncert:
                    m.setenv("GMG_MG_FORCE_UNCERT", "1")
                ss = gm.SeqSet(ctx, seqs=reads)
                score(ss)
                got = (*ss.get_orfs(), *ss.get_starts())
                ss.close()
            if want is None:
                want = got
                continue
            assert got[0].tobytes() == want[0].tobytes() and (got[1] == want[1]).all(), (route, uncert)
            assert (got[3] == want[3]).all() and got[2].tobytes() == want[2].tobytes(), (route, uncert)
    assert len(want[2]) > 0
    return want


@pytest.mark.parametrize("min_gene_len", [75, 9])
def test_single_model(gm, ctx, genome, model, monkeypatch, min_gene_len):
    w, gene, om = model
    reads = read_set(genome, w, 100 + w)
    gc = gm.SeqSet(ctx, seqs=reads).gc_fraction()
    indep = gm.ICM.Build_Indep_WO_Stops(ctx, gc)
    p = gm.Params(True, min_gene_len=min_gene_len)
    p.set_ignore_score_len(gc)

    def score(ss):
        ss.find_orfs(p)
        ss.score_orfs_mg(gene, indep, p)

    orfs, ooff, starts, soff = run_routes(gm, ctx, monkeypatch, reads, score)
    a = np.frombuffer(b"".join(reads), np.uint8)
    off = np.concatenate([[0], np.cumsum([len(r) for r in reads])]).astype(np.int64)
    CP.check_scoring("mg", a, off, range(len(reads)), orfs, ooff, starts, soff, om, gc, ("taa", "tag", "tga"),
                     ignore_score_len=p.ignore_score_len, min_gene_len=min_gene_len)


def test_per_read_gc(gm, ctx, genome, model, monkeypatch):
    """score_orfs_mg_gc: every read with the independent model of its own (distinct) GC value"""
    w, gene, om = model
    reads = read_set(genome, w, 200 + w)
    gc = np.random.default_rng(w).random(len(reads))
    p = gm.Params(True, min_gene_len=9)
    p.c.ignore_score_len = 1000

    def score(ss):
        ss.find_orfs(p)
        ss.score_orfs_mg_gc(gene, gc, p)

    orfs, ooff, starts, soff = run_routes(gm, ctx, monkeypatch, reads, score)
    op = O.params(True, min_gene_len=9)
    op.ignore_score_len = 1000
    for i, r in enumerate(reads):
        oi = O.build_indep(float(gc[i]))
        o0, o1 = ooff[i], ooff[i + 1]
        woff, wst = O.mg_score_orfs(om, oi, O.filter_lower(r), op, orfs[o0:o1])
        O.lib().orc_icm_free(oi)
        for k in range(o1 - o0):
            assert starts[soff[o0 + k]:soff[o0 + k + 1]].tobytes() == wst[woff[k]:woff[k + 1]].tobytes(), f"read {i} ORF {k}"
