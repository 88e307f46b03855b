"""Batched training (gmg_icm_train_many, ICMTraining.Train_Models, build-icm -B): every model of a batch is byte-identical
to training it alone, on every counting and level-finish route, in any order, and the batch costs the same number of
kernel launches whatever its size."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_lib as O

sys.path.insert(0, os.path.join(O.ROOT, "tools"))
import workloads as W  # noqa: E402

pytestmark = pytest.mark.gpu
G = O.GOLDEN
EXE = os.path.join(O.ROOT, "glimmer_mg_b200", "host", "bin", "build-icm")
GOLD_SETS = ("seqs.cluster-4.run1.filt.gene.fasta.gz", "seqs.cluster-5.run1.filt.gene.fasta.gz", "NC_000915.train.gz")
SHAPES = ((12, 7, 3), (12, 3, 1), (10, 5, 1))
# build_icm_cluster5.sha256.json keys by (shape, reverse)
DIGEST_KEY = {((12, 7, 3), True): "-r", ((12, 7, 3), False): "", ((10, 5, 1), True): "-r -d 5 -w 10 -p 1"}


@pytest.fixture(scope="module")
def gm():
    import glimmer_mg_b200 as g
    return g


@pytest.fixture(scope="module")
def ctx(gm):
    c = gm.Context(0)
    yield c
    c.close()


def _golden(name):
    return [s.lower() for _, s in O.read_fasta(os.path.join(G, name))]


def _cluster(k, n_clusters=16):
    """The training genes of config 5's cluster k (tests/test_gpu_configs.py::_cluster, without the genome)."""
    gc = float(np.linspace(0.30, 0.70, n_clusters)[k])
    ts, toff = W.coding(1500, 333, seed=W.READS100_SEED * 1000 + 500 + k, freq=W.reweight_gc(W.codon_freq(), gc))
    raw = ts.tobytes()
    return [raw[toff[i]:toff[i + 1]].decode() for i in range(len(toff) - 1)]


@pytest.fixture(scope="module")
def batch():
    """(name, strings) of the mixed batch: golden sets, 16 synthetic clusters, edge cases, one set twice."""
    sets = [(n, _golden(n)) for n in GOLD_SETS]
    sets += [(f"cluster{k}", _cluster(k)) for k in range(16)]
    sets += [("empty", []), ("one", [_cluster(3)[0]]), ("short", ["acgtacg", "ac", "t"])]
    sets.append(("cluster-5 again", sets[1][1]))
    return sets


def _alone(gm, ctx, shape, strs, reverse):
    try:
        return gm.ICMTraining(ctx, *shape).Train_Model(strs, reverse=reverse).image()
    except gm.GmgError as e:
        return e


def _many(gm, ctx, shape, sets, reverse):
    return [m.image() for m in gm.ICMTraining(ctx, *shape).Train_Models(sets, reverse=reverse)]


def _check_batch(gm, ctx, shape, sets, reverse, want):
    """Train_Models on `sets` equals `want` (images, or the error of a set that fails alone, which fails the batch)."""
    if any(isinstance(w, Exception) for w in want):
        with pytest.raises(gm.GmgError):
            _many(gm, ctx, shape, sets, reverse)
        keep = [i for i, w in enumerate(want) if not isinstance(w, Exception)]
        sets, want = [sets[i] for i in keep], [want[i] for i in keep]
    got = _many(gm, ctx, shape, sets, reverse)
    assert len(got) == len(want)
    for k, (a, b) in enumerate(zip(got, want)):
        assert a == b, f"model {k} of the batch differs from training it alone ({shape}, reverse={reverse})"


@pytest.mark.parametrize("reverse", [True, False])
@pytest.mark.parametrize("shape", SHAPES)
def test_batch_models_equal_single_training(gm, ctx, batch, tmp_path, shape, reverse):
    strs = [s for _, s in batch]
    want = [_alone(gm, ctx, shape, s, reverse) for s in strs]
    _check_batch(gm, ctx, shape, strs, reverse, want)
    digests = json.load(open(os.path.join(G, "build_icm_cluster5.sha256.json")))
    for k, name in enumerate(GOLD_SETS):
        s = [x[::-1] for x in strs[k]] if reverse else strs[k]
        o = O.lib().orc_icm_train(O.cstr_array(s), len(s), *shape)
        path = str(tmp_path / f"oracle{k}.icm")
        O.lib().orc_icm_write(o, path.encode())
        with open(path, "rb") as fp:
            assert want[k] == fp.read(), f"{name} {shape} reverse={reverse}: differs from the oracle"
        key = DIGEST_KEY.get((shape, reverse))
        if name.startswith("seqs.cluster-5") and key is not None:
            assert (hashlib.sha256(want[k]).hexdigest(), len(want[k])) == (digests[key]["sha256"], digests[key]["bytes"])


@pytest.mark.parametrize("env", [("GMG_K4_MI", "0"), ("GMG_K4_MI", "2"), ("GMG_K4_HIST", "1"), ("GMG_K4_MANY_GROUP", "1"),
                                 ("GMG_K4_MANY_GROUP", "5"), ("GMG_K4_MANY_GROUP", "1000")])
def test_batch_routes_give_the_same_bytes(gm, ctx, batch, monkeypatch, env):
    """Level finish on the host / on the device with every node re-done on the host, every model through the
    single-model histogram route, and groups of 1, 5 and all models: the bytes of training each set alone."""
    strs = [s for _, s in batch]
    want = [_alone(gm, ctx, (12, 7, 3), s, True) for s in strs]
    monkeypatch.setenv(*env)
    _check_batch(gm, ctx, (12, 7, 3), strs, True, want)


def test_batch_order_does_not_matter(gm, ctx, batch):
    strs = [s for name, s in batch if name != "empty"]
    base = _many(gm, ctx, (12, 7, 3), strs, True)
    perm = np.random.default_rng(11).permutation(len(strs))
    got = _many(gm, ctx, (12, 7, 3), [strs[i] for i in perm], True)
    for j, i in enumerate(perm):
        assert got[j] == base[i], f"model of set {i} changed when moved to position {j}"


def test_batch_is_one_pass_not_a_loop(gm, ctx):
    """With one group, the launches of a call do not grow with the number of direct-path models (the 32-model batch
    repeats the 4 sets of the small one, so both flag nodes at the same levels)."""
    sets = [_cluster(k) for k in (0, 5, 10, 15)]
    ss = [gm.SeqSet(ctx, seqs=s) for s in sets]
    tr = gm.ICMTraining(ctx, 12, 7, 3)
    counts = []
    for m in (4, 32):
        tr.Train_Models(ss * (m // 4), reverse=True)  # warm
        before = ctx.launches
        models = tr.Train_Models(ss * (m // 4), reverse=True)
        counts.append(ctx.launches - before)
        assert len(models) == m
    assert counts[0] == counts[1] and counts[0] <= 4 * 8, counts


def _write_fasta(path, strs):
    with open(path, "wb") as fp:
        for i, s in enumerate(strs):
            s = s.encode() if isinstance(s, str) else s
            fp.write(b">g%d\n" % i)
            for a in range(0, len(s), 60):
                fp.write(s[a:a + 60] + b"\n")
    return path


@pytest.mark.parametrize("opts", [["-r"], ["-r", "-p", "1"], ["-r", "-F"], ["-r", "-t"]])
def test_cli_batch_writes_what_single_runs_write(tmp_path, batch, opts):
    assert os.path.exists(EXE), "glimmer_mg_b200/host/bin/build-icm missing: run __graft_entry__.build()"
    inputs = [_write_fasta(str(tmp_path / f"in{k}.fa"), batch[i][1]) for k, i in enumerate((0, 1, 5, 20))]
    with open(tmp_path / "list", "w") as fp:
        for k, f in enumerate(inputs):
            fp.write(f"{f} {tmp_path / f'batch{k}.icm'}\n\n")
    r = subprocess.run([EXE, *opts, "-B", str(tmp_path / "list")], capture_output=True, timeout=600, stdin=subprocess.DEVNULL)
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    for k, f in enumerate(inputs):
        with open(f, "rb") as fin:
            s = subprocess.run([EXE, *opts, str(tmp_path / f"single{k}.icm")], stdin=fin, capture_output=True, timeout=600)
        assert s.returncode == 0, s.stderr.decode()[-2000:]
        assert open(tmp_path / f"batch{k}.icm", "rb").read() == open(tmp_path / f"single{k}.icm", "rb").read(), (opts, k)


@pytest.mark.parametrize("bad", ["empty", "missing"])
def test_cli_batch_rejects_bad_input_before_writing(tmp_path, batch, bad):
    good = _write_fasta(str(tmp_path / "good.fa"), batch[1][1])
    bad_path = str(tmp_path / "bad.fa")
    if bad == "empty":
        open(bad_path, "w").close()
    with open(tmp_path / "list", "w") as fp:
        fp.write(f"{good} {tmp_path / 'a.icm'}\n{bad_path} {tmp_path / 'b.icm'}\n")
    r = subprocess.run([EXE, "-r", "-B", str(tmp_path / "list")], capture_output=True, timeout=600)
    want = b"ERROR:  Cannot create model--no input data" if bad == "empty" else b"ERROR:  Could not open file  " + bad_path.encode()
    assert r.returncode != 0 and want in r.stderr and bad_path.encode() in r.stderr, r.stderr
    assert not os.path.exists(tmp_path / "a.icm") and not os.path.exists(tmp_path / "b.icm")
