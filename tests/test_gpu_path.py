"""Path queries (KGEModel.path_rank_statistics, predict_path_topk; kge_eval_path_query_vectors, kge_eval_path_bits*).

One-hop forward paths must give rank_statistics' and predict_topk's results bit for bit on every counting path.  Longer
paths (inverse hops, ragged padding) are checked against the fold and raw scores of tests/path_oracle.c, with the answer
sets of a Python breadth-first search over the triple list; the traversal against that search on a graph with a hub, on
both filter-index layouts; and the fast counting paths against exact=True, also after an ambiguous-list overflow."""
import collections
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import kge_oracle as O

import path_oracle as P
from test_gpu_rank_stats import numpy_stats
from test_gpu_topk import FLAGS, MODELS, MODES, assert_same, load, make, oracle_topk, random_triples

gpu = pytest.mark.gpu
GAMMA = {"TransE": 9.0, "RotatE": 24.0, "pRotatE": 24.0, "ComplEx": 200.0, "DistMult": 500.0}


def bfs(triples, anchor, path, mode, nrel):
    """The answer set of one path query: the frontier {anchor} mapped hop by hop through the triple list."""
    fwd, bwd = collections.defaultdict(set), collections.defaultdict(set)
    for h, r, t in triples:
        fwd[(h, r)].add(t)
        bwd[(r, t)].add(h)
    hops = [int(h) for h in path if h != -1]
    front = {int(anchor)}
    for h in (reversed(hops) if mode == "head-batch" else hops):
        nxt = set()
        for e in front:
            if mode == "tail-batch":
                nxt |= fwd[(e, h)] if h < nrel else bwd[(h - nrel, e)]
            else:
                nxt |= bwd[(h, e)] if h < nrel else fwd[(e, h - nrel)]
        front = nxt
    return front


def answer_masks(triples, anchors, paths, mode, nentity, nrel):
    mask = np.zeros((len(anchors), nentity), dtype=bool)
    for i, (a, p) in enumerate(zip(anchors, paths)):
        mask[i, sorted(bfs(triples, a, p, mode, nrel))] = True
    return mask


def random_paths(rng, Q, L, nentity, nrel, ragged=True):
    anchors = rng.randint(nentity, size=Q)
    paths = rng.randint(2 * nrel, size=(Q, L))
    if ragged:
        for i in range(0, Q, 3):
            paths[i, rng.randint(1, L + 1):] = -1
    return anchors, paths


def one_hop(test, mode):
    t = np.asarray(test, dtype=np.int64)
    anchors, answers = (t[:, 2], t[:, 0]) if mode == "head-batch" else (t[:, 0], t[:, 2])
    return anchors, t[:, 1:2].copy(), answers


# ------------------------------------------------------------------------------------------------ L = 1 identity
SHAPES = [(14951, 1345, 1000), (300, 7, 10), (300, 7, 12)]


@gpu
@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("shape", SHAPES, ids=["full", "d10", "d12"])
def test_one_hop_path_equals_the_one_hop_calls(model, shape):
    nentity, nrel, d = shape
    m, st = make(model, nentity, nrel, d, GAMMA[model], seed=4)
    m = load(m, st)
    all_true = random_triples(nentity, nrel, 20000 if nentity > 1000 else 2000, seed=5, tail_range=nentity)
    rng = np.random.RandomState(6)
    test = [all_true[i] for i in rng.choice(len(all_true), 80, replace=False)]
    for mode in MODES:
        anchors, paths, answers = one_hop(test, mode)
        for exact in (False, True):
            want = m.rank_statistics(test, all_true, mode, exact=exact)
            got = m.path_rank_statistics(anchors, paths, answers, all_true, mode, exact=exact)
            np.testing.assert_array_equal(got, want, err_msg="%s %s exact=%s" % (model, mode, exact))
        for exclude in (None, all_true):
            queries = np.asarray(test, dtype=np.int64)
            want = m.predict_topk(queries, mode, k=20, exclude_triples=exclude)
            got = m.predict_path_topk(anchors, paths, mode, k=20, exclude_triples=exclude)
            assert_same(got[0], got[1], want[0].cpu().numpy(), want[1].cpu().numpy(), (model, mode, exclude is None))


# ------------------------------------------------------------------------------------------------ multi-hop vs oracle
@gpu
@pytest.mark.parametrize("model", MODELS)
def test_multi_hop_against_the_oracle(model):
    nentity, nrel, d, gamma = 300, 6, 12, GAMMA[model]
    m, st = make(model, nentity, nrel, d, gamma, seed=7)
    m = load(m, st)
    rho = O.embedding_range(gamma, d)
    triples = random_triples(nentity, nrel, 1500, seed=8, tail_range=nentity)
    rng = np.random.RandomState(9)
    for L in (2, 3):
        for mode in MODES:
            anchors, paths = random_paths(rng, 40, L, nentity, nrel)
            q = P.path_query_vectors(model, st, anchors, paths, mode, rho)
            raw = P.scores_from_q(model, st, q, mode, gamma, rho)
            mask = answer_masks(triples, anchors, paths, mode, nentity, nrel)
            ids, scores = oracle_topk(raw, mask, 25)
            got = m.predict_path_topk(anchors, paths, mode, k=25, exclude_triples=triples)
            assert_same(got[0], got[1], ids, scores, (model, L, mode))
            ids, scores = oracle_topk(raw, np.zeros_like(mask), 25)
            got = m.predict_path_topk(anchors, paths, mode, k=25)
            assert_same(got[0], got[1], ids, scores, (model, L, mode, "no exclusion"))
            answers = rng.randint(nentity, size=40)
            fake = [(a, 0, a) for a in answers]                  # numpy_stats reads the positive column only
            want = numpy_stats(raw, fake, mode, mask)
            stats, counts = m.path_rank_statistics(anchors, paths, answers, triples, mode, return_answer_counts=True)
            np.testing.assert_array_equal(stats, want, err_msg="%s L=%d %s" % (model, L, mode))
            np.testing.assert_array_equal(counts, mask.sum(1))


@gpu
@pytest.mark.parametrize("model", MODELS)
def test_fast_paths_equal_exact_also_after_an_overflow(model, monkeypatch):
    nentity, nrel, d = 2000, 9, 64
    m, st = make(model, nentity, nrel, d, GAMMA[model], seed=10)
    st["entity_embedding"][1000:] = st["entity_embedding"][:1000]       # twins: exact ties, so ambiguous pairs
    m = load(m, st)
    triples = random_triples(nentity, nrel, 8000, seed=11, tail_range=nentity)
    rng = np.random.RandomState(12)
    anchors, paths = random_paths(rng, 300, 3, nentity, nrel)
    answers = rng.randint(nentity, size=300)
    for mode in MODES:
        exact = m.path_rank_statistics(anchors, paths, answers, triples, mode, exact=True)
        np.testing.assert_array_equal(m.path_rank_statistics(anchors, paths, answers, triples, mode), exact)
        monkeypatch.setenv("KGE_EVAL_AMB_CAP", "4")
        np.testing.assert_array_equal(m.path_rank_statistics(anchors, paths, answers, triples, mode, query_chunk=128),
                                      exact)
        monkeypatch.delenv("KGE_EVAL_AMB_CAP")
        if model != "TransE":                             # the first pass overflowed its list of 4 pairs
            assert max(m._ws.get("gemm_last_ambiguous", 0), m._ws.get("two_stage_last_ambiguous", 0)) > 4


@gpu
@pytest.mark.parametrize("model", MODELS)
def test_inverse_hop_equals_the_other_mode(model):
    """(a, ~r, ?) and (?, r, a) have the same answer set; RotatE, ComplEx and DistMult also the same q and op."""
    nentity, nrel, d = 256, 5, 16
    m, st = make(model, nentity, nrel, d, GAMMA[model], seed=13)
    m = load(m, st)
    triples = random_triples(nentity, nrel, 2500, seed=14, tail_range=nentity)
    rng = np.random.RandomState(15)
    anchors, rels = rng.randint(nentity, size=50), rng.randint(nrel, size=(50, 1))
    a = m.predict_path_topk(anchors, rels + nrel, "tail-batch", k=nentity, exclude_triples=triples)
    b = m.predict_path_topk(anchors, rels, "head-batch", k=nentity, exclude_triples=triples)
    ia, ib = a[0].cpu().numpy(), b[0].cpu().numpy()
    for i in range(50):
        assert set(ia[i][ia[i] >= 0]) == set(ib[i][ib[i] >= 0])
    if model in ("RotatE", "ComplEx", "DistMult"):
        assert_same(a[0], a[1], ib, b[1].cpu().numpy(), model)


# ------------------------------------------------------------------------------------------------ traversal
def hub_graph(seed):
    """8000 entities, 6 relations; entity 0 links to 6000 tails under relation 0, everything else is sparse, and
    relation 5 is used once (so most frontiers through it empty)."""
    rng = np.random.RandomState(seed)
    nentity, nrel = 8000, 6
    tri = {(0, 0, int(t)) for t in rng.choice(nentity, 6000, replace=False)}
    tri |= {(int(rng.randint(nentity)), int(rng.randint(5)), int(rng.randint(nentity))) for _ in range(20000)}
    tri.add((1, 5, 2))
    return nentity, nrel, sorted(tri)


@gpu
@pytest.mark.parametrize("host_index", [False, True], ids=["dense", "sorted"])
def test_traversal_counts_equal_bfs(host_index, monkeypatch):
    if host_index:
        monkeypatch.setenv("KGE_FILTER_HOST_INDEX", "1")
    nentity, nrel, triples = hub_graph(16)
    m, st = make("DistMult", nentity, nrel, 8, 500.0, seed=17)
    m = load(m, st)
    rng = np.random.RandomState(18)
    for L in (1, 2, 3, 4):
        anchors, paths = random_paths(rng, 60, L, nentity, nrel)
        anchors[:10] = 0                                  # through the hub
        paths[:10, 0] = 0
        paths[10:15, 0] = 5                               # a frontier that empties
        for mode in MODES:
            mask = answer_masks(triples, anchors, paths, mode, nentity, nrel)
            _, counts = m.path_rank_statistics(anchors, paths, np.zeros(60, np.int64), list(triples), mode,
                                               return_answer_counts=True)
            np.testing.assert_array_equal(counts, mask.sum(1), err_msg="L=%d %s" % (L, mode))
    assert mask[:10].sum() > 0


@gpu
def test_exclusion_is_exactly_the_answer_set_complement():
    nentity, nrel = 200, 4
    m, st = make("RotatE", nentity, nrel, 8, 24.0, seed=19)
    m = load(m, st)
    triples = random_triples(nentity, nrel, 700, seed=20, tail_range=nentity)
    rng = np.random.RandomState(21)
    for mode in MODES:
        anchors, paths = random_paths(rng, 30, 3, nentity, nrel)
        ids = m.predict_path_topk(anchors, paths, mode, k=nentity, exclude_triples=triples)[0].cpu().numpy()
        mask = answer_masks(triples, anchors, paths, mode, nentity, nrel)
        for i in range(30):
            assert set(ids[i][ids[i] >= 0]) == set(np.nonzero(~mask[i])[0])
            assert np.all(ids[i][(~mask[i]).sum():] == -1)


# ------------------------------------------------------------------------------------------------ errors
@gpu
def test_bad_ids_raise_and_the_next_call_is_clean():
    nentity, nrel = 100, 4
    m, st = make("ComplEx", nentity, nrel, 8, 200.0, seed=22)
    m = load(m, st)
    triples = random_triples(nentity, nrel, 300, seed=23, tail_range=nentity)
    good_a, good_p, good_t = np.array([1, 2]), np.array([[0, 5], [1, -1]]), np.array([3, 4])
    bad = [(np.array([1, nentity]), good_p, good_t),                   # anchor
           (good_a, np.array([[0, 2 * nrel], [1, -1]]), good_t),       # hop id
           (good_a, np.array([[0, -2], [1, -1]]), good_t),             # negative hop id
           (good_a, np.array([[-1, 1], [1, -1]]), good_t),             # a hop after padding
           (good_a, good_p, np.array([3, -1]))]                        # answer
    want = m.path_rank_statistics(good_a, good_p, good_t, triples, "tail-batch")
    for a, p, t in bad:
        with pytest.raises(IndexError):
            m.path_rank_statistics(a, p, t, triples, "tail-batch")
        np.testing.assert_array_equal(m.path_rank_statistics(good_a, good_p, good_t, triples, "tail-batch"), want)
        if t is good_t:                                   # (predict_path_topk takes no answers)
            with pytest.raises(IndexError):
                m.predict_path_topk(a, p, "head-batch", exclude_triples=triples)
            m.predict_path_topk(good_a, good_p, "head-batch", exclude_triples=triples)
    for a, p in ((good_a, good_p[:, None]), (good_a[:1], good_p), (good_a, good_p[:, :0])):
        with pytest.raises(ValueError):
            m.predict_path_topk(a, p, "tail-batch")
    with pytest.raises(ValueError):
        m.predict_path_topk(good_a, good_p, "single")


# ------------------------------------------------------------------------------------------------ two ranks
def _gpu0_shareable():
    from test_gpu_topk import _gpu0_shareable as shareable
    return shareable()


@gpu
@pytest.mark.skipif(torch.cuda.is_available() and not _gpu0_shareable(), reason="GPU 0 is in an exclusive compute mode")
def test_path_calls_two_ranks_sharing_one_gpu():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "path_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, KGE_TEST_SAME_GPU="1"))
    if not (res.returncode == 0 and res.stdout.strip().endswith("ok")):
        sys.stderr.write(res.stdout[-3000:] + "\n" + res.stderr[-8000:])
    assert res.returncode == 0 and res.stdout.strip().endswith("ok"), "path worker failed (output on stderr)"
