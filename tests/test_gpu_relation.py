"""KGEModel.filtered_relation_ranks / predict_relations and the kge_eval_relation_* C ABI (relation prediction).

The oracle is the C oracle's 'single'-mode forward over every (h, r', t): the canonical exact scores, bit-identical to the
device's.  Ranks (stable descending tie rule, filtered relations skipped) and top-k lists (score descending, then id
ascending, NaN last) are formed from them in numpy.  The relation filter table and the ABI argument checks at the end need
no GPU.
"""
import ctypes
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import c_oracle as C
from oracle import kge_oracle as O

gpu = pytest.mark.gpu
FLAGS = {"TransE": (False, False), "DistMult": (False, False), "ComplEx": (True, True),
         "RotatE": (True, False), "pRotatE": (False, False)}
MODELS = list(FLAGS)
FULL = [("TransE", 14541, 237, 1000, 9.0), ("RotatE", 14951, 1345, 1000, 24.0), ("ComplEx", 40943, 11, 500, 200.0),
        ("RotatE", 123182, 37, 500, 24.0), ("pRotatE", 14951, 1345, 1000, 24.0), ("DistMult", 14951, 1345, 2000, 500.0)]


# make / load / assert_same: the patterns of test_gpu_topk.py
def make(model, nentity, nrel, d, gamma, seed=0, scale=3.0):
    from knowledgegraphembedding_b200 import KGEModel
    de, dr = FLAGS[model]
    st = O.init_tables(model, nentity, nrel, d, gamma, de, dr, seed=seed)
    st["entity_embedding"] = (st["entity_embedding"] * scale).astype(np.float32)
    m = KGEModel(model, nentity, nrel, d, gamma, double_entity_embedding=de, double_relation_embedding=dr)
    return m, st


def load(m, st):
    with torch.no_grad():
        m.entity_embedding.copy_(torch.from_numpy(st["entity_embedding"]))
        m.relation_embedding.copy_(torch.from_numpy(st["relation_embedding"]))
        if "modulus" in st and hasattr(m, "modulus"):
            m.modulus.copy_(torch.from_numpy(np.asarray(st["modulus"])))
    return m.cuda()


def assert_same(got_ids, got_scores, ids, scores, what=""):
    got_ids, got_scores = got_ids.cpu().numpy(), got_scores.cpu().numpy()
    np.testing.assert_array_equal(got_ids, ids, err_msg=str(what))
    a, b = got_scores.copy(), scores.copy()
    assert np.array_equal(np.isnan(a), np.isnan(b)), what
    a[np.isnan(a)] = 0.0
    b[np.isnan(b)] = 0.0
    a[a == 0] = 0.0                                     # -0.0 reads as +0.0
    b[b == 0] = 0.0
    np.testing.assert_array_equal(a.view(np.uint32), b.view(np.uint32), err_msg=str(what))


def assert_bits(got, want, what=""):
    got = got.cpu().numpy() if isinstance(got, torch.Tensor) else np.asarray(got)
    np.testing.assert_array_equal(got.view(np.uint32), np.asarray(want, dtype=np.float32).view(np.uint32),
                                  err_msg=str(what))


def random_triples(nentity, nrel, n, seed, tail_range=200):
    rng = np.random.RandomState(seed)
    return sorted({(int(rng.randint(nentity)), int(rng.randint(nrel)), int(rng.randint(min(tail_range, nentity))))
                   for _ in range(n)})


def relation_scores(model, st, queries, gamma, d, nrel):
    """[Q, nrel]: the C oracle's 'single' score of (h, r', t) for every query and relation."""
    q = np.asarray(queries, dtype=np.int64).reshape(-1, 3)
    sample = np.repeat(q, nrel, axis=0)
    sample[:, 1] = np.tile(np.arange(nrel), len(q))
    return C.forward(model, st, sample, "single", gamma, O.embedding_range(gamma, d)).reshape(len(q), nrel)


def relation_mask(triples, queries, nrel):
    """[Q, nrel]: (h, r', t) in triples."""
    q = np.asarray(queries, dtype=np.int64).reshape(-1, 3)
    mask = np.zeros((len(q), nrel), dtype=bool)
    if triples:
        by_pair = {}
        for h, r, t in triples:
            by_pair.setdefault((h, t), []).append(r)
        for i, (h, _, t) in enumerate(q.tolist()):
            mask[i, by_pair.get((h, t), [])] = True
    return mask


def oracle_ranks(raw, queries, filt):
    """1 + #{r' != r unfiltered: s > s_pos} + #{r' < r unfiltered: s == s_pos}; plus the dumped scores (a filtered
    column holds s_pos - 1)."""
    q = np.asarray(queries, dtype=np.int64).reshape(-1, 3)
    ranks = np.empty(len(q), dtype=np.int64)
    dumped = raw.copy()
    cols = np.arange(raw.shape[1])
    for i, r in enumerate(q[:, 1]):
        sp = raw[i, r]
        keep = ~filt[i] | (cols == r)
        ranks[i] = 1 + np.sum(keep & (cols != r) & ((raw[i] > sp) | ((raw[i] == sp) & (cols < r))))
        dumped[i, ~keep] = np.float32(sp) + np.float32(-1.0)
    return ranks, dumped


def oracle_topk(raw, mask, k):
    Q = raw.shape[0]
    ids = np.full((Q, k), -1, dtype=np.int64)
    scores = np.full((Q, k), -np.inf, dtype=np.float32)
    for q in range(Q):
        cand = np.nonzero(~mask[q])[0]
        s = raw[q, cand]
        nan = np.isnan(s)
        order = np.lexsort((cand, np.where(nan, 0.0, -s.astype(np.float64)), nan))[:k]
        ids[q, :order.size] = cand[order]
        scores[q, :order.size] = s[order]
    return ids, scores


def check_against_oracle(m, model, st, queries, all_true, gamma, d, nrel, ks, what):
    raw = relation_scores(model, st, queries, gamma, d, nrel)
    filt = relation_mask(all_true, queries, nrel)
    want_ranks, want_dump = oracle_ranks(raw, queries, filt)
    ranks, dump = m.filtered_relation_ranks(queries, all_true, return_scores=True)
    np.testing.assert_array_equal(ranks, want_ranks, err_msg=str(what))
    assert_bits(dump, want_dump, what)
    for exclude in (None, all_true):
        mask = relation_mask(exclude, queries, nrel)
        for k in ks:
            ids, scores = m.predict_relations(queries, k=k, exclude_triples=exclude)
            assert ids.shape == (len(queries), k) and ids.dtype == torch.int64 and scores.dtype == torch.float32
            assert ids.device == m.entity_embedding.device
            assert_same(ids, scores, *oracle_topk(raw, mask, k), what=(what, k, exclude is not None))


# ------------------------------------------------------------------------------------------------ bit-exact vs oracle
@gpu
@pytest.mark.parametrize("model,nentity,nrel,d,gamma", FULL)
def test_relation_bit_exact_at_baseline_shapes(model, nentity, nrel, d, gamma):
    m, st = make(model, nentity, nrel, d, gamma)
    m = load(m, st)
    all_true = random_triples(nentity, nrel, 30000, seed=2, tail_range=40)      # several relations per (h, t)
    rng = np.random.RandomState(3)
    queries = [all_true[i] for i in rng.choice(len(all_true), 24, replace=False)]
    check_against_oracle(m, model, st, queries, all_true, gamma, d, nrel, (1, 10, 256), model)


@gpu
@pytest.mark.parametrize("model", MODELS)
def test_relation_score_is_the_entity_score(model):
    """s(h, r, t) of the relation kernel == column t of the tail-batch entity scores of (h, r, ?) == the score
    predict_topk returns for t."""
    nentity, nrel, gamma = 500, 37, 24.0
    d = {"ComplEx": 500, "DistMult": 2000}.get(model, 1000)
    m, st = make(model, nentity, nrel, d, gamma, seed=5)
    m = load(m, st)
    rng = np.random.RandomState(9)
    queries = [(int(rng.randint(nentity)), int(rng.randint(nrel)), int(rng.randint(nentity))) for _ in range(16)]
    _, rel = m.filtered_relation_ranks(queries, [], return_scores=True)
    _, ent = m.filtered_ranks(queries, [], "tail-batch", return_scores=True)
    rel, ent = rel.cpu().numpy(), ent.cpu().numpy()
    for i, (h, r, t) in enumerate(queries):
        assert rel[i, r].view(np.uint32) == ent[i, t].view(np.uint32), (model, i)
    exclude = [(h, r, e) for h, r, t in queries for e in range(nentity) if e != t]
    ids, scores = m.predict_topk(queries, "tail-batch", k=1, exclude_triples=exclude)
    assert ids[:, 0].tolist() == [t for _, _, t in queries]
    assert_bits(scores[:, 0], [rel[i, r] for i, (_, r, _) in enumerate(queries)], model)


@gpu
@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("d", [10, 12])
def test_relation_small_ragged_shapes(model, d):
    """d = 10 takes the unaligned staging path; nrelation around the 64-relation tile; numpy input."""
    nentity, gamma = 300, 6.0
    for nrel in (2, 11, 63, 64, 65, 200):
        m, st = make(model, nentity, nrel, d, gamma, seed=1, scale=1.0)
        m = load(m, st)
        all_true = random_triples(nentity, nrel, 3000, seed=4, tail_range=30)
        queries = np.asarray(all_true[:100], dtype=np.int64)
        check_against_oracle(m, model, st, queries, all_true, gamma, d, nrel, (7, 100), (model, d, nrel))


@gpu
def test_relation_ties_ascending_ids_nan_last_and_signed_zero():
    model, nentity, nrel, d, gamma = "TransE", 200, 70, 16, 6.0
    m, st = make(model, nentity, nrel, d, gamma, seed=3, scale=1.0)
    R = st["relation_embedding"]
    R[10:50] = R[10]                                    # 40 identical rows: 40 tied scores
    R[3] = np.nan                                       # a NaN row: ranked after every number, never counted
    m = load(m, st)
    queries = [(1, 10, 2), (150, 30, 3), (30, 3, 100), (7, 49, 7)]
    raw = relation_scores(model, st, queries, gamma, d, nrel)
    ids, scores = m.predict_relations(queries, k=nrel)
    assert_same(ids, scores, *oracle_topk(raw, np.zeros_like(raw, dtype=bool), nrel))
    for row in ids.cpu().numpy():
        assert row[-1] == 3
        pos = [int(np.nonzero(row == j)[0][0]) for j in range(10, 50)]
        assert pos == list(range(pos[0], pos[0] + 40))   # tied ids adjacent and ascending
    ranks = m.filtered_relation_ranks(queries, [])
    np.testing.assert_array_equal(ranks, oracle_ranks(raw, queries, np.zeros_like(raw, dtype=bool))[0])
    assert ranks[0] == 1 + np.sum(raw[0] > raw[0, 10])                  # ascending ids inside the tie
    assert ranks[1] == 1 + np.sum(raw[1] > raw[1, 30]) + 20
    assert ranks[3] == 1 + np.sum(raw[3] > raw[3, 49]) + 39
    assert ranks[2] == 1                                # a NaN positive: nothing counts
    # DistMult with a +0.0 and a -0.0 relation row: both score zero and tie, in ascending id order
    m, st = make("DistMult", nentity, 5, d, gamma, seed=3, scale=1.0)
    st["relation_embedding"][1] = 0.0
    st["relation_embedding"][3] = -0.0
    m = load(m, st)
    queries = [(1, 3, 2), (150, 1, 3)]
    raw = relation_scores("DistMult", st, queries, gamma, d, 5)
    ids, scores = m.predict_relations(queries, k=5)
    assert_same(ids, scores, *oracle_topk(raw, np.zeros_like(raw, dtype=bool), 5))
    for row in ids.cpu().numpy():
        p1, p3 = int(np.nonzero(row == 1)[0][0]), int(np.nonzero(row == 3)[0][0])
        assert p3 == p1 + 1
    np.testing.assert_array_equal(m.filtered_relation_ranks(queries, []),
                                  oracle_ranks(raw, queries, np.zeros_like(raw, dtype=bool))[0])


# ------------------------------------------------------------------------------------------------ vs the filtered ranks
@gpu
@pytest.mark.parametrize("model", MODELS)
def test_relation_topk_agrees_with_ranks(model):
    """exclude = all true triples except the test triples (whose (h, t) pairs are distinct): the candidates of a query are
    exactly those its filtered rank counts, plus its answer, so the answer sits at position rank - 1 when rank <= k."""
    nentity, nrel, gamma = 14951, 1345, 24.0
    d = {"ComplEx": 500, "DistMult": 2000}.get(model, 1000)
    m, st = make(model, nentity, nrel, d, gamma, seed=5)
    m = load(m, st)
    all_true = random_triples(nentity, nrel, 30000, seed=7, tail_range=30)
    seen, test = set(), []
    for tr in all_true[::29]:
        if (tr[0], tr[2]) not in seen:
            seen.add((tr[0], tr[2]))
            test.append(tr)
    test_set = set(test)
    exclude = [tr for tr in all_true if tr not in test_set]
    ranks = m.filtered_relation_ranks(test, all_true)
    hits = 0
    for k in (10, 256):
        ids = m.predict_relations(test, k=k, exclude_triples=exclude)[0].cpu().numpy()
        for q, (tr, r) in enumerate(zip(test, ranks)):
            if r <= k:
                assert ids[q, r - 1] == tr[1], (model, k, q, r)
                hits += 1
            else:
                assert tr[1] not in ids[q], (model, k, q, r)
    assert hits > 0


# ------------------------------------------------------------------------------------------------ boundaries
@gpu
def test_relation_chunking_empty_queries_and_padding():
    model, nentity, nrel, d, gamma = "RotatE", 301, 5, 12, 6.0
    m, st = make(model, nentity, nrel, d, gamma, seed=2, scale=1.0)
    m = load(m, st)
    rng = np.random.RandomState(6)
    queries = np.stack([rng.randint(nentity, size=5000), rng.randint(nrel, size=5000), rng.randint(nentity, size=5000)], 1)
    all_true = random_triples(nentity, nrel, 20000, seed=8, tail_range=nentity)
    raw = relation_scores(model, st, queries, gamma, d, nrel)
    ranks = m.filtered_relation_ranks(queries, all_true)                             # Q > 4096: two chunks
    np.testing.assert_array_equal(ranks, oracle_ranks(raw, queries, relation_mask(all_true, queries, nrel))[0])
    ids, scores = m.predict_relations(torch.from_numpy(queries), k=3)
    assert_same(ids, scores, *oracle_topk(raw, np.zeros_like(raw, dtype=bool), 3))
    assert m.filtered_relation_ranks([], all_true).shape == (0,)
    ids, scores = m.predict_relations([], k=3)
    assert tuple(ids.shape) == (0, 3) and tuple(scores.shape) == (0, 3)
    # k larger than the relations left: 2 of the 5 relations excluded for the first query
    h, t = int(queries[0, 0]), int(queries[0, 2])
    exclude = [(h, 1, t), (h, 4, t)]
    q = [(h, 0, t), (h, 0, (t + 1) % nentity)]
    ids, scores = m.predict_relations(q, k=64, exclude_triples=exclude)
    raw = relation_scores(model, st, q, gamma, d, nrel)
    assert_same(ids, scores, *oracle_topk(raw, relation_mask(exclude, q, nrel), 64))
    assert sorted(ids[0, :3].tolist()) == [0, 2, 3] and (ids[0, 3:] == -1).all() and torch.isneginf(scores[0, 3:]).all()
    assert sorted(ids[1, :5].tolist()) == list(range(5)) and (ids[1, 5:] == -1).all()


@gpu
def test_relation_slices_sum_and_merge_to_full_range():
    from knowledgegraphembedding_b200 import _lib, shard_bounds
    from knowledgegraphembedding_b200.model import _ptr, _stream
    lib = _lib.load()
    for model, nrel in (("RotatE", 200), ("pRotatE", 11), ("ComplEx", 65)):
        nentity, d, gamma = 1003, 64, 12.0
        m, st = make(model, nentity, nrel, d, gamma, seed=4, scale=1.0)
        m = load(m, st)
        dev = m.entity_embedding.device
        rng = np.random.RandomState(8)
        test = np.stack([rng.randint(nentity, size=100), rng.randint(nrel, size=100), rng.randint(nentity, size=100)], 1)
        q = torch.from_numpy(test).to(dev)
        Q, k, words = len(test), 50, (nrel + 31) // 32
        desc, stt = m._descriptor(), _stream(dev)
        rel_table, phase = m._relation_operands(desc, dev, stt)
        tail = _lib.MODE_IDS["tail-batch"]
        qvec = torch.empty(Q * m.entity_dim, device=dev)
        pos = torch.empty(Q, device=dev)
        _lib.call("kge_eval_query_vectors", ctypes.byref(desc), tail, _ptr(q), Q, _ptr(qvec), None, stt)
        _lib.call("kge_eval_positive_scores", ctypes.byref(desc), tail, _ptr(qvec), _ptr(q), Q, _ptr(phase), _ptr(pos),
                  stt)
        bits = torch.zeros(Q * words, dtype=torch.int32, device=dev)

        def count(b, e):
            counts = torch.zeros(Q, dtype=torch.int32, device=dev)
            _lib.call("kge_eval_relation_count_ranks", ctypes.byref(desc), _ptr(q), Q, _ptr(rel_table), _ptr(phase),
                      _ptr(pos), _ptr(bits), b, e, _ptr(counts), None, stt)
            return counts

        def select(b, e):
            sb = int(lib.kge_eval_relation_topk_scratch_bytes(ctypes.byref(desc), Q, b, e, k))
            assert sb >= 0 and (sb == 0) == (b == e)
            scratch = torch.empty(max(sb, 1), dtype=torch.uint8, device=dev)
            keys = torch.empty((Q, k), dtype=torch.int64, device=dev)
            _lib.call("kge_eval_relation_topk", ctypes.byref(desc), _ptr(q), Q, _ptr(rel_table), _ptr(phase), None, b,
                      e, k, _ptr(keys), _ptr(scratch), sb, None, stt)
            return keys

        full_counts, full = count(0, nrel), select(0, nrel)
        slices = [shard_bounds(nrel, r, 8, align=64) for r in range(8)]     # mostly empty for 11 and 65 relations
        assert any(b == e for b, e in slices)
        assert torch.equal(sum(count(b, e) for b, e in slices), full_counts), model
        for b, e in slices:
            if b == e:
                assert not select(b, e).any()              # an empty slice: every key empty
        parts = torch.stack([select(b, e) for b, e in slices], dim=1).contiguous()
        merged = torch.empty_like(full)
        ids = torch.empty((Q, k), dtype=torch.int64, device=dev)
        scores = torch.empty((Q, k), dtype=torch.float32, device=dev)
        _lib.call("kge_eval_topk_merge", _ptr(parts), Q, 8, k, _ptr(merged), _ptr(ids), _ptr(scores), stt)
        assert torch.equal(merged, full), model
        raw = relation_scores(model, st, test, gamma, d, nrel)
        assert_same(ids, scores, *oracle_topk(raw, np.zeros_like(raw, dtype=bool), k), what=model)
        np.testing.assert_array_equal(full_counts.cpu().numpy() + 1,
                                      oracle_ranks(raw, test, np.zeros_like(raw, dtype=bool))[0])


def _run_worker(n, **env):
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "relation_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, **env))
    if not (res.returncode == 0 and res.stdout.strip().endswith("ok")):
        sys.stderr.write(res.stdout[-3000:] + "\n" + res.stderr[-8000:])
    assert res.returncode == 0 and res.stdout.strip().endswith("ok"), "relation worker failed (output on stderr)"


def _gpu0_shareable():
    """Two processes can hold contexts on GPU 0 only in the default compute mode."""
    try:
        import pynvml
        pynvml.nvmlInit()
        mode = pynvml.nvmlDeviceGetComputeMode(pynvml.nvmlDeviceGetHandleByIndex(0))
        return mode == pynvml.NVML_COMPUTEMODE_DEFAULT
    except Exception:
        return True


@gpu
@pytest.mark.skipif(torch.cuda.is_available() and not _gpu0_shareable(), reason="GPU 0 is in an exclusive compute mode")
def test_relation_multi_rank_two_ranks_sharing_one_gpu():
    _run_worker(2, KGE_TEST_SAME_GPU="1")


@gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_relation_multi_rank_one_gpu_per_rank():
    _run_worker(min(torch.cuda.device_count(), 8))


# ------------------------------------------------------------------------------------------------ other paths, API
@gpu
def test_relation_calls_leave_entity_paths_unchanged():
    model, nentity, nrel, d, gamma = "pRotatE", 3001, 11, 64, 12.0
    m, st = make(model, nentity, nrel, d, gamma, seed=7, scale=1.0)
    m = load(m, st)
    all_true = random_triples(nentity, nrel, 5000, seed=10, tail_range=nentity)
    test = all_true[:300]
    for mode in ("head-batch", "tail-batch"):
        ranks = m.filtered_ranks(test, all_true, mode)
        ids, scores = m.predict_topk(test, mode, k=20, exclude_triples=all_true)
        m.filtered_relation_ranks(test, all_true)
        m.predict_relations(test, k=256, exclude_triples=all_true)
        np.testing.assert_array_equal(m.filtered_ranks(test, all_true, mode), ranks)
        ids2, scores2 = m.predict_topk(test, mode, k=20, exclude_triples=all_true)
        assert torch.equal(ids2, ids) and torch.equal(scores2.view(torch.int32), scores.view(torch.int32))


@gpu
def test_relation_errors():
    m, st = make("TransE", 100, 3, 8, 6.0, scale=1.0)
    m = load(m, st)
    q = [(1, 0, 2)]
    for k in (0, 257, True, 2.5):
        with pytest.raises(ValueError):
            m.predict_relations(q, k=k)
    with pytest.raises(IndexError):
        m.predict_relations([(1, 0, 2), (100, 0, 2)], k=3)                  # head out of range
    with pytest.raises(IndexError):
        m.predict_relations([(1, 0, -1)], k=3)                              # tail out of range
    with pytest.raises(IndexError):
        m.filtered_relation_ranks([(1, 3, 2)], [])                           # relation out of range
    with pytest.raises(IndexError):
        m.filtered_relation_ranks([(1, 0, 100)], [])                         # tail out of range
    ids, _ = m.predict_relations([(1, 10**9, 2)], k=3)                      # the relation slot is ignored
    assert ids.shape == (1, 3) and sorted(ids[0].tolist()) == [0, 1, 2]
    assert m.filtered_relation_ranks(q, []).shape == (1,)                  # the error flag was cleared


# ------------------------------------------------------------------------------------------------ no GPU needed
def test_relation_filter_table_matches_a_python_set():
    from knowledgegraphembedding_b200.filter_index import relation_table
    nentity, nrel = 97, 13
    triples = random_triples(nentity, nrel, 4000, seed=11, tail_range=20)
    keys, offsets, rels = relation_table(triples, nentity)
    assert keys.dtype == np.int64 and offsets.dtype == np.int64 and rels.dtype == np.int32
    assert np.all(np.diff(keys) > 0) and offsets[0] == 0 and offsets[-1] == len(triples) == rels.size
    got = set()
    for i, key in enumerate(keys.tolist()):
        h, t = divmod(key, nentity)
        got.update((h, int(r), t) for r in rels[offsets[i]:offsets[i + 1]])
    assert got == set(triples)
    keys, offsets, rels = relation_table([], nentity)
    assert keys.size == 0 and offsets.tolist() == [0] and rels.size == 0


def test_relation_abi_argument_errors_without_a_gpu():
    from knowledgegraphembedding_b200 import _lib
    lib = _lib.load()
    desc = _lib.KgeModelStruct(model=_lib.TRANSE, device=0, nentity=100, nrelation=40, hidden_dim=8, entity_dim=8,
                               relation_dim=8, gamma=6.0, embedding_range=1.0, entity=16, relation=16, modulus=None)
    d = ctypes.byref(desc)
    for k in (0, 257):
        assert lib.kge_eval_relation_topk_scratch_bytes(d, 10, 0, 40, k) == _lib.ERR_INVALID
        assert b"outside [1, 256]" in lib.kge_last_error()
        assert lib.kge_eval_relation_topk(d, 16, 10, None, None, None, 0, 40, k, 16, 16, 1 << 20, None,
                                          None) == _lib.ERR_INVALID
    for b, e in ((0, 41), (-1, 5), (30, 20)):
        assert lib.kge_eval_relation_topk_scratch_bytes(d, 10, b, e, 5) == _lib.ERR_INVALID
        assert b"relation slice" in lib.kge_last_error()
        assert lib.kge_eval_relation_topk(d, 16, 10, None, None, None, b, e, 5, 16, 16, 1 << 20, None,
                                          None) == _lib.ERR_INVALID
        assert lib.kge_eval_relation_count_ranks(d, 16, 10, None, None, 16, 16, b, e, 16, None, None) == _lib.ERR_INVALID
        assert b"relation slice" in lib.kge_last_error()
    assert lib.kge_eval_relation_topk_scratch_bytes(d, -1, 0, 40, 5) == _lib.ERR_INVALID
    assert lib.kge_eval_relation_topk_scratch_bytes(d, 65535 * 64 + 1, 0, 40, 5) == _lib.ERR_INVALID
    assert b"queries per call" in lib.kge_last_error()
    # scratch: Q * ceil(slice / k) * k keys; none for an empty slice or no queries
    assert lib.kge_eval_relation_topk_scratch_bytes(d, 10, 0, 40, 7) == 8 * 10 * 42
    assert lib.kge_eval_relation_topk_scratch_bytes(d, 10, 0, 40, 256) == 8 * 10 * 256
    assert lib.kge_eval_relation_topk_scratch_bytes(d, 10, 20, 20, 5) == 0
    assert lib.kge_eval_relation_topk_scratch_bytes(d, 0, 0, 40, 5) == 0
    assert lib.kge_eval_relation_topk(d, 16, 10, None, None, None, 0, 40, 5, 16, 16, 8 * 10 * 40 - 1, None,
                                      None) == _lib.ERR_INVALID
    assert b"scratch" in lib.kge_last_error()
    assert lib.kge_eval_relation_topk(d, None, 10, None, None, None, 0, 40, 5, 16, 16, 1 << 20, None,
                                      None) == _lib.ERR_INVALID
    assert b"null pointer" in lib.kge_last_error()
    assert lib.kge_eval_relation_topk(d, 16, 10, None, None, None, 0, 40, 5, None, 16, 1 << 20, None,
                                      None) == _lib.ERR_INVALID
    assert b"null pointer" in lib.kge_last_error()
    for args in ((None, 16, 16, 16), (16, None, 16, 16), (16, 16, None, 16), (16, 16, 16, None)):
        queries, pos, bits, counts = args
        assert lib.kge_eval_relation_count_ranks(d, queries, 10, None, None, pos, bits, 0, 40, counts, None,
                                                 None) == _lib.ERR_INVALID
        assert b"null pointer" in lib.kge_last_error()
    for name, entity_dim in (("RotatE", 16), ("pRotatE", 8)):
        desc.model, desc.entity_dim, desc.modulus = _lib.MODEL_IDS[name], entity_dim, 16
        assert lib.kge_eval_relation_count_ranks(d, 16, 10, None, 16, 16, 16, 0, 40, 16, None, None) == _lib.ERR_INVALID
        assert b"kge_eval_relation_table" in lib.kge_last_error()
    assert lib.kge_eval_relation_count_ranks(d, 16, 10, 16, None, 16, 16, 0, 40, 16, None, None) == _lib.ERR_INVALID
    assert b"kge_eval_phase_table" in lib.kge_last_error()
    assert lib.kge_eval_relation_table(d, None, None) == _lib.ERR_INVALID
    desc.model, desc.entity_dim, desc.modulus = _lib.TRANSE, 8, None
    assert lib.kge_eval_relation_table(d, None, None) == 0            # TransE uses the relation table as it is
    assert lib.kge_eval_relation_filter_bits(16, 16, 16, 5, 16, 10, 100, 40, None, None) == _lib.ERR_INVALID
    assert lib.kge_eval_relation_filter_bits(None, 16, 16, 5, 16, 10, 100, 40, 16, None) == _lib.ERR_INVALID
    assert b"null filter index" in lib.kge_last_error()
    assert lib.kge_eval_relation_filter_bits(16, 16, 16, 5, 16, 10, 100, 0, 16, None) == _lib.ERR_INVALID
    assert lib.kge_eval_relation_filter_bits(16, 16, 16, 5, None, 0, 100, 40, 16, None) == 0
