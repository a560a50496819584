"""KGEModel.predict_topk and the kge_eval_topk / kge_eval_topk_merge C ABI (top-k link prediction).

The oracle is the C oracle with an empty filter (raw exact scores, bit-identical to the device's canonical scores); the
exclusion is applied in numpy and the order is score descending, then id ascending, NaN last.  The ABI argument checks
at the end need no GPU.
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
MODES = ("head-batch", "tail-batch")


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


def raw_scores(model, st, queries, mode, gamma, d, nentity, nrel):
    from knowledgegraphembedding_b200 import FilterIndex
    off, ent = FilterIndex([], nentity, nrel).csr(queries, mode)
    return C.eval_scores(model, st, queries, mode, gamma, O.embedding_range(gamma, d), off, ent)


def excluded(exclude, queries, mode, nentity, nrel):
    from knowledgegraphembedding_b200 import FilterIndex
    mask = np.zeros((len(queries), nentity), dtype=bool)
    if exclude:
        off, ent = FilterIndex(exclude, nentity, nrel).csr(queries, mode)
        mask[np.repeat(np.arange(len(queries)), np.diff(off)), ent] = True
    return mask


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


def random_triples(nentity, nrel, n, seed, tail_range=200):
    rng = np.random.RandomState(seed)
    return sorted({(int(rng.randint(nentity)), int(rng.randint(nrel)), int(rng.randint(min(tail_range, nentity))))
                   for _ in range(n)})


# ------------------------------------------------------------------------------------------------ bit-exact vs oracle
@gpu
@pytest.mark.parametrize("model,nentity,nrel,d,gamma", FULL)
def test_topk_bit_exact_at_baseline_shapes(model, nentity, nrel, d, gamma):
    m, st = make(model, nentity, nrel, d, gamma)
    m = load(m, st)
    all_true = random_triples(nentity, nrel, 30000, seed=2)
    rng = np.random.RandomState(3)
    queries = [all_true[i] for i in rng.choice(len(all_true), 24, replace=False)]
    for mode in MODES:
        raw = raw_scores(model, st, queries, mode, gamma, d, nentity, nrel)
        for exclude in (None, all_true):
            mask = excluded(exclude, queries, mode, nentity, nrel)
            for k in (1, 10, 256):
                ids, scores = m.predict_topk(queries, mode, k=k, exclude_triples=exclude)
                assert ids.shape == (24, k) and ids.dtype == torch.int64 and scores.dtype == torch.float32
                assert ids.device == m.entity_embedding.device
                assert_same(ids, scores, *oracle_topk(raw, mask, k), what=(model, mode, k, exclude is not None))


@gpu
@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("d", [10, 12])
def test_topk_small_ragged_shapes(model, d):
    """d = 10 takes the unaligned staging path; nentity and Q are not multiples of 64; numpy input."""
    nentity, nrel, gamma = 1000, 7, 6.0
    m, st = make(model, nentity, nrel, d, gamma, seed=1, scale=1.0)
    m = load(m, st)
    all_true = random_triples(nentity, nrel, 3000, seed=4, tail_range=nentity)
    queries = np.asarray(all_true[:100], dtype=np.int64)
    for mode in MODES:
        raw = raw_scores(model, st, queries, mode, gamma, d, nentity, nrel)
        for k, exclude in ((7, all_true), (100, None)):
            ids, scores = m.predict_topk(queries, mode, k=k, exclude_triples=exclude)
            assert_same(ids, scores, *oracle_topk(raw, excluded(exclude, queries, mode, nentity, nrel), k),
                        what=(model, d, mode, k))


@gpu
def test_topk_chunking_empty_queries_and_padding():
    model, nentity, nrel, d, gamma = "TransE", 301, 5, 12, 6.0
    m, st = make(model, nentity, nrel, d, gamma, seed=2, scale=1.0)
    m = load(m, st)
    rng = np.random.RandomState(6)
    queries = np.stack([rng.randint(nentity, size=5000), rng.randint(nrel, size=5000), rng.randint(nentity, size=5000)], 1)
    raw = raw_scores(model, st, queries, "tail-batch", gamma, d, nentity, nrel)
    ids, scores = m.predict_topk(torch.from_numpy(queries), "tail-batch", k=5)        # Q > 4096: two chunks
    assert_same(ids, scores, *oracle_topk(raw, np.zeros_like(raw, dtype=bool), 5))
    ids, scores = m.predict_topk([], "head-batch", k=3)
    assert tuple(ids.shape) == (0, 3) and tuple(scores.shape) == (0, 3)
    # k larger than the candidates left: every entity but 40 excluded for the (h, r) of the first query
    h, r = int(queries[0, 0]), int(queries[0, 1])
    exclude = [(h, r, t) for t in range(40, nentity)]
    q = [(h, r, 0), (h, (r + 1) % nrel, 0)]
    ids, scores = m.predict_topk(q, "tail-batch", k=64, exclude_triples=exclude)
    raw = raw_scores(model, st, q, "tail-batch", gamma, d, nentity, nrel)
    want_ids, want_scores = oracle_topk(raw, excluded(exclude, q, "tail-batch", nentity, nrel), 64)
    assert_same(ids, scores, want_ids, want_scores)
    assert (ids[0, 40:] == -1).all() and torch.isneginf(scores[0, 40:]).all()
    assert sorted(ids[0, :40].tolist()) == list(range(40))
    assert (ids[1] >= 0).all()


@gpu
def test_topk_ties_ascending_ids_and_nan_last():
    model, nentity, nrel, d, gamma = "TransE", 200, 3, 16, 6.0
    m, st = make(model, nentity, nrel, d, gamma, seed=3, scale=1.0)
    E = st["entity_embedding"]
    E[100:164] = E[100]                                 # 64 identical rows: 64 tied scores
    E[7] = np.nan                                       # a NaN row: ranked after every number
    m = load(m, st)
    queries = [(1, 0, 2), (150, 2, 3), (30, 1, 100)]
    raw = raw_scores(model, st, queries, "tail-batch", gamma, d, nentity, nrel)
    ids, scores = m.predict_topk(queries, "tail-batch", k=nentity)
    assert_same(ids, scores, *oracle_topk(raw, np.zeros_like(raw, dtype=bool), nentity))
    for row in ids.cpu().numpy():
        assert row[-1] == 7
        pos = [int(np.nonzero(row == j)[0][0]) for j in range(100, 164)]
        assert pos == list(range(pos[0], pos[0] + 64))   # tied ids adjacent and ascending
    assert torch.isnan(scores[:, -1]).all() and not torch.isnan(scores[:, :-1]).any()


# ------------------------------------------------------------------------------------------------ vs the filtered ranks
@gpu
@pytest.mark.parametrize("model", MODELS)
def test_topk_agrees_with_filtered_ranks(model):
    """exclude = all true triples minus the test triples (whose open-slot keys are distinct), so the candidates of a query
    are exactly those its filtered rank counts, plus its answer: the answer sits at position rank - 1 when rank <= k."""
    nentity, nrel, gamma = 14951, 1345, 24.0
    d = {"ComplEx": 500, "DistMult": 2000}.get(model, 1000)
    m, st = make(model, nentity, nrel, d, gamma, seed=5)
    m = load(m, st)
    all_true = random_triples(nentity, nrel, 30000, seed=7)
    for mode in MODES:
        seen, test = set(), []
        for tr in all_true[::97]:
            key = (tr[1], tr[2]) if mode == "head-batch" else (tr[0], tr[1])
            if key not in seen:
                seen.add(key)
                test.append(tr)
        test_set = set(test)
        exclude = [tr for tr in all_true if tr not in test_set]
        ranks = m.filtered_ranks(test, all_true, mode)
        col = 0 if mode == "head-batch" else 2
        hits = 0
        for k in (10, 256):
            ids = m.predict_topk(test, mode, k=k, exclude_triples=exclude)[0].cpu().numpy()
            for q, (tr, r) in enumerate(zip(test, ranks)):
                if r <= k:
                    assert ids[q, r - 1] == tr[col], (mode, k, q, r)
                    hits += 1
                else:
                    assert tr[col] not in ids[q], (mode, k, q, r)
        assert hits > 0


# ------------------------------------------------------------------------------------------------ ABI level
@gpu
def test_topk_entity_slices_merge_to_full_range():
    from knowledgegraphembedding_b200 import _lib, shard_bounds
    from knowledgegraphembedding_b200.model import _ptr, _stream
    model, nentity, nrel, d, gamma = "RotatE", 5003, 17, 64, 12.0
    m, st = make(model, nentity, nrel, d, gamma, seed=4, scale=1.0)
    m = load(m, st)
    dev = m.entity_embedding.device
    lib = _lib.load()
    rng = np.random.RandomState(8)
    test = np.stack([rng.randint(nentity, size=100), rng.randint(nrel, size=100), rng.randint(nentity, size=100)], 1)
    q = torch.from_numpy(test).to(dev)
    Q, k = len(test), 50
    desc, stt = m._descriptor(), _stream(dev)
    for mode in MODES:
        mid = _lib.MODE_IDS[mode]
        qvec = torch.empty(Q * m.entity_dim, device=dev)
        _lib.call("kge_eval_query_vectors", ctypes.byref(desc), mid, _ptr(q), Q, _ptr(qvec), None, stt)

        def select(b, e):
            sb = int(lib.kge_eval_topk_scratch_bytes(ctypes.byref(desc), Q, b, e, k))
            scratch = torch.empty(max(sb, 1), dtype=torch.uint8, device=dev)
            keys = torch.empty((Q, k), dtype=torch.int64, device=dev)
            _lib.call("kge_eval_topk", ctypes.byref(desc), mid, _ptr(qvec), Q, None, None, b, e, k, _ptr(keys),
                      _ptr(scratch), sb, stt)
            return keys

        full = select(0, nentity)
        parts = torch.stack([select(*shard_bounds(nentity, r, 8)) for r in range(8)], dim=1).contiguous()
        merged = torch.empty_like(full)
        ids = torch.empty((Q, k), dtype=torch.int64, device=dev)
        scores = torch.empty((Q, k), dtype=torch.float32, device=dev)
        _lib.call("kge_eval_topk_merge", _ptr(parts), Q, 8, k, _ptr(merged), _ptr(ids), _ptr(scores), stt)
        assert torch.equal(merged, full), mode
        raw = raw_scores(model, st, test, mode, gamma, d, nentity, nrel)
        assert_same(ids, scores, *oracle_topk(raw, np.zeros_like(raw, dtype=bool), k), what=mode)


def _run_worker(n, **env):
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "topk_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, **env))
    if not (res.returncode == 0 and res.stdout.strip().endswith("ok")):
        sys.stderr.write(res.stdout[-3000:] + "\n" + res.stderr[-8000:])
    assert res.returncode == 0 and res.stdout.strip().endswith("ok"), "top-k worker failed (output on stderr)"


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
def test_topk_multi_rank_two_ranks_sharing_one_gpu():
    _run_worker(2, KGE_TEST_SAME_GPU="1")


@gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_topk_multi_rank_one_gpu_per_rank():
    _run_worker(min(torch.cuda.device_count(), 8))


# ------------------------------------------------------------------------------------------------ resources, API
@gpu
def test_topk_never_allocates_the_score_matrix():
    model, nentity, nrel, d, gamma = "RotatE", 14951, 1345, 1000, 24.0
    m, st = make(model, nentity, nrel, d, gamma, seed=6)
    m = load(m, st)
    all_true = random_triples(nentity, nrel, 30000, seed=9)
    rng = np.random.RandomState(1)
    Q, k = 4096, 100
    queries = np.stack([rng.randint(nentity, size=Q), rng.randint(nrel, size=Q), rng.randint(nentity, size=Q)], 1)
    m.predict_topk(queries, "tail-batch", k=k, exclude_triples=all_true)      # builds the filter index (80 MB)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    m.predict_topk(queries, "tail-batch", k=k, exclude_triples=all_true)
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated() - base < Q * nentity * 4 // 2


@gpu
def test_topk_leaves_filtered_ranks_unchanged():
    model, nentity, nrel, d, gamma = "RotatE", 3001, 11, 64, 12.0
    m, st = make(model, nentity, nrel, d, gamma, seed=7, scale=1.0)
    m = load(m, st)
    all_true = random_triples(nentity, nrel, 5000, seed=10, tail_range=nentity)
    test = all_true[:300]
    for mode in MODES:
        before = m.filtered_ranks(test, all_true, mode)
        m.predict_topk(test, mode, k=256, exclude_triples=all_true)
        np.testing.assert_array_equal(m.filtered_ranks(test, all_true, mode), before)


@gpu
def test_topk_errors():
    m, st = make("TransE", 100, 3, 8, 6.0, scale=1.0)
    m = load(m, st)
    q = [(1, 0, 2)]
    for k in (0, 257, 2.5):
        with pytest.raises(ValueError):
            m.predict_topk(q, "tail-batch", k=k)
    with pytest.raises(ValueError):
        m.predict_topk(q, "single", k=3)
    with pytest.raises(IndexError):
        m.predict_topk([(1, 0, 2), (100, 0, 2)], "tail-batch", k=3)      # fixed side out of range
    with pytest.raises(IndexError):
        m.predict_topk([(1, 3, 2)], "head-batch", k=3)                     # relation out of range
    ids, _ = m.predict_topk([(1, 0, 10**9)], "tail-batch", k=3)           # the predicted slot is ignored
    assert ids.shape == (1, 3)


def test_topk_abi_argument_errors_without_a_gpu():
    from knowledgegraphembedding_b200 import _lib
    lib = _lib.load()
    desc = _lib.KgeModelStruct(model=_lib.TRANSE, device=0, nentity=100, nrelation=3, hidden_dim=8, entity_dim=8,
                               relation_dim=8, gamma=6.0, embedding_range=1.0, entity=16, relation=16, modulus=None)
    d = ctypes.byref(desc)
    for k in (0, 257):
        assert lib.kge_eval_topk_scratch_bytes(d, 10, 0, 100, k) == _lib.ERR_INVALID
        assert b"outside [1, 256]" in lib.kge_last_error()
        assert lib.kge_eval_topk(d, _lib.TAIL_BATCH, 16, 10, None, None, 0, 100, k, 16, 16, 1 << 20, None) == _lib.ERR_INVALID
        assert lib.kge_eval_topk_merge(16, 10, 2, k, 32, None, None, None) == _lib.ERR_INVALID
    assert lib.kge_eval_topk_scratch_bytes(d, 10, 50, 101, 5) == _lib.ERR_INVALID
    assert b"entity slice" in lib.kge_last_error()
    assert lib.kge_eval_topk(d, _lib.TAIL_BATCH, 16, 10, None, None, 60, 50, 5, 16, 16, 1 << 20, None) == _lib.ERR_INVALID
    assert lib.kge_eval_topk(d, _lib.TAIL_BATCH, None, 10, None, None, 0, 100, 5, 16, 16, 1 << 20, None) == _lib.ERR_INVALID
    assert b"null pointer" in lib.kge_last_error()
    assert lib.kge_eval_topk(d, _lib.TAIL_BATCH, 16, 10, None, None, 0, 100, 5, None, 16, 1 << 20, None) == _lib.ERR_INVALID
    assert lib.kge_eval_topk(d, _lib.SINGLE, 16, 10, None, None, 0, 100, 5, 16, 16, 1 << 20, None) == _lib.ERR_INVALID
    assert b"negative batch mode 0" in lib.kge_last_error()
    assert lib.kge_eval_topk(d, _lib.TAIL_BATCH, 16, 10, None, None, 0, 100, 5, 16, 16, 0, None) == _lib.ERR_INVALID
    assert b"scratch" in lib.kge_last_error()
    assert lib.kge_eval_topk_merge(None, 10, 2, 5, 32, None, None, None) == _lib.ERR_INVALID
    assert lib.kge_eval_topk_merge(16, 10, 2, 5, None, None, None, None) == _lib.ERR_INVALID
    assert lib.kge_eval_topk_merge(16, 10, 0, 5, 32, None, None, None) == _lib.ERR_INVALID
    assert lib.kge_eval_topk_scratch_bytes(d, 0, 0, 100, 5) == 0
