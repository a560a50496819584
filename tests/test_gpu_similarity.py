"""KGEModel.nearest_neighbors and the kge_similarity_* C ABI (similarity search over the embedding tables).

Scores are compared with == on the raw bits against ko_similarity (tests/similarity_oracle.c), ids against a stable
descending sort of its [Q, rows] matrix (score descending, then id ascending, NaN last, -0.0 == +0.0) with the self
column removed when exclude_self is set.  The ABI argument checks and the input checks at the end need no GPU.
"""
import ctypes
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

import similarity_oracle as S
from conftest import ROOT
from oracle import kge_oracle as O

gpu = pytest.mark.gpu
METRICS = ("dot", "cosine", "l2", "l1")
FLAGS = {"TransE": (False, False), "DistMult": (False, False), "ComplEx": (True, True),
         "RotatE": (True, False), "pRotatE": (False, False)}


def make(model, nentity, nrel, d, gamma=12.0, seed=0, scale=3.0):
    """A KGEModel on the GPU with the U(-rho, rho) tables of the oracle (entities scaled by `scale`), and the tables."""
    from knowledgegraphembedding_b200 import KGEModel
    de, dr = FLAGS[model]
    st = O.init_tables(model, nentity, nrel, d, gamma, de, dr, seed=seed)
    st["entity_embedding"] = (st["entity_embedding"] * scale).astype(np.float32)
    m = KGEModel(model, nentity, nrel, d, gamma, double_entity_embedding=de, double_relation_embedding=dr)
    return set_tables(m.cuda(), st["entity_embedding"], st["relation_embedding"])


def set_tables(m, E, R):
    with torch.no_grad():
        m.entity_embedding.copy_(torch.from_numpy(np.ascontiguousarray(E, dtype=np.float32)))
        m.relation_embedding.copy_(torch.from_numpy(np.ascontiguousarray(R, dtype=np.float32)))
    return m, m.entity_embedding.detach().cpu().numpy(), m.relation_embedding.detach().cpu().numpy()


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


def check_ids(m, X, table, ids, metric, k, exclude_self=True, what=""):
    """nearest_neighbors of the id queries `ids` against the oracle."""
    got = m.nearest_neighbors(ids, table=table, k=k, metric=metric, exclude_self=exclude_self)
    assert got[0].shape == (len(ids), k) and got[0].dtype == torch.int64 and got[1].dtype == torch.float32
    assert got[0].device == m.entity_embedding.device and got[1].device == m.entity_embedding.device
    raw = S.similarity(X, X[np.asarray(ids)], metric)
    want = S.topk(raw, k, np.asarray(ids) if exclude_self else None)
    assert_same(*got, *want, what=(what, table, metric, k, exclude_self))
    return got


# ------------------------------------------------------------------------------------------------ bit-exact vs oracle
FULL = [("TransE", 14541, 237, 1000, "entity"),          # FB15k-237 TransE
        ("ComplEx", 40943, 11, 500, "entity"),           # wn18rr ComplEx -de -dr: width 1000
        ("RotatE", 14951, 1345, 1000, "entity"),         # FB15k RotatE -de: width 2000
        ("RotatE", 14951, 1345, 1000, "relation")]       # its relation table: 1345 x 1000 phases


@gpu
@pytest.mark.parametrize("model,nentity,nrel,d,table", FULL)
def test_similarity_bit_exact_at_full_shapes(model, nentity, nrel, d, table):
    m, E, R = make(model, nentity, nrel, d)
    X = E if table == "entity" else R
    ids = np.random.RandomState(1).choice(X.shape[0], 64, replace=False)
    for metric in METRICS:
        raw = S.similarity(X, X[ids], metric)
        for k in (1, 10, 256):
            for exclude_self in ((True, False) if k == 10 else (True,)):
                got = m.nearest_neighbors(torch.from_numpy(ids), table=table, k=k, metric=metric,
                                          exclude_self=exclude_self)
                assert_same(*got, *S.topk(raw, k, ids if exclude_self else None), what=(model, table, metric, k))


# ------------------------------------------------------------------------------------------------ ties and specials
@gpu
def test_similarity_ties_zero_nan_and_inf_rows():
    m, E, R = make("TransE", 250, 3, 16, seed=2, scale=1.0)
    E[100:140] = E[100]                                 # 40 identical rows: equal scores, ids ascending
    E[7] = 0.0                                          # zero row: cosine 0/0 = NaN, ranked last
    E[11, 3] = np.nan                                   # a NaN row
    E[13, 0], E[14, 5] = np.inf, -np.inf                # infinite rows
    m, E, R = set_tables(m, E, R)
    ids = [100, 120, 7, 11, 13, 14, 0, 5]
    for metric in METRICS:
        for exclude_self in (True, False):
            got_ids, got_scores = check_ids(m, E, "entity", ids, metric, 250, exclude_self)
            row = got_ids[0].cpu().numpy()                    # query 100: its 39 duplicates are adjacent and ascending
            dup = [int(np.nonzero(row == j)[0][0]) for j in range(101 if exclude_self else 100, 140)]
            assert dup == list(range(dup[0], dup[0] + len(dup))), metric
            if metric == "cosine":
                assert torch.isnan(got_scores[2, got_ids[2] >= 0]).all()     # the zero row's own query: all NaN
                n = int((got_ids[0] >= 0).sum())                # 0/0, NaN and inf/inf rows: NaN, after every number
                assert set(got_ids[0, n - 4:n].tolist()) == {7, 11, 13, 14} and torch.isnan(got_scores[0, n - 4:n]).all()
    # l2 self-distance: -0.0, equal to +0.0 and first when the query's own row stays
    got_ids, got_scores = m.nearest_neighbors([5, 0], k=3, metric="l2", exclude_self=False)
    assert got_ids[:, 0].tolist() == [5, 0] and (got_scores[:, 0] == 0).all()


@gpu
def test_similarity_fewer_rows_than_k_and_one_row():
    m, E, R = make("DistMult", 50, 5, 12, seed=3, scale=1.0)
    for metric in METRICS:
        got_ids, got_scores = check_ids(m, R, "relation", [0, 4], metric, 10, True)
        assert (got_ids[:, 4:] == -1).all() and torch.isneginf(got_scores[:, 4:]).all()
        got_ids, _ = check_ids(m, R, "relation", [0, 4], metric, 10, False)
        assert (got_ids[:, :5] >= 0).all() and (got_ids[:, 5:] == -1).all()
    m1, E1, R1 = make("TransE", 40, 1, 8, seed=4, scale=1.0)          # a one-row relation table
    for metric in METRICS:
        got_ids, got_scores = m1.nearest_neighbors([0], table="relation", k=3, metric=metric)
        assert (got_ids == -1).all() and torch.isneginf(got_scores).all()
        check_ids(m1, R1, "relation", [0], metric, 3, False)


# ------------------------------------------------------------------------------------------------ widths, vector queries
@gpu
@pytest.mark.parametrize("width", [5, 8, 23, 37, 50, 64])
def test_similarity_widths_and_misaligned_vector_queries(width):
    """Widths that are not multiples of 4 take the staging path without cp.async; so does a query view whose pointer is
    not 16-byte aligned, at any width."""
    m, E, R = make("TransE", 1000, 7, width, seed=width, scale=1.0)
    rng = np.random.RandomState(width)
    ids = rng.choice(1000, 37, replace=False)
    V = rng.standard_normal((19, width)).astype(np.float32)
    buf = torch.zeros(19 * width + 1, dtype=torch.float32, device="cuda")
    view = buf[1:].view(19, width)                       # contiguous, 4 bytes past an aligned address
    view.copy_(torch.from_numpy(V))
    assert view.data_ptr() % 16 != 0
    for metric in METRICS:
        check_ids(m, E, "entity", ids, metric, 20, what=width)
        check_ids(m, R, "relation", [0, 6], metric, 5, what=width)
        for items in (view, V):
            got = m.nearest_neighbors(items, k=50, metric=metric)
            assert_same(*got, *S.topk(S.similarity(E, V, metric), 50), what=(width, metric, type(items)))


@gpu
def test_similarity_vector_queries_equal_id_queries():
    m, E, R = make("RotatE", 3001, 11, 40, seed=5)
    ids = np.arange(0, 3001, 47)
    vec = m.entity_embedding.detach()[torch.from_numpy(ids).cuda()]
    for metric in METRICS:
        v_ids, v_scores = m.nearest_neighbors(vec, k=31, metric=metric)
        i_ids, i_scores = m.nearest_neighbors(ids, k=30, metric=metric, exclude_self=False)
        assert torch.equal(v_ids[:, :30], i_ids), metric
        assert torch.equal(v_scores[:, :30].view(torch.int32), i_scores.view(torch.int32)), metric
        s_ids, s_scores = m.nearest_neighbors(ids, k=30, metric=metric, exclude_self=True)
        for q, own in enumerate(ids):
            keep = (v_ids[q] != int(own)).nonzero().flatten()[:30]
            assert torch.equal(s_ids[q], v_ids[q, keep]), (metric, q)
            assert torch.equal(s_scores[q].view(torch.int32), v_scores[q, keep].view(torch.int32)), (metric, q)


# ------------------------------------------------------------------------------------------------ chunks, slices, ranks
@gpu
def test_similarity_chunking():
    m, E, R = make("DistMult", 700, 5, 48, seed=6, scale=1.0)
    ids = np.random.RandomState(7).randint(700, size=5000)           # two chunks of the call
    for metric in ("cosine", "l1"):
        whole = m.nearest_neighbors(ids, k=12, metric=metric)
        parts = [m.nearest_neighbors(ids[:4096], k=12, metric=metric), m.nearest_neighbors(ids[4096:], k=12, metric=metric)]
        assert torch.equal(whole[0], torch.cat([p[0] for p in parts]))
        assert torch.equal(whole[1].view(torch.int32), torch.cat([p[1] for p in parts]).view(torch.int32))
        assert_same(*whole, *S.topk(S.similarity(E, E[ids], metric), 12, ids), what=metric)
    ids, scores = m.nearest_neighbors([], k=3)
    assert tuple(ids.shape) == (0, 3) and tuple(scores.shape) == (0, 3)


@gpu
def test_similarity_row_slices_merge_to_the_whole_table():
    from knowledgegraphembedding_b200 import _lib
    from knowledgegraphembedding_b200.model import _ptr, _stream
    m, E, R = make("ComplEx", 3000, 7, 30, seed=8)
    dev = m.entity_embedding.device
    lib = _lib.load()
    desc, st = m._descriptor(), _stream(dev)
    ids = torch.from_numpy(np.random.RandomState(9).randint(3000, size=100)).to(dev)
    Q, k, rows, width = 100, 40, 3000, m.entity_dim
    ent = _lib.TABLE_ENTITY
    qvec = torch.empty((Q, width), device=dev)
    qnorm, xnorm = torch.empty(Q, device=dev), torch.empty(rows, device=dev)
    _lib.call("kge_similarity_rows", ctypes.byref(desc), ent, _ptr(ids), Q, _ptr(qvec), None, st)
    _lib.call("kge_similarity_norms", ctypes.byref(desc), ent, _ptr(qvec), Q, _ptr(qnorm), st)
    _lib.call("kge_similarity_norms", ctypes.byref(desc), ent, None, rows, _ptr(xnorm), st)
    for metric in METRICS:
        sim = _lib.SIM_IDS[metric]

        def select(b, e):
            sb = int(lib.kge_similarity_topk_scratch_bytes(ctypes.byref(desc), ent, Q, b, e, k))
            scratch = torch.empty(max(sb, 1), dtype=torch.uint8, device=dev)
            keys = torch.empty((Q, k), dtype=torch.int64, device=dev)
            _lib.call("kge_similarity_topk", ctypes.byref(desc), ent, sim, _ptr(qvec), _ptr(qnorm), _ptr(xnorm),
                      _ptr(ids), Q, b, e, k, _ptr(keys), _ptr(scratch), sb, st)
            return keys

        full = select(0, rows)
        parts = torch.stack([select(0, 1024), select(1024, rows)], dim=1).contiguous()
        merged = torch.empty_like(full)
        out_ids = torch.empty((Q, k), dtype=torch.int64, device=dev)
        out_scores = torch.empty((Q, k), dtype=torch.float32, device=dev)
        _lib.call("kge_eval_topk_merge", _ptr(parts), Q, 2, k, _ptr(merged), _ptr(out_ids), _ptr(out_scores), st)
        assert torch.equal(merged, full), metric
        host_ids = ids.cpu().numpy()
        assert_same(out_ids, out_scores, *S.topk(S.similarity(E, E[host_ids], metric), k, host_ids), what=metric)


def _run_worker(n, **env):
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "similarity_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, **env))
    if not (res.returncode == 0 and res.stdout.strip().endswith("ok")):
        sys.stderr.write(res.stdout[-3000:] + "\n" + res.stderr[-8000:])
    assert res.returncode == 0 and res.stdout.strip().endswith("ok"), "similarity worker failed (output on stderr)"


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
def test_similarity_multi_rank_two_ranks_sharing_one_gpu():
    _run_worker(2, KGE_TEST_SAME_GPU="1")


@gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_similarity_multi_rank_one_gpu_per_rank():
    _run_worker(min(torch.cuda.device_count(), 8))


# ------------------------------------------------------------------------------------------------ errors
@gpu
def test_similarity_bad_ids_raise_once():
    m, E, R = make("TransE", 100, 3, 8, seed=10, scale=1.0)
    for bad in ([1, 100], [-1], [3, 2, 1000]):
        with pytest.raises(IndexError):
            m.nearest_neighbors(bad, k=3)
        check_ids(m, E, "entity", [1, 2, 99], "cosine", 3)            # the flag was cleared
    with pytest.raises(IndexError):
        m.nearest_neighbors([3], table="relation", k=2)
    check_ids(m, R, "relation", [0, 2], "l2", 2)


@gpu
def test_similarity_leaves_predict_topk_unchanged():
    m, E, R = make("RotatE", 2001, 11, 32, seed=11)
    queries = [(i, i % 11, 0) for i in range(0, 2001, 37)]
    before = m.predict_topk(queries, "tail-batch", k=50)
    m.nearest_neighbors(np.arange(0, 2001, 5), k=200, metric="l2")
    after = m.predict_topk(queries, "tail-batch", k=50)
    assert torch.equal(before[0], after[0]) and torch.equal(before[1].view(torch.int32), after[1].view(torch.int32))


def test_similarity_abi_argument_errors_without_a_gpu():
    from knowledgegraphembedding_b200 import _lib
    lib = _lib.load()
    desc = _lib.KgeModelStruct(model=_lib.TRANSE, device=0, nentity=100, nrelation=3, hidden_dim=8, entity_dim=8,
                               relation_dim=8, gamma=6.0, embedding_range=1.0, entity=16, relation=16, modulus=None)
    d = ctypes.byref(desc)
    E, R = _lib.TABLE_ENTITY, _lib.TABLE_RELATION
    topk = lib.kge_similarity_topk
    for k in (0, 257):
        assert lib.kge_similarity_topk_scratch_bytes(d, E, 10, 0, 100, k) == _lib.ERR_INVALID
        assert b"outside [1, 256]" in lib.kge_last_error()
        assert topk(d, E, 0, 16, None, None, None, 10, 0, 100, k, 16, 16, 1 << 20, None) == _lib.ERR_INVALID
    assert lib.kge_similarity_topk_scratch_bytes(d, 2, 10, 0, 100, 5) == _lib.ERR_INVALID
    assert b"table 2" in lib.kge_last_error()
    assert lib.kge_similarity_topk_scratch_bytes(d, R, 10, 0, 4, 5) == _lib.ERR_INVALID    # 3 relation rows
    assert b"row slice [0,4) outside [0,3)" in lib.kge_last_error()
    assert lib.kge_similarity_topk_scratch_bytes(d, E, 65535 * 64 + 1, 0, 100, 5) == _lib.ERR_INVALID
    assert b"queries per call" in lib.kge_last_error()
    assert lib.kge_similarity_topk_scratch_bytes(d, E, 0, 0, 100, 5) == 0
    assert lib.kge_similarity_topk_scratch_bytes(d, E, 10, 50, 50, 5) == 0
    assert topk(d, E, 4, 16, 16, 16, None, 10, 0, 100, 5, 16, 16, 1 << 20, None) == _lib.ERR_INVALID
    assert b"metric 4" in lib.kge_last_error()
    assert topk(d, E, -1, 16, 16, 16, None, 10, 0, 100, 5, 16, 16, 1 << 20, None) == _lib.ERR_INVALID
    assert topk(d, E, 0, None, None, None, None, 10, 0, 100, 5, 16, 16, 1 << 20, None) == _lib.ERR_INVALID
    assert b"null pointer" in lib.kge_last_error()
    assert topk(d, E, 0, 16, None, None, None, 10, 0, 100, 5, None, 16, 1 << 20, None) == _lib.ERR_INVALID
    assert topk(d, E, 1, 16, None, 16, None, 10, 0, 100, 5, 16, 16, 1 << 20, None) == _lib.ERR_INVALID
    assert b"cosine needs" in lib.kge_last_error()
    assert topk(d, E, 1, 16, 16, None, None, 10, 0, 100, 5, 16, 16, 1 << 20, None) == _lib.ERR_INVALID
    assert topk(d, E, 0, 16, None, None, None, 10, 60, 50, 5, 16, 16, 1 << 20, None) == _lib.ERR_INVALID
    assert topk(d, E, 0, 16, None, None, None, 10, 0, 100, 5, 16, 16, 0, None) == _lib.ERR_INVALID
    assert b"scratch" in lib.kge_last_error()
    assert topk(d, 7, 0, 16, None, None, None, 10, 0, 100, 5, 16, 16, 1 << 20, None) == _lib.ERR_INVALID
    assert lib.kge_similarity_rows(d, E, None, 10, 16, None, None) == _lib.ERR_INVALID
    assert b"null pointer" in lib.kge_last_error()
    assert lib.kge_similarity_rows(d, E, 16, 10, None, None, None) == _lib.ERR_INVALID
    assert lib.kge_similarity_rows(d, 5, 16, 10, 16, None, None) == _lib.ERR_INVALID
    assert lib.kge_similarity_norms(d, E, None, 99, 16, None) == _lib.ERR_INVALID
    assert b"n = 100 rows" in lib.kge_last_error()
    assert lib.kge_similarity_norms(d, R, 16, 10, None, None) == _lib.ERR_INVALID
    assert lib.kge_similarity_norms(d, E, 16, -1, 16, None) == _lib.ERR_INVALID
    desc.nentity = 0
    assert lib.kge_similarity_norms(d, E, None, 0, 16, None) == _lib.ERR_INVALID           # check_model: empty model
    assert lib.kge_similarity_rows(None, E, 16, 10, 16, None, None) == _lib.ERR_INVALID


def test_similarity_input_checks_without_a_gpu():
    from knowledgegraphembedding_b200 import KGEModel
    m = KGEModel("RotatE", 30, 4, 6, 12.0, double_entity_embedding=True)           # entity width 12, relation 6
    bad = [dict(items=[1], metric="cos"), dict(items=[1], table="entities"), dict(items=[1], k=0),
           dict(items=[1], k=257), dict(items=[1], k=2.5), dict(items=[1], k=True),
           dict(items=np.zeros((2, 6), dtype=np.float32)),                           # entity width is 12
           dict(items=np.zeros((2, 12), dtype=np.float32), table="relation"),
           dict(items=np.zeros((2, 12), dtype=np.int64)), dict(items=torch.zeros(2, 12, dtype=torch.int32)),
           dict(items=np.zeros(3, dtype=np.float32)), dict(items=torch.zeros(3)), dict(items=[0.5, 1.0]),
           dict(items=np.zeros((2, 3, 12), dtype=np.float32)), dict(items=np.array([True, False]))]
    for kw in bad:
        with pytest.raises(ValueError):
            m.nearest_neighbors(**kw)
    with pytest.raises(RuntimeError, match="CUDA device"):                           # valid arguments: no CPU fallback
        m.nearest_neighbors([1, 2], k=3)
