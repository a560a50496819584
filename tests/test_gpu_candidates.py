"""Candidate-list ranking (KGEModel.candidate_rank_statistics, kge_eval_candidate_rank_stats): the six counters of
rank_statistics over each query's own list of entities, and the canonical scores of the listed entries.  Checked
against numpy counts over the C oracle's raw scores at the listed ids (lists with duplicates, the positive itself and
-1 padding in the middle and at the end), against rank_statistics and filtered_ranks when every list is a permutation
of all entities, on the tie tables of test_gpu_rank_stats, at unaligned widths and d = 100 over 100 k entities, over
query chunks, the host-sorted filter index, column slices and two ranks; without a GPU, the argument checks of the ABI
entry and the input checks of the method."""
import ctypes
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import kge_oracle as O
from test_gpu_rank_stats import FLAGS, filter_mask, raw_scores, tie_case

gpu = pytest.mark.gpu
MODES = ("head-batch", "tail-batch")


def positives(test, mode):
    return np.array([t[0] if mode == "head-batch" else t[2] for t in test], dtype=np.int64)


def random_lists(rng, pos, nentity, C, extra=()):
    """[Q, C] lists: random ids with duplicates, the positive, a few -1 in the middle and at the end, and `extra` ids."""
    Q = len(pos)
    cand = rng.randint(nentity, size=(Q, C)).astype(np.int64)
    for q in range(Q):
        if C < 4 and rng.rand() < 0.5:                     # short lists: half of them hold only random ids
            continue
        fill = [int(pos[q])] + [int(e) for e in extra]
        if C > 1:
            fill.append(int(cand[q, 0]))                   # a duplicate
        slots = rng.permutation(C)[:len(fill)]
        cand[q, slots] = fill[:len(slots)]
        if C >= 4:
            cand[q, rng.randint(1, C - 1)] = -1            # padding in the middle
            cand[q, C - 1 - rng.randint(2):] = -1          # and at the end
        elif rng.rand() < 0.3:
            cand[q, rng.randint(C)] = -1
    return cand


def numpy_candidate_stats(raw, pos, mask, cand):
    """The definition over the listed entries: j != pos, each entry counted as often as listed, padding ignored."""
    Q = len(pos)
    rows = np.arange(Q)[:, None]
    valid = (cand >= 0) & (cand != pos[:, None])
    safe = np.where(cand >= 0, cand, 0)
    s = raw[rows, safe]
    sp = raw[np.arange(Q), pos][:, None]
    with np.errstate(invalid="ignore"):
        gt, eq = (s > sp) & valid, (s == sp) & valid
    before, after = cand < pos[:, None], cand > pos[:, None]
    kept = ~mask[rows, safe] if mask is not None else np.ones_like(valid)
    cols = [gt & kept, eq & before & kept, eq & after & kept, gt, eq & before, eq & after]
    return np.stack([c.sum(1) for c in cols], 1).astype(np.int64)


def expected_scores(raw, pos, cand):
    out = raw[np.arange(len(pos))[:, None], np.where(cand >= 0, cand, 0)].astype(np.float32)
    out[cand < 0] = -np.inf
    return out


def assert_bits_equal(got, want, msg=""):
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    assert got.shape == want.shape, msg
    nan = np.isnan(want)
    np.testing.assert_array_equal(np.isnan(got), nan, err_msg=msg)
    np.testing.assert_array_equal(got.view(np.uint32)[~nan], want.view(np.uint32)[~nan], err_msg=msg)


def check_against_oracle(m, raw, test, mode, mask, all_true, cand, **kw):
    pos = positives(test, mode)
    got, sc = m.candidate_rank_statistics(test, cand, mode, exclude_triples=all_true, return_scores=True, **kw)
    assert got.dtype == np.int64 and got.shape == (len(test), 6)
    np.testing.assert_array_equal(got, numpy_candidate_stats(raw, pos, mask, cand), err_msg=mode)
    assert sc.dtype == torch.float32 and sc.device == m.entity_embedding.device
    assert_bits_equal(sc.cpu().numpy(), expected_scores(raw, pos, cand), mode)
    return got


# ------------------------------------------------------------------------------------------------ full-size shapes
@gpu
@pytest.mark.parametrize("model,nentity,nrel,d,gamma", __import__("test_gpu_parity").FULL)
def test_candidate_statistics_bit_exact_vs_c_oracle(model, nentity, nrel, d, gamma):
    """The shapes of test_full_size_eval_bit_exact_vs_c_oracle, lists of 1, 37 and 1000 entries: counts and scores equal
    the oracle's raw scores at the listed ids, and the raw realistic rank is OGB's 1 + #> + #= / 2."""
    from knowledgegraphembedding_b200 import ranks_from_statistics
    from test_gpu_parity import make_model
    de, dr = FLAGS[model]
    st = O.init_tables(model, nentity, nrel, d, gamma, de, dr, seed=0)
    st["entity_embedding"] = (st["entity_embedding"] * 3.0).astype(np.float32)
    rng = np.random.RandomState(2)
    all_true = sorted({(int(rng.randint(nentity)), int(rng.randint(nrel)), int(rng.randint(200))) for _ in range(30000)})
    test = [all_true[i] for i in rng.choice(len(all_true), 24, replace=False)]
    m = make_model(model, nentity, nrel, d, gamma, st)
    for mode in MODES:
        raw = raw_scores(model, st, test, mode, gamma, d)
        mask = filter_mask(test, all_true, mode, nentity, nrel)
        pos = positives(test, mode)
        for C in (1, 37, 1000):
            # half of each list drawn from the filtered entities of the query, so that exclusion is exercised
            cand = random_lists(rng, pos, nentity, C)
            for q in range(len(test)):
                true_j = np.nonzero(mask[q])[0]
                if true_j.size and C > 2:
                    cand[q, 1:C // 2] = np.where(cand[q, 1:C // 2] >= 0, rng.choice(true_j, C // 2 - 1), -1)
                    cand[q, C // 2] = pos[q]
            got = check_against_oracle(m, raw, test, mode, mask, all_true, cand)
            s = expected_scores(raw, pos, cand)
            sp = raw[np.arange(len(test)), pos][:, None]
            neg = (cand >= 0) & (cand != pos[:, None])
            ogb = 1.0 + ((s > sp) & neg).sum(1) + ((s == sp) & neg).sum(1) / 2.0
            np.testing.assert_array_equal(ranks_from_statistics(got, filtered=False, ties="realistic"), ogb)


# ------------------------------------------------------------------------------------------------ all-entity agreement
@gpu
@pytest.mark.parametrize("model", ["TransE", "DistMult", "ComplEx", "RotatE", "pRotatE"])
def test_permutation_lists_give_rank_statistics(model):
    """Every list a random permutation of all entities: the statistics are rank_statistics' on the default path and on
    exact=True, with and without exclusion, and the scores are filtered_ranks' raw scores at the permutation."""
    from test_gpu_parity import make_model
    nentity, nrel, d, gamma, st, test, all_true = tie_case(model, seed=31)
    m = make_model(model, nentity, nrel, d, gamma, st)
    rng = np.random.RandomState(5)
    perm = np.stack([rng.permutation(nentity) for _ in test]).astype(np.int64)
    for mode in MODES:
        with_ex, sc = m.candidate_rank_statistics(test, torch.from_numpy(perm).cuda(), mode, exclude_triples=all_true,
                                                  return_scores=True)
        without = m.candidate_rank_statistics(test, perm, mode)
        for exact in (False, True):
            np.testing.assert_array_equal(with_ex, m.rank_statistics(test, all_true, mode, exact=exact))
            np.testing.assert_array_equal(without, m.rank_statistics(test, [], mode, exact=exact))
        _, full = m.filtered_ranks(test, [], mode, return_scores=True)
        assert_bits_equal(sc.cpu().numpy(), full.gather(1, torch.from_numpy(perm).cuda()).cpu().numpy(), mode)


@gpu
@pytest.mark.parametrize("model", ["TransE", "DistMult", "ComplEx", "RotatE", "pRotatE"])
def test_tie_tables(model):
    """The tie tables of test_gpu_rank_stats (copies of positives on both sides of their id, zero rows, NaN rows, a zero
    and a NaN positive), with those rows in every list: counts and scores equal the oracle's."""
    from test_gpu_parity import make_model
    nentity, nrel, d, gamma, st, test, all_true = tie_case(model, seed=32)
    m = make_model(model, nentity, nrel, d, gamma, st)
    E = st["entity_embedding"]
    rows = E.reshape(nentity, -1)
    zero = np.nonzero((rows == 0).all(1))[0]
    nan = np.nonzero(np.isnan(rows).any(1))[0]
    rng = np.random.RandomState(6)
    for mode in MODES:
        pos = positives(test, mode)
        copies = [np.nonzero((rows == rows[p]).all(1))[0] for p in pos]
        raw = raw_scores(model, st, test, mode, gamma, d)
        mask = filter_mask(test, all_true, mode, nentity, nrel)
        cand = random_lists(rng, pos, nentity, 300, extra=list(zero[:6]) + list(nan[:4]))
        for q in range(len(test)):
            c = copies[q][copies[q] != pos[q]][:8]
            cand[q, 100:100 + c.size] = c
        got = check_against_oracle(m, raw, test, mode, mask, all_true, cand)
        assert got[:, 4].sum() + got[:, 5].sum() > 50, "the lists meet too few ties"
        nan_q = 65 if mode == "head-batch" else 66       # the NaN positive counts nothing
        assert (got[nan_q] == 0).all()


# ------------------------------------------------------------------------------------------------ edge cases
@gpu
@pytest.mark.parametrize("model,nentity,d", [("TransE", 2003, 37), ("RotatE", 2003, 50), ("pRotatE", 2003, 23),
                                             ("ComplEx", 2003, 30), ("RotatE", 100003, 100), ("DistMult", 100003, 100)])
def test_widths(model, nentity, d):
    """Unaligned widths (d not a multiple of 4: the plain-load staging) and d = 100 over 100 k entities."""
    from test_gpu_parity import make_model
    nrel, gamma = 13, 12.0
    de, dr = FLAGS[model]
    st = O.init_tables(model, nentity, nrel, d, gamma, de, dr, seed=3)
    rng = np.random.RandomState(3)
    all_true = sorted({(int(rng.randint(nentity)), int(rng.randint(nrel)), int(rng.randint(100))) for _ in range(4000)})
    test = [all_true[i] for i in rng.choice(len(all_true), 16, replace=False)]
    m = make_model(model, nentity, nrel, d, gamma, st)
    for mode in MODES:
        raw = raw_scores(model, st, test, mode, gamma, d)
        mask = filter_mask(test, all_true, mode, nentity, nrel)
        check_against_oracle(m, raw, test, mode, mask, all_true, random_lists(rng, positives(test, mode), nentity, 500))


@gpu
def test_query_chunk_and_host_filter_index(monkeypatch):
    """query_chunk=7 and the host-sorted filter index give the result of the default chunk and the device index."""
    from test_gpu_parity import make_model
    nentity, nrel, d, gamma, st, test, all_true = tie_case("RotatE", seed=33)
    m = make_model("RotatE", nentity, nrel, d, gamma, st)
    rng = np.random.RandomState(7)
    for mode in MODES:
        cand = random_lists(rng, positives(test, mode), nentity, 200)
        want, want_sc = m.candidate_rank_statistics(test, cand, mode, exclude_triples=all_true, return_scores=True)
        got, sc = m.candidate_rank_statistics(test, cand, mode, exclude_triples=all_true, query_chunk=7,
                                              return_scores=True)
        np.testing.assert_array_equal(got, want)
        assert torch.equal(sc.view(torch.int32), want_sc.view(torch.int32))
        with monkeypatch.context() as mp:
            mp.setenv("KGE_FILTER_HOST_INDEX", "1")
            fresh = list(all_true)                       # a new list object: a new cache entry, the sorted index
            np.testing.assert_array_equal(m.candidate_rank_statistics(test, cand, mode, exclude_triples=fresh,
                                                                      query_chunk=7), want)
            assert m._filter_cache["tables"][(mode, m.entity_embedding.device)][0] == "sorted"
        np.testing.assert_array_equal(m.candidate_rank_statistics(test, cand.tolist(), mode, exclude_triples=all_true),
                                      want)


@gpu
def test_bad_ids_raise_once():
    from test_gpu_parity import make_model
    nentity, nrel, d, gamma, st, test, all_true = tie_case("TransE", seed=34)
    m = make_model("TransE", nentity, nrel, d, gamma, st)
    cand = random_lists(np.random.RandomState(8), positives(test, "tail-batch"), nentity, 40)
    want = m.candidate_rank_statistics(test, cand, "tail-batch")
    for bad in (nentity, -2, 1 << 40):
        wrong = cand.copy()
        wrong[3, 5] = bad
        with pytest.raises(IndexError):
            m.candidate_rank_statistics(test, wrong, "tail-batch")
        np.testing.assert_array_equal(m.candidate_rank_statistics(test, cand, "tail-batch"), want)
    with pytest.raises(ValueError):
        m.candidate_rank_statistics(test, cand, "single")
    with pytest.raises(ValueError):
        m.candidate_rank_statistics(test, cand[:-1], "tail-batch")


# ------------------------------------------------------------------------------------------------ slices, ranks
@gpu
@pytest.mark.parametrize("model", ["ComplEx", "pRotatE"])
def test_column_slices_sum_to_full_statistics(model):
    """Column slices through the ABI add up to the method's statistics, and each slice writes only its own scores."""
    from knowledgegraphembedding_b200 import _lib as L
    from knowledgegraphembedding_b200.model import _ptr, _stream
    from test_gpu_parity import make_model
    nentity, nrel, d, gamma, st, test, all_true = tie_case(model, seed=35)
    m = make_model(model, nentity, nrel, d, gamma, st)
    mode = "head-batch"
    cand = random_lists(np.random.RandomState(9), positives(test, mode), nentity, 333)
    want, want_sc = m.candidate_rank_statistics(test, cand, mode, return_scores=True)
    dev = m.entity_embedding.device
    desc, stt, mid = m._descriptor(), _stream(dev), L.MODE_IDS[mode]
    Q, De = len(test), m.entity_dim
    q = torch.tensor(test, dtype=torch.int64, device=dev)
    c = torch.from_numpy(cand).to(dev)
    qvec, pos = torch.empty(Q * De, device=dev), torch.empty(Q, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    phase = None
    if model == "pRotatE":
        phase = torch.empty(nentity * De, device=dev)
        L.call("kge_eval_phase_table", ctypes.byref(desc), _ptr(phase), stt)
    L.call("kge_eval_query_vectors", ctypes.byref(desc), mid, _ptr(q), Q, _ptr(qvec), _ptr(err), stt)
    L.call("kge_eval_positive_scores", ctypes.byref(desc), mid, _ptr(qvec), _ptr(q), Q, _ptr(phase), _ptr(pos), stt)
    total = torch.zeros((Q, 6), dtype=torch.int32, device=dev)
    scores = torch.full((Q, 333), 7.0, device=dev)
    cuts = [0, 1, 128, 129, 300, 333]
    for b, e in zip(cuts[:-1], cuts[1:]):
        part = torch.zeros((Q, 6), dtype=torch.int32, device=dev)
        L.call("kge_eval_candidate_rank_stats", ctypes.byref(desc), mid, _ptr(qvec), _ptr(q), Q, _ptr(phase), _ptr(pos),
               _ptr(c), 333, b, e, None, _ptr(part), _ptr(scores), _ptr(err), stt)
        total += part
        assert bool((scores[:, e:] == 7.0).all())
    torch.cuda.synchronize()
    assert err.item() == 0
    np.testing.assert_array_equal(total.cpu().numpy(), want)
    assert torch.equal(scores.view(torch.int32), want_sc.view(torch.int32))


def _run_worker(n, **env):
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "candidate_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, **env))
    if not (res.returncode == 0 and res.stdout.strip().endswith("ok")):
        sys.stderr.write(res.stdout[-3000:] + "\n" + res.stderr[-8000:])
    assert res.returncode == 0 and res.stdout.strip().endswith("ok"), "candidate worker failed (output on stderr)"


@gpu
def test_candidate_statistics_two_ranks_sharing_one_gpu():
    from test_gpu_topk import _gpu0_shareable
    if not _gpu0_shareable():
        pytest.skip("GPU 0 is in an exclusive compute mode")
    _run_worker(2, KGE_TEST_SAME_GPU="1")


# ------------------------------------------------------------------------------------------------ no GPU needed
def test_candidate_abi_argument_errors_without_a_gpu():
    from knowledgegraphembedding_b200 import _lib as L
    lib = L.load()
    desc = L.KgeModelStruct(model=L.ROTATE, device=0, nentity=100, nrelation=5, hidden_dim=8, entity_dim=16,
                            relation_dim=8, gamma=6.0, embedding_range=1.0, entity=16, relation=16, modulus=None)
    dd = ctypes.byref(desc)

    def call(mode=L.TAIL_BATCH, qvec=16, queries=16, Q=10, pos=16, cand=16, ld=50, b=0, e=50, stats=16, err=16):
        return lib.kge_eval_candidate_rank_stats(dd, mode, qvec, queries, Q, None, pos, cand, ld, b, e, None, stats,
                                                 None, err, None)
    assert call(mode=L.SINGLE) == L.ERR_INVALID and b"negative batch mode" in lib.kge_last_error()
    for kw in (dict(qvec=None), dict(queries=None), dict(pos=None), dict(cand=None), dict(stats=None), dict(err=None)):
        assert call(**kw) == L.ERR_INVALID and b"null pointer" in lib.kge_last_error(), kw
    assert call(Q=-1) == L.ERR_INVALID and b"negative query count" in lib.kge_last_error()
    for ld in (0, -3):
        assert call(ld=ld, e=0) == L.ERR_INVALID and b"row length" in lib.kge_last_error()
    for b, e in ((0, 51), (-1, 5), (30, 20)):
        assert call(b=b, e=e) == L.ERR_INVALID and b"column slice" in lib.kge_last_error()


def test_candidate_input_checks_without_a_gpu():
    from knowledgegraphembedding_b200 import KGEModel
    m = KGEModel("TransE", 50, 4, 8, 6.0)                 # on the CPU: the checks run before any device work
    test = [(1, 2, 3), (4, 0, 5)]
    good = np.array([[1, 2, -1], [7, 8, 9]])
    for bad_mode in ("single", "tail", None):
        with pytest.raises(ValueError, match="negative batch mode"):
            m.candidate_rank_statistics(test, good, bad_mode)
    for bad in (good[0], good[:1], good.astype(np.float32), [[1, 2], [3]], torch.ones(2, 3, dtype=torch.bool),
                np.zeros((2, 3, 1), np.int64)):
        with pytest.raises(ValueError, match="candidates must be"):
            m.candidate_rank_statistics(test, bad, "head-batch")
    for bad in ([(1, 2)], np.zeros((2, 4), np.int64), np.zeros((2, 3), np.float64)):
        with pytest.raises(ValueError, match="queries must be"):
            m.candidate_rank_statistics(bad, good, "head-batch")
    for chunk in (0, -1, 2.5, True):
        with pytest.raises(ValueError, match="query_chunk"):
            m.candidate_rank_statistics(test, good, "tail-batch", query_chunk=chunk)
    with pytest.raises(RuntimeError, match="CUDA device"):                  # well-formed: only then the device check
        m.candidate_rank_statistics(test, good, "tail-batch")
