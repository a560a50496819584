"""Rank statistics (KGEModel.rank_statistics, kge_eval_count_rank_stats*): per query the counts of candidates j != pos
that score above the positive, tie with it before its id, or tie with it after its id, among the unfiltered candidates
(columns 0-2) and among all candidates (columns 3-5).  Checked against numpy counts over the C oracle's raw scores with
the filter applied as a mask, against filtered_ranks (filtered and with an empty filter list), across the exact,
two-stage and tcgen05 paths on tables full of exact ties, over entity slices, after an ambiguous-list overflow and on
several ranks; without a GPU, ranks_from_statistics and the argument checks of the new ABI entries."""
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
MODES = ("head-batch", "tail-batch")


def _lib():
    from knowledgegraphembedding_b200 import _lib as L
    return L


def raw_scores(model, st, test, mode, gamma, d):
    """[Q, nentity] canonical scores with no filter (C oracle)."""
    return C.eval_scores(model, st, test, mode, gamma, O.embedding_range(gamma, d), np.zeros(len(test) + 1, np.int64),
                         np.zeros(0, np.int32))


def filter_mask(test, all_true, mode, nentity, nrel):
    from knowledgegraphembedding_b200 import FilterIndex
    off, ent = FilterIndex(all_true, nentity, nrel).csr(test, mode)
    mask = np.zeros((len(test), nentity), bool)
    for q in range(len(test)):
        mask[q, ent[off[q]:off[q + 1]]] = True
    return mask


def numpy_stats(raw, test, mode, mask):
    """The definition: six counts per query over j != pos, the filter as a mask (a filtered column keeps its score)."""
    pos = np.array([t[0] if mode == "head-batch" else t[2] for t in test])
    sp = raw[np.arange(len(test)), pos][:, None]
    j = np.arange(raw.shape[1])[None, :]
    other = j != pos[:, None]
    with np.errstate(invalid="ignore"):
        gt, eq = (raw > sp) & other, (raw == sp) & other
    before, after, kept = j < pos[:, None], j > pos[:, None], ~mask
    cols = [gt & kept, eq & before & kept, eq & after & kept, gt, eq & before, eq & after]
    return np.stack([c.sum(1) for c in cols], 1).astype(np.int64)


def check_agrees_with_ranks(m, stats, test, all_true, mode, exact):
    np.testing.assert_array_equal(1 + stats[:, 0] + stats[:, 1], m.filtered_ranks(test, all_true, mode, exact=exact))
    np.testing.assert_array_equal(1 + stats[:, 3] + stats[:, 4], m.filtered_ranks(test, [], mode, exact=exact))


# ------------------------------------------------------------------------------------------------ full-size shapes
@gpu
@pytest.mark.parametrize("model,nentity,nrel,d,gamma", __import__("test_gpu_parity").FULL)
def test_rank_statistics_bit_exact_vs_c_oracle(model, nentity, nrel, d, gamma):
    """The shapes of test_full_size_eval_bit_exact_vs_c_oracle, on the default path (tcgen05 / two-stage / exact) and on
    exact=True: the statistics equal numpy counts over the oracle's raw scores, and give filtered_ranks' filtered and
    raw ranks."""
    from test_gpu_parity import FLAGS, make_model
    de, dr = FLAGS[model]
    st = O.init_tables(model, nentity, nrel, d, gamma, de, dr, seed=0)
    st["entity_embedding"] = (st["entity_embedding"] * 3.0).astype(np.float32)
    rng = np.random.RandomState(2)
    all_true = sorted({(int(rng.randint(nentity)), int(rng.randint(nrel)), int(rng.randint(200))) for _ in range(30000)})
    test = [all_true[i] for i in rng.choice(len(all_true), 24, replace=False)]
    m = make_model(model, nentity, nrel, d, gamma, st)
    for mode in MODES:
        want = numpy_stats(raw_scores(model, st, test, mode, gamma, d), test, mode,
                           filter_mask(test, all_true, mode, nentity, nrel))
        for exact in (False, True):
            got = m.rank_statistics(test, all_true, mode, exact=exact)
            assert got.dtype == np.int64 and got.shape == (len(test), 6)
            np.testing.assert_array_equal(got, want, err_msg="%s %s exact=%s" % (model, mode, exact))
            check_agrees_with_ranks(m, got, test, all_true, mode, exact)


# ------------------------------------------------------------------------------------------------ dense ties
FLAGS = {"TransE": (False, False), "DistMult": (False, False), "ComplEx": (True, True), "RotatE": (True, False),
         "pRotatE": (False, False)}


def tie_case(model, seed):
    """Tables full of exact ties: copies of the positives' rows on both sides of the positive's id (some of them
    filtered), all-zero rows (DistMult: +-0 scores, and a zero positive), NaN rows, and one query whose positive is a
    NaN row."""
    nentity, nrel, d, gamma = 3001, 7, 64, 12.0
    de, dr = FLAGS[model]
    st = O.init_tables(model, nentity, nrel, d, gamma, de, dr, seed=seed)
    E = st["entity_embedding"]
    rng = np.random.RandomState(seed)
    Q = 96
    pos = 500 + rng.choice(2000, Q, replace=False)
    rels = rng.randint(nrel, size=Q)
    copies = {}
    for p in pos[:64]:                                 # 3 copies of each of 64 positives, before and after it
        copies[int(p)] = [int(c) for c in (p - 1 - rng.randint(400), p + 1 + rng.randint(400), rng.randint(nentity))
                          if c not in pos]
        E[copies[int(p)]] = E[p]
    zero = rng.choice(nentity, 40, replace=False)
    zero = zero[~np.isin(zero, pos[:64])]
    E[zero] = 0.0
    nan = np.setdiff1d(rng.choice(nentity, 10, replace=False), pos[:64])
    E[nan] = np.nan
    E[pos[64]] = 0.0                                   # a positive that ties with every zero row
    E[pos[65]] = np.nan                                # a NaN positive: counts nothing
    st["entity_embedding"] = E
    # head-batch ranks h = pos[i], tail-batch ranks t = pos[i - 1]: every mode meets the copies, the zero and NaN rows
    test = [(int(p), int(r), int(p2)) for p, r, p2 in zip(pos, rels, np.roll(pos, 1))]
    rng2 = np.random.RandomState(seed + 1)
    all_true = set(test)
    for (h, r, t) in test:                             # filter one copy of each side, a zero row and random rows
        if copies.get(h):
            all_true.add((copies[h][0], r, t))
        if copies.get(t):
            all_true.add((h, r, copies[t][-1]))
        all_true.add((int(zero[0]), r, t))
        all_true.add((h, r, int(zero[1])))
        for _ in range(8):
            all_true.add((int(rng2.randint(nentity)), r, t))
            all_true.add((h, r, int(rng2.randint(nentity))))
    return nentity, nrel, d, gamma, st, test, sorted(all_true)


@gpu
@pytest.mark.parametrize("model", ["TransE", "DistMult", "ComplEx", "RotatE", "pRotatE"])
def test_dense_ties_identical_on_every_path(model):
    from test_gpu_parity import make_model
    nentity, nrel, d, gamma, st, test, all_true = tie_case(model, seed=21)
    m = make_model(model, nentity, nrel, d, gamma, st)
    for mode in MODES:
        want = numpy_stats(raw_scores(model, st, test, mode, gamma, d), test, mode,
                           filter_mask(test, all_true, mode, nentity, nrel))
        assert want[:, 4].sum() + want[:, 5].sum() > 100, "the case has too few ties"
        assert (want[65 if mode == "head-batch" else 66] == 0).all()       # the NaN positive
        fast = m.rank_statistics(test, all_true, mode)
        exact = m.rank_statistics(test, all_true, mode, exact=True)
        np.testing.assert_array_equal(exact, want, err_msg=mode)
        np.testing.assert_array_equal(fast, want, err_msg=mode)
        check_agrees_with_ranks(m, fast, test, all_true, mode, False)


@gpu
@pytest.mark.parametrize("name", ["rotate_tiny_1e-3", "protate_modulus_1e-3"])
def test_dense_ties_of_the_band_cases(name):
    """The tiny-distance RotatE table (thousands of exact ties with s_pos) and the small-modulus pRotatE table of the
    two-stage band test: two-stage statistics equal the exact kernel's, and numpy counts over its score dump (the
    oracle's bits, pinned by the parity tests)."""
    from test_gpu_two_stage_band import build, true_triples
    model, gamma, d, st, test, m = build(name)
    nentity = st["entity_embedding"].shape[0]
    test = test[:1024]
    all_true = true_triples(test, nentity, seed=7)
    for mode in MODES:
        _, sc = m.filtered_ranks(test, [], mode, return_scores=True)
        want = numpy_stats(sc.cpu().numpy(), test, mode, filter_mask(test, all_true, mode, nentity, 5))
        if name.startswith("rotate"):
            assert want[:, 4].sum() + want[:, 5].sum() > 100
        np.testing.assert_array_equal(m.rank_statistics(test, all_true, mode, exact=True), want)
        np.testing.assert_array_equal(m.rank_statistics(test, all_true, mode), want)
        del sc


# ------------------------------------------------------------------------------------------------ slices, overflow
def _abi_stats(m, test, all_true, mode, path, slices):
    """Statistics of one ABI entry ('exact', 'two_stage', 'gemm') summed over entity slices."""
    L = _lib()
    from knowledgegraphembedding_b200 import FilterIndex
    from knowledgegraphembedding_b200.model import _ptr, _stream
    dev = m.entity_embedding.device
    nentity, De = m.entity_embedding.shape
    desc, stt, mid = m._descriptor(), _stream(dev), L.MODE_IDS[mode]
    Q = len(test)
    q = torch.tensor(test, dtype=torch.int64, device=dev)
    off, ent = FilterIndex(all_true, nentity, m.relation_embedding.shape[0]).csr(test, mode)
    d_off, d_ent = torch.from_numpy(off).to(dev), torch.from_numpy(ent).to(dev)
    bits = torch.zeros(Q * ((nentity + 31) // 32), dtype=torch.int32, device=dev)
    qvec = torch.empty(Q * De, device=dev)
    pos = torch.empty(Q, device=dev)
    phase = None
    if m.model_name == "pRotatE":
        phase = torch.empty(nentity * De, device=dev)
        L.call("kge_eval_phase_table", ctypes.byref(desc), _ptr(phase), stt)
    L.call("kge_eval_filter_bits", _ptr(d_off), _ptr(d_ent), Q, nentity, _ptr(bits), stt)
    L.call("kge_eval_query_vectors", ctypes.byref(desc), mid, _ptr(q), Q, _ptr(qvec), None, stt)
    L.call("kge_eval_positive_scores", ctypes.byref(desc), mid, _ptr(qvec), _ptr(q), Q, _ptr(phase), _ptr(pos), stt)
    cap = Q * nentity + 64
    amb = torch.empty(2 * cap, dtype=torch.int32, device=dev)
    amb_count = torch.zeros(2, dtype=torch.int32, device=dev)
    if path == "gemm":
        ehi, elo, qhi, qlo = (torch.empty(n * De, device=dev) for n in (nentity, nentity, Q, Q))
        enorm, qnorm = torch.empty(nentity, device=dev), torch.empty(Q, device=dev)
        L.call("kge_eval_gemm_split", _ptr(m.entity_embedding), nentity, De, _ptr(ehi), _ptr(elo), _ptr(enorm), stt)
        L.call("kge_eval_gemm_split", _ptr(qvec), Q, De, _ptr(qhi), _ptr(qlo), _ptr(qnorm), stt)
    total = torch.zeros((Q, 6), dtype=torch.int32, device=dev)
    for b, e in slices:
        part = torch.zeros((Q, 6), dtype=torch.int32, device=dev)
        if path == "exact":
            L.call("kge_eval_count_rank_stats", ctypes.byref(desc), mid, _ptr(qvec), _ptr(q), Q, _ptr(phase), _ptr(pos),
                   _ptr(bits), b, e, _ptr(part), stt)
        elif path == "two_stage":
            L.call("kge_eval_count_rank_stats_two_stage", ctypes.byref(desc), mid, _ptr(qvec), _ptr(q), Q, _ptr(phase),
                   _ptr(pos), _ptr(bits), b, e, _ptr(part), _ptr(amb), cap, _ptr(amb_count), stt)
        else:
            L.call("kge_eval_gemm_count_rank_stats", ctypes.byref(desc), mid, _ptr(qvec), _ptr(qhi), _ptr(qlo),
                   _ptr(qnorm), _ptr(q), Q, _ptr(pos), _ptr(bits), _ptr(ehi), _ptr(elo), _ptr(enorm), b, e, _ptr(part),
                   _ptr(amb), cap, _ptr(amb_count), stt)
        total += part
    torch.cuda.synchronize()
    assert amb_count[1].item() == 0
    return total.cpu().numpy().astype(np.int64)


@gpu
@pytest.mark.parametrize("model,path", [("TransE", "exact"), ("RotatE", "exact"), ("RotatE", "two_stage"),
                                        ("pRotatE", "two_stage"), ("DistMult", "gemm"), ("ComplEx", "gemm")])
def test_entity_slices_sum_to_full_statistics(model, path):
    """Slices cut at multiples of 32 (the tcgen05 entry's rule) and at the 128-aligned shards of a multi-GPU run add up
    to the full-range statistics of rank_statistics."""
    from knowledgegraphembedding_b200 import shard_bounds
    from test_gpu_parity import make_model
    nentity, nrel, d, gamma, st, test, all_true = tie_case(model, seed=22)
    m = make_model(model, nentity, nrel, d, gamma, st)
    cuts = [0, 32, 96, 992, 1504, 2016, 2880, nentity]
    for mode in MODES:
        full = m.rank_statistics(test, all_true, mode)
        np.testing.assert_array_equal(_abi_stats(m, test, all_true, mode, path, list(zip(cuts[:-1], cuts[1:]))), full)
        shards = [shard_bounds(nentity, r, 8, align=128) for r in range(8)]
        np.testing.assert_array_equal(_abi_stats(m, test, all_true, mode, path, shards), full)


@gpu
@pytest.mark.parametrize("model", ["RotatE", "pRotatE", "ComplEx"])
def test_ambiguous_list_overflow_gives_the_same_statistics(model, monkeypatch):
    from test_gpu_parity import make_model
    nentity, nrel, d, gamma, st, test, all_true = tie_case(model, seed=23)
    m = make_model(model, nentity, nrel, d, gamma, st)
    want = {mode: m.rank_statistics(test, all_true, mode, exact=True) for mode in MODES}
    monkeypatch.setenv("KGE_EVAL_AMB_CAP", "1")
    for mode in MODES:
        np.testing.assert_array_equal(m.rank_statistics(test, all_true, mode, query_chunk=32), want[mode])


# ------------------------------------------------------------------------------------------------ several ranks
def _run_worker(n, **env):
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "rank_stats_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, **env))
    if not (res.returncode == 0 and res.stdout.strip().endswith("ok")):
        sys.stderr.write(res.stdout[-3000:] + "\n" + res.stderr[-8000:])
    assert res.returncode == 0 and res.stdout.strip().endswith("ok"), "rank statistics worker failed (output on stderr)"


@gpu
def test_rank_statistics_two_ranks_sharing_one_gpu():
    from test_gpu_topk import _gpu0_shareable
    if not _gpu0_shareable():
        pytest.skip("GPU 0 is in an exclusive compute mode")
    _run_worker(2, KGE_TEST_SAME_GPU="1")


@gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_rank_statistics_one_gpu_per_rank():
    _run_worker(min(torch.cuda.device_count(), 8))


# ------------------------------------------------------------------------------------------------ no GPU needed
def test_ranks_from_statistics():
    from knowledgegraphembedding_b200 import ranks_from_statistics
    stats = np.array([[0, 0, 0, 0, 0, 0], [3, 1, 2, 5, 4, 6], [7, 0, 3, 9, 0, 3]], dtype=np.int64)
    for filtered, (g, eb, ea) in ((True, (0, 1, 2)), (False, (3, 4, 5))):
        G, EB, EA = stats[:, g], stats[:, eb], stats[:, ea]
        opt = ranks_from_statistics(stats, filtered, "optimistic")
        assert opt.dtype == np.int64 and opt.tolist() == (1 + G).tolist()
        assert ranks_from_statistics(stats, filtered=filtered).tolist() == (1 + G + EB).tolist()
        assert ranks_from_statistics(stats, filtered, "pessimistic").tolist() == (1 + G + EB + EA).tolist()
        real = ranks_from_statistics(stats, filtered, "realistic")
        assert real.dtype == np.float64 and real.tolist() == (1 + G + (EB + EA) / 2).tolist()
    assert ranks_from_statistics(stats, ties="realistic").tolist() == [1.0, 5.5, 9.5]
    assert ranks_from_statistics(stats.astype(np.int32)).tolist() == [1, 5, 8]
    for bad in (stats[:, :5], stats[0], stats.astype(np.float64)):
        with pytest.raises(ValueError, match="integer table"):
            ranks_from_statistics(bad)
    with pytest.raises(ValueError, match="ties must be"):
        ranks_from_statistics(stats, ties="random")


def test_rank_stats_abi_argument_errors_without_a_gpu():
    L = _lib()
    lib = L.load()
    desc = L.KgeModelStruct(model=L.ROTATE, device=0, nentity=100, nrelation=5, hidden_dim=8, entity_dim=16,
                            relation_dim=8, gamma=6.0, embedding_range=1.0, entity=16, relation=16, modulus=None)
    d = ctypes.byref(desc)

    def exact(mode=L.TAIL_BATCH, b=0, e=100, stats=16, qvec=16):
        return lib.kge_eval_count_rank_stats(d, mode, qvec, 16, 10, None, 16, 16, b, e, stats, None)

    def two_stage(mode=L.TAIL_BATCH, b=0, e=100, amb=16, cap=10, amb_count=16, stats=16):
        return lib.kge_eval_count_rank_stats_two_stage(d, mode, 16, 16, 10, None, 16, 16, b, e, stats, amb, cap,
                                                       amb_count, None)
    for call in (exact, two_stage):
        assert call(mode=L.SINGLE) == L.ERR_INVALID and b"negative batch mode" in lib.kge_last_error()
        for b, e in ((0, 101), (-1, 5), (30, 20)):
            assert call(b=b, e=e) == L.ERR_INVALID and b"entity slice" in lib.kge_last_error()
        assert call(stats=None) == L.ERR_INVALID and b"null pointer" in lib.kge_last_error()
    assert exact(qvec=None) == L.ERR_INVALID and b"null pointer" in lib.kge_last_error()
    for kw in (dict(amb=None), dict(cap=0), dict(amb_count=None)):
        assert two_stage(**kw) == L.ERR_INVALID and b"ambiguous-pair buffers" in lib.kge_last_error()
    desc.model, desc.entity_dim = L.DISTMULT, 8

    def gemm(mode=L.TAIL_BATCH, b=0, e=100, stats=16, amb=16, cap=10):
        return lib.kge_eval_gemm_count_rank_stats(d, mode, 16, 16, 16, 16, 16, 10, 16, 16, 16, 16, 16, b, e, stats, amb,
                                                  cap, 16, None)
    assert gemm(mode=L.SINGLE) == L.ERR_INVALID and b"negative batch mode" in lib.kge_last_error()
    for b, e in ((16, 100), (0, 101), (64, 32)):
        assert gemm(b=b, e=e) == L.ERR_INVALID and b"entity slice" in lib.kge_last_error()
    for kw in (dict(stats=None), dict(amb=None), dict(cap=0)):
        assert gemm(**kw) == L.ERR_INVALID and b"null pointer" in lib.kge_last_error()
    desc.model = L.TRANSE
    assert gemm() == L.ERR_INVALID and b"tcgen05 path serves" in lib.kge_last_error()
