"""Negative sampler (SURVEY 8f-1; reference: codes/dataloader.py:13-119,165-186)."""
import numpy as np
import pytest

from conftest import load_golden
from oracle import kge_oracle as O


def countries():
    g = load_golden("countries_S1")
    tri = [tuple(int(v) for v in r) for r in g["train"]]
    return g, tri, int(g["nentity"]), int(g["nrelation"])


def test_philox_known_answers():
    """Random123's published Philox4x32-10 vectors pin the oracle's stream (the device stream is compared with it)."""
    kat = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
           ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
           ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
            (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for ctr, key, want in kat:
        got = O._philox4x32_10(*[[c] for c in ctr], *key)
        assert tuple(int(x[0]) for x in got) == want


def test_weights_and_true_lists_match_reference():
    from knowledgegraphembedding_b200.sampler import subsampling_weights, true_lists
    g, tri, nentity, nrel = countries()
    w = subsampling_weights(tri)
    np.testing.assert_array_equal(w, O.subsampling_weight(tri))
    index = {t: i for i, t in enumerate(tri)}
    for step in range(4):       # weights the reference's TrainDataset produced for its own batches (golden)
        rows = [index[tuple(int(v) for v in p)] for p in g[f"pos{step}"].astype(np.int64)]
        np.testing.assert_array_equal(w[rows], g[f"w{step}"])
    th, tt = O.true_head_and_tail(tri)
    for mode in ("head-batch", "tail-batch"):
        start, length, ents = true_lists(tri, nentity, nrel, mode)
        for i, (h, r, t) in enumerate(tri[:200]):
            want = sorted(th[(r, t)] if mode == "head-batch" else tt[(h, r)])
            assert ents[start[i]:start[i] + length[i]].tolist() == want
    # the reference's own negatives never hit the true set; neither may the oracle's
    neg = O.sample_negatives(tri, list(range(16)), "tail-batch", nentity, 8, seed=1, step=1)
    for b in range(16):
        h, r, t = tri[b]
        assert not set(neg[b].tolist()) & tt[(h, r)]
    with pytest.raises(ValueError):
        true_lists(tri, nentity, nrel, "sideways")


@pytest.mark.gpu
def test_device_negatives_bit_exact_vs_oracle_and_filtered():
    import torch
    from knowledgegraphembedding_b200.sampler import GpuTrainDataset
    g, tri, nentity, nrel = countries()
    rng = np.random.RandomState(0)
    th, tt = O.true_head_and_tail(tri)
    for mode in ("head-batch", "tail-batch"):
        ds = GpuTrainDataset(tri, nentity, nrel, 24, mode, 64, "cuda", seed=5)
        index = rng.randint(len(tri), size=40)
        pos, neg, w, md = ds.sample(torch.from_numpy(index), step=7)
        assert md == mode and neg.dtype == torch.int64 and neg.shape == (40, 24) and neg.is_cuda
        want = O.sample_negatives(tri, index, mode, nentity, 24, seed=5, step=7)
        np.testing.assert_array_equal(neg.cpu().numpy(), want)                 # same Philox stream, same rejections
        np.testing.assert_array_equal(pos.cpu().numpy(), np.asarray(tri)[index])
        np.testing.assert_array_equal(w.cpu().numpy(), O.subsampling_weight(tri)[index])
    # large draw: never a true entity, and uniform over the complement (chi-square, 271 entities)
    ds = GpuTrainDataset(tri, nentity, nrel, 4096, "tail-batch", 64, "cuda", seed=9)
    index = np.zeros(64, dtype=np.int64)                                       # the same triple 64 times
    _, neg, _, _ = ds.sample(torch.from_numpy(index), step=1)
    neg = neg.cpu().numpy().ravel()
    h, r, t = tri[0]
    true = tt[(h, r)]
    assert not set(np.unique(neg).tolist()) & true
    allowed = nentity - len(true)
    counts = np.bincount(neg, minlength=nentity)
    expected = neg.size / allowed
    chi2 = ((counts[[e for e in range(nentity) if e not in true]] - expected) ** 2 / expected).sum()
    assert chi2 < allowed + 6 * np.sqrt(2 * allowed)                            # mean k, sd sqrt(2k)


@pytest.mark.gpu
def test_bidirectional_iterator_contract_and_training():
    """First call tail-batch, then alternating (dataloader.py:171-177); every epoch visits each triple once with a
    ragged last batch; the 4-tuple feeds train_step directly."""
    import types

    import torch
    from knowledgegraphembedding_b200 import KGEModel
    from knowledgegraphembedding_b200.sampler import BidirectionalGpuIterator
    g, tri, nentity, nrel = countries()
    it = BidirectionalGpuIterator(tri, nentity, nrel, 16, 200, "cuda", seed=3)
    modes, seen_tail = [], []
    nb = (len(tri) + 199) // 200
    for _ in range(2 * nb):
        pos, neg, w, mode = next(it)
        modes.append(mode)
        if mode == "tail-batch":
            seen_tail.append(pos.cpu().numpy())
    assert modes[:4] == ["tail-batch", "head-batch", "tail-batch", "head-batch"]
    seen = np.concatenate(seen_tail)
    assert seen.shape[0] == len(tri) and seen_tail[-1].shape[0] == len(tri) - 200 * (nb - 1)
    assert sorted(map(tuple, seen.tolist())) == sorted(tri)
    m = KGEModel("RotatE", nentity, nrel, 32, 6.0, double_entity_embedding=True).cuda()
    opt = torch.optim.Adam(filter(lambda p: p.requires_grad, m.parameters()), lr=1e-3)
    args = types.SimpleNamespace(cuda=True, negative_adversarial_sampling=True, adversarial_temperature=1.0,
                                 uni_weight=False, regularization=0.0)
    losses = [KGEModel.train_step(m, opt, it, args)["loss"] for _ in range(30)]
    assert np.isfinite(losses).all() and np.mean(losses[-5:]) < np.mean(losses[:5])


@pytest.mark.gpu
def test_forty_steps_track_the_cpu_oracle_on_countries():
    """40 consecutive train_steps on countries_S1 (device-sampled batches, alternating modes, one LR decay with the
    Adam re-creation of run.py:315-322): every step's losses stay within 1e-4 of the C oracle fed the same batches,
    and the final tables agree except for a vanishing fraction of sign-ambiguous Adam elements."""
    import types

    import torch
    from conftest import outlier_fraction, relinf
    from knowledgegraphembedding_b200 import KGEModel
    from knowledgegraphembedding_b200.sampler import BidirectionalGpuIterator
    from oracle import c_oracle as C
    g, tri, nentity, nrel = countries()
    d, gamma = 64, 2.0
    st = O.init_tables("RotatE", nentity, nrel, d, gamma, True, False, seed=4)
    m = KGEModel("RotatE", nentity, nrel, d, gamma, double_entity_embedding=True)
    with torch.no_grad():
        m.entity_embedding.copy_(torch.from_numpy(st["entity_embedding"]))
        m.relation_embedding.copy_(torch.from_numpy(st["relation_embedding"]))
    m = m.cuda()
    ts = C.TrainState("RotatE", st, gamma, d)
    it = BidirectionalGpuIterator(tri, nentity, nrel, 32, 256, "cuda", seed=8)
    args = types.SimpleNamespace(cuda=True, negative_adversarial_sampling=True, adversarial_temperature=1.0,
                                 uni_weight=False, regularization=0.0)
    lr = 5e-4
    opt = torch.optim.Adam(filter(lambda p: p.requires_grad, m.parameters()), lr=lr)
    for step in range(40):
        if step == 25:
            lr /= 10
            opt = torch.optim.Adam(filter(lambda p: p.requires_grad, m.parameters()), lr=lr)
            ts.reset_optimizer()
        batch = next(it)
        log = KGEModel.train_step(m, opt, iter([batch]), args)
        ref = C.train_step(ts, tuple(b.cpu().numpy() if hasattr(b, "cpu") else b for b in batch), lr=lr,
                           adversarial=True, alpha=1.0)
        for k in ref:
            assert abs(log[k] - ref[k]) <= 1e-4 * abs(ref[k]), (step, k, log[k], ref[k])
    E = m.entity_embedding.detach().cpu().numpy()
    assert outlier_fraction(E, ts.state["entity_embedding"], 1e-4) < 2e-3
    assert relinf(m.relation_embedding.detach().cpu().numpy(), ts.state["relation_embedding"]) < 1e-3
