"""GPU parity tests: the CUDA path (through the C ABI, via the KGEModel drop-in) against
  * the golden vectors produced by the unmodified reference (tests/golden/*.npz),
  * the CPU oracles (oracle/kge_oracle.py numpy, oracle/kge_oracle.c) on seeded inputs,
  * at BASELINE.json's full sizes: bit-exact evaluation scores/ranks vs the C oracle, and size-independent
    properties for the train path.
Tolerance (north_star): scores, loss, updated embeddings within 1e-5 relative (fp32); ranks bit-exact.
"""
import os
import types

import numpy as np
import pytest
import torch

from conftest import GOLDEN, load_golden, outlier_fraction, relinf
from oracle import c_oracle as C
from oracle import kge_oracle as O

pytestmark = pytest.mark.gpu

TOL = 1e-5
MODELS = ["TransE", "DistMult", "ComplEx", "RotatE", "pRotatE"]
FLAGS = {"TransE": (False, False), "DistMult": (False, False), "ComplEx": (True, True),
         "RotatE": (True, False), "pRotatE": (False, False)}
DIST = ("TransE", "RotatE", "pRotatE")       # score = gamma - distance: tolerance is relative to the distance


def KGE():
    from knowledgegraphembedding_b200 import KGEModel
    return KGEModel


def make_model(model, nentity, nrelation, d, gamma, state=None):
    de, dr = FLAGS[model]
    m = KGE()(model_name=model, nentity=nentity, nrelation=nrelation, hidden_dim=d, gamma=gamma,
              double_entity_embedding=de, double_relation_embedding=dr)
    if state is not None:
        with torch.no_grad():
            m.entity_embedding.copy_(torch.from_numpy(np.asarray(state["entity_embedding"])))
            m.relation_embedding.copy_(torch.from_numpy(np.asarray(state["relation_embedding"])))
            if model == "pRotatE" and "modulus" in state:
                m.modulus.copy_(torch.from_numpy(np.asarray(state["modulus"])))
    return m.cuda()


def score_err(model, got, want, gamma):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    if model in DIST:
        return float(np.max(np.abs(got - want)) / max(np.max(np.abs(gamma - want)), 1e-30))
    return relinf(got, want)


def ns(**kw):
    base = dict(cuda=True, negative_adversarial_sampling=False, adversarial_temperature=1.0, uni_weight=False,
                regularization=0.0, countries=False, regions=None, test_batch_size=4, cpu_num=2,
                test_log_steps=100000, nentity=0, nrelation=0)
    base.update(kw)
    return types.SimpleNamespace(**base)


def golden_state(g, prefix="init_"):
    st = {"entity_embedding": g[prefix + "entity_embedding"], "relation_embedding": g[prefix + "relation_embedding"]}
    if prefix + "modulus" in g.files:
        st["modulus"] = g[prefix + "modulus"]
    return st


# ------------------------------------------------------------------------------------------------ forward / autograd
@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("d", [12, 10])
def test_forward_and_autograd_vs_reference_golden(model, d):
    g = np.load(os.path.join(GOLDEN, f"small_{model}_d{d}.npz"))
    gamma = float(g["gamma"])
    m = make_model(model, int(g["nentity"]), int(g["nrelation"]), d, gamma, golden_state(g))
    pos, neg = torch.from_numpy(g["positive"]), torch.from_numpy(g["negative"])
    cot = torch.from_numpy(g["cotangent"]).cuda()
    for mode in O.MODES:
        m.zero_grad()
        s = m(pos) if mode == "single" else m((pos, neg), mode)
        assert s.shape == g["score_" + mode].shape and s.dtype == torch.float32
        assert score_err(model, s.detach().cpu().numpy(), g["score_" + mode], gamma) < TOL, (model, mode)
        (s * cot[:, :s.shape[1]]).sum().backward()
        assert relinf(m.entity_embedding.grad.cpu().numpy(), g["dE_" + mode]) < TOL, (model, mode)
        assert relinf(m.relation_embedding.grad.cpu().numpy(), g["dR_" + mode]) < TOL, (model, mode)
        if model == "pRotatE":
            assert relinf(m.modulus.grad.cpu().numpy(), g["dM_" + mode]) < TOL


@pytest.mark.parametrize("model", MODELS)
def test_public_score_methods(model):
    """KGEModel.TransE/.../pRotatE(head, relation, tail, mode) on gathered rows == forward() (model.py:166-249)."""
    g = np.load(os.path.join(GOLDEN, f"small_{model}_d12.npz"))
    gamma = float(g["gamma"])
    m = make_model(model, int(g["nentity"]), int(g["nrelation"]), 12, gamma, golden_state(g))
    pos, neg = torch.from_numpy(g["positive"]).cuda(), torch.from_numpy(g["negative"]).cuda()
    E, R = m.entity_embedding.detach(), m.relation_embedding.detach()
    fn = getattr(m, model)
    for mode in ("head-batch", "tail-batch"):
        if mode == "head-batch":
            head, tail = E[neg.view(-1)].view(neg.shape[0], neg.shape[1], -1), E[pos[:, 2]].unsqueeze(1)
        else:
            head, tail = E[pos[:, 0]].unsqueeze(1), E[neg.view(-1)].view(neg.shape[0], neg.shape[1], -1)
        s = fn(head, R[pos[:, 1]].unsqueeze(1), tail, mode)
        assert score_err(model, s.detach().cpu().numpy(), g["score_" + mode], gamma) < TOL
    s = fn(E[pos[:, 0]].unsqueeze(1), R[pos[:, 1]].unsqueeze(1), E[pos[:, 2]].unsqueeze(1), "single")
    assert score_err(model, s.detach().cpu().numpy(), g["score_single"], gamma) < TOL


# ------------------------------------------------------------------------------------------------ train_step
CFGS = {
    "adv_sub": dict(negative_adversarial_sampling=True, adversarial_temperature=0.7, uni_weight=False),
    "adv_uni": dict(negative_adversarial_sampling=True, adversarial_temperature=1.0, uni_weight=True),
    "mean_sub": dict(negative_adversarial_sampling=False, uni_weight=False),
    "adv_sub_reg": dict(negative_adversarial_sampling=True, adversarial_temperature=1.0, uni_weight=False,
                        regularization=1e-3),
}


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("d", [12, 10])
@pytest.mark.parametrize("cfg", list(CFGS))
@pytest.mark.parametrize("path", ["default", "single_read", "two_sweep"])
def test_train_steps_vs_reference_golden(model, d, cfg, path, monkeypatch):
    """4 train_steps with the run.py call sequence (incl. the Adam re-creation of run.py:315-322) through
      default      what train_step picks: the single-read path with the entity table's Adam update fused into the
                   entity pass when rows are 16-byte multiples (no entity gradient is materialised: .grad stays None),
      single_read  the single-read (split + entity-major) path with dense gradients + kge_adam_step,
      two_sweep    the two-sweep atomic kernel + kge_adam_step."""
    monkeypatch.delenv("KGE_KEEP_GRADS", raising=False)
    if path == "single_read":
        monkeypatch.setenv("KGE_FORCE_SPLIT", "1")
        monkeypatch.setenv("KGE_KEEP_GRADS", "1")
    elif path == "two_sweep":
        monkeypatch.setenv("KGE_NO_SPLIT", "1")
    g = np.load(os.path.join(GOLDEN, f"small_{model}_d{d}.npz"))
    m = make_model(model, int(g["nentity"]), int(g["nrelation"]), d, float(g["gamma"]), golden_state(g))
    lr = 1e-3
    opt = torch.optim.Adam(filter(lambda p: p.requires_grad, m.parameters()), lr=lr)
    batches = [(torch.from_numpy(g[f"train_{cfg}_pos{i}"]), torch.from_numpy(g[f"train_{cfg}_neg{i}"]),
                torch.from_numpy(g[f"train_{cfg}_w{i}"]), "tail-batch" if i % 2 == 0 else "head-batch")
               for i in range(4)]
    it = iter(batches)
    args = ns(**CFGS[cfg])
    for step in range(4):
        if step == 2:
            lr /= 10
            opt = torch.optim.Adam(filter(lambda p: p.requires_grad, m.parameters()), lr=lr)
        log = KGE().train_step(m, opt, it, args)
        ref = g[f"train_{cfg}_logs"][step]
        keys = (["regularization"] if "reg" in cfg else []) + ["positive_sample_loss", "negative_sample_loss", "loss"]
        assert list(log.keys()) == keys and all(isinstance(v, float) for v in log.values())
        got = [log.get("regularization", 0.0), log["positive_sample_loss"], log["negative_sample_loss"], log["loss"]]
        np.testing.assert_allclose(got, ref, rtol=TOL, atol=1e-7)
        if step == 0:
            if m.entity_embedding.grad is None:       # fused entity optimizer (needs rows that are 16-byte multiples)
                assert path != "single_read" and d % 4 == 0
            else:
                assert path in ("single_read", "two_sweep") or d % 4 != 0
                assert relinf(m.entity_embedding.grad.cpu().numpy(), g[f"train_{cfg}_gE0"]) < TOL
            assert relinf(m.relation_embedding.grad.cpu().numpy(), g[f"train_{cfg}_gR0"]) < TOL
            if model == "pRotatE":
                assert relinf(m.modulus.grad.cpu().numpy(), g[f"train_{cfg}_gM0"]) < TOL
    assert relinf(m.entity_embedding.detach().cpu().numpy(), g[f"train_{cfg}_E"]) < TOL
    assert relinf(m.relation_embedding.detach().cpu().numpy(), g[f"train_{cfg}_R"]) < TOL
    if model == "pRotatE":
        assert relinf(m.modulus.detach().cpu().numpy(), g[f"train_{cfg}_M"]) < TOL
    # the optimizer state is torch's own layout: it round-trips through a stock Adam (run.py:106,283)
    sd = opt.state_dict()
    assert [float(sd["state"][k]["step"]) for k in sorted(sd["state"])] == list(g[f"train_{cfg}_adam_steps"])
    torch.optim.Adam(filter(lambda p: p.requires_grad, m.parameters()), lr=lr).load_state_dict(sd)


@pytest.mark.parametrize("path", ["default", "single_read"])
def test_train_step_matches_autograd_path_full_width(path, monkeypatch):
    if path == "single_read":
        monkeypatch.setenv("KGE_FORCE_SPLIT", "1")
    monkeypatch.setenv("KGE_KEEP_GRADS", "1")
    _full_width_case()


def _full_width_case():
    """cfg-3 row shape (RotatE, d=1000, N=256, 14,951 entities): fused train grads vs (a) the numpy oracle,
    (b) forward() + torch loss + the autograd backward kernel."""
    import torch.nn.functional as F
    nentity, nrel, d, gamma, B, N = 14951, 1345, 1000, 24.0, 48, 256
    st = O.init_tables("RotatE", nentity, nrel, d, gamma, True, False, seed=0)
    rng = np.random.RandomState(1)
    pos = np.stack([rng.randint(nentity, size=B), rng.randint(nrel, size=B), rng.randint(nentity, size=B)], 1)
    neg = rng.randint(nentity, size=(B, N))
    w = np.sqrt(1.0 / rng.randint(8, 200, size=B)).astype(np.float32)
    for mode in ("tail-batch", "head-batch"):
        m = make_model("RotatE", nentity, nrel, d, gamma, st)
        opt = torch.optim.Adam(m.parameters(), lr=1e-4)
        args = ns(negative_adversarial_sampling=True, adversarial_temperature=1.0)
        log = KGE().train_step(m, opt, iter([(torch.from_numpy(pos), torch.from_numpy(neg), torch.from_numpy(w), mode)]), args)
        gE, gR = m.entity_embedding.grad.cpu().numpy(), m.relation_embedding.grad.cpu().numpy()
        # (a) numpy oracle
        ts = O.TrainState("RotatE", st, gamma, d)
        olog, og = O.train_step(ts, (pos, neg, w, mode), lr=1e-4, adversarial=True, alpha=1.0, return_grads=True)
        for k in ("positive_sample_loss", "negative_sample_loss", "loss"):
            assert abs(log[k] - olog[k]) <= TOL * abs(olog[k])
        assert relinf(gE, og["entity_embedding"]) < TOL and relinf(gR, og["relation_embedding"]) < TOL
        assert outlier_fraction(m.entity_embedding.detach().cpu().numpy(), ts.state["entity_embedding"]) < 1e-4
        # (b) the differentiable forward() path of the same library
        m2 = make_model("RotatE", nentity, nrel, d, gamma, st)
        tp, tn, tw = torch.from_numpy(pos).cuda(), torch.from_numpy(neg).cuda(), torch.from_numpy(w).cuda()
        sneg = m2((tp, tn), mode)
        nl = (F.softmax(sneg, dim=1).detach() * F.logsigmoid(-sneg)).sum(dim=1)
        pl = F.logsigmoid(m2(tp)).squeeze(1)
        loss = (-(tw * pl).sum() / tw.sum() - (tw * nl).sum() / tw.sum()) / 2
        loss.backward()
        assert abs(loss.item() - log["loss"]) <= TOL * abs(log["loss"])
        assert relinf(m2.entity_embedding.grad.cpu().numpy(), gE) < TOL
        assert relinf(m2.relation_embedding.grad.cpu().numpy(), gR) < TOL


def test_adam_kernel_vs_torch_adam(monkeypatch):
    """kge_adam_step == torch.optim.Adam (foreach CUDA path) over 5 steps of random gradients."""
    monkeypatch.setenv("KGE_KEEP_GRADS", "1")           # the dense gradients feed the stock optimizer below
    torch.manual_seed(0)
    m = make_model("TransE", 5000, 11, 36, 9.0)
    ref = [p.detach().clone().requires_grad_(True) for p in (m.entity_embedding, m.relation_embedding)]
    ropt = torch.optim.Adam(ref, lr=3e-4)
    opt = torch.optim.Adam(m.parameters(), lr=3e-4)
    args = ns(negative_adversarial_sampling=True)
    B, N = 64, 32
    for step in range(5):
        pos = torch.stack([torch.randint(5000, (B,)), torch.randint(11, (B,)), torch.randint(5000, (B,))], 1)
        neg = torch.randint(5000, (B, N))
        w = torch.rand(B) + 0.1
        KGE().train_step(m, opt, iter([(pos, neg, w, "tail-batch" if step % 2 == 0 else "head-batch")]), args)
        for r, p in zip(ref, (m.entity_embedding, m.relation_embedding)):
            r.grad = p.grad.detach().clone()          # same gradients into stock Adam
        ropt.step()
        for r, p in zip(ref, (m.entity_embedding, m.relation_embedding)):
            assert relinf(p.detach().cpu().numpy(), r.detach().cpu().numpy()) < 1e-6
    for r, p in zip(ref, (m.entity_embedding, m.relation_embedding)):
        for key in ("exp_avg", "exp_avg_sq"):
            assert relinf(opt.state[p][key].cpu().numpy(), ropt.state[r][key].cpu().numpy()) < 1e-6


# ------------------------------------------------------------------------------------------------ filtered ranking
def as_triples(a):
    return [tuple(int(v) for v in row) for row in a]


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("d", [12, 10])
def test_filtered_ranks_vs_reference_golden(model, d):
    g = np.load(os.path.join(GOLDEN, f"small_{model}_d{d}.npz"))
    gamma, nentity = float(g["gamma"]), int(g["nentity"])
    st = {"entity_embedding": g["eval_E"], "relation_embedding": g["eval_R"]}
    if model == "pRotatE":
        st["modulus"] = g["init_modulus"]
    m = make_model(model, nentity, int(g["nrelation"]), d, gamma, st)
    test, all_true = as_triples(g["eval_test"]), as_triples(g["eval_all_true"])
    rows, ranks = [], []
    for mode in ("head-batch", "tail-batch"):
        r, s = m.filtered_ranks(test, all_true, mode, return_scores=True)
        s = s.cpu().numpy()
        # identical score matrix => identical ranks: the reference procedure (argsort) on OUR matrix
        pos_col = [t[0] if mode == "head-batch" else t[2] for t in test]
        np.testing.assert_array_equal(r, [O.rank_from_scores(row, p) for row, p in zip(s, pos_col)])
        # bit-exact against the C oracle (same IEEE op sequence)
        from knowledgegraphembedding_b200 import FilterIndex
        off, ent = FilterIndex(all_true, nentity, int(g["nrelation"])).csr(test, mode)
        cs = C.eval_scores(model, st, test, mode, gamma, O.embedding_range(gamma, d), off, ent)
        np.testing.assert_array_equal(s.view(np.uint32), cs.view(np.uint32))
        rows.append(s)
        ranks.append(r)
    assert score_err(model, np.concatenate(rows), g["eval_scores"], gamma) < TOL
    np.testing.assert_array_equal(np.concatenate(ranks), g["eval_ranks"])        # ranks bit-exact vs the reference
    metrics = KGE().test_step(m, test, all_true, ns(nentity=nentity, nrelation=int(g["nrelation"])))
    assert list(metrics.keys()) == ["MRR", "MR", "HITS@1", "HITS@3", "HITS@10"]
    np.testing.assert_allclose([metrics[k] for k in metrics], g["eval_metrics"], rtol=0, atol=1e-12)


def test_countries_s1_end_to_end():
    """Real dataset, reference-sampled batches: 4 train steps, AUC-PR (model.py:322-344) and filtered ranks."""
    g = load_golden("countries_S1")
    d, gamma, nentity, nrel = int(g["d"]), float(g["gamma"]), int(g["nentity"]), int(g["nrelation"])
    from test_oracle_golden import countries_init
    assert (d, g["pos0"].shape[0], g["neg0"].shape[1]) == (500, 512, 64)     # BASELINE configs[0] at its stated shape
    m = make_model("RotatE", nentity, nrel, d, gamma, countries_init(g))
    opt = torch.optim.Adam(filter(lambda p: p.requires_grad, m.parameters()), lr=float(g["lr"]))
    regions = [int(r) for r in g["regions"]]
    args = ns(negative_adversarial_sampling=True, countries=True, regions=regions, nentity=nentity, nrelation=nrel)
    for step in range(4):
        batch = (torch.from_numpy(g[f"pos{step}"].astype(np.int64)), torch.from_numpy(g[f"neg{step}"].astype(np.int64)),
                 torch.from_numpy(g[f"w{step}"]), "tail-batch" if step % 2 == 0 else "head-batch")
        log = KGE().train_step(m, opt, iter([batch]), args)
        np.testing.assert_allclose([log["positive_sample_loss"], log["negative_sample_loss"], log["loss"]],
                                   g["logs"][step], rtol=TOL)
    E = m.entity_embedding.detach().cpu().numpy()
    assert outlier_fraction(E, g["final_E"], TOL) < 1e-3
    assert relinf(m.relation_embedding.detach().cpu().numpy(), g["final_R"]) < TOL
    test = as_triples(g["test"])
    all_true = as_triples(np.concatenate([g["train"], g["valid"], g["test"]]))
    with torch.no_grad():
        m.entity_embedding.copy_(torch.from_numpy(g["final_E"]))
        m.relation_embedding.copy_(torch.from_numpy(g["final_R"]))
    auc = KGE().test_step(m, test, all_true, args)["auc_pr"]
    assert abs(auc - float(g["auc_pr"])) < 1e-6
    args.countries = False
    metrics = KGE().test_step(m, test, all_true, args)
    ranks = np.concatenate([m.filtered_ranks(test, all_true, mode) for mode in ("head-batch", "tail-batch")])
    np.testing.assert_array_equal(ranks, g["ranks"])
    np.testing.assert_allclose([metrics[k] for k in ("MRR", "MR", "HITS@1", "HITS@3", "HITS@10")], g["metrics"],
                               rtol=0, atol=1e-12)


def test_wn18rr_real_dataset_ranks():
    """wn18rr (40,943 entities, full train+valid+test filter): ranks vs the reference's and vs the C oracle."""
    g = np.load(os.path.join(GOLDEN, "wn18rr_eval.npz"))
    d, gamma, nentity, nrel = int(g["d"]), float(g["gamma"]), int(g["nentity"]), int(g["nrelation"])
    st = O.init_tables("RotatE", nentity, nrel, d, gamma, True, False, seed=int(g["seed"]))
    st["entity_embedding"] = (st["entity_embedding"] * float(g["scale"])).astype(np.float32)
    assert float(st["entity_embedding"].astype(np.float64).sum()) == float(g["table_checksum"])
    m = make_model("RotatE", nentity, nrel, d, gamma, st)
    test, all_true = as_triples(g["test"]), as_triples(g["all_true"])
    from knowledgegraphembedding_b200 import FilterIndex
    index = FilterIndex(all_true, nentity, nrel)
    got = []
    for mode in ("head-batch", "tail-batch"):
        r = m.filtered_ranks(test, all_true, mode)
        off, ent = index.csr(test, mode)
        cs = C.eval_scores("RotatE", st, test, mode, gamma, O.embedding_range(gamma, d), off, ent)
        np.testing.assert_array_equal(r, C.ranks_from_scores(cs, test, mode))           # bit-exact vs the oracle
        got.append(r)
    got = np.concatenate(got)
    want = g["ranks"]
    # vs the torch reference: libm sin/cos and reduction order differ, so a rank may move across a near tie only
    assert np.max(np.abs(got - want)) <= 2 and np.mean(got != want) < 0.02
    metrics = KGE().test_step(m, test, all_true, ns(nentity=nentity, nrelation=nrel))
    np.testing.assert_allclose([metrics[k] for k in ("MRR", "MR", "HITS@1", "HITS@3", "HITS@10")], g["metrics"], rtol=2e-4)


FULL = [("TransE", 14541, 237, 1000, 9.0), ("RotatE", 14951, 1345, 1000, 24.0), ("ComplEx", 40943, 11, 500, 200.0),
        ("RotatE", 123182, 37, 500, 24.0), ("pRotatE", 14951, 1345, 1000, 24.0), ("DistMult", 14951, 1345, 2000, 500.0)]


@pytest.mark.parametrize("model,nentity,nrel,d,gamma", FULL)
def test_full_size_eval_bit_exact_vs_c_oracle(model, nentity, nrel, d, gamma):
    """BASELINE.json config shapes: all-entity scores (+filter bias) and ranks of a query sample are bit-identical
    to the C oracle; ranks also equal the argsort procedure on the same matrix."""
    de, dr = FLAGS[model]
    st = O.init_tables(model, nentity, nrel, d, gamma, de, dr, seed=0)
    st["entity_embedding"] = (st["entity_embedding"] * 3.0).astype(np.float32)
    rng = np.random.RandomState(2)
    all_true = sorted({(int(rng.randint(nentity)), int(rng.randint(nrel)), int(rng.randint(200))) for _ in range(30000)})
    test = [all_true[i] for i in rng.choice(len(all_true), 24, replace=False)]
    m = make_model(model, nentity, nrel, d, gamma, st)
    from knowledgegraphembedding_b200 import FilterIndex
    index = FilterIndex(all_true, nentity, nrel)
    rho = O.embedding_range(gamma, d)
    for mode in ("head-batch", "tail-batch"):
        r, s = m.filtered_ranks(test, all_true, mode, return_scores=True)
        s = s.cpu().numpy()
        off, ent = index.csr(test, mode)
        cs = C.eval_scores(model, st, test, mode, gamma, rho, off, ent)
        np.testing.assert_array_equal(s.view(np.uint32), cs.view(np.uint32))
        np.testing.assert_array_equal(r, C.ranks_from_scores(cs, test, mode))
        pos_col = [t[0] if mode == "head-batch" else t[2] for t in test]
        np.testing.assert_array_equal(r[:6], [O.rank_from_scores(row, p) for row, p in zip(s[:6], pos_col[:6])])


def test_entity_sharded_counts_sum_to_full():
    """The multi-GPU eval path: counts over disjoint entity slices add up to the single-GPU ranks (bit-exact)."""
    import ctypes
    from knowledgegraphembedding_b200 import _lib, FilterIndex, shard_bounds
    from knowledgegraphembedding_b200.model import _ptr, _stream
    model, nentity, nrel, d, gamma = "RotatE", 5003, 17, 64, 12.0
    st = O.init_tables(model, nentity, nrel, d, gamma, True, False, seed=4)
    m = make_model(model, nentity, nrel, d, gamma, st)
    rng = np.random.RandomState(0)
    all_true = sorted({(int(rng.randint(nentity)), int(rng.randint(nrel)), int(rng.randint(50))) for _ in range(4000)})
    test = all_true[:100]
    for mode in ("head-batch", "tail-batch"):
        full = m.filtered_ranks(test, all_true, mode)
        dev = m.entity_embedding.device
        q = torch.tensor(test, dtype=torch.int64, device=dev)
        off, ent = FilterIndex(all_true, nentity, nrel).csr(test, mode)
        d_off, d_ent = torch.from_numpy(off).to(dev), torch.from_numpy(ent).to(dev)
        words = (nentity + 31) // 32
        bits = torch.zeros(len(test) * words, dtype=torch.int32, device=dev)
        qvec = torch.empty(len(test) * m.entity_dim, device=dev)
        pos = torch.empty(len(test), device=dev)
        desc, mid, stt = m._descriptor(), _lib.MODE_IDS[mode], _stream(dev)
        _lib.call("kge_eval_filter_bits", _ptr(d_off), _ptr(d_ent), len(test), nentity, _ptr(bits), stt)
        _lib.call("kge_eval_query_vectors", ctypes.byref(desc), mid, _ptr(q), len(test), _ptr(qvec), None, stt)
        _lib.call("kge_eval_positive_scores", ctypes.byref(desc), mid, _ptr(qvec), _ptr(q), len(test), None, _ptr(pos), stt)
        total = torch.zeros(len(test), dtype=torch.int32, device=dev)
        for rank in range(8):
            b, e = shard_bounds(nentity, rank, 8)
            part = torch.zeros(len(test), dtype=torch.int32, device=dev)
            _lib.call("kge_eval_count_ranks", ctypes.byref(desc), mid, _ptr(qvec), _ptr(q), len(test), None, _ptr(pos),
                      _ptr(bits), b, e, _ptr(part), None, stt)
            total += part
        np.testing.assert_array_equal(total.cpu().numpy() + 1, full)


def test_device_filter_lookup_equals_host_csr_bitmap():
    """kge_eval_filter_bits_lookup (index resident on the device) sets exactly the bits of the host CSR path, which is
    pinned to dataloader.py:134-154 by the CPU tests; includes queries whose key has no true triple and empty indexes."""
    from knowledgegraphembedding_b200 import _lib, FilterIndex
    from knowledgegraphembedding_b200.model import _ptr, _stream
    dev = torch.device("cuda", 0)
    rng = np.random.RandomState(5)
    for nentity, nrel, ntrue, nq in ((5003, 17, 6000, 700), (33, 2, 40, 50), (100, 3, 0, 10)):
        all_true = sorted({(int(rng.randint(nentity)), int(rng.randint(nrel)), int(rng.randint(min(nentity, 60))))
                           for _ in range(ntrue)})
        test = [(int(rng.randint(nentity)), int(rng.randint(nrel)), int(rng.randint(min(nentity, 70)))) for _ in range(nq)]
        test += all_true[:nq]
        index = FilterIndex(all_true, nentity, nrel)
        q = torch.tensor(test, dtype=torch.int64, device=dev)
        words = (nentity + 31) // 32
        for mode in ("head-batch", "tail-batch"):
            off, ent = index.csr(test, mode)
            d_off = torch.from_numpy(off).to(dev)
            d_ent = torch.from_numpy(ent).to(dev) if ent.size else torch.zeros(1, dtype=torch.int32, device=dev)
            want = torch.full((len(test) * words,), -1, dtype=torch.int32, device=dev)
            got = torch.full((len(test) * words,), -1, dtype=torch.int32, device=dev)
            _lib.call("kge_eval_filter_bits", _ptr(d_off), _ptr(d_ent), len(test), nentity, _ptr(want), _stream(dev))
            keys, offsets, values = index.table(mode)
            d_keys = torch.from_numpy(np.ascontiguousarray(keys)).to(dev)
            d_offsets = torch.from_numpy(np.ascontiguousarray(offsets)).to(dev)
            d_values = torch.from_numpy(np.ascontiguousarray(values)).to(dev) if values.size else d_ent
            _lib.call("kge_eval_filter_bits_lookup", _ptr(d_keys) if keys.size else None,
                      _ptr(d_offsets) if keys.size else None, _ptr(d_values) if keys.size else None, int(keys.size),
                      _ptr(q), len(test), _lib.MODE_IDS[mode], nentity, nrel, _ptr(got), _stream(dev))
            assert torch.equal(got, want), (nentity, mode)
            if ntrue:
                assert int((want != 0).sum()) > 0
            # the index built ON the device (counting sort into a direct-address CSR) holds the same runs as the host's
            # sorted-key index, and its lookup sets the same bits
            lib = _lib.load()
            tri = torch.tensor(all_true, dtype=torch.int64, device=dev).reshape(-1, 3)
            d_off32 = torch.full((nentity * nrel + 1,), -7, dtype=torch.int32, device=dev)
            d_ent32 = torch.zeros(max(len(all_true), 1), dtype=torch.int32, device=dev)
            sbytes = int(lib.kge_eval_filter_index_scratch_bytes(nentity, nrel))
            scratch = torch.empty(sbytes, dtype=torch.uint8, device=dev)
            flag = torch.zeros(1, dtype=torch.int32, device=dev)
            _lib.call("kge_eval_filter_index_build", _ptr(tri) if len(all_true) else None, len(all_true),
                      _lib.MODE_IDS[mode], nentity, nrel, _ptr(d_off32), _ptr(d_ent32), _ptr(scratch), sbytes, _ptr(flag),
                      _stream(dev))
            dense = torch.full((len(test) * words,), -1, dtype=torch.int32, device=dev)
            _lib.call("kge_eval_filter_bits_lookup_dense", _ptr(d_off32), _ptr(d_ent32), _ptr(q), len(test),
                      _lib.MODE_IDS[mode], nentity, nrel, _ptr(dense), _stream(dev))
            assert torch.equal(dense, want), (nentity, mode, "device-built index")
            assert int(flag.item()) == 0
            off32, ent32 = d_off32.cpu().numpy(), d_ent32.cpu().numpy()
            assert off32[0] == 0 and off32[-1] == len(all_true) and np.all(np.diff(off32) >= 0)
            for k, lo, hi in zip(keys.tolist(), offsets[:-1].tolist(), offsets[1:].tolist()):
                assert sorted(ent32[off32[k]:off32[k + 1]].tolist()) == sorted(values[lo:hi].tolist())
            assert int(np.count_nonzero(np.diff(off32))) == keys.size       # no run outside the host index's keys


# ------------------------------------------------------------------------------------------------ API behaviour
def test_api_errors_and_state_dict():
    K = KGE()
    with pytest.raises(ValueError, match="model Foo not supported"):
        K("Foo", 10, 2, 4, 1.0)
    with pytest.raises(ValueError, match="RotatE should use --double_entity_embedding"):
        K("RotatE", 10, 2, 4, 1.0)
    with pytest.raises(ValueError, match="ComplEx should use"):
        K("ComplEx", 10, 2, 4, 1.0, double_entity_embedding=True)
    m = K("pRotatE", 10, 2, 4, 6.0).cuda()
    assert list(m.state_dict().keys()) == ["gamma", "embedding_range", "entity_embedding", "relation_embedding", "modulus"]
    assert [n for n, p in m.named_parameters() if p.requires_grad] == ["entity_embedding", "relation_embedding", "modulus"]
    with pytest.raises(ValueError, match="mode sideways not supported"):
        m((torch.zeros(2, 3, dtype=torch.long), torch.zeros(2, 4, dtype=torch.long)), "sideways")
    m2 = K("pRotatE", 10, 2, 4, 6.0)
    m2.load_state_dict({k: v.cpu() for k, v in m.state_dict().items()})
    m2 = m2.cuda()
    s = torch.tensor([[1, 0, 2], [3, 1, 4]])
    assert torch.equal(m(s), m2(s))
    with pytest.raises(IndexError):
        m(torch.tensor([[1, 0, 10]]))          # entity id == nentity
        m._raise_if_bad_index()
    cpu = K("TransE", 10, 2, 4, 6.0)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        cpu(s)


def test_ragged_last_batch_and_non_adam_optimizer():
    """The last batch of an epoch is smaller than -b (run.py:246-260 has no drop_last); any optimizer object works."""
    torch.manual_seed(1)
    m = make_model("RotatE", 300, 5, 20, 6.0)
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    args = ns(negative_adversarial_sampling=True)
    for B in (16, 5, 1):
        pos = torch.stack([torch.randint(300, (B,)), torch.randint(5, (B,)), torch.randint(300, (B,))], 1)
        log = KGE().train_step(m, opt, iter([(pos, torch.randint(300, (B, 7)), torch.rand(B) + 0.1, "head-batch")]), args)
        assert np.isfinite(log["loss"])
    before = m.entity_embedding.detach().clone()
    sgd = torch.optim.SGD(m.parameters(), lr=0.1)
    pos = torch.stack([torch.randint(300, (8,)), torch.randint(5, (8,)), torch.randint(300, (8,))], 1)
    KGE().train_step(m, sgd, iter([(pos, torch.randint(300, (8, 7)), torch.rand(8) + 0.1, "tail-batch")]), args)
    torch.testing.assert_close(m.entity_embedding.detach(), before - 0.1 * m.entity_embedding.grad)


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("mode", ["head-batch", "tail-batch"])
def test_single_read_path_matches_two_sweep_kernel(model, mode, monkeypatch):
    """The single-read path (row_kernel_split + entity_kernel) against the two-sweep atomic kernel and the numpy
    oracle on a medium shape, adversarial and uniform losses."""
    nentity, nrel, d, gamma, B, N = 3000, 7, 128, 6.0, 37, 50
    de, dr = FLAGS[model]
    monkeypatch.setenv("KGE_KEEP_GRADS", "1")
    st = O.init_tables(model, nentity, nrel, d, gamma, de, dr, seed=5)
    rng = np.random.RandomState(6)
    pos = np.stack([rng.randint(nentity, size=B), rng.randint(nrel, size=B), rng.randint(nentity, size=B)], 1)
    neg = rng.randint(60, size=(B, N))                  # few distinct candidates => long entity segments
    w = np.sqrt(1.0 / rng.randint(8, 200, size=B)).astype(np.float32)
    for adv in (True, False):
        args = ns(negative_adversarial_sampling=adv, adversarial_temperature=0.5)
        out = {}
        for tag in ("split", "two_sweep"):
            if tag == "two_sweep":
                monkeypatch.setenv("KGE_NO_SPLIT", "1")
                monkeypatch.delenv("KGE_FORCE_SPLIT", raising=False)
            else:
                monkeypatch.delenv("KGE_NO_SPLIT", raising=False)
                monkeypatch.setenv("KGE_FORCE_SPLIT", "1")
            m = make_model(model, nentity, nrel, d, gamma, st)
            opt = torch.optim.Adam(filter(lambda p: p.requires_grad, m.parameters()), lr=1e-4)
            log = KGE().train_step(m, opt, iter([(torch.from_numpy(pos), torch.from_numpy(neg), torch.from_numpy(w), mode)]), args)
            out[tag] = (log, m.entity_embedding.grad.cpu().numpy().copy(), m.relation_embedding.grad.cpu().numpy().copy(),
                        m.modulus.grad.cpu().numpy().copy() if model == "pRotatE" else None)
        monkeypatch.delenv("KGE_NO_SPLIT", raising=False)
        monkeypatch.delenv("KGE_FORCE_SPLIT", raising=False)
        ts = O.TrainState(model, st, gamma, d)
        olog, og = O.train_step(ts, (pos, neg, w, mode), lr=1e-4, adversarial=adv, alpha=0.5, return_grads=True)
        for tag in out:
            log, gE, gR, gM = out[tag]
            assert abs(log["loss"] - olog["loss"]) <= TOL * abs(olog["loss"]), tag
            assert relinf(gE, og["entity_embedding"]) < TOL, (tag, adv)
            assert relinf(gR, og["relation_embedding"]) < TOL, (tag, adv)
            if gM is not None:
                assert relinf(gM, og["modulus"]) < TOL, (tag, adv)


@pytest.mark.parametrize("model,nentity,nrel,d,gamma,nq", [
    ("ComplEx", 40943, 11, 500, 200.0, 300),        # wn18rr shape (BASELINE.json configs[3]); K = 1000 is not a multiple of 32
    ("DistMult", 14951, 1345, 2000, 500.0, 200),    # FB15k shape of best_config.sh
    ("ComplEx", 517, 5, 12, 20.0, 130),             # tiles mostly out of bounds, Q and nentity not multiples of 128
    ("DistMult", 4099, 3, 36, 20.0, 129),
])
def test_tcgen05_eval_ranks_identical_to_exact_kernel(model, nentity, nrel, d, gamma, nq, monkeypatch):
    """DistMult/ComplEx all-entity scoring on the tcgen05 path (3xTF32 + exact re-score of the ambiguous band) gives
    the same integer ranks as the exact SIMT tile kernel, which is bit-exact against the C oracle."""
    de, dr = FLAGS[model]
    st = O.init_tables(model, nentity, nrel, d, gamma, de, dr, seed=3)
    st["entity_embedding"] = (st["entity_embedding"] * 5.0).astype(np.float32)
    rng = np.random.RandomState(4)
    all_true = sorted({(int(rng.randint(nentity)), int(rng.randint(nrel)), int(rng.randint(min(nentity, 300))))
                       for _ in range(20000)})
    test = [all_true[i] for i in rng.choice(len(all_true), nq, replace=False)]
    m = make_model(model, nentity, nrel, d, gamma, st)
    for mode in ("head-batch", "tail-batch"):
        monkeypatch.setenv("KGE_EVAL_SIMT", "1")
        exact = m.filtered_ranks(test, all_true, mode)
        monkeypatch.delenv("KGE_EVAL_SIMT")
        m._ws.pop('gemm_last_ambiguous', None)
        fast = m.filtered_ranks(test, all_true, mode)
        assert 'gemm_last_ambiguous' in m._ws, "tcgen05 path was not taken"
        np.testing.assert_array_equal(fast, exact)
        # the band is narrow: only a small fraction of the Q x nentity pairs needs the exact re-score
        assert m._ws['gemm_last_ambiguous'] < 0.05 * nq * nentity + 64


def test_batch_sharded_rows_sum_to_full_batch(monkeypatch):
    monkeypatch.setenv("KGE_FORCE_SPLIT", "1")
    _sharded_rows_case()


def _sharded_rows_case():
    """The multi-GPU train path: every rank runs kge_train_rows on its row slice with the global weight sum; the
    gradient buffers and per-row losses add up to the single-GPU result (what the NCCL all-reduce then delivers)."""
    import ctypes
    from knowledgegraphembedding_b200 import _lib, shard_bounds
    from knowledgegraphembedding_b200.model import _ptr, _stream
    nentity, nrel, d, gamma, B, N = 4000, 9, 64, 9.0, 50, 40
    st = O.init_tables("RotatE", nentity, nrel, d, gamma, True, False, seed=8)
    m = make_model("RotatE", nentity, nrel, d, gamma, st)
    dev = m.entity_embedding.device
    rng = np.random.RandomState(9)
    pos = torch.from_numpy(np.stack([rng.randint(nentity, size=B), rng.randint(nrel, size=B), rng.randint(nentity, size=B)], 1)).to(dev)
    neg = torch.from_numpy(rng.randint(nentity, size=(B, N))).to(dev)
    w = torch.from_numpy(np.sqrt(1.0 / rng.randint(8, 200, size=B)).astype(np.float32)).to(dev)
    wsum = w.sum().reshape(1)
    desc, stt = m._descriptor(), _stream(dev)

    def run(world):
        gE, gR = torch.zeros_like(m.entity_embedding), torch.zeros_like(m.relation_embedding)
        rows = torch.zeros(2, B, device=dev)
        for rank in range(world):
            b, e = shard_bounds(B, rank, world)
            nb = _lib.load().kge_train_workspace_bytes(ctypes.byref(desc), e - b, N)
            wsp = torch.empty(nb, dtype=torch.uint8, device=dev)
            _lib.call("kge_train_rows", ctypes.byref(desc), _lib.HEAD_BATCH, _lib.LOSS_NEG_ADVERSARIAL, 1.0, _ptr(pos),
                      _ptr(neg), _ptr(w), _ptr(wsum), B, b, e - b, N, _ptr(rows[0]), _ptr(rows[1]), _ptr(gE), _ptr(gR),
                      None, None, _ptr(wsp), nb, None, stt)
        torch.cuda.synchronize()
        return gE.cpu().numpy(), gR.cpu().numpy(), rows.cpu().numpy()

    full = run(1)
    for world in (2, 3, 8):
        part = run(world)
        assert relinf(part[0], full[0]) < 1e-6 and relinf(part[1], full[1]) < 1e-6
        np.testing.assert_allclose(part[2], full[2], rtol=1e-6)


@pytest.mark.parametrize("nentity,nrel,d,gamma,nq,scale", [
    (14951, 1345, 1000, 24.0, 160, 1.0),      # FB15k shape at random init: scores nearly tied (worst case for the band)
    (14951, 1345, 1000, 24.0, 160, 4.0),
    (123182, 37, 500, 24.0, 48, 2.0),         # YAGO3-10 shape
    (1031, 5, 36, 6.0, 200, 3.0),
])
def test_two_stage_rotate_eval_ranks_identical_to_exact_kernel(nentity, nrel, d, gamma, nq, scale, monkeypatch):
    """RotatE filtered ranking through the fast tile pass + exact re-score of the undecidable band gives the same
    integer ranks as the exact kernel (which is bit-exact against the C oracle)."""
    st = O.init_tables("RotatE", nentity, nrel, d, gamma, True, False, seed=12)
    st["entity_embedding"] = (st["entity_embedding"] * scale).astype(np.float32)
    rng = np.random.RandomState(13)
    all_true = sorted({(int(rng.randint(nentity)), int(rng.randint(nrel)), int(rng.randint(min(nentity, 400))))
                       for _ in range(20000)})
    test = [all_true[i] for i in rng.choice(len(all_true), nq, replace=False)]
    m = make_model("RotatE", nentity, nrel, d, gamma, st)
    for mode in ("head-batch", "tail-batch"):
        monkeypatch.setenv("KGE_EVAL_SIMT", "1")
        exact = m.filtered_ranks(test, all_true, mode)
        monkeypatch.delenv("KGE_EVAL_SIMT")
        m._ws.pop('two_stage_last_ambiguous', None)
        fast = m.filtered_ranks(test, all_true, mode)
        assert 'two_stage_last_ambiguous' in m._ws, "two-stage path was not taken"
        np.testing.assert_array_equal(fast, exact)
        assert m._ws['two_stage_last_ambiguous'] < 0.02 * nq * nentity + 64


@pytest.mark.parametrize("nentity,nrel,d,gamma,nq,scale", [
    (14951, 1345, 1000, 24.0, 160, 1.0),      # FB15k shape at random init
    (14951, 1345, 1000, 24.0, 96, 5.0),       # phases up to +-5 pi: the reduction by pi runs over several periods
    (1031, 5, 36, 6.0, 200, 3.0),
    (1031, 5, 36, 6.0, 64, 3.0e4),            # absurd phases (|t| up to 1e5): the fast pass answers NaN -> exact re-score
])
def test_two_stage_protate_eval_ranks_identical_to_exact_kernel(nentity, nrel, d, gamma, nq, scale, monkeypatch):
    """pRotatE filtered ranking through the fast tile pass (reduction by pi + sin.approx) + exact re-score of the
    undecidable band gives the same integer ranks as the exact kernel (bit-exact against the C oracle)."""
    st = O.init_tables("pRotatE", nentity, nrel, d, gamma, False, False, seed=12)
    st["entity_embedding"] = (st["entity_embedding"] * scale).astype(np.float32)
    rng = np.random.RandomState(13)
    all_true = sorted({(int(rng.randint(nentity)), int(rng.randint(nrel)), int(rng.randint(min(nentity, 400))))
                       for _ in range(20000)})
    test = [all_true[i] for i in rng.choice(len(all_true), nq, replace=False)]
    m = make_model("pRotatE", nentity, nrel, d, gamma, st)
    if scale > 1e3:
        monkeypatch.setenv("KGE_EVAL_AMB_CAP", str(nq * nentity + 64))     # every pair may be undecidable here
    for mode in ("head-batch", "tail-batch"):
        monkeypatch.setenv("KGE_EVAL_SIMT", "1")
        exact = m.filtered_ranks(test, all_true, mode)
        monkeypatch.delenv("KGE_EVAL_SIMT")
        m._ws.pop('two_stage_last_ambiguous', None)
        fast = m.filtered_ranks(test, all_true, mode)
        assert 'two_stage_last_ambiguous' in m._ws, "two-stage path was not taken"
        np.testing.assert_array_equal(fast, exact)
        if scale <= 1e3:
            assert m._ws['two_stage_last_ambiguous'] < 0.02 * nq * nentity + 64


def test_pinned_negatives_are_read_in_place(monkeypatch):
    """KGE_ZERO_COPY=1 with a pinned host batch: the candidate ids are not staged on the device, the single-read row
    kernel reads them from host memory through its prefetched windows and leaves the int32 copy for the counting sort.
    Same losses and tables as the (default) staged copy and as a pageable batch; includes an id window that ends in the
    middle (N = 40)."""
    torch.manual_seed(1)
    nentity, nrel, d, gamma, B, N = 700, 5, 32, 9.0, 200, 40
    st = O.init_tables("RotatE", nentity, nrel, d, gamma, True, False, seed=5)
    args = ns(negative_adversarial_sampling=True)
    batches = []
    for i in range(3):
        pos = torch.stack([torch.randint(nentity, (B,)), torch.randint(nrel, (B,)), torch.randint(nentity, (B,))], 1)
        batches.append((pos, torch.randint(nentity, (B, N)), torch.rand(B) + 0.1, "tail-batch" if i % 2 == 0 else "head-batch"))
    out = {}
    for tag in ("pinned", "staged", "pageable"):
        if tag == "pinned":
            monkeypatch.setenv("KGE_ZERO_COPY", "1")
        else:
            monkeypatch.delenv("KGE_ZERO_COPY", raising=False)
        m = make_model("RotatE", nentity, nrel, d, gamma, st)
        opt = torch.optim.Adam(filter(lambda p: p.requires_grad, m.parameters()), lr=1e-3)
        feed = [(p.pin_memory(), n.pin_memory(), w.pin_memory(), md) if tag != "pageable" else (p, n, w, md)
                for p, n, w, md in batches]
        logs = [KGE().train_step(m, opt, iter([b]), args) for b in feed]
        assert ('stage_neg' in m._ws) == (tag != "pinned"), tag          # zero-copy: no device staging buffer for the ids
        out[tag] = (logs, m.entity_embedding.detach().cpu().numpy().copy())
    for tag in ("staged", "pageable"):
        for a, b in zip(out["pinned"][0], out[tag][0]):
            assert all(abs(a[k] - b[k]) <= 1e-6 * abs(b[k]) for k in b), (tag, a, b)
        assert outlier_fraction(out["pinned"][1], out[tag][1]) < 1e-4, tag
    # an out-of-range id in a pinned batch is flagged like in a staged one
    m = make_model("RotatE", nentity, nrel, d, gamma, st)
    opt = torch.optim.Adam(filter(lambda p: p.requires_grad, m.parameters()), lr=1e-3)
    bad = batches[0][1].clone()
    bad[7, 33] = nentity + 5
    monkeypatch.setenv("KGE_ZERO_COPY", "1")
    with pytest.raises(IndexError):
        KGE().train_step(m, opt, iter([(batches[0][0].pin_memory(), bad.pin_memory(), batches[0][2].pin_memory(), "tail-batch")]), args)


def test_train_step_pulls_exactly_one_batch_per_call():
    """The reference's iterator contract (model.py:261): one next(train_iterator) per train_step, at the call; a finite
    iterator of K batches yields exactly K steps and raises StopIteration at call K+1; two iterators used alternately
    (e.g. separate head / tail loaders) lose no batch."""
    torch.manual_seed(0)
    st = O.init_tables("RotatE", 500, 5, 16, 6.0, True, False, seed=2)
    args = ns(negative_adversarial_sampling=True)
    batches = []
    for i in range(3):
        pos = torch.stack([torch.randint(500, (32,)), torch.randint(5, (32,)), torch.randint(500, (32,))], 1)
        batches.append((pos.pin_memory(), torch.randint(500, (32, 16)).pin_memory(), (torch.rand(32) + 0.1).pin_memory(),
                        "tail-batch" if i % 2 == 0 else "head-batch"))

    class Counting:
        def __init__(self, items):
            self.items, self.pulled = list(items), 0

        def __iter__(self):
            return self

        def __next__(self):
            if self.pulled >= len(self.items):
                raise StopIteration
            self.pulled += 1
            return self.items[self.pulled - 1]

    m = make_model("RotatE", 500, 5, 16, 6.0, st)
    opt = torch.optim.Adam(filter(lambda p: p.requires_grad, m.parameters()), lr=1e-3)
    it = Counting(batches)
    for k in range(3):
        KGE().train_step(m, opt, it, args)
        assert it.pulled == k + 1
    with pytest.raises(StopIteration):
        KGE().train_step(m, opt, it, args)
    a, b = Counting(batches[:2]), Counting(batches[1:])
    m2 = make_model("RotatE", 500, 5, 16, 6.0, st)
    opt2 = torch.optim.Adam(filter(lambda p: p.requires_grad, m2.parameters()), lr=1e-3)
    seq = [KGE().train_step(m2, opt2, x, args)["loss"] for x in (a, b, a, b)]
    ref2 = make_model("RotatE", 500, 5, 16, 6.0, st)
    opt3 = torch.optim.Adam(filter(lambda p: p.requires_grad, ref2.parameters()), lr=1e-3)
    want = [KGE().train_step(ref2, opt3, iter([x]), args)["loss"] for x in (batches[0], batches[1], batches[1], batches[2])]
    np.testing.assert_allclose(seq, want, rtol=1e-6)
    assert a.pulled == 2 and b.pulled == 2


@pytest.mark.parametrize("model,reg", [("RotatE", 0.0), ("ComplEx", 1e-3), ("pRotatE", 0.0), ("TransE", 0.0),
                                       ("DistMult", 1e-3)])
def test_fused_entity_optimizer_matches_dense_adam(model, reg, monkeypatch):
    """kge_train_rows_adam (Adam for the entity table inside the entity-major pass, no dense entity gradient) against
    the same step with dense gradients + kge_adam_step (KGE_KEEP_GRADS=1): losses, tables and moments over 3 steps;
    entities that no pair touches are still updated (dense Adam semantics); with -r the L3 term is included."""
    nentity, nrel, d, gamma, B, N = 3001, 7, 64, 6.0, 64, 300
    de, dr = FLAGS[model]
    st = O.init_tables(model, nentity, nrel, d, gamma, de, dr, seed=5)
    rng = np.random.RandomState(6)
    batches = []
    for i in range(3):
        pos = np.stack([rng.randint(nentity, size=B), rng.randint(nrel, size=B), rng.randint(nentity, size=B)], 1)
        batches.append((torch.from_numpy(pos), torch.from_numpy(rng.randint(nentity // 2, size=(B, N))),
                        torch.from_numpy(np.sqrt(1.0 / rng.randint(8, 200, size=B)).astype(np.float32)),
                        "tail-batch" if i % 2 == 0 else "head-batch"))
    args = ns(negative_adversarial_sampling=True, regularization=reg)
    out = {}
    for tag in ("dense", "fused"):
        if tag == "dense":
            monkeypatch.setenv("KGE_KEEP_GRADS", "1")
        else:
            monkeypatch.delenv("KGE_KEEP_GRADS")
        m = make_model(model, nentity, nrel, d, gamma, st)
        opt = torch.optim.Adam(filter(lambda p: p.requires_grad, m.parameters()), lr=1e-3)
        it = iter(batches)
        logs = [KGE().train_step(m, opt, it, args) for _ in range(3)]
        assert (m.entity_embedding.grad is None) == (tag == "fused"), "fused entity optimizer was (not) taken"
        mom = opt.state[m.entity_embedding]
        out[tag] = (logs, m.entity_embedding.detach().cpu().numpy().copy(), m.relation_embedding.detach().cpu().numpy().copy(),
                    mom["exp_avg"].cpu().numpy().copy(), mom["exp_avg_sq"].cpu().numpy().copy(), float(mom["step"]))
    for a, b in zip(out["dense"][0], out["fused"][0]):
        assert list(a) == list(b) and all(abs(a[k] - b[k]) <= 1e-6 * abs(a[k]) for k in a)
    # three free-running steps: the kinked models (|x|, |sin x|) amplify summation-order noise between the two paths
    # from the second step on (tests/test_gpu_fullshape.py::sync_state explains); the smooth ones stay at 1e-5
    mtol = 1e-5 if model in ("RotatE", "ComplEx", "DistMult") else 2e-3
    assert outlier_fraction(out["fused"][1], out["dense"][1]) < 1e-4 and relinf(out["fused"][2], out["dense"][2]) < max(mtol, 1e-5)
    assert relinf(out["fused"][3], out["dense"][3]) < mtol and relinf(out["fused"][4], out["dense"][4]) < mtol
    assert out["fused"][5] == out["dense"][5] == 3.0
    # the upper half of the entity ids never appears as a negative: those rows still move (m decays, v stays 0 ...)
    untouched = np.setdiff1d(np.arange(nentity // 2, nentity), np.concatenate([b[0][:, [0, 2]].numpy().ravel() for b in batches]))
    assert untouched.size > 100
    if reg == 0.0:          # zero gradient, zero moments: the row must not move at all
        np.testing.assert_array_equal(out["fused"][1][untouched], out["dense"][1][untouched])
        np.testing.assert_array_equal(out["fused"][1][untouched], st["entity_embedding"][untouched])
    else:                   # the L3 gradient moves every row; the fused update uses MUFU rcp / sqrt (within 2^-22 of the step)
        np.testing.assert_allclose(out["fused"][1][untouched], out["dense"][1][untouched], rtol=2e-6, atol=0)
        assert np.abs(out["fused"][1][untouched] - st["entity_embedding"][untouched]).max() > 0


def test_bad_index_leaves_model_and_optimizer_untouched():
    """An out-of-range id raises IndexError like the reference's index_select -- and, as there, before any state
    changed: the optimizer kernels see the error flag and skip the update, the step counters are rolled back."""
    for B, N, nentity in ((64, 300, 3001), (8, 16, 500)):          # single-read (fused optimizer) and two-sweep paths
        st = O.init_tables("RotatE", nentity, 7, 64, 6.0, True, False, seed=5)
        m = make_model("RotatE", nentity, 7, 64, 6.0, st)
        opt = torch.optim.Adam(filter(lambda p: p.requires_grad, m.parameters()), lr=1e-3)
        args = ns(negative_adversarial_sampling=True)
        rng = np.random.RandomState(1)

        def batch(bad):
            pos = np.stack([rng.randint(nentity, size=B), rng.randint(7, size=B), rng.randint(nentity, size=B)], 1)
            neg = rng.randint(nentity, size=(B, N))
            if bad:
                neg[B // 2, N // 2] = nentity
            return (torch.from_numpy(pos), torch.from_numpy(neg), torch.rand(B) + 0.1, "tail-batch")

        KGE().train_step(m, opt, iter([batch(False)]), args)
        before = (m.entity_embedding.detach().clone(), m.relation_embedding.detach().clone(),
                  opt.state[m.entity_embedding]["exp_avg"].clone(), float(opt.state[m.entity_embedding]["step"]))
        with pytest.raises(IndexError):
            KGE().train_step(m, opt, iter([batch(True)]), args)
        assert torch.equal(m.entity_embedding.detach(), before[0]) and torch.equal(m.relation_embedding.detach(), before[1])
        assert torch.equal(opt.state[m.entity_embedding]["exp_avg"], before[2])
        assert float(opt.state[m.entity_embedding]["step"]) == before[3] == 1.0
        log = KGE().train_step(m, opt, iter([batch(False)]), args)     # and the model keeps training afterwards
        assert np.isfinite(log["loss"]) and float(opt.state[m.entity_embedding]["step"]) == 2.0


@pytest.mark.parametrize("model", ["RotatE", "ComplEx"])
def test_two_stage_overflow_falls_back_to_exact(model, monkeypatch):
    """A full ambiguous-pair list (capacity forced to 2) is detected at the call's single sync and the chunk is
    re-ranked by the exact kernel: same ranks."""
    de, dr = FLAGS[model]
    nentity, nrel, d, gamma = 2500, 5, 32, 6.0
    st = O.init_tables(model, nentity, nrel, d, gamma, de, dr, seed=21)
    rng = np.random.RandomState(22)
    all_true = sorted({(int(rng.randint(nentity)), int(rng.randint(nrel)), int(rng.randint(200))) for _ in range(5000)})
    test = all_true[:150]
    m = make_model(model, nentity, nrel, d, gamma, st)
    monkeypatch.setenv("KGE_EVAL_SIMT", "1")
    exact = m.filtered_ranks(test, all_true, "tail-batch", query_chunk=64)
    monkeypatch.delenv("KGE_EVAL_SIMT")
    monkeypatch.setenv("KGE_EVAL_AMB_CAP", "2")
    np.testing.assert_array_equal(m.filtered_ranks(test, all_true, "tail-batch", query_chunk=64), exact)
    monkeypatch.delenv("KGE_EVAL_AMB_CAP")
    np.testing.assert_array_equal(m.filtered_ranks(test, all_true, "tail-batch", query_chunk=64), exact)
