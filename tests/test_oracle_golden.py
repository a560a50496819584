"""Pin the CPU oracle (oracle/kge_oracle.py) against vectors produced by the unmodified reference
(tests/golden/make_golden.py).  CPU only."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, load_golden, outlier_fraction, relinf
from oracle import kge_oracle as O

MODELS = ["TransE", "DistMult", "ComplEx", "RotatE", "pRotatE"]
DS = [12, 10]
TOL = 1e-5          # north_star: scores, loss and updated embeddings within 1e-5 relative (fp32)


def load(model, d):
    return np.load(os.path.join(GOLDEN, f"small_{model}_d{d}.npz"))


def state_of(g, prefix="init_"):
    st = {"entity_embedding": g[prefix + "entity_embedding"], "relation_embedding": g[prefix + "relation_embedding"]}
    if prefix + "modulus" in g.files:
        st["modulus"] = g[prefix + "modulus"]
    return st


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("d", DS)
def test_forward_scores(model, d):
    g = load(model, d)
    st = state_of(g)
    for mode in O.MODES:
        sample = g["positive"] if mode == "single" else (g["positive"], g["negative"])
        s = O.forward(model, st, sample, mode, float(g["gamma"]), d)
        assert s.shape == g["score_" + mode].shape
        assert relinf(s, g["score_" + mode]) < TOL, (model, mode)


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("d", DS)
def test_score_backward(model, d):
    g = load(model, d)
    st = state_of(g)
    for mode in O.MODES:
        sample = g["positive"] if mode == "single" else (g["positive"], g["negative"])
        cot = g["cotangent"][:, :1] if mode == "single" else g["cotangent"]
        grads = O.score_backward(model, st, sample, mode, cot, float(g["gamma"]), d)
        assert relinf(grads["entity_embedding"], g["dE_" + mode]) < TOL, (model, mode)
        assert relinf(grads["relation_embedding"], g["dR_" + mode]) < TOL, (model, mode)
        if model == "pRotatE":
            assert relinf(grads["modulus"], g["dM_" + mode]) < TOL


CFGS = {
    "adv_sub": dict(adversarial=True, alpha=0.7, uni_weight=False),
    "adv_uni": dict(adversarial=True, alpha=1.0, uni_weight=True),
    "mean_sub": dict(adversarial=False, uni_weight=False),
    "adv_sub_reg": dict(adversarial=True, alpha=1.0, uni_weight=False, regularization=1e-3),
}


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("d", DS)
@pytest.mark.parametrize("cfg", list(CFGS))
def test_train_steps(model, d, cfg):
    g = load(model, d)
    ts = O.TrainState(model, state_of(g), float(g["gamma"]), d)
    lr = 1e-3
    for step in range(4):
        if step == 2:                       # run.py:315-322
            lr /= 10
            ts.reset_optimizer()
        batch = (g[f"train_{cfg}_pos{step}"], g[f"train_{cfg}_neg{step}"], g[f"train_{cfg}_w{step}"],
                 "tail-batch" if step % 2 == 0 else "head-batch")
        log, grads = O.train_step(ts, batch, lr=lr, return_grads=True, **CFGS[cfg])
        ref = g[f"train_{cfg}_logs"][step]
        got = [log.get("regularization", 0.0), log["positive_sample_loss"], log["negative_sample_loss"], log["loss"]]
        np.testing.assert_allclose(got, ref, rtol=TOL, atol=1e-7)
        if step == 0:
            assert relinf(grads["entity_embedding"], g[f"train_{cfg}_gE0"]) < TOL
            assert relinf(grads["relation_embedding"], g[f"train_{cfg}_gR0"]) < TOL
            if model == "pRotatE":
                assert relinf(grads["modulus"], g[f"train_{cfg}_gM0"]) < TOL
    assert relinf(ts.state["entity_embedding"], g[f"train_{cfg}_E"]) < TOL
    assert relinf(ts.state["relation_embedding"], g[f"train_{cfg}_R"]) < TOL
    if model == "pRotatE":
        assert relinf(ts.state["modulus"], g[f"train_{cfg}_M"]) < TOL
    # Adam was re-created before step 2, so each parameter saw 2 steps since (run.py:318-321)
    assert all(st["step"] == s for st, s in zip(ts.adam.values(), g[f"train_{cfg}_adam_steps"]))


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("d", DS)
def test_filtered_ranks(model, d):
    g = load(model, d)
    st = {"entity_embedding": g["eval_E"], "relation_embedding": g["eval_R"]}
    if model == "pRotatE":
        st["modulus"] = g["init_modulus"]
    test = [tuple(int(v) for v in row) for row in g["eval_test"]]
    all_true = [tuple(int(v) for v in row) for row in g["eval_all_true"]]
    ranks, scores = O.filtered_ranks(model, st, test, all_true, int(g["nentity"]), float(g["gamma"]), d,
                                     return_scores=True)
    assert relinf(scores, g["eval_scores"]) < TOL
    np.testing.assert_array_equal(ranks, g["eval_ranks"])          # bit-exact ranks
    m = O.metrics_from_ranks(ranks)
    np.testing.assert_allclose([m[k] for k in ("MRR", "MR", "HITS@1", "HITS@3", "HITS@10")], g["eval_metrics"],
                               rtol=0, atol=1e-12)
    # the rank procedure itself, on the reference's own score rows (identical matrix => identical ranks)
    pos_col = [t[0] for t in test] + [t[2] for t in test]
    again = [O.rank_from_scores(row, p) for row, p in zip(g["eval_scores"], pos_col)]
    np.testing.assert_array_equal(again, g["eval_ranks"])


def countries_init(g):
    """The initial tables of the countries golden: the portable numpy initialiser, checksummed against the file."""
    st = O.init_tables("RotatE", int(g["nentity"]), int(g["nrelation"]), int(g["d"]), float(g["gamma"]), True, False,
                       seed=int(g["init_seed"]))
    assert float(st["entity_embedding"].astype(np.float64).sum()) == float(g["init_checksum"])
    return st


def fullwidth_batches(nentity, nrelation, B, N, steps, seed):
    """Same seeded batches as tests/golden/make_golden.py:fullwidth_batches."""
    rng = np.random.RandomState(seed)
    out = []
    for step in range(steps):
        pos = np.stack([rng.randint(nentity, size=B), rng.randint(nrelation, size=B), rng.randint(nentity, size=B)], 1)
        neg = rng.randint(nentity, size=(B, N))
        w = np.sqrt(1.0 / rng.randint(8, 200, size=B)).astype(np.float32)
        out.append((pos.astype(np.int64), neg.astype(np.int64), w, "tail-batch" if step % 2 == 0 else "head-batch"))
    return out


def check_fullwidth_step(g, step, log, gE, gR):
    """One step of the full-width golden (reference outputs): losses, per-row / per-column sums of |grad| and the
    sampled gradient rows, all within TOL."""
    np.testing.assert_allclose([log["positive_sample_loss"], log["negative_sample_loss"], log["loss"]],
                               g["logs"][step], rtol=TOL)
    gE64, gR64 = np.abs(np.asarray(gE, np.float64)), np.abs(np.asarray(gR, np.float64))
    assert relinf(gE64.sum(1), g[f"gE{step}_abs_rowsum"]) < TOL, step
    assert relinf(gE64.sum(0), g[f"gE{step}_abs_colsum"]) < TOL, step
    assert relinf(gR64.sum(1), g[f"gR{step}_abs_rowsum"]) < TOL, step
    if step == 0:
        assert relinf(np.asarray(gE)[g["ent_rows"]], g["gE0_rows"]) < TOL
        assert relinf(np.asarray(gR)[g["rel_rows"]], g["gR0_rows"]) < TOL


def check_fullwidth_final(g, E, R):
    lr = float(g["lr"])
    Er, Rr = np.asarray(E)[g["ent_rows"]], np.asarray(R)[g["rel_rows"]]
    assert outlier_fraction(Er, g["final_E_rows"], TOL) < 1e-3 and outlier_fraction(Rr, g["final_R_rows"], TOL) < 1e-3
    assert np.max(np.abs(Er - g["final_E_rows"])) <= 3 * 2 * lr and np.max(np.abs(Rr - g["final_R_rows"])) <= 3 * 2 * lr


def test_fullwidth_reference_golden_pins_both_oracles():
    """BASELINE configs[2] row shape (14,951 x 2000 table, N=256, 192 rows, 3 steps) produced by the unmodified
    reference: pins the C oracle -- the full-size checker of the GPU tests and bench.py's CPU port -- at full width,
    and the numpy oracle on the first step."""
    from oracle import c_oracle as C
    g = load_golden("fullwidth_RotatE_fb15k")
    nentity, nrel, d, gamma = int(g["nentity"]), int(g["nrelation"]), int(g["d"]), float(g["gamma"])
    st = O.init_tables("RotatE", nentity, nrel, d, gamma, True, False, seed=int(g["init_seed"]))
    assert float(st["entity_embedding"].astype(np.float64).sum()) == float(g["init_checksum"])
    batches = fullwidth_batches(nentity, nrel, int(g["B"]), int(g["N"]), 3, int(g["batch_seed"]))
    ts = C.TrainState("RotatE", st, gamma, d)
    for step, b in enumerate(batches):
        log, grads = C.train_step(ts, b, lr=float(g["lr"]), adversarial=True, alpha=1.0, return_grads=True)
        check_fullwidth_step(g, step, log, grads["entity_embedding"], grads["relation_embedding"])
    check_fullwidth_final(g, ts.state["entity_embedding"], ts.state["relation_embedding"])
    tn = O.TrainState("RotatE", st, gamma, d)
    log, grads = O.train_step(tn, batches[0], lr=float(g["lr"]), adversarial=True, alpha=1.0, return_grads=True)
    check_fullwidth_step(g, 0, log, grads["entity_embedding"], grads["relation_embedding"])


def test_countries_s1_real_dataset():
    g = load_golden("countries_S1")
    d, gamma = int(g["d"]), float(g["gamma"])
    lr = float(g["lr"])
    ts = O.TrainState("RotatE", countries_init(g), gamma, d)
    assert [g[f"pos{i}"].shape[0] for i in range(4)] == [512, 512, 87, 512]      # stated -b 512, ragged third batch
    for step in range(4):
        batch = (g[f"pos{step}"].astype(np.int64), g[f"neg{step}"].astype(np.int64), g[f"w{step}"],
                 "tail-batch" if step % 2 == 0 else "head-batch")
        log = O.train_step(ts, batch, lr=lr, adversarial=True, alpha=1.0)
        np.testing.assert_allclose([log["positive_sample_loss"], log["negative_sample_loss"], log["loss"]],
                                   g["logs"][step], rtol=TOL)
    # 4 Adam steps: elements whose gradient cancels to rounding noise may move by up to lr*2 per step
    assert outlier_fraction(ts.state["entity_embedding"], g["final_E"], TOL) < 1e-3
    assert relinf(ts.state["entity_embedding"], g["final_E"]) < 4 * 2 * lr / np.abs(g["final_E"]).max()
    assert relinf(ts.state["relation_embedding"], g["final_R"]) < TOL
    test = [tuple(int(v) for v in r) for r in g["test"]]
    sample, y_true = O.countries_samples(test, [int(r) for r in g["regions"]])
    np.testing.assert_array_equal(y_true, g["y_true"])
    final = {"entity_embedding": g["final_E"], "relation_embedding": g["final_R"]}
    y = O.forward("RotatE", final, sample, "single", gamma, d)[:, 0]
    assert relinf(y, g["y_score"]) < TOL
    assert abs(O.average_precision(y_true, g["y_score"]) - float(g["auc_pr"])) < 1e-12
    all_true = [tuple(int(v) for v in r) for r in np.concatenate([g["train"], g["valid"], g["test"]])]
    ranks = O.filtered_ranks("RotatE", final, test, all_true, int(g["nentity"]), gamma, d)
    np.testing.assert_array_equal(ranks, g["ranks"])


def test_wn18rr_real_dataset_ranks():
    g = np.load(os.path.join(GOLDEN, "wn18rr_eval.npz"))
    d, gamma, nentity = int(g["d"]), float(g["gamma"]), int(g["nentity"])
    st = O.init_tables("RotatE", nentity, int(g["nrelation"]), d, gamma, True, False, seed=int(g["seed"]))
    st["entity_embedding"] = (st["entity_embedding"] * float(g["scale"])).astype(np.float32)
    assert float(st["entity_embedding"].astype(np.float64).sum()) == float(g["table_checksum"])
    test = [tuple(int(v) for v in r) for r in g["test"][:60]]
    all_true = [tuple(int(v) for v in r) for r in g["all_true"]]
    nq = len(g["test"])
    ranks = O.filtered_ranks("RotatE", st, test, all_true, nentity, gamma, d)
    want = np.concatenate([g["ranks"][:60], g["ranks"][nq:nq + 60]])
    # numpy and torch differ in libm sin/cos and reduction order: a rank may move only across a near tie
    assert np.max(np.abs(ranks - want)) <= 1 and np.mean(ranks != want) < 0.05
