"""Train-path parity AT THE BENCHMARKED SHAPES (BASELINE.json configs 1-5), through the kernel variant the launcher
picks by default -- the persistent multi-row `row_kernel_split` + counting sort + `entity_kernel` + Adam at B=1024 --
against
  * the unmodified reference's outputs at full width (tests/golden/fullwidth_RotatE_fb15k.npz: 14,951 x 2000 table,
    N=256, 192 rows, 3 steps; countries_S1.npz at -b 512 -d 500 -n 64), and
  * the C oracle (oracle/kge_oracle.c, pinned to those goldens by tests/test_oracle_golden.py) at the full batch.
Tolerance (north_star): losses and updated tables within 1e-5 relative (fp32); full-batch gradients see GRAD_TOL."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, load_golden, outlier_fraction, relinf
from oracle import c_oracle as C
from oracle import kge_oracle as O
from test_gpu_parity import FLAGS, KGE, make_model, ns
from test_oracle_golden import check_fullwidth_final, check_fullwidth_step, fullwidth_batches

pytestmark = pytest.mark.gpu
TOL = 1e-5
# Gradients of a full batch: dL/ds_ij carries the softmax weight exp(alpha * s_ij) / Z, so an absolute score error
# delta moves every weight -- and every gradient contribution -- by alpha * delta RELATIVE.  Scores are gamma - distance
# with distance ~ 25-30 at these shapes: two correct fp32 evaluations of the same 1000-term sum already differ by a few
# ulp(32) = 4e-6 each (the north-star score tolerance, 1e-5 relative to the distance, would allow 3e-4).  Measured on
# B200 against the C oracle: 1.3e-5 at cfg 3.  Losses and updated tables keep the plain 1e-5.
GRAD_TOL = 5e-5


def tbatch(b):
    return (torch.from_numpy(b[0]), torch.from_numpy(b[1]), torch.from_numpy(b[2]), b[3])


@pytest.mark.parametrize("path", ["default", "single_read"])
def test_fullwidth_steps_vs_reference_golden(path, monkeypatch):
    """cfg-3 row shape against the REFERENCE's own outputs.  192 rows x 256 negatives is below the launcher's
    pairs-per-entity threshold, so "default" is the two-sweep TMA kernel; "single_read" forces the split path, whose
    persistent CTAs then walk 1-2 rows each (192 > 148 SMs, not a multiple)."""
    if path == "single_read":
        monkeypatch.setenv("KGE_FORCE_SPLIT", "1")
    monkeypatch.setenv("KGE_KEEP_GRADS", "1")
    g = load_golden("fullwidth_RotatE_fb15k")
    nentity, nrel, d, gamma = int(g["nentity"]), int(g["nrelation"]), int(g["d"]), float(g["gamma"])
    st = O.init_tables("RotatE", nentity, nrel, d, gamma, True, False, seed=int(g["init_seed"]))
    m = make_model("RotatE", nentity, nrel, d, gamma, st)
    opt = torch.optim.Adam(filter(lambda p: p.requires_grad, m.parameters()), lr=float(g["lr"]))
    args = ns(negative_adversarial_sampling=True, adversarial_temperature=1.0)
    batches = fullwidth_batches(nentity, nrel, int(g["B"]), int(g["N"]), 3, int(g["batch_seed"]))
    for step, b in enumerate(batches):
        log = KGE().train_step(m, opt, iter([tbatch(b)]), args)
        check_fullwidth_step(g, step, log, m.entity_embedding.grad.cpu().numpy(), m.relation_embedding.grad.cpu().numpy())
    check_fullwidth_final(g, m.entity_embedding.detach().cpu().numpy(), m.relation_embedding.detach().cpu().numpy())


# (id, model, nentity, nrelation, d, gamma, B, N, lr, regularization, steps)
SHAPES = [
    ("cfg3_rotate_fb15k", "RotatE", 14951, 1345, 1000, 24.0, 1024, 256, 1e-4, 0.0, 3),      # the bench.py workload
    ("cfg3_rows_not_multiple", "RotatE", 14951, 1345, 1000, 24.0, 777, 256, 1e-4, 0.0, 2),   # 777 = 5 * 148 + 37 rows
    ("cfg2_transe_fb15k237", "TransE", 14541, 237, 1000, 9.0, 1024, 256, 5e-5, 0.0, 2),
    ("cfg4_complex_wn18rr_reg", "ComplEx", 40943, 11, 500, 200.0, 512, 1024, 2e-3, 5e-6, 2),
    ("cfg5_rotate_yago310", "RotatE", 123182, 37, 500, 24.0, 1024, 400, 2e-4, 0.0, 2),
    ("protate_fb15k", "pRotatE", 14951, 1345, 1000, 24.0, 1024, 256, 1e-4, 0.0, 2),
    ("distmult_fb15k_reg", "DistMult", 14951, 1345, 2000, 500.0, 1024, 256, 1e-3, 2e-6, 2),
]


def sync_state(m, opt, ts, model):
    """Copy the oracle's tables and Adam moments into the model / optimizer: the next step then starts from identical
    inputs on both sides.  (Comparing free-running trajectories is ill-conditioned: |x| and |sin x| have kinks, and
    Adam's first steps are sign-like, so ulp-level differences in the tables change single gradient elements by O(1) --
    measured on the CPU oracle alone: ulp noise in the tables moves the next step's gradient by 2e-2 (pRotatE),
    4e-3 (TransE), 7e-5 (RotatE) in the infinity norm.)"""
    names = [("entity_embedding", m.entity_embedding), ("relation_embedding", m.relation_embedding)]
    if model == "pRotatE":
        names.append(("modulus", m.modulus))
    with torch.no_grad():
        for name, p in names:
            p.copy_(torch.from_numpy(ts.state[name]))
            opt.state[p]["exp_avg"].copy_(torch.from_numpy(ts.m[name]))
            opt.state[p]["exp_avg_sq"].copy_(torch.from_numpy(ts.v[name]))


@pytest.mark.parametrize("keep_grads", [True, False], ids=["grads", "fused_optimizer"])
@pytest.mark.parametrize("case", SHAPES, ids=[s[0] for s in SHAPES])
def test_full_batch_train_steps_vs_c_oracle(case, keep_grads, monkeypatch):
    """Full batches of every BASELINE config through KGEModel.train_step with the launcher's default kernel choice,
    alternating tail/head steps, against the C oracle's full-batch steps on the same inputs: losses, (with
    KGE_KEEP_GRADS=1) the dense gradients, the updated tables and the Adam moments of every step.  After each step the
    oracle's state is copied into the model (sync_state), so every step is compared from identical inputs."""
    _, model, nentity, nrel, d, gamma, B, N, lr, reg, steps = case
    if keep_grads:
        monkeypatch.setenv("KGE_KEEP_GRADS", "1")       # materialise p.grad (the fused entity-pass optimizer does not)
    else:
        monkeypatch.delenv("KGE_KEEP_GRADS", raising=False)
    de, dr = FLAGS[model]
    st = O.init_tables(model, nentity, nrel, d, gamma, de, dr, seed=0)
    m = make_model(model, nentity, nrel, d, gamma, st)
    opt = torch.optim.Adam(filter(lambda p: p.requires_grad, m.parameters()), lr=lr)
    args = ns(negative_adversarial_sampling=True, adversarial_temperature=1.0, regularization=reg)
    ts = C.TrainState(model, st, gamma, d)
    batches = fullwidth_batches(nentity, nrel, B, N, steps, seed=1)
    params = [("entity_embedding", m.entity_embedding), ("relation_embedding", m.relation_embedding)]
    for step, b in enumerate(batches):
        log = KGE().train_step(m, opt, iter([tbatch(b)]), args)
        ref, grads = C.train_step(ts, b, lr=lr, adversarial=True, alpha=1.0, regularization=reg, return_grads=True)
        assert list(log) == list(ref)
        for k in ref:
            assert abs(log[k] - ref[k]) <= TOL * abs(ref[k]), (step, k, log[k], ref[k])
        assert (m.entity_embedding.grad is None) == (not keep_grads), "fused entity optimizer was (not) taken"
        if keep_grads:
            assert relinf(m.entity_embedding.grad.cpu().numpy(), grads["entity_embedding"]) < GRAD_TOL, step
        assert relinf(m.relation_embedding.grad.cpu().numpy(), grads["relation_embedding"]) < GRAD_TOL, step
        if model == "pRotatE":
            assert relinf(m.modulus.grad.cpu().numpy(), grads["modulus"]) < GRAD_TOL, step
            assert relinf(m.modulus.detach().cpu().numpy(), ts.state["modulus"]) < TOL
        # updated tables: all but a vanishing fraction within 1e-5, nothing beyond the Adam step bound (an element
        # whose gradient cancels to rounding noise may take the other sign of lr in the first steps)
        for name, p in params:
            got, want = p.detach().cpu().numpy(), ts.state[name]
            assert outlier_fraction(got, want, TOL) < 1e-4, (step, name)
            assert np.max(np.abs(got - want)) <= 2.0 * lr + TOL * np.abs(want).max(), (step, name)
            mom = opt.state[p]
            assert float(mom["step"]) == step + 1
            assert relinf(mom["exp_avg"].cpu().numpy(), ts.m[name]) < GRAD_TOL, (step, name)
            assert relinf(mom["exp_avg_sq"].cpu().numpy(), ts.v[name]) < 2 * GRAD_TOL, (step, name)
        sync_state(m, opt, ts, model)


def test_wn18rr_rank_differences_are_near_ties():
    """SURVEY section 7 hard part 1b: where our filtered rank differs from the torch reference's on wn18rr, the
    candidates that flipped sides are within a few ulp of the positive score -- i.e. the difference is a libm /
    reduction-order near-tie, never a wrong comparison.  For every differing query: the number of candidates whose
    score lies within 4 ulp(|distance|) of s_pos bounds |our rank - reference rank|."""
    g = np.load(os.path.join(GOLDEN, "wn18rr_eval.npz"))
    d, gamma, nentity, nrel = int(g["d"]), float(g["gamma"]), int(g["nentity"]), int(g["nrelation"])
    st = O.init_tables("RotatE", nentity, nrel, d, gamma, True, False, seed=int(g["seed"]))
    st["entity_embedding"] = (st["entity_embedding"] * float(g["scale"])).astype(np.float32)
    m = make_model("RotatE", nentity, nrel, d, gamma, st)
    test = [tuple(int(v) for v in r) for r in g["test"]]
    all_true = [tuple(int(v) for v in r) for r in g["all_true"]]
    nq, want = len(test), g["ranks"]
    differing = 0
    for mi, mode in enumerate(("head-batch", "tail-batch")):
        r, s = m.filtered_ranks(test, all_true, mode, return_scores=True)
        s = s.cpu().numpy()
        ref = want[mi * nq:(mi + 1) * nq]
        for i in np.nonzero(r != ref)[0]:
            differing += 1
            pos = test[i][0] if mode == "head-batch" else test[i][2]
            sp = s[i, pos]
            ulp = np.spacing(np.float32(abs(gamma - sp)))          # the score is gamma - distance: ulp of the distance
            near = int(np.sum(np.abs(s[i].astype(np.float64) - float(sp)) <= 4.0 * float(ulp))) - 1
            assert near >= abs(int(r[i]) - int(ref[i])) > 0, (mode, i, int(r[i]), int(ref[i]), near)
    assert differing < 0.02 * 2 * nq
