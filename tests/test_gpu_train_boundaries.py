"""KGEModel.train_step and the autograd path at every row / entity kernel instantiation and launcher boundary, against
a float64 restatement (oracle/kge_oracle.py with compute_dtype=float64).

Every case runs its first step under torch.profiler and checks that the kernels which ran -- demangled template
arguments and block sizes -- are the ones test_train_launch_rules.expected_launch restates for the case, so a change of
the launcher cannot quietly route a boundary case to the default path.  The case table lives in
test_train_launch_rules.py, where a CPU test checks that it reaches every instantiation in the library.

Tolerances are calibrated per case: the numpy oracle also runs in float32, and the GPU's distance to float64 may be at
most K times the float32 oracle's distance, or a floor, whichever is larger."""
import json

import numpy as np
import pytest
import torch

from conftest import outlier_fraction, relinf
from oracle import kge_oracle as O
from test_gpu_parity import FLAGS, KGE, make_model, ns
from test_train_launch_rules import AUTOGRAD, CASES, F64_BUDGET, TRAIN_KERNELS, expected_autograd

pytestmark = pytest.mark.gpu

# Calibration: GPU error / float32-oracle error, and the floors for cases where the float32 oracle happens to be
# (nearly) exact.  Measured on a B200 at a 1000 W power limit (each test prints its worst ratio, floors included):
# at most 2.8 on the train step (softmax-order RotatE), 5.3 on the autograd path (pRotatE d = 1024, the sin of the
# phase).
K = 8.0
FLOOR_LOSS = 2e-6              # relative error of a loss value
FLOOR_GRAD = 2e-5              # relinf of a gradient or a first moment (the second moment gets twice)
FLOOR_SCORE = 2e-6             # relinf of a score matrix
LR, GAMMA, NREL = 1e-3, 12.0, 5
ENV_KEYS = ("KGE_KEEP_GRADS", "KGE_FORCE_SPLIT", "KGE_NO_SPLIT", "KGE_NO_TMA", "KGE_SPLIT_VARIANT", "KGE_SPLIT_RING",
            "KGE_SPLIT_CTAS", "KGE_ENTITY_PARTS", "KGE_ENTITY_WARPS", "KGE_ENTITY_DEPTH", "KGE_L2_HINTS",
            "KGE_ZERO_COPY", "KGE_ROW_PHASES")


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def set_env(monkeypatch, env):
    for k in ENV_KEYS:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


def observe(fn, tmp_path):
    """Run fn under torch.profiler; the train-path kernels that ran, as sorted [((name, template args), block)]."""
    import re
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    path = tmp_path / "trace.json"
    prof.export_chrome_trace(str(path))
    with open(path) as f:
        events = json.load(f)["traceEvents"]
    got = []
    for ev in events:
        if ev.get("cat") != "kernel":
            continue
        m = re.search(r"kge::(\w+)<([^>]*)>", ev["name"])
        if not m or m.group(1) not in TRAIN_KERNELS:
            continue
        args = tuple({"true": 1, "false": 0}.get(a.strip(), None) if a.strip() in ("true", "false") else int(a)
                     for a in m.group(2).split(","))
        got.append(((m.group(1), args), int(ev["args"]["block"][0])))
    return sorted(got), out


def calibrated(got, want64, want32, floor, measure=relinf):
    """GPU distance to float64 within max(K x the float32 oracle's distance, floor)."""
    e, e32 = measure(got, want64), measure(want32, want64)
    return e <= max(K * e32, floor), (e, e32)


def rel(a, b):
    return abs(float(a) - float(b)) / max(abs(float(b)), 1e-30)


# ---------------------------------------------------------------------------------------------------- inputs
def make_inputs(case, rows):
    """Tables and two batches.  Step 1 draws every id from the lower half of the entity range and step 2 from the
    upper half, so that step 2 has entities with pairs in step 1 and none now (dense Adam still moves them), and step 1
    has entities without any pair."""
    model, d, N, n = case.model, case.d, case.N, case.nentity
    de, dr = FLAGS[model]
    gamma = 60.0 if case.data == "saturate" else GAMMA
    st = O.init_tables(model, n, NREL, d, gamma, de, dr, seed=7)
    rng = np.random.RandomState(11)
    head = case.mode == "head-batch"
    batches = []
    for s in range(case.steps):
        lo, hi = (0, n // 2) if s == 0 else (n // 2, n)
        pos = np.stack([rng.randint(lo, hi, rows), rng.randint(NREL, size=rows), rng.randint(lo, hi, rows)], 1)
        neg = rng.randint(lo, hi, (rows, N))
        w = np.sqrt(1.0 / rng.randint(8, 200, size=rows)).astype(np.float32)
        batches.append([pos, neg, w])
    E, R = st["entity_embedding"], st["relation_embedding"]
    fixed_col = 2 if head else 0                     # the positive's fixed side; its answer is the other one
    if case.data in ("kink_equal", "kink_partial", "kink_tiny") or (case.data == "saturate" and model != "DistMult"):
        R[0] = 0.0                                    # zero translation / zero phase
        for b in batches:
            b[0][:, 1] = 0
    if case.data == "kink_equal":
        for b in batches:                             # candidates equal to q: the fixed entity itself
            b[1][:, ::5] = b[0][:, fixed_col][:, None]
    elif case.data == "kink_partial":
        E[:] = np.round(E * 1024) / 1024              # sums of table entries are exact in fp32 and float64
        for b in batches:
            for r in range(rows):                     # a candidate sharing every second coordinate with q
                c = b[1][r, 0]
                E[c, ::2] = E[b[0][r, fixed_col], ::2]
    elif case.data == "kink_tiny":
        zero, tiny = 1, 2
        for b in batches:
            b[0][:, fixed_col] = zero
            b[1][:, ::4] = tiny
        E[zero] = 0.0
        E[tiny] = 1e-12                               # |q - x| = sqrt(2) 1e-12: far above the FLT_MIN guard's reach
    elif case.data == "one_entity":
        for b in batches:
            b[1][:] = b[1][0, 0]
    elif case.data == "duplicates":
        for b in batches:
            b[1][:] = b[1][:, :4][:, rng.randint(4, size=N)]
    elif case.data == "own_ids":
        for b in batches:
            b[1][:, 0::4] = b[0][:, 0][:, None]
            b[1][:, 1::4] = b[0][:, 2][:, None]
    elif case.data == "saturate":
        for b in batches:
            b[0][: rows // 2, 2 - fixed_col] = b[0][: rows // 2, fixed_col]   # score gamma exactly: logsigmoid(60)
            b[1][:, 0] = b[0][:, fixed_col]
        scale_to_saturate(model, st, batches, case.mode, gamma, d)
    elif case.data.startswith("order_"):
        E *= 8.0                                      # score spread ~ 30: alpha * spread > 104, early weights underflow
        for _ in range(2):                            # gamma: negative scores around 0, where sigmoid(s) matters
            s = O.forward(model, st, (batches[0][0], batches[0][1]), case.mode, gamma, d, np.float64)
            gamma = float(np.round(2 * (gamma - np.mean(s))) / 2)
        for b in batches:
            s = O.forward(model, st, (b[0], b[1]), case.mode, gamma, d, np.float64)
            order = np.argsort(s, axis=1, kind="stable")
            if case.data == "order_dec":
                order = order[:, ::-1]
            b[1] = np.take_along_axis(b[1], order, axis=1)
    return st, gamma, [(b[0], b[1], b[2], case.mode) for b in batches]


def scale_to_saturate(model, st, batches, mode, gamma, d):
    """Scores down to about gamma - 260 = -200 (distance models) or +-200 (DistMult)."""
    allneg = np.concatenate([b[1] for b in batches])
    allpos = np.concatenate([b[0] for b in batches])
    s = O.forward(model, st, (allpos, allneg), mode, gamma, d, np.float64)
    if model == "TransE":
        f = 260.0 / np.max(gamma - s)
        st["entity_embedding"] *= np.float32(f)
        st["relation_embedding"] *= np.float32(f)
    elif model == "pRotatE":
        st["modulus"] *= np.float32(260.0 / np.max(gamma - s))
    else:
        st["entity_embedding"] *= np.float32(np.sqrt(200.0 / np.max(np.abs(s))))


# ---------------------------------------------------------------------------------------------------- reference
def ref_step(model, state, batch, gamma, d, adv, reg, dtype):
    """Losses and gradients of one train step; grads = score gradients only, l3 = the L3 term's gradients.  The
    candidates are gathered in column blocks of at most F64_BUDGET elements (scores and gradients are sums over
    independent candidates), so N = 8192 at the widest rows stays in float64 too."""
    pos, neg, w, mode = batch
    De = state["entity_embedding"].shape[1]
    c = max(1, F64_BUDGET // (len(pos) * De))
    cols = [slice(i, i + c) for i in range(0, neg.shape[1], c)]
    sn = np.concatenate([O.forward(model, state, (pos, neg[:, j]), mode, gamma, d, dtype) for j in cols], axis=1)
    sp = O.forward(model, state, pos, "single", gamma, d, dtype)
    pl, nl, loss, dneg, dpos = O.loss_and_dscore(sn, sp, w, adv > 0, adv if adv > 0 else 1.0, False, dtype)
    grads = O.score_backward(model, state, pos, "single", dpos, gamma, d, dtype)
    for j in cols:
        g1 = O.score_backward(model, state, (pos, neg[:, j]), mode, dneg[:, j], gamma, d, dtype)
        grads = {k: grads[k] + g1[k] for k in grads}
    log = {}
    l3 = {k: np.zeros_like(v) for k, v in grads.items()}
    if reg:
        E, R = state["entity_embedding"].astype(np.float64), state["relation_embedding"].astype(np.float64)
        val = reg * (np.sum(np.abs(E) ** 3) + np.sum(np.abs(R) ** 3))
        l3["entity_embedding"], l3["relation_embedding"] = 3 * reg * E * np.abs(E), 3 * reg * R * np.abs(R)
        loss = loss + dtype(val)
        log["regularization"] = val
    log.update(positive_sample_loss=pl, negative_sample_loss=nl, loss=loss)
    return log, grads, l3


def sync_state(m, opt, ref, params):
    with torch.no_grad():
        for name, p in params:
            p.copy_(torch.from_numpy(ref["p"][name]))
            opt.state[p]["exp_avg"].copy_(torch.from_numpy(ref["m"][name]))
            opt.state[p]["exp_avg_sq"].copy_(torch.from_numpy(ref["v"][name]))


# ---------------------------------------------------------------------------------------------------- train step
@pytest.mark.parametrize("case", CASES, ids=lambda c: c.id)
def test_train_step_boundary(case, monkeypatch, tmp_path):
    set_env(monkeypatch, case.env)
    S = sms()
    rows = case.rows(S)
    st, gamma, batches = make_inputs(case, rows)
    m = make_model(case.model, case.nentity, NREL, case.d, gamma, st)       # fresh model: the plan is cached per shape
    opt = torch.optim.Adam(filter(lambda p: p.requires_grad, m.parameters()), lr=LR)
    args = ns(negative_adversarial_sampling=case.adv > 0, adversarial_temperature=case.adv or 1.0,
              regularization=case.reg)
    params = [("entity_embedding", m.entity_embedding), ("relation_embedding", m.relation_embedding)]
    if case.model == "pRotatE":
        params.append(("modulus", m.modulus))
    want = case.launch(S)
    fused = want["fused_entity_adam"]
    ref = {"p": {k: np.array(v, np.float32) for k, v in st.items()},
           "m": {k: np.zeros_like(v, np.float32) for k, v in st.items()},
           "v": {k: np.zeros_like(v, np.float32) for k, v in st.items()}}
    worst = 0.0
    for step, batch in enumerate(batches):
        tb = (torch.from_numpy(batch[0]), torch.from_numpy(batch[1]), torch.from_numpy(batch[2]), batch[3])
        if step == 0:
            ran, log = observe(lambda: KGE().train_step(m, opt, iter([tb]), args), tmp_path)
            assert ran == sorted(want["kernels"]), (ran, want["kernels"])
        else:
            log = KGE().train_step(m, opt, iter([tb]), args)
        assert all(np.isfinite(v) for v in log.values()), log
        st_now = {k: v.copy() for k, v in ref["p"].items()}
        l64, g64, r64 = ref_step(case.model, st_now, batch, gamma, case.d, case.adv, case.reg, np.float64)
        l32, g32, _ = ref_step(case.model, st_now, batch, gamma, case.d, case.adv, case.reg, np.float32)
        assert list(log) == list(l64)
        for k in l64:
            ok, e = calibrated(log[k], l64[k], l32[k], FLOOR_LOSS, rel)
            worst = max(worst, e[0] / max(e[1], FLOOR_LOSS / K))
            assert ok, (step, k, log[k], float(l64[k]), e)
        assert (m.entity_embedding.grad is None) == fused
        for name, p in params:          # p.grad holds the L3 term too: autograd of loss + regularization
            if p.grad is None:
                continue
            ok, e = calibrated(p.grad.cpu().numpy(), g64[name] + r64[name], g32[name] + r64[name], FLOOR_GRAD)
            worst = max(worst, e[0] / max(e[1], FLOOR_GRAD / K))
            assert ok, (step, name, e)
        # Adam on the float64 gradients (the L3 term is the optimizer's, also in the fused entity pass)
        for name, p in params:
            g = (g64[name] + r64[name]).astype(np.float32)
            g_32 = (g32[name] + r64[name]).astype(np.float32)
            m64, v64 = ref["m"][name].copy(), ref["v"][name].copy()
            m32 = m64 * np.float32(0.9) + np.float32(0.1) * g_32
            v32 = v64 * np.float32(0.999) + np.float32(0.001) * g_32 * g_32
            O.adam_update(ref["p"][name], g, ref["m"][name], ref["v"][name], step + 1, LR)
            mom = opt.state[p]
            # fused entity pass: the step's entity gradient is only visible through the moments
            ok, e = calibrated(mom["exp_avg"].cpu().numpy(), ref["m"][name], m32, FLOOR_GRAD)
            assert ok, (step, name, "exp_avg", e)
            ok, e = calibrated(mom["exp_avg_sq"].cpu().numpy(), ref["v"][name], v32, 2 * FLOOR_GRAD)
            assert ok, (step, name, "exp_avg_sq", e)
            got, wantp = p.detach().cpu().numpy(), ref["p"][name]
            # an entity whose gradient cancels to ~eps takes an Adam step that its rounding decides (conftest.py
            # outlier_fraction): measured on B200, one such row of 600 in the adversarial softmax-order cases
            assert outlier_fraction(got, wantp, 1e-5) < 1e-2, (step, name)
            assert np.max(np.abs(got - wantp)) <= 2.0 * LR + 1e-5 * np.abs(wantp).max(), (step, name)
        sync_state(m, opt, ref, params)
    print("calibration %s: worst gpu/fp32 error ratio %.3g" % (case.id, worst))


# ---------------------------------------------------------------------------------------------------- autograd
@pytest.mark.parametrize("model,d", AUTOGRAD, ids=lambda v: str(v))
def test_autograd_boundary(model, d, monkeypatch, tmp_path):
    """model((pos, neg), mode) / model(pos) and .backward() of a random cotangent against float64 forward /
    score_backward: the forward-only TMA kernel, the split kernel without a loss (and pRotatE's modulus gradient
    from the entity pass), and the direct-load kernels."""
    set_env(monkeypatch, {})
    B, N, n = 8, 64, 80
    de, dr = FLAGS[model]
    st = O.init_tables(model, n, NREL, d, GAMMA, de, dr, seed=3)
    rng = np.random.RandomState(5)
    pos = np.stack([rng.randint(n, size=B), rng.randint(NREL, size=B), rng.randint(n, size=B)], 1)
    neg = rng.randint(n, size=(B, N))
    worst = 0.0
    for mode in ("single", "head-batch", "tail-batch"):
        mm = make_model(model, n, NREL, d, GAMMA, st)
        sample = (pos, neg) if mode != "single" else pos
        cot = rng.standard_normal((B, 1 if mode == "single" else N))

        def run():
            s = mm(torch.from_numpy(pos)) if mode == "single" else \
                mm((torch.from_numpy(pos), torch.from_numpy(neg)), mode)
            (s * torch.from_numpy(cot).float().cuda()).sum().backward()
            return s.detach().cpu().numpy()
        ran, s = observe(run, tmp_path)
        assert ran == sorted(expected_autograd(model, mode, d, N, B, n, {}, sms())["kernels"]), (mode, ran)
        s64 = O.forward(model, st, sample, mode, GAMMA, d, np.float64)
        s32 = O.forward(model, st, sample, mode, GAMMA, d, np.float32)
        ok, e = calibrated(s, s64, s32, FLOOR_SCORE)
        worst = max(worst, e[0] / max(e[1], FLOOR_SCORE / K))
        assert ok, (mode, "score", e)
        g64 = O.score_backward(model, st, sample, mode, cot, GAMMA, d, np.float64)
        g32 = O.score_backward(model, st, sample, mode, cot.astype(np.float32), GAMMA, d, np.float32)
        got = {"entity_embedding": mm.entity_embedding.grad, "relation_embedding": mm.relation_embedding.grad}
        if model == "pRotatE":
            got["modulus"] = mm.modulus.grad
        for name, g in got.items():
            ok, e = calibrated(g.cpu().numpy(), g64[name], g32[name], FLOOR_GRAD)
            worst = max(worst, e[0] / max(e[1], FLOOR_GRAD / K))
            assert ok, (mode, name, e)
    print("calibration autograd %s d=%d: worst gpu/fp32 error ratio %.3g" % (model, d, worst))
