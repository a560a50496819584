"""Pins the error band of the two-stage RotatE / pRotatE ranking (count_ranks_kernel<OP, true, true> in
csrc/kge_eval.cu).  Its counts equal the exact kernel's only if every fast score s_f lies within
eps(s_f) = c_abs + c_rel * |gamma - s_f| + c_ulp * |s_f|  (kge_eval_two_stage_band) of the canonical score s_c.  Here the
fast scores are dumped by the ranking kernel itself (kge_eval_count_ranks_two_stage_approx) and compared with

  * s_c, the exact kernel's scores_out (bit-identical to the C oracle): |s_f - s_c| <= eps(s_f);
  * s64, a float64 restatement of the same scores from the same fp32 operands (the library's query vectors and entity
    table, or pRotatE's phase table; the pRotatE phase difference t = q -/+ x is taken as the fp32 value the model
    defines, everything after it is float64).  With u = 2^-24, T = sum_k |term_k| and the canonical order (blocks of
    KC = 32 consecutive k summed from 0, block sums added in order), the canonical fp32 score satisfies
        |s_c - s64| <= C + u |s_c|        (u |s_c|: the final rounding of gamma - p)
        RotatE:  C = (KC + ceil(d / KC) + 3) u T          (sums; 3 u per term: two differences, square, fma, sqrt)
        pRotatE: C = |mod| ((KC + ceil(d / KC)) u S + 1.6 u d) + u |mod| S    (S = sum |sin t|; 1.6 u per term:
                 sin_rep's error, pinned below by test_sincos_rep_error_over_the_fast_pass_range; u |mod| S: the
                 rounding of acc * mod)
    each times 1.01 for the second-order terms; and the fast score |s_f - s64| <= eps(s_f) + C + u |s_c|;
  * the ranks: two-stage == exact kernel (with a filter), == the C oracle where that is cheap, and the counts of entity
    slices add up to the full ranks.

The cases are the regimes where a band goes wrong: tiny distances (dense exact ties: the scores of two sums that
straddle a rounding boundary of gamma - acc differ by one ulp however close the sums are), a trained-down pRotatE
modulus, phases up to and across the 4e4 limit of the fast reduction, phases at odd multiples of pi/2, a negative
modulus, a partial 32-chunk, and the largest d of the fast pass (and the first one past it)."""
import ctypes
import math

import numpy as np
import pytest
import torch

from oracle import c_oracle as C
from oracle import kge_oracle as O

gpu = pytest.mark.gpu
KC, U = 32, 2.0 ** -24
MODES = ("head-batch", "tail-batch")


def _lib():
    from knowledgegraphembedding_b200 import _lib as L
    return L


def band_of(model, entity_dim, modulus=1.0):
    L = _lib()
    out = (ctypes.c_float * 3)()
    L.call("kge_eval_two_stage_band", L.MODEL_IDS[model], entity_dim, modulus, out)
    return [float(v) for v in out]


# ------------------------------------------------------------------------------------------------ cases
def rotate_case(nentity, d, gamma, scale, nq, seed, near=False):
    """RotatE tables at init scale times `scale`; with `near`, the answer of every query is moved to within the table's
    own spread of the query vector (E[t] = E[h] o r + noise, which also puts E[h] next to the head-batch query of the
    same triple): s_pos then sits among the other candidates, where tiny distances give dense exact ties."""
    st = O.init_tables("RotatE", nentity, 5, d, gamma, True, False, seed=seed)
    E = st["entity_embedding"].astype(np.float64) * scale
    rng = np.random.RandomState(seed + 1)
    heads = rng.choice(nentity // 2, nq, replace=False)
    tails = nentity // 2 + rng.choice(nentity - nentity // 2, nq, replace=False)
    rels = rng.randint(5, size=nq)
    if near:
        rho = O.embedding_range(gamma, d)
        ph = st["relation_embedding"].astype(np.float64)[rels] / (rho / math.pi)
        h = E[heads, :d] + 1j * E[heads, d:]
        t = h * np.exp(1j * ph) + scale * rho * (rng.uniform(-1, 1, h.shape) + 1j * rng.uniform(-1, 1, h.shape))
        E[tails] = np.concatenate([t.real, t.imag], 1)
    st["entity_embedding"] = E.astype(np.float32)
    return st, [(int(h), int(r), int(t)) for h, r, t in zip(heads, rels, tails)]


def protate_case(nentity, d, gamma, nq, seed, phase=None, mod_scale=1.0):
    """pRotatE tables at init, or with every entity and relation phase drawn by `phase(rng, shape)` (radians)."""
    st = O.init_tables("pRotatE", nentity, 5, d, gamma, False, False, seed=seed)
    rng = np.random.RandomState(seed + 1)
    if phase is not None:
        to_table = O.embedding_range(gamma, d) / math.pi          # phase = table / (rho / pi)
        st["entity_embedding"] = (phase(rng, (nentity, d)) * to_table).astype(np.float32)
        st["relation_embedding"] = (phase(rng, (5, d)) * to_table).astype(np.float32)
    st["modulus"] = (st["modulus"].astype(np.float64) * mod_scale).astype(np.float32)
    test = [(int(rng.randint(nentity)), int(rng.randint(5)), int(rng.randint(nentity))) for _ in range(nq)]
    return st, test


def half_pi_multiples(rng, shape):
    """phases at multiples of pi/2 plus 1e-3 noise; with relation phases of the same kind, about half of the phase
    differences sit next to an odd multiple (|sin| near 1, the reduced argument near +-pi/2)."""
    return 0.5 * math.pi * rng.randint(-60, 61, size=shape) + rng.uniform(-1e-3, 1e-3, size=shape)


CASES = {
    # RotatE
    "rotate_fb15k_init": lambda: ("RotatE", 24.0) + rotate_case(14951, 1000, 24.0, 1.0, 128, seed=31),
    "rotate_tiny_1e-2": lambda: ("RotatE", 24.0) + rotate_case(32 * 1024 + 45, 4, 24.0, 1e-2, 4096, seed=32, near=True),
    "rotate_tiny_1e-3": lambda: ("RotatE", 24.0) + rotate_case(32 * 1024 + 45, 4, 24.0, 1e-3, 4096, seed=33, near=True),
    "rotate_d36_gamma200": lambda: ("RotatE", 200.0) + rotate_case(4099, 36, 200.0, 1e-3, 512, seed=34, near=True),
    "rotate_d2048": lambda: ("RotatE", 24.0) + rotate_case(2085, 2048, 24.0, 1.0, 64, seed=35),
    # pRotatE
    "protate_fb15k_init": lambda: ("pRotatE", 24.0) + protate_case(14951, 1000, 24.0, 96, seed=41),
    "protate_phase_3.9e4": lambda: ("pRotatE", 24.0) + protate_case(
        3001, 36, 24.0, 256, seed=42, phase=lambda rng, s: rng.uniform(-1.3e4, 1.3e4, size=s)),
    "protate_phase_across_4e4": lambda: ("pRotatE", 24.0) + protate_case(
        3001, 36, 24.0, 256, seed=43, phase=lambda rng, s: rng.uniform(-1.55e4, 1.55e4, size=s)),
    "protate_odd_half_pi": lambda: ("pRotatE", 24.0) + protate_case(3001, 36, 24.0, 256, seed=44, phase=half_pi_multiples),
    "protate_modulus_1e-3": lambda: ("pRotatE", 24.0) + protate_case(14951, 1000, 24.0, 96, seed=45, mod_scale=1e-3),
    "protate_negative_modulus": lambda: ("pRotatE", 24.0) + protate_case(3001, 100, 24.0, 256, seed=46, mod_scale=-1.0),
}
ORACLE_CASES = {"rotate_tiny_1e-3", "rotate_d36_gamma200", "protate_phase_across_4e4", "protate_odd_half_pi",
                "protate_negative_modulus"}


def build(name):
    from test_gpu_parity import make_model
    model, gamma, st, test = CASES[name]()
    d = st["entity_embedding"].shape[1] // (2 if model == "RotatE" else 1)
    return model, gamma, d, st, test, make_model(model, st["entity_embedding"].shape[0], 5, d, gamma, st)


def true_triples(test, nentity, seed):
    rng = np.random.RandomState(seed)
    extra = {(int(rng.randint(nentity)), int(rng.randint(5)), int(rng.randint(min(nentity, 300)))) for _ in range(20000)}
    return sorted(extra | set(test))


# ------------------------------------------------------------------------------------------------ float64 reference
def operands(m, test, mode):
    """The fp32 operands every kernel scores: query vectors [Q, De] and the candidate table (entity or phase table)."""
    L = _lib()
    from knowledgegraphembedding_b200.model import _ptr, _stream
    dev = m.entity_embedding.device
    desc, st = m._descriptor(), _stream(dev)
    q = torch.tensor(test, dtype=torch.int64, device=dev)
    qvec = torch.empty(len(test), m.entity_dim, device=dev)
    L.call("kge_eval_query_vectors", ctypes.byref(desc), L.MODE_IDS[mode], _ptr(q), len(test), _ptr(qvec), None, st)
    X = m.entity_embedding.detach()
    if m.model_name == "pRotatE":
        X = torch.empty_like(X)
        L.call("kge_eval_phase_table", ctypes.byref(desc), _ptr(X), st)
    torch.cuda.synchronize()
    return qvec, X


def reference64(m, test, mode, gamma, modulus):
    """(s64, C, big): float64 scores, the canonical bound C of the module docstring (before u |s_c|), and for pRotatE
    the pairs with a phase difference |t| >= 4e4 (where the fast pass must answer NaN)."""
    qvec, X = operands(m, test, mode)
    Q, N = qvec.shape[0], X.shape[0]
    rot = m.model_name == "RotatE"
    d = X.shape[1] // 2 if rot else X.shape[1]
    nb = (d + KC - 1) // KC
    s64 = torch.empty(Q, N, dtype=torch.float64, device=qvec.device)
    bound = torch.empty_like(s64)
    big = torch.zeros(Q, N, dtype=torch.bool, device=qvec.device)
    step = max(1, (1 << 26) // (Q * d))
    for j0 in range(0, N, step):
        x = X[j0:j0 + step]
        if rot:
            q64, x64 = qvec.double(), x.double()
            a = q64[:, None, :d] - x64[None, :, :d]
            b = q64[:, None, d:] - x64[None, :, d:]
            T = torch.sqrt(a * a + b * b).sum(-1)
            s64[:, j0:j0 + step] = gamma - T
            bound[:, j0:j0 + step] = 1.01 * (KC + nb + 3) * U * T
        else:
            t = (x[None] + qvec[:, None]) if mode == "head-batch" else (qvec[:, None] - x[None])   # fp32, as the model
            big[:, j0:j0 + step] = (t.abs() >= 4.0e4).any(-1)
            S = torch.sin(t.double()).abs().sum(-1)
            s64[:, j0:j0 + step] = gamma - modulus * S
            bound[:, j0:j0 + step] = 1.01 * (abs(modulus) * ((KC + nb) * U * S + 1.6 * U * d) + U * abs(modulus) * S)
    return s64, bound, big


# ------------------------------------------------------------------------------------------------ GPU tests
@gpu
@pytest.mark.parametrize("name", list(CASES))
def test_fast_scores_inside_band_and_float64(name, monkeypatch):
    model, gamma, d, st, test, m = build(name)
    nentity = st["entity_embedding"].shape[0]
    modulus = float(st["modulus"].reshape(-1)[0]) if model == "pRotatE" else 1.0
    c_abs, c_rel, c_ulp = band_of(model, m.entity_dim, modulus)
    monkeypatch.setenv("KGE_EVAL_AMB_CAP", str(len(test) * nentity + 64))   # dense ties: most pairs may be undecidable
    all_true = true_triples(test, nentity, seed=len(name))
    for mode in MODES:
        _, sc = m.filtered_ranks(test, [], mode, return_scores=True)        # no filter: the plain score matrix
        m._ws.pop("two_stage_last_ambiguous", None)
        _, sf = m.filtered_ranks(test, [], mode, return_approx=True)
        assert sf is not None and "two_stage_last_ambiguous" in m._ws, "two-stage path was not taken"
        sc, sf = sc.double(), sf.double()
        s64, canon, big = reference64(m, test, mode, gamma, modulus)
        canon = canon + U * sc.abs()
        finite = torch.isfinite(sf)
        if model == "pRotatE":      # the fast pass gives up (NaN) exactly where a phase difference reaches 4e4
            assert torch.equal(~finite, big), (name, mode, int((~finite).sum()), int(big.sum()))
        else:
            assert bool(finite.all())
        eps = c_abs + c_rel * (gamma - sf).abs() + c_ulp * sf.abs()
        err = (sf - sc).abs()
        ratio = torch.where(finite, err / eps, torch.zeros_like(err))
        worst = float(ratio.max())
        # the canonical scores against float64, then the fast ones against float64 through the band
        c_ratio = float(((sc - s64).abs() / canon).max())
        f_ratio = float(torch.where(finite, (sf - s64).abs() / (eps + canon), torch.zeros_like(err)).max())
        nbad = int((ratio > 1).sum())
        ties = int((sc == sc.gather(1, torch.tensor([t[0] if mode == "head-batch" else t[2] for t in test],
                                                     device=sc.device)[:, None])).sum()) - len(test)
        print(f"{name} {mode}: max |s_f - s_c| / eps = {worst:.3f} ({nbad} pairs outside), |s_c - s64| / bound = "
              f"{c_ratio:.3f}, |s_f - s64| / (eps + bound) = {f_ratio:.3f}, {ties} exact ties with s_pos, "
              f"{int((~finite).sum())} NaN")
        assert nbad == 0, (name, mode, worst, nbad)
        assert c_ratio <= 1.0, (name, mode, c_ratio)
        assert f_ratio <= 1.0, (name, mode, f_ratio)
        # ranks: two-stage (with a filter) == exact kernel, and == the C oracle where that is cheap
        m._ws.pop("two_stage_last_ambiguous", None)
        fast = m.filtered_ranks(test, all_true, mode)
        amb = m._ws["two_stage_last_ambiguous"]
        exact = m.filtered_ranks(test, all_true, mode, exact=True)
        print(f"{name} {mode}: {amb} undecidable pairs ({amb / (len(test) * nentity):.2e} of all), "
              f"{int((fast != exact).sum())} ranks differ")
        np.testing.assert_array_equal(fast, exact)
        if name in ORACLE_CASES:
            from knowledgegraphembedding_b200 import FilterIndex
            sub = test[:512]
            off, ent = FilterIndex(all_true, nentity, 5).csr(sub, mode)
            cs = C.eval_scores(model, st, sub, mode, gamma, O.embedding_range(gamma, d), off, ent)
            np.testing.assert_array_equal(fast[:len(sub)], C.ranks_from_scores(cs, sub, mode))


def _two_stage_counts(m, test, all_true, mode, slices, dump=None, amb_init=0):
    """Counts of kge_eval_count_ranks_two_stage_approx summed over entity slices, and the last call's amb_count."""
    L = _lib()
    from knowledgegraphembedding_b200 import FilterIndex
    from knowledgegraphembedding_b200.model import _ptr, _stream
    dev = m.entity_embedding.device
    nentity = m.entity_embedding.shape[0]
    desc, st, mid = m._descriptor(), _stream(dev), L.MODE_IDS[mode]
    Q = len(test)
    q = torch.tensor(test, dtype=torch.int64, device=dev)
    off, ent = FilterIndex(all_true, nentity, m.relation_embedding.shape[0]).csr(test, mode)
    d_off, d_ent = torch.from_numpy(off).to(dev), torch.from_numpy(ent).to(dev)
    bits = torch.zeros(Q * ((nentity + 31) // 32), dtype=torch.int32, device=dev)
    qvec, phase = operands(m, test, mode)
    phase = phase if m.model_name == "pRotatE" else None
    pos = torch.empty(Q, device=dev)
    L.call("kge_eval_filter_bits", _ptr(d_off), _ptr(d_ent), Q, nentity, _ptr(bits), st)
    L.call("kge_eval_positive_scores", ctypes.byref(desc), mid, _ptr(qvec), _ptr(q), Q, _ptr(phase), _ptr(pos), st)
    cap = Q * nentity + 64
    amb = torch.empty(2 * cap, dtype=torch.int32, device=dev)
    amb_count = torch.full((2,), amb_init, dtype=torch.int32, device=dev)
    total = torch.zeros(Q, dtype=torch.int32, device=dev)
    for b, e in slices:
        part = torch.zeros(Q, dtype=torch.int32, device=dev)
        L.call("kge_eval_count_ranks_two_stage_approx", ctypes.byref(desc), mid, _ptr(qvec), _ptr(q), Q, _ptr(phase),
               _ptr(pos), _ptr(bits), b, e, _ptr(part), _ptr(amb), cap, _ptr(amb_count),
               _ptr(dump) if dump is not None else None, st)
        total += part
    torch.cuda.synchronize()
    return total.cpu().numpy().astype(np.int64) + 1, amb_count.cpu().numpy()


@gpu
@pytest.mark.parametrize("name", ["rotate_tiny_1e-3", "rotate_d36_gamma200", "protate_modulus_1e-3",
                                  "protate_phase_across_4e4"])
def test_two_stage_entity_slices_sum_to_full_ranks(name):
    """Entity sharding of the two-stage path: the counts over the 8 aligned shards of a multi-GPU run, and over
    unaligned slices, add up to the full ranks of the exact kernel."""
    from knowledgegraphembedding_b200 import shard_bounds
    model, gamma, d, st, test, m = build(name)
    nentity = st["entity_embedding"].shape[0]
    test = test[:1024]
    all_true = true_triples(test, nentity, seed=7)
    cuts = [0, 1, 63, 64 * 5 + 3, nentity // 3, nentity // 2 + 17, nentity - 65, nentity - 1, nentity]
    for mode in MODES:
        exact = m.filtered_ranks(test, all_true, mode, exact=True)
        aligned, _ = _two_stage_counts(m, test, all_true, mode, [shard_bounds(nentity, r, 8, align=128) for r in range(8)])
        np.testing.assert_array_equal(aligned, exact)
        ragged, _ = _two_stage_counts(m, test, all_true, mode, list(zip(cuts[:-1], cuts[1:])))
        np.testing.assert_array_equal(ragged, exact)


@gpu
def test_rotate_d2052_has_no_fast_pass():
    """d = 2052 is past the d the band is proven for: the two-stage entry runs the exact kernel (no fast pass zeroes
    amb_count, the dump holds the exact scores) and the band export refuses the shape."""
    st, test = rotate_case(1100, 2052, 24.0, 1.0, 64, seed=36)
    from test_gpu_parity import make_model
    m = make_model("RotatE", 1100, 5, 2052, 24.0, st)
    with pytest.raises(ValueError, match="no two-stage pass"):
        band_of("RotatE", m.entity_dim)
    all_true = true_triples(test, 1100, seed=3)
    for mode in MODES:
        _, sc = m.filtered_ranks(test, [], mode, return_scores=True)
        dump = torch.full((len(test), 1100), float("nan"), device=sc.device)
        _, amb_count = _two_stage_counts(m, test, [], mode, [(0, 1100)], dump=dump, amb_init=-7)
        assert amb_count.tolist() == [-7, -7], "a fast pass ran"
        assert torch.equal(dump.view(torch.int32), sc.view(torch.int32))
        ranks, amb_count = _two_stage_counts(m, test, all_true, mode, [(0, 1100)], amb_init=-7)
        assert amb_count.tolist() == [-7, -7]
        np.testing.assert_array_equal(ranks, m.filtered_ranks(test, all_true, mode, exact=True))
        np.testing.assert_array_equal(m.filtered_ranks(test, all_true, mode), ranks)


# ------------------------------------------------------------------------------------------------ no GPU needed
def test_sincos_rep_error_over_the_fast_pass_range():
    """The canonical sine / cosine (kge_math.h sincos_rep, restated by the C oracle) within 1.6 * 2^-24 of the true
    values over the fp32 reduction (|t| < 4e4, where the fast pRotatE pass answers) and the fp64 branch beyond it: the
    per-term error the pRotatE float64 bound above relies on."""
    rng = np.random.RandomState(11)
    near = 0.5 * np.pi * rng.randint(-25000, 25001, 400000) + rng.uniform(-1e-3, 1e-3, 400000)
    for x in (rng.uniform(-4e4, 4e4, 2000000), rng.uniform(4e4, 1e6, 1000000) * rng.choice([-1, 1], 1000000), near,
              np.float32([4e4, -4e4, np.nextafter(np.float32(4e4), np.float32(0)), 1e6, -1e6, 39999.99])):
        x = np.asarray(x, np.float32)
        s, c = C.sincos(x)
        x64 = x.astype(np.float64)
        assert np.max(np.abs(s - np.sin(x64))) < 1.6 * U
        assert np.max(np.abs(c - np.cos(x64))) < 1.6 * U


def test_two_stage_abi_argument_errors_without_a_gpu():
    L = _lib()
    lib = L.load()
    out = (ctypes.c_float * 3)()
    assert lib.kge_eval_two_stage_band(L.ROTATE, 2000, 1.0, out) == 0
    assert list(out) == [np.float32(1e-12), np.float32(1.6e-5), 2.0 ** -22]
    rot = list(out)
    assert lib.kge_eval_two_stage_band(L.ROTATE, 4096, 1.0, out) == 0 and list(out) == rot     # d = 2048: largest
    for mod in (0.013, -0.013):                                                               # |modulus| * d * 2e-6
        assert lib.kge_eval_two_stage_band(L.PROTATE, 1000, mod, out) == 0
        np.testing.assert_allclose(out[0], 0.013 * 1000 * 2e-6, rtol=1e-6)
        assert out[1] == np.float32(1.2e-5) and out[2] == 2.0 ** -22
    assert lib.kge_eval_two_stage_band(L.PROTATE, 2048, 1.0, out) == 0
    for model, entity_dim in ((L.ROTATE, 4098), (L.ROTATE, 7), (L.ROTATE, 0), (L.PROTATE, 2049), (L.PROTATE, -4)):
        assert lib.kge_eval_two_stage_band(model, entity_dim, 1.0, out) == L.ERR_INVALID
        assert b"no two-stage pass" in lib.kge_last_error()
    for model in (L.TRANSE, L.DISTMULT, L.COMPLEX, 9):
        assert lib.kge_eval_two_stage_band(model, 64, 1.0, out) == L.ERR_INVALID
        assert b"no two-stage pass" in lib.kge_last_error()
    assert lib.kge_eval_two_stage_band(L.ROTATE, 64, 1.0, None) == L.ERR_INVALID
    assert b"null pointer" in lib.kge_last_error()

    desc = L.KgeModelStruct(model=L.ROTATE, device=0, nentity=100, nrelation=5, hidden_dim=8, entity_dim=16,
                            relation_dim=8, gamma=6.0, embedding_range=1.0, entity=16, relation=16, modulus=None)
    d = ctypes.byref(desc)

    def call(mode=L.TAIL_BATCH, b=0, e=100, amb=16, cap=10, amb_count=16, qvec=16):
        return lib.kge_eval_count_ranks_two_stage_approx(d, mode, qvec, 16, 10, None, 16, 16, b, e, 16, amb, cap,
                                                         amb_count, 16, None)
    for kw in (dict(amb=None), dict(cap=0), dict(amb_count=None)):
        assert call(**kw) == L.ERR_INVALID
        assert b"ambiguous-pair buffers" in lib.kge_last_error()
    assert call(mode=L.SINGLE) == L.ERR_INVALID and b"negative batch mode" in lib.kge_last_error()
    for b, e in ((0, 101), (-1, 5), (30, 20)):
        assert call(b=b, e=e) == L.ERR_INVALID and b"entity slice" in lib.kge_last_error()
    assert call(qvec=None) == L.ERR_INVALID and b"null pointer" in lib.kge_last_error()
