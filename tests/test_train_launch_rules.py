"""The train step's kernel choice, restated in Python, and the case table of tests/test_gpu_train_boundaries.py.

`expected_launch` restates split_path_shape_ok / plan_split (csrc/kge_train.cu), launch_rows_v and launch_entity_pass
(csrc/kge_train_launch.cuh) for one KGEModel.train_step with a stock torch.optim.Adam on one GPU: which row kernel runs
with which template arguments and block size, whether a separate launch scores the positive triples, and which entity
kernel (if any) finishes the backward.  The GPU tests compare it with the kernels that torch.profiler observes, so every
boundary case provably runs the kernel it is meant to run; the CPU tests below check that the case table reaches every
row / entity kernel instantiation that the library contains."""
import os
import struct

import pytest

MODELS = ("TransE", "DistMult", "ComplEx", "RotatE", "pRotatE")
MODEL_ID = {m: i for i, m in enumerate(MODELS)}
CPLX = ("ComplEx", "RotatE")
SMEM = 227 * 1024                      # dynamic shared memory the launcher plans with (bytes per block)
B200_SMS = 148
F64_BUDGET = 10 ** 7                   # gathered B * N * entity_dim of a float64 reference


def dims(model, d):
    """(entity_dim, relation_dim) of a KGEModel with hidden_dim d and the flags its model needs."""
    return (2 * d if model in CPLX else d), (2 * d if model == "ComplEx" else d)


def _atoi(s):
    s = s.strip()
    n = len(s) - len(s.lstrip("+-"))
    while n < len(s) and s[n].isdigit():
        n += 1
    try:
        return int(s[:n])
    except ValueError:
        return 0


def split_warps(cplx, nch, var):
    f = (2 if cplx else 1) * nch
    if var == 0:
        return 13 if f >= 16 else 16
    if var == 1:
        return 12 if f >= 16 else 16
    if var == 2:
        return 8 if f >= 16 else (12 if f >= 8 else 16)
    if var == 3:
        return 12 if f >= 16 else 16
    return 16


def split_variant(env):
    v = env.get("KGE_SPLIT_VARIANT")
    return int(v) if v is not None and len(v) == 1 and v in "01234" else 2


def shape_ok(rows, N, De, d, cplx, nentity, fused, env):
    """split_path_shape_ok."""
    if "KGE_NO_SPLIT" in env or "KGE_NO_TMA" in env:
        return False
    if d % 4 or De % 4 or d // 4 > 32 * (8 if cplx else 16):
        return False
    if N < 8 or nentity >= 2 ** 31 or rows * (N + 3) >= 2 ** 31:
        return False
    return fused or rows * N >= 6 * nentity or "KGE_FORCE_SPLIT" in env


def entity_pass(model, d, fused, env, sms):
    """launch_entity_pass: (('entity_kernel', (MODEL, HEAD, S, FUSED)) without HEAD, block, depth)."""
    cplx = model in CPLX
    nunits = d // 4
    two = nunits >= 64 and not env.get("KGE_ENTITY_PARTS", "").startswith("1")
    slotbytes = (2 if cplx else 1) * ((8 if cplx else 16) // (2 if two else 1)) * 32 * 16
    We = (20 if not fused else 16) if two else 12
    if "KGE_ENTITY_WARPS" in env:
        v = _atoi(env["KGE_ENTITY_WARPS"])
        if 1 <= v <= We:
            We = v
    depth = 2
    while depth < 4 and 16 + We * (depth + 1) * (slotbytes + 16) <= SMEM:
        depth += 1
    if "KGE_ENTITY_DEPTH" in env:
        v = _atoi(env["KGE_ENTITY_DEPTH"])
        if 2 <= v <= depth:
            depth = v
    while We > 1 and 16 + We * depth * (slotbytes + 16) > SMEM:
        We -= 1
    return (2 if two else 1), We * 32, depth


def launch_rows(model, head, d, N, rows, nentity, env, sms, *, do_loss, positive_loss, want_adam, workspace, gE):
    """launch_rows + launch_rows_v: dict(row=(name, args), block, grid, fused_positive, entity, entity_block, ...)."""
    De, Dr = dims(model, d)
    cplx = model in CPLX
    M = MODEL_ID[model]
    vec4 = Dr % 4 == 0 and d % 4 == 0 and De % 4 == 0
    nunits = d // 4
    out = dict(fused_positive=False, entity=None, entity_block=None)
    if vec4 and nunits <= 32 * (8 if cplx else 16) and "KGE_NO_TMA" not in env:
        split = (workspace and (gE or want_adam) and not (do_loss and positive_loss) and
                 shape_ok(rows, N, De, d, cplx, nentity, want_adam, env))
        if split:
            Hs = 2 if cplx else 1
            chunks = (nunits + 31) // 32
            nch = 4 if chunks <= 4 else (8 if chunks <= 8 else 16)
            var = split_variant(env)
            hs = Hs * 128 * nch
            fixed_s = 4 * (hs + ((De + 3) & ~3) + 2 * ((d + 3) & ~3) + 2 * N + 32 + 2 * (2 * De + Dr)) + 32
            wpr = 2 if var >= 3 else 1
            wcap = split_warps(cplx, nch, var) // wpr
            Ws = wcap
            if N < 4 * Ws:
                Ws = (N + 3) // 4 if N >= 16 else 4
            Ws = min(Ws, wcap)

            def group_bytes(depth):
                return depth * (hs * 4 + 8) + 16 + 4
            ring, ring_max = 2, 2
            while ring_max < 4 and fixed_s + Ws * group_bytes(ring_max + 1) <= SMEM:
                ring_max += 1
            if "KGE_SPLIT_RING" in env:
                v = _atoi(env["KGE_SPLIT_RING"])
                if 2 <= v <= ring_max:
                    ring = v
            while Ws > 1 and fixed_s + Ws * group_bytes(ring) > SMEM:
                Ws -= 1
            ctas = 1
            if env.get("KGE_SPLIT_CTAS", "").startswith("2"):
                if wpr == 1 and Ws >= 8 and 2 * (fixed_s + (Ws // 2) * group_bytes(ring) + 1024) <= SMEM:
                    ctas, Ws = 2, Ws // 2
            if Ws >= (2 if wpr == 2 else 4) and fixed_s + Ws * group_bytes(ring) <= SMEM:
                out.update(row=("row_kernel_split", (M, int(head), nch, var)), block=Ws * wpr * 32,
                           grid=min(rows, sms * ctas), ring=ring, ctas=ctas, fused_positive=do_loss)
                S, eblock, depth = entity_pass(model, d, want_adam, env, sms)
                out.update(entity=("entity_kernel", (M, int(head), S, int(want_adam))), entity_block=eblock,
                           entity_depth=depth)
                return out
        # two-sweep TMA kernel
        Dq4 = (De + 3) & ~3
        fixed = 4 * (2 * Dq4 + (2 * N if do_loss else 0) + 32) + 16
        rowbytes = De * 4
        W = ((SMEM - fixed) % 2 ** 64) // (2 * rowbytes + 16)      # size_t arithmetic, then (int)
        W = (W + 2 ** 31) % 2 ** 32 - 2 ** 31
        W = min(W, 16)
        if N < 4 * W:
            W = (N + 3) // 4 if N >= 16 else 4
        if W >= 4 and fixed + W * (2 * rowbytes + 16) <= SMEM:
            out.update(row=("row_kernel_tma", (M, int(head))), block=W * 32, grid=rows)
            return out
    threads = 512 if N >= 16 else (256 if N >= 4 else 128)
    out.update(row=("row_kernel", (M, int(head), 4 if vec4 else 1)), block=threads, grid=rows)
    return out


def train_plan(model, d, N, rows, nentity, env, fused):
    """plan_split (16-byte aligned tables)."""
    De, Dr = dims(model, d)
    return Dr % 4 == 0 and N <= 8192 and shape_ok(rows, N, De, d, model in CPLX, nentity, fused, env)


def expected_launch(model, mode, d, N, rows, nentity, env, sms):
    """What KGEModel.train_step with torch.optim.Adam launches on one GPU for a [rows, N] batch in `mode`.
    Returns dict(kernels=[((name, template args), block), ...] in launch order, fused_entity_adam=bool, ...);
    fused_entity_adam False means the dense gradient + kge_adam_step."""
    head = mode == "head-batch"
    fused = "KGE_KEEP_GRADS" not in env and train_plan(model, d, N, rows, nentity, env, True)
    r = launch_rows(model, head, d, N, rows, nentity, env, sms, do_loss=True, positive_loss=False,
                    want_adam=fused, workspace=True, gE=not fused)
    if fused and r["entity"] is None:
        raise AssertionError("kge_train_plan promised the fused entity optimizer but the launcher declined")
    kernels = [(r["row"], r["block"])]
    if not r["fused_positive"]:
        p = launch_rows(model, False, d, 1, rows, nentity, env, sms, do_loss=True, positive_loss=True,
                        want_adam=False, workspace=False, gE=True)
        kernels.append((p["row"], p["block"]))
    if r["entity"] is not None:
        kernels.append((r["entity"], r["entity_block"]))
    return dict(kernels=kernels, fused_entity_adam=fused, rows=r)


def expected_autograd(model, mode, d, N, rows, nentity, env, sms):
    """model(sample, mode) then .backward(): kge_score_forward and kge_score_backward."""
    head = mode == "head-batch"
    single = mode == "single"
    n = 1 if single else N
    f = launch_rows(model, head, d, n, rows, nentity, env, sms, do_loss=False, positive_loss=False, want_adam=False,
                    workspace=False, gE=False)
    b = launch_rows(model, head, d, n, rows, nentity, env, sms, do_loss=False, positive_loss=False, want_adam=False,
                    workspace=not single, gE=True)
    kernels = [(f["row"], f["block"]), (b["row"], b["block"])]
    if b["entity"] is not None:
        kernels.append((b["entity"], b["entity_block"]))
    return dict(kernels=kernels)


def reachable_instantiations():
    """Every row / entity kernel that launch_rows_model<MODEL> / launch_entity_model<MODEL> (kge_train_inst.cu, one
    translation unit per model) can launch: the launcher's dispatch, enumerated."""
    out = set()
    for model in MODELS:
        M, cplx = MODEL_ID[model], model in CPLX
        for h in (0, 1):
            for nch in ((4, 8) if cplx else (4, 8, 16)):
                for var in range(5):
                    out.add(("row_kernel_split", (M, h, nch, var)))
            out.add(("row_kernel_tma", (M, h)))
            for v in (4, 1):
                out.add(("row_kernel", (M, h, v)))
            for s in (1, 2):
                for fz in (0, 1):
                    out.add(("entity_kernel", (M, h, s, fz)))
    return out


# ---------------------------------------------------------------------------------------------------- case table
# A case: id, model, mode, d (hidden_dim: half the row of ComplEx / RotatE), N, B (rows; an int or a function of the
# SM count), nentity, env, and `data`, the input generator of the GPU test (see test_gpu_train_boundaries.make_inputs).
# reg (L3 coefficient), adv (self-adversarial alpha, 0 = uniform loss), steps (train steps compared).
class Case:
    def __init__(self, cid, model, mode, d, N, B, nentity, env=None, data="split", reg=0.0, adv=1.0, steps=2,
                 switch=()):
        self.id, self.model, self.mode, self.d, self.N, self.B = cid, model, mode, d, N, B
        self.nentity, self.env, self.data, self.reg, self.adv = nentity, dict(env or {}), data, reg, adv
        self.steps, self.switch = steps, switch

    def rows(self, sms):
        return self.B(sms) if callable(self.B) else self.B

    def launch(self, sms):
        return expected_launch(self.model, self.mode, self.d, self.N, self.rows(sms), self.nentity, self.env, sms)


MODES = ("head-batch", "tail-batch")
KEEP = {"KGE_KEEP_GRADS": "1"}


def _m(mode):
    return "h" if mode == "head-batch" else "t"


def _cases():
    cs = []
    # every row_kernel_split instantiation: each NCH at the smallest width above its lower boundary (unit counts
    # 33 / 129 / 257 = 1 mod 32 leave the most pad), each variant, all models, both modes; fused entity optimizer
    for model in MODELS:
        for mode in MODES:
            for nch, d in ((4, 132), (8, 516), (16, 1028)):
                if model in CPLX and nch == 16:
                    continue
                for var in range(5):
                    env = {} if var == 2 else {"KGE_SPLIT_VARIANT": str(var)}
                    cs.append(Case("split-%s-%s-nch%d-var%d" % (model, _m(mode), nch, var), model, mode, d, 32, 4,
                                   300, env))
    # the upper side of every width boundary (d/4 = 128, 256, 512), the rows too wide for the TMA ring (513 real,
    # 257 complex units: row_kernel<..., 4>) and rows that are not 16-byte multiples (row_kernel<..., 1>; RotatE
    # d = 1026 has entity_dim % 4 == 0 but an unaligned half row), default variant
    for model in MODELS:
        widths = (512, 1024, 1028, 1026) if model in CPLX else (512, 1024, 2048, 2052, 1026)
        for mode in MODES:
            for d in widths:
                cs.append(Case("width-%s-%s-d%d" % (model, _m(mode), d), model, mode, d, 32, 4, 300))
            # sparse pairs with dense gradients: the two-sweep TMA kernel + kge_adam_step
            cs.append(Case("sparse-%s-%s" % (model, _m(mode)), model, mode, 132, 32, 4, 3000, KEEP))
    # entity kernel: 63 / 64 / 65 units (one part; two parts, two of odd length upp = 33 / 32), fused and dense
    for model in MODELS:
        for mode in MODES:
            for units in (63, 64, 65):
                for keep in (False, True):
                    cs.append(Case("entity-%s-%s-u%d-%s" % (model, _m(mode), units, "dense" if keep else "fused"),
                                   model, mode, 4 * units, 64, 8, 80, KEEP if keep else {}))
    # tuning switches, one real and one complex model, both modes (the largest entity warp count is the default)
    switches = [("ring3", {"KGE_SPLIT_RING": "3"}), ("ring4", {"KGE_SPLIT_RING": "4"}),
                ("ctas2", {"KGE_SPLIT_CTAS": "2"}), ("parts1", {"KGE_ENTITY_PARTS": "1"}),
                ("ewarps1", {"KGE_ENTITY_WARPS": "1"}),
                ("edepth2", {"KGE_ENTITY_DEPTH": "2"}), ("edepth4", {"KGE_ENTITY_DEPTH": "4", "KGE_ENTITY_WARPS": "4"}),
                ("l2hints", {"KGE_L2_HINTS": "1"}), ("nosplit", {"KGE_NO_SPLIT": "1"}), ("notma", {"KGE_NO_TMA": "1"})]
    for name, env in switches:
        for model in ("TransE", "RotatE"):
            for mode in MODES:
                d, N = (132, 64) if name in ("ring3", "ring4", "ctas2") else (260, 32)
                cs.append(Case("switch-%s-%s-%s" % (name, model, _m(mode)), model, mode, d, N, 8, 200, env,
                               switch=tuple(env)))
    # candidate-list lengths: fewer candidates than warps (1-3, two-sweep and direct kernels), the split threshold
    # (7 / 8), the short-list warp rule (15 / 16 and 4 Ws - 1 / 4 Ws)
    for model, wsn in (("TransE", 64), ("RotatE", 48)):
        for i, N in enumerate((1, 2, 3, 7, 8, 15, 16, wsn - 1, wsn)):
            mode = MODES[i % 2]
            cs.append(Case("N%d-%s-%s" % (N, model, _m(mode)), model, mode, 132, N, 6, 30))
            if N <= 3:
                cs.append(Case("N%d-%s-%s-notma" % (N, model, _m(mode)), model, mode, 132, N, 6, 30,
                               {"KGE_NO_TMA": "1"}))
    # the plan's N <= 8192 limit at the widest row of each kind (the float64 reference gathers them in column blocks)
    for model, d in (("DistMult", 2048), ("ComplEx", 1024)):
        for N, B in ((8192, 2), (8193, 1)):
            cs.append(Case("Nlimit%d-%s" % (N, model), model, "tail-batch" if N % 2 else "head-batch", d, N, B, 4000,
                           steps=1))
    # persistent CTAs: one row, one row short of / exactly / one past one row per SM, two rows per SM plus one
    rowcounts = (("1", 1), ("sms-1", lambda s: s - 1), ("sms", lambda s: s), ("sms+1", lambda s: s + 1),
                 ("2sms+1", lambda s: 2 * s + 1))
    for model in ("TransE", "RotatE", "pRotatE"):
        for i, (name, B) in enumerate(rowcounts):
            mode = MODES[i % 2]
            cs.append(Case("rows%s-%s-%s" % (name, model, _m(mode)), model, mode, 132, 16, B, 400))
    # numerical edges
    for model in ("TransE", "RotatE"):
        for order in ("inc", "dec"):
            for adv in (8.0, 0.0):
                cs.append(Case("softmax-%s-%s-%s" % (order, "adv" if adv else "uniform", model), model, "tail-batch",
                               132, 64, 8, 600, data="order_" + order, adv=adv))
    for model in ("TransE", "DistMult", "pRotatE"):
        cs.append(Case("saturate-%s" % model, model, "head-batch", 132, 32, 8, 300, data="saturate"))
    for model in ("TransE", "RotatE", "pRotatE"):
        for mode in MODES:
            cs.append(Case("kink-equal-%s-%s" % (model, _m(mode)), model, mode, 132, 32, 8, 300, data="kink_equal"))
    for model in ("TransE", "pRotatE"):
        cs.append(Case("kink-partial-%s" % model, model, "tail-batch", 132, 32, 8, 300, data="kink_partial"))
    cs.append(Case("kink-tiny-RotatE", "RotatE", "tail-batch", 132, 32, 8, 300, data="kink_tiny"))
    for keep in (False, True):
        tag = "dense" if keep else "fused"
        env = KEEP if keep else {}
        cs.append(Case("segment-one-entity-%s" % tag, "RotatE", "head-batch", 132, 256, 40, 300, env, data="one_entity"))
        cs.append(Case("segment-duplicates-%s" % tag, "TransE", "tail-batch", 132, 64, 16, 40, env, data="duplicates"))
        cs.append(Case("segment-own-ids-%s" % tag, "ComplEx", "tail-batch", 132, 32, 8, 300, env, data="own_ids"))
        cs.append(Case("segment-sparse-%s" % tag, "DistMult", "head-batch", 260, 16, 8, 5000,
                       dict(env, KGE_FORCE_SPLIT="1"), data="split"))
    for model in ("RotatE", "ComplEx", "TransE"):
        cs.append(Case("l3-%s" % model, model, "tail-batch", 260, 32, 8, 300, reg=1e-3))
    return cs


CASES = _cases()

# autograd path: one width on each side of every NCH / TMA / alignment boundary, all models, all three modes
AUTOGRAD_WIDTHS = {"real": (132, 512, 516, 1024, 1028, 2048, 2052, 1026),
                   "cplx": (132, 512, 516, 1024, 1028, 1026)}
AUTOGRAD = [(model, d) for model in MODELS for d in AUTOGRAD_WIDTHS["cplx" if model in CPLX else "real"]]


# ---------------------------------------------------------------------------------------------------- CPU tests
def _dynamic_symbols(path):
    """Names in the .dynsym section of a 64-bit little-endian ELF shared object."""
    with open(path, "rb") as f:
        data = f.read()
    assert data[:4] == b"\x7fELF" and data[4] == 2 and data[5] == 1
    shoff, = struct.unpack_from("<Q", data, 0x28)
    shentsize, shnum = struct.unpack_from("<HH", data, 0x3A)
    secs = [struct.unpack_from("<IIQQQQIIQQ", data, shoff + i * shentsize) for i in range(shnum)]
    names = []
    for _, stype, _, _, off, size, link, _, _, entsize in secs:
        if stype != 11:                                  # SHT_DYNSYM
            continue
        stroff = secs[link][4]
        for k in range(size // entsize):
            st_name, = struct.unpack_from("<I", data, off + k * entsize)
            end = data.index(b"\0", stroff + st_name)
            names.append(data[stroff + st_name:end].decode())
    return names


def _parse_mangled(sym):
    """_ZN3kge16row_kernel_splitILi3ELb1ELi8ELi2EEEv... -> ('row_kernel_split', (3, 1, 8, 2))."""
    import re
    m = re.match(r"_ZN3kge(\d+)", sym)
    if not m:
        return None
    n, p = int(m.group(1)), m.end()
    name = sym[p:p + n]
    a = re.match(r"I((?:L[ib]\d+E)+)E", sym[p + n:])
    if not a:
        return None
    return name, tuple(int(v) for v in re.findall(r"L[ib](\d+)E", a.group(1)))


TRAIN_KERNELS = ("row_kernel_split", "row_kernel_tma", "row_kernel", "entity_kernel")


def test_library_instantiations_are_the_launchers_dispatch():
    """The row / entity kernels compiled into the library are exactly those the restated dispatch can launch."""
    from knowledgegraphembedding_b200 import build
    if not os.path.exists(build.LIB):
        pytest.skip("libkge_b200.so is not built")
    got = {k for k in map(_parse_mangled, _dynamic_symbols(build.LIB)) if k and k[0] in TRAIN_KERNELS}
    assert got == reachable_instantiations()


def test_case_table_reaches_every_instantiation():
    reached = {}
    for c in CASES:
        for kernel, _ in c.launch(B200_SMS)["kernels"]:
            reached.setdefault(kernel, c.id)
    for model, d in AUTOGRAD:
        for mode in ("single", "head-batch", "tail-batch"):
            for kernel, _ in expected_autograd(model, mode, d, 64, 8, 80, {}, B200_SMS)["kernels"]:
                reached.setdefault(kernel, "autograd")
    missing = sorted(reachable_instantiations() - set(reached))
    assert not missing, missing
    assert set(reached) <= reachable_instantiations()


def test_case_table_shapes():
    ids = [c.id for c in CASES]
    assert len(ids) == len(set(ids))
    for c in CASES:
        De, _ = dims(c.model, c.d)
        assert c.rows(B200_SMS) * c.N * De <= F64_BUDGET or c.id.startswith("Nlimit"), c.id
        c.launch(B200_SMS)                        # no case is one the launcher refuses


@pytest.mark.parametrize("case", [c for c in CASES if c.id.startswith("switch-")], ids=lambda c: c.id)
def test_every_switch_changes_the_launch(case):
    """A switch case that launched what the default launches would test nothing."""
    base = expected_launch(case.model, case.mode, case.d, case.N, case.rows(B200_SMS), case.nentity,
                           {k: v for k, v in case.env.items() if k not in case.switch}, B200_SMS)
    got = case.launch(B200_SMS)
    r, r0 = got["rows"], base["rows"]
    keys = ("row", "block", "ring", "ctas", "entity", "entity_block", "entity_depth")
    if case.env.get("KGE_L2_HINTS"):
        assert got["kernels"][0][0][0] == "row_kernel_split" and got["fused_entity_adam"]   # a flag of both kernels
    else:
        assert [r.get(k) for k in keys] != [r0.get(k) for k in keys]


def test_boundary_cases_land_where_they_claim():
    by = {c.id: c.launch(B200_SMS) for c in CASES}

    def row(cid):
        return by[cid]["kernels"][0]
    # NCH and TMA boundaries
    assert row("width-TransE-t-d512")[0] == ("row_kernel_split", (0, 0, 4, 2))
    assert row("split-TransE-t-nch8-var2")[0] == ("row_kernel_split", (0, 0, 8, 2))
    assert row("width-TransE-t-d1024")[0] == ("row_kernel_split", (0, 0, 8, 2))
    assert row("split-TransE-t-nch16-var2")[0] == ("row_kernel_split", (0, 0, 16, 2))
    assert row("width-TransE-t-d2048")[0] == ("row_kernel_split", (0, 0, 16, 2))
    assert row("width-TransE-t-d2052")[0] == ("row_kernel", (0, 0, 4))
    assert row("width-RotatE-h-d1024")[0] == ("row_kernel_split", (3, 1, 8, 2))
    assert row("width-RotatE-h-d1028")[0] == ("row_kernel", (3, 1, 4))
    assert row("width-RotatE-h-d1026")[0] == ("row_kernel", (3, 1, 1))
    # entity kernel parts
    assert by["entity-TransE-t-u63-fused"]["kernels"][-1][0] == ("entity_kernel", (0, 0, 1, 1))
    assert by["entity-TransE-t-u64-dense"]["kernels"][-1][0] == ("entity_kernel", (0, 0, 2, 0))
    assert by["entity-TransE-t-u65-fused"]["kernels"][-1][0] == ("entity_kernel", (0, 0, 2, 1))
    # N: the split threshold and the plan limit
    assert row("N7-TransE-t")[0][0] == "row_kernel_tma" and row("N8-TransE-h")[0][0] == "row_kernel_split"
    assert row("N3-TransE-h-notma") == (("row_kernel", (0, 1, 4)), 128)
    assert by["Nlimit8192-DistMult"]["fused_entity_adam"] and not by["Nlimit8193-DistMult"]["fused_entity_adam"]
    assert by["Nlimit8192-ComplEx"]["fused_entity_adam"] and not by["Nlimit8193-ComplEx"]["fused_entity_adam"]
    # the widest real row at N = 8192 keeps about 19 KB above the four warps the split kernel needs
    s = launch_rows("DistMult", False, 2048, 8192, 2, 4000, {}, B200_SMS, do_loss=True, positive_loss=False,
                    want_adam=True, workspace=True, gE=False)
    assert s["row"][0] == "row_kernel_split" and s["block"] == 5 * 32
    # persistent CTAs: grid = min(rows, SMs)
    assert by["rows2sms+1-TransE-h"]["rows"]["grid"] == B200_SMS
    assert by["rowssms-1-TransE-t"]["rows"]["grid"] == B200_SMS - 1
