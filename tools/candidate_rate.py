#!/usr/bin/env python
"""Candidate-list ranking rate (KGEModel.candidate_rank_statistics): 4096 queries per mode against C = 500 and 1000
random candidates each, with and without exclude_triples, at five shapes -- four BASELINE ones (the YAGO3-10 table,
493 MB, is larger than the 126 MB L2) and a synthetic ogbl-wikikg2-sized RotatE (2,500,604 entities, 535 relations,
d = 100, a 2 GB table).  Per configuration:
  kernel      CUDA events around kge_eval_candidate_rank_stats (summed over the call's query chunks), pairs/s, and the
              gathered row bytes per second against the project's HBM copy peak (6468.6 GB/s) and the L2-gather ceiling
              (15.8 TB/s, DESIGN.md section 3.1);
  tile        the exact all-entity tile kernel's cost per pair (filtered_ranks(..., exact=True) on the same queries),
              where all-entity ranking is feasible;
  e2e         host clock around the whole call, ending in its host sync;
  workaround  model((positive, candidates), mode) and model(positive) (the training row kernels, no filter), then the
              six counters with torch comparisons, end to end.
Each timed result is checked against the canonical scores of a query sample: filtered_ranks(..., return_scores=True)
gathered at the candidate ids, with the exclusion as a mask.  The true-triple lists are synthetic (bench.py's
generator); the wikikg2 shape uses 2 M of them.  Prints the card's name and power limit first, then one JSON line per
configuration.

    python tools/candidate_rate.py [--reps 5] [--shapes all|small] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from knowledgegraphembedding_b200 import FilterIndex, KGEModel  # noqa: E402

SHAPES = [  # name, model, nentity, nrelation, hidden_dim, gamma, -de, -dr, true triples, all-entity tile reference
    ("RotatE FB15k", "RotatE", 14951, 1345, 1000, 24.0, True, False, 483142, True),
    ("TransE FB15k-237", "TransE", 14541, 237, 1000, 9.0, False, False, 272115, True),
    ("ComplEx wn18rr", "ComplEx", 40943, 11, 500, 200.0, True, True, 86835, True),
    ("RotatE YAGO3-10", "RotatE", 123182, 37, 500, 24.0, True, False, 1079040, True),
    ("RotatE wikikg2-size", "RotatE", 2500604, 535, 100, 24.0, True, False, 2000000, False),
]
NQ, CS, SAMPLE = 4096, (500, 1000), 32
HBM_COPY_GBS, L2_GATHER_GBS = 6468.6, 15800.0


def kernel_ms(m, key, fn, reps):
    fn()
    m._ws[key] = events = []
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    m._ws[key] = None
    return sum(a.elapsed_time(b) for a, b in events) / reps


def e2e_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        out = fn()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0) / reps, out


def sample_stats(m, queries, cand, mode, index):
    """numpy counts of the first SAMPLE queries over filtered_ranks' exact raw scores at the listed ids."""
    test = queries[:SAMPLE]
    _, sc = m.filtered_ranks(test, [], mode, return_scores=True)
    c = cand[:SAMPLE].to(sc.device)
    s = sc.gather(1, c).cpu().numpy()
    pos = np.array([q[0] if mode == "head-batch" else q[2] for q in test])
    sp = sc[torch.arange(len(test)), torch.from_numpy(pos).to(sc.device)].cpu().numpy()[:, None]
    cn = c.cpu().numpy()
    other = cn != pos[:, None]
    kept = np.ones_like(other)
    if index is not None:
        off, ent = index.csr(test, mode)
        for q in range(len(test)):
            kept[q] = ~np.isin(cn[q], ent[off[q]:off[q + 1]])
    with np.errstate(invalid="ignore"):
        gt, eq = (s > sp) & other, (s == sp) & other
    before, after = cn < pos[:, None], cn > pos[:, None]
    cols = [gt & kept, eq & before & kept, eq & after & kept, gt, eq & before, eq & after]
    return np.stack([x.sum(1) for x in cols], 1).astype(np.int64)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--shapes", choices=("all", "small"), default="all")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("tools/candidate_rate.py measures on the GPU; no CUDA device found")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    header = {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi[:2]}
    print(json.dumps(header), flush=True)
    rows = [header]
    shapes = SHAPES if args.shapes == "all" else SHAPES[:1]
    for name, model, nentity, nrel, dim, gamma, de, dr, ntrue, tile_ref in shapes:
        torch.manual_seed(0)
        m = KGEModel(model, nentity, nrel, dim, gamma, double_entity_embedding=de, double_relation_embedding=dr).cuda()
        row_bytes = 4 * m.entity_dim
        all_true, rng = bench.synthetic_triples(nentity, nrel, ntrue, seed=2)
        queries = [all_true[i] for i in rng.choice(len(all_true), NQ, replace=False)]
        index = FilterIndex(all_true, nentity, nrel)
        gen = torch.Generator(device="cuda").manual_seed(3)
        for mode in ("head-batch", "tail-batch"):
            head = mode == "head-batch"
            tile_ns = None
            if tile_ref:
                tile_ms = kernel_ms(m, "eval_events", lambda: m.filtered_ranks(queries, [], mode, exact=True), args.reps)
                tile_ns = 1e6 * tile_ms / (NQ * nentity)
            pos_sample = torch.tensor(queries, dtype=torch.int64, device="cuda")
            for C in CS:
                cand = torch.randint(nentity, (NQ, C), generator=gen, device="cuda", dtype=torch.int64)

                def workaround():
                    with torch.no_grad():
                        s = m((pos_sample, cand), mode)
                        sp = m(pos_sample)
                    p = pos_sample[:, 0 if head else 2][:, None]
                    other = cand != p
                    gt, eq = (s > sp) & other, (s == sp) & other
                    eb, ea = eq & (cand < p), eq & (cand > p)
                    return torch.stack([x.sum(1) for x in (gt, eb, ea)], 1).cpu().numpy()

                w_ms, _ = e2e_ms(workaround, args.reps)
                for excl in (False, True):
                    ex = all_true if excl else None
                    call = lambda: m.candidate_rank_statistics(queries, cand, mode, exclude_triples=ex)   # noqa: E731
                    k_ms = kernel_ms(m, "candidate_events", call, args.reps)
                    c_ms, got = e2e_ms(call, args.reps)
                    want = sample_stats(m, queries, cand, mode, index if excl else None)
                    assert np.array_equal(got[:SAMPLE], want), (name, mode, C, excl)
                    pairs = NQ * C
                    gbs = pairs * row_bytes / (k_ms * 1e6)
                    row = {"shape": name, "mode": mode, "queries": NQ, "candidates": C, "exclude": excl,
                           "d": m.entity_dim // (2 if de else 1), "row_bytes": row_bytes,
                           "kernel_ms": round(k_ms, 4), "pairs_per_s": float("%.4g" % (pairs / (k_ms * 1e-3))),
                           "gathered_GBs": round(gbs, 1), "of_hbm_copy_peak": round(gbs / HBM_COPY_GBS, 3),
                           "of_l2_gather_ceiling": round(gbs / L2_GATHER_GBS, 3),
                           "ns_per_pair": round(1e6 * k_ms / pairs, 5),
                           "tile_ns_per_pair": round(tile_ns, 5) if tile_ns is not None else None,
                           "e2e_ms": round(c_ms, 3), "workaround_e2e_ms": round(w_ms, 3),
                           "speedup_vs_workaround": round(w_ms / c_ms, 2), "sample_checked": SAMPLE}
                    print(json.dumps(row), flush=True)
                    rows.append(row)
                del cand
        del m
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()
