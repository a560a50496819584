#!/usr/bin/env python
"""Relation prediction rate (KGEModel.filtered_relation_ranks / predict_relations) at four BASELINE shapes, 4096 seeded
synthetic queries (h, r, t) drawn from as many synthetic true triples as the dataset has, next to two references:
  entity   the exact count kernel of the tail-batch entity ranking at the same model and d (filtered_ranks(...,
           exact=True)), kernel-only: its time per (query, entity) pair beside the relation kernel's per (query, relation);
  forward  the workaround without this feature: model(sample) in 'single' mode over every (h, r', t), then the
           filtered ranks in torch (the [Q, nrelation] filter mask is built beforehand and not timed), end to end.
The relation kernel is timed with CUDA events (kge_eval_relation_count_ranks; kge_eval_relation_topk + merge for the
top-k); filtered_relation_ranks and predict_relations(k=10) end to end.  Every timed result is checked against a stable
descending sort of the dumped exact scores.  Prints the card's name and power limit first, then one JSON line per shape.

    python tools/relation_rate.py [--reps 5] [--out FILE]
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
from knowledgegraphembedding_b200 import KGEModel  # noqa: E402

SHAPES = [  # name, model, nentity, nrelation, hidden_dim, gamma, -de, -dr, true triples (synthetic, as many as the dataset)
    ("RotatE FB15k", "RotatE", 14951, 1345, 1000, 24.0, True, False, 483142),
    ("TransE FB15k-237", "TransE", 14541, 237, 1000, 9.0, False, False, 272115),
    ("ComplEx wn18rr", "ComplEx", 40943, 11, 500, 200.0, True, True, 86835),
    ("RotatE YAGO3-10", "RotatE", 123182, 37, 500, 24.0, True, False, 1079040),
]
NQ, K = 4096, 10
NO_TRIPLES = []             # one object: the model caches the filter index per list object


def timed(fn, reps):
    fn()                                                   # warm-up (modules, buffers, filter index)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps, out


def kernel_ms(m, key, fn, reps):
    fn()
    m._ws[key] = events = []
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    m._ws[key] = None
    return sum(a.elapsed_time(b) for a, b in events) / reps


def relation_mask(triples, queries, nrel):
    by_pair = {}
    for h, r, t in triples:
        by_pair.setdefault((h, t), []).append(r)
    mask = np.zeros((len(queries), nrel), dtype=bool)
    for i, (h, _, t) in enumerate(queries):
        mask[i, by_pair.get((h, t), [])] = True
    return torch.from_numpy(mask).cuda()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("tools/relation_rate.py measures on the GPU; no CUDA device found")
    card = torch.cuda.get_device_name(0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    header = {"device": card, "nvidia_smi": smi[:2]}
    print(json.dumps(header), flush=True)
    rows = [header]
    for name, model, nentity, nrel, dim, gamma, de, dr, ntrue in SHAPES:
        torch.manual_seed(0)
        m = KGEModel(model, nentity, nrel, dim, gamma, double_entity_embedding=de, double_relation_embedding=dr).cuda()
        all_true, rng = bench.synthetic_triples(nentity, nrel, ntrue, seed=2)
        queries = [all_true[i] for i in rng.choice(len(all_true), NQ, replace=False)]
        q_dev = torch.tensor(queries, dtype=torch.int64, device="cuda")
        cols = torch.arange(nrel, device="cuda")
        filt = relation_mask(all_true, queries, nrel) & (cols[None, :] != q_dev[:, 1:2])     # r' != r
        with torch.no_grad():
            # ---- relation kernel and entity count kernel, kernel-only -----------------------------------------------
            rel_ms = kernel_ms(m, "relation_events", lambda: m.filtered_relation_ranks(queries, all_true), args.reps)
            ent_ms = kernel_ms(m, "eval_events", lambda: m.filtered_ranks(queries, all_true, "tail-batch", exact=True),
                               args.reps)
            topk_ms = kernel_ms(m, "relation_topk_events",
                                lambda: m.predict_relations(queries, k=K, exclude_triples=all_true), args.reps)
            # ---- end to end, checked against a stable sort of the dumped exact scores ----------------------------------
            ranks_s, ranks = timed(lambda: m.filtered_relation_ranks(queries, all_true), args.reps)
            dumped = m.filtered_relation_ranks(queries, all_true, return_scores=True)[1]   # filtered: s_pos - 1
            order = torch.sort(dumped, dim=1, descending=True, stable=True)[1]
            want = (order == q_dev[:, 1:2]).int().argmax(dim=1) + 1
            assert np.array_equal(ranks, want.cpu().numpy()), name
            raw = m.filtered_relation_ranks(queries, NO_TRIPLES, return_scores=True)[1]
            excluded = relation_mask(all_true, queries, nrel)            # every true (h, r', t), r' = r included
            vals, ids_want = torch.sort(raw.masked_fill(excluded, float("-inf")), dim=1, descending=True, stable=True)
            ids_want = torch.where(torch.isneginf(vals), torch.full_like(ids_want, -1), ids_want)   # padding slots
            topk_s, (ids, scores) = timed(lambda: m.predict_relations(queries, k=K, exclude_triples=all_true),
                                          args.reps)
            assert torch.equal(ids, ids_want[:, :K]), name
            assert torch.equal(scores, vals[:, :K]), name

            # ---- the workaround: model(sample) over every (h, r', t), ranks in torch ------------------------------------
            def forward_ranks():
                sample = q_dev.repeat_interleave(nrel, dim=0)
                sample[:, 1] = cols.repeat(NQ)
                s = m(sample).view(NQ, nrel)
                sp = s.gather(1, q_dev[:, 1:2])
                beat = ((s > sp) | ((s == sp) & (cols[None, :] < q_dev[:, 1:2]))) & ~filt
                beat &= cols[None, :] != q_dev[:, 1:2]
                return beat.sum(dim=1) + 1

            fwd_s, fwd_ranks = timed(forward_ranks, args.reps)
            mismatch = int((fwd_ranks.cpu().numpy() != ranks).sum())
        pairs_rel, pairs_ent = NQ * nrel, NQ * nentity
        row = {"shape": name, "queries": NQ, "nrelation": nrel, "dim": dim,
               "relation_kernel_ms": round(rel_ms, 4), "ns_per_query_relation": round(1e6 * rel_ms / pairs_rel, 4),
               "entity_count_kernel_ms": round(ent_ms, 3), "ns_per_query_entity": round(1e6 * ent_ms / pairs_ent, 4),
               "pair_cost_ratio": round((rel_ms / pairs_rel) / (ent_ms / pairs_ent), 2),
               "relation_topk10_kernel_ms": round(topk_ms, 4),
               "filtered_relation_ranks_e2e_ms": round(1e3 * ranks_s, 3),
               "predict_relations_k10_e2e_ms": round(1e3 * topk_s, 3),
               "forward_workaround_e2e_ms": round(1e3 * fwd_s, 3),
               "speedup_vs_forward": round(fwd_s / ranks_s, 2),
               "forward_rank_mismatches": mismatch}
        print(json.dumps(row), flush=True)
        rows.append(row)
        del m, raw, dumped, order
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()
