#!/usr/bin/env python
"""Top-k link prediction rate (KGEModel.predict_topk) at three BASELINE shapes, 4096 queries per mode, k = 10/100/256,
with and without exclude_triples, next to two references on the same queries:
  count    the exact count kernel of the filtered ranking (filtered_ranks(..., exact=True)), kernel-only;
  workaround  filtered_ranks(return_scores=True), excluded columns masked, then torch.topk, end to end.
predict_topk is timed end to end and kernel-only (CUDA events around kge_eval_topk + kge_eval_topk_merge).  On the timed
inputs its result is checked against a stable descending sort of the exact score matrix with the excluded columns
removed.  Prints the card's name and power limit first, then one JSON line per configuration.

    python tools/topk_rate.py [--reps 3] [--out FILE]
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

SHAPES = [  # name, model, nentity, nrelation, hidden_dim, gamma, -de, -dr, true triples (synthetic, as many as the dataset)
    ("RotatE FB15k", "RotatE", 14951, 1345, 1000, 24.0, True, False, 483142),
    ("ComplEx wn18rr", "ComplEx", 40943, 11, 500, 200.0, True, True, 86835),
    ("TransE FB15k-237", "TransE", 14541, 237, 1000, 9.0, False, False, 272115),
]
NQ, KS = 4096, (10, 100, 256)
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("tools/topk_rate.py measures on the GPU; no CUDA device found")
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
        index = FilterIndex(all_true, nentity, nrel)
        for mode in ("head-batch", "tail-batch"):
            count_ms = kernel_ms(m, "eval_events", lambda: m.filtered_ranks(queries, all_true, mode, exact=True),
                                 args.reps)
            raw = m.filtered_ranks(queries, NO_TRIPLES, mode, return_scores=True)[1]     # exact scores, nothing filtered
            off, ent = index.csr(queries, mode)
            mask = torch.zeros((NQ, nentity), dtype=torch.bool)
            mask[torch.from_numpy(np.repeat(np.arange(NQ), np.diff(off))), torch.from_numpy(ent.astype(np.int64))] = True
            mask = mask.cuda()
            for exclude in (None, all_true):
                masked = raw.masked_fill(mask, float("-inf")) if exclude is not None else raw
                order_vals, order_ids = torch.sort(masked, dim=1, descending=True, stable=True)
                for k in KS:
                    e2e_s, (ids, scores) = timed(lambda: m.predict_topk(queries, mode, k=k, exclude_triples=exclude),
                                                 args.reps)
                    assert torch.equal(ids, order_ids[:, :k]), (name, mode, k)
                    assert torch.equal(scores, order_vals[:, :k]), (name, mode, k)
                    topk_ms = kernel_ms(m, "topk_events",
                                        lambda: m.predict_topk(queries, mode, k=k, exclude_triples=exclude), args.reps)

                    def workaround():
                        filt = all_true if exclude is not None else NO_TRIPLES
                        s = m.filtered_ranks(queries, filt, mode, return_scores=True)[1]
                        if exclude is not None:
                            s.masked_fill_(mask, float("-inf"))
                        return torch.topk(s, k, dim=1)

                    wa_s, _ = timed(workaround, args.reps)
                    row = {"shape": name, "mode": mode, "k": k, "exclude": exclude is not None, "queries": NQ,
                           "topk_kernel_ms": round(topk_ms, 3), "count_kernel_ms": round(count_ms, 3),
                           "ratio_to_count": round(topk_ms / count_ms, 3),
                           "topk_e2e_ms": round(1e3 * e2e_s, 3), "topk_queries_per_s": round(NQ / e2e_s),
                           "workaround_e2e_ms": round(1e3 * wa_s, 3), "speedup_vs_workaround": round(wa_s / e2e_s, 2)}
                    print(json.dumps(row), flush=True)
                    rows.append(row)
                del masked, order_vals, order_ids
            del raw, mask
            torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()
