#!/usr/bin/env python
"""Rank statistics rate (KGEModel.rank_statistics) at four BASELINE shapes, 4096 queries per mode, on the default path
of each model (two-stage RotatE / pRotatE, tcgen05 ComplEx, exact TransE), next to
  count       filtered_ranks on the same queries and path: the kernel it shares the query loop with;
  workaround  filtered_ranks(return_scores=True) with an empty filter list (exact kernel, [Q, nentity] raw scores), then
              the six counters with torch comparisons and the filter as a mask, end to end.
Kernel times are CUDA events around the count step (the same hook for both calls), the two calls alternated in one
process; end-to-end times are host clocks around whole calls ending in their host sync.  The statistics are checked
against the workaround's and against the filtered ranks on the timed inputs.  Prints the card's name and power limit
first, then one JSON line per shape and mode.

    python tools/rank_stats_rate.py [--reps 5] [--out FILE]
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
    ("pRotatE FB15k", "pRotatE", 14951, 1345, 1000, 24.0, False, False, 483142),
    ("ComplEx wn18rr", "ComplEx", 40943, 11, 500, 200.0, True, True, 86835),
    ("TransE FB15k-237", "TransE", 14541, 237, 1000, 9.0, False, False, 272115),
]
NQ = 4096
PATHS = {"RotatE": "two-stage", "pRotatE": "two-stage", "ComplEx": "tcgen05", "TransE": "exact"}
NO_TRIPLES = []             # one object: the model caches the filter index per list object


def kernel_ms(m, fn):
    m._ws["eval_events"] = events = []
    fn()
    torch.cuda.synchronize()
    m._ws["eval_events"] = None
    return sum(a.elapsed_time(b) for a, b in events)


def e2e_s(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("tools/rank_stats_rate.py measures on the GPU; no CUDA device found")
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
            count = lambda: m.filtered_ranks(queries, all_true, mode)            # noqa: E731
            stats = lambda: m.rank_statistics(queries, all_true, mode)           # noqa: E731
            ranks, got = count(), stats()                                        # warm-up (modules, buffers, index)
            assert np.array_equal(1 + got[:, 0] + got[:, 1], ranks), (name, mode)
            off, ent = index.csr(queries, mode)
            mask = torch.zeros((NQ, nentity), dtype=torch.bool)
            mask[torch.from_numpy(np.repeat(np.arange(NQ), np.diff(off))), torch.from_numpy(ent.astype(np.int64))] = True
            mask = mask.cuda()
            pos = torch.tensor([q[0] if mode == "head-batch" else q[2] for q in queries], device="cuda")
            j = torch.arange(nentity, device="cuda")[None, :]
            before, after = j < pos[:, None], j > pos[:, None]

            def workaround():
                s = m.filtered_ranks(queries, NO_TRIPLES, mode, return_scores=True)[1]
                sp = s.gather(1, pos[:, None])
                gt, eq = s > sp, s == sp
                eb, ea, kept = eq & before, eq & after, ~mask
                cols = (gt & kept, eb & kept, ea & kept, gt, eb, ea)
                return torch.stack([c.sum(1) for c in cols], 1).cpu().numpy()

            assert np.array_equal(workaround(), got), (name, mode)
            ks, kc, es, ec, ew = [], [], [], [], []
            for _ in range(args.reps):                                           # alternated: count, stats
                kc.append(kernel_ms(m, count))
                ks.append(kernel_ms(m, stats))
            for _ in range(args.reps):
                ec.append(e2e_s(count)[0])
                es.append(e2e_s(stats)[0])
                ew.append(e2e_s(workaround)[0])
            ks_m, kc_m = float(np.median(ks)), float(np.median(kc))
            row = {"shape": name, "mode": mode, "queries": NQ,
                   "path": PATHS[model],
                   "stats_kernel_ms": round(ks_m, 3), "count_kernel_ms": round(kc_m, 3),
                   "kernel_ratio": round(ks_m / kc_m, 3),
                   "stats_kernel_ms_range": [round(min(ks), 3), round(max(ks), 3)],
                   "count_kernel_ms_range": [round(min(kc), 3), round(max(kc), 3)],
                   "stats_e2e_ms": round(1e3 * float(np.median(es)), 3),
                   "count_e2e_ms": round(1e3 * float(np.median(ec)), 3),
                   "workaround_e2e_ms": round(1e3 * float(np.median(ew)), 3),
                   "speedup_vs_workaround": round(float(np.median(ew)) / float(np.median(es)), 2),
                   "raw_ties_per_query": round(float((got[:, 4] + got[:, 5]).mean()), 3)}
            print(json.dumps(row), flush=True)
            rows.append(row)
            del mask, before, after
            torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()
