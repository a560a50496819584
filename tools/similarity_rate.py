#!/usr/bin/env python
"""Similarity search rate (KGEModel.nearest_neighbors) over four entity tables and one relation table, 4096 id queries,
k = 10 / 100, all four metrics, next to two references on the same shapes:
  topk        predict_topk's kernel (kge_eval_topk + merge) on a DistMult table of the same rows and width, kernel-only:
              the same tile loop with the link-prediction epilogue;
  workaround  the torch route a user takes without this call: X[ids] @ X.T (cosine: of the normalised rows) or
              torch.cdist (l2, l1), the self column set to -inf, then torch.topk; TF32 off.  End to end.
nearest_neighbors is timed end to end and kernel-only (CUDA events around kge_similarity_topk + kge_eval_topk_merge); the
cost per (query, row) pair is kernel time / (queries x rows).  Every timed result is checked on a subset of queries
against a stable descending sort of the exact score matrix of tests/similarity_oracle.c.  Prints the card's name and
power limit first, then one JSON line per configuration.

    python tools/similarity_rate.py [--reps 3] [--check 32] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from knowledgegraphembedding_b200 import KGEModel  # noqa: E402
import similarity_oracle as SO  # noqa: E402

SHAPES = [  # name, model, nentity, nrelation, hidden_dim, -de, -dr, table
    ("RotatE FB15k entities", "RotatE", 14951, 1345, 1000, True, False, "entity"),        # width 2000
    ("TransE FB15k-237 entities", "TransE", 14541, 237, 1000, False, False, "entity"),
    ("ComplEx wn18rr entities", "ComplEx", 40943, 11, 500, True, True, "entity"),
    ("RotatE YAGO3-10 entities", "RotatE", 123182, 37, 500, True, False, "entity"),
    ("RotatE FB15k relations", "RotatE", 14951, 1345, 1000, True, False, "relation"),     # 1345 x 1000
]
NQ, KS, METRICS = 4096, (10, 100), ("dot", "cosine", "l2", "l1")


def timed(fn, reps):
    fn()                                                   # warm-up (modules, buffers)
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


def workaround(X, ids, metric, k):
    q = X[ids]
    if metric == "dot":
        s = q @ X.T
    elif metric == "cosine":
        s = torch.nn.functional.normalize(q, dim=1) @ torch.nn.functional.normalize(X, dim=1).T
    else:
        s = -torch.cdist(q, X, p=2.0 if metric == "l2" else 1.0)
    s[torch.arange(len(ids), device=X.device), ids] = float("-inf")
    return torch.topk(s, k, dim=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--check", type=int, default=32, help="queries checked against the reference per configuration")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("tools/similarity_rate.py measures on the GPU; no CUDA device found")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    card = torch.cuda.get_device_name(0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    header = {"device": card, "nvidia_smi": smi[:2]}
    print(json.dumps(header), flush=True)
    rows_out = [header]
    for name, model, nentity, nrel, dim, de, dr, table in SHAPES:
        torch.manual_seed(0)
        m = KGEModel(model, nentity, nrel, dim, 12.0, double_entity_embedding=de, double_relation_embedding=dr).cuda()
        X = (m.entity_embedding if table == "entity" else m.relation_embedding).detach()
        rows, width = X.shape
        ids = torch.from_numpy(np.random.RandomState(1).randint(rows, size=NQ)).cuda()
        sub = ids[:args.check].cpu().numpy()
        Xh = X.cpu().numpy()
        # predict_topk's kernel on a DistMult table of the same rows and width (OP_MUL, the dot-product tile loop)
        ref = KGEModel("DistMult", rows, 7, width, 12.0).cuda()
        queries = np.stack([np.arange(NQ) % rows, np.arange(NQ) % 7, np.zeros(NQ, dtype=np.int64)], 1)
        for metric in METRICS:
            want_ids, want_scores = SO.topk(SO.similarity(Xh, Xh[sub], metric), max(KS), sub)
            for k in KS:
                call = lambda: m.nearest_neighbors(ids, table=table, k=k, metric=metric)     # noqa: E731
                e2e_s, (got_ids, got_scores) = timed(call, args.reps)
                assert np.array_equal(got_ids[:len(sub)].cpu().numpy(), want_ids[:, :k]), (name, metric, k)
                got = got_scores[:len(sub)].cpu().numpy()
                assert np.array_equal(got.view(np.uint32), want_scores[:, :k].view(np.uint32)), (name, metric, k)
                nn_ms = kernel_ms(m, "nn_events", call, args.reps)
                topk_ms = kernel_ms(ref, "topk_events", lambda: ref.predict_topk(queries, "tail-batch", k=k), args.reps)
                wa_s, _ = timed(lambda: workaround(X, ids, metric, k), args.reps)
                pairs = NQ * rows
                row = {"shape": name, "rows": rows, "width": width, "metric": metric, "k": k, "queries": NQ,
                       "kernel_ms": round(nn_ms, 3), "ps_per_pair": round(1e9 * nn_ms / pairs, 2),
                       "predict_topk_kernel_ms": round(topk_ms, 3),
                       "predict_topk_ps_per_pair": round(1e9 * topk_ms / pairs, 2),
                       "e2e_ms": round(1e3 * e2e_s, 3), "workaround_e2e_ms": round(1e3 * wa_s, 3),
                       "speedup_vs_workaround": round(wa_s / e2e_s, 2)}
                print(json.dumps(row), flush=True)
                rows_out.append(row)
        del m, ref, X
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rows_out, f, indent=1)


if __name__ == "__main__":
    main()
