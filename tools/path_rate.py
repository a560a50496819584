#!/usr/bin/env python
"""Path-query rate (KGEModel.path_rank_statistics) at four dataset shapes, on seeded synthetic graphs with skewed (Zipf)
degrees and as many triples as the dataset (nothing is downloaded), with 4096 random-walk queries per mode at L = 1, 2, 3
on the default counting path of each model.  Per shape, mode and L it prints
  fold_ms           kge_eval_path_query_vectors of the 4096 queries;
  traversal_ms      the answer-set traversal (kge_eval_path_bits_dense, all hops) and traversal_ms_per_hop;
  count_kernel_ms   the count / stats kernel of the call (CUDA events of the eval_events hook), beside
  one_hop_kernel_ms the same kernel in rank_statistics on 4096 one-hop queries of the same graph;
  path_e2e_ms / one_hop_e2e_ms  both calls end to end (host clock around the call, which ends in its host sync).
Device times are CUDA events, medians over --reps; the card's name and power limit come first, then one JSON line per row.
At L = 1 the statistics are checked against rank_statistics on the same queries.

    python tools/path_rate.py [--reps 5] [--out FILE]
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
from knowledgegraphembedding_b200 import KGEModel, _lib  # noqa: E402
from knowledgegraphembedding_b200.model import _stream  # noqa: E402

SHAPES = [  # name, model, nentity, nrelation, hidden_dim, gamma, -de, -dr, triples
    ("TransE FB15k-237", "TransE", 14541, 237, 1000, 9.0, False, False, 272115),
    ("RotatE FB15k", "RotatE", 14951, 1345, 1000, 24.0, True, False, 483142),
    ("ComplEx wn18rr", "ComplEx", 40943, 11, 500, 200.0, True, True, 86835),
    ("RotatE YAGO3-10", "RotatE", 123182, 37, 500, 24.0, True, False, 1079040),
]
NQ = 4096


def skewed_graph(nentity, nrel, n, seed):
    """n distinct triples with Zipf(1.2) head, relation and tail ranks over shuffled ids (hubs with thousands of edges)."""
    rng = np.random.RandomState(seed)
    perm_e, perm_r = rng.permutation(nentity), rng.permutation(nrel)
    got = np.zeros((0, 3), dtype=np.int64)
    while got.shape[0] < n:
        m = 2 * (n - got.shape[0])
        h = perm_e[(rng.zipf(1.2, m) - 1) % nentity]
        r = perm_r[(rng.zipf(1.2, m) - 1) % nrel]
        t = perm_e[(rng.zipf(1.2, m) - 1) % nentity]
        got = np.unique(np.concatenate([got, np.stack([h, r, t], 1)]), axis=0)
    return got[rng.permutation(got.shape[0])[:n]]


def random_walks(tri, L, mode, rng):
    """NQ walks of L hops along the graph, each hop along a random edge at the current entity (inverted when the walk
    takes it backwards); answers are where the walks end."""
    nrel = int(tri[:, 1].max()) + 1
    out = {}
    for h, r, t in tri:
        out.setdefault(int(h), []).append((int(r), int(t)))
        out.setdefault(int(t), []).append((int(r) + nrel, int(h)))
    starts = list(out)
    anchors, paths, answers = [], [], []
    while len(anchors) < NQ:
        a = e = starts[rng.randint(len(starts))]
        hops = []
        for _ in range(L):
            hop, e = out[e][rng.randint(len(out[e]))]
            hops.append(hop)
        anchors.append(a)
        paths.append(hops)
        answers.append(e)
    paths = np.array(paths, dtype=np.int64)
    if mode == "head-batch":       # the same walk read backwards: (?, reversed path, end), answer = start
        anchors, answers = answers, anchors
        paths = np.where(paths >= nrel, paths - nrel, paths + nrel)[:, ::-1].copy()
    return np.array(anchors), paths, np.array(answers)


def events_ms(fn, reps):
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b))
    return float(np.median(out))


def hook_ms(m, fn):
    m._ws["eval_events"] = events = []
    fn()
    torch.cuda.synchronize()
    m._ws["eval_events"] = None
    return sum(a.elapsed_time(b) for a, b in events)


def e2e_ms(fn, reps):
    out = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        out.append(1e3 * (time.perf_counter() - t0))
    return float(np.median(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("tools/path_rate.py measures on the GPU; no CUDA device found")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    header = {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi[:2]}
    print(json.dumps(header), flush=True)
    rows = [header]
    for name, model, nentity, nrel, dim, gamma, de, dr, ntrue in SHAPES:
        torch.manual_seed(0)
        m = KGEModel(model, nentity, nrel, dim, gamma, double_entity_embedding=de, double_relation_embedding=dr).cuda()
        tri = skewed_graph(nentity, nrel, ntrue, seed=1)
        triples = [tuple(int(v) for v in row) for row in tri]
        rng = np.random.RandomState(2)
        dev = m.entity_embedding.device
        st = _stream(dev)
        words = (nentity + 31) // 32
        for mode in ("head-batch", "tail-batch"):
            one = np.asarray(triples, dtype=np.int64)[rng.choice(len(triples), NQ, replace=False)]
            one_list = [tuple(int(v) for v in row) for row in one]
            m.rank_statistics(one_list, triples, mode)                            # warm-up (modules, index)
            one_kernel = hook_ms(m, lambda: m.rank_statistics(one_list, triples, mode))
            one_e2e = e2e_ms(lambda: m.rank_statistics(one_list, triples, mode), args.reps)
            for L in (1, 2, 3):
                anchors, paths, answers = random_walks(tri, L, mode, rng)
                got = m.path_rank_statistics(anchors, paths, answers, triples, mode)     # warm-up
                if L == 1:                                   # forward hops: the one-hop call's numbers
                    fw = paths[:, 0] < nrel
                    q = np.zeros((int(fw.sum()), 3), dtype=np.int64)
                    q[:, 1] = paths[fw, 0]
                    q[:, 0 if mode == "head-batch" else 2] = answers[fw]
                    q[:, 2 if mode == "head-batch" else 0] = anchors[fw]
                    assert np.array_equal(got[fw], m.rank_statistics([tuple(r) for r in q.tolist()], triples, mode))
                path, _ = m._path_queries(anchors, paths, mode, triples)
                desc, err, mid = m._descriptor(), m._err_flag(), _lib.MODE_IDS[mode]
                qvec = torch.empty(NQ * m.entity_dim, device=dev)
                bits = torch.empty(NQ * words, dtype=torch.int32, device=dev)
                fold = events_ms(lambda: m._path_chunk(path, 0, NQ, mid, desc, None, qvec, None, err, st), args.reps)
                both = events_ms(lambda: m._path_chunk(path, 0, NQ, mid, desc, bits, qvec, None, err, st), args.reps)
                kernel = hook_ms(m, lambda: m.path_rank_statistics(anchors, paths, answers, triples, mode))
                e2e = e2e_ms(lambda: m.path_rank_statistics(anchors, paths, answers, triples, mode), args.reps)
                row = {"shape": name, "mode": mode, "L": L, "queries": NQ,
                       "mean_answers": round(float(m.path_rank_statistics(
                           anchors, paths, answers, triples, mode, return_answer_counts=True)[1].mean()), 1),
                       "fold_ms": round(fold, 3), "traversal_ms": round(both - fold, 3),
                       "traversal_ms_per_hop": round((both - fold) / L, 3),
                       "count_kernel_ms": round(kernel, 3), "one_hop_kernel_ms": round(one_kernel, 3),
                       "path_e2e_ms": round(e2e, 3), "one_hop_e2e_ms": round(one_e2e, 3)}
                print(json.dumps(row), flush=True)
                rows.append(row)
        m._ws.clear()
        del m
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()
