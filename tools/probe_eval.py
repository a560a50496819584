#!/usr/bin/env python
"""Time the evaluation kernels of one workload with CUDA events.  --two-stage times the count step of the two-stage
path (RotatE, pRotatE: fast tile pass + exact re-score) instead of the exact kernel and reports the share of
(query, entity) pairs the fast pass left undecidable."""
import argparse
import ctypes
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench import WORKLOADS  # noqa: E402
from knowledgegraphembedding_b200 import KGEModel, _lib  # noqa: E402
from knowledgegraphembedding_b200.model import _ptr, _stream  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--workload", default="rotate_fb15k")
ap.add_argument("--queries", type=int, default=1024)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--two-stage", action="store_true")
a = ap.parse_args()
model, nentity, nrel, d, gamma, B, N, lr, de, dr = WORKLOADS[a.workload][:10]
m = KGEModel(model, nentity, nrel, d, gamma, double_entity_embedding=de, double_relation_embedding=dr).cuda()
dev = m.entity_embedding.device
rng = np.random.RandomState(0)
Q = a.queries
q = torch.from_numpy(np.stack([rng.randint(nentity, size=Q), rng.randint(nrel, size=Q), rng.randint(nentity, size=Q)], 1)).to(dev)
words = (nentity + 31) // 32
bits = torch.zeros(Q * words, dtype=torch.int32, device=dev)
qvec = torch.empty(Q * m.entity_dim, device=dev)
pos = torch.empty(Q, device=dev)
counts = torch.zeros(Q, dtype=torch.int32, device=dev)
desc, st = m._descriptor(), _stream(dev)
cap = Q * 256
amb = torch.empty(2 * cap, dtype=torch.int32, device=dev)
amb_count = torch.zeros(2, dtype=torch.int32, device=dev)
phase = None
if model == "pRotatE":
    phase = torch.empty(nentity * m.entity_dim, device=dev)
    _lib.call("kge_eval_phase_table", ctypes.byref(desc), _ptr(phase), st)
for mode in ("head-batch", "tail-batch"):
    mid = _lib.MODE_IDS[mode]
    times = {"qvec": [], "pos": [], "count": []}
    for rep in range(a.reps):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        _lib.call("kge_eval_query_vectors", ctypes.byref(desc), mid, _ptr(q), Q, _ptr(qvec), None, st)
        ev[1].record()
        _lib.call("kge_eval_positive_scores", ctypes.byref(desc), mid, _ptr(qvec), _ptr(q), Q, _ptr(phase), _ptr(pos), st)
        ev[2].record()
        if a.two_stage:
            _lib.call("kge_eval_count_ranks_two_stage", ctypes.byref(desc), mid, _ptr(qvec), _ptr(q), Q, _ptr(phase),
                      _ptr(pos), _ptr(bits), 0, nentity, _ptr(counts), _ptr(amb), cap, _ptr(amb_count), st)
        else:
            _lib.call("kge_eval_count_ranks", ctypes.byref(desc), mid, _ptr(qvec), _ptr(q), Q, _ptr(phase), _ptr(pos),
                      _ptr(bits), 0, nentity, _ptr(counts), None, st)
        ev[3].record()
        torch.cuda.synchronize()
        for k, i in (("qvec", 0), ("pos", 1), ("count", 2)):
            times[k].append(ev[i].elapsed_time(ev[i + 1]))
    best = {k: min(v) for k, v in times.items()}
    tot = sum(best.values())
    undecidable = ""
    if a.two_stage:
        n, overflow = amb_count.tolist()
        undecidable = f", {n / (Q * nentity):.2e} of the pairs undecidable" + (" (list overflowed)" if overflow else "")
    print(f"{a.workload} {mode}: Q={Q} qvec {best['qvec']:.3f} ms, pos {best['pos']:.3f} ms, count {best['count']:.3f} ms "
          f"-> {Q / tot * 1e3:.0f} queries/s (kernels only); one-pass-per-query HBM equiv "
          f"{Q * nentity * m.entity_dim * 4 / (best['count'] * 1e-3) / 1e9:.0f} GB/s{undecidable}")
