"""ctypes loader of tests/similarity_oracle.c (the reference of KGEModel.nearest_neighbors) and the stable sort the
similarity tests compare against.  TEST INFRASTRUCTURE.  The library is compiled into a temporary directory on first
use, so the tree stays untouched."""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
METRICS = {"dot": 0, "cosine": 1, "l2": 2, "l1": 3}
_lib = None


def load():
    global _lib
    if _lib is None:
        path = os.path.join(tempfile.mkdtemp(prefix="kge_sim_oracle_"), "libsimilarity_oracle.so")
        subprocess.run(["gcc", "-O2", "-std=c11", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-shared",
                        "-o", path, os.path.join(HERE, "similarity_oracle.c"), "-lm"], check=True)
        _lib = ctypes.CDLL(path)
    return _lib


def similarity(table, queries, metric):
    """[Q, rows] float32 scores of every (query, row) pair, bit-identical to the device's canonical scores."""
    X = np.ascontiguousarray(table, dtype=np.float32)
    q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, X.shape[1])
    out = np.empty((q.shape[0], X.shape[0]), dtype=np.float32)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)      # noqa: E731
    load().ko_similarity(p(X), ctypes.c_int64(X.shape[0]), ctypes.c_int(X.shape[1]), p(q), ctypes.c_int64(q.shape[0]),
                         ctypes.c_int(METRICS[metric]), p(out))
    return out


def topk(scores, k, self_ids=None):
    """ids int64 [Q, k] and scores float32 [Q, k] of a stable descending sort of each row (score descending, then id
    ascending, NaN last, -0.0 == +0.0), with column self_ids[q] left out; empty slots hold id -1 and score -inf."""
    Q, rows = scores.shape
    ids = np.full((Q, k), -1, dtype=np.int64)
    out = np.full((Q, k), -np.inf, dtype=np.float32)
    for q in range(Q):
        cand = np.arange(rows)
        if self_ids is not None and 0 <= self_ids[q] < rows:
            cand = cand[cand != self_ids[q]]
        s = scores[q, cand]
        nan = np.isnan(s)
        order = np.lexsort((cand, np.where(nan, 0.0, -s.astype(np.float64)), nan))[:k]
        ids[q, :order.size] = cand[order]
        out[q, :order.size] = s[order]
    return ids, out
