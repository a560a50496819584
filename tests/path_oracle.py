"""ctypes loader of tests/path_oracle.c (the reference of KGEModel's path queries).  TEST INFRASTRUCTURE.  The library
is compiled into a temporary directory on first use, so the tree stays untouched."""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

from oracle.c_oracle import MODEL_IDS, _f32, _i64, _modulus, _p

HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def load():
    global _lib
    if _lib is None:
        path = os.path.join(tempfile.mkdtemp(prefix="kge_path_oracle_"), "libpath_oracle.so")
        subprocess.run(["gcc", "-O2", "-std=c11", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-shared",
                        "-o", path, os.path.join(HERE, "path_oracle.c"), "-lm"], check=True)
        _lib = ctypes.CDLL(path)
    return _lib


def path_query_vectors(model, state, anchors, paths, mode, rho):
    """[Q, entity_dim] path query vectors of anchors [Q] along paths [Q, L] (DESIGN.md section 3.13)."""
    E, R = _f32(state["entity_embedding"]), _f32(state["relation_embedding"])
    a, p = _i64(anchors).reshape(-1), _i64(paths)
    p = p.reshape(a.shape[0], -1)
    out = np.empty((a.shape[0], E.shape[1]), dtype=np.float32)
    load().ko_path_query_vectors(MODEL_IDS[model], int(mode == "head-batch"), _p(E), _p(R), ctypes.c_int64(R.shape[0]),
                                 E.shape[1], R.shape[1], ctypes.c_float(rho), _p(a), _p(p), ctypes.c_int64(a.shape[0]),
                                 ctypes.c_int64(p.shape[1]), _p(out))
    return out


def scores_from_q(model, state, qvec, mode, gamma, rho):
    """[Q, nentity] unfiltered scores of every entity against the query vectors qvec [Q, entity_dim]."""
    E = _f32(state["entity_embedding"])
    q = _f32(qvec).reshape(-1, E.shape[1])
    out = np.empty((q.shape[0], E.shape[0]), dtype=np.float32)
    load().ko_scores_from_q(MODEL_IDS[model], int(mode == "head-batch"), _p(E), ctypes.c_int64(E.shape[0]), E.shape[1],
                            ctypes.c_float(gamma), ctypes.c_float(rho), ctypes.c_float(_modulus(state)), _p(q),
                            ctypes.c_int64(q.shape[0]), _p(out))
    return out
