"""Path queries without a GPU: the reference fold of tests/path_oracle.c (ko_path_query_vectors) against the C oracle's
one-hop query vectors bit for bit and against a float64 composition at L = 2..4, and the argument checks of the path
entries of the C ABI."""
import ctypes

import numpy as np
import pytest

from oracle import c_oracle as C
from oracle import kge_oracle as O

import path_oracle as P

FLAGS = {"TransE": (False, False), "DistMult": (False, False), "ComplEx": (True, True),
         "RotatE": (True, False), "pRotatE": (False, False)}
MODES = ("head-batch", "tail-batch")


def tables(model, nentity=40, nrel=6, d=37, gamma=12.0):
    de, dr = FLAGS[model]
    return O.init_tables(model, nentity, nrel, d, gamma, de, dr, seed=3), O.embedding_range(gamma, d)


@pytest.mark.parametrize("model", list(FLAGS))
@pytest.mark.parametrize("mode", MODES)
def test_one_hop_fold_is_the_query_vector(model, mode):
    st, rho = tables(model)
    rng = np.random.RandomState(1)
    anchors, rels = rng.randint(40, size=64), rng.randint(6, size=64)
    want = C.query_vectors(model, st, np.stack([anchors, rels, anchors], 1), mode, rho)
    got = P.path_query_vectors(model, st, anchors, rels[:, None], mode, rho)
    np.testing.assert_array_equal(got.view(np.uint32), want.view(np.uint32))


def fold64(model, st, rho, a, path, mode, nrel):
    """The fold in float64 and a bound of the magnitudes it adds or multiplies (for the rounding bound)."""
    E = st["entity_embedding"].astype(np.float64)
    R = st["relation_embedding"].astype(np.float64)
    cplx = model in ("ComplEx", "RotatE")
    d = E.shape[1] // 2 if cplx else E.shape[1]
    scale = rho / (3.14159262358979323846 if model == "pRotatE" else np.pi)
    hops = [h for h in path if h != -1]
    head = mode == "head-batch"
    q = E[a, :d] + 1j * E[a, d:] if cplx else E[a].copy()
    if model == "pRotatE":
        q = q / scale
    if head and model in ("TransE", "pRotatE"):
        q = -q
    mag = np.abs(q)
    for h in (reversed(hops) if head else hops):
        inv, r = h >= nrel, h % nrel
        if model in ("TransE", "pRotatE"):
            v = R[r] / (scale if model == "pRotatE" else 1.0)
            q = q - v if inv else q + v
            mag = mag + np.abs(v)
        elif model == "DistMult":
            q = q * R[r]
            mag = mag * np.abs(R[r])
        else:
            v = R[r, :d] + 1j * R[r, d:] if model == "ComplEx" else np.exp(1j * R[r] / scale)
            q = q * (np.conj(v) if inv != head else v)
            mag = mag * np.abs(v)
    return (np.concatenate([q.real, q.imag]) if cplx else q), (np.concatenate([mag, mag]) if cplx else mag)


@pytest.mark.parametrize("model", list(FLAGS))
@pytest.mark.parametrize("mode", MODES)
def test_multi_hop_fold_within_rounding_of_float64(model, mode):
    """L = 2..4 with inverse hops and padding: every element within 8 L 2^-24 of the magnitudes the fold combines."""
    nrel = 6
    st, rho = tables(model, nrel=nrel)
    rng = np.random.RandomState(2)
    for L in (2, 3, 4):
        anchors = rng.randint(40, size=32)
        paths = rng.randint(2 * nrel, size=(32, L))
        for i in range(0, 32, 4):                      # ragged rows: padded after at least one hop
            paths[i, rng.randint(1, L):] = -1
        got = P.path_query_vectors(model, st, anchors, paths, mode, rho).astype(np.float64)
        for i in range(32):
            want, mag = fold64(model, st, rho, anchors[i], paths[i], mode, nrel)
            assert np.all(np.abs(got[i] - want) <= 8 * L * 2.0 ** -24 * mag + 1e-30), (L, i)


def test_path_abi_argument_errors_without_a_gpu():
    from knowledgegraphembedding_b200 import _lib
    lib = _lib.load()
    desc = _lib.KgeModelStruct(model=_lib.TRANSE, device=0, nentity=4, nrelation=2, hidden_dim=4, entity_dim=4,
                               relation_dim=4, gamma=1.0, embedding_range=0.1, entity=8, relation=8, modulus=None)
    tail = _lib.TAIL_BATCH
    rc = lib.kge_eval_path_query_vectors(ctypes.byref(desc), tail, None, 16, 3, 2, 16, None, None)
    assert rc == _lib.ERR_INVALID and b"null pointer" in lib.kge_last_error()
    rc = lib.kge_eval_path_query_vectors(ctypes.byref(desc), tail, 16, 16, 3, 0, 16, None, None)
    assert rc == _lib.ERR_INVALID and b"at least one hop" in lib.kge_last_error()
    rc = lib.kge_eval_path_query_vectors(ctypes.byref(desc), tail, 16, 16, -1, 2, 16, None, None)
    assert rc == _lib.ERR_INVALID and b"bad query count" in lib.kge_last_error()
    rc = lib.kge_eval_path_query_vectors(ctypes.byref(desc), _lib.SINGLE, 16, 16, 3, 2, 16, None, None)
    assert rc == _lib.ERR_INVALID
    dense = (16, 16, None, None)
    rc = lib.kge_eval_path_bits_dense(*dense, None, 16, 3, 2, tail, 4, 2, 16, 32, None, None)
    assert rc == _lib.ERR_INVALID and b"null pointer" in lib.kge_last_error()
    rc = lib.kge_eval_path_bits_dense(*dense, 16, 16, 3, 0, tail, 4, 2, 16, 32, None, None)
    assert rc == _lib.ERR_INVALID and b"at least one hop" in lib.kge_last_error()
    rc = lib.kge_eval_path_bits_dense(*dense, 16, 16, -1, 2, tail, 4, 2, 16, 32, None, None)
    assert rc == _lib.ERR_INVALID and b"bad arguments" in lib.kge_last_error()
    rc = lib.kge_eval_path_bits_dense(*dense, 16, 16, 3, 2, tail, 4, 2, 16, 16, None, None)
    assert rc == _lib.ERR_INVALID and b"two buffers" in lib.kge_last_error()
    rc = lib.kge_eval_path_bits_dense(16, None, None, None, 16, 16, 3, 2, tail, 4, 2, 16, 32, None, None)
    assert rc == _lib.ERR_INVALID and b"half of a filter index" in lib.kge_last_error()
    sorted_ix = (16, 16, 16, 5, None, None, None, 0)
    rc = lib.kge_eval_path_bits(*sorted_ix, 16, None, 3, 2, tail, 4, 2, 16, 32, None, None)
    assert rc == _lib.ERR_INVALID and b"null pointer" in lib.kge_last_error()
    rc = lib.kge_eval_path_bits(*sorted_ix, 16, 16, 3, 0, tail, 4, 2, 16, 32, None, None)
    assert rc == _lib.ERR_INVALID and b"at least one hop" in lib.kge_last_error()
    rc = lib.kge_eval_path_bits(None, None, None, 5, None, None, None, 0, 16, 16, 3, 2, tail, 4, 2, 16, 32, None, None)
    assert rc == _lib.ERR_INVALID and b"null filter index" in lib.kge_last_error()
    rc = lib.kge_eval_path_bits(*sorted_ix, 16, 16, 3, 2, _lib.SINGLE, 4, 2, 16, 32, None, None)
    assert rc == _lib.ERR_INVALID and b"mode 0 not supported" in lib.kge_last_error()
