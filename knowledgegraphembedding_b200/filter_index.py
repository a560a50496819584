"""Host-side filter index for filtered ranking.

Replaces the per-query python set scan of the reference's TestDataset (codes/dataloader.py:134-154: one
`(h, r, t) in triple_set` lookup per entity per query) by two sorted-key CSR tables built once per
`all_true_triples` list:
    head-batch query (?, r, t)  ->  every h with (h, r, t) true
    tail-batch query (h, r, ?)  ->  every t with (h, r, t) true
The device turns the lists of one query chunk into the filter bitmap (kge_eval_filter_bits).
relation_table() is the index of relation prediction, (h, t) -> every r with (h, r, t) true.
Pure numpy; covered by CPU tests.
"""
import numpy as np


class FilterIndex:
    def __init__(self, all_true_triples, nentity, nrelation):
        tri = np.asarray(all_true_triples, dtype=np.int64).reshape(-1, 3)
        self.nentity, self.nrelation = int(nentity), int(nrelation)
        self.ntriples = tri.shape[0]
        h, r, t = tri[:, 0], tri[:, 1], tri[:, 2]
        self._tables = {
            "head-batch": self._group(r * self.nentity + t, h),
            "tail-batch": self._group(h * self.nrelation + r, t),
        }

    @staticmethod
    def _group(keys, values):
        order = np.argsort(keys, kind="stable")
        keys, values = keys[order], values[order]
        ukeys, starts = np.unique(keys, return_index=True)
        offsets = np.append(starts, keys.size).astype(np.int64)
        return ukeys, offsets, values.astype(np.int32)

    def _query_keys(self, queries, mode):
        q = np.asarray(queries, dtype=np.int64).reshape(-1, 3)
        if mode == "head-batch":
            return q[:, 1] * self.nentity + q[:, 2]
        if mode == "tail-batch":
            return q[:, 0] * self.nrelation + q[:, 1]
        raise ValueError('negative batch mode %s not supported' % mode)       # dataloader.py:147

    def table(self, mode):
        """(sorted unique keys int64 [K], run offsets int64 [K+1], entities int32 [nnz]) of one mode: what the device
        keeps resident for kge_eval_filter_bits_lookup."""
        if mode not in self._tables:
            raise ValueError('negative batch mode %s not supported' % mode)    # dataloader.py:147
        return self._tables[mode]

    def csr(self, queries, mode):
        """(offsets int64 [Q+1], entities int32 [nnz]) : the true entities of every query's open slot."""
        ukeys, offsets, values = self._tables[mode] if mode in self._tables else (None, None, None)
        qk = self._query_keys(queries, mode)
        nq = qk.size
        if ukeys.size == 0:
            return np.zeros(nq + 1, dtype=np.int64), np.zeros(0, dtype=np.int32)
        pos = np.searchsorted(ukeys, qk)
        pos_c = np.minimum(pos, ukeys.size - 1)
        found = ukeys[pos_c] == qk
        start = np.where(found, offsets[pos_c], 0)
        length = np.where(found, offsets[pos_c + 1] - offsets[pos_c], 0)
        out_off = np.zeros(nq + 1, dtype=np.int64)
        np.cumsum(length, out=out_off[1:])
        total = int(out_off[-1])
        # gather all slices at once: index = start[q] + (i - out_off[q]) for i in the q-th output run
        run = np.repeat(np.arange(nq), length)
        idx = np.repeat(start - out_off[:-1], length) + np.arange(total)
        ents = values[idx] if total else np.zeros(0, dtype=np.int32)
        assert run.size == total
        return out_off, np.ascontiguousarray(ents, dtype=np.int32)


def relation_table(all_true_triples, nentity):
    """Relation-prediction index of a list of true triples: (sorted unique keys h*nentity+t int64 [K], run offsets int64
    [K+1], relation ids int32 [nnz]); run i holds every r with (h, r, t) true for key i.  The key space nentity^2 is too
    large for a direct-address table, so the keys are sorted and the device looks them up by binary search
    (kge_eval_relation_filter_bits)."""
    tri = np.asarray(all_true_triples, dtype=np.int64).reshape(-1, 3)
    return FilterIndex._group(tri[:, 0] * int(nentity) + tri[:, 2], tri[:, 1])
