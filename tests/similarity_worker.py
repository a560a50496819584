"""Worker of tests/test_gpu_similarity.py::test_similarity_multi_rank_* (one process per rank, launched with
torch.distributed.run).

Every rank computes KGEModel.nearest_neighbors once as a single process (before the process group exists) and once as
a rank of the group, where it selects over its row slice and merges the lists of all ranks.  The two results must be
identical on every rank.  KGE_TEST_SAME_GPU=1: every rank on cuda:0 over gloo; otherwise one GPU per rank over NCCL.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from knowledgegraphembedding_b200 import KGEModel     # noqa: E402
from oracle import kge_oracle as O                    # noqa: E402

# (model, nentity, nrelation, hidden_dim, double entity, double relation): the 17-row relation table leaves every rank
# but the first with an empty slice
CASES = [("RotatE", 5003, 17, 64, True, False), ("ComplEx", 1001, 300, 18, True, True)]


def build(model, nentity, nrel, d, de, dr, dev):
    st = O.init_tables(model, nentity, nrel, d, 12.0, de, dr, seed=11)
    m = KGEModel(model, nentity, nrel, d, 12.0, double_entity_embedding=de, double_relation_embedding=dr)
    with torch.no_grad():
        m.entity_embedding.copy_(torch.from_numpy(st["entity_embedding"] * 3.0))
        m.relation_embedding.copy_(torch.from_numpy(st["relation_embedding"]))
    return m.to(dev)


def runs(dev):
    out = []
    rng = np.random.RandomState(5)
    for model, nentity, nrel, d, de, dr in CASES:
        m = build(model, nentity, nrel, d, de, dr, dev)
        for table, rows in (("entity", nentity), ("relation", nrel)):
            ids = rng.randint(rows, size=150)
            width = m.entity_dim if table == "entity" else m.relation_dim
            vectors = rng.standard_normal((40, width)).astype(np.float32)
            for metric in ("dot", "cosine", "l2", "l1"):
                for items, k in ((ids, 10), (vectors, 256)):
                    got_ids, got_scores = m.nearest_neighbors(items, table=table, k=k, metric=metric)
                    out.append((model, table, metric, k, got_ids.cpu().numpy(), got_scores.cpu().numpy()))
    return out


def main():
    same = os.environ.get("KGE_TEST_SAME_GPU") == "1"
    local = 0 if same else int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    single = runs(dev)
    if same:
        dist.init_process_group("gloo")
    else:
        dist.init_process_group("nccl", device_id=dev)
    sharded = runs(dev)
    for (model, table, metric, k, ids1, s1), (_, _, _, _, ids2, s2) in zip(single, sharded):
        what = (model, table, metric, k, dist.get_rank())
        assert np.array_equal(ids1, ids2), what
        assert np.array_equal(s1.view(np.uint32), s2.view(np.uint32)), what
    dist.barrier()
    dist.destroy_process_group()
    if int(os.environ.get("RANK", "0")) == 0:
        print("ok", flush=True)


if __name__ == "__main__":
    main()
