"""Worker of tests/test_gpu_relation.py::test_relation_multi_rank_* (one process per rank, launched with
torch.distributed.run).

Every rank computes KGEModel.filtered_relation_ranks and predict_relations once as a single process (before the process
group exists) and once as a rank of the group, where it works on its relation slice (shard_bounds(nrelation, rank,
world, align=64): empty on some ranks for the small relation counts) and the counts are all-reduced / the key lists
merged.  The two results must be identical on every rank.  KGE_TEST_SAME_GPU=1: every rank on cuda:0 over gloo;
otherwise one GPU per rank over NCCL.
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

FLAGS = {"TransE": (False, False), "RotatE": (True, False), "pRotatE": (False, False), "ComplEx": (True, True),
         "DistMult": (False, False)}
CASES = [("RotatE", 1003, 200, 64, 12.0), ("pRotatE", 777, 11, 12, 6.0), ("ComplEx", 1001, 130, 32, 20.0),
         ("TransE", 500, 2, 16, 6.0)]


def build(model, nentity, nrel, d, gamma, dev):
    de, dr = FLAGS[model]
    st = O.init_tables(model, nentity, nrel, d, gamma, de, dr, seed=11)
    m = KGEModel(model, nentity, nrel, d, gamma, double_entity_embedding=de, double_relation_embedding=dr)
    with torch.no_grad():
        m.entity_embedding.copy_(torch.from_numpy(st["entity_embedding"] * 3.0))
        m.relation_embedding.copy_(torch.from_numpy(st["relation_embedding"]))
    return m.to(dev)


def inputs(nentity, nrel):
    rng = np.random.RandomState(5)
    all_true = sorted({(int(rng.randint(nentity)), int(rng.randint(nrel)), int(rng.randint(20))) for _ in range(3000)})
    queries = [all_true[i] for i in rng.choice(len(all_true), 150, replace=False)]
    return queries, all_true


def runs(dev):
    out = []
    for model, nentity, nrel, d, gamma in CASES:
        m = build(model, nentity, nrel, d, gamma, dev)
        queries, all_true = inputs(nentity, nrel)
        out.append((model, "ranks", m.filtered_relation_ranks(queries, all_true), None))
        for k, exclude in ((10, all_true), (256, None)):
            ids, scores = m.predict_relations(queries, k=k, exclude_triples=exclude)
            out.append((model, k, ids.cpu().numpy(), scores.cpu().numpy()))
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
    for (model, what, a1, s1), (_, _, a2, s2) in zip(single, sharded):
        assert np.array_equal(a1, a2), (model, what, dist.get_rank())
        if s1 is not None:
            assert np.array_equal(s1.view(np.uint32), s2.view(np.uint32)), (model, what, dist.get_rank())
    dist.barrier()
    dist.destroy_process_group()
    if int(os.environ.get("RANK", "0")) == 0:
        print("ok", flush=True)


if __name__ == "__main__":
    main()
