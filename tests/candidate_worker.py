"""Worker of tests/test_gpu_candidates.py::test_candidate_statistics_two_ranks_sharing_one_gpu (one process per rank,
launched with torch.distributed.run).

Every rank computes KGEModel.candidate_rank_statistics once as a single process (before the process group exists) and
once as a rank of the group, where it counts over its slice of the candidate columns and the tallies of all ranks are
summed.  The two results must be identical on every rank.  KGE_TEST_SAME_GPU=1: every rank on cuda:0 over gloo;
otherwise one GPU per rank over NCCL.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from knowledgegraphembedding_b200 import KGEModel                  # noqa: E402
from test_gpu_candidates import positives, random_lists            # noqa: E402
from test_gpu_rank_stats import FLAGS, tie_case                    # noqa: E402

MODELS = ("RotatE", "pRotatE", "ComplEx", "DistMult", "TransE")


def runs(dev):
    out = []
    for model in MODELS:
        nentity, nrel, d, gamma, st, test, all_true = tie_case(model, seed=36)
        de, dr = FLAGS[model]
        m = KGEModel(model, nentity, nrel, d, gamma, double_entity_embedding=de, double_relation_embedding=dr)
        with torch.no_grad():
            m.entity_embedding.copy_(torch.from_numpy(st["entity_embedding"]))
            m.relation_embedding.copy_(torch.from_numpy(st["relation_embedding"]))
        m = m.to(dev)
        rng = np.random.RandomState(10)
        for mode in ("head-batch", "tail-batch"):
            cand = random_lists(rng, positives(test, mode), nentity, 517)
            out.append((model, mode, m.candidate_rank_statistics(test, cand, mode, exclude_triples=all_true)))
            out.append((model, mode, m.candidate_rank_statistics(test, cand, mode, query_chunk=13)))
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
    for (model, mode, s1), (_, _, s2) in zip(single, sharded):
        assert np.array_equal(s1, s2), (model, mode, dist.get_rank())
    m = KGEModel("TransE", 10, 2, 4, 6.0).to(dev)
    try:
        m.candidate_rank_statistics([(1, 0, 2)], [[3, 4]], "tail-batch", return_scores=True)
        raise AssertionError("return_scores under a process group must raise")
    except ValueError:
        pass
    dist.barrier()
    dist.destroy_process_group()
    if int(os.environ.get("RANK", "0")) == 0:
        print("ok", flush=True)


if __name__ == "__main__":
    main()
