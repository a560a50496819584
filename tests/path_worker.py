"""Worker of tests/test_gpu_path.py::test_path_calls_two_ranks_sharing_one_gpu (one process per rank, launched with
torch.distributed.run).

Every rank computes KGEModel.path_rank_statistics and predict_path_topk once as a single process (before the process
group exists) and once as a rank of the group, where it builds every query's whole answer set, counts or selects over its
entity slice and combines the results of all ranks.  The two results must be identical on every rank.
KGE_TEST_SAME_GPU=1: every rank on cuda:0 over gloo; otherwise one GPU per rank over NCCL.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from topk_worker import build                         # noqa: E402

# two-stage (RotatE, pRotatE), tcgen05 (ComplEx) and exact (TransE) counting
CASES = [("RotatE", 5003, 17, 64, 12.0), ("pRotatE", 777, 5, 12, 6.0), ("ComplEx", 1001, 7, 32, 20.0),
         ("TransE", 640, 6, 16, 9.0)]


def runs(dev):
    out = []
    for model, nentity, nrel, d, gamma in CASES:
        m = build(model, nentity, nrel, d, gamma, dev)
        rng = np.random.RandomState(7)
        triples = sorted({(int(rng.randint(nentity)), int(rng.randint(nrel)), int(rng.randint(nentity)))
                          for _ in range(6 * nentity)})
        anchors, paths = rng.randint(nentity, size=120), rng.randint(2 * nrel, size=(120, 3))
        paths[::4, 2] = -1
        answers = rng.randint(nentity, size=120)
        for mode in ("head-batch", "tail-batch"):
            stats, counts = m.path_rank_statistics(anchors, paths, answers, triples, mode, return_answer_counts=True)
            ids, scores = m.predict_path_topk(anchors, paths, mode, k=16, exclude_triples=triples)
            out.append((model, mode, stats, counts, ids.cpu().numpy(), scores.cpu().numpy().view(np.uint32)))
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
    for one, many in zip(single, sharded):
        for a, b in zip(one[2:], many[2:]):
            assert np.array_equal(a, b), (one[0], one[1], dist.get_rank())
    dist.barrier()
    dist.destroy_process_group()
    if int(os.environ.get("RANK", "0")) == 0:
        print("ok", flush=True)


if __name__ == "__main__":
    main()
