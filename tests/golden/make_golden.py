#!/usr/bin/env python
"""Generate the golden vectors under tests/golden/ by RUNNING THE UNMODIFIED REFERENCE.

Run in the build container only (needs /root/reference):

    python tests/golden/make_golden.py

The reference (kahrabian/KnowledgeGraphEmbedding, codes/model.py + codes/dataloader.py) ships no tests
or fixtures, so parity is pinned on its own outputs for seeded inputs.  Nothing here is read at test
time except the .npz files this script writes; the GPU box has no /root/reference.

Files written
  small_<Model>_d<d>.npz   forward scores (3 modes), 4 train steps x 4 loss configs, filtered ranks
  countries_S1.npz         real dataset: 4 RotatE train steps on reference-sampled batches, AUC-PR, ranks
                           (+ countries_S1.2.npz: the second half of the final entity table)
  fullwidth_RotatE_fb15k.npz  BASELINE configs[2] row shape (14,951 x 2000 table, N=256), 192 rows, 3 train steps
                           (+ fullwidth_RotatE_fb15k.2.npz: the sampled rows of the updated tables)
  runpy_logs.json          codes/run.py end to end (countries_S1 train/valid/test + resume, wn18rr --do_test -init): log lines
  wn18rr_eval.npz          real dataset: filtered ranks of a seeded RotatE model on 400 test triples
"""
import argparse
import os
import sys
import types

import numpy as np
import torch

REF = os.environ.get("KGE_REFERENCE", "/root/reference")
sys.path.insert(0, os.path.join(REF, "codes"))
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))

import dataloader as ref_data          # noqa: E402  (reference)
import model as ref_model              # noqa: E402  (reference)
from oracle import kge_oracle as O     # noqa: E402  (only for the portable numpy table initialiser)

torch.set_num_threads(4)

FLAGS = {"TransE": (False, False), "DistMult": (False, False), "ComplEx": (True, True),
         "RotatE": (True, False), "pRotatE": (False, False)}
GAMMA = {"TransE": 9.0, "DistMult": 20.0, "ComplEx": 20.0, "RotatE": 6.0, "pRotatE": 6.0}


def make_ref(model_name, nentity, nrelation, d, gamma, seed, scale=1.0):
    de, dr = FLAGS[model_name]
    m = ref_model.KGEModel(model_name=model_name, nentity=nentity, nrelation=nrelation, hidden_dim=d,
                           gamma=gamma, double_entity_embedding=de, double_relation_embedding=dr)
    st = O.init_tables(model_name, nentity, nrelation, d, gamma, de, dr, seed=seed)
    if scale != 1.0:       # "trained-like" spread of scores (random-init scores are nearly all equal)
        st["entity_embedding"] = (st["entity_embedding"] * scale).astype(np.float32)
    with torch.no_grad():
        m.entity_embedding.copy_(torch.from_numpy(st["entity_embedding"]))
        m.relation_embedding.copy_(torch.from_numpy(st["relation_embedding"]))
    return m, st


def ns(**kw):
    base = dict(cuda=False, negative_adversarial_sampling=False, adversarial_temperature=1.0,
                uni_weight=False, regularization=0.0, countries=False, regions=None,
                test_batch_size=4, cpu_num=2, test_log_steps=100000, nentity=0, nrelation=0)
    base.update(kw)
    return types.SimpleNamespace(**base)


def stable_ranks(m, test_triples, all_true, nentity, nrelation):
    """Per-query ranks via the reference's TestDataset + forward, stable descending order."""
    ranks, scores = [], []
    for mode in ("head-batch", "tail-batch"):
        ds = ref_data.TestDataset(test_triples, all_true, nentity, nrelation, mode)
        for i in range(len(ds)):
            pos, neg, bias, _ = ds[i]
            with torch.no_grad():
                s = m((pos[None], neg[None]), mode)[0] + bias
            arg = pos[0] if mode == "head-batch" else pos[2]
            order = torch.argsort(s, descending=True, stable=True)
            hit = (order == arg).nonzero()
            assert hit.size(0) == 1
            ranks.append(1 + hit.item())
            scores.append(s.numpy().copy())
    return np.asarray(ranks, dtype=np.int64), np.stack(scores)


TRAIN_CFGS = {
    "adv_sub": dict(negative_adversarial_sampling=True, adversarial_temperature=0.7, uni_weight=False),
    "adv_uni": dict(negative_adversarial_sampling=True, adversarial_temperature=1.0, uni_weight=True),
    "mean_sub": dict(negative_adversarial_sampling=False, uni_weight=False),
    "adv_sub_reg": dict(negative_adversarial_sampling=True, adversarial_temperature=1.0, uni_weight=False,
                        regularization=1e-3),
}


def small_case(model_name, d, out):
    nentity, nrelation, B, N = 37, 5, 6, 9
    gamma = GAMMA[model_name]
    rng = np.random.RandomState(1234 + d)
    positive = np.stack([rng.randint(nentity, size=B), rng.randint(nrelation, size=B),
                         rng.randint(nentity, size=B)], axis=1).astype(np.int64)
    negative = rng.randint(nentity, size=(B, N)).astype(np.int64)
    weight = np.sqrt(1.0 / rng.randint(8, 200, size=B)).astype(np.float32)
    m, st = make_ref(model_name, nentity, nrelation, d, gamma, seed=d)
    data = dict(nentity=nentity, nrelation=nrelation, d=d, gamma=gamma, positive=positive,
                negative=negative, weight=weight, **{"init_" + k: v for k, v in st.items()})
    tp, tn = torch.from_numpy(positive), torch.from_numpy(negative)
    with torch.no_grad():
        data["score_single"] = m(tp).numpy()
        data["score_head-batch"] = m((tp, tn), "head-batch").numpy()
        data["score_tail-batch"] = m((tp, tn), "tail-batch").numpy()
    # autograd of a plain weighted score sum (exercises forward()'s differentiability per mode)
    cot = rng.standard_normal((B, N)).astype(np.float32)
    data["cotangent"] = cot
    for mode in ("single", "head-batch", "tail-batch"):
        m.zero_grad()
        s = m(tp) if mode == "single" else m((tp, tn), mode)
        (s * torch.from_numpy(cot[:, :s.shape[1]])).sum().backward()
        data["dE_" + mode] = m.entity_embedding.grad.numpy().copy()
        data["dR_" + mode] = m.relation_embedding.grad.numpy().copy()
        if model_name == "pRotatE":
            data["dM_" + mode] = m.modulus.grad.numpy().copy()
    # train steps: 4 steps alternating tail/head like BidirectionalOneShotIterator (dataloader.py:171-177)
    for cname, cfg in TRAIN_CFGS.items():
        m, _ = make_ref(model_name, nentity, nrelation, d, gamma, seed=d)
        lr = 1e-3
        opt = torch.optim.Adam(filter(lambda p: p.requires_grad, m.parameters()), lr=lr)
        batches = []
        for step in range(4):
            pos_s = np.stack([rng.randint(nentity, size=B), rng.randint(nrelation, size=B),
                              rng.randint(nentity, size=B)], axis=1).astype(np.int64)
            neg_s = rng.randint(nentity, size=(B, N)).astype(np.int64)
            w_s = np.sqrt(1.0 / rng.randint(8, 200, size=B)).astype(np.float32)
            batches.append((pos_s, neg_s, w_s, "tail-batch" if step % 2 == 0 else "head-batch"))
        it = iter([(torch.from_numpy(a), torch.from_numpy(b), torch.from_numpy(c), md)
                   for a, b, c, md in batches])
        args = ns(**cfg)
        logs = []
        for step in range(4):
            if step == 2:      # run.py:315-322: LR decay re-creates Adam (moments dropped)
                lr = lr / 10
                opt = torch.optim.Adam(filter(lambda p: p.requires_grad, m.parameters()), lr=lr)
            log = ref_model.KGEModel.train_step(m, opt, it, args)
            logs.append([log.get("regularization", 0.0), log["positive_sample_loss"],
                         log["negative_sample_loss"], log["loss"]])
            if step == 0:
                data[f"train_{cname}_gE0"] = m.entity_embedding.grad.numpy().copy()
                data[f"train_{cname}_gR0"] = m.relation_embedding.grad.numpy().copy()
                if model_name == "pRotatE":
                    data[f"train_{cname}_gM0"] = m.modulus.grad.numpy().copy()
        data[f"train_{cname}_logs"] = np.asarray(logs, dtype=np.float64)
        for i, (a, b, c, md) in enumerate(batches):
            data[f"train_{cname}_pos{i}"], data[f"train_{cname}_neg{i}"], data[f"train_{cname}_w{i}"] = a, b, c
        data[f"train_{cname}_E"] = m.entity_embedding.detach().numpy().copy()
        data[f"train_{cname}_R"] = m.relation_embedding.detach().numpy().copy()
        if model_name == "pRotatE":
            data[f"train_{cname}_M"] = m.modulus.detach().numpy().copy()
        sd = opt.state_dict()["state"]
        data[f"train_{cname}_adam_steps"] = np.asarray([float(sd[k]["step"]) for k in sorted(sd)])
    # filtered ranking on a small KG
    m, st = make_ref(model_name, nentity, nrelation, d, gamma, seed=d + 1, scale=8.0)
    all_true = sorted({(int(rng.randint(nentity)), int(rng.randint(nrelation)), int(rng.randint(nentity)))
                       for _ in range(160)})
    test = [all_true[i] for i in rng.choice(len(all_true), size=14, replace=False)]
    ranks, scores = stable_ranks(m, test, all_true, nentity, nrelation)
    metrics = ref_model.KGEModel.test_step(m, test, all_true, ns(nentity=nentity, nrelation=nrelation))
    data.update(eval_E=st["entity_embedding"], eval_R=st["relation_embedding"],
                eval_all_true=np.asarray(all_true, dtype=np.int64), eval_test=np.asarray(test, dtype=np.int64),
                eval_ranks=ranks, eval_scores=scores,
                eval_metrics=np.asarray([metrics[k] for k in ("MRR", "MR", "HITS@1", "HITS@3", "HITS@10")]))
    np.savez_compressed(out, **data)
    print("wrote", out, {k: round(v, 4) for k, v in metrics.items()})


def read_triples(path, e2id, r2id):
    out = []
    with open(path) as f:
        for line in f:
            h, r, t = line.strip().split("\t")
            out.append((e2id[h], r2id[r], e2id[t]))
    return out


def read_dict(path):
    d = {}
    with open(path) as f:
        for line in f:
            i, name = line.strip().split("\t")
            d[name] = int(i)
    return d


def load_dataset(name):
    root = os.path.join(REF, "data", name)
    e2id, r2id = read_dict(os.path.join(root, "entities.dict")), read_dict(os.path.join(root, "relations.dict"))
    tr, va, te = (read_triples(os.path.join(root, f + ".txt"), e2id, r2id) for f in ("train", "valid", "test"))
    return e2id, r2id, tr, va, te


def save_split(out, data, tail):
    """np.savez_compressed of `data` into <name>.npz and <name>.2.npz, so that neither file exceeds 1 MB:
    `tail` maps a key to the first row that goes to the second file (0: the whole array).  tests/conftest.py:load_golden
    joins them again."""
    head = {k: v for k, v in data.items() if tail.get(k) != 0}
    for k, row in tail.items():
        if row:
            head[k] = data[k][:row]
    np.savez_compressed(out, **head)
    np.savez_compressed(out[:-len(".npz")] + ".2.npz", **{k: data[k][row:] for k, row in tail.items()})


def countries_case(out):
    e2id, r2id, tr, va, te = load_dataset("countries_S1")
    with open(os.path.join(REF, "data", "countries_S1", "regions.list")) as f:
        regions = [e2id[line.strip()] for line in f]
    # BASELINE.json configs[0] at its stated shape: -n 64 -b 512 -d 500 -g 0.1 -adv -de (512 rows > 148 SMs)
    nentity, nrelation, d, gamma, B, N = len(e2id), len(r2id), 500, 0.1, 512, 64
    np.random.seed(7)                                   # TrainDataset samples with the global numpy RNG
    torch.manual_seed(7)
    batches = []
    order = np.random.permutation(len(tr))              # 1111 train triples: 512, 512, a ragged 87, then 512 again
    cuts = [(0, B), (B, 2 * B), (2 * B, len(tr)), (0, B)]
    for step, (lo, hi) in enumerate(cuts):
        mode = "tail-batch" if step % 2 == 0 else "head-batch"
        ds = ref_data.TrainDataset(tr, nentity, nrelation, N, mode)
        items = [ds[int(i)] for i in order[lo:hi]]
        batches.append(ref_data.TrainDataset.collate_fn(items))
    m, st = make_ref("RotatE", nentity, nrelation, d, gamma, seed=3)
    lr = 1e-4                                           # best_config uses 2e-6; larger so 4 steps move the tables
    opt = torch.optim.Adam(filter(lambda p: p.requires_grad, m.parameters()), lr=lr)
    args = ns(negative_adversarial_sampling=True, adversarial_temperature=1.0, countries=True,
              regions=regions, nentity=nentity, nrelation=nrelation)
    logs = []
    for log in (ref_model.KGEModel.train_step(m, opt, iter([b]), args) for b in batches):
        logs.append([log["positive_sample_loss"], log["negative_sample_loss"], log["loss"]])
    auc = ref_model.KGEModel.test_step(m, te, tr + va + te, args)["auc_pr"]
    sample, y_true = O.countries_samples(te, regions)
    with torch.no_grad():
        y_score = m(torch.from_numpy(sample)).squeeze(1).numpy()
    args.countries = False
    all_true = tr + va + te
    metrics = ref_model.KGEModel.test_step(m, te, all_true, args)
    ranks, _ = stable_ranks(m, te, all_true, nentity, nrelation)
    data = dict(nentity=nentity, nrelation=nrelation, d=d, gamma=gamma, lr=lr, init_seed=3, regions=np.asarray(regions),
                train=np.asarray(tr, dtype=np.int32), valid=np.asarray(va, dtype=np.int32),
                test=np.asarray(te, dtype=np.int32),      # initial tables: O.init_tables(seed=init_seed), checksummed
                init_checksum=np.float64(st["entity_embedding"].astype(np.float64).sum()),
                logs=np.asarray(logs), final_E=m.entity_embedding.detach().numpy(),
                final_R=m.relation_embedding.detach().numpy(), auc_pr=auc, y_score=y_score, y_true=y_true,
                ranks=ranks, metrics=np.asarray([metrics[k] for k in ("MRR", "MR", "HITS@1", "HITS@3", "HITS@10")]))
    for i, (p, n, w, md) in enumerate(batches):
        data[f"pos{i}"], data[f"neg{i}"], data[f"w{i}"] = p.numpy().astype(np.int16), n.numpy().astype(np.int16), w.numpy()
    save_split(out, data, {"final_E": nentity // 2})
    print("wrote", out, "auc_pr", auc, metrics)


def fullwidth_batches(nentity, nrelation, B, N, steps, seed):
    """Seeded batches of the full-width case (the tests regenerate them with the same call)."""
    rng = np.random.RandomState(seed)
    out = []
    for step in range(steps):
        pos = np.stack([rng.randint(nentity, size=B), rng.randint(nrelation, size=B), rng.randint(nentity, size=B)], 1)
        neg = rng.randint(nentity, size=(B, N))
        w = np.sqrt(1.0 / rng.randint(8, 200, size=B)).astype(np.float32)
        out.append((pos.astype(np.int64), neg.astype(np.int64), w, "tail-batch" if step % 2 == 0 else "head-batch"))
    return out


def fullwidth_case(out):
    """BASELINE.json configs[2] row shape through the UNMODIFIED reference: RotatE, 14,951 x 2000 entity table,
    1,345 relations, N = 256 negatives, gamma 24, -adv, lr 1e-4 -- with B = 192 positive rows (more rows than the
    148 SMs and not a multiple of them: the persistent multi-row loop of the CUDA row kernel), 3 alternating
    steps.  The reference needs ~50 s per 1024-row step on this container, hence 192 rows.  Tables and batches
    are regenerated from seeds by the tests; stored are the losses and, because whole tables would be 120 MB,
    per-row sums of |gradient| (no cancellation) plus sampled full rows of the gradients and the updated tables."""
    nentity, nrelation, d, gamma, B, N, lr = 14951, 1345, 1000, 24.0, 192, 256, 1e-4
    torch.set_num_threads(8)
    m, st = make_ref("RotatE", nentity, nrelation, d, gamma, seed=0)
    batches = fullwidth_batches(nentity, nrelation, B, N, 3, seed=77)
    opt = torch.optim.Adam(filter(lambda p: p.requires_grad, m.parameters()), lr=lr)
    args = ns(negative_adversarial_sampling=True, adversarial_temperature=1.0)
    rng = np.random.RandomState(5)
    touched = np.unique(np.concatenate([batches[0][1].reshape(-1), batches[0][0][:, 0], batches[0][0][:, 2]]))
    ent_rows = np.sort(rng.choice(touched, 48, replace=False))
    rel_rows = np.sort(rng.choice(np.unique(batches[0][0][:, 1]), 24, replace=False))
    data = dict(nentity=nentity, nrelation=nrelation, d=d, gamma=gamma, B=B, N=N, lr=lr, batch_seed=77, init_seed=0,
                ent_rows=ent_rows, rel_rows=rel_rows,
                init_checksum=np.float64(st["entity_embedding"].astype(np.float64).sum()))
    logs = []
    for step, b in enumerate(batches):
        tb = (torch.from_numpy(b[0]), torch.from_numpy(b[1]), torch.from_numpy(b[2]), b[3])
        log = ref_model.KGEModel.train_step(m, opt, iter([tb]), args)
        logs.append([log["positive_sample_loss"], log["negative_sample_loss"], log["loss"]])
        gE, gR = m.entity_embedding.grad.numpy(), m.relation_embedding.grad.numpy()
        data[f"gE{step}_abs_rowsum"] = np.abs(gE.astype(np.float64)).sum(1)
        data[f"gR{step}_abs_rowsum"] = np.abs(gR.astype(np.float64)).sum(1)
        data[f"gE{step}_abs_colsum"] = np.abs(gE.astype(np.float64)).sum(0)
        if step == 0:
            data["gE0_rows"], data["gR0_rows"] = gE[ent_rows].copy(), gR[rel_rows].copy()
        print("full-width step", step, log)
    data["logs"] = np.asarray(logs, dtype=np.float64)
    data["final_E_rows"] = m.entity_embedding.detach().numpy()[ent_rows].copy()
    data["final_R_rows"] = m.relation_embedding.detach().numpy()[rel_rows].copy()
    save_split(out, data, {"final_E_rows": 0, "final_R_rows": 0})
    print("wrote", out)


def wn18rr_case(out, nq=400):
    e2id, r2id, tr, va, te = load_dataset("wn18rr")
    nentity, nrelation, d, gamma = len(e2id), len(r2id), 16, 6.0
    m, st = make_ref("RotatE", nentity, nrelation, d, gamma, seed=11, scale=6.0)
    all_true = tr + va + te
    test = te[:nq]
    ranks, _ = stable_ranks(m, test, all_true, nentity, nrelation)
    metrics = ref_model.KGEModel.test_step(m, test, all_true,
                                           ns(nentity=nentity, nrelation=nrelation, test_batch_size=8, cpu_num=8))
    np.savez_compressed(out, nentity=nentity, nrelation=nrelation, d=d, gamma=gamma, seed=11, scale=6.0,
                        all_true=np.asarray(all_true, dtype=np.int32), test=np.asarray(test, dtype=np.int32),
                        ranks=ranks.astype(np.int32),
                        metrics=np.asarray([metrics[k] for k in ("MRR", "MR", "HITS@1", "HITS@3", "HITS@10")]),
                        table_checksum=np.float64(st["entity_embedding"].astype(np.float64).sum()))
    print("wrote", out, metrics, "stable-rank metrics", O.metrics_from_ranks(ranks))


def runpy_case(out):
    """codes/run.py end to end on the UNMODIFIED reference (CPU): the logged training losses, AUC-PR and filtered metrics
    that tests/test_gpu_runpy.py expects from the same commands on the drop-in (tests/runpy_cases.py)."""
    import json
    import tempfile
    sys.path.insert(0, os.path.join(HERE, ".."))
    import runpy_cases as RC
    data, run_py = os.path.join(REF, "data"), os.path.join(REF, "codes", "run.py")
    work = tempfile.mkdtemp(prefix="kge_runpy_golden_")
    RC.prepare_wn18rr(data, work)
    cmds = RC.commands(data, work)
    logs = {}
    for name in ("countries_train", "countries_resume", "wn18rr_test"):
        RC.run_case(run_py, cmds[name], reference=True, cuda=False)
        log_dir = {"countries_train": f"{work}/countries", "countries_resume": f"{work}/countries_resumed",
                   "wn18rr_test": f"{work}/wn18rr_ckpt"}[name]
        logs[name] = RC.parse_log(os.path.join(log_dir, "train.log" if "countries" in name else "test.log"))
        print(name, len(logs[name]), "metric lines; last:", logs[name][-1])
    with open(out, "w") as f:
        json.dump({"torch": torch.__version__, "seed": 0, "logs": logs}, f, indent=1)
    print("wrote", out)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="")
    a = ap.parse_args()
    if a.only in ("", "small"):
        for name in FLAGS:
            for d in (12, 10):
                small_case(name, d, os.path.join(HERE, f"small_{name}_d{d}.npz"))
    if a.only in ("", "countries"):
        countries_case(os.path.join(HERE, "countries_S1.npz"))
    if a.only in ("", "fullwidth"):
        fullwidth_case(os.path.join(HERE, "fullwidth_RotatE_fb15k.npz"))
    if a.only in ("", "runpy"):
        runpy_case(os.path.join(HERE, "runpy_logs.json"))
    if a.only in ("", "wn18rr"):
        wn18rr_case(os.path.join(HERE, "wn18rr_eval.npz"))
