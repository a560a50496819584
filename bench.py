#!/usr/bin/env python
"""bench.py -- RotatE FB15k (BASELINE.json configs[2]: 14,951 entities, 1,345 relations, d=1000, -n 256 -b 1024
-g 24 -adv -de) train-step throughput in negative-sample scores/s, plus filtered-eval queries/s.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun by the driver)
    python bench.py --impl reference ...                     (the reference's CPU path on the host cores)
    python bench.py ... --dump-outputs DIR                   (also write what the timed steps computed, DIR/*.npy)

One JSON line on stdout (rank 0).  A "step" is one full KGEModel.train_step: gather+score+loss+backward, dense
Adam, loss read-back excluded for `value` (inputs resident in HBM) and included for `e2e` (host batches).

Reference arm: the UNMODIFIED reference (baseline/_ref/codes, copied from /root/reference by __graft_entry__.build();
git-ignored, travels with gpurun) through its own KGEModel.train_step on torch-CPU with every host thread, on a bounded
sample of rows per step (the reference needs ~50 s for one full 1024-row step); when baseline/_ref is absent the C/OpenMP
restatement oracle/kge_oracle.c is timed instead (kind "port").  The GPU arm also reports, as extras, the port's full-batch
rate, the reference's own torch-CUDA eager path on the same B200 ("reference_cuda": the practical bar), an oracle parity
check of the timed path, and the other BASELINE configs (TransE FB15k-237, ComplEx wn18rr incl. the tcgen05 eval, RotatE
YAGO3-10).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
REF_CODES = os.path.join(ROOT, "baseline", "_ref", "codes")

WORKLOADS = {
    # name: (model, nentity, nrelation, d, gamma, B, N, lr, de, dr, regularization, filter triples)   [best_config.sh]
    "rotate_fb15k": ("RotatE", 14951, 1345, 1000, 24.0, 1024, 256, 1e-4, True, False, 0.0, 483142),
    "transe_fb15k237": ("TransE", 14541, 237, 1000, 9.0, 1024, 256, 5e-5, False, False, 0.0, 272115),
    "rotate_yago310": ("RotatE", 123182, 37, 500, 24.0, 1024, 400, 2e-4, True, False, 0.0, 1079040),
    "complex_wn18rr": ("ComplEx", 40943, 11, 500, 200.0, 512, 1024, 2e-3, True, True, 5e-6, 86835),
    "distmult_fb15k": ("DistMult", 14951, 1345, 2000, 500.0, 1024, 256, 1e-3, False, False, 2e-6, 483142),
}
METRIC = "rotate_negative_sample_scores_per_sec_train_step"


def make_config(wl, world):
    """The `config` object of BOTH arms (same keys and values: the driver compares them)."""
    model, nentity, nrel, d, gamma, B, N, lr, de, dr, reg, _ = WORKLOADS[wl]
    return {"workload": wl, "score_function": model, "nentity": nentity, "nrelation": nrel, "hidden_dim": d,
            "negative_sample_size": N, "batch_size_per_gpu": B, "positives_per_step": B * world, "gamma": gamma,
            "adversarial": True, "double_entity_embedding": de, "double_relation_embedding": dr,
            "regularization": reg, "learning_rate": lr,
            "sharding": f"positive rows over {world} rank(s), tables replicated; eval: entity slices",
            "l2_policy": "no flush: each step streams >= 0.5 GB of tables+moments (> 126 MB L2)"}


def make_batches(nentity, nrel, B, N, count, seed):
    rng = np.random.RandomState(seed)
    out = []
    for i in range(count):
        pos = np.stack([rng.randint(nentity, size=B), rng.randint(nrel, size=B), rng.randint(nentity, size=B)], 1)
        neg = rng.randint(nentity, size=(B, N))
        w = np.sqrt(1.0 / rng.randint(8, 200, size=B)).astype(np.float32)
        out.append((pos.astype(np.int64), neg.astype(np.int64), w, "tail-batch" if i % 2 == 0 else "head-batch"))
    return out


def train_bytes(B, N, De, Dr):
    """Algorithmic bytes of score + loss + backward (DESIGN.md section 5 / SURVEY 8d `A_train`)."""
    return B * N * De * 4 * 2 + B * N * 8 + 2 * B * (De + Dr) * 4 + B * 28


def adam_bytes(numel):
    """SURVEY 8d `A_adam`: read p, g, m, v; write p, m, v."""
    return 7 * numel * 4


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed regions: in-process NVML every 5 ms (pynvml; a query costs
    tens of microseconds of a host thread), or an `nvidia-smi -lms 100` child as the fallback."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index
        self.nvml, self.samples, self.bits, self.stop_flag, self.thread = None, [], 0, False, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # LOCAL_RANK indexes the visible devices; NVML wants the physical one
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.gpu]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else self.gpu
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.QUERY}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _poll(self):
        nv = self.nvml
        reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_flag:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)))
                self.bits |= int(reasons(self.handle))
            except Exception:
                pass
            time.sleep(0.005)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=1.0)
            return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                    "reasons": sorted(n for b, n in self.REASONS.items() if self.bits & b), "samples": len(self.samples),
                    "source": "nvml, 5 ms period, over the timed train regions"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 8 for n, v in zip(names, r[4:8]) if v.startswith("Active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "source": "nvidia-smi -lms 100"}


def ncu_traffic(wl):
    """DRAM bytes per train-path launch, NOT measured in this run: read from the committed `ncu --set full` capture of
    the same command (dram__bytes_read.sum + dram__bytes_write.sum of the row kernel + entity kernel)."""
    if wl != "rotate_fb15k":
        return None, None
    import csv
    import glob
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "prof_train_r*.raw.csv")), reverse=True):
        rows = list(csv.reader(open(path)))
        hdr, units = rows[0], rows[1]
        per_kernel = {}                                 # the capture may hold several launches (steps) of each kernel
        for r in rows[2:]:
            kind = "row" if "row_kernel_split" in r[0] else ("entity" if "entity_kernel" in r[0] else None)
            if kind is None:
                continue
            t = 0.0
            for name in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                i = hdr.index(name)
                scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[units[i]]
                t += float(r[i]) * scale
            per_kernel.setdefault(kind, []).append(t)
        total = sum(sum(v) / len(v) for v in per_kernel.values())
        if total:
            return total, "not measured in this run: " + os.path.relpath(path, ROOT) + " (ncu --set full of this command)"
    return None, None


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
            return p, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops_sustained": 1418.0}, "fallback (B200_PROFILING.md)"


def row_sample(table, budget, seed=0):
    """Rows of a (rows, dim) device table as float32 host data, at most `budget` bytes: every row when they fit, else a
    fixed seeded sample of rows in ascending order (the same rows on every run of the same workload)."""
    t = table.detach().reshape(table.shape[0], -1)
    k = min(t.shape[0], max(1, budget // (t.shape[1] * 4)))
    if k < t.shape[0]:
        rows = np.sort(np.random.RandomState(seed).choice(t.shape[0], k, replace=False))
        t = t[rows]
    return t.float().cpu().numpy()


def train_outputs(m, loss_buffer):
    """What a caller of the timed train step receives from its last call: the loss buffer's [positive_sample_loss,
    negative_sample_loss, loss, regularization] and every trainable table (each at most 28 MB: a seeded row sample)."""
    out = {"train_losses": loss_buffer[:4].cpu().numpy()}
    for name, p in m.named_parameters():
        if p.requires_grad:
            out[name] = row_sample(p, 28 << 20)
    return out


def dump_outputs(path, arrays):
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        np.save(os.path.join(path, name + ".npy"), a if a.dtype in (np.float32, np.float64) else a.astype(np.float64))


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


# ---------------------------------------------------------------------------------------------- reference helpers
def load_reference():
    """The unmodified reference modules from baseline/_ref/codes (None when the copy is absent)."""
    if not os.path.exists(os.path.join(REF_CODES, "model.py")):
        return None
    import importlib.util
    mods = {}
    for name in ("dataloader", "model"):
        spec = importlib.util.spec_from_file_location("kge_reference_" + name, os.path.join(REF_CODES, name + ".py"))
        mod = importlib.util.module_from_spec(spec)
        if name == "model":                       # model.py does `from dataloader import TestDataset`
            sys.modules.setdefault("dataloader", mods["dataloader"])
        spec.loader.exec_module(mod)
        mods[name] = mod
    return mods


def reference_model(mods, wl, tables, device):
    import torch
    model, nentity, nrel, d, gamma, B, N, lr, de, dr, reg, _ = WORKLOADS[wl]
    m = mods["model"].KGEModel(model_name=model, nentity=nentity, nrelation=nrel, hidden_dim=d, gamma=gamma,
                               double_entity_embedding=de, double_relation_embedding=dr)
    with torch.no_grad():
        m.entity_embedding.copy_(torch.from_numpy(tables["entity_embedding"]))
        m.relation_embedding.copy_(torch.from_numpy(tables["relation_embedding"]))
    return m.to(device)


def reference_args(wl, cuda):
    model, nentity, nrel, d, gamma, B, N, lr, de, dr, reg, _ = WORKLOADS[wl]
    return types.SimpleNamespace(cuda=cuda, negative_adversarial_sampling=True, adversarial_temperature=1.0,
                                 uni_weight=False, regularization=reg, countries=False, regions=None,
                                 test_batch_size=16, cpu_num=2, test_log_steps=100000, nentity=nentity, nrelation=nrel)


def time_reference_train(mods, wl, rows, steps, warmup, cuda):
    """The unmodified reference KGEModel.train_step (model.py:251-312) on `rows` positive rows x N negatives per step,
    full tables, stock torch.optim.Adam; returns (scores/s, seconds per step)."""
    import torch
    from oracle import kge_oracle as O
    model, nentity, nrel, d, gamma, B, N, lr, de, dr, reg, _ = WORKLOADS[wl]
    tables = O.init_tables(model, nentity, nrel, d, gamma, de, dr, seed=0)
    dev = torch.device("cuda") if cuda else torch.device("cpu")
    m = reference_model(mods, wl, tables, dev)
    opt = torch.optim.Adam(filter(lambda p: p.requires_grad, m.parameters()), lr=lr)
    args = reference_args(wl, cuda)
    batches = [(torch.from_numpy(p), torch.from_numpy(n), torch.from_numpy(w), md)
               for p, n, w, md in make_batches(nentity, nrel, rows, N, steps + warmup, seed=1)]
    if cuda:
        batches = [(p.pin_memory(), n.pin_memory(), w.pin_memory(), md) for p, n, w, md in batches]
    it = iter(batches)
    for _ in range(warmup):
        mods["model"].KGEModel.train_step(m, opt, it, args)
    if cuda:
        torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        mods["model"].KGEModel.train_step(m, opt, it, args)        # (its .item() calls synchronise)
    if cuda:
        torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return rows * N / dt, dt


def time_reference_eval(mods, wl, all_true, test, cuda):
    """The unmodified reference KGEModel.test_step (model.py:314-429: TestDataset + DataLoader + forward + argsort) on a
    few test triples; returns (queries/s, seconds, metrics)."""
    import torch
    from oracle import kge_oracle as O
    model, nentity, nrel, d, gamma, B, N, lr, de, dr, reg, _ = WORKLOADS[wl]
    tables = O.init_tables(model, nentity, nrel, d, gamma, de, dr, seed=0)
    m = reference_model(mods, wl, tables, torch.device("cuda") if cuda else torch.device("cpu"))
    args = reference_args(wl, cuda)
    t0 = time.perf_counter()
    metrics = mods["model"].KGEModel.test_step(m, test, all_true, args)
    if cuda:
        torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return 2 * len(test) / dt, dt, metrics


def cpu_port_train(wl, rows, steps, warmup, threads):
    """The reference's train_step restated by the C/OpenMP oracle on the host cores, on the first `rows` positive rows
    of each batch at full width (N negatives, full tables incl. the dense Adam)."""
    from oracle import c_oracle as C
    from oracle import kge_oracle as O
    model, nentity, nrel, d, gamma, B, N, lr, de, dr, reg, _ = WORKLOADS[wl]
    C.set_num_threads(threads)
    st = O.init_tables(model, nentity, nrel, d, gamma, de, dr, seed=0)
    batches = make_batches(nentity, nrel, rows, N, steps + warmup, seed=1)
    state = C.TrainState(model, st, gamma, d)
    for b in batches[:warmup]:
        C.train_step(state, b, lr=lr, adversarial=True, alpha=1.0, regularization=reg)
    t0 = time.perf_counter()
    for b in batches[warmup:]:
        C.train_step(state, b, lr=lr, adversarial=True, alpha=1.0, regularization=reg)
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return rows * N / dt, dt, C.num_threads()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = max(1, int(os.environ.get("WORLD_SIZE", str(args.gpus))))
    wl = args.workload
    model, nentity, nrel, d, gamma, B, N, lr, de, dr, reg, _ = WORKLOADS[wl]
    cores = host_cores()
    mods = None if args.reference_kind == "port" else load_reference()
    if mods is not None:
        import torch
        torch.set_num_threads(cores)              # torchrun exports OMP_NUM_THREADS=1: use every host core explicitly
        rows = args.cpu_rows or 16
        value, dt = time_reference_train(mods, wl, rows, args.steps, args.warmup, cuda=False)
        kind = "reference"
        sample = (f"unmodified reference (baseline/_ref/codes/model.py KGEModel.train_step, torch {torch.__version__} CPU, "
                  f"{torch.get_num_threads()} threads): {rows} of the {B * world} positive rows of a step x {N} negatives "
                  f"at full width per step, full {nentity} x {d * (2 if de else 1)} tables, stock torch.optim.Adam included")
        pv, pdt, pthreads = cpu_port_train(wl, B, 2, 1, cores)
        extra = {"cpu_port": {"value": pv, "unit": "scores/s", "cores": pthreads, "kind": "port",
                              "sample": f"oracle/kge_oracle.c (C/OpenMP restatement), full {B}-row batch, 2 steps after 1"}}
    else:
        rows = args.cpu_rows or B
        value, dt, cores = cpu_port_train(wl, rows, args.steps, args.warmup, cores)
        kind = "port"
        sample = (f"oracle/kge_oracle.c (C/OpenMP restatement of model.py:251-312; baseline/_ref absent): {rows} of "
                  f"{B * world} positive rows x {N} negatives per step at full width, full-table dense Adam included")
        extra = {}
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "scores/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": make_config(wl, world),
        "cpu_baseline": {"value": value, "unit": "scores/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "scores/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        **extra,
    }
    emit(line)


# ---------------------------------------------------------------------------------------------- GPU arm
def synthetic_triples(nentity, nrel, count, seed):
    rng = np.random.RandomState(seed)
    h, r, t = rng.randint(nentity, size=count), rng.randint(nrel, size=count), rng.randint(nentity, size=count)
    keys = np.unique((h.astype(np.int64) * nrel + r) * nentity + t)
    h, rem = np.divmod(keys, nrel * nentity)
    r, t = np.divmod(rem, nentity)
    return list(zip(h.tolist(), r.tolist(), t.tolist())), rng


class Bench:
    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.args = torch, dist, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def timed(self, fn, steps, warmup):
        torch = self.torch
        for i in range(warmup):
            fn(i)
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(warmup + i)
        e1.record()
        self.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(ms, op=self.dist.ReduceOp.MAX)               # max over ranks
        return float(ms.item())

    def build_model(self, wl):
        torch = self.torch
        from knowledgegraphembedding_b200 import KGEModel
        from oracle import kge_oracle as O          # only the portable synthetic table initialiser
        model, nentity, nrel, d, gamma, B, N, lr, de, dr, reg, _ = WORKLOADS[wl]
        st = O.init_tables(model, nentity, nrel, d, gamma, de, dr, seed=0)
        m = KGEModel(model, nentity, nrel, d, gamma, double_entity_embedding=de, double_relation_embedding=dr)
        with torch.no_grad():
            m.entity_embedding.copy_(torch.from_numpy(st["entity_embedding"]))
            m.relation_embedding.copy_(torch.from_numpy(st["relation_embedding"]))
        m = m.to(self.dev)
        opt = torch.optim.Adam(filter(lambda p: p.requires_grad, m.parameters()), lr=lr)
        targs = types.SimpleNamespace(cuda=True, negative_adversarial_sampling=True, adversarial_temperature=1.0,
                                      uni_weight=False, regularization=reg)
        return m, opt, targs, st

    def train(self, wl, steps, warmup, e2e=True, outputs=False):
        """value (device-resident inputs), kernel timing, e2e (public KGEModel.train_step on pinned host batches).
        outputs: also return train_outputs() of the last timed device step (taken before the e2e steps go on)."""
        torch = self.torch
        from knowledgegraphembedding_b200 import KGEModel
        model, nentity, nrel, d, gamma, B, N, lr, de, dr, reg, _ = WORKLOADS[wl]
        world, dev = self.world, self.dev
        Bg = B * world                                   # weak scaling: every rank keeps B rows of the global batch
        m, opt, targs, _ = self.build_model(wl)
        pool = make_batches(nentity, nrel, Bg, N, min(steps + warmup, 32), seed=1)            # same batches on every rank
        dev_pool = [(torch.from_numpy(p).to(dev), torch.from_numpy(n).to(dev), torch.from_numpy(w).to(dev), md)
                    for p, n, w, md in pool]
        m.train()

        device_out = {}

        def step_device(i):
            device_out["loss"] = m.train_step_async(opt, dev_pool[i % len(dev_pool)], targs)

        m._ws['kernel_events'] = None
        for i in range(warmup):
            step_device(i)
        m._ws['kernel_events'] = events = []
        m._ws['exchange_events'] = xevents = []
        ms_total = self.timed(step_device, steps, 0)
        m._ws['kernel_events'] = m._ws['exchange_events'] = None
        out = {"ms_per_step": ms_total / steps, "value": Bg * N / (ms_total / steps * 1e-3),
               "row_ms": float(np.mean([a.elapsed_time(b) for a, b in events])) if events else None,
               "exchange_ms": float(np.mean([a.elapsed_time(b) for a, b in xevents])) if xevents else None,
               "fused_entity_adam": m.entity_embedding.grad is None, "model": m, "opt": opt, "targs": targs}
        if outputs:
            out["outputs"] = train_outputs(m, device_out["loss"])
        px = m._ws.get('peer')
        out["peer"] = px
        out["shard"] = m._ws.get('shard') or None
        out["nreg"] = int(m._ws.get('exchange_regions', 1)) if px else 1
        if e2e:
            pin_pool = [(torch.from_numpy(p).pin_memory(), torch.from_numpy(n).pin_memory(),
                         torch.from_numpy(w).pin_memory(), md) for p, n, w, md in pool]
            # a training loop recycles its pinned buffers (the pinned-memory allocator hands freed blocks out again), so
            # the device has read every buffer before: one untimed copy per pool entry; the timed steps still copy
            # their whole batch host -> device
            for p, n, w, _ in pin_pool:
                p.to(dev), n.to(dev), w.to(dev)
            torch.cuda.synchronize(dev)
            it_state = {"i": 0}

            class HostIterator:
                def __next__(self):
                    b = pin_pool[it_state["i"] % len(pin_pool)]
                    it_state["i"] += 1
                    return b

            host_it, last = HostIterator(), {}

            def step_host(i):
                last.update(KGEModel.train_step(m, opt, host_it, targs))

            out["ms_e2e"] = self.timed(step_host, steps, warmup) / steps
            out["e2e_value"] = Bg * N / (out["ms_e2e"] * 1e-3)
            out["last_loss"] = last.get("loss")
            # every rank copies its own rows (+ the whole weight vector); one 32-byte loss read-back
            out["h2d"] = world * (B * 3 * 8 + B * N * 8 + Bg * 4)
            out["d2h"] = 8 * 4
        return out

    def parity(self, wl, steps=2):
        """The timed path against the C oracle on the same seeded full batches (losses 1e-5, tables outlier bound);
        raises if it fails: a fast kernel whose results differ from the reference's is not done.  Multi-GPU: the ranks
        step the GLOBAL batch (B rows per rank) together, rank 0 runs the oracle's single-device step on all of it."""
        torch = self.torch
        from knowledgegraphembedding_b200 import KGEModel
        model, nentity, nrel, d, gamma, B, N, lr, de, dr, reg, _ = WORKLOADS[wl]
        m, opt, targs, st = self.build_model(wl)
        ts = None
        if self.rank == 0:
            from oracle import c_oracle as C
            C.set_num_threads(host_cores())              # (torchrun exports OMP_NUM_THREADS=1)
            ts = C.TrainState(model, st, gamma, d)
        worst = 0.0
        for b in make_batches(nentity, nrel, B * self.world, N, steps, seed=11):
            log = KGEModel.train_step(m, opt, iter([tuple(torch.from_numpy(x) if isinstance(x, np.ndarray) else x
                                                          for x in b)]), targs)
            if ts is not None:
                ref = C.train_step(ts, b, lr=lr, adversarial=True, alpha=1.0, regularization=reg)
                worst = max(worst, max(abs(log[k] - ref[k]) / abs(ref[k]) for k in ref))
            self.barrier()       # the other ranks wait here on the host, not inside the next step's bounded GPU barrier
        self.barrier()
        if ts is None:
            return None
        E = m.entity_embedding.detach().cpu().numpy()
        bad = float(np.mean(np.abs(E - ts.state["entity_embedding"]) > 1e-5 * np.abs(ts.state["entity_embedding"]).max()))
        ok = worst <= 1e-5 and bad < 1e-4
        res = {"against": "oracle/kge_oracle.c full-batch train_step (pinned to the reference's goldens)", "steps": steps,
               "global_rows": B * self.world, "max_rel_loss_err": worst, "entity_table_outlier_fraction": bad,
               "tolerance": 1e-5, "ok": bool(ok)}
        if not ok:
            raise SystemExit("bench.py parity check failed: " + json.dumps(res))
        return res

    def eval(self, wl, m, nq, reps=3):
        """KGEModel.filtered_ranks end to end (host triples in, host ranks out), entity-sharded over the ranks: once cold
        (filter index built from the python list + uploads) and warm (index cached, as across valid/test of one run)."""
        model, nentity, nrel, d, gamma, B, N, lr, de, dr, reg, ntrue = WORKLOADS[wl]
        all_true, rng = synthetic_triples(nentity, nrel, ntrue, seed=2)
        test = [all_true[i] for i in rng.choice(len(all_true), nq, replace=False)]
        self.barrier()
        t0 = time.perf_counter()
        for mode in ("head-batch", "tail-batch"):
            m.filtered_ranks(test, all_true, mode)
        self.barrier()
        cold_s = time.perf_counter() - t0
        m._ws['eval_events'] = eval_events = []
        self.barrier()
        t0 = time.perf_counter()
        ranks = {}
        for _ in range(reps):
            for mode in ("head-batch", "tail-batch"):
                ranks[mode] = m.filtered_ranks(test, all_true, mode)   # host triples in, host ranks out
        self.barrier()
        eval_s = (time.perf_counter() - t0) / reps
        m._ws['eval_events'] = None
        kernel_ms = sum(a.elapsed_time(b) for a, b in eval_events) / reps
        return {"metric": "filtered_eval_queries_per_sec", "value": 2 * nq / eval_s, "queries": 2 * nq, "seconds": eval_s,
                "what": "KGEModel.filtered_ranks end to end, warm: host triples -> H2D -> filter lookup + count kernels -> "
                        "host ranks; the filter index of all_true_triples is cached from the cold call",
                "cold": {"value": 2 * nq / cold_s, "seconds": cold_s,
                         "what": "first call: python list of all true triples -> int64 array on the host, H2D, filter index built on the device (counting sort)"},
                "count_kernel_ms": kernel_ms, "count_kernel_queries_per_sec": 2 * nq / (kernel_ms * 1e-3) if kernel_ms else None,
                "sharding": f"entities/{self.world}", "filter_triples": len(all_true)}, all_true, test, ranks


def run_gpu(args):
    b = Bench(args)
    torch, world, rank, dev = b.torch, b.world, b.rank, b.dev
    wl = args.workload
    model, nentity, nrel, d, gamma, B, N, lr, de, dr, reg, _ = WORKLOADS[wl]
    pk, peak_src = peaks()
    sampler = ClockSampler(b.local)
    sampler.start()
    tr = b.train(wl, args.steps, args.warmup, outputs=bool(args.dump_outputs) and rank == 0)
    clocks = sampler.stop()
    m = tr["model"]
    De, Dr = m.entity_dim, m.relation_dim
    ev, all_true, test, eval_ranks = b.eval(wl, m, args.eval_queries)

    # ---- the other BASELINE configs (cfg 2, 4, 5), shorter runs ------------------------------------------------------
    extras = {}
    if not args.no_extras:
        del tr["model"], tr["opt"]
        m = None
        torch.cuda.empty_cache()
        for name in ("transe_fb15k237", "complex_wn18rr", "rotate_yago310"):
            if name == wl:
                continue
            w = WORKLOADS[name]
            t2 = b.train(name, args.steps, args.warmup)
            m2 = t2["model"]
            a_tr = train_bytes(w[5], w[6], m2.entity_dim, m2.relation_dim)
            a_ad = adam_bytes(m2.entity_embedding.numel() + m2.relation_embedding.numel())
            e2, _, _, _ = b.eval(name, m2, 2048 if name != "rotate_yago310" else 1024, reps=2)
            entry = {"config": make_config(name, world), "value": t2["value"], "unit": "scores/s",
                     "ms_per_step": t2["ms_per_step"], "e2e": {"value": t2["e2e_value"], "ms_per_step": t2["ms_e2e"]},
                     "fused_entity_adam": t2["fused_entity_adam"],
                     "full_step_roofline": {"bound": "hbm", "algorithmic_bytes": a_tr + a_ad,
                                            "achieved": (a_tr + a_ad) / (t2["ms_per_step"] * 1e-3) / 1e9,
                                            "peak": pk["hbm_gbs"], "unit": "GB/s",
                                            "frac": (a_tr + a_ad) / (t2["ms_per_step"] * 1e-3) / 1e9 / pk["hbm_gbs"]},
                     "eval": e2}
            if name == "complex_wn18rr" and e2["count_kernel_ms"]:
                # tcgen05 path: 3 TF32 MMAs (hi*hi + hi*lo + lo*hi) per product => 3 x 2 x Q x nentity x 2d tensor flops
                flops = 3 * 2.0 * e2["queries"] * w[1] * m2.entity_dim / world
                tf = flops / (e2["count_kernel_ms"] * 1e-3) / 1e12
                tpeak = pk.get("bf16_tflops_sustained", 1418.0) / 2.0
                entry["eval"]["roofline"] = {"bound": "tensor", "kernel": "gemm_count_kernel (tcgen05.mma kind::tf32, 3xTF32 split)",
                                             "achieved": tf, "peak": tpeak, "unit": "TFLOP/s", "frac": tf / tpeak,
                                             "peak_source": peak_src + " bf16_tflops_sustained / 2 (TF32 rate)",
                                             "note": "kernel time includes the exact re-score of the ambiguous band"}
            extras[name] = entry
            del t2, m2
            torch.cuda.empty_cache()

    parity = b.parity(wl) if not args.no_parity else None

    if rank != 0:
        if world > 1:
            b.dist.destroy_process_group()
        return

    # ---- rooflines -----------------------------------------------------------------------------------------------------
    sm_mhz = (clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965.0)
    if model == "RotatE" and ev["count_kernel_ms"]:
        # what bounds the distance-model ranking kernel: one square root per (query, entity, complex dimension) on the
        # MUFU pipe, 16 results per clock and SM (DESIGN.md section 3.3 / SURVEY 8d); peak at the sampled SM clock
        sqrt_per_s = ev["queries"] * nentity * d / (ev["count_kernel_ms"] * 1e-3) / world      # per GPU: its entity slice
        peak_sqrt = 148 * 16 * sm_mhz * 1e6
        ev["roofline"] = {"bound": "mufu (1 sqrt per query x entity x complex dim, 16/clk/SM)",
                          "achieved": sqrt_per_s / 1e9, "peak": peak_sqrt / 1e9, "unit": "Gsqrt/s per GPU",
                          "frac": sqrt_per_s / peak_sqrt}
    a_train = train_bytes(B, N, De, Dr)
    a_adam_e = adam_bytes(nentity * De)
    fused = tr["fused_entity_adam"]
    roofline = None
    if tr["row_ms"]:
        a_bytes = a_train + (a_adam_e if fused else 0)
        ach = a_bytes / (tr["row_ms"] * 1e-3) / 1e9
        traffic, traffic_src = ncu_traffic(wl)
        roofline = {"bound": "hbm",
                    "kernel": ("kge_train_rows_adam: row_kernel_split + counting sort + entity_kernel with the entity table's "
                               "Adam update fused in" if fused else
                               "kge_train_rows: row_kernel_split + counting sort + entity_kernel"),
                    "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"],
                    "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src + " hbm_gbs",
                    "algorithmic_bytes_per_launch": a_bytes,
                    "algorithmic_bytes_what": "A_train (gather + scatter formulation of the reference, SURVEY 8d)"
                                              + (" + A_adam of the entity table (7 streams)" if fused else ""),
                    "avg_launch_ms": tr["row_ms"]}
        l2 = os.path.join(ROOT, "profiles", "l2_gather_r2.json")
        if os.path.exists(l2):
            try:
                rows = [json.loads(x) for x in open(l2) if x.strip().startswith("{")]
                best = max(r["gather_gbs_depth2"] for r in rows if "fits_L2" in r["table"])
                roofline["l2_gather"] = {"what": "the kernel does not stream from HBM: the 120 MB table is L2-resident; measured "
                                                 "L2->SM ceiling for this access pattern (tools/l2_gather_bench.cu, 8 KB rows, "
                                                 "cp.async.bulk, random ids), not measured in this run",
                                         "peak_gbs": best, "gather_bytes_per_launch": B * N * De * 4}
            except Exception:
                pass
    cores = host_cores()
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        mods = load_reference()
        if mods is not None:
            torch.set_num_threads(cores)
            rows = args.cpu_rows or 16
            v, dt = time_reference_train(mods, wl, rows, 3, 1, cuda=False)
            cpu = {"value": v, "unit": "scores/s", "cores": cores, "kind": "reference",
                   "sample": f"unmodified reference (baseline/_ref/codes/model.py KGEModel.train_step, torch CPU, {cores} "
                             f"threads): {rows} of {B} positive rows x {N} negatives per step at full width, full tables, "
                             f"stock Adam; 3 steps after 1 warm-up ({dt:.2f} s/step)"}
            qv, qdt, _ = time_reference_eval(mods, wl, all_true, test[:16], cuda=False)
            ev["cpu_baseline"] = {"value": qv, "unit": "queries/s", "cores": cores, "kind": "reference",
                                  "sample": f"unmodified reference KGEModel.test_step (TestDataset + DataLoader + forward + "
                                            f"argsort) on 16 test triples x 2 modes, same tables and filter list ({qdt:.1f} s)"}
            try:                                    # the practical bar: the reference's own eager torch-CUDA path, same B200
                torch.cuda.empty_cache()
                cv, cdt = time_reference_train(mods, wl, B, 5, 2, cuda=True)
                cq, cqdt, _ = time_reference_eval(mods, wl, all_true, test[:64], cuda=True)
                ref_cuda = {"what": "unmodified reference with args.cuda=True on this GPU (eager torch kernels)",
                            "train_value": cv, "train_unit": "scores/s", "train_ms_per_step": cdt * 1e3,
                            "eval_value": cq, "eval_unit": "queries/s", "eval_queries": 128,
                            "speedup_e2e_train": tr["e2e_value"] / cv, "speedup_eval": ev["value"] / cq}
            except Exception as exc:                # e.g. out of memory on a smaller device
                ref_cuda = {"unavailable": repr(exc)[:200]}
        else:
            ref_cuda = {"unavailable": "baseline/_ref/codes absent"}
        pv, pdt, pthreads = cpu_port_train(wl, B, 3, 1, cores)
        port = {"value": pv, "unit": "scores/s", "cores": pthreads, "kind": "port",
                "sample": f"oracle/kge_oracle.c (C/OpenMP restatement), full {B}-row batch, 3 steps after 1 warm-up"}
        if cpu is None:
            cpu = port
    else:
        ref_cuda = port = None
    px = tr["peer"]
    sh = tr["shard"]
    if sh:
        exchange_path = ("entity-sharded optimizer over nvlink_peer_memory/%s: row kernel stores q / dL/ds / ids into every rank's "
                         "gather area, owners run sort + entity-major backward + fused Adam and store the updated rows into "
                         "every replica (kge_train_rows_sharded / kge_train_entity_sharded); exposed = wait for the relation-table exchange "
                         "(kge_peer_reduce_adam on a second stream) + final barrier" % sh['peer'].backend)
    else:
        exchange_path = ("nvlink_peer_memory/%s%s (kge_peer_reduce_adam)" % (px.backend, "+nvswitch_multicast" if px.multicast else "")
                         if px else ("nccl_allreduce + kge_adam_step" if world > 1 else
                                     ("entity Adam fused in kge_train_rows_adam + kge_adam_step over R" if fused else "kge_adam_step")))
    # kernels of libkge_b200.so per step: weight_sum, row_kernel_split, scan_tiles, scan_apply, scatter_pairs,
    # entity_kernel per region, loss_finalize, and adam_kernel (1 GPU / NCCL path) or peer_reduce_adam + peer_finish per region
    nreg = tr["nreg"]
    line = {
        "metric": METRIC, "value": tr["value"], "unit": "scores/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": tr["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": make_config(wl, world),
        # sharded step: weight_sum, push_ids, row_kernel_split, 2 barriers, 2 gathered_pairs, 2 scans, entity_kernel,
        # peer_reduce_adam, peer_finish, loss_finalize
        "clocks": clocks, "gpu_launches": (13 if sh else 6 + nreg + (2 * nreg if px else 1)) * args.steps,
        "e2e": {"value": tr["e2e_value"], "unit": "scores/s", "ms_per_step": tr["ms_e2e"], "h2d_bytes_per_step": tr["h2d"],
                "d2h_bytes_per_step": tr["d2h"], "last_loss": tr["last_loss"],
                "what": "KGEModel.train_step (default settings: one next() per call, H2D on the compute stream) on pinned "
                        "host batches, log dict read back every step"},
        "roofline": roofline, "cpu_baseline": cpu, "cpu_port": port, "reference_cuda": ref_cuda, "parity_check": parity,
        "full_step_roofline": {"bound": "hbm", "algorithmic_bytes": a_train + adam_bytes(nentity * De + nrel * Dr),
                               "achieved": (a_train + adam_bytes(nentity * De + nrel * Dr)) / (tr["ms_per_step"] * 1e-3) / 1e9,
                               "peak": pk["hbm_gbs"], "unit": "GB/s",
                               "frac": (a_train + adam_bytes(nentity * De + nrel * Dr)) / (tr["ms_per_step"] * 1e-3) / 1e9 / pk["hbm_gbs"]},
        "exchange": {"path": exchange_path, "exposed_exchange_and_optimizer_ms": tr["exchange_ms"],
                     "regions_per_step": nreg,
                     "bytes_reduced_per_rank": (4 * nrel * Dr if sh else 4 * (nentity * De + nrel * Dr)) if world > 1 else 0,
                     "nvlink_bytes_in_per_rank": (int((world - 1) * (4 * nentity * De / world + B * (De + 2 * N) * 4
                                                                      + 3 * B * De * 4 / world)) if sh else None)},
        "eval": ev, "workloads": extras,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {**tr["outputs"], "eval_ranks_head_batch": eval_ranks["head-batch"],
                                         "eval_ranks_tail_batch": eval_ranks["tail-batch"]})
    emit(line)
    if world > 1:
        b.dist.destroy_process_group()


_REAL_STDOUT = None


def protect_stdout():
    """Libraries (NCCL's version banner, for one) print to stdout; the driver wants exactly one JSON line there.
    Route fd 1 to stderr for the run and keep the real stdout for the result line."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    protect_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed train steps of every GPU workload, at least 1 (the CPU baselines reported beside "
                         "them keep their own short fixed counts: one reference step takes seconds)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="rotate_fb15k", choices=list(WORKLOADS))
    ap.add_argument("--cpu-rows", type=int, default=0,
                    help="positive rows per CPU step (0 = 16 for the reference's torch-CPU path, the full batch for the port)")
    ap.add_argument("--reference-kind", default="auto", choices=["auto", "port"],
                    help="--impl reference: 'auto' = the unmodified reference when baseline/_ref exists, else the C port")
    ap.add_argument("--eval-queries", type=int, default=8192)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the other BASELINE configs")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--negatives", type=int, default=0, help="experiments: override the workload's negative_sample_size")
    ap.add_argument("--batch", type=int, default=0, help="experiments: override the workload's batch size per GPU")
    ap.add_argument("--entities", type=int, default=0, help="experiments: override the workload's entity count")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="GPU arm, rank 0: after the run, write DIR/<name>.npy (float32/float64, < 64 MB in all) with what "
                         "the last timed train step returned (train_losses, and the updated tables: entity_embedding is a "
                         "seeded row sample when it exceeds 28 MB) and the ranks of the last timed evaluation")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU arm computed: it does not apply to --impl reference")
    if args.negatives or args.batch or args.entities:     # (shows up in `config`: not the BASELINE workload any more)
        w = list(WORKLOADS[args.workload])
        w[1], w[5], w[6] = args.entities or w[1], args.batch or w[5], args.negatives or w[6]
        w[11] = min(w[11], 20 * w[1])
        WORKLOADS[args.workload] = tuple(w)
    if args.impl == "reference":
        # torchrun exports OMP_NUM_THREADS=1 to every rank: the CPU arm uses all host cores explicitly
        os.environ["OMP_NUM_THREADS"] = str(host_cores())
        run_reference(args)
    else:
        if args.warmup < 3:
            args.warmup = 3
        run_gpu(args)


if __name__ == "__main__":
    main()
