#!/usr/bin/env python
"""bench.py — CTR examples/sec of the Wide&Deep train step on N B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torch.distributed.run)
    python bench.py --impl reference ...                      (optimised CPU restatement of the reference step, host cores)
    python bench.py --workload criteo|multihot|wide           (default criteo = BASELINE.json configs[1] / [2])
    python bench.py --dump-outputs DIR ...                    (also store what the last timed step computed: see dump_outputs)

Workloads (config.workload), one "step" = ids + forward + sum-reduced sigmoid-CE + backward + all optimizers:
  criteo    configs[1] (N = 1) / configs[2] (N > 1): synthetic Criteo shape, 13 dense + 26 categorical (Criteo-Kaggle
            cardinalities, 33.76 M embedding rows x 32), wide = 26 hash columns + 13 bucketized + 8 crosses @ 1 M buckets, MLP
            1024-512-256 (relu, BN affine), Adagrad deep / FTRL wide, 8192 examples per GPU per step (weak scaling).
  multihot  configs[3]: one hashed multihot slot (Poisson(30) ids per example), 64-wide embedding, ResDnn 4 x 512, 12.5 M table
            rows PER GPU (100 M at N = 8, row-sharded), 8192 examples per GPU.
  wide      configs[4]: wide-only, 9 hashed fields + 32 hashed crosses into 125 M buckets PER GPU (1 B at N = 8, row-sharded),
            FTRL, 131072 examples per GPU (1 M at N = 8).
N > 1: the batch is split by example; every table larger than 16384 rows is ROW-SHARDED over the ranks and exchanged through peer
memory by the library's own kernels (wide_deep_b200/csrc/shard.cu), smaller tables are replicated and their gradients travel with
the dense gradients in one two-shot all-reduce over peer memory.  WD_DP_MODE=lists selects round 1's replicated-table path
(NCCL all-gather of (row, gradient) lists) instead.

JSON keys beyond the base contract:
  value     examples/s with the step's inputs already resident in HBM (a ring of distinct batches, so the rows a step touches are
            not the ones the previous step left in L2)
  e2e       the same metric fed from pinned host memory the way estimator.train feeds it: wd_batch_prefetch_slot refills two
            alternating slots on the upload stream (the copy of step i+1 overlaps step i, like dataset.prefetch in the reference),
            then the step, then a device -> host read of its loss — all inside the timed region
  roofline  the dominant kernel group, timed live with CUDA events on the model stream (a few profiled steps, N = 1): criteo = the
            nine MLP GEMM launches vs the measured bf16 tensor peak; multihot = embedding gather + pool vs measured HBM bandwidth;
            wide = the wide-table kernels vs HBM bandwidth.  `kernels` carries the per-phase times and the gather's HBM figure.
  dtype     arithmetic of the MLP GEMMs ("bf16x3" = fp32 operands split into bf16 hi + lo, three tensor-core products, fp32
            accumulation); `parity` re-checks the engine against the oracle in this run, `strict_engine` = the same step on tf32x3
  cpu_baseline  the optimised CPU restatement (oracle/fast.py) on the host cores, same workload, bounded sample
Before the W warm-up steps every ring slot is visited three times untimed (two eager steps + the CUDA-graph capture of that slot), so
the timed K steps replay graphs only.  WD_STEP_TRACE=1 (N = 1) / WD_SHARD_TRACE=1 (N > 1) print a stream / flag-barrier timeline of
one replayed step to stderr (profiles/r2_step_timelines.md).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

RING = 8
DENSE_EXCHANGE_ROWS = int(os.environ.get("WD_DENSE_EXCHANGE_ROWS", "16384"))
# arithmetic the MLP GEMMs run in (tables, optimizers, pooling and every reduction are fp32 in all engines)
DTYPE_OF_ENGINE = {"bf16x3": "bf16x3 (fp32 operands split into bf16 hi+lo, 3 tensor-core products, fp32 accumulate; 2^-16)",
                   "tc3x": "tf32x3 (fp32 operands split into tf32 hi+lo, 3 tensor-core products, fp32 accumulate; 2^-21)",
                   "tc1x": "tf32", "ffma": "f32", "auto": "tf32x3 (library default)"}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_burst=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, source="fallback")


def usable_cores():
    """Host cores this process may actually use: logical CPUs, limited by the affinity mask and by the container's cgroup CPU
    quota (the GPU box shows 128 logical CPUs behind a 16-CPU quota; 128 OpenMP threads on 16 CPUs' worth of time run 40x
    slower than 16).  This is the `cores` the CPU arm reports and the thread count it runs with."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        t = open("/sys/fs/cgroup/cpu.max").read().split()
        if t[0] != "max":
            n = min(n, max(1, int(float(t[0]) / float(t[1]) + 0.5)))
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, int(q / p + 0.5)))
        except Exception:
            pass
    return max(1, n)


def gemm_traffic_from_profile(engine, batch):
    """DRAM bytes of the GEMM launches of one step, from the newest committed ncu capture that matches (engine, batch):
    profiles/*_gemm_traffic.json = {"engine", "batch", "dram_bytes_per_step", "command", "source"} written by
    tools/ncu_summary.py --traffic from the `ncu --set full` raw CSV.  (None, reason) when no capture matches — never a constant."""
    import glob
    best = None
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_gemm_traffic.json"))):
        try:
            d = json.load(open(path))
        except Exception:
            continue
        if d.get("engine") == engine and int(d.get("batch", -1)) == int(batch):
            best = (float(d["dram_bytes_per_step"]), os.path.relpath(path, ROOT))
    return best if best else (None, "no committed ncu capture for engine=%s batch=%d" % (engine, batch))


class ClockSampler(object):
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe).

    A step is ~1 ms, so `nvidia-smi -lms` (>= 100 ms per sample) would miss short runs: NVML is polled in-process every 2 ms from a
    thread (same counters nvidia-smi reads); nvidia-smi is the fallback when the NVML binding is missing."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc, self.nvml, self.stop_flag = index, [], None, None, False
        self.sm, self.mx, self.reasons, self.power = [], [], set(), []

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        ids = [v for v in vis.split(",") if v.strip()]
        if ids and self.index < len(ids) and ids[self.index].strip().isdigit():
            return int(ids[self.index])
        return self.index

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
            self.mx = [float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))]
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv = self.nvml
        names = [("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                 ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap)]
        while not self.stop_flag:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for name, bit in names:
                    if mask & bit:
                        self.reasons.add(name)
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            time.sleep(0.002)

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) >= 8 and f[0] == str(self._physical_index()):
                self.rows.append(f)

    def stop(self):
        if self.nvml:
            self.stop_flag = True
            self.t.join(timeout=1.0)
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_min_mhz": min(self.sm) if self.sm else None,
                    "sm_max_mhz": max(self.mx) if self.mx else None, "reasons": sorted(self.reasons), "samples": len(self.sm),
                    "power_w": float(np.median(self.power)) if self.power else None, "source": "nvml, 2 ms poll during both timed regions"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows), "source": "nvidia-smi -lms 100"}


# ------------------------------------------------------------------------------------------------ workloads
class Workload(object):
    """One BASELINE.json configuration: conf dicts, synthetic batches (product Batch + the oracle's raw dict), bookkeeping."""

    def __init__(self, name, world, batch=None):
        from wide_deep_b200 import synthetic
        self.name, self.world = name, max(1, world)
        self.syn = synthetic
        if name == "criteo":
            self.fc, self.cross, self.model, self.emb = synthetic.criteo_conf()
            self.model_type, self.batch = "wide_deep", batch or 8192
            n_cat = sum(1 for c in self.fc.values() if c["type"] == "category")
            self.n_cat, self.n_dense = n_cat, len(self.fc) - n_cat
            self.ids_per_row = len(self.fc) + len(self.cross)
            self.keys_per_row = n_cat
            self.P = (n_cat * self.emb + self.n_dense) * 1024 + 1024 * 512 + 512 * 256 + 256
            self.desc = ("synthetic Criteo shape: 13 dense + 26 categorical (Criteo-Kaggle cardinalities, 33.76M rows), emb 32, "
                         "wide 26 hash + 13 bucketized + 8 crosses@1M, MLP 1024-512-256 relu+BN, Adagrad/FTRL; train step")
            self.l2 = "ring of %d distinct resident batches; touched rows per step ~60 MB, tables 8.6 GB >> 126 MB L2" % RING
        elif name == "multihot":
            self.rows = 12_500_000 * self.world
            self.fc, self.cross, self.model, self.emb = synthetic.multihot_conf(rows=self.rows)
            self.model_type, self.batch = "deep", batch or 8192
            self.n_cat, self.n_dense, self.ids_per_row, self.keys_per_row = 1, 0, 128, 128
            self.P = 64 * 512 + (512 + 64) * 512 + (1024 + 64) * 512 + (1536 + 64) * 512 + (2048 + 64)
            self.desc = ("one hashed multihot slot, Poisson(30) ids per example clipped to [1,128], %d rows (12.5M per GPU) x 64, mean "
                         "pooling, ResDnn 4x512 (resnet concatenations) relu+BN, Adagrad; train step" % self.rows)
            self.l2 = "ring of %d distinct resident batches; ~246K random 256-byte rows per step of a 6.4 GB table >> 126 MB L2" % RING
        elif name == "wide":
            self.rows = 125_000_000 * self.world
            self.fc, self.cross, self.model, self.emb = synthetic.wide_conf(total_cross_rows=self.rows)
            self.model_type, self.batch = "wide", batch or 131072
            self.n_cat, self.n_dense = len(self.fc), 0
            self.ids_per_row = len(self.fc) + len(self.cross)
            self.keys_per_row = len(self.fc)
            self.P = 0
            self.desc = ("wide-only: 9 hashed key fields + 32 hashed pairwise crosses into %d buckets (125M per GPU), FTRL(0.1, l1 0.5, "
                         "l2 1); train step" % self.rows)
            self.l2 = "ring of %d distinct resident batches; 4.2M random 16-byte records per step of a 2 GB table >> 126 MB L2" % RING
        else:
            raise SystemExit("unknown workload %r" % name)

    def config(self, per_gpu_batch, exchange):
        n = self.world
        return {"workload": self.desc, "global_batch": per_gpu_batch * n, "per_gpu_batch": per_gpu_batch,
                "parallelism": "dp%d" % n if n > 1 else "single",
                "tables": ("tables > %d rows row-sharded over the ranks, smaller ones replicated" % DENSE_EXCHANGE_ROWS) if (n > 1 and exchange == "sharded")
                else "replicated", "ids": "uniform", "exchange": exchange_text(exchange) if n > 1 else "none", "l2": self.l2}

    def arrays(self, B, step):
        """Host arrays of one batch: (keys uint64[nnz], offsets int32[B * F + 1] | None, dense float32[B, Nd] | None, label)."""
        if self.name == "criteo":
            keys, dense, label = self.syn.criteo_batch_arrays(self.fc, B, step=step)
            return keys.reshape(-1), None, dense, label
        if self.name == "multihot":
            keys, offs, label = self.syn.multihot_batch_arrays(B, step=step)
            return keys, offs, None, label
        keys, label = self.syn.wide_batch_arrays(self.fc, B, step=step)
        return keys.reshape(-1), None, None, label

    def raw(self, B, arrays):
        """The same batch in the oracle's format (feature -> CSR of fingerprints / float column)."""
        keys, offs, dense, label = arrays
        cats = [f for f, c in self.fc.items() if c["type"] == "category"]
        dn = [f for f, c in self.fc.items() if c["type"] == "continuous"]
        raw = {}
        if offs is None:
            k2 = keys.reshape(B, len(cats))
            for j, f in enumerate(cats):
                raw[f] = (np.arange(B + 1, dtype=np.int64), np.ascontiguousarray(k2[:, j]))
        else:
            raw[cats[0]] = (offs.astype(np.int64), keys)
        for j, f in enumerate(dn):
            raw[f] = np.ascontiguousarray(dense[:, j])
        return raw, label

    def plan(self, B, engine, rank=0, exchange="sharded"):
        from wide_deep_b200.plan import Plan
        n = self.world
        kw = dict(max_batch=B, embedding_dim_override=self.emb, gemm_engine=engine, max_keys=B * self.keys_per_row)
        if n > 1 and exchange == "sharded":
            kw.update(max_nnz=B * self.ids_per_row, dense_exchange_max_rows=DENSE_EXCHANGE_ROWS, shard_world=n, shard_rank=rank,
                      shard_slack=float(os.environ.get("WD_SHARD_SLACK", "1.5")))
        elif n > 1:
            kw.update(max_nnz=B * self.ids_per_row * n, dense_exchange_max_rows=DENSE_EXCHANGE_ROWS)
        else:
            kw.update(max_nnz=B * self.ids_per_row)
        return Plan(self.fc, self.cross, self.model, self.model_type, **kw)


def exchange_text(exchange):
    if exchange == "sharded":
        return ("peer-memory exchange by the library's kernels: ids -> owners, owner-side pooled partial sums -> requesters, owners "
                "pull gradients inside their segmented reduction + apply; dense gradients and the gradient blocks of tables <= %d rows: "
                "two-shot all-reduce over peer memory; flag barriers; no NCCL on the data path" % DENSE_EXCHANGE_ROWS)
    return ("dense all-reduce (NCCL) of MLP/wide-bias gradients + gradient blocks of tables <= %d rows; all-gather + on-device "
            "re-reduction of (row, gradient) lists for the larger tables" % DENSE_EXCHANGE_ROWS)


# ------------------------------------------------------------------------------------------- reference arm
def fast_fill(om, seed=1):
    """Parameters for the CPU arm, filled by torch's multi-threaded generators (OracleModel.init's numpy truncated normal takes
    minutes on the multi-GB tables; the timed step does not depend on the values)."""
    import torch
    from oracle import columns as C
    g = torch.Generator().manual_seed(seed)
    P = om.params = {}
    if om.use_wide:
        for c in om.wide_cols:
            P[om.wname(c)] = np.zeros(c.num_buckets, dtype=np.float32)
        P["linear/linear_model/bias_weights"] = np.zeros(1, dtype=np.float32)
    if om.use_deep:
        for c in om.deep_cols:
            if isinstance(c, C.Embedding):
                t = torch.empty((c.cat.num_buckets, c.dim), dtype=torch.float32)
                t.normal_(0.0, float(1.0 / np.sqrt(c.dim)), generator=g).clamp_(-2.0 / np.sqrt(c.dim), 2.0 / np.sqrt(c.dim))
                P[om.ename(c)] = t.numpy()
        for t_i in range(len(om.towers)):
            dims = om.layer_dims(t_i)
            for l, (i, o) in enumerate(dims):
                scope = "dnn/dnn_%d/" % (t_i + 1) + ("hiddenlayer_%d" % l if l < len(dims) - 1 else "logits")
                lim = float(np.sqrt(6.0 / (i + o)))
                P[scope + "/kernel"] = torch.empty((i, o)).uniform_(-lim, lim, generator=g).numpy()
                P[scope + "/bias"] = np.zeros(o, dtype=np.float32)
                if om.bn and l < len(dims) - 1:
                    P[scope + "/batch_normalization/gamma"] = np.ones(o, dtype=np.float32)
                    P[scope + "/batch_normalization/beta"] = np.zeros(o, dtype=np.float32)
    om.slots = {}
    for k, v in P.items():
        o = om.opt_lin if k.startswith("linear/") else om.opt_dnn
        if o["kind"] == "adagrad":
            om.slots[k] = {"acc": torch.full(v.shape, o["init_acc"], dtype=torch.float32).numpy()}
        elif o["kind"] == "ftrl":
            om.slots[k] = {"n": torch.full(v.shape, o["init_acc"], dtype=torch.float32).numpy(), "z": torch.zeros(v.shape, dtype=torch.float32).numpy()}
        else:
            om.slots[k] = {}
    return om


def oracle_examples_per_sec(wl, batch_rows, steps, warmup, threads, budget_s=None):
    """Time the OPTIMISED CPU restatement (oracle/fast.py: torch-CPU matmuls + embedding_bag + sparse row updates, C hashing;
    checked against oracle/model.py by tests/test_oracle_fast.py) on the same workload with every host thread; returns
    (examples/s, seconds per step, steps timed).  torch.distributed.run exports OMP_NUM_THREADS=1: overridden explicitly."""
    os.environ["OMP_NUM_THREADS"] = str(threads)
    os.environ["MKL_NUM_THREADS"] = str(threads)
    import torch
    torch.set_num_threads(threads)
    from oracle import fast as OF, model as OM
    om = OM.OracleModel(wl.fc, wl.cross, wl.model, wl.model_type, embedding_dim_override=wl.emb, acc=np.float32)
    fm = OF.FastCpuModel(fast_fill(om), threads=threads)
    times = []
    for s in range(warmup + steps):
        raw, label = wl.raw(batch_rows, wl.arrays(batch_rows, s))
        t0 = time.perf_counter()
        fm.train_step(raw, label)
        dt = time.perf_counter() - t0
        if s >= warmup:
            times.append(dt)
            if budget_s is not None and sum(times) > budget_s:
                break
    sec = float(np.mean(times))
    return batch_rows / sec, sec, len(times)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = usable_cores()
    wl = Workload(args.workload, args.gpus, args.batch)
    # the same step as the GPU arm: same tables, same GLOBAL batch (N x per-GPU batch: the CPU arm is the whole box's host cores,
    # whatever N is), a bounded number of steps
    rows = wl.batch * max(1, args.gpus)
    warm = max(1, min(args.warmup, 2))
    v, sec, steps = oracle_examples_per_sec(wl, rows, max(1, args.steps), warm, threads, budget_s=90.0)   # K steps or 90 s of CPU work
    sample = "%d steps of %d examples (same tables/config as the GPU arm at N=%d), %d threads" % (steps, rows, args.gpus, threads)
    exchange = "sharded" if os.environ.get("WD_DP_MODE", "sharded") != "lists" else "lists"
    out = {"impl": "reference", "metric": "CTR examples/sec (train step)", "value": v, "unit": "examples/s", "n_gpus": args.gpus,
           "steps": steps, "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": wl.config(wl.batch, exchange),
           "cpu_baseline": {"value": v, "unit": "examples/s", "cores": threads, "kind": "port", "sample": sample,
                            "note": "optimised CPU restatement of the reference step (oracle/fast.py: torch-CPU sgemm + embedding_bag + "
                                    "sparse row updates, C hashing); TensorFlow 1.x is not installable here"},
           "e2e": {"value": v, "unit": "examples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def parity_check(engine, rows=2048):
    """Checker leg (oracle = test infrastructure): max relative logit error of `engine` against the CPU oracle on the benchmark
    model with every table scaled by 1e-3 (same columns, same 845-1024-512-256 towers, same kernels), parameters copied from the
    oracle.  The bar is BASELINE.json's: |gpu - oracle| <= 1e-4 * max(|oracle|, 1).  (tests/test_gpu_bench_engine.py holds the
    same engine to the same bar under pytest, plus a 50-step drift bound.)"""
    from oracle import model as OM
    from tests.helpers import copy_params_to_product
    from wide_deep_b200 import synthetic
    from wide_deep_b200.model import Batch, WideDeepModel
    from wide_deep_b200.plan import Plan
    fc, cross, model, emb = synthetic.criteo_conf(scale=1e-3)
    n_cat = sum(1 for c in fc.values() if c["type"] == "category")
    om = OM.OracleModel(fc, cross, model, "wide_deep", embedding_dim_override=emb).init(7)
    plan = Plan(fc, cross, model, "wide_deep", max_batch=rows, embedding_dim_override=emb, gemm_engine=engine,
                max_nnz=rows * (len(fc) + len(cross)), max_keys=rows * n_cat)
    pm = WideDeepModel(plan)
    copy_params_to_product(om, pm)
    keys, dense, label = synthetic.criteo_batch_arrays(fc, rows, step=123)
    cats = [f for f, c in fc.items() if c["type"] == "category"]
    dn = [f for f, c in fc.items() if c["type"] == "continuous"]
    raw = {f: (np.arange(rows + 1, dtype=np.int64), np.ascontiguousarray(keys[:, j])) for j, f in enumerate(cats)}
    for j, f in enumerate(dn):
        raw[f] = np.ascontiguousarray(dense[:, j])
    b = Batch(rows, keys.reshape(-1), None, dense, label)
    logits, _ = pm.forward(b)
    _, cache = om.forward(raw)
    ref = cache["logits"]
    err = np.abs(logits - ref) / np.maximum(np.abs(ref), 1.0)
    loss = pm.train_step(b)
    ref_loss, _ = om.train_step(raw, label)
    del pm
    return {"engine": engine, "max_rel_logit_err": float(err.max()), "rms_rel_logit_err": float(np.sqrt((err ** 2).mean())),
            "rel_loss_err": float(abs(loss - ref_loss) / max(abs(ref_loss), 1.0)), "bar": 1e-4, "pass": bool(err.max() <= 1e-4),
            "sample": "%d examples, benchmark model with tables scaled 1e-3, parameters copied from the oracle" % rows}


DUMP_BUDGET_BYTES = 56 << 20            # array data of one --dump-outputs directory; with the .npy headers it stays under 64 MB


def dump_outputs(model, loss, out_dir):
    """--dump-outputs: what the timed train step leaves its caller after its last step, as float32 .npy files: `loss.npy` (the
    step's sum-reduced loss) and every parameter and optimizer slot under its checkpoint key with '/' -> '.' (`<name>.npy`,
    `<name>.slotN.npy`).  MLP and bias tensors are stored whole; the budget left is shared out over the embedding tables and
    wide columns, smallest first, and one larger than its share is stored as a fixed sample of its rows, drawn by a generator
    seeded with the file name, so runs with the same arguments store the same rows.  N > 1: rank 0's replica and row shards."""
    import zlib
    from wide_deep_b200.plan import T_EMB_TABLE, T_WIDE_COL
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), np.array([loss], dtype=np.float32))
    arrays = [(name, s) for name in model.tensor_names() for s in range(model.n_slots(name) + 1)]
    share = {a: int(np.prod(model.plan.local_shape(a[0]))) for a in arrays}
    tables = sorted((a for a in arrays if model.plan.tensor_names[a[0]][0] in (T_EMB_TABLE, T_WIDE_COL)), key=share.get)
    left = DUMP_BUDGET_BYTES // 4 - 1 - sum(n for a, n in share.items() if a not in tables)
    for i, a in enumerate(tables):
        share[a] = min(share[a], left // (len(tables) - i))
        left -= share[a]
    for name, s in arrays:
        key = name.replace("/", ".") + (".slot%d" % s if s else "")
        x = model.get_tensor(name, slot=s)
        if x.size > share[(name, s)]:
            rows = np.random.default_rng(zlib.crc32(key.encode())).choice(x.shape[0], share[(name, s)] // (x.size // x.shape[0]), replace=False)
            x = x[np.sort(rows)]
        np.save(os.path.join(out_dir, key + ".npy"), x)


# ------------------------------------------------------------------------------------------------ our arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--workload", default=os.environ.get("WD_WORKLOAD", "criteo"), choices=["criteo", "multihot", "wide"])
    ap.add_argument("--batch", type=int, default=None, help="examples per GPU per step (default: the workload's)")
    ap.add_argument("--engine", default=os.environ.get("WD_GEMM_ENGINE", "bf16x3"),
                    help="MLP GEMM engine: bf16x3 (tcgen05 kind::f16 on bf16 hi/lo copies, 2^-16 products; re-checked against the "
                         "oracle in this run) | tc3x (tcgen05 kind::tf32 3-pass, 2^-21, the library default) | ffma (fp32 CUDA cores)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the loss, parameters and optimizer slots of the last one to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs stores what the GPU step computed; the reference arm has nothing to store")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    torch.cuda.set_device(local)
    exchange = "lists" if os.environ.get("WD_DP_MODE", "sharded") == "lists" else "sharded"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from wide_deep_b200.model import Batch, WideDeepModel
    wl = Workload(args.workload, world, args.batch)
    B = wl.batch
    plan = wl.plan(B, args.engine, rank, exchange)
    model = WideDeepModel(plan, device=local)
    model.init(seed=0x5EED0005)          # identical replicas on every rank (shards of sharded tables draw their own stream)
    trainer = None
    if world > 1 and exchange == "sharded":
        from wide_deep_b200.sharded import ShardedTrainer
        trainer = ShardedTrainer(model)
    elif world > 1:
        from wide_deep_b200.parallel import DataParallelTrainer
        trainer = DataParallelTrainer(model, fixed_rows=plan.exchange_rows(B))

    # distinct batches per (rank, ring slot) in pinned host memory
    host = []
    for s in range(RING):
        keys, offs, dense, label = wl.arrays(B, rank * 1000 + s)
        pins = [torch.from_numpy(keys.view(np.int64).copy()).pin_memory(), torch.from_numpy(label.copy()).pin_memory()]
        po = torch.from_numpy(offs.copy()).pin_memory() if offs is not None else None
        pd = torch.from_numpy(dense.copy()).pin_memory() if dense is not None else None
        b = Batch(B, pins[0].numpy().view(np.uint64), None if po is None else po.numpy(), None if pd is None else pd.numpy(), pins[1].numpy())
        host.append((b, (pins, po, pd)))
    for s in range(RING):
        model.upload_slot(s, host[s][0])
    model.sync()
    stream = torch.cuda.ExternalStream(model.stream(), device=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(steps):
            fn(i)
        e1.record(stream)
        model.sync()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def step_resident(i):
        if trainer:
            trainer.step_slot(i % RING, want_loss=False)
        else:
            model.train_step_slot(i % RING, want_loss=False)

    # end to end: every step's inputs come from pinned host memory and its loss goes back to the host.  Two extra slots are
    # refilled alternately with wd_batch_prefetch_slot — the copy of step i+1 runs on the upload stream while step i computes, as
    # tf.data's prefetch does in the reference's input_fn — and each step ends with a device->host read of its loss.
    E2E0 = RING

    def step_e2e(i):
        model.prefetch_slot(E2E0 + (i + 1) % 2, host[(i + 1) % RING][0])
        if trainer and exchange == "sharded":
            return trainer.step_slot(E2E0 + i % 2, want_loss=True)
        if trainer:
            trainer.step_slot(E2E0 + i % 2, want_loss=False)
            return model.last_loss()
        return model.train_step_slot(E2E0 + i % 2, want_loss=True)

    # untimed: every ring slot runs its two eager steps and its graph capture (3 visits per slot) BEFORE the W warm-up steps, so the
    # timed region replays graphs only (a capture inside the timed region costs a host-side stall that shows up as rank skew)
    for i in range(3 * RING):
        step_resident(i)
    model.sync()
    launches0 = model.launch_count()
    for i in range(args.warmup):
        step_resident(i)
    model.sync()
    per_step_launches = (model.launch_count() - launches0) // max(args.warmup, 1)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    ms = timed(step_resident, args.steps)
    if args.dump_outputs:                                # before the e2e steps train the model further
        if rank == 0:
            dump_outputs(model, model.last_loss(), args.dump_outputs)
        barrier()
    model.prefetch_slot(E2E0, host[0][0])
    for i in range(8):                                   # both e2e slots past their eager steps (graphs captured)
        step_e2e(i)
    ms_e2e = timed(lambda i: step_e2e(i + 8), args.steps)
    clk = clocks.stop() if rank == 0 else None

    if trainer and exchange == "lists" and os.environ.get("WD_DP_PROFILE"):
        for i in range(3):
            prof = trainer.profile_step(i % RING)
        if rank == 0:
            sys.stderr.write("dp phases (ms from step start): %s\n" % json.dumps({k: round(v, 3) for k, v in prof.items()}))

    if trainer and exchange == "sharded" and os.environ.get("WD_SHARD_TRACE"):
        # flag-barrier timeline of one replayed step per rank (globaltimer, us from that rank's step start): enter / leave of the
        # barriers A (ids delivered), B (pooled sums delivered), Cw / Ce (dlogit / dX0 exist; side streams), G (gradient arenas
        # final), R (slices reduced), END; "work" = step start -> last kernel before END
        import ctypes
        for i in range(3):
            step_resident(i)
        tr = np.zeros(16, dtype=np.uint64)
        model._lib.wd_debug_shard_trace(model._h, tr.ctypes.data_as(ctypes.c_void_p))
        t0 = int(tr[14])
        names = ["A", "B", "Cw", "Ce", "G", "R", "END"]
        mine = {n: [round((int(tr[2 * k]) - t0) / 1e3, 1), round((int(tr[2 * k + 1]) - t0) / 1e3, 1)] for k, n in enumerate(names)}
        mine["work_end"] = round((int(tr[15]) - t0) / 1e3, 1)
        allr = [None] * world
        dist.all_gather_object(allr, mine)
        if rank == 0:
            sys.stderr.write("shard barrier timeline (us, [enter, leave]): %s\n" % json.dumps(allr))

    if not trainer and os.environ.get("WD_STEP_TRACE"):
        # stream timeline of one replayed step (globaltimer stamps inside the step's CUDA graph; us from the step's start)
        import ctypes
        for i in range(3):
            step_resident(i)
        tr = np.zeros(16, dtype=np.uint64)
        model._lib.wd_debug_step_trace(model._h, tr.ctypes.data_as(ctypes.c_void_p))
        names = ["start", "ids", "gather", "head", "towers_bwd", "main_end", "group_emb_end", "group_wide_end", "reduce_emb_beg",
                 "reduce_emb_end", "reduce_wide_beg", "reduce_wide_end", "apply_emb_end", "apply_wide_end"]
        sys.stderr.write("step timeline (us): %s\n" % json.dumps({n: round((int(tr[k]) - int(tr[0])) / 1e3, 1) for k, n in enumerate(names)}))

    # per-kernel timings (CUDA events between stages on the model stream), a few profiled steps
    phases = {}
    if not trainer:
        model.set_profile(True)
        nprof = 5
        for i in range(nprof):
            model.train_step_slot(i % RING, want_loss=True)
            for k, v in model.last_timings().items():
                phases[k] = phases.get(k, 0.0) + v / nprof
        model.set_profile(False)

    if rank == 0:
        peaks = load_peaks()
        gb = B * world
        value = gb * args.steps / (ms / 1e3)
        e2e = gb * args.steps / (ms_e2e / 1e3)
        has_mlp = wl.model_type != "wide"
        out = {"metric": "CTR examples/sec (train step)", "value": value, "unit": "examples/s", "n_gpus": world,
               "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
               "scaling": "weak", "vs_baseline": None, "dtype": DTYPE_OF_ENGINE.get(args.engine, "f32") if has_mlp else "f32 (no MLP: integer ids + fp32 FTRL)",
               "data": "synthetic", "config": wl.config(B, exchange),
               "e2e": {"value": e2e, "unit": "examples/s", "ms_per_step": ms_e2e / args.steps,
                       "h2d_bytes_per_step": host[0][0].h2d_bytes(), "d2h_bytes_per_step": 8,
                       "input": "pinned host batches, wd_batch_prefetch_slot into two alternating slots (copy of step i+1 overlaps step i), loss read every step"},
               "gpu_launches": int(per_step_launches * args.steps), "launches_per_step": int(per_step_launches),
               "clocks": clk, "gemm_engine": args.engine if has_mlp else None}
        nnz_avg = host[0][0].keys.shape[0] / float(B) if wl.name == "multihot" else float(wl.n_cat)
        if phases and wl.name == "criteo":
            gemm_ms = sum(v for k, v in phases.items() if k.startswith("gemm_"))
            flops = 6.0 * B * wl.P                                # 2BP forward + 4BP backward (SURVEY 8d)
            ach = flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
            traffic, traffic_src = gemm_traffic_from_profile(args.engine, B)
            out["roofline"] = {"kernel": "mlp gemm (fwd+dgrad+wgrad)", "bound": "tensor", "achieved": ach, "peak": peaks["bf16_sustained"],
                               "unit": "TFLOP/s", "frac": ach / peaks["bf16_sustained"],
                               # the GEMMs run inside a long step, back to back with the rest of it: the SUSTAINED peak applies; the
                               # fraction against the burst figure (a kernel timed alone) is given beside it
                               "peak_burst": peaks["bf16_burst"], "frac_burst": ach / peaks["bf16_burst"], "peak_applies": "sustained",
                               # dram__bytes_read.sum + dram__bytes_write.sum summed over the GEMM launches of one step, read from the
                               # committed ncu capture of this engine / batch size (profiles/*_gemm_traffic.json); null when there is none
                               "traffic": traffic, "traffic_unit": "bytes per step (all GEMM launches of one step)", "traffic_source": traffic_src,
                               "peak_source": peaks["source"] + " dense bf16.  achieved = algorithmic fp32 FLOPs (6*B*P) / GEMM time; "
                                              "both split engines issue 3 tensor-core products per algorithmic one, so the fp32-"
                                              "equivalent ceiling is 1/3 of the bf16 peak for bf16x3 and 1/6 for tc3x",
                               "tensor_pipe_frac": 3.0 * ach / peaks["bf16_sustained"] * (2.0 if args.engine == "tc3x" else 1.0),
                               "share_of_step": gemm_ms / phases.get("total", 1.0)}
        if phases and has_mlp:
            # SURVEY 8(d) K3: ids + offsets + rows + pooled output
            gather_bytes = B * (nnz_avg * (4 * wl.emb + 4) + 4 * wl.n_cat + 4 * wl.n_cat * wl.emb)
            g_ms = phases.get("emb_fwd", 0.0)
            g_ach = gather_bytes / (g_ms * 1e-3) / 1e9 if g_ms > 0 else 0.0
            gk = {"bound": "hbm", "achieved": g_ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": g_ach / peaks["hbm_gbs"],
                  "algorithmic_bytes": gather_bytes, "ms": g_ms}
            out["kernels"] = {"emb_gather_pool_fwd": gk, "phases_ms": {k: round(v, 4) for k, v in phases.items()}}
            if wl.name == "multihot":
                # the table-bound kernels of this workload: gather + pool (K3) and the backward gradient sums + Adagrad (K8)
                u = min(nnz_avg * B, wl.rows)
                bwd_bytes = 4 * B * wl.emb + 4 * nnz_avg * B + 16 * u * wl.emb
                b_ms = phases.get("emb_grad_sum", 0.0) + phases.get("sparse_apply", 0.0)
                out["roofline"] = dict(gk, kernel="emb gather + mean pool (forward)", traffic=None, peak_source=peaks["source"] + " HBM copy bandwidth",
                                       share_of_step=g_ms / phases.get("total", 1.0))
                out["kernels"]["emb_grad_sum_apply_bwd"] = {"bound": "hbm", "achieved": bwd_bytes / (b_ms * 1e-3) / 1e9 if b_ms > 0 else 0.0,
                                                            "peak": peaks["hbm_gbs"], "unit": "GB/s", "algorithmic_bytes": bwd_bytes, "ms": b_ms}
        if phases and wl.name == "wide":
            nnz = float(wl.ids_per_row) * B
            w_bytes = nnz * 8 + 4 * B + 4 * nnz + 4 * B + 24 * nnz          # SURVEY 8(d) K4 + K9 (U_w ~ nnz: uniform ids)
            w_ms = phases.get("wide_fwd", 0.0) + phases.get("wide_grad_sum", 0.0) + phases.get("sparse_apply", 0.0)
            ach = w_bytes / (w_ms * 1e-3) / 1e9 if w_ms > 0 else 0.0
            out["roofline"] = {"kernel": "wide logit gather + gradient sums + FTRL (excludes the id hashing and the sort)", "bound": "hbm",
                               "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"], "traffic": None,
                               "algorithmic_bytes": w_bytes, "ms": w_ms, "peak_source": peaks["source"] + " HBM copy bandwidth",
                               "share_of_step": w_ms / phases.get("total", 1.0)}
            out["kernels"] = {"phases_ms": {k: round(v, 4) for k, v in phases.items()}}
        if not args.no_cpu_baseline and world == 1 and args.engine != "tc3x" and wl.name == "criteo":
            # the same step on the fp32-faithful engine (3xTF32, the library default), for reference next to the headline
            m2 = WideDeepModel(wl.plan(B, "tc3x"), device=local)
            m2.init(seed=0x5EED0005)
            for s_ in range(RING):
                m2.upload_slot(s_, host[s_][0])
            st2 = torch.cuda.ExternalStream(m2.stream(), device=torch.device("cuda", local))
            for i in range(6):
                m2.train_step_slot(i % RING, want_loss=False)
            m2.sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st2)
            for i in range(40):
                m2.train_step_slot(i % RING, want_loss=False)
            e1.record(st2)
            m2.sync()
            out["strict_engine"] = {"gemm_engine": "tc3x", "value": B * 40 / (e0.elapsed_time(e1) / 1e3), "unit": "examples/s",
                                    "ms_per_step": e0.elapsed_time(e1) / 40, "steps": 40}
            del m2
        if not args.no_cpu_baseline and world == 1:
            if wl.name == "criteo":
                out["parity"] = parity_check(args.engine)
            del model
            threads = usable_cores()
            v, sec, nst = oracle_examples_per_sec(wl, B, 10, 2, threads, budget_s=20.0)
            out["cpu_baseline"] = {"value": v, "unit": "examples/s", "cores": threads, "kind": "port",
                                   "sample": "%d steps of %d examples, same tables/config (oracle/fast.py: torch-CPU + C hashing, fp32)" % (nst, B)}
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    sys.dont_write_bytecode = True                       # the benchmark leaves the tree as it found it
    main()
