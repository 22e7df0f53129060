#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (BASELINE.json metric: CTR forward+backward samples/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--ids uniform|zipf]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch.  Workloads (BASELINE.json `configs`):
  deepfm_cfg5          configs[4] on ONE GPU (default at N=1): DeepFM, 40 fields, embed_dim 32, batch 65536, 100 M-row
                       vocabulary (12.8 GB fp32, fits one GPU): fused lookup+FM2 forward, then its backward.
  deepfm_cfg5_sharded  configs[4] as named: the vocabulary ROW-SHARDED over the N GPUs (default at N>1; 32 GB shard per rank,
                       B = 65536 per rank): rows pulled / gradient rows pushed over NVLink inside the kernels.
  dcn_cfg2 | xdeepfm_cfg3 | din_cfg4   configs[1..3]: lookup + cross stack / CIN / DIN attention, forward+backward.
Prints ONE JSON line (rank 0).  Keys beyond the base contract:
  value        device-resident throughput (inputs already in HBM), CUDA-event timed, max over ranks
  e2e          same metric through the public autograd API with HOST (pinned) ids/labels: H2D copies, loss, D2H of the loss
               inside the timed region
  roofline     achieved algorithmic GB/s (or TFLOP/s) of the dominant kernel vs MEASURED_PEAKS.json
  sustained    the same step looped for >= 2 s with the clock sampler running
  configs      (default line only) samples/s + roofline fraction of configs 2, 3, 4 from short runs in the same process
  cpu_baseline the restated reference (oracle port, torch CPU op-for-op) timed on this box's host cores
--impl reference times that CPU restatement as the reference arm (TF 1.14 itself cannot be installed).
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import sys
import threading
import time

# NCCL writes its banner / NCCL_DEBUG output to stdout by default; stdout of this script carries exactly one JSON line
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":   # level VERSION (env or /etc/nccl.conf) ignores NCCL_DEBUG_FILE;
    os.environ["NCCL_DEBUG"] = "WARN"                                # WARN prints the same banner, through the debug file

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

DEEPFM = {
    "deepfm_cfg5": dict(model="DeepFM lookup+FM2", B=65536, F=40, D=32, rows_per_field=2_500_000, id_batches=8),
    # 6.25 M rows/field PER RANK (32 GB shard each; 2 G rows = 256 GB at 8 GPUs): the vocabulary outgrows one GPU
    "deepfm_cfg5_sharded": dict(model="DeepFM lookup+FM2, row-sharded tables", B=65536, F=40, D=32,
                                rows_per_field_per_rank=6_250_000, rows_per_field=2_500_000, id_batches=8, sharded=True),
    "deepfm_small": dict(model="DeepFM lookup+FM2", B=8192, F=40, D=32, rows_per_field=100_000, id_batches=4),
    "deepfm_small_sharded": dict(model="DeepFM lookup+FM2, row-sharded tables", B=8192, F=40, D=32,
                                 rows_per_field_per_rank=100_000, rows_per_field=100_000, id_batches=4, sharded=True),
}
LAYER_WORKLOADS = ("dcn_cfg2", "xdeepfm_cfg3", "din_cfg4")


def deepfm_config(workload, model, B, world, F, D, rows, ids_desc, NB):
    """`config` of a replicated-table DeepFM line.  ONE builder for the GPU arm and for `--impl reference`: when the CPU arm runs
    the same B / table / id batches its config dict is equal to the GPU arm's, key for key (it says what ran when it could not)."""
    return {"workload": workload, "model": model, "global_batch": B * world, "B_per_gpu": B, "F": F, "D": D,
            "rows_per_field": rows, "vocab_rows_total": rows * F, "ids": ids_desc,
            "parallelism": ("replicated tables (12.8 GB fits one device), data-parallel ranks, no exchange" if world > 1
                            else "single device, no exchange"),
            "l2": f"inputs larger than the last-level cache: {NB} rotating id batches over a {rows * F * D * 4 / 1e9:.1f} GB table; "
                  f"tile/d_tile/row_grads are {B * F * D * 4 / 1e6:.0f} MB each"}
NVLINK_PEAK_GBS = 770.0       # B200_PROFILING.md: measured peer copy, per direction per GPU


def measured_peaks():
    d = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            d.update(hbm_gbs=float(j["hbm_gbs"]), bf16_tflops=float(j["bf16_tflops"]),
                     bf16_tflops_sustained=float(j.get("bf16_tflops_sustained", j["bf16_tflops"])),
                     source="measured (MEASURED_PEAKS.json)")
        except Exception:
            pass
    return d


def bytes_per_sample(F, D):
    """Algorithmic bytes (SURVEY 8d): idx = 8 B, elt = 4 B."""
    fwd = F * (8 + 2 * D * 4) + 4          # read id, read row, write tile ; write logit
    bwd = F * (3 * D * 4) + 4              # read d_tile, read tile, write row-grads ; read d_logit
    return fwd, bwd


def kernel_source_hash():
    h = hashlib.sha256()
    for f in ("embed_fm2.cu", "ctr_common.cuh"):
        h.update(open(os.path.join(ROOT, "recalgorithm_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:16]


def measured_traffic(workload, ids_kind):
    """DRAM bytes per launch of the gather from the committed ncu capture -- only while the kernel source still hashes to
    what was profiled (ncu cannot run inside the bench); otherwise null + the reason."""
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        t = json.load(open(tp)).get(workload, {})
    except Exception:
        return None, "profiles/traffic.json missing"
    if ids_kind != "uniform":
        return None, "ncu capture was taken with uniform ids"
    if t.get("kernel_source_sha256_16") != kernel_source_hash():
        return None, f"stale: kernel source changed since {t.get('source', 'the capture')} (hash {t.get('kernel_source_sha256_16')} != {kernel_source_hash()})"
    return t.get("embed_fm2_fwd_dram_bytes_per_launch"), t.get("source")


class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU DURING the timed region (NVML, 10 ms period)."""

    def __init__(self, index: int):
        self.index, self.samples, self.reasons = index, [], set()
        self.max_mhz, self._stop, self._thr = None, threading.Event(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake_slowdown": 0x80, "sync_boost": 0x10}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.01)

    def start(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        return self

    def stop(self):
        self._stop.set()
        if self._thr is not None:
            self._thr.join()
        return {"sm_mhz": (statistics.median(self.samples) if self.samples else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


class Dist:
    def __init__(self):
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world > 1:
            import torch.distributed as dist
            self.dist = dist
            torch.cuda.set_device(self.local)
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        else:
            self.dist = None
            torch.cuda.set_device(0)
        self.dev = torch.device("cuda", self.local if self.world > 1 else 0)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max(self, x: float) -> float:
        if self.world == 1:
            return x
        t = torch.tensor([x], device=self.dev, dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def gather(self, x: float):
        if self.world == 1:
            return [x]
        t = torch.tensor([x], device=self.dev, dtype=torch.float64)
        out = [torch.zeros_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [float(o.item()) for o in out]


def timed_steps(dd: Dist, step, steps, n_marks=0):
    """EXACTLY `steps` steps bracketed by barrier + synchronize; returns (total ms = max over ranks, mean ms per mark)."""
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(n_marks + 1)] for _ in range(steps)] if n_marks else None
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dd.barrier()
    t0.record()
    for i in range(steps):
        step(i, evs[i] if evs else None)
    t1.record()
    dd.barrier()
    ms = dd.max(t0.elapsed_time(t1))
    marks = [statistics.mean(e[j].elapsed_time(e[j + 1]) for e in evs) for j in range(n_marks)] if evs else []
    return ms, marks


DUMP_BYTES = 60_000_000


def dump_outputs(path, whole, per_sample):
    """--dump-outputs: writes `whole`'s tensors in full and, of `per_sample`'s (batch-major) tensors, the same fixed, seeded
    sample of batch rows (ascending, as many as keep the total within DUMP_BYTES), as float32 `path/<name>.npy`.  The bench
    inputs are seeded, so two builds run with the same arguments can be compared file by file."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    arrays = {k: t.detach().float().cpu().numpy() for k, t in whole.items()}
    B = next(iter(per_sample.values())).shape[0]
    row_bytes = sum(t[0].numel() * 4 for t in per_sample.values())
    n = min(B, (DUMP_BYTES - sum(a.nbytes for a in arrays.values())) // row_bytes)
    rows = torch.randperm(B, generator=torch.Generator().manual_seed(0))[:n].sort().values
    for k, t in per_sample.items():
        arrays[k] = t.detach().index_select(0, rows.to(t.device)).float().cpu().numpy()
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def sustained_run(dd: Dist, step, ms_per_step, units_per_step, seconds=2.0):
    """The same step looped for >= `seconds` with the clock sampler running (the headline region is only milliseconds)."""
    n = max(50, int(seconds * 1e3 / max(ms_per_step, 1e-3)) + 1)
    sampler = ClockSampler(dd.local if dd.world > 1 else 0).start()
    ms, _ = timed_steps(dd, step, n)
    clocks = sampler.stop()
    return {"seconds": ms * 1e-3, "steps": n, "ms_per_step": ms / n, "value": dd.world * units_per_step * n / (ms * 1e-3), "clocks": clocks}


# ----------------------------------------------------------------------------------------------------
# CPU restatement of the reference model_fn slice (oracle port): used by cpu_baseline and --impl reference
# ----------------------------------------------------------------------------------------------------
def usable_cores():
    """Cores this process may really use: affinity mask capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period))))
    except Exception:
        pass
    return n


def host_table_rows(cfg):
    """Rows per field for the CPU arm: the GPU arm's full table when host RAM allows, else halved until it fits (the config
    keys of the CPU line state what actually ran)."""
    want = cfg["rows_per_field"]
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = 32 << 30
    per_row = cfg["F"] * cfg["D"] * 4 * 1.3            # table + sparse-gradient headroom
    while want * per_row > 0.6 * avail and want > 10_000:
        want //= 2
    return want


_cpu_model_cache = {}


def cpu_reference_run(cfg, steps, warmup, budget_s=90.0):
    """Forward+backward of the restated reference on the host cores at the GPU arm's B and table size (RAM permitting);
    returns (samples/s, ms/step, info).  The per-step batch is cut only if `steps` full batches would exceed `budget_s`."""
    from oracle import torch_cpu_model as M            # the only oracle use in bench.py (the measured baseline)
    cores = usable_cores()
    rows = host_table_rows(cfg)
    key = (cfg["F"], cfg["D"], rows)
    if key not in _cpu_model_cache:
        _cpu_model_cache[key] = M.DeepFMLookupFM2CPU(cfg["F"], cfg["D"], rows, seed=1234)
    model = _cpu_model_cache[key]
    B = cfg["B"]
    g = torch.Generator().manual_seed(1234)
    NB = cfg["id_batches"]                    # as many rotating id batches as the GPU arm
    batches = [(torch.randint(0, rows, (B, cfg["F"]), generator=g), (torch.rand((B, 1), generator=g) < 0.0356).float())
               for _ in range(NB)]
    probe = [(i[:8192].contiguous(), l[:8192].contiguous()) for i, l in batches[:2]]
    best = None                               # give the CPU arm its best thread count: many-core hosts oversubscribe on small ops
    for nt in sorted({min(cores, c) for c in (4, 8, 16, 32, 64, cores)}):
        torch.set_num_threads(nt)
        model.step(*probe[0])
        t0 = time.perf_counter()
        model.step(*probe[1])
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, nt)
    threads = best[1]
    torch.set_num_threads(threads)
    est = best[0] * B / 8192
    sample_B = B
    if est * (steps + warmup) > budget_s:
        sample_B = max(4096, int(B * budget_s / (est * (steps + warmup))) // 4096 * 4096)
        batches = [(i[:sample_B].contiguous(), l[:sample_B].contiguous()) for i, l in batches]
    for i in range(warmup):
        model.step(*batches[i % NB])
    t0 = time.perf_counter()
    for i in range(steps):
        model.step(*batches[i % NB])
    dt = time.perf_counter() - t0
    info = {"cores": threads, "host_cores_usable": cores, "kind": "port", "B": sample_B, "rows_per_field": rows,
            "same_config_as_gpu_arm": bool(sample_B == B and rows == cfg["rows_per_field"]),
            "sample": f"B={sample_B} per step x {steps} steps, F={cfg['F']}, D={cfg['D']}, {rows} rows/field "
                      f"({cfg['F'] * rows * cfg['D'] * 4 / 1e9:.1f} GB of tables), uniform ids; fwd+bwd of per-field gathers + "
                      "add_n/square FM2 + dense(1) deep head + sigmoid-CE (torch CPU op-for-op restatement of "
                      "DeepFM/deepfm.py:178-235; TF 1.14 not installable)"}
    return sample_B * steps / dt, dt / steps * 1e3, info


CPU_LAYER_SAMPLE_B = {"xdeepfm_cfg3": 1024}      # the reference materialises a (B, D, hk*m) outer product: 2 GB at B = 8192


def cpu_layer_baseline(name, budget_s=5.0, steps=None, warmup=1):
    """Forward+backward of the reference-restated lookup + interaction chain of config `name` (oracle/torch_cpu_layers.py: the
    reference's ops as written, e.g. the materialised CIN outer product) on the host cores; a bounded sample of the workload
    (about `budget_s` seconds of timed steps, or exactly `steps`).  Returns the cpu_baseline object of that config."""
    from oracle import torch_cpu_layers as C         # oracle use #2 of bench.py: again only as the measured baseline
    cls, B_full = C.BUILDERS[name]
    B = CPU_LAYER_SAMPLE_B.get(name, B_full)
    cores = usable_cores()
    model = cls()
    gen = torch.Generator().manual_seed(1234)
    batches = [model.make_batch(B, gen) for _ in range(2)]
    best = None
    for nt in sorted({min(cores, c) for c in (16, 64)}):             # many-core hosts oversubscribe on these small ops
        torch.set_num_threads(nt)
        model.step(*batches[0])
        t0 = time.perf_counter()
        model.step(*batches[1])
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, nt)
    torch.set_num_threads(best[1])
    for i in range(max(0, warmup - 1)):
        model.step(*batches[i % 2])
    n = int(steps) if steps else max(2, min(50, int(budget_s / max(best[0], 1e-4))))
    t0 = time.perf_counter()
    for i in range(n):
        model.step(*batches[i % 2])
    dt = time.perf_counter() - t0
    return {"value": B * n / dt, "unit": "samples/s", "ms_per_step": dt / n * 1e3, "cores": best[1], "host_cores_usable": cores,
            "kind": "port", "B": B, "same_config_as_gpu_arm": bool(B == B_full),
            "sample": f"B={B} per step x {n} steps (GPU arm: B={B_full}); per-field gathers + the interaction layers as the reference "
                      f"writes them, forward + backward (torch CPU op-for-op restatement, oracle/torch_cpu_layers.py; TF 1.14 not installable)"}


def safe_cpu_layer_baseline(name, budget_s):
    """The CPU baseline must never cost the GPU line: any failure is reported in place of the number."""
    try:
        return cpu_layer_baseline(name, budget_s)
    except Exception as ex:                                            # noqa: BLE001
        return {"unavailable": f"{type(ex).__name__}: {str(ex)[:160]}"}


LAYER_MODELS = {"dcn_cfg2": "DCN lookup + 3 cross layers", "xdeepfm_cfg3": "xDeepFM lookup + CIN [128,128]",
                "din_cfg4": "DIN lookup + attention"}


def run_reference_arm_layers(args):
    """`--impl reference --workload dcn_cfg2|xdeepfm_cfg3|din_cfg4`: the CPU restatement of that chain as the reference arm."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cb = cpu_layer_baseline(args.workload, steps=args.steps, warmup=args.warmup)
    line = {"metric": "ctr_fwd_bwd_samples_per_sec", "value": cb["value"], "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": args.workload, "model": LAYER_MODELS[args.workload], "B": cb["B"], "rows_per_field": 1_000_000,
                       "ids": "uniform int64"},
            "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_reference_arm(args, cfg):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    sps, ms, info = cpu_reference_run(cfg, args.steps, max(args.warmup, 1))
    line = {"metric": "ctr_fwd_bwd_samples_per_sec", "value": sps, "unit": "samples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            # the GPU arm's N = 1 config, key for key (B / rows differ only if the host could not hold or finish them); launched
            # with N > 1 the CPU arm still runs this single-process configuration, and says so
            "config": deepfm_config(args.workload, cfg["model"], info["B"], 1, cfg["F"], cfg["D"], info["rows_per_field"],
                                    "uniform int64", cfg["id_batches"])
                      | ({"note": "CPU arm runs the single-process configuration (one batch of B per step) at every N"}
                         if args.gpus > 1 else {}),
            "cpu_baseline": {"value": sps, "unit": "samples/s", **info},
            "e2e": {"value": sps, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------
# e2e harness: pinned host inputs -> H2D (double-buffered on a copy stream) -> public autograd API -> loss D2H
# ----------------------------------------------------------------------------------------------------
def h2d_probe(dev, nbytes):
    """Pinned-host -> device copy rate for one step's input size (explains the e2e bound: the copy of step i+1 overlaps the
    compute of step i, so a step cannot be shorter than its H2D copy)."""
    src = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    dst = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    for _ in range(2):
        dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(10):
        dst.copy_(src, non_blocking=True)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 10
    return {"h2d_GBps_measured": nbytes / (ms * 1e-3) / 1e9, "h2d_ms_per_step_alone": ms}


def e2e_loop(dd: Dist, B, F, host_ids, host_labels, model_step, steps, cuda_graph=False):
    """model_step(ids_dev, labels_dev) -> loss tensor (runs forward+backward through the public API).  Every step's H2D copy
    of ids+labels and the D2H of its loss are inside the timed region; the loss is READ on the host one step late (so the
    launch latency of step i hides behind step i-1; the last loss is read before the closing event).
    cuda_graph=True: the same public-API calls are captured ONCE per input slot with torch.cuda.graph (they only enqueue work
    on the current stream) and every step replays the graph -- one launch per step instead of ~20, the H2D copies and the
    loss read-back stay outside the graph, per step."""
    dev = dd.dev
    copy_stream = torch.cuda.Stream(device=dev)
    main_stream = torch.cuda.current_stream(dev)
    id_dtype = host_ids[0].dtype
    slots = [(torch.empty((B, F), dtype=id_dtype, device=dev), torch.empty((B, 1), device=dev)) for _ in range(2)]
    ev_ready = [torch.cuda.Event() for _ in range(2)]
    ev_free = [torch.cuda.Event() for _ in range(2)]
    loss_host = torch.zeros(2, dtype=torch.float32).pin_memory()
    ev_loss = [torch.cuda.Event() for _ in range(2)]
    losses = []
    nb = len(host_ids)

    def read_loss(i):
        ev_loss[i % 2].synchronize()
        losses.append(float(loss_host[i % 2]))

    def issue_copy(i):
        sl = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ev_free[sl])
            slots[sl][0].copy_(host_ids[i % nb], non_blocking=True)
            slots[sl][1].copy_(host_labels[i % nb], non_blocking=True)
            ev_ready[sl].record(copy_stream)

    graphs = None
    if cuda_graph:
        graphs = []
        for sl in range(2):
            slots[sl][0].copy_(host_ids[0]); slots[sl][1].copy_(host_labels[0])
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(main_stream)
            with torch.cuda.stream(side):
                for _ in range(3):
                    model_step(*slots[sl])
            main_stream.wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                static_loss = model_step(*slots[sl])
            graphs.append((g, static_loss))

    def one(i):
        sl = i % 2
        main_stream.wait_event(ev_ready[sl])
        if graphs is not None:
            graphs[sl][0].replay()
            loss = graphs[sl][1]
        else:
            loss = model_step(*slots[sl])
        ev_free[sl].record(main_stream)
        loss_host[sl:sl + 1].copy_(loss.detach().reshape(1), non_blocking=True)   # D2H of the step's result
        ev_loss[sl].record(main_stream)
        issue_copy(i + 2)                                                           # next use of this slot
        if i > 0:
            read_loss(i - 1)

    for sl in range(2):
        ev_free[sl].record(main_stream)
    issue_copy(0)
    issue_copy(1)
    for i in range(3):
        one(i)
    read_loss(2)
    dd.barrier()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(3, 3 + steps):
        one(i)
    read_loss(3 + steps - 1)
    e1.record()
    dd.barrier()
    ms = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)   # never less than the wall clock
    return dd.max(ms), losses


# ----------------------------------------------------------------------------------------------------
# DeepFM lookup+FM2 (configs[4]): one GPU / replicas, or row-sharded over the ranks
# ----------------------------------------------------------------------------------------------------
def make_ids(args, rows, B, F, NB, dev, gen):
    if args.ids == "zipf":
        # SURVEY 8d config 5, second case: Zipf(1.05) over each field's vocabulary (hot rows are served by L2), inverse CDF
        cdf = torch.cumsum(torch.arange(1, rows + 1, device=dev, dtype=torch.float64) ** -1.05, 0)
        cdf /= cdf[-1].clone()
        sets = [torch.searchsorted(cdf, torch.rand((B, F), device=dev, generator=gen, dtype=torch.float64)).clamp_(max=rows - 1)
                for _ in range(NB)]
        return sets, "Zipf(1.05) int64 (hot rows L2-resident: not the HBM worst case)"
    return [torch.randint(0, rows, (B, F), device=dev, generator=gen) for _ in range(NB)], "uniform int64"


def run_deepfm(args, cfg, dd: Dist):
    from recalgorithm_b200 import _lib, autograd, ops
    dev, world, rank = dd.dev, dd.world, dd.rank
    sharded_mode = bool(cfg.get("sharded"))
    B, F, D, NB = cfg["B"], cfg["F"], cfg["D"], cfg["id_batches"]
    peaks = measured_peaks()
    fwd_b, bwd_b = bytes_per_sample(F, D)
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    d_tile = torch.randn((B, F, D), device=dev, generator=gen) * 0.01      # upstream grad of the deep part
    d_fm2 = torch.randn((B,), device=dev, generator=gen) * 0.01            # upstream grad of the logit
    tile = torch.empty((B, F, D), device=dev)
    fm2 = torch.empty((B, 1), device=dev)
    sampler_idx = dd.local if world > 1 else 0

    def replica_setup():
        rows = int(os.environ.get("CTR_BENCH_ROWS", cfg["rows_per_field"]))      # experiment knob (table-size sweeps)
        tables = autograd.EmbeddingTables([rows] * F, D, device=dev, init=None)
        tables.weight.normal_(0, D ** -0.5, generator=gen)
        id_sets, ids_desc = make_ids(args, rows, B, F, NB, dev, gen)
        row_grads = torch.empty((B, F, D), device=dev)

        def step(i, ev=None):
            if ev:
                ev[0].record()
            ops.embed_fm2_fwd(tables.weight, tables.field_row_offset, id_sets[i % NB], tile=tile, fm2=fm2)
            if ev:
                ev[1].record()
            ops.embed_fm2_bwd(tile, d_tile, d_fm2, row_grads=row_grads)
            if ev:
                ev[2].record()
        return tables, rows, id_sets, ids_desc, step, row_grads

    if not sharded_mode:
        # ------------------------------------------------------------------ one GPU (or N replicas, no exchange step)
        tables, rows, id_sets, ids_desc, step, row_grads = replica_setup()
        for i in range(args.warmup):
            step(i)
        dd.barrier()
        launches0 = _lib.kernel_launches()
        sampler = ClockSampler(sampler_idx).start()
        ms_total, (fwd_ms, bwd_ms) = timed_steps(dd, step, args.steps, n_marks=2)
        clocks = sampler.stop()
        launches = _lib.kernel_launches() - launches0
        if args.dump_outputs and rank == 0:
            # the buffers still hold the last timed step: later measurements reuse them
            dump_outputs(args.dump_outputs, whole={"fm2": fm2}, per_sample={"tile": tile, "row_grads": row_grads})
        value = world * B * args.steps / (ms_total * 1e-3)
        sustained = sustained_run(dd, step, ms_total / args.steps, B)

        # e2e: public autograd API, int32 ids over PCIe, lookup + FM2 + fused dense(1) head -> sigmoid-CE -> backward
        e2e_steps = max(3, min(args.steps, 50))
        w_deep = (torch.randn((F * D, 1), device=dev, generator=gen) * 0.01).requires_grad_()
        ids_host = [s.int().cpu().pin_memory() for s in id_sets[:4]]
        lab_host = [(torch.rand((B, 1)) < 0.0356).float().pin_memory() for _ in range(4)]

        def model_fused(ids_dev, lab_dev):
            tables.zero_grad()
            w_deep.grad = None
            f_, lin = autograd.lookup_fm2_linear(tables, ids_dev, w_deep)          # deep head fused into the gather
            loss = autograd.sigmoid_cross_entropy_mean(f_, lab_dev, logit_b=lin)   # add_n of the logits + sigmoid-CE + its gradient, one launch
            loss.backward()
            return loss

        def model_unfused(ids_dev, lab_dev):
            tables.zero_grad()
            w_deep.grad = None
            t_, f_ = autograd.lookup_fm2(tables, ids_dev)
            logit = f_ + t_.reshape(B, F * D) @ w_deep                              # dense(1) consumer of the tile in torch
            loss = torch.nn.functional.binary_cross_entropy_with_logits(logit, lab_dev)
            loss.backward()
            return loss

        e2e_ms_eager, losses_eager = e2e_loop(dd, B, F, ids_host, lab_host, model_fused, e2e_steps)
        e2e_ms_unf, losses_unf = e2e_loop(dd, B, F, ids_host, lab_host, model_unfused, e2e_steps)
        try:
            e2e_ms, losses = e2e_loop(dd, B, F, ids_host, lab_host, model_fused, e2e_steps, cuda_graph=True)
            e2e_mode = "cuda graph replay of the public-API step"
        except Exception as exc:                                   # capture refused on this stack: the eager number is the e2e number
            e2e_ms, losses, e2e_mode = e2e_ms_eager, losses_eager, f"eager (graph capture failed: {type(exc).__name__}: {exc})"
        if e2e_ms > e2e_ms_eager:
            e2e_ms, losses, e2e_mode = e2e_ms_eager, losses_eager, "eager (the graph replay was not faster)"
        e2e_value = world * B * e2e_steps / (e2e_ms * 1e-3)
        pcie = h2d_probe(dev, B * F * 4 + B * 4)
        if rank != 0:
            return
        ach_fwd = fwd_b * B / (fwd_ms * 1e-3) / 1e9
        ach_bwd = bwd_b * B / (bwd_ms * 1e-3) / 1e9
        ach_step = (fwd_b + bwd_b) * B * args.steps / (ms_total * 1e-3) / 1e9
        traffic, traffic_src = measured_traffic(args.workload, args.ids)
        hbm = peaks["hbm_gbs"]
        line = {
            "metric": "ctr_fwd_bwd_samples_per_sec", "value": value, "unit": "samples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": deepfm_config(args.workload, cfg["model"], B, world, F, D, rows, ids_desc, NB),
            "roofline": {"bound": "hbm", "kernel": "embed_fm2_fwd_kernel<8> (fused gather + FM2)", "achieved": ach_fwd,
                         "peak": hbm, "unit": "GB/s", "frac": ach_fwd / hbm, "traffic": traffic, "traffic_source": traffic_src,
                         "kernel_source_sha256_16": kernel_source_hash(), "peak_source": peaks["source"],
                         "algorithmic_bytes_per_launch": fwd_b * B, "avg_launch_ms": fwd_ms},
            "roofline_bwd": {"kernel": "embed_fm2_bwd_kernel", "achieved": ach_bwd, "frac": ach_bwd / hbm,
                             "algorithmic_bytes_per_launch": bwd_b * B, "avg_launch_ms": bwd_ms},
            "roofline_step": {"achieved": ach_step, "frac": ach_step / hbm, "bytes_per_sample": fwd_b + bwd_b},
            "sustained": sustained,
            "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": B * F * 4 + B * 4,
                    "d2h_bytes_per_step": 4, "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps, "loss_last": losses[-1], **pcie,
                    "what": "pinned-host int32 ids + labels -> H2D (double-buffered on a copy stream) -> autograd.lookup_fm2_linear "
                            "(gather + FM2 + dense(1) deep head in one kernel; ids widened on device) -> autograd.sigmoid_cross_entropy_mean (logit sum + loss + gradient, one launch) -> backward "
                            "(ctr_embed_fm2_lin_bwd -> IndexedSlices + d_w) -> loss D2H to pinned memory, read on the host one step later",
                    "launch": e2e_mode,
                    "eager": {"value": world * B * e2e_steps / (e2e_ms_eager * 1e-3), "ms_per_step": e2e_ms_eager / e2e_steps,
                              "loss_last": losses_eager[-1], "what": "the same step issued call by call (no graph)"},
                    "unfused_head": {"value": world * B * e2e_steps / (e2e_ms_unf * 1e-3), "ms_per_step": e2e_ms_unf / e2e_steps,
                                     "loss_last": losses_unf[-1],
                                     "what": "same, with autograd.lookup_fm2 + a torch matmul head (the tile is re-streamed by cuBLAS)"}},
            "gpu_launches": int(launches), "clocks": clocks,
        }
        if world == 1 and not args.no_extra and args.ids == "uniform":
            # the same step on Zipf(1.05) ids (SURVEY 8d's second case): hot rows are served by the 126 MB L2, so the
            # algorithmic rate may exceed the HBM peak -- reported beside the uniform (L2-miss) headline, never instead of it
            zargs = argparse.Namespace(**{**vars(args), "ids": "zipf"})
            zsets, zdesc = make_ids(zargs, rows, B, F, NB, dev, gen)

            def zstep(i, ev=None):
                if ev:
                    ev[0].record()
                ops.embed_fm2_fwd(tables.weight, tables.field_row_offset, zsets[i % NB], tile=tile, fm2=fm2)
                if ev:
                    ev[1].record()
                ops.embed_fm2_bwd(tile, d_tile, d_fm2, row_grads=row_grads_z)
                if ev:
                    ev[2].record()
            row_grads_z = torch.empty((B, F, D), device=dev)
            for i in range(3):
                zstep(i)
            zn = min(args.steps, 50)
            zms, (zf, zb) = timed_steps(dd, zstep, zn, n_marks=2)
            line["zipf"] = {"value": B * zn / (zms * 1e-3), "unit": "samples/s", "ms_per_step": zms / zn, "ids": zdesc,
                            "fwd_ms": zf, "bwd_ms": zb, "fwd_algorithmic_GBps": fwd_b * B / (zf * 1e-3) / 1e9,
                            "fwd_frac_of_hbm_peak": fwd_b * B / (zf * 1e-3) / 1e9 / hbm,
                            "note": "algorithmic bytes over time; rows that hit L2 never reach HBM, so this is not an HBM utilisation"}
            del zsets, row_grads_z
        if world == 1 and not args.no_extra:
            line["configs"] = {}
            del tables, id_sets
            torch.cuda.empty_cache()
            for name in LAYER_WORKLOADS:
                line["configs"][name] = layer_workload_measure(dd, name, steps=min(args.steps, 30), warmup=3, brief=True)[0]
                torch.cuda.empty_cache()
        if world == 1 and not args.no_cpu_baseline:
            for name in line.get("configs", {}):                           # the reference's CPU path beside each of configs 2-4
                line["configs"][name]["cpu_baseline"] = safe_cpu_layer_baseline(name, budget_s=4.0)
            try:
                sps, ms, info = cpu_reference_run(cfg, steps=4, warmup=1, budget_s=30.0)
                line["cpu_baseline"] = {"value": sps, "unit": "samples/s", "ms_per_step": ms, **info}
            except Exception as ex:                                        # noqa: BLE001  (e.g. a host without the RAM for the tables)
                line["cpu_baseline"] = {"unavailable": f"{type(ex).__name__}: {str(ex)[:160]}"}
        print(json.dumps(line), flush=True)
        return

    # ---------------------------------------------------------------------- row-sharded over the ranks (SURVEY 8e)
    if world < 2:
        raise SystemExit(f"{args.workload} needs --gpus >= 2 (launch under torchrun)")
    from recalgorithm_b200 import sharded as shard_mod
    rows = cfg["rows_per_field_per_rank"] * world
    if os.environ.get("CTR_BENCH_ROWS"):
        rows = int(os.environ["CTR_BENCH_ROWS"])
    plan = torch.empty((B, F), dtype=torch.int32, device=dev)
    align_token = torch.zeros((1,), device=dev)

    def make_sharded(rows_):
        tb = shard_mod.ShardedEmbeddingTables([rows_] * F, D, batch_per_rank=B, device=dev, init="normal",
                                              shard_backend=args.shard_backend, vmm_align=args.vmm_align << 20)
        sets, desc = make_ids(args, rows_, B, F, NB, dev, gen)

        def step_(i, ev=None):
            ids = sets[i % NB]
            if ev:
                ev[0].record()
            tb.plan(ids, plan=plan, side_stream=True)                      # queue slots + row indices, on a side stream BESIDE the pull
            if ev:
                ev[1].record()
            tb.lookup_fm2(ids, tile=tile, fm2=fm2)                         # rows pulled from the owners over NVLink
            if ev:
                ev[2].record()
            tb.bwd_push(tile, d_tile, d_fm2, plan)                         # gradient rows stored straight into the owners' queues
            if ev:
                ev[3].record()
            if args.align_steps and world > 1:
                # what the dense-gradient all-reduce of a real step does as a side effect: it keeps the ranks' pull / push phases
                # aligned (stream-ordered 1-element NCCL all-reduce, no host sync).  Unaligned ranks load one NVLink direction with
                # push payload AND read responses while the other idles.
                dd.dist.all_reduce(align_token)
        return tb, sets, desc, step_

    tables, id_sets, ids_desc, step = make_sharded(rows)

    for i in range(args.warmup):
        step(i)
    dd.barrier()
    launches0 = _lib.kernel_launches()
    sampler = ClockSampler(sampler_idx).start()
    ms_total, (plan_ms, fwd_ms, push_ms) = timed_steps(dd, step, args.steps, n_marks=3)
    clocks = sampler.stop()
    launches = _lib.kernel_launches() - launches0
    tables.finish_push()                                                # raises if a receive queue overflowed
    value = world * B * args.steps / (ms_total * 1e-3)
    per_rank = {"plan_ms": dd.gather(plan_ms), "pull_ms": dd.gather(fwd_ms), "bwd_push_ms": dd.gather(push_ms)}
    sustained = sustained_run(dd, step, ms_total / args.steps, B)
    tables.finish_push()

    # e2e through the public sharded API: pinned int32 ids -> H2D -> lookup_fm2_autograd -> head + loss -> backward (push)
    e2e_steps = max(3, min(args.steps, 50))
    w_deep = (torch.randn((F * D, 1), device=dev, generator=gen) * 0.01).requires_grad_()
    ids_host = [s.int().cpu().pin_memory() for s in id_sets[:4]]
    lab_host = [(torch.rand((B, 1)) < 0.0356).float().pin_memory() for _ in range(4)]

    def model_sharded(ids_dev, lab_dev):
        w_deep.grad = None
        f_, lin = shard_mod.lookup_fm2_linear_autograd(tables, ids_dev, w_deep)     # dense(1) deep head fused into the gather
        loss = autograd.sigmoid_cross_entropy_mean(f_, lab_dev, logit_b=lin)
        loss.backward()
        if world > 1:
            dd.dist.all_reduce(w_deep.grad)                    # the replicated dense head's gradient: summed over the data-parallel ranks
        return loss

    e2e_ms, losses = e2e_loop(dd, B, F, ids_host, lab_host, model_sharded, e2e_steps)
    tables.finish_push()
    e2e_eager = {"value": world * B * e2e_steps / (e2e_ms * 1e-3), "ms_per_step": e2e_ms / e2e_steps, "loss_last": losses[-1],
                 "what": "the same step issued call by call (no graph)"}
    e2e_mode = "eager"
    if args.e2e_graph:
        # the same public-API step (side-stream plan, NCCL all-reduce of d_w included) captured once per input slot and replayed:
        # at 2-4 GPUs the eager step is bound by the host issuing ~25 calls, not by the GPUs
        try:
            g_ms, g_losses = e2e_loop(dd, B, F, ids_host, lab_host, model_sharded, e2e_steps, cuda_graph=True)
            tables.finish_push()
            if g_ms < e2e_ms:
                e2e_ms, losses, e2e_mode = g_ms, g_losses, "cuda graph replay of the public-API step"
            else:
                e2e_mode = "eager (the graph replay was not faster)"
        except Exception as ex:                                              # noqa: BLE001  (reported, the eager number stands)
            e2e_mode = f"eager (graph capture failed: {type(ex).__name__}: {str(ex)[:120]})"
    e2e_value = world * B * e2e_steps / (e2e_ms * 1e-3)
    del tables
    torch.cuda.empty_cache()

    # BASELINE's literal vocabulary (100 M rows in total, 12.8 GB) split over the same ranks: the shard is 12.8 GB / N per GPU
    v100 = None
    if not args.no_extra and "rows_per_field" in cfg:
        rows100 = cfg["rows_per_field"]
        tb100, _s, _d, step100 = make_sharded(rows100)
        for i in range(3):
            step100(i)
        n100 = min(args.steps, 50)
        ms100, (p100, f100, b100) = timed_steps(dd, step100, n100, n_marks=3)
        tb100.finish_push()
        nvb = B * F * D * 4 * (world - 1) / world
        v100 = {"value": world * B * n100 / (ms100 * 1e-3), "ms_per_step": ms100 / n100, "rows_per_field": rows100,
                "vocab_rows_total": rows100 * F, "shard_bytes_per_gpu": rows100 * F * D * 4 // world,
                "plan_ms": p100, "pull_ms": f100, "bwd_push_ms": b100, "pull_GBps": nvb / (f100 * 1e-3) / 1e9,
                "push_GBps": nvb / (b100 * 1e-3) / 1e9,
                "what": "the same step on BASELINE's literal 100 M-row vocabulary row-sharded over the ranks (1.6-6.4 GB shards instead "
                        "of 32 GB: same link traffic per step, DESIGN 6)"}
        del tb100, step100
        torch.cuda.empty_cache()

    # the zero-traffic split of the same batch (replicated 12.8 GB table) for comparison -- NOT the headline at N > 1
    rep = None
    if not args.no_extra:
        _t, _rows, _ids, _desc, rstep, _rg = replica_setup()
        for i in range(3):
            rstep(i)
        rms, _ = timed_steps(dd, rstep, min(args.steps, 50))
        rep = {"value": world * B * min(args.steps, 50) / (rms * 1e-3), "ms_per_step": rms / min(args.steps, 50),
               "what": "replicated 12.8 GB table per rank, no exchange (the table fits one GPU): upper bound, zero NVLink traffic"}
    if rank != 0:
        return
    remote = (world - 1) / world
    nv_bytes = B * F * D * 4 * remote                       # payload crossing NVLink per rank per direction, each way
    hbm = peaks["hbm_gbs"]
    pull_nv_ms = nv_bytes / NVLINK_PEAK_GBS / 1e6
    pull_hbm_ms = (fwd_b * B - nv_bytes) / hbm / 1e6          # local rows + ids + the tile write
    push_hbm_ms = (F * 2 * D * 4 + 8) * B / hbm / 1e6         # tile + d_tile read (row_grads never written)
    bound_ms = max(pull_nv_ms, pull_hbm_ms) + max(pull_nv_ms, push_hbm_ms)
    pull_gbs = [nv_bytes / (t * 1e-3) / 1e9 for t in per_rank["pull_ms"]]
    push_gbs = [nv_bytes / (t * 1e-3) / 1e9 for t in per_rank["bwd_push_ms"]]
    print("[bench] per-rank NVLink GB/s  pull: " + " ".join(f"{x:.0f}" for x in pull_gbs) + "   push: " +
          " ".join(f"{x:.0f}" for x in push_gbs), file=sys.stderr, flush=True)
    line = {
        "metric": "ctr_fwd_bwd_samples_per_sec", "value": value, "unit": "samples/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "model": cfg["model"], "global_batch": B * world, "B_per_gpu": B, "F": F,
                   "D": D, "rows_per_field": rows, "vocab_rows_total": rows * F, "table_bytes_total": rows * F * D * 4,
                   "shard_bytes_per_gpu": rows * F * D * 4 // world, "ids": ids_desc,
                   "shard_backend": args.shard_backend + (f" (align {args.vmm_align} MiB)" if args.shard_backend == "vmm" else ""),
                   "rank_alignment": "1-element NCCL all-reduce per step (stream-ordered, no host sync)" if args.align_steps else "none (free-running ranks)",
                   "parallelism": f"row-sharded: tables split over {world} GPUs (global row % {world}); forward pulls rows over NVLink "
                                  "inside the gather kernel, backward stores gradient rows into the owners' queues (fused "
                                  "compute+exchange kernels, no NCCL data collective)",
                   "l2": "inputs larger than L2 (rotating id batches over a 32 GB shard per GPU)"},
        "roofline": {"bound": "nvlink", "kernel": "embed_fm2_fwd_kernel<8,sharded> (peer-pull gather + FM2)",
                     "achieved": nv_bytes / (fwd_ms * 1e-3) / 1e9, "peak": NVLINK_PEAK_GBS, "unit": "GB/s",
                     "frac": nv_bytes / (fwd_ms * 1e-3) / 1e9 / NVLINK_PEAK_GBS, "traffic": None,
                     "peak_source": "B200_PROFILING.md: measured peer copy 770 GB/s per direction per GPU",
                     "nvlink_bytes_per_direction_per_rank": nv_bytes, "avg_launch_ms": fwd_ms,
                     "push": {"kernel": "embed_fm2_bwd_push_kernel<8,12> (backward fused with the gradient exchange)",
                              "achieved": nv_bytes / (push_ms * 1e-3) / 1e9, "frac": nv_bytes / (push_ms * 1e-3) / 1e9 / NVLINK_PEAK_GBS,
                              "avg_launch_ms": push_ms},
                     "plan_ms": plan_ms, "per_rank_pull_GBps": pull_gbs, "per_rank_push_GBps": push_gbs,
                     "step_bound_ms": bound_ms, "step_frac_of_bound": bound_ms / (ms_total / args.steps),
                     "bound_terms_ms": {"pull_nvlink": pull_nv_ms, "pull_hbm": pull_hbm_ms, "push_nvlink": pull_nv_ms, "push_hbm": push_hbm_ms},
                     "link_ceiling_note": "tools/peerbench.cu (all ranks active, 128 B rows): pull tops out at ~650 GB/s, push at ~690 GB/s"},
        "sustained": sustained,
        "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": B * F * 4 + B * 4, "d2h_bytes_per_step": 4,
                "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps, "loss_last": losses[-1], "launch": e2e_mode, "eager": e2e_eager,
                "what": "per rank: pinned-host int32 ids + labels -> H2D -> sharded.lookup_fm2_linear_autograd (peer-pull gather + FM2 + "
                        "dense(1) deep head in one kernel, queue plan beside it) -> sigmoid-CE (ctr_sigmoid_ce) -> backward (ctr_embed_fm2_lin_bwd_push: "
                        "gradient rows into the owners' queues + d_w) -> NCCL all-reduce of the replicated head's d_w -> loss D2H, read one step later"},
        "vocab_100m": v100, "replicas": rep, "gpu_launches": int(launches), "clocks": clocks,
        "comm_nranks": int(dd.dist.get_world_size()), "comm_backend": "nccl (handles, barriers, 1-element alignment all-reduce; no data-plane collective)",
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------
# configs 2, 3, 4: lookup + interaction layer chains
# ----------------------------------------------------------------------------------------------------
def layer_workload_measure(dd: Dist, name, steps, warmup, brief=False):
    from tools import workloads as W
    peaks = measured_peaks()
    wl = W.BUILDERS[name]()
    flush = torch.empty(64 * 1024 * 1024, device=dd.dev)      # 256 MB: these working sets fit the 126 MB L2, flush it every step
    marks = wl["marks"]

    def step(i, ev=None):
        flush.zero_()
        wl["step"](ev)

    for i in range(warmup):
        step(i)
    # per-stage events bracket the stages only (the flush sits before event 0): step time = sum of the stages
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(len(marks) + 1)] for _ in range(steps)]
    dd.barrier()
    for i in range(steps):
        step(i, evs[i])
    dd.barrier()
    per = {m: statistics.mean(e[j].elapsed_time(e[j + 1]) for e in evs) for j, m in enumerate(marks)}
    ms_step = dd.max(statistics.mean(e[0].elapsed_time(e[-1]) for e in evs))
    out = {"value": dd.world * wl["B"] / (ms_step * 1e-3), "unit": "samples/s", "ms_per_step": ms_step, "stage_ms": per,
           "roofline": wl["roofline"](per, ms_step, peaks), "config": wl["config"], "dtype": wl["dtype"], "steps": steps,
           "what": "lookup fwd + interaction fwd + interaction bwd + lookup bwd (IndexedSlices); no dense tail; L2 flushed before every step"}
    if name == "dcn_cfg2":
        g = W.graphed(lambda: wl["step"](None))
        for _ in range(3):
            g()
        ts = []
        for _ in range(steps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); g(); b.record()
            ts.append((a, b))
        torch.cuda.synchronize()
        gms = statistics.mean(a.elapsed_time(b) for a, b in ts)
        out["cuda_graph"] = {"ms_per_step": gms, "value": dd.world * wl["B"] / (gms * 1e-3), "what": "the same C-ABI calls captured once, one graph replay per step"}
    if brief:
        out = {k: out[k] for k in ("value", "unit", "ms_per_step", "stage_ms", "roofline", "config") if k in out} | (
            {"cuda_graph": out["cuda_graph"]} if "cuda_graph" in out else {})
    return out, wl


def run_layer_workload(args, dd: Dist):
    from recalgorithm_b200 import _lib
    sampler = ClockSampler(dd.local if dd.world > 1 else 0).start()
    n0 = _lib.kernel_launches()
    res, wl = layer_workload_measure(dd, args.workload, args.steps, args.warmup)
    launches = _lib.kernel_launches() - n0
    clocks = sampler.stop()
    sustained = sustained_run(dd, lambda i, ev=None: wl["step"](None), res["ms_per_step"], wl["B"])
    sustained["l2"] = "NOT flushed in this loop (its purpose is the clock record under seconds of load)"
    if dd.rank != 0:
        return
    line = {"metric": "ctr_fwd_bwd_samples_per_sec", "value": res["value"], "unit": "samples/s", "n_gpus": dd.world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": res["dtype"], "data": "synthetic",
            "config": {**res["config"], "l2": "flushed (256 MB write) before every step; flush excluded from the step time",
                       "parallelism": "independent replicas" if dd.world > 1 else "1 GPU"},
            "roofline": res["roofline"], "stage_ms": res["stage_ms"], "sustained": sustained,
            "e2e": None, "gpu_launches": int(launches), "clocks": clocks, "what": res["what"]}
    if "cuda_graph" in res:
        line["cuda_graph"] = res["cuda_graph"]
    if dd.world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = safe_cpu_layer_baseline(args.workload, budget_s=15.0)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(DEEPFM) + list(LAYER_WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the configs 2-4 / replica side measurements")
    ap.add_argument("--shard-backend", default="symm", choices=["symm", "vmm"],
                    help="allocation of the table shard in the sharded workloads: torch symmetric memory or ctr_vmm_alloc")
    ap.add_argument("--vmm-align", type=int, default=0, help="MiB; size/address alignment of ctr_vmm_alloc (0 = driver granularity)")
    ap.add_argument("--align-steps", type=int, default=1,
                    help="sharded workloads: 1 = every step ends with a stream-ordered 1-element NCCL all-reduce that keeps the ranks' "
                         "phases aligned (stands in for the dense-gradient all-reduce of a real step); 0 = free-running ranks")
    ap.add_argument("--e2e-graph", type=int, default=1,
                    help="sharded workloads: 1 = also time the e2e step as a CUDA-graph replay and report the faster form")
    ap.add_argument("--ids", default="uniform", choices=["uniform", "zipf"],
                    help="id distribution of the synthetic batches (default: uniform = every row an HBM miss)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32, at most 60 MB): fm2 in "
                         "full, tile and row_grads for a fixed, seeded sample of batch rows (replicated DeepFM workloads, rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.workload is None:
        # BASELINE config 5 names the row-sharded split: it is the headline whenever there is more than one GPU
        args.workload = "deepfm_cfg5_sharded" if (world > 1 and args.impl == "ours") else "deepfm_cfg5"
    if args.dump_outputs and (args.impl != "ours" or args.workload not in DEEPFM or DEEPFM[args.workload].get("sharded")):
        ap.error("--dump-outputs covers the replicated DeepFM workloads of --impl ours only")
    if args.impl == "reference":
        if args.workload in LAYER_WORKLOADS:
            run_reference_arm_layers(args)
        else:
            run_reference_arm(args, DEEPFM[args.workload])
        return
    dd = Dist()
    if args.workload in DEEPFM:
        run_deepfm(args, DEEPFM[args.workload], dd)
    else:
        run_layer_workload(args, dd)
    if dd.world > 1 and torch.distributed.is_initialized():
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
