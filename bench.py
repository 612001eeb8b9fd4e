#!/usr/bin/env python
"""bench.py -- predict QPS of the route -> ensure-resident -> predict hot path on a Zipf
multi-model mix (BASELINE.json metric), one process per GPU.

Workload (config.workload): the per-GPU shard of BASELINE.json configs[2] -- the configuration the
north_star target is quoted on: N GPUs serve 125*N per-tenant 3-layer MLPs (9216^4 fp32,
1 019 326 464 B each), Zipf(alpha=1.0) request stream, ring replicas = min(2, N).  Per-GPU work is
fixed as N grows (weak scaling); at N=8 it is exactly configs[2] (1000 models, replicas 2).

A "step" is one batcher tick: `--tick` (default 1024) requests per GPU drawn from the seeded Zipf
trace, routed with the consistent-hash ring, grouped per resident model and executed.
  value  : whole-job req/s with the step's inputs already resident in HBM (device pointers through
           tfsc_predict_device), timed with CUDA events on the launching stream.
  e2e    : the same ticks through the public C ABI (tfsc_predict / tfsc_predict_member) with HOST buffers from
           `--clients` closed-loop client threads (transfers of inputs and results inside the timed
           region), plus p50/p99 latency and a client sweep for the QPS that still meets p50 < 5 ms.
  forward: at N > 1 a fraction `--forward-frac` of the requests ENTERS at a rank that does not own the model
           (a6, taskhandler.go:95-147): their rows sit in the ingress rank's forward window and the owner reads /
           writes them over NVLink (gather / scatter kernels), in both the value and the e2e region.
  cache_pressure: a short phase with the HBM-resident set capped below the working set (uniform trace, BASELINE
           configs[4]-style storm): hit %, reloads, H2D GB/s against the PCIe roofline, load-stall p99.
  extra  : device-resident ResNet-50 (configs[1]) and BERT-base (configs[3]) model speed, N=1 only.
  --impl reference : the reference's CPU path restated (ring -> LRU/top-N residency -> per-request,
           unbatched fp32 forward on all host cores, oracle C), on a bounded sample.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DIMS = [9216, 9216, 9216, 9216]
MODEL_BYTES = 1019326464
MODELS_PER_GPU = 125
IN_DIM, OUT_DIM = DIMS[0], DIMS[-1]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--tick", type=int, default=1024, help="requests per GPU per step")
    ap.add_argument("--clients", type=int, default=1024, help="closed-loop client threads per GPU (e2e)")
    ap.add_argument("--models-per-gpu", type=int, default=MODELS_PER_GPU)
    ap.add_argument("--arena-gib", type=float, default=160.0)
    ap.add_argument("--host-gib", type=float, default=0.0, help="pinned host tier per GPU (0 = auto)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = same as --steps")
    ap.add_argument("--cpu-sample", type=int, default=48, help="requests in the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true", help="profiling runs only (ncu): device-resident part alone")
    ap.add_argument("--light-clients", type=int, default=16, help="clients per GPU of the light-load latency probe (0 = skip)")
    ap.add_argument("--dims", type=int, nargs="*", default=None, help="override model dims (debug only)")
    ap.add_argument("--forward-frac", type=float, default=0.25,
                    help="N > 1: fraction of requests whose ingress rank is not the owner (forward hop over NVLink)")
    ap.add_argument("--no-extras", action="store_true", help="skip cache_pressure / sweep / extra model lines (profiling runs)")
    ap.add_argument("--pressure-resident", type=int, default=32, help="HBM-resident cap of the cache_pressure phase")
    ap.add_argument("--preheat-s", type=float, default=2.0, help="untimed seconds of real passes right before the timed region")
    ap.add_argument("--samplers", default="smi+nvml", choices=["smi+nvml", "smi", "nvml", "none"],
                    help="clock samplers running during the timed regions (A/B their perturbation with 'none')")
    ap.add_argument("--replica-pick", default="balanced", choices=["balanced", "hot-spread", "random", "first", "hash"],
                    help="replica choice among the ring's GetN candidates (reference: random)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the results of the last one as DIR/predict_y.npy (float32, at most 64 MB: "
                         "a larger result is cut to a fixed seeded sample of its rows); at N > 1 one file per rank, predict_y_rank<r>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be >= 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the results of the b200 path only")
    return a


DUMP_MAX_BYTES = 64 << 20


def sample_rows(y: np.ndarray, max_bytes: int, seed: int = 0) -> np.ndarray:
    """y itself when it fits in max_bytes, else a fixed seeded sample of its rows, kept in their original order."""
    keep = max_bytes // max(1, y[:1].nbytes)
    if len(y) <= keep:
        return y
    return y[np.sort(np.random.default_rng(seed).choice(len(y), keep, replace=False))]


def effective_cpus() -> int:
    """CPUs this process may actually use: min(os.cpu_count(), sched affinity, cgroup-v2 cpu.max quota). The GPU boxes
    expose 128 logical CPUs but cap the container at 16 CPUs of quota; running 128 busy threads there only earns
    CFS throttling."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(per))))
    except Exception:
        pass
    return max(1, n)


# ------------------------------------------------------------------------------- workload ------
def splitmix(i: np.ndarray) -> np.ndarray:
    z = (i.astype(np.uint64) + np.uint64(0x9E3779B97F4A7C15))
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def build_workload(n_gpus, models_per_gpu, tick, n_steps, seed=42, pick_policy="balanced", forward_frac=0.0):
    """Global request stream + ring routing, identical on every rank (no communication)."""
    import tfservingcache_b200 as t
    from tools.traces import zipf_trace
    n_models = models_per_gpu * n_gpus
    replicas = min(2, n_gpus)
    members = [f"gpu{i}:0:0" for i in range(n_gpus)]
    cluster = t.ClusterConnection(replicas)
    cluster.update([t.ServingService.from_string(m) for m in members])
    owners = np.empty((n_models, replicas), dtype=np.int32)
    for j in range(n_models):
        nodes = cluster.find_node_for_key(t.model_key(f"m{j}", "1"))  # nodeForKey, taskhandler.go:84-92
        owners[j] = [int(s.host[3:]) for s in nodes]
    total = tick * n_gpus * n_steps
    trace = zipf_trace(n_models, total, 1.0, seed)
    # replica choice (taskhandler.go:91 picks at random; default here: primary unless the model is hot) with the
    # library's deterministic picker, fed the same global request sequence on every rank so all ranks agree
    picker = t.ReplicaPicker(pick_policy, seed, 0.25)
    keys = [t.model_key(f"m{j}", "1") for j in range(n_models)]
    own = [[int(v) for v in owners[j]] for j in range(n_models)]
    pick = np.fromiter((picker.pick_ids(keys[m], own[m], n_gpus) for m in trace.tolist()), dtype=np.int64, count=total)
    dest = owners[trace, pick]
    # ingress rank of every request: the owner itself, or (fraction forward_frac) another rank chosen uniformly -- the
    # front load balancer of a real deployment does not know the ring
    ingress = dest.copy()
    if n_gpus > 1 and forward_frac > 0:
        rng = np.random.default_rng(seed + 7)
        fw = rng.random(total) < forward_frac
        other = (dest + rng.integers(1, n_gpus, size=total)) % n_gpus
        ingress = np.where(fw, other, dest).astype(dest.dtype)
    return dict(n_models=n_models, replicas=replicas, members=members, trace=trace, dest=dest, owners=owners,
                pick_policy=pick_policy, ingress=ingress, forward_frac=forward_frac if n_gpus > 1 else 0.0)


def step_groups(wl, rank, step, tick_global):
    """Requests of `step` owned by `rank`, grouped per model: [(model, count)] in first-arrival order."""
    lo, hi = step * tick_global, (step + 1) * tick_global
    mine = wl["trace"][lo:hi][wl["dest"][lo:hi] == rank]
    order, counts = [], {}
    for m in mine.tolist():
        if m not in counts:
            order.append(m)
            counts[m] = 0
        counts[m] += 1
    return mine, [(m, counts[m]) for m in order]


def step_plan(wl, rank, step, tick_global):
    """Owner-side plan of one step: for every model group owned by `rank`, how many rows entered locally and, for the
    forwarded rows, (ingress rank, slot index k in that rank's forward window). k enumerates ALL forwarded requests of
    the ingress rank in the step, so owners writing results into the same window never collide."""
    lo, hi = step * tick_global, (step + 1) * tick_global
    tr, de, ing = wl["trace"][lo:hi], wl["dest"][lo:hi], wl["ingress"][lo:hi]
    fw = ing != de
    slot_k = np.zeros(hi - lo, np.int64)
    for p in np.unique(ing[fw]).tolist():
        sel = np.nonzero(fw & (ing == p))[0]
        slot_k[sel] = np.arange(len(sel))
    order, local, fwd = [], {}, {}
    for i in np.nonzero(de == rank)[0].tolist():
        m = int(tr[i])
        if m not in local:
            order.append(m)
            local[m], fwd[m] = 0, []
        if fw[i]:
            fwd[m].append((int(ing[i]), int(slot_k[i])))
        else:
            local[m] += 1
    return [(m, local[m], fwd[m]) for m in order]


def pass_plan(rows, tc_min=9):
    """Mirror of launch_dense (csrc/kernels.cu): groups of >= 9 rows take the tcgen05 path, 64 rows per
    pass; what is left (<= 8 rows) takes one SIMT streaming pass."""
    out, r = [], rows
    while tc_min > 0 and r >= tc_min:
        rr = min(64, r)
        out.append(("tc", rr))
        r -= rr
    while r > 0:
        rr = min(8, r)
        out.append(("simt", rr))
        r -= rr
    return out


def algorithmic_bytes(groups, dims):
    """SURVEY 8(d): per launch of one dense layer = W + bias + rows*(in+out)*4; every pass streams W once."""
    total, launches, tc = 0, 0, 0
    tc_min = int(os.environ.get("TFSC_TC_MIN_ROWS", "9"))
    for _m, rows in groups:
        for kind, rr in pass_plan(rows, tc_min):
            for l in range(len(dims) - 1):
                total += dims[l] * dims[l + 1] * 4 + dims[l + 1] * 4 + rr * (dims[l] + dims[l + 1]) * 4
                launches += 1
                tc += kind == "tc"
    return total, launches


# ---------------------------------------------------------------------------------- clocks ------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index, enabled=True):
        self.rows, self.proc, self.idx, self.windows, self.enabled = [], None, gpu_index, [], enabled

    def start(self):
        if not self.enabled:   # one nvidia-smi loop per box (local rank 0), as in the profiling recipe: eight concurrent
            return             # loops each polling all eight GPUs perturb the very kernels they are meant to watch
        try:
            # all GPUs of the box are sampled (rank 0 only): a multi-GPU run can be slowed by one throttled device
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([time.time()] + [c.strip() for c in line.split(",")])

    def mark(self, t0, t1):
        """A timed window (value or e2e region); only samples inside the marked windows are reported."""
        self.windows.append((t0, t1))

    def stop(self):
        if not self.enabled:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "per_gpu": []}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        per = {}
        for row in self.rows:
            ts, r = row[0], row[1:]
            if self.windows and not any(a - 0.05 <= ts <= b + 0.05 for a, b in self.windows):
                continue
            try:
                g = int(r[0])
                d = per.setdefault(g, {"sm": [], "pw": [], "reasons": set()})
                d["sm"].append(float(r[1]))
                d["pw"].append(float(r[3]))
                if g == self.idx:
                    sm.append(float(r[1]))
                    mx = max(mx, float(r[2]))
                for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                    if r[col].lower().startswith("active"):
                        d["reasons"].add(name)
                        if g == self.idx:
                            reasons.add(name)
            except Exception:
                pass
        per_gpu = [{"gpu": g, "sm_mhz": float(np.median(d["sm"])), "power_w": round(float(np.median(d["pw"])), 1),
                    "reasons": sorted(d["reasons"])} for g, d in sorted(per.items())]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm), "per_gpu": per_gpu}


class NvmlSampler:
    """Per-rank sampler of this rank's own GPU through NVML (20 ms period; nvidia-smi needs > 200 ms per query on an
    8-GPU box). Reports median SM clock, max clock, median power and the throttle reasons seen inside the marked
    timed windows. Any failure degrades to an empty record -- it must never break the bench."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, gpu_index, period_s=0.02):
        self.idx, self.rows, self.windows, self.ok, self._stop, self.period_s = gpu_index, [], [], False, False, period_s
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def start(self):
        if self.ok:
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()

    def _run(self):
        nv = self.nv
        reasons_fn = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons", None)
        while not self._stop:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                rs = int(reasons_fn(self.h)) if reasons_fn else 0
                try:
                    mem = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_MEM)
                    temp = nv.nvmlDeviceGetTemperature(self.h, nv.NVML_TEMPERATURE_GPU)
                except Exception:
                    mem, temp = -1, -1
                self.rows.append((time.time(), sm, pw, rs, mem, temp))
            except Exception:
                pass
            time.sleep(self.period_s)

    def mark(self, t0, t1):
        self.windows.append((t0, t1))

    def stop(self):
        self._stop = True
        rows = [r for r in self.rows if any(a <= r[0] <= b for a, b in self.windows)] if self.windows else self.rows
        if not self.ok or not rows:
            return None
        mask = 0
        for r in rows:
            mask |= r[3]
        return {"sm_mhz": float(np.median([r[1] for r in rows])), "sm_min_mhz": float(min(r[1] for r in rows)),
                "sm_max_mhz": float(self.max_sm), "power_w": round(float(np.median([r[2] for r in rows])), 1),
                "mem_mhz": float(np.median([r[4] for r in rows])), "temp_c": float(np.median([r[5] for r in rows])),
                "reasons": sorted(n for b, n in self.REASONS.items() if mask & b), "samples": len(rows)}


# ------------------------------------------------------------------------------- b200 impl ------
def pin_to_gpu_numa(gpu_index):
    """Bind this rank (and every thread it will start: client threads, batcher, completer, forwarder) to the CPUs NVML lists as
    local to its GPU (topo: GPUs 0-3 <-> CPUs 0-31,64-95, GPUs 4-7 <-> 32-63,96-127 on the 8-GPU box). Pinned staging memory is
    then allocated on the GPU's NUMA node and the PCIe path of the zero-copy gather / scatter does not cross sockets."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cpus = {64 * w + b for w, m in enumerate(words) for b in range(64) if (int(m) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"{len(cpus)} CPUs local to GPU {gpu_index}"
    except Exception as ex:  # never fatal
        return f"not pinned ({type(ex).__name__})"
    return "not pinned"


def workload_string(models_per_gpu, dims, replicas, pick_policy):
    """config.workload, identical for the b200 arm and the reference arm (same workload, two implementations)"""
    model_bytes = sum(dims[i] * dims[i + 1] * 4 + dims[i + 1] * 4 for i in range(len(dims) - 1))
    return (f"BASELINE configs[2] per-GPU shard: {models_per_gpu} per-tenant 3-layer MLP "
            f"({'x'.join(map(str, dims))} fp32, {model_bytes} B) per GPU, Zipf alpha=1.0, ring replicas={replicas} "
            f"(replica pick: {pick_policy}); at 8 GPUs = configs[2] (1000 models)")


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    return json.load(open(path)) if os.path.exists(path) else {}


def graph_model_speed(kind, steps=30):
    """extra.<kind>: device-resident speed of one BASELINE configs[1] / configs[3] model (synthetic weights, batch 8):
    tfsc_predict_device in a loop, CUDA events. Returns a small dict for the bench line."""
    import torch
    import tfservingcache_b200 as t
    if kind == "resnet50":
        man = t.modelformat.resnet50_manifest()
        rows, in_elems, out_elems, flop = 8, 224 * 224 * 3, 1000, 8.2e9
        x = torch.rand(rows, in_elems, device="cuda")
    else:
        man = t.modelformat.bert_manifest()
        rows, in_elems, out_elems, flop = 8, 128, 2, 22.4e9   # ~180 GFLOP per 8 x 128 request
        x = torch.randint(1, 30522, (rows, in_elems), device="cuda", dtype=torch.int32)
    y = torch.empty(rows, out_elems, device="cuda")
    cfg = {"modelProvider.type": "synthetic", "modelProvider.synthetic.template": "manifest",
           "modelProvider.synthetic.manifest": man, "modelProvider.synthetic.count": 2, "gpu.devices": [torch.cuda.current_device()],
           "gpu.arenaBytes": 2 << 30, "serving.maxConcurrentModels": 2, "modelCache.size": 4 << 30, "gpu.maxBatch": 8}
    stream = torch.cuda.Stream()
    with t.Server(cfg) as srv, torch.cuda.stream(stream):
        srv.ensure(0, "m0", 1)
        l0 = t._lib.lib.tfsc_kernel_launches()
        for _ in range(3):
            srv.predict_device(0, "m0", 1, x.data_ptr(), rows, y.data_ptr(), stream.cuda_stream)
        torch.cuda.synchronize()
        per_pass = (t._lib.lib.tfsc_kernel_launches() - l0) // 3
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            srv.predict_device(0, "m0", 1, x.data_ptr(), rows, y.data_ptr(), stream.cuda_stream)
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
    tfl = flop * rows / (ms * 1e-3) / 1e12
    peak = _peaks().get("bf16_tflops_sustained", 1405.4)
    return {"batch": rows, "ms_per_batch": round(ms, 3), "items_per_s": round(rows / (ms * 1e-3), 1), "tflops": round(tfl, 2),
            "frac_of_bf16_sustained": round(tfl / peak, 4), "launches_per_batch": int(per_pass), "weights_bytes": man["weights_bytes"],
            "note": "fp32 in/out, 3xTF32 tcgen05 GEMMs; device-resident inputs, one model, CUDA events"}


def _phase(rank, t0, name):
    """progress marker on stderr (rank 0): where the time of a run goes, and where a hang sits"""
    if rank == 0:
        print(f"[bench +{time.time() - t0:6.1f}s] {name}", file=sys.stderr, flush=True)


def run_b200(args):
    import torch
    import torch.distributed as dist
    t_start = time.time()

    import tfservingcache_b200 as t
    from tfservingcache_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    assert torch.cuda.is_available(), "bench.py needs a B200; the library has no CPU fallback"
    torch.cuda.set_device(local)
    cpus_total = effective_cpus()          # before the NUMA pinning narrows the affinity mask
    numa = pin_to_gpu_numa(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dims = args.dims or DIMS
    in_dim, out_dim = dims[0], dims[-1]
    inb, outb = in_dim * 4, out_dim * 4
    model_bytes = sum(dims[i] * dims[i + 1] * 4 + dims[i + 1] * 4 for i in range(len(dims) - 1))
    W, K = args.warmup, args.steps
    e2e_steps = args.e2e_steps or K
    n_steps_total = W + K + W + e2e_steps
    fwd_frac = args.forward_frac if world > 1 else 0.0
    wl = build_workload(world, args.models_per_gpu, args.tick, n_steps_total, pick_policy=args.replica_pick, forward_frac=fwd_frac)
    tick_global = args.tick * world

    free_b, _tot = torch.cuda.mem_get_info()
    arena = min(int(args.arena_gib * 2**30), int(free_b * 0.9))
    my_models = sorted({int(m) for m in np.unique(wl["trace"][wl["dest"] == rank])})
    host_gib = args.host_gib
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", world))
    if host_gib <= 0:
        avail_kb = 0
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable"):
                avail_kb = int(line.split()[1])
        host_gib = min(len(my_models) * model_bytes / 2**30 * 1.02 + 1, avail_kb / 2**20 * 0.7 / max(local_world, 1))
    cfg = {"modelProvider.type": "synthetic", "modelProvider.synthetic.dims": dims,
           "modelProvider.synthetic.count": wl["n_models"], "modelProvider.synthetic.namePrefix": "m",
           "modelProvider.synthetic.threads": max(1, min(32, cpus_total // max(local_world, 1))),
           "gpu.devices": [local], "gpu.arenaBytes": arena, "gpu.maxBatch": 64, "gpu.maxRequestRows": 4096,
           "gpu.stagingSlots": 4, "modelCache.size": int(host_gib * 2**30), "serving.maxConcurrentModels": 1 << 20,
           # routing is done above with the library's ring + picker over the GLOBAL member list (identical on every rank);
           # requests are handed to the cache tier of the chosen member (tfsc_predict_member / tfsc_predict_device)
           "proxy.replicasPerModel": wl["replicas"], "gpu.members": wl["members"], "gpu.localMembers": [wl["members"][rank]],
           "proxy.seed": 1, "proxy.replicaPick": "first"}
    win_slot = 128 << 10
    if world > 1:
        sock_dir = os.environ.get("TFSC_SOCK_DIR", f"/tmp/tfsc_fwd_{os.environ.get('MASTER_PORT', '0')}")
        os.makedirs(sock_dir, exist_ok=True)
        # window: [x rows | y rows] of one tick's forwarded requests in the value region; slots of 128 KB for the e2e region
        n_slots = max(512, (2 * args.tick * max(inb, outb) + win_slot - 1) // win_slot + 8)
        cfg.update({"cluster.rank": rank, "cluster.endpoints": [os.path.join(sock_dir, f"r{r}.sock") for r in range(world)],
                    "cluster.slotBytes": win_slot, "cluster.windowSlots": int(n_slots), "proxy.grpcTimeout": 60.0})
    _phase(rank, t_start, "workload built")
    srv = t.Server(cfg)

    # page every model this rank owns into HBM once (cold loads are not part of the steady-state metric;
    # with replicas=2 the owned set can exceed the arena and LRU paging continues inside the timed steps)
    t_load = time.time()
    for m in my_models:
        srv.ensure(0, f"m{m}", 1)
    load_s = time.time() - t_load
    _phase(rank, t_start, f"shard resident ({len(my_models)} models, {load_s:.1f} s)")

    # a dedicated non-default stream: handle 0 (the legacy default stream) means "the node's own compute
    # stream" to tfsc_predict_device, and the CUDA events below must sit on the stream the kernels run on
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    sptr = stream.cuda_stream
    assert sptr != 0
    max_rows = args.tick * 4
    x_dev = torch.randn(max_rows, in_dim, device="cuda", dtype=torch.float32,
                        generator=torch.Generator(device="cuda").manual_seed(0))   # same inputs in every run (--dump-outputs)
    y_dev = torch.empty(max_rows, out_dim, device="cuda", dtype=torch.float32)
    xb_dev = torch.empty(max_rows, in_dim, device="cuda", dtype=torch.float32)    # gathered batches (groups with forwarded rows)
    yb_dev = torch.empty(max_rows, out_dim, device="cuda", dtype=torch.float32)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # forward windows: mine holds the rows that ENTER here for other owners; the peers' windows are mapped (CUDA IPC)
    pwin = {}
    if world > 1:
        _r, my_win, my_win_bytes, _slot = srv.fwd_window()
        y_base = (my_win_bytes // 2) & ~255                     # value region layout: x rows from 0, y rows from y_base
        assert args.tick * inb <= y_base and args.tick * outb <= my_win_bytes - y_base
        _lib.check(_lib.lib.tfsc_device_memcpy(my_win, x_dev.data_ptr(), min(args.tick * inb, x_dev.numel() * 4)))
        barrier()
        for d in range(1, world):                 # ring schedule: at step d every rank dials a different peer
            p = (rank + d) % world
            pwin[p] = srv.fwd_peer_window(p)[0]
        barrier()
        _phase(rank, t_start, "peer windows mapped")

    # the request trace of every value-region step is grouped before the clock starts: the timed loop is route ->
    # ensure-resident -> gather -> predict launches -> scatter only, not numpy bookkeeping of the synthetic trace
    SegArr = _lib.TfscCopySeg
    plans = {}
    for s in range(W + K):
        groups = step_plan(wl, rank, s, tick_global)
        launches, gsegs, ssegs = [], [], []
        loff = boff = 0
        fwd_rows = 0
        fwd_idx = []   # rows of yb_dev that hold the results of forwarded requests
        for m, n_local, fl in groups:
            n = n_local + len(fl)
            if not fl:
                launches.append((f"m{m}".encode(), n, x_dev.data_ptr() + loff * inb, y_dev.data_ptr() + loff * outb))
                loff += n
                continue
            # a group with forwarded rows is assembled in one batch buffer (as the batcher does): local rows + peer rows
            xb, yb = xb_dev.data_ptr() + boff * inb, yb_dev.data_ptr() + boff * outb
            if n_local:
                gsegs.append((x_dev.data_ptr() + loff * inb, xb, n_local * inb))
                ssegs.append((yb, y_dev.data_ptr() + loff * outb, n_local * outb))
                loff += n_local
            for j, (p, k) in enumerate(fl):
                gsegs.append((pwin[p] + k * inb, xb + (n_local + j) * inb, inb))                      # NVLink read
                ssegs.append((yb + (n_local + j) * outb, pwin[p] + y_base + k * outb, outb))          # NVLink write
                fwd_idx.append(boff + n_local + j)
            launches.append((f"m{m}".encode(), n, xb, yb))
            boff += n
            fwd_rows += len(fl)
        ga = (SegArr * len(gsegs))(*[SegArr(a, b, c) for a, b, c in gsegs]) if gsegs else None
        sa = (SegArr * len(ssegs))(*[SegArr(a, b, c) for a, b, c in ssegs]) if ssegs else None
        plans[s] = dict(groups=[(m, nl + len(fl)) for m, nl, fl in groups], launches=launches, gather=ga, n_g=len(gsegs),
                        scatter=sa, n_s=len(ssegs), fwd_rows=fwd_rows, n_local=loff, fwd_idx=fwd_idx)
    lib = _lib.lib
    h = srv._h

    def device_step(step):
        p = plans[step]
        if p["n_g"]:
            _lib.check(lib.tfsc_k_copy_segments(p["gather"], p["n_g"], sptr))
        for name, rows, xp, yp in p["launches"]:
            lib.tfsc_model_ensure_async(h, 0, name, 1)      # route -> ensure-resident (all hits once the shard is resident)
            rc = lib.tfsc_predict_device(h, 0, name, 1, xp, rows, yp, sptr)
            if rc < 0:
                _lib.check(rc, "predict_device")
        if p["n_s"]:
            _lib.check(lib.tfsc_k_copy_segments(p["scatter"], p["n_s"], sptr))
        return p

    # ---- value: inputs resident in HBM ----------------------------------------------------------
    for s in range(W):
        device_step(s)
    barrier()
    # pre-heat: the W warm-up steps follow ~45 s of cold loads with an idle GPU; run real passes for --preheat-s more so
    # clocks, power state and the driver's launch path are in steady state when the clock starts (r1: N=1 varied 36-48 k)
    t_heat, i_heat = time.time(), 0
    while time.time() - t_heat < args.preheat_s:
        device_step(i_heat % max(W, 1))
        torch.cuda.synchronize()
        i_heat += 1
    barrier()
    flush.fill_(1)  # inputs (>= 1 GB of weights per launch) already exceed L2; flush once anyway
    sampler = ClockSampler(local, enabled=(local == 0 and "smi" in args.samplers))
    sampler.start()
    nvml = NvmlSampler(local, period_s=0.1)   # every rank watches its own GPU
    if "nvml" in args.samplers:
        nvml.start()
    launches0 = lib.tfsc_kernel_launches()
    st0 = srv.stats()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    alg_bytes, n_req, n_dense, fwd_rows_value = 0, 0, 0, 0
    t_host0 = time.perf_counter()
    t_wall0 = time.time()
    for s in range(W, W + K):
        p = device_step(s)
        b, l = algorithmic_bytes(p["groups"], dims)
        alg_bytes += b
        n_dense += l
        n_req += sum(r for _m, r in p["groups"])
        fwd_rows_value += p["fwd_rows"]
    ev1.record(stream)
    host_enqueue_ms = (time.perf_counter() - t_host0) * 1e3
    barrier()
    sampler.mark(t_wall0, time.time())
    nvml.mark(t_wall0, time.time())
    elapsed_ms = ev0.elapsed_time(ev1)
    my_elapsed_ms, my_req = elapsed_ms, n_req
    launches = lib.tfsc_kernel_launches() - launches0
    st1 = srv.stats()
    if args.dump_outputs:
        # the results of the last timed step as its callers receive them: the rows of the requests that entered here, then
        # those computed here for requests that entered at another rank (each request once over all ranks), in plan order
        last = plans[W + K - 1]
        y = torch.cat([y_dev[:last["n_local"]], yb_dev[torch.tensor(last["fwd_idx"], dtype=torch.long, device="cuda")]])
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "predict_y.npy" if world == 1 else f"predict_y_rank{rank}.npy"),
                sample_rows(y.cpu().numpy(), DUMP_MAX_BYTES // world))

    _phase(rank, t_start, "value region done")
    # ---- e2e: host buffers through the C ABI, closed-loop clients ----------------------------------------------
    lg = C.CDLL(os.path.join(ROOT, "tools", "libtfsc_loadgen.so"))
    lg.tfsc_loadgen_run.restype = C.c_int64
    names = b"".join(f"m{j}".encode().ljust(16, b"\0") for j in range(wl["n_models"]))
    n_inputs = 256
    inputs_h = torch.randn(n_inputs, in_dim).pin_memory()
    outputs_h = torch.empty(args.clients, out_dim).pin_memory()
    predict_ptr = C.cast(lib.tfsc_predict, C.c_void_p)
    member_ptr = C.cast(lib.tfsc_predict_member, C.c_void_p)

    def e2e_requests(step_lo, step_hi, trace=None):
        """requests that ENTER at this rank in the step range: (model ids, member = owner rank chosen by the front tier)"""
        lo, hi = step_lo * tick_global, step_hi * tick_global
        sel = wl["ingress"][lo:hi] == rank
        tr = (trace if trace is not None else wl["trace"])[lo:hi][sel]
        return tr.astype(np.int32), wl["dest"][lo:hi][sel].astype(np.int32)

    def e2e_run(req, mem, want_lat, clients=None):
        clients = clients or args.clients
        req, mem = np.ascontiguousarray(req), np.ascontiguousarray(mem)
        lat = np.zeros(max(1, len(req)), np.float32)
        el = C.c_double()
        failed = lg.tfsc_loadgen_run(predict_ptr, C.c_void_p(h), names, 16, b"1", req.ctypes.data_as(C.c_void_p),
                                     C.c_int64(len(req)), C.c_void_p(inputs_h.data_ptr()), C.c_int64(n_inputs), in_dim,
                                     C.c_void_p(outputs_h.data_ptr()), out_dim, clients,
                                     lat.ctypes.data_as(C.c_void_p) if want_lat else None, C.byref(el),
                                     member_ptr, mem.ctypes.data_as(C.c_void_p))
        return len(req), failed, el.value, lat[:len(req)]

    e0 = W + K
    if not args.skip_e2e:
        e2e_run(*e2e_requests(e0, e0 + W), False)
    barrier()
    ste0 = srv.stats()
    if args.skip_e2e:
        n_e2e, failed, el_s, lat = 0, 0, 1.0, np.zeros(1, np.float32)
    else:
        t_e0 = time.time()
        n_e2e, failed, el_s, lat = e2e_run(*e2e_requests(e0 + W, e0 + W + e2e_steps), True)
        sampler.mark(t_e0, time.time())
        nvml.mark(t_e0, time.time())
    torch.cuda.synchronize()
    barrier()
    ste1 = srv.stats()
    clocks = sampler.stop()
    my_nvml = nvml.stop()
    if my_nvml and (clocks.get("sm_mhz") is None or clocks.get("samples", 0) < 3):
        clocks.update({k: my_nvml[k] for k in ("sm_mhz", "sm_max_mhz", "reasons", "samples")})
        clocks["source"] = "nvml"
    if my_nvml:
        clocks["nvml"] = my_nvml

    def allsum(vals):
        if world == 1:
            return [float(v) for v in vals]
        tt = torch.tensor(vals, device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.SUM)
        return [float(v) for v in tt]

    def allmax(vals):
        if world == 1:
            return [float(v) for v in vals]
        tt = torch.tensor(vals, device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return [float(v) for v in tt]

    _phase(rank, t_start, "e2e region done")
    # ---- latency-bounded throughput: closed-loop client sweep (north_star: cache-hit p50 < 5 ms) -----------------
    sweep, light = [], None
    if not args.skip_e2e and not args.no_extras:
        req_all, mem_all = e2e_requests(e0 + W, e0 + W + e2e_steps)
        for c in (args.light_clients, 64, 128, 256, 512):
            if c <= 0 or c > args.clients:
                continue
            n_l = min(len(req_all), c * 40)
            barrier()
            _n, f_l, el_l, lat_l = e2e_run(req_all[:n_l], mem_all[:n_l], True, clients=c)
            qps_all, = allsum([n_l / el_l])
            p50_w, p99_w = allmax([float(np.percentile(lat_l, 50)) / 1e3, float(np.percentile(lat_l, 99)) / 1e3])
            sweep.append({"clients_per_gpu": c, "qps": round(qps_all, 1), "p50_ms": round(p50_w, 3), "p99_ms": round(p99_w, 3),
                          "failed": int(f_l)})
        if sweep:
            light = dict(sweep[0])
    ok = [p for p in sweep if p["p50_ms"] < 5.0]
    qps_at_p50_5ms = max(ok, key=lambda p: p["qps"]) if ok else None

    _phase(rank, t_start, "client sweep done")
    # ---- cache under pressure: resident cap below the working set, uniform storm (configs[4]) ---------------------
    pressure = None
    if not args.skip_e2e and not args.no_extras and len(my_models) > args.pressure_resident:
        from tools.traces import uniform_trace
        barrier()
        srv.set_max_resident(0, args.pressure_resident)
        n_p = 3 * args.tick      # per rank, whatever N is (the phase runs at PCIe speed: ~240 req/s per GPU)
        utrace = np.asarray(my_models, np.int64)[uniform_trace(len(my_models), n_p, seed=7 + rank)]   # this rank's own models
        sp0 = srv.stats()
        tp0 = time.time()
        _n, f_p, el_p, lat_p = e2e_run(utrace.astype(np.int32), np.full(n_p, rank, np.int32), True, clients=min(args.clients, 256))
        sp1 = srv.stats()
        srv.set_max_resident(0, 1 << 20)
        tot = max(1, sp1["cache_total"] - sp0["cache_total"])
        h2d = sp1["h2d_weight_bytes"] - sp0["h2d_weight_bytes"]
        qps_p, h2d_all = allsum([n_p / el_p, h2d / el_p / 1e9])
        p50_p, p99_p = allmax([float(np.percentile(lat_p, 50)) / 1e3, float(np.percentile(lat_p, 99)) / 1e3])
        pressure = {"trace": f"uniform over this rank's {len(my_models)} models, 256 clients per GPU", "resident_cap": args.pressure_resident,
                    "ideal_hit_pct": round(100.0 * args.pressure_resident / len(my_models), 1), "requests_per_gpu": int(n_p),
                    "qps": round(qps_p, 1), "hit_pct_rank0": round(100.0 * (sp1["cache_hits_total"] - sp0["cache_hits_total"]) / tot, 2),
                    "reloads_rank0": int(tot - (sp1["cache_hits_total"] - sp0["cache_hits_total"]) - (sp1["cache_misses_total"] - sp0["cache_misses_total"])),
                    "evictions_hbm_rank0": int(sp1["evictions_hbm"] - sp0["evictions_hbm"]),
                    "h2d_weight_GBps_all_gpus": round(h2d_all, 2), "h2d_weight_GBps_per_gpu": round(h2d_all / world, 2),
                    "pcie_roofline_GBps_per_gpu": 55.0, "load_stall_p50_ms": round(p50_p, 3), "load_stall_p99_ms": round(p99_p, 3),
                    "failed": int(f_p), "seconds": round(time.time() - tp0, 2)}
        # bring the shard back for anything that follows
        for m in my_models:
            srv.ensure_async(0, f"m{m}", 1)
        srv.sync(0)

    _phase(rank, t_start, "cache pressure phase done")
    per_rank = None
    fwd_out = ste1["fwd_out_requests"] - ste0["fwd_out_requests"]
    fwd_bytes = (ste1["fwd_peer_bytes_read"] - ste0["fwd_peer_bytes_read"]) + (ste1["fwd_peer_bytes_written"] - ste0["fwd_peer_bytes_written"])
    if world > 1:
        nv = my_nvml or {}
        rmask = sum(b for b, n in NvmlSampler.REASONS.items() if n in nv.get("reasons", []))
        diag = torch.tensor([my_elapsed_ms, host_enqueue_ms, my_req, n_dense, nv.get("sm_mhz", -1), nv.get("sm_min_mhz", -1),
                             nv.get("power_w", -1), rmask, n_e2e, el_s], device="cuda", dtype=torch.float64)
        allr = [torch.zeros_like(diag) for _ in range(world)]
        dist.all_gather(allr, diag)
        per_rank = [{"device_ms": round(float(v[0]), 2), "host_enqueue_ms": round(float(v[1]), 2), "requests": int(v[2]),
                     "launches": int(v[3]), "us_per_launch": round(float(v[0]) * 1e3 / max(1.0, float(v[3])), 2),
                     "sm_mhz": float(v[4]), "sm_min_mhz": float(v[5]), "power_w": float(v[6]),
                     "reasons": sorted(n for b, n in NvmlSampler.REASONS.items() if int(v[7]) & b),
                     "e2e_requests": int(v[8]), "e2e_s": round(float(v[9]), 3)} for v in allr]
    elapsed_ms, el_s = allmax([elapsed_ms, el_s])
    n_req_all, n_e2e_all, launches_all, alg_sum, failed_all, n_dense, fwd_rows_all, fwd_out_all, fwd_bytes_all = allsum(
        [n_req, n_e2e, launches, alg_bytes, failed, n_dense, fwd_rows_value, fwd_out, fwd_bytes])
    alg_bytes = alg_sum / world   # per-GPU average bytes over the max-over-ranks time

    peaks = _peaks()
    if "hbm_gbs" in peaks:
        peak, peak_src = peaks["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        peak, peak_src = 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"
    achieved = alg_bytes / (elapsed_ms * 1e-3) / 1e9  # this rank's dense launches are the whole timed region
    traffic = None
    tp = os.path.join(ROOT, "profiles", "dense_traffic.json")
    if os.path.exists(tp):
        traffic = json.load(open(tp)).get("dram_bytes_per_launch")

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_base = cpu_reference(args.cpu_sample, dims, warm=4)

    extra = None
    if rank == 0 and world == 1 and not args.no_extras and not args.skip_e2e:
        srv.close()
        srv = None
        extra = {}
        for kind in ("resnet50", "bert_base"):
            try:
                extra[kind] = graph_model_speed(kind)
            except Exception as ex:  # an extra line must never cost the headline
                extra[kind] = {"error": repr(ex)[:200]}

    roof = {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
            "traffic": traffic,
            "kernel": "dense_cluster_kernel<R> (<=8 rows, 2-CTA clusters, TMA ring, DSMEM K-fold, PDL) + dense_tc_kernel<RP> (9..64 rows, tcgen05 3xTF32, PDL): fused xW+b+ReLU",
            "peak_source": peak_src, "launches_timed": int(n_dense), "avg_launch_us": round(elapsed_ms * 1e3 * world / max(1, n_dense), 2),
            "note": "per-GPU average algorithmic bytes / max-over-ranks device time; gather / scatter launches of forwarded rows are inside the timed region"}
    workload = workload_string(args.models_per_gpu, dims, wl["replicas"], wl["pick_policy"])
    if rank == 0:
        value = n_req_all / (elapsed_ms * 1e-3)
        e2e_val = n_e2e_all / el_s
        line = {
            "metric": "predict_qps", "value": round(value, 1), "unit": "req/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": round(elapsed_ms / K, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload,
                       "models_total": wl["n_models"], "tick_requests_per_gpu": args.tick, "max_rows_per_pass": "8 (SIMT) / 64 (tcgen05 3xTF32)",
                       "l2": "inputs larger than L2 (>=1 GB of weights streamed per model pass); L2 flushed before timing",
                       "arena_gib": round(arena / 2**30, 1), "host_tier_gib": round(host_gib, 1), "cold_load_s": round(load_s, 1),
                       "preheat_s": args.preheat_s, "samplers": args.samplers, "cpu_affinity": numa},
            "e2e": {"value": round(e2e_val, 1), "unit": "req/s",
                    "h2d_bytes_per_step": int((ste1["h2d_input_bytes"] - ste0["h2d_input_bytes"] + ste1["h2d_weight_bytes"] - ste0["h2d_weight_bytes"]) / e2e_steps),
                    "d2h_bytes_per_step": int((ste1["d2h_output_bytes"] - ste0["d2h_output_bytes"]) / e2e_steps),
                    "transfer": "inputs: client memcpy into pinned staging, gather kernel reads it over PCIe; results: scatter kernel writes pinned staging (bytes counted per request row, rank 0)",
                    "clients_per_gpu": args.clients, "steps": e2e_steps, "failed": int(failed_all),
                    "p50_ms": round(float(np.percentile(lat, 50)) / 1e3, 3), "p99_ms": round(float(np.percentile(lat, 99)) / 1e3, 3),
                    "mean_batch_rows": round((ste1["batched_rows"] - ste0["batched_rows"]) / max(1, ste1["batches"] - ste0["batches"]), 2),
                    "light_load": light, "sweep": sweep,
                    "qps_at_p50_5ms": qps_at_p50_5ms},
            "hbm_cache_hit_pct": round(100.0 * (st1["cache_hits_total"] - st0["cache_hits_total"]) / max(1, st1["cache_total"] - st0["cache_total"]), 2),
            "gpu_launches": int(launches_all),
            "clocks": clocks,
            "roofline": roof,
        }
        if world > 1:
            line["forward"] = {"fraction": fwd_frac,
                               "value_region": {"forwarded_requests_per_step": round(fwd_rows_all / K, 1),
                                                "nvlink_bytes_per_step": int(fwd_rows_all * (inb + outb) / K)},
                               "e2e_region": {"forwarded_requests": int(fwd_out_all), "nvlink_bytes_per_step": int(fwd_bytes_all / e2e_steps),
                                              "mean_rtt_ms_rank0": round(1e3 * (ste1["fwd_rtt_seconds_sum"] - ste0["fwd_rtt_seconds_sum"]) / max(1, fwd_out), 3)},
                               "path": "ingress window (HBM, CUDA IPC) -> owner gather kernel over NVLink -> kernels -> scatter kernel over NVLink; control: unix socket"}
        if pressure:
            line["cache_pressure"] = pressure
        if extra:
            line["extra"] = extra
        if per_rank:
            line["per_rank"] = per_rank
        if cpu_base:
            line["cpu_baseline"] = cpu_base
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()    # nobody closes its window while a peer may still use it
    _phase(rank, t_start, "line printed, closing")
    if srv is not None:
        srv.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ---------------------------------------------------------------------------- reference arm ------
def cpu_reference(n_sample, dims, warm=4, steps=None):
    """The reference's path restated on the host CPU (oracle): ring lookup -> LRU + top-N residency
    (hit path) -> ONE unbatched fp32 forward per request (the reference never batches) with the
    oracle's multi-threaded C GEMV on all host cores -- the stand-in for CPU TF-Serving (absent)."""
    from oracle import cachemanager as ocm
    from oracle import models as omodels
    from oracle import ring as oring
    from oracle.lrucache import Model, ModelIdentifier
    from tools.traces import zipf_trace

    cores = min(effective_cpus(), 256)
    liborc = C.CDLL(os.path.join(ROOT, "oracle", "liboracle_ref.so"))
    n_models = MODELS_PER_GPU
    trace = zipf_trace(n_models, 4096, 1.0, 42)
    # bounded sample: the requests that touch the 12 most popular models of the trace
    top = [int(m) for m in np.argsort(-np.bincount(trace, minlength=n_models))[:12]]
    sample = [int(m) for m in trace if int(m) in top][: n_sample + warm]
    man = omodels.mlp_manifest(dims)

    I4 = C.c_int64 * len(dims)
    I3 = C.c_int64 * (len(dims) - 1)
    c_dims = I4(*dims)
    c_woff = I3(*[L["w_offset"] for L in man["layers"]])
    c_boff = I3(*[L["b_offset"] for L in man["layers"]])
    c_relu = (C.c_int * (len(dims) - 1))(*[1 if L["activation"] == "relu" else 0 for L in man["layers"]])
    liborc.oracle_mlp_forward_mt.restype = C.c_int

    def synth(j):
        blob = np.empty(man["weights_bytes"] // 4, np.float32)

        def fill(tid, off, n, scale):
            per = (n + 31) // 32
            ths = []
            for c in range(32):
                lo, hi = c * per, min(n, (c + 1) * per)
                if lo < hi:
                    th = threading.Thread(target=liborc.oracle_synth_fill, args=(
                        C.c_void_p(blob.ctypes.data + (off + lo) * 4), C.c_uint32(1000 + j), C.c_uint32(tid), C.c_uint64(lo),
                        C.c_uint64(hi - lo), C.c_float(scale)))
                    th.start()
                    ths.append(th)
            [th.join() for th in ths]
        for l, L in enumerate(man["layers"]):
            fill(2 * l, L["w_offset"] // 4, L["in"] * L["out"], omodels.weight_scale(L["in"]))
            fill(2 * l + 1, L["b_offset"] // 4, L["out"], omodels.BIAS_SCALE)
        return blob

    weights = {j: synth(j) for j in top}

    class Prov:
        def model_size(self, name, ver):
            return man["weights_bytes"]

        def load_model(self, name, ver):
            return Model(ModelIdentifier(name, ver), f"{name}/{ver}", man["weights_bytes"])

    cluster = oring.ClusterConnection(1)
    cluster.update([oring.ServingService("gpu0", 0, 0)])
    cm = ocm.CacheManager(Prov(), 1 << 50, 1 << 20)
    x = np.random.default_rng(0).standard_normal((1, dims[0])).astype(np.float32)
    y = np.empty((1, dims[-1]), np.float32)

    def one(j):
        oring.node_for_key(cluster, f"m{j}", "1", lambda n: 0)   # taskhandler.go:84-92
        cm.handle_model_request(f"m{j}", "1")                    # cachemanager.go:294-309 (hit path)
        rc = liborc.oracle_mlp_forward_mt(C.c_void_p(weights[j].ctypes.data), len(dims) - 1, c_dims, c_woff, c_boff, c_relu,
                                          C.c_void_p(x.ctypes.data), C.c_int64(1), C.c_void_p(y.ctypes.data), cores)
        assert rc == 0
        return y

    for j in sample[:warm]:
        one(j)
    t0 = time.perf_counter()
    for j in sample[warm:]:
        one(j)
    dt = time.perf_counter() - t0
    n = len(sample) - warm
    return {"value": round(n / dt, 2), "unit": "req/s", "cores": cores, "kind": "port",
            "sample": f"{n} unbatched requests (1 row each) of the Zipf trace restricted to its 12 most popular of {n_models} "
                      f"models, all cached+resident (hit path), oracle C fp32 split-K GEMV (AVX2) on {cores} threads; restated reference "
                      f"path (ring -> LRU -> forward), TF-Serving itself is not available",
            "seconds": round(dt, 2)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    dims = args.dims or DIMS
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # each "step" is a bounded sample of the workload; K steps + W warm-up end within minutes
    per_step = max(4, args.cpu_sample // 4)
    base = cpu_reference(per_step * args.steps, dims, warm=max(1, per_step * args.warmup // 4))
    line = {"impl": "reference", "metric": "predict_qps", "value": base["value"], "unit": "req/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * base["seconds"] / args.steps, 2),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(args.models_per_gpu, dims, min(2, world), args.replica_pick),
                       "reference_sample": f"CPU reference path, bounded sample of {per_step} requests per step; at N > 1 still ONE CPU "
                                           f"process on rank 0 (the reference's CPU path does not use the GPUs), ms_per_step = sample time / steps"},
            "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": base["value"], "unit": "req/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    import faulthandler
    faulthandler.enable()   # a native crash prints the Python stack it happened under
    # a hang leaves the stacks of all threads in stderr (driver limit per N: 870 s)
    faulthandler.dump_traceback_later(int(os.environ.get("TFSC_BENCH_DUMP_S", "600")), exit=False)
    a = parse_args()
    try:
        if a.impl == "reference":
            run_reference(a)
        else:
            run_b200(a)
    except BaseException:
        import traceback
        traceback.print_exc()
        sys.stderr.flush()
        os._exit(1)  # do not leave the other ranks waiting in a collective
