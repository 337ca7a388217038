#!/usr/bin/env python
"""bench.py -- column-iterations/s of the GLOM column update on N B200s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one batch: ``Glom.forward(img, iters=12)`` at BASELINE
configs[1] per GPU (dim=512 L=6 224/14, batch 32, bf16 tensor-core precision), i.e. 12 Jacobi column
updates of 32x256 columns x 6 levels = 589,824 column-iterations per GPU per step.  N > 1 shards the
batch (configs[2]: 32 images per GPU, no data-path collective) => weak scaling.

Regime (what the numbers mean): after the W warm-up steps the same forward runs back to back for
``--preheat-s`` seconds (default 2 s) so that the timed K steps see the SUSTAINED state of the part (1 kW power
cap, SM clock ~1.4-1.5 GHz), not a sub-second burst at 1.965 GHz.  The SM clock is measured on the device itself
(``glom_b200_clock_probe``: cycles per %globaltimer nanosecond) immediately before and after the timed region and
printed next to NVML's (lagging) reading; ``roofline.peak`` is the measured sustained cuBLAS rate when that clock is
in the sustained band and the burst rate otherwise, and both fractions are printed.

Printed (rank 0, ONE JSON line):
  value      whole-job column-iterations/s with the images already resident in HBM, device-timed
             (CUDA events on the launch stream, barrier + synchronize both sides, MAX over ranks)
  e2e        same metric through the public API with HOST buffers: pinned-host images -> H2D,
             forward, D2H of the returned state into pinned host memory, all inside the timed region
  roofline   dominant kernel: algorithmic FLOPs per launch / its average duration from CUDA events recorded
             around every launch in the timed region
  other_configs  BASELINE configs[3] (per-GPU shape) and configs[4] (3-frame continuation), and a training step
  cpu_baseline   the reference's own CPU forward on this box's host cores (bounded sample; rank 0, N = 1 only)

``--impl reference`` times the UNMODIFIED reference package (``$GLOM_REF_PATH`` -> ``oracle/_ref``; torch CPU, all
host threads) on the same shapes; if it is not importable on the box it times ``oracle/glom_oracle_torch.py`` (a
torch-CPU restatement pinned on the reference's golden outputs) and says so.

``--dump-outputs DIR`` writes, after the timed steps, what the last timed step returned (rank 0's shard) as
``DIR/levels.npy``: float32 ``(columns, levels, dim)`` for a fixed seeded sample of DUMP_COLUMNS (image, patch)
columns in (image, patch) order, or every column when the batch has no more (<= 50 MB).  Inputs and weights are
seeded, so two builds run with the same arguments can be compared output for output.

bench.py writes nothing into the tree: a library older than its sources is rebuilt into a temporary directory.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CFG = dict(dim=512, levels=6, image_size=224, patch_size=14)
CFG3 = dict(dim=1024, levels=8, image_size=384, patch_size=16)      # BASELINE configs[3], 8 images per GPU, 16 iters
ITERS = 12
BATCH_PER_GPU = 32
N_PATCH = (CFG["image_size"] // CFG["patch_size"]) ** 2
METRIC = "column-iterations/sec (BxNxLxiters) at dim=512 L=6 224/14"
UNIT = "column-iterations/s"
NOMINAL_FLOP_PER_CLK = 148 * 8192.0        # dense bf16: 4096 MAC/clk/SM x 148 SMs (2.25 PFLOP/s at ~1.86 GHz)
DUMP_COLUMNS = 4096                         # x levels x dim x 4 B = 50 MB at configs[1] (the full state is 100 MB)
DUMP_SEED = 0


def flops_per_col_iter(d, L, n, iters=None):
    """Tensor FLOPs per column-iteration: 16 d^2 (2L-1)/L + 4 n d   (SURVEY 8d).  With `iters`: the FLOPs the engine
    EXECUTES per column-iteration of a call of that many steps -- the first GEMM of MLP group 0 (bottom-up net of level 0,
    whose input, the tokens, does not change during a call) runs in the call's first step only: 8 d^2 / L per
    column-iteration less in the later steps.  Rooflines use the executed figure, never the larger algorithmic one."""
    f = 16.0 * d * d * (2 * L - 1) / L + 4.0 * n * d
    if iters:
        f -= 8.0 * d * d / L * (iters - 1) / iters
    return f


def bytes_per_iter(d, L, n, B, s_state=2, s_w=2):
    """Algorithmic HBM bytes per iteration (SURVEY 8d)."""
    return 2 * B * n * L * d * s_state + (2 * L - 1) * (8 * d * d + 5 * d) * s_w + B * n * d * 2 + n * d * 2


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            j = json.load(f)
        return dict(hbm_gbs=j["hbm_gbs"], sustained=j.get("bf16_tflops_sustained", j["bf16_tflops"]),
                    burst=j["bf16_tflops"], sm_max_mhz=j.get("sm_max_mhz", 1965.0),
                    sustained_mhz=(j.get("clocks_under_load") or {}).get("sm_mhz_median"),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, sustained=1400.0, burst=1590.0, sm_max_mhz=1965.0, sustained_mhz=1300.0,
                source="fallback (B200_PROFILING.md)")


# ------------------------------------------------------------------------------------ CPU arm
def cpu_model_name():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def find_reference():
    """The unmodified reference package, if importable on this box: (module, where) or (None, why)."""
    tried = []
    for cand in (os.environ.get("GLOM_REF_PATH"), os.path.join(ROOT, "oracle", "_ref")):
        if not cand or not os.path.isdir(os.path.join(cand, "glom_pytorch")):
            continue
        sys.path.insert(0, cand)
        try:
            import importlib
            mod = importlib.import_module("glom_pytorch")
            if os.path.realpath(os.path.dirname(mod.__file__)).startswith(os.path.realpath(cand)):
                return mod, cand
            tried.append(f"{cand}: shadowed by {mod.__file__}")
        except Exception as e:      # einops missing, ...
            tried.append(f"{cand}: {type(e).__name__}: {e}")
        finally:
            if sys.path and sys.path[0] == cand:
                sys.path.pop(0)
    return None, "; ".join(tried) or "no glom_pytorch package under $GLOM_REF_PATH or oracle/_ref"


class CpuArm:
    """The reference's CPU forward at configs[1] shapes (dim=512 L=6 224/14, fp32, no_grad), all host threads.
    kind = "reference": the unmodified package's ``Glom.forward``; kind = "port": the torch restatement in oracle/."""

    def __init__(self):
        import torch
        self.torch = torch
        mod, where = find_reference()
        torch.manual_seed(0)
        if mod is not None:
            self.kind, self.where = "reference", where
            self.model = mod.Glom(**CFG).eval()
            self.params = None
        else:
            from oracle import glom_oracle_torch as OT
            import glom_pytorch_b200 as G
            self.kind, self.where = "port", f"oracle/glom_oracle_torch.py ({where})"
            self.params = {k: v.detach() for k, v in G.Glom(**CFG).state_dict().items()}
            self.OT = OT
        self.threads = None

    def forward(self, img, iters):
        torch = self.torch
        with torch.no_grad():
            if self.kind == "reference":
                return self.model(img, iters=iters)
            return self.OT.glom_forward(self.params, img, patch_size=CFG["patch_size"], iters=iters)

    def images(self, batch):
        g = self.torch.Generator().manual_seed(1)
        return self.torch.randn(batch, 3, CFG["image_size"], CFG["image_size"], generator=g)

    def calibrate(self, budget_s):
        """Pick the thread count (all logical CPUs or half: SMT rarely helps oneDNN) and the largest batch in
        {1..32} whose 12-iteration forward is expected to take <= budget_s.  Returns (batch, est seconds)."""
        torch = self.torch
        ncpu = os.cpu_count() or 1
        try:
            ncpu = len(os.sched_getaffinity(0))
        except (AttributeError, OSError):
            pass
        x = self.images(2)
        best = None
        for nt in sorted({ncpu, max(1, ncpu // 2)}, reverse=True):
            torch.set_num_threads(nt)
            self.forward(x, 1)                                    # warm the thread pool / oneDNN primitives
            t0 = time.perf_counter()
            self.forward(x, 2)
            dt = time.perf_counter() - t0
            if best is None or dt < best[1]:
                best = (nt, dt)
        self.threads = best[0]
        torch.set_num_threads(self.threads)
        per_img_iter = best[1] / (2 * 2)
        batch = 1
        for b in (2, 4, 8, 16, 32):
            if per_img_iter * b * ITERS <= budget_s:
                batch = b
        return batch, per_img_iter * batch * ITERS

    def time(self, batch, iters, reps, warm=1):
        x = self.images(batch)
        for _ in range(warm):
            self.forward(x, iters)
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            self.forward(x, iters)
            ts.append(time.perf_counter() - t0)
        sec = statistics.median(ts)
        spread = (max(ts) - min(ts)) / sec if len(ts) > 1 else 0.0
        return batch * N_PATCH * CFG["levels"] * iters / sec, sec, spread

    def describe(self, batch, iters, reps, sec, spread):
        what = ("unmodified reference glom_pytorch.Glom.forward from " + self.where) if self.kind == "reference" \
            else ("torch-CPU restatement " + self.where)
        return (f"{what}; torch {self.torch.__version__} CPU fp32 no_grad, {self.threads} threads; dim=512 L=6 224/14 "
                f"batch={batch} iters={iters}; median of {reps} reps after warm-up, {sec:.2f} s each, "
                f"(max-min)/median {spread:.2f}")


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    arm = CpuArm()
    steps = max(1, args.steps)
    # a step = one forward of a bounded sample of configs[1]: all 12 iterations, as many of the 32 images as keep
    # warm-up + K steps within a few minutes on this host
    batch, _ = arm.calibrate(budget_s=min(6.0, 150.0 / (steps + max(1, args.warmup))))
    v, sec, spread = arm.time(batch, ITERS, steps, warm=max(1, min(args.warmup, 2)))
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"BASELINE configs[1] shapes: dim=512 L=6 224/14 iters={ITERS}; CPU sample batch={batch} "
                               f"of 32 per step (the metric is per column-iteration)",
                   "batch": batch, "iters": ITERS},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": arm.threads, "kind": arm.kind, "cpu": cpu_model_name(),
                         "logical_cpus": os.cpu_count(), "sample": arm.describe(batch, ITERS, steps, sec, spread)},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------ host placement
def bind_to_gpu_numa(local_rank):
    """Pin this process (and the threads / pinned allocations it creates afterwards) to the CPUs local to its GPU
    (sysfs local_cpulist of the GPU's PCI function).  Returns a short record for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        idx = local_rank
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                idx = int(vis.split(",")[local_rank])
            except (ValueError, IndexError):
                idx = local_rank
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        with open(f"/sys/bus/pci/devices/{bus}/local_cpulist") as f:
            cpulist = f.read().strip()
        cpus = set()
        for part in cpulist.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        allowed = cpus & os.sched_getaffinity(0)
        if not allowed:
            return {"bound": False, "why": "local cpulist outside the allowed set", "local_cpulist": cpulist}
        os.sched_setaffinity(0, allowed)
        node = None
        try:
            with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
                node = int(f.read().strip())
        except (OSError, ValueError):
            pass
        return {"bound": True, "local_cpulist": cpulist, "numa_node": node, "cpus": len(allowed)}
    except Exception as e:
        return {"bound": False, "why": f"{type(e).__name__}: {e}"}


# ------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples SM clock, power and throttle reasons DURING the timed region: an NVML polling thread (every
    ~5 ms); falls back to `nvidia-smi -lms` if pynvml is unavailable.  NVML's clock / power readings lag the device by
    up to a second -- the device-side probe (see device_clock_mhz) is the authoritative clock."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.thread = None
        self.samples = []
        self._stop = False
        self.max_mhz = None

    def _poll(self):
        import pynvml
        h = self.handle
        while not self._stop:
            try:
                sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                pw = pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0
                rs = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(
                    pynvml, "nvmlDeviceGetCurrentClocksEventReasons") else pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.samples.append((sm, pw, rs))
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        try:
            import threading
            import pynvml
            pynvml.nvmlInit()
            idx = self.gpu
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                try:
                    idx = int(vis.split(",")[self.gpu])
                except (ValueError, IndexError):
                    idx = self.gpu
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.thread is not None:
            import pynvml
            self._stop = True
            self.thread.join(timeout=2)
            if not self.samples:
                return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["no samples"]}
            bits = {"hw_slowdown": getattr(pynvml, "nvmlClocksEventReasonHwSlowdown", 0x8),
                    "hw_thermal_slowdown": getattr(pynvml, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                    "sw_thermal_slowdown": getattr(pynvml, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                    "sw_power_cap": getattr(pynvml, "nvmlClocksEventReasonSwPowerCap", 0x4)}
            pmax = max(p for _, p, _ in self.samples)
            load = [s for s in self.samples if s[1] > 0.5 * pmax] or self.samples
            reasons = sorted(k for k, b in bits.items() if any(s[2] & b for s in load))
            return {"sm_mhz": statistics.median(s[0] for s in load), "sm_max_mhz": self.max_mhz,
                    "power_w_max": pmax, "power_w_median_under_load": statistics.median(s[1] for s in load),
                    "samples": len(self.samples), "samples_under_load": len(load), "reasons": reasons,
                    "how": "NVML polled every ~5 ms during the timed region"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        load = [s for s, p in zip(sm, power) if p > 0.5 * max(power)] or sm
        return {"sm_mhz": statistics.median(load), "sm_max_mhz": max(mx), "power_w_max": max(power),
                "samples": len(sm), "reasons": sorted(reasons), "how": "nvidia-smi -lms 100"}


# ------------------------------------------------------------------------------------ ours
def sample_columns(levels):
    """(B, n, L, d) -> (k, L, d): the fixed seeded sample of --dump-outputs, gathered on the device."""
    import torch
    cols = levels.reshape(-1, levels.shape[-2], levels.shape[-1])
    if cols.shape[0] > DUMP_COLUMNS:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(cols.shape[0], DUMP_COLUMNS, replace=False))
        cols = cols.index_select(0, torch.from_numpy(idx).to(cols.device))
    return cols.float()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch-per-gpu", type=int, default=BATCH_PER_GPU)
    ap.add_argument("--iters", type=int, default=ITERS)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--preheat-s", type=float, default=2.0,
                    help="seconds of back-to-back forwards before the timed region (sustained power / clock state)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true", help="skip configs[3] / configs[4] / training extras")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--train", action="store_true", help="(kept for compatibility: the training step is timed by default)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned to DIR/levels.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    try:
        orig_affinity = os.sched_getaffinity(0)
    except (AttributeError, OSError):
        orig_affinity = None
    numa = bind_to_gpu_numa(local_rank)       # before torch creates threads / pinned buffers
    import torch
    import torch.distributed as dist
    from glom_pytorch_b200 import _native
    from glom_pytorch_b200.build import build_library, is_stale
    if "GLOM_B200_LIB" not in os.environ and is_stale():
        # time the current sources, but build them outside the tree (which may be read-only)
        import atexit
        import shutil
        import tempfile
        tmp = tempfile.mkdtemp(prefix="glom_b200_bench_")
        atexit.register(shutil.rmtree, tmp, True)
        _native.LIB_PATH = build_library(out_dir=tmp)
    distributed = world > 1
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29511")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
        dist.barrier(device_ids=[local_rank])
    import glom_pytorch_b200 as G
    from glom_pytorch_b200.sharding import shard_range

    if args.warmup < 3:
        args.warmup = 3          # timing rule: at least 3 warm-up steps
    B, T = args.batch_per_gpu, args.iters
    d, L = CFG["dim"], CFG["levels"]
    global_batch = B * world
    s, e = shard_range(global_batch, rank, world)
    assert e - s == B

    torch.manual_seed(0)                                    # identical default init on every rank ...
    model = G.Glom(**CFG, precision=args.precision).to(dev).eval()
    if distributed:                                         # ... and rank 0's weights broadcast over NCCL anyway
        for prm in model.parameters():
            dist.broadcast(prm.data, src=0)

    # synthetic images: 4 rotating pinned host buffers (global batch generated per seed, this rank's shard)
    NBUF = 4
    host_imgs, dev_imgs = [], []
    for i in range(NBUF):
        g = torch.Generator().manual_seed(1 + i)
        full = torch.randn(global_batch, 3, CFG["image_size"], CFG["image_size"], generator=g)
        host_imgs.append(full[s:e].contiguous().pin_memory())
        dev_imgs.append(host_imgs[-1].to(dev))
    host_out = torch.empty(B, N_PATCH, L, d, dtype=torch.float32).pin_memory()
    stream = torch.cuda.current_stream(dev)
    probe_buf = torch.zeros(8, dtype=torch.int64, device=dev)

    def barrier():
        if distributed:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize(dev)

    def enqueue_clock_probe(slot):
        _native.clock_probe(probe_buf.data_ptr() + 16 * slot, 150, stream.cuda_stream)

    def preheat(fn, seconds):
        """Run fn() back to back for `seconds` of device time (checked every 8 calls)."""
        if seconds <= 0:
            return 0
        n = 0
        t0 = time.perf_counter()
        while True:
            for _ in range(8):
                fn()
                n += 1
            torch.cuda.synchronize(dev)
            if time.perf_counter() - t0 >= seconds:
                return n

    launches = 0
    with torch.no_grad():
        # -------- device-resident throughput (value) + per-kernel events (roofline), same timed region
        for i in range(args.warmup):
            model(dev_imgs[i % NBUF], iters=T)
        barrier()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        preheat_steps = preheat(lambda: model(dev_imgs[0], iters=T), args.preheat_s)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if distributed:
            dist.barrier(device_ids=[local_rank])
        enqueue_clock_probe(0)
        torch.cuda.synchronize(dev)
        _native.kernel_clocks(reset=True)        # in-kernel (clock64, %globaltimer) samples of the timed region only
        ev0.record(stream)
        for i in range(args.steps):
            last = None                          # free the previous result first: the allocator reuses one output block
            last = model(dev_imgs[i % NBUF], iters=T)
            launches += model.last_launches
        ev1.record(stream)
        enqueue_clock_probe(1)
        barrier()
        ms_dev = ev0.elapsed_time(ev1)
        kernel_clk = _native.kernel_clocks(reset=True)
        dump = sample_columns(last) if args.dump_outputs and rank == 0 else None   # stays on the device until the end
        del last
        # -------- the same K steps again, back to back, with CUDA events around EVERY kernel launch (library hook):
        # per-kernel durations for the roofline.  Kept out of the region above because an event between two kernels
        # disables their programmatic (PDL) overlap and costs ~1 us each: the instrumented pass is a few % slower.
        _native.profile_begin()
        ep0, ep1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ep0.record(stream)
        for i in range(args.steps):
            model(dev_imgs[i % NBUF], iters=T)
        ep1.record(stream)
        enqueue_clock_probe(2)
        barrier()
        ms_prof = ep0.elapsed_time(ep1)
        prof = _native.profile_end()
        clocks = sampler.stop() if rank == 0 else None
        pb = probe_buf.cpu().tolist()
        dev_mhz = [1e3 * pb[2 * k] / pb[2 * k + 1] if pb[2 * k + 1] else None for k in range(3)]

        # -------- PCIe bandwidth of the buffers the e2e loop moves (attribution of e2e - value)
        def copy_gbs(dst, src, reps=3):
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            dst.copy_(src, non_blocking=True)
            torch.cuda.synchronize(dev)
            c0.record(stream)
            for _ in range(reps):
                dst.copy_(src, non_blocking=True)
            c1.record(stream)
            torch.cuda.synchronize(dev)
            return src.numel() * src.element_size() * reps / (c0.elapsed_time(c1) * 1e-3) / 1e9
        dev_out_probe = torch.empty(B, N_PATCH, L, d, dtype=torch.float32, device=dev)
        pcie = {"h2d_gbs": copy_gbs(dev_imgs[0], host_imgs[0]), "d2h_gbs": copy_gbs(host_out, dev_out_probe)}
        del dev_out_probe

        # -------- end to end through the public API with host buffers: every step copies its images from pinned
        # host memory and its result back to pinned host memory inside the timed region.  Copies run on extra
        # streams (one per direction), double-buffered, so step i's D2H and step i+2's H2D overlap step i+1's compute.
        h2d_stream, d2h_stream = torch.cuda.Stream(dev), torch.cuda.Stream(dev)   # one per copy engine / PCIe direction
        d2h_stream2 = torch.cuda.Stream(dev)           # the 100 MB result goes back as two halves on two DMA queues
        host_outs = [host_out, torch.empty_like(host_out).pin_memory()]

        def e2e_loop(nsteps):
            staged = None
            ready = torch.cuda.Event()
            with torch.cuda.stream(h2d_stream):
                staged = host_imgs[0].to(dev, non_blocking=True)
                ready.record(h2d_stream)
            for i in range(nsteps):
                stream.wait_event(ready)                       # this step's images are on the device
                x = staged
                if i + 1 < nsteps:                             # prefetch the next step's images
                    nxt_ready = torch.cuda.Event()
                    with torch.cuda.stream(h2d_stream):
                        staged = host_imgs[(i + 1) % NBUF].to(dev, non_blocking=True)
                        nxt_ready.record(h2d_stream)
                out = model(x, iters=T)                        # public API call on the compute stream
                done = torch.cuda.Event()
                done.record(stream)
                x.record_stream(stream)
                half = (out.shape[0] + 1) // 2
                for q, (lo, hi) in ((d2h_stream, (0, half)), (d2h_stream2, (half, out.shape[0]))):
                    if lo >= hi:
                        continue
                    with torch.cuda.stream(q):                 # result back to the host
                        q.wait_event(done)
                        host_outs[i % 2][lo:hi].copy_(out[lo:hi], non_blocking=True)
                        out.record_stream(q)
                if i + 1 < nsteps:
                    ready = nxt_ready
            stream.wait_stream(d2h_stream)                     # the last D2H is inside the timed region
            stream.wait_stream(d2h_stream2)

        e2e_loop(max(4, args.warmup))                   # allocator and copy queues reach their steady state
        e2e_attempts = []
        for attempt in range(2):
            barrier()
            ee0, ee1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ee0.record(stream)
            e2e_loop(args.steps)
            ee1.record(stream)
            barrier()
            e2e_attempts.append(ee0.elapsed_time(ee1))
            # the copies hide behind the compute (PCIe needs ~2.1 of the ~5.7 ms): an end-to-end pass far above the
            # device-resident one is a host / PCIe hiccup (seen once on a fresh box: 18 ms per step) -> re-measured ONCE,
            # both attempts are reported
            if e2e_attempts[-1] <= 1.15 * ms_dev:
                break
        ms_e2e = min(e2e_attempts)

    # -------- the other BASELINE configs on this GPU (same sustained state; short: the box is already hot)
    other = {}
    peaks = measured_peaks()
    if not args.no_other_configs and args.precision == "bf16":
        def timed(fn, reps, warm=3):
            with torch.no_grad():
                for _ in range(warm):
                    fn()
                barrier()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                for _ in range(reps):
                    fn()
                b.record(stream)
                barrier()
            return a.elapsed_time(b) / reps

        def entry(ms, col_iters, fci, what):
            tf = fci * col_iters / (ms * 1e-3) / 1e12
            return {"workload": what, "ms_per_step": ms, "value": col_iters * world / (ms * 1e-3), "unit": UNIT,
                    "tflops_per_gpu": tf, "frac_sustained": tf / peaks["sustained"], "frac_burst": tf / peaks["burst"]}
        # configs[4]: 3-frame continuation 12 -> 10 -> 6 with the state carried (README.md:105-111), incl. tokeniser
        # (the carried tensor is the one the previous call returned, so the engine resumes from the shadows it still
        # holds -- glom_b200_forward_resume -- and each next frame is tokenised on a side stream while the current one runs)
        def chain():
            lv = model(dev_imgs[0], iters=12)
            model.stage_tokens(dev_imgs[1])
            lv = model(dev_imgs[1], iters=10, levels=lv)
            model.stage_tokens(dev_imgs[2])
            return model(dev_imgs[2], iters=6, levels=lv)
        ms4 = timed(chain, max(3, args.steps // 8))
        other["configs[4]"] = entry(ms4, B * N_PATCH * L * 28, flops_per_col_iter(d, L, N_PATCH, 28.0 / 3),
                                    f"3-frame continuation iters 12->10->6, batch={B}/GPU, three forward calls incl. tokeniser")
        ms_ra = timed(lambda: model(dev_imgs[0], iters=T, return_all=True), max(3, args.steps // 8))
        other["configs[1] return_all"] = entry(ms_ra, B * N_PATCH * L * T, flops_per_col_iter(d, L, N_PATCH, T),
                                               f"configs[1] with return_all=True ({T + 1} slabs written)")
        # configs[3]: dim=1024 L=8 384/16 iters=16, 8 images per GPU
        torch.manual_seed(0)
        m3 = G.Glom(**CFG3, precision="bf16").to(dev).eval()
        n3 = (CFG3["image_size"] // CFG3["patch_size"]) ** 2
        img3 = torch.randn(8, 3, CFG3["image_size"], CFG3["image_size"], generator=torch.Generator().manual_seed(5)).to(dev)
        ms3 = timed(lambda: m3(img3, iters=16), max(3, args.steps // 8))
        other["configs[3]"] = entry(ms3, 8 * n3 * CFG3["levels"] * 16, flops_per_col_iter(CFG3["dim"], CFG3["levels"], n3, 16),
                                    "dim=1024 L=8 384/16 iters=16, batch=8/GPU (the 8-GPU config's per-GPU shard)")
        del m3, img3
        torch.cuda.empty_cache()

    train = None
    if not args.no_train and not args.no_other_configs and args.precision == "bf16":
        from glom_pytorch_b200.dp import allreduce_gradients
        model.train()
        tt = 7 if T >= 7 else T
        group = dist.group.WORLD if distributed else None

        def train_step(img):
            model.zero_grad(set_to_none=True)
            loss = model(img, iters=T, return_all=True)[tt, :, :, -1].square().mean()
            loss.backward()
            if distributed:
                allreduce_gradients(model, group)
        for _ in range(2):
            train_step(dev_imgs[0])
        barrier()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        nrep = max(3, args.steps // 8)
        f_ms = b_ms = c_ms = 0.0
        for i in range(nrep):
            model.zero_grad(set_to_none=True)
            ev[0].record(stream)
            loss = model(dev_imgs[i % NBUF], iters=T, return_all=True)[tt, :, :, -1].square().mean()
            ev[1].record(stream)
            loss.backward()
            ev[2].record(stream)
            if distributed:
                allreduce_gradients(model, group)
            ev[3].record(stream)
            torch.cuda.synchronize(dev)
            f_ms += ev[0].elapsed_time(ev[1]); b_ms += ev[1].elapsed_time(ev[2]); c_ms += ev[2].elapsed_time(ev[3])
        tms = torch.tensor([(f_ms + b_ms + c_ms) / nrep], device=dev, dtype=torch.float64)
        if distributed:
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        train = {"forward_ms": f_ms / nrep, "backward_ms": b_ms / nrep, "grad_allreduce_ms": c_ms / nrep, "reps": nrep,
                 "step_ms_max_over_ranks": tms.item(),
                 "value": global_batch * N_PATCH * L * T / (tms.item() * 1e-3),
                 "unit": "column-iterations/s (fwd+bwd" + ("+NCCL gradient all-reduce)" if distributed else ")"),
                 "loss": f"mean(all_levels[{tt}, :, :, -1] ** 2)", "peak_mem_gib": torch.cuda.max_memory_allocated(dev) / 2 ** 30}
        model.eval()

    if distributed:
        t = torch.tensor([ms_dev, ms_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_dev, ms_e2e = t.tolist()
        mh = torch.tensor([m or 0.0 for m in dev_mhz], device=dev, dtype=torch.float64)
        mh_min = mh.clone()
        dist.all_reduce(mh_min, op=dist.ReduceOp.MIN)
        dev_mhz_min = mh_min.tolist()
    else:
        dev_mhz_min = dev_mhz

    col_iters_step = global_batch * N_PATCH * L * T
    value = col_iters_step * args.steps / (ms_dev * 1e-3)
    e2e_value = col_iters_step * args.steps / (ms_e2e * 1e-3)

    if rank == 0:
        rows = B * N_PATCH
        G_ = 2 * L - 1
        kern = {}
        # executed FLOPs per launch, averaged over the T launches of a call: MLP group 0 runs in the first step only
        merged_env = os.environ.get("GLOM_B200_MERGED_MLP", "0") == "1"
        reuse_g0 = os.environ.get("GLOM_B200_REUSE_BU0", "1") != "0" and not merged_env
        g1 = (G_ - (T - 1) / T) if (reuse_g0 and T > 0) else G_
        flops = {"gemm1_gelu": 2.0 * rows * 4 * d * d * g1,
                 "gemm2_combine": 2.0 * rows * d * (8 * d * (L - 1) + 4 * d),
                 "attention": 4.0 * N_PATCH * N_PATCH * d * B * L}
        flops["mlp_fused"] = 2.0 * rows * 4 * d * d * G_ + flops["gemm2_combine"]
        algo_bytes = {"gemm1_gelu": rows * d * 2 * g1 + g1 * 4 * d * d * 2 + rows * g1 * 4 * d * 2,
                      "gemm2_combine": rows * G_ * 4 * d * 2 + L * d * 8 * d * 2 + rows * L * d * (4 + 2 + 4 + 2 + 2),
                      # fused MLP kernel: state shadows + tokens in, weights once, fp32 state in/out, C in, shadows out
                      "mlp_fused": rows * d * 2 * G_ + (G_ * 4 * d * d + L * d * 8 * d) * 2 + rows * L * d * (4 + 2 + 4 + 2 + 2)}
        for k, (ms, cnt) in prof.items():
            if cnt:
                kern[k] = {"launches": cnt, "avg_us": ms / cnt * 1e3, "ms_per_step": ms / args.steps}
                if k in flops and args.precision == "bf16":
                    kern[k]["tflops"] = flops[k] / (ms / cnt * 1e-3) / 1e12
        cand = [k for k in ("mlp_fused", "gemm1_gelu", "gemm2_combine") if k in kern]
        dom = max(cand, key=lambda k: kern[k]["ms_per_step"]) if cand else "gemm1_gelu"
        names = {"mlp_fused": "mlp_kernel (persistent grouped GEMM1+GELU -> GEMM2+combine tiles, tcgen05, H kept in L2)",
                 "gemm1_gelu": "gemm_kernel<0,256> (grouped GEMM1 + bias + exact-erf GELU, tcgen05)",
                 "gemm2_combine": "gemm_kernel<1,256> (grouped GEMM2 + 4-way combine, tcgen05)"}
        traffic = None
        try:   # per-launch DRAM bytes of the dominant kernel from the committed ncu --set full capture
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                traffic = json.load(f)["kernels"][dom]["dram_bytes"] if args.batch_per_gpu == BATCH_PER_GPU else None
        except (OSError, KeyError, ValueError):
            traffic = None
        # regime: the device-side clock decides which measured peak is the denominator
        mhz = [m for m in dev_mhz_min[:2] if m]
        clk = sum(mhz) / len(mhz) if mhz else None
        band = 0.85 * peaks["sm_max_mhz"]
        regime = "unknown" if clk is None else ("sustained" if clk < band else "burst")
        peak = peaks["burst"] if regime == "burst" else peaks["sustained"]
        ach = kern.get(dom, {}).get("tflops")
        whole_tf = flops_per_col_iter(d, L, N_PATCH, T) * col_iters_step / world / (ms_dev / args.steps * 1e-3) / 1e12
        roof = {"bound": "tensor", "kernel": names.get(dom, dom), "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                "frac": (ach / peak) if ach else None,
                "frac_of_sustained_peak": (ach / peaks["sustained"]) if ach else None,
                "frac_of_burst_peak": (ach / peaks["burst"]) if ach else None,
                "frac_of_clock_scaled_nominal": (ach * 1e12 / (NOMINAL_FLOP_PER_CLK * clk * 1e6)) if (ach and clk) else None,
                "regime": regime,
                "regime_rule": f"device SM clock {clk:.0f} MHz {'<' if regime == 'sustained' else '>='} 0.85 x {peaks['sm_max_mhz']:.0f} "
                               f"-> peak = bf16_tflops{'_sustained' if regime != 'burst' else ''}" if clk else "no device clock",
                "peaks": {"sustained": peaks["sustained"], "burst": peaks["burst"], "hbm_gbs": peaks["hbm_gbs"],
                          "sustained_measured_at_mhz": peaks["sustained_mhz"], "source": peaks["source"]},
                "traffic": traffic, "traffic_source": "profiles/traffic.json (ncu --set full, dram__bytes_read+write)",
                "algorithmic_bytes": algo_bytes.get(dom),
                "flops_per_launch": flops.get(dom),
                "whole_step": {"tflops": whole_tf,
                               "hbm_gbs_algorithmic": bytes_per_iter(d, L, N_PATCH, B) * T /
                               (ms_dev / args.steps * 1e-3) / 1e9,
                               "frac_tensor": whole_tf / peak, "frac_of_sustained_peak": whole_tf / peaks["sustained"],
                               "frac_of_burst_peak": whole_tf / peaks["burst"]},
                "instrumented_ms_per_step": ms_prof / args.steps,
                "how": "per-kernel CUDA events (library hook) over a second pass of the same K steps right after the timed "
                       "region, same sustained state; `value` / `ms_per_step` come from the un-instrumented pass",
                "kernels": kern}
        roof["whole_step"]["frac_hbm"] = roof["whole_step"]["hbm_gbs_algorithmic"] / peaks["hbm_gbs"]
        if traffic and kern.get(dom):
            # the dominant kernel's HBM side: its arithmetic intensity sits at the ridge of the measured peaks, and the
            # in-kernel counters show it waiting for operands, so both rooflines are printed
            gbs = traffic / (kern[dom]["avg_us"] * 1e-6) / 1e9
            roof["hbm"] = {"achieved_gbs": gbs, "peak_gbs": peaks["hbm_gbs"], "frac": gbs / peaks["hbm_gbs"],
                           "dram_bytes_per_launch": traffic,
                           "flop_per_dram_byte": (flops.get(dom) or 0) / traffic,
                           "ridge_flop_per_byte": peak * 1e12 / (peaks["hbm_gbs"] * 1e9),
                           "read_write_ceiling_gbs": 3200.0,
                           "read_write_ceiling_source": "profiles/r2_dram_pattern_probe.txt: a kernel that only reads and "
                                                        "writes a tensor with the GEMM2 epilogue's access pattern, one "
                                                        "512-thread CTA per SM (copy bandwidth: MEASURED_PEAKS.json)"}
        if clocks is not None:
            # the SM clock INSIDE the tensor-core kernels of the un-instrumented timed region (rank 0): cycles and
            # %globaltimer ns bracketing each kernel's working phase, summed per kernel kind
            clocks["in_kernel_sm_mhz"] = {k: round(v[0], 1) for k, v in kernel_clk.items()}
            clocks["in_kernel_ms_per_step"] = {k: v[1] / args.steps for k, v in kernel_clk.items()}
            clocks["block0_wait_fractions"] = {k: dict(zip(("mma_lane_waits_operands", "mma_lane_waits_accumulator",
                                                            "tma_lane_waits_slot", "epilogue_warp0_waits_accumulator",
                                                            "epilogue_warp0_busy", "consensus_output_work"), v[2]))
                                               for k, v in kernel_clk.items() if any(v[2])}
            clocks["device_sm_mhz_before"] = dev_mhz_min[0]
            clocks["device_sm_mhz_after"] = dev_mhz_min[1]
            clocks["device_sm_mhz_after_instrumented_pass"] = dev_mhz_min[2]
            clocks["device_how"] = ("glom_b200_clock_probe: clock64 cycles per %globaltimer ns over 150 us, one thread, "
                                    "enqueued right before / after the timed region (min over ranks)")
            clocks["preheat_s"] = args.preheat_s
            clocks["preheat_steps"] = preheat_steps
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "f32",
            "data": "synthetic",
            "images_per_s": global_batch * args.steps / (ms_dev * 1e-3),
            "config": {"workload": f"BASELINE configs[{1 if world == 1 else 2}]: dim=512 L=6 224/14 iters={T} "
                                   f"batch={B}/GPU (global {global_batch}), Glom.forward incl. tokeniser",
                       "global_batch": global_batch, "iters": T, "parallelism": f"dp{world} (batch shards, no collective)",
                       "regime": f"{args.preheat_s:g} s of back-to-back forwards before the timed region (sustained power state)",
                       "l2": "per-step working set ~1 GB (state 100 MB fp32 + shadows, H 369 MB, weights 46 MB) "
                             "> 126 MB L2; input images rotate over 4 buffers; no explicit flush"},
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": host_imgs[0].numel() * 4 * world,
                    "d2h_bytes_per_step": host_out.numel() * 4 * world,
                    "attempts_ms_per_step": [a / args.steps for a in e2e_attempts],
                    "pcie": pcie, "host_numa": numa},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": roof,
        }
        if other:
            line["other_configs"] = other
        if train is not None:
            line["train"] = train
        if dump is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "levels.npy"), dump.cpu().numpy())
        if world == 1 and not args.no_cpu_baseline:
            # the reference arm's own code path, in a child process with the ORIGINAL CPU affinity (this process and
            # its thread pools are pinned to the GPU's NUMA node), on a bounded sample: 3 timed forwards
            def unbind():
                if orig_affinity:
                    os.sched_setaffinity(0, orig_affinity)
            try:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "3",
                                    "--warmup", "1"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                                   timeout=600, preexec_fn=unbind)
                ref_line = json.loads(r.stdout.strip().splitlines()[-1])
                line["cpu_baseline"] = ref_line["cpu_baseline"]
            except Exception as ex:
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "unavailable",
                                        "sample": f"CPU arm failed: {type(ex).__name__}: {ex}"}
        print(json.dumps(line), flush=True)
    if distributed:
        dist.barrier(device_ids=[local_rank])
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
