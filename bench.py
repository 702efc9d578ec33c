#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (BASELINE.json): MNIST-16x16 images/sec at batch 1M on the
FC 4bitsym width-64 model (BitNetMCU_model_fc.h), int32 logits bit-exact, achieved HBM GB/s vs measured peak.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--model fc] [--batch 1048576]

A "step" = one pass of the whole chain (processfclayer x4 + ReLUNorm x4, BitMnistInference dll.c:95-121) over one
batch of synthetic int8 images resident in HBM.  N > 1: launched by torchrun, one rank per GPU, the batch shards by
rank with no data-path collective (weak scaling: 1M images per GPU).  Prints ONE JSON line on rank 0.

value        : whole-job images/s, device-timed (CUDA events), max over ranks, inputs resident in HBM, PLAIN launches
               (ordinary stream semantics: what a drop-in caller gets by default)
value_two_streams : same steps, plain launches alternating between two streams (ordinary CUDA semantics for independent batches)
value_overlapped_launches : same steps with BNM_OPT_LAUNCH_OVERLAP = 2 (consecutive launches declared independent; the
               bench double-buffers inputs and outputs, which is what that mode asks for)
value_sustained: >= 1 s of back-to-back plain launches, with the nvidia-smi clock sampler covering THAT region
e2e          : same metric through bnm_infer_batch with PINNED HOST buffers, H2D + D2H inside the timed region
roofline     : dominant kernel fc_chain_kernel: 296 algorithmic B/image x batch / mean launch duration (CUDA events)
configs      : every other BASELINE.json config (Binary-160, Ternary-64, 2bitsym-96, CNN-64, CNN-48 at 2^20; FC at 2^22),
               each with value, roofline against its real bound (HBM, or the integer-ALU pipe for the CNN front-end) and a
               full-batch parity flag against the oracle
latency_us_batch1: the drop-in Inference() (gcc-built shim, one image per call) next to the reference DLL's Inference()
cpu_baseline : the reference's own C code (oracle/_ref, all host cores) on a bounded sample, rank 0, N = 1
--impl reference: that CPU reference as the timed arm (rank 0 only)
"""
import argparse
import ctypes as Ct
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from (which may be read-only)


def _baseline_metric():
    """The headline metric, verbatim from BASELINE.json (the achieved-HBM half of it is the `roofline` object)."""
    try:
        with open(os.path.join(ROOT, "BASELINE.json")) as f:
            return str(json.load(f)["metric"])
    except Exception:
        return "MNIST-16x16 images/sec at batch 1M; achieved HBM GB/s vs B200 peak"


METRIC = _baseline_metric()
UNIT = "images/s"

# BASELINE.json configs 3-5 besides the headline (config 2): (fixture model, images per GPU)
EXTRA_CONFIGS = [("binary160", 1 << 20), ("ternary64", 1 << 20), ("2bitsym96", 1 << 20), ("cnn", 1 << 20), ("cnn_48", 1 << 20),
                 ("fc", 1 << 22)]


def load_model(name):
    from bitnetmcu_b200.model import Model
    return Model.load(os.path.join(ROOT, "tests", "golden", "models", name + ".bnm"))


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)", float(d.get("sm_max_mhz", 1965.0))
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)", 1965.0


def synth_images(n, img_bytes, seed, dist="uniform"):
    """Synthetic int8 images of the reference's input shape (no dataset in this sandbox).  SURVEY.md 8d config 2:
    (i) "uniform" int8; (ii) "mnist": background near -20 with a blob of strokes up to 127, the value profile of
    BitNetMCU_MNIST_test_data.h (normalised MNIST scaled to +-127) -- the GPU time must not depend on which."""
    rng = np.random.default_rng(seed)
    if dist == "uniform":
        return rng.integers(-128, 128, size=(n, img_bytes), dtype=np.int8)
    side = int(round(img_bytes ** 0.5))
    out = np.full((n, side, side), -20, dtype=np.int8)
    if side * side != img_bytes:
        return rng.integers(-128, 128, size=(n, img_bytes), dtype=np.int8)
    chunk = 1 << 16
    yy, xx = np.mgrid[0:side, 0:side].astype(np.float32)
    for b in range(0, n, chunk):
        m = min(chunk, n - b)
        cy, cx = rng.uniform(5, side - 5, (2, m, 1, 1)).astype(np.float32)
        ang = rng.uniform(0, np.pi, (m, 1, 1)).astype(np.float32)
        # a thick stroke through (cy, cx) at angle ang: distance to the line, faded at the ends
        d = np.abs((yy - cy) * np.cos(ang) - (xx - cx) * np.sin(ang))
        along = np.abs((yy - cy) * np.sin(ang) + (xx - cx) * np.cos(ang))
        ink = np.clip(1.6 - d, 0, 1) * np.clip(5.5 - along, 0, 1)
        out[b:b + m] = np.clip(-20 + 147 * ink + rng.integers(-2, 3, size=ink.shape), -128, 127).astype(np.int8)
    return out.reshape(n, img_bytes)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING a timed region (B200_PROFILING.md recipe).  Auxiliary: whatever
    goes wrong here (UUID-style CUDA_VISIBLE_DEVICES, no nvidia-smi) must never abort the measurement."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    @staticmethod
    def device_selector(local_rank):
        """What to hand to `nvidia-smi -i`: an index or a UUID string, from CUDA_VISIBLE_DEVICES when it is set."""
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "").strip()
        try:
            if vis:
                items = [v.strip() for v in vis.split(",") if v.strip()]
                item = items[local_rank] if local_rank < len(items) else items[0]
                return item            # "3" or "GPU-xxxx" / "MIG-...": nvidia-smi -i takes either
            import torch
            return str(torch.cuda.current_device())
        except Exception:
            return str(local_rank)

    def __init__(self, selector):
        self.sel = str(selector)
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", self.sel, f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        try:
            for line in self.proc.stdout:
                self.lines.append((time.perf_counter(), line.strip()))
        except Exception:
            pass

    def stop(self, t0, t1, region):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "region": region}
        time.sleep(0.15)
        try:
            self.proc.terminate()
        except Exception:
            pass
        inside = [l.split(", ") for t, l in self.lines if t0 <= t <= t1]
        rows = inside or [l.split(", ") for t, l in self.lines if t0 - 0.1 <= t <= t1 + 0.2] or [l.split(", ") for _, l in self.lines]
        sm, smax, power, reasons = [], [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1])); smax.append(float(r[2])); power.append(float(r[3]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "reasons": sorted(reasons), "samples": len(sm),
                "samples_inside_region": len(inside), "region": region}


def host_cpu_budget():
    """(logical CPUs, cgroup CPU quota in cores or None): the GPU boxes expose many logical CPUs under a smaller quota."""
    n = os.cpu_count() or 1
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, p = f.read().split()
        if q != "max":
            quota = float(q) / float(p)
    except Exception:
        pass
    return n, quota


def checker_threads():
    ncpu, quota = host_cpu_budget()
    return max(1, int(quota + 0.5)) if quota else ncpu


def cpu_reference_rate(model, images, budget_s=1.0, reps=3):
    """Time the reference's own C implementation (oracle/_ref: BitNetMCU_inference.c compiled unmodified + our batch
    driver, images fanned over host threads) -- or the oracle port when _ref is absent -- on a bounded sample.  The thread
    count is the better of "all logical CPUs" and "the cgroup quota" (over-subscribing a quota-limited box is slower)."""
    from oracle.oracle import Oracle, Reference
    if Reference.available():
        impl, kind = Reference(), "reference"
    else:
        impl, kind = Oracle(), "port"
    ncpu, quota = host_cpu_budget()
    cands = sorted({ncpu, max(1, int(quota + 0.5)) if quota else ncpu})
    probe = images[: min(len(images), 32768)]
    best_threads, rate = ncpu, 0.0
    for th in cands:
        impl.infer(model, probe[:2048], threads=th)
        t = time.perf_counter(); impl.infer(model, probe, threads=th); dt = time.perf_counter() - t
        if len(probe) / dt > rate:
            rate, best_threads = len(probe) / dt, th
    n = int(min(len(images), max(32768, rate * budget_s)))
    best = None
    for _ in range(reps):
        t = time.perf_counter(); impl.infer(model, images[:n], threads=best_threads); dt = time.perf_counter() - t
        best = dt if best is None else min(best, dt)
    return {"value": n / best, "unit": UNIT, "cores": best_threads, "kind": kind,
            "sample": f"{n} of the {len(images)} synthetic images, best of {reps}, {best_threads} pthreads "
                      f"({ncpu} logical CPUs, cgroup quota {('%.1f' % quota) if quota else 'none'}), gcc -O3 -march=x86-64-v3"}, impl, n, best_threads


def run_reference_arm(args):
    """--impl reference: the reference's CPU implementation of the same path/config on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    import __graft_entry__ as g
    try:
        g.build_oracle()
    except Exception:
        pass
    model = load_model(args.model)
    images = synth_images(args.batch, model.img_bytes, 1234, args.dist)
    base, impl, n, threads = cpu_reference_rate(model, images, budget_s=1.0, reps=1)
    for _ in range(args.warmup):
        impl.infer(model, images[:n], threads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        logits, labels = impl.infer(model, images[:n], threads=threads)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"logits": logits, "labels": labels})
    value = n * args.steps / dt
    base["value"] = value
    base["sample"] = f"each step = {n} of the {args.batch} synthetic images; " + base["sample"].split(", best of")[1].split(", ", 1)[1]
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int8", "data": "synthetic" if args.dist == "uniform" else "synthetic (MNIST-like value profile)",
        "config": {"workload": workload_name(args.model, model, args.batch), "batch_per_gpu": args.batch, "sample_per_step": n},
        "cpu_baseline": base,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), file=RESULT_OUT, flush=True)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays, seed=0):
    """Write each array (all with the same leading row count) as out_dir/<name>.npy: float32, or float64 where float32 would not
    hold its integers exactly.  Above DUMP_LIMIT_BYTES in all, a fixed seeded sample of rows is written instead, with the
    indices of those rows as out_dir/rows.npy."""
    os.makedirs(out_dir, exist_ok=True)
    exact32 = lambda a: a.size == 0 or (-(1 << 24) <= a.min() and a.max() <= (1 << 24))
    arrays = {k: a.astype(np.float32 if exact32(a) else np.float64) for k, a in arrays.items()}
    n = next(iter(arrays.values())).shape[0]
    row_bytes = sum(a.nbytes // max(n, 1) for a in arrays.values())
    if n * row_bytes > DUMP_LIMIT_BYTES:
        keep = DUMP_LIMIT_BYTES // (row_bytes + 8)
        rows = np.sort(np.random.default_rng(seed).choice(n, size=keep, replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def workload_name(name, model, batch):
    return f"{name}: {model.describe()} | batch {batch} x {model.img_bytes} B int8 per GPU"


RESULT_OUT = sys.stdout


def claim_stdout():
    """stdout must carry exactly ONE JSON line.  Libraries loaded later write to file descriptor 1 behind Python's back
    (NCCL prints its "NCCL version ..." banner there at NCCL_DEBUG=VERSION/WARN), so keep a private copy of the real
    stdout for the result and point descriptor 1 at stderr for everything else."""
    global RESULT_OUT
    sys.stdout.flush()
    RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ------------------------------------------------------------------------------------------------------------------
# measurement helpers (GPU arm)
# ------------------------------------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(local_rank):
    """Pin this process (and therefore its first-touch pinned allocations) to the CPUs of the NUMA node its GPU hangs off
    (GPU0-3 <-> node 0, GPU4-7 <-> node 1 on these boxes): the e2e arm streams 268 MB per step through pinned host memory, and a
    rank running on the far socket pays the inter-socket hop on every byte.  Best effort; returns a short description."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id if hasattr(torch.cuda.get_device_properties(local_rank), "pci_bus_id") else None
        dom = getattr(torch.cuda.get_device_properties(local_rank), "pci_domain_id", 0)
        dev = getattr(torch.cuda.get_device_properties(local_rank), "pci_device_id", 0)
        if bus is None:
            return "pci bus id unavailable"
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0"
        node = int(open(path + "/numa_node").read().strip())
        cpulist = open(path + "/local_cpulist").read().strip()
        cpus = set()
        for part in cpulist.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if node < 0 or not cpus:
            return f"numa_node {node}: not bound"
        os.sched_setaffinity(0, cpus)
        return f"bound to NUMA node {node} ({len(cpus)} CPUs)"
    except Exception as ex:
        return f"not bound: {ex}"


class Ctx:
    """torch plumbing shared by the measurements of one process / rank."""

    def __init__(self):
        import torch
        import torch.distributed as tdist
        from bitnetmcu_b200 import dist as bdist
        self.torch, self.tdist = torch, tdist
        self.rank, self.local_rank, self.world = bdist.env_rank_world()
        if self.world > 1:
            os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # NCCL's INFO log: stderr, not stdout (see claim_stdout)
            bdist.init_process_group("nccl")
        torch.cuda.set_device(self.local_rank)
        self.numa = bind_to_gpu_numa_node(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.stream = torch.cuda.current_stream(self.dev)

    def barrier(self):
        if self.world > 1:
            self.tdist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.tdist.all_reduce(t, op=self.tdist.ReduceOp.MAX)
        return float(t.item())

    def timed_steps(self, step, steps, warmup):
        """warmup untimed steps, then exactly `steps` steps between two events on the launching stream, barrier + synchronize on
        both sides; returns (max-over-ranks ms per step, this rank's ms per step)."""
        torch = self.torch
        for i in range(warmup):
            step(i)
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        for i in range(steps):
            step(i)
        e1.record(self.stream)
        self.barrier()
        local = e0.elapsed_time(e1) / steps
        return self.max_over_ranks(local), local


class DeviceBatch:
    """Two image buffers alternated per step (each n x 256 B = 268 MB at 1M: larger than the 126 MB L2) and double-buffered
    outputs: consecutive launches touch disjoint buffers."""

    def __init__(self, ctx, eng, host_imgs):
        torch = ctx.torch
        n, C = host_imgs.shape[0], eng.n_classes
        self.n = n
        self.d_in = [torch.from_numpy(host_imgs).to(ctx.dev), torch.from_numpy(np.ascontiguousarray(host_imgs[::-1])).to(ctx.dev)]
        self.d_logits = [torch.empty((n, C), dtype=torch.int32, device=ctx.dev) for _ in range(2)]
        self.d_labels = [torch.empty(n, dtype=torch.int32, device=ctx.dev) for _ in range(2)]
        self.eng, self.ctx = eng, ctx

    def step(self, i):
        self.eng.infer_device(self.d_in[i & 1], self.d_logits[i & 1], self.d_labels[i & 1], self.ctx.stream.cuda_stream)

    def snapshot(self):
        return [(self.d_logits[k].cpu().numpy(), self.d_labels[k].cpu().numpy().view(np.uint32)) for k in range(2)]


def int_alu_peak_ops(sm_max_mhz):
    """Integer-ALU roofline of the CNN front-end: the dot-product unit issues one IDP.4A warp instruction per 2 cycles per SM
    sub-partition (tools/alu_rates.cu, profiles/r1_micro_alu_rates.txt: 2.00 cycles) = 64 lanes/clk/SM x 4 MAC x 2 ops, 148 SMs,
    at the maximum SM clock.  (conv2/conv3 take int16/int32 activations and can only use IDP.2A / IMAD = 2 / 1 MAC per lane.)"""
    return 148 * 64 * 8 * sm_max_mhz * 1e6


def epilogue_alu_bound(model, sm_max_mhz):
    """Second ceiling of the fused FC kernel: the integer ALU pipe of the in-TMEM ReLUNorm.  Every hidden-layer accumulator costs
    2.33 ALU-pipe instructions (VIADDMNMX.RELU + 1/2 VIMNMX3 + 3/4 PRMT; the shift is an IMAD on the FMA pipe) at one warp
    instruction per 2 cycles per SM sub-partition (tools/alu_rates.cu): images/s <= 148 SMs x 4 x 32 lanes / (accumulators x 2.33 x 2
    cycles) x clock.  Wide models (Binary-160: 480 hidden accumulators per image) hit this ceiling far below the HBM roofline."""
    fc = model.fc_layers
    acc = sum(l.n_out for l in fc[:-1])
    ips = 148 * 4 * 32 / (max(acc, 1) * 2.33 * 2) * sm_max_mhz * 1e6
    return {"hidden_accumulators_per_image": acc, "images_per_s": ips, "alu_instructions_per_accumulator": 2.33}


def run_config(ctx, name, batch, steps, warmup, args, check_parity=True, host_imgs=None):
    """One BASELINE config: device-timed plain launches, its roofline, full-batch parity against the oracle (rank 0)."""
    from bitnetmcu_b200 import _lib
    from bitnetmcu_b200.engine import Engine
    model = load_model(name)
    eng = Engine(model, device=ctx.local_rank)
    n, C = batch, eng.n_classes
    if host_imgs is None or host_imgs.shape[0] != n:
        host_imgs = synth_images(n, eng.img_bytes, 4321 + ctx.rank, args.dist)
    db = DeviceBatch(ctx, eng, host_imgs)
    eng.set_option(_lib.OPT_LAUNCH_OVERLAP, 0)
    ms, _ = ctx.timed_steps(db.step, steps, warmup)
    value = ctx.world * n / (ms * 1e-3)
    peak_gbs, peak_src, sm_max = measured_peaks()
    bytes_per_image = eng.img_bytes + 4 * C
    hbm_ach = bytes_per_image * n / (ms * 1e-3) / 1e9
    cnn = model.model_class == 1
    if cnn:
        ops = 2.0 * model.macs_per_image * n / (ms * 1e-3)
        peak_ops = int_alu_peak_ops(sm_max)
        roof = {"bound": "int_alu", "achieved": ops / 1e12, "peak": peak_ops / 1e12, "unit": "Top/s", "frac": ops / peak_ops,
                "peak_source": f"IDP.4A issue rate (1 warp instruction / 2 cycles / SM sub-partition, tools/alu_rates.cu) x 148 SMs x {sm_max:.0f} MHz",
                "macs_per_image": model.macs_per_image, "hbm_frac": hbm_ach / peak_gbs, "traffic": traffic_for(name, n)}
    else:
        roof = {"bound": "hbm", "achieved": hbm_ach, "peak": peak_gbs, "unit": "GB/s", "frac": hbm_ach / peak_gbs,
                "peak_source": peak_src, "algorithmic_bytes_per_image": bytes_per_image, "traffic": traffic_for(name, n),
                "alu_pipe_bound": epilogue_alu_bound(model, sm_max)}
        roof["alu_pipe_bound"]["frac"] = value / ctx.world / roof["alu_pipe_bound"]["images_per_s"]
    out = {"name": name, "workload": workload_name(name, model, n), "value": value, "unit": UNIT, "ms_per_step": ms, "steps": steps,
           "warmup": warmup, "gpu_launches_per_step": eng.launch_count(n), "launch_semantics": "plain launches",
           "path": "tcgen05" if eng.active_path == _lib.PATH_TCGEN05 else "layers", "roofline": roof}
    if cnn:
        out["cnn_frontend"] = {0: "auto (tensor cores when covered)", 1: "CUDA cores", 2: "tensor cores"}.get(int(eng.lib.bnm_model_get_option(eng.handle, _lib.OPT_CNN_FRONTEND)))
    if cnn:   # e2e through the C ABI with pinned host buffers for the CNN config too (three-stream chunk pipeline, per-slot feature buffers)
        try:
            out["e2e"] = e2e_through_c_abi(ctx, eng, host_imgs, steps=3, warm=2)
        except Exception as ex:
            out["e2e"] = {"error": str(ex)[:200]}
    if check_parity and ctx.rank == 0:
        try:
            from oracle.oracle import Oracle
            got_l, got_b = db.snapshot()[0]
            t0 = time.perf_counter()
            ns = n if n <= (1 << 20) else (1 << 18)
            oo, ol = Oracle().infer(model, host_imgs[:ns], threads=checker_threads())
            ok = bool(zlib.crc32(got_l[:ns].tobytes()) == zlib.crc32(oo.tobytes()) and np.array_equal(got_b[:ns], ol))
            out["parity"] = ok
            out["parity_check"] = (f"logits CRC-32 + labels of {'the full batch' if ns == n else 'the first %d images' % ns} of the timed launches "
                                   f"vs the oracle ({time.perf_counter() - t0:.1f} s of CPU)")
        except Exception as ex:
            out["parity"] = f"oracle unavailable: {ex}"
    eng.close()
    del db
    ctx.torch.cuda.empty_cache()
    return out


def e2e_through_c_abi(ctx, eng, host_imgs, steps, warm=3, keep=None):
    """The metric end to end through bnm_infer_batch: pinned host buffers in, pinned host buffers out, H2D + kernels + D2H inside the
    timed region (wall clock around `steps` calls, max over ranks).  keep: dict that receives the result arrays of the last call."""
    from bitnetmcu_b200 import _lib
    lib = _lib.load()
    n, C = host_imgs.shape[0], eng.n_classes
    nb_in, nb_log, nb_lab = n * eng.img_bytes, n * C * 4, n * 4
    p_in, p_log, p_lab = lib.bnm_host_alloc(nb_in), lib.bnm_host_alloc(nb_log), lib.bnm_host_alloc(nb_lab)
    try:
        h_in = np.ctypeslib.as_array((Ct.c_int8 * nb_in).from_address(p_in)).reshape(n, eng.img_bytes)
        h_log = np.ctypeslib.as_array((Ct.c_int32 * (n * C)).from_address(p_log)).reshape(n, C)
        h_lab = np.ctypeslib.as_array((Ct.c_uint32 * n).from_address(p_lab))
        h_in[:] = host_imgs
        eng.set_option(_lib.OPT_CHUNK_IMAGES, 1 << 17)
        for _ in range(warm):
            eng.infer(h_in, out_logits=h_log, out_labels=h_lab)
        ctx.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            eng.infer(h_in, out_logits=h_log, out_labels=h_lab)
        ctx.torch.cuda.synchronize()
        dt = ctx.max_over_ranks(time.perf_counter() - t0)
        if keep is not None:
            keep["logits"], keep["labels"] = h_log.copy(), h_lab.copy()
        return {"value": ctx.world * n * steps / dt, "unit": UNIT, "h2d_bytes_per_step": nb_in, "d2h_bytes_per_step": nb_log + nb_lab,
                "ms_per_step": 1e3 * dt / steps, "api": "bnm_infer_batch (pinned host buffers, 3-stream chunk pipeline)"}
    finally:
        lib.bnm_host_free(p_in); lib.bnm_host_free(p_log); lib.bnm_host_free(p_lab)


def run_float_input(ctx, name, batch, steps, warmup, args):
    """SURVEY.md 8f rank 3: float32 images in (1 024 B/image), the scaling of test_inference.py:140-141 fused into the FC kernel's load
    stage (bnm_infer_batch_device_f32) -- next to the chain of the scaling kernel and the int8 kernel it replaces.  Parity: the fused
    launch's full batch against the chain's, and a slice against NumPy scaling + oracle."""
    from bitnetmcu_b200 import engine as E
    from bitnetmcu_b200.engine import Engine
    torch = ctx.torch
    model = load_model(name)
    eng = Engine(model, device=ctx.local_rank)
    n, C = batch, eng.n_classes
    rng = np.random.default_rng(99 + ctx.rank)
    host = rng.normal(size=(1 << 16, eng.img_bytes)).astype(np.float32)
    d_x = [torch.from_numpy(host).to(ctx.dev).repeat(n >> 16, 1).contiguous() for _ in range(2)]
    d_x[1].mul_(1.5)
    d_q = torch.empty((n, eng.img_bytes), dtype=torch.int8, device=ctx.dev)
    d_log = [torch.empty((n, C), dtype=torch.int32, device=ctx.dev) for _ in range(2)]
    d_lab = [torch.empty(n, dtype=torch.int32, device=ctx.dev) for _ in range(2)]
    st = ctx.stream.cuda_stream

    def fused(i):
        eng.infer_device_f32(d_x[i & 1], d_log[0], d_lab[0], st)

    def chained(i):
        E.quantize_images_device(d_x[i & 1], d_q, st)
        eng.infer_device(d_q, d_log[1], d_lab[1], st)
    ms_f, _ = ctx.timed_steps(fused, steps, warmup)
    ms_c, _ = ctx.timed_steps(chained, steps, warmup)
    fused(1); chained(1)
    torch.cuda.synchronize()
    same = bool(torch.equal(d_log[0], d_log[1]) and torch.equal(d_lab[0], d_lab[1]))
    parity = same
    if ctx.rank == 0:
        try:
            from oracle.oracle import Oracle
            x = (host[:4096] * np.float32(1.5))
            scale = np.float32(127.0) / np.maximum(np.abs(x).max(axis=-1, keepdims=True), np.float32(1e-5))
            q = np.round(x * scale).clip(-128, 127).astype(np.int8)
            oo, ol = Oracle().infer(model, q, threads=checker_threads())
            parity = bool(same and np.array_equal(d_log[0][:4096].cpu().numpy(), oo) and np.array_equal(d_lab[0][:4096].cpu().numpy().astype(np.uint32), ol))
        except Exception as ex:
            parity = f"oracle unavailable: {ex}"
    peak, peak_src, _ = measured_peaks()
    bpi = 4 * eng.img_bytes + 4 * C
    out = {"name": name + "_float_input", "workload": f"{name}: float32 images [{n}][{eng.img_bytes}] -> int32 logits, input scaling fused into the FC kernel",
           "value": ctx.world * n / (ms_f * 1e-3), "unit": UNIT, "ms_per_step": ms_f, "steps": steps, "warmup": warmup, "gpu_launches_per_step": 1,
           "value_chained_kernels": ctx.world * n / (ms_c * 1e-3), "ms_per_step_chained_kernels": ms_c,
           "roofline": {"bound": "hbm", "achieved": bpi * n / (ms_f * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": bpi * n / (ms_f * 1e-3) / 1e9 / peak,
                        "algorithmic_bytes_per_image": bpi, "peak_source": peak_src, "traffic": None,
                        "chained_kernels_bytes_per_image": bpi + 2 * eng.img_bytes},
           "parity": parity, "parity_check": "fused launch == scaling kernel + int8 kernel on the full batch; first 4096 images == NumPy scaling + oracle"}
    eng.close()
    del d_x, d_q, d_log, d_lab
    torch.cuda.empty_cache()
    return out


_TRAFFIC = None


def traffic_for(name, n):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture (profiles/traffic.json);
    not re-measured inside a bench run (nothing printed under a profiler is a bench value)."""
    global _TRAFFIC
    if _TRAFFIC is None:
        try:
            _TRAFFIC = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        except Exception:
            _TRAFFIC = {}
    return _TRAFFIC.get(f"{name}:{n}")


def latency_batch1(model_name="fc", calls=10000):
    """Single-image latency of the drop-in: host/bitnetmcu_b200_latency.c (plain C, gcc) dlopen()s a DLL and calls its exported
    Inference() `calls` times over the ten reference digits -- once for the gcc-built shim of THIS library (host/bitnetmcu_b200_dll.c +
    a header written from the fixture model), once for the reference's own DLL (oracle/_ref, when it travelled)."""
    from bitnetmcu_b200 import _lib
    from bitnetmcu_b200.pack import write_header
    out = {"calls": calls, "model": model_name}
    tmp = tempfile.mkdtemp(prefix="bnm_lat_")
    try:
        m = load_model(model_name)
        write_header(m, os.path.join(tmp, "BitNetMCU_model.h"))
        libdir = os.path.dirname(_lib.LIB_PATH)
        dll = os.path.join(tmp, "Bitnet_inf.dll")
        exe = os.path.join(tmp, "latency")
        subprocess.run(["gcc", "-O2", "-fPIC", "-shared", "-D_DLL", "-o", dll, os.path.join(ROOT, "host", "bitnetmcu_b200_dll.c"), "-I" + tmp,
                        "-I" + os.path.join(ROOT, "include"), "-L" + libdir, "-lbitnetmcu_b200", "-Wl,-rpath," + libdir], check=True, capture_output=True)
        subprocess.run(["gcc", "-O2", "-o", exe, os.path.join(ROOT, "host", "bitnetmcu_b200_latency.c"), "-ldl"], check=True, capture_output=True)
        d = np.load(os.path.join(ROOT, "tests", "golden", "digits.npz"))
        d["images"].astype(np.int8).tofile(os.path.join(tmp, "digits.bin"))
        want = ",".join(str(int(v)) for v in d["labels"])

        def run(path):
            r = subprocess.run([exe, path, os.path.join(tmp, "digits.bin"), str(calls)], capture_output=True, text=True, timeout=300)
            return json.loads(r.stdout.strip().splitlines()[-1])
        ours = run(dll)
        out["ours_us"] = ours["us_per_call"]
        out["ours_labels_ok"] = ours["labels"] == want
        ref = os.path.join(ROOT, "oracle", "_ref", f"Bitnet_inf_{model_name}.so")
        if os.path.exists(ref):
            r = run(ref)
            out["reference_us"] = r["us_per_call"]
            out["reference_labels_ok"] = r["labels"] == want
        else:
            out["reference_us"] = None
        out["note"] = "one image per call through the exported Inference(): H2D + launch + D2H + sync per call (ours), one CPU core (reference)"
    except Exception as ex:
        out["error"] = str(ex)[:300]
    return out


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="fc")
    ap.add_argument("--batch", type=int, default=1 << 20, help="images per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the `configs` block (the other BASELINE.json configs)")
    ap.add_argument("--configs-multi-gpu", action="store_true", help="run the `configs` block at N > 1 as well (default: N = 1 only, "
                    "they are single-GPU workloads and every one of them synchronises the ranks)")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--sustain-seconds", type=float, default=1.0)
    ap.add_argument("--path", default="auto", choices=["auto", "layers", "tcgen05"])
    ap.add_argument("--dist", default="uniform", choices=["uniform", "mnist"], help="synthetic image distribution (SURVEY.md 8d config 2)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the logits and labels of the last timed step as DIR/<name>.npy (rank 0; "
                    "inputs are seeded, so runs with the same arguments can be compared output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference_arm(args)

    from bitnetmcu_b200 import _lib
    from bitnetmcu_b200.engine import Engine
    ctx = Ctx()
    torch, rank, world = ctx.torch, ctx.rank, ctx.world
    model = load_model(args.model)
    path = {"auto": _lib.PATH_AUTO, "layers": _lib.PATH_LAYERS, "tcgen05": _lib.PATH_TCGEN05}[args.path]
    eng = Engine(model, device=ctx.local_rank, path=path)
    n, C = args.batch, eng.n_classes

    # ---- device-resident inputs, larger than L2, alternated per step
    host_imgs = synth_images(n, eng.img_bytes, 1234 + rank, args.dist)
    db = DeviceBatch(ctx, eng, host_imgs)

    # ---- headline: K steps, plain launches (ordinary stream semantics)
    eng.set_option(_lib.OPT_LAUNCH_OVERLAP, 0)
    ms_per_step, local_ms = ctx.timed_steps(db.step, args.steps, args.warmup)
    value = world * n / (ms_per_step * 1e-3)
    snap_plain = db.snapshot()
    launches = args.steps * eng.launch_count(n)

    # ---- the same steps, still plain launches, alternating between TWO streams: the ordinary CUDA way for a caller to say that
    # consecutive (double-buffered) batches are independent -- the tail of one launch then overlaps the head of the next
    ms_two = None
    try:
        two = [torch.cuda.Stream(device=ctx.dev), torch.cuda.Stream(device=ctx.dev)]

        def step2(i):
            eng.infer_device(db.d_in[i & 1], db.d_logits[i & 1], db.d_labels[i & 1], two[i & 1].cuda_stream)
        for i in range(4):
            step2(i)
        ctx.barrier()
        t0e, e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0e.record(two[0]); two[1].wait_event(t0e)
        for i in range(args.steps):
            step2(i)
        e0.record(two[0]); e1.record(two[1])
        ctx.barrier()
        ms_two = ctx.max_over_ranks(max(t0e.elapsed_time(e0), t0e.elapsed_time(e1)) / args.steps)
    except Exception as ex:
        log("two-stream measurement failed:", ex)

    # ---- the same steps with consecutive launches declared independent (BNM_OPT_LAUNCH_OVERLAP = 2)
    eng.set_option(_lib.OPT_LAUNCH_OVERLAP, 2)
    ms_overlap, _ = ctx.timed_steps(db.step, args.steps, 3)
    snap_overlap = db.snapshot()
    eng.set_option(_lib.OPT_LAUNCH_OVERLAP, 0)

    # ---- sustained: >= sustain_seconds of back-to-back plain launches, clocks sampled over exactly this region
    for i in range(3):
        db.step(i)
    ctx.barrier()
    sampler = ClockSampler(ClockSampler.device_selector(ctx.local_rank))
    sampler.start()
    time.sleep(0.3)
    ctx.barrier()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_s0 = time.perf_counter()
    s0.record(ctx.stream)
    n_sus = 0
    while True:
        for _ in range(64):
            db.step(n_sus); n_sus += 1
        torch.cuda.synchronize()
        if time.perf_counter() - t_s0 >= args.sustain_seconds:
            break
    s1.record(ctx.stream)
    torch.cuda.synchronize()
    t_s1 = time.perf_counter()
    sus_ms = ctx.max_over_ranks(s0.elapsed_time(s1))
    clocks = sampler.stop(t_s0, t_s1, f"the value_sustained loop ({n_sus} back-to-back plain launches, {sus_ms / 1e3:.2f} s), which runs the same "
                                      "kernel on the same buffers right after the timed steps (the timed region itself is ~1 ms, below the 100 ms sampling period)")
    sustained = {"value": world * n * n_sus / (sus_ms * 1e-3), "unit": UNIT, "seconds": sus_ms / 1e3, "launches": n_sus,
                 "ms_per_step": sus_ms / n_sus, "note": "a host synchronise every 64 launches is inside the region"}

    # ---- one launch timed alone with its own event pair (no overlap with neighbours, includes the event/launch gap)
    durs = []
    for i in range(args.steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(ctx.stream); db.step(i); b.record(ctx.stream)
        durs.append((a, b))
    torch.cuda.synchronize()
    kernel_ms_isolated = statistics.mean(a.elapsed_time(b) for a, b in durs)

    single_kernel_step = eng.launch_count(n) == 1
    kernel_ms = local_ms if single_kernel_step else kernel_ms_isolated
    bytes_per_image = eng.img_bytes + 4 * C          # SURVEY.md 8d: 256 B read + 10 x int32 written = 296 B (labels +4 B not counted)
    peak, peak_src, _ = measured_peaks()
    gbs = lambda ms: bytes_per_image * n / (ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": gbs(kernel_ms), "peak": peak, "unit": "GB/s", "frac": gbs(kernel_ms) / peak,
                "traffic": traffic_for(args.model, n), "kernel": "fc_chain_kernel" if eng.active_path == _lib.PATH_TCGEN05 else "layer kernels",
                "kernel_ms": kernel_ms, "kernel_ms_isolated_launch": kernel_ms_isolated,
                "frac_two_streams": (gbs(ms_two) / peak) if (ms_two and single_kernel_step) else None,
                "frac_overlapped_launches": gbs(ms_overlap) / peak if single_kernel_step else None,
                "frac_sustained": gbs(sus_ms / n_sus) / peak if single_kernel_step else None,
                "algorithmic_bytes_per_image": bytes_per_image, "peak_source": peak_src,
                "launch_semantics": "frac = plain launches (ordinary stream semantics)"}

    # ---- e2e through the C ABI with pinned host buffers + parity of everything timed above (oracle = checker only)
    parity = None
    e2e = None
    if not args.no_e2e:
        keep = {}
        e2e = e2e_through_c_abi(ctx, eng, host_imgs, steps=args.steps, warm=3, keep=keep)
        h_log, h_lab = keep["logits"], keep["labels"]
        try:
            from oracle.oracle import Oracle
            ns = min(n, 1 << 16)
            oo, ol = Oracle().infer(model, host_imgs[:ns], threads=checker_threads())
            parity = bool(np.array_equal(h_log[:ns], oo) and np.array_equal(h_lab[:ns], ol))
            # ... and the device path's results, the whole batch, both buffers (buffer 1 holds the images in reverse order), plain
            # and overlapped launches, against the e2e result that was just checked
            for snap in (snap_plain, snap_overlap):
                parity = parity and bool(np.array_equal(snap[0][0], h_log) and np.array_equal(snap[0][1], h_lab)
                                         and np.array_equal(snap[1][0], h_log[::-1]) and np.array_equal(snap[1][1], h_lab[::-1]))
        except Exception as ex:  # the checker being unavailable must not hide the measurement
            parity = f"oracle unavailable: {ex}"

    # ---- N > 1: the result exchange (SURVEY.md 8e), timed separately -- `value` keeps the logits sharded
    gather = None
    if world > 1:
        try:
            from bitnetmcu_b200 import gather as bgather
            gather = bgather.bench_gathers(ctx, eng, db, ms_per_step)
        except Exception as ex:
            gather = {"error": str(ex)[:300]}

    del db
    torch.cuda.empty_cache()

    # ---- the other BASELINE.json configs
    configs = None
    if not args.no_configs and (world == 1 or args.configs_multi_gpu):
        configs = []
        shared = None
        for name, batch in EXTRA_CONFIGS:
            try:
                if shared is None or shared.shape[0] != batch:
                    shared = host_imgs if batch == n else synth_images(batch, 256, 977 + rank, args.dist)
                t0 = time.perf_counter()
                c = run_config(ctx, name, batch, steps=10 if batch <= (1 << 20) else 5, warmup=3, args=args, host_imgs=shared)
                log(f"config {name}@{batch}: {c['value'] / 1e9:.3f} G img/s, frac {c['roofline']['frac']:.3f}, parity {c.get('parity')}, {time.perf_counter() - t0:.1f} s")
                configs.append(c)
            except Exception as ex:
                configs.append({"name": name, "error": str(ex)[:300]})
        try:
            c = run_float_input(ctx, "fc", 1 << 20, steps=10, warmup=3, args=args)
            log(f"config {c['name']}: fused {c['value'] / 1e9:.3f} G img/s (frac {c['roofline']['frac']:.3f}), chained {c['value_chained_kernels'] / 1e9:.3f}, parity {c['parity']}")
            configs.append(c)
        except Exception as ex:
            configs.append({"name": "fc_float_input", "error": str(ex)[:300]})

    cpu_base = None
    latency = None
    if rank == 0 and world == 1:
        if not args.no_cpu_baseline:
            try:
                cpu_base, _, _, _ = cpu_reference_rate(model, host_imgs, budget_s=1.0, reps=3)
            except Exception as ex:
                cpu_base = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "unavailable", "sample": str(ex)}
        if not args.no_latency:
            latency = latency_batch1(args.model)

    if rank == 0:
        if args.dump_outputs:
            last_logits, last_labels = snap_plain[(args.steps - 1) & 1]   # DeviceBatch alternates its two buffers per step
            dump_outputs(args.dump_outputs, {"logits": last_logits, "labels": last_labels})
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int8", "data": "synthetic" if args.dist == "uniform" else "synthetic (MNIST-like value profile)",
            "config": {"workload": workload_name(args.model, model, n), "batch_per_gpu": n, "global_batch": n * world,
                       "parallelism": f"dp{world} (batch sharded, logits stay sharded; no data-path collective)",
                       "l2": "inputs larger than L2: two 268 MB image buffers alternated per step, TMA evict-first loads",
                       "path": "tcgen05" if eng.active_path == _lib.PATH_TCGEN05 else "layers",
                       "launch_semantics": "plain launches (BNM_OPT_LAUNCH_OVERLAP = 0): ordinary stream semantics",
                       "host_numa": ctx.numa},
            "value_two_streams": (world * n / (ms_two * 1e-3)) if ms_two else None,
            "value_overlapped_launches": world * n / (ms_overlap * 1e-3),
            "value_sustained": sustained,
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu_base,
            "parity_vs_oracle_sample": parity, "gather": gather, "configs": configs,
            "configs_note": None if configs is not None else "the other BASELINE configs are reported by the N = 1 run", "latency_us_batch1": latency,
        }
        print(json.dumps(out), file=RESULT_OUT, flush=True)
    eng.close()
    if world > 1:
        ctx.tdist.destroy_process_group()


if __name__ == "__main__":
    main()
