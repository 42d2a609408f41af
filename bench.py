#!/usr/bin/env python3
"""bench.py -- the SRCNN hot path on B200, BASELINE.json's configurations.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workloads c3,c2,c4,c5] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  Every timed loop of `--impl ours` runs exactly K steps.
`--dump-outputs DIR` writes, after the timed loops, what the last step of each loop returned
(rank 0's share) as DIR/<workload>_<entry>.npy; see dump_sample.  Workloads (BASELINE.json
`configs`):
  * c3 (primary: `metric`/`value`/`e2e`/`roofline`): INFERENCE of one 4096x4096 luma image with
    the 9-1-5 n1=64 n2=32 network, halo row-sharded across the N ranks (no collective; strong
    scaling).  A step = one forward pass of the whole image.  MPix/s = input pixels / step time.
  * c2 (`train`): TRAINING, one epoch over 4096 synthetic 33x33 patches PER RANK (weak scaling):
    forward + backward in chunks of 2048, ONE all-reduce of the flat 8129-float gradient through
    the product's own communicator (srcnn_allreduce_grads), momentum + weight-decay update.
  * c4 (`train_c4`): the 9-5-5 network, 65 536 patches in TOTAL split data-parallel across the
    ranks (strong scaling), same step.
  * c5 (`c5`): the 9-1-5 n1=128 n2=64 network on 256 frames of 1920x1080 in TOTAL, frames split
    across the ranks (strong scaling, no collective).
`value`s are measured with inputs resident in HBM; every `e2e` goes through the host-buffer
C-ABI entry (srcnn_infer_rows_host / srcnn_train_chunks_host / srcnn_infer_frames_host) with
pinned HOST buffers, H2D and D2H inside the timed region.  `--impl reference` times the
reference's own kernels (oracle/_ref; the oracle port when that was not built) on all host cores.
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
sys.path.insert(0, os.path.join(ROOT, "tests"))

IMG = 4096
PATCH = 33
MOMENTUM, DECAY = 0.9, 0.001
LR = np.array([1e-4, 1e-4, 1e-5], np.float32)   # example_config.json:8-10
C2_PATCHES_PER_RANK = 4096
C4_PATCHES_TOTAL = 65536
C5_FRAMES_TOTAL, C5_W, C5_H = 256, 1920, 1080

NETS = {"c3": (64, 32, 9, 1, 5), "c2": (64, 32, 9, 1, 5), "c4": (64, 32, 9, 5, 5),
        "c5": (128, 64, 9, 1, 5)}


def net_pad(cfg):
    return cfg[2] + cfg[3] + cfg[4] - 3


def fwd_flop(cfg, w, h):
    """Algorithmic forward FLOPs of one w x h sample: each layer's own output extent x 2 f^2 k n
    (SURVEY 8d)."""
    n1, n2, f1, f2, f3 = cfg
    w1, h1 = w - f1 + 1, h - f1 + 1
    w2, h2 = w1 - f2 + 1, h1 - f2 + 1
    w3, h3 = w2 - f3 + 1, h2 - f3 + 1
    return 2.0 * (w1 * h1 * f1 * f1 * n1 + w2 * h2 * f2 * f2 * n1 * n2 + w3 * h3 * f3 * f3 * n2)


def train_flop_per_patch(cfg):
    """forward + deltas + weight gradients of one 33x33 patch (SURVEY 8d: 23.05 MFLOP for 9-1-5
    64/32, 168.9 MFLOP for 9-5-5)."""
    n1, n2, f1, f2, f3 = cfg
    w1 = PATCH - f1 + 1
    w2 = w1 - f2 + 1
    w3 = w2 - f3 + 1
    fwd = fwd_flop(cfg, PATCH, PATCH)
    d2 = 2.0 * w2 * w2 * n2 * f3 * f3            # deltas 2 <- 3
    d1 = 2.0 * w1 * w1 * n1 * f2 * f2 * n2       # deltas 1 <- 2
    gw = 2.0 * (w3 * w3 * f3 * f3 * n2 + w2 * w2 * f2 * f2 * n1 * n2 + w1 * w1 * f1 * f1 * n1)
    return fwd + d2 + d1 + gw


def train_bytes_per_patch(cfg):
    """Algorithmic HBM bytes of one patch through a training chunk, per kernel of the chunk
    (every tensor the backward needs is materialised once and read by each consumer)."""
    n1, n2, f1, f2, f3 = cfg
    w1 = PATCH - f1 + 1
    w2 = w1 - f2 + 1
    w3 = w2 - f3 + 1
    px = 4 * PATCH * PATCH
    o1, o2, o3 = 4 * w1 * w1 * n1, 4 * w2 * w2 * n2, 4 * w3 * w3
    if f2 == 1:   # 9-1-5: d1 lives inside the layer-1 gradient kernel
        return {"forward_fused": px + o1 + o2 + o3,
                "bwd3_fused (d3, d2, gW3)": px + o3 + o2 + o3 + o2,
                "wgrad1_fused (d1 + gW1)": o2 + o1 + px,
                "wgrad2 (gW2)": o2 + o1}
    return {"forward l1": px + o1, "forward l2": o1 + o2, "forward l3": o2 + o3,
            "bwd3_fused (d3, d2, gW3)": px + o3 + o2 + o3 + o2,
            "deltas l1": o2 + o1 + o1, "gW2": o2 + o1, "gW1": o1 + px}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), "measured"
    return 6650.0, 1590.0, "fallback"


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed
    ncu --set full capture (profiles/traffic.json, written by tools/ncu_summary.py)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None, None
    d = json.load(open(p)).get(kernel)
    if not d:
        return None, None
    return d.get("dram_bytes"), d.get("source")


class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU while the timed regions run: NVML in a
    thread every 10 ms (the training steps last tens of milliseconds), `nvidia-smi -lms 100` as
    a subprocess when NVML cannot be loaded."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    BITS = [0x8, 0x40, 0x20, 0x4]      # nvmlClocksEventReason{HwSlowdown,HwThermal,SwThermal,SwPowerCap}

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []           # [time, sm MHz, max sm MHz, set of reasons]
        self.proc = None
        self.nvml = None
        self.source = None
        self._stop = False

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            get_reasons(h)
            self.nvml = (pynvml, h, mx, get_reasons)
            self.source = "nvml, 10 ms"
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi -lms 100"
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll(self):
        pynvml, h, mx, get_reasons = self.nvml
        while not self._stop:
            try:
                sm = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                bits = int(get_reasons(h))
                self.rows.append([time.time(), sm, mx,
                                  {n for n, b in zip(self.NAMES, self.BITS) if bits & b}])
            except Exception:
                pass
            time.sleep(0.01)

    def _read(self):
        for line in self.proc.stdout:
            c = [x.strip() for x in line.split(",")]
            try:
                self.rows.append([time.time(), float(c[0]), float(c[1]),
                                  {n for n, v in zip(self.NAMES, c[3:7])
                                   if v.lower().startswith("active")}])
            except Exception:
                continue

    def summary(self, t0=None, t1=None):
        """clocks / throttle reasons of the samples taken in [t0, t1] (all samples by default)"""
        rows = [r for r in list(self.rows)
                if (t0 is None or r[0] >= t0) and (t1 is None or r[0] <= t1)]
        reasons = set()
        for r in rows:
            reasons |= r[3]
        return {"sm_mhz": float(np.median([r[1] for r in rows])) if rows else None,
                "sm_max_mhz": max(r[2] for r in rows) if rows else None,
                "reasons": sorted(reasons), "samples": len(rows), "source": self.source}

    def stop(self):
        if not self.proc and not self.nvml:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML, no nvidia-smi"]}
        time.sleep(0.15)
        self._stop = True
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        return self.summary()


def bind_to_gpu_numa_node(gpu_index):
    """Run this rank on the cores of its GPU's NUMA node BEFORE the pinned buffers are allocated
    (first touch puts their pages on that node): with 8 ranks copying at once, buffers on the far
    socket share the inter-socket link.  Best effort; returns the node or None."""
    try:
        bus = subprocess.check_output(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=pci.bus_id",
                                       "--format=csv,noheader"], text=True).strip().lower()
        # nvidia-smi prints an 8-digit domain (00000000:1b:00.0), sysfs uses 4 digits
        if bus.count(":") == 2 and len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def synthetic_params(cfg, seed=1234):
    from helpers import make_params
    rng = np.random.default_rng(seed + cfg[0] + 7 * cfg[3])
    return make_params(rng, *cfg)


def frames_like(rng, n, h, w):
    """n distinct synthetic frames: a few generated ones, rolled (cheap on the host)."""
    from helpers import luma_image
    base = [luma_image(rng, h, w) for _ in range(min(n, 4))]
    out = np.empty((n, h, w), np.float32)
    for i in range(n):
        out[i] = np.roll(base[i % len(base)], 17 * (i // len(base)), axis=1)
    return out


DUMP_SAMPLE = 1 << 20


def dump_sample(a):
    """An output as it is dumped: whole when it has at most DUMP_SAMPLE values, else the values
    at DUMP_SAMPLE distinct flat indices drawn by default_rng(0) (sorted), so that two builds
    given the same arguments are compared at the same positions.  Four sampled outputs of 4 MB
    keep a dump of every workload far below 64 MB."""
    a = np.ascontiguousarray(a, np.float32).reshape(-1)
    if a.size <= DUMP_SAMPLE:
        return a.copy()
    idx = np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))
    return a[idx]


def workload_config(n, wl):
    return {"workload": "C3: SRCNN 9-1-5 n1=64 n2=32 inference, one 4096x4096 luma image, halo "
                        "row bands over %d GPU(s)" % n,
            "secondary": {"train": "C2: 9-1-5 training, 4096 patches 33x33 PER GPU (weak), chunks "
                                   "of 2048, momentum + weight decay, one all-reduce of 8129 floats",
                          "train_c4": "C4: 9-5-5 training, 65536 patches in total split over the "
                                      "GPUs (strong), one all-reduce of 57281 floats",
                          "c5": "C5: 9-1-5 n1=128 n2=64 inference of 256 frames 1920x1080 in total, "
                                "frames split over the GPUs (strong)"},
            "workloads_run": wl, "net": "9-1-5 n1=64 n2=32", "image": [IMG, IMG],
            "patch": [PATCH, PATCH], "halo_rows": 12,
            "parallelism": "inference: row bands / frames, no collective; training: dp%d, one "
                           "all-reduce per update (NCCL communicator owned by the C-ABI)" % n,
            "l2": "inference rotates 4 input/output buffer pairs (>= 4x the band size) so no step "
                  "finds its input in the 126 MB L2; training streams > 1 GB of activations per "
                  "epoch; C5 walks >= 265 MB of frames per step"}


# ======================================================================= reference arm
def reference_numbers(args, wl):
    """The reference's own CPU implementation of the path on the host cores (oracle/_ref)."""
    from helpers import luma_image, patches
    from oracle.loader import NetState, Oracle, have
    kind = "reference" if have("reference") else "port"
    orc = Oracle(kind)
    # all host cores, also under torchrun (which exports OMP_NUM_THREADS=1)
    orc.set_num_threads(len(os.sched_getaffinity(0)))
    cores = orc.num_threads()
    rng = np.random.default_rng(1234)
    out = {"kind": kind, "cores": cores}
    if "c3" in wl:
        cfg = NETS["c3"]
        pad = net_pad(cfg)
        net = NetState(*cfg, synthetic_params(cfg))
        rows = min(args.ref_rows, IMG - pad)
        band = luma_image(rng, rows + pad, IMG)
        t = []
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            orc.net_forward(net, band, IMG, rows + pad, 1)
            t.append(time.perf_counter() - t0)
        sec = float(np.mean(t[args.warmup:]))
        frac = rows / float(IMG - pad)
        out["c3"] = {"mpix": IMG * IMG * frac / 1e6 / sec, "sec_per_step": sec, "frac": frac,
                     "sample": "%d of %d output rows of the 4096-wide image per step (%.1f%% of "
                               "C3)%s" % (rows, IMG - pad, 100 * frac,
                                          "" if frac == 1.0 else ", scaled linearly")}
    for key, npat in (("c2", args.ref_patches), ("c4", max(64, args.ref_patches // 4))):
        if key in wl:
            cfg = NETS[key]
            net = NetState(*cfg, synthetic_params(cfg))
            x, gt = patches(rng, npat, PATCH, PATCH)
            tt = []
            for i in range(2):
                t0 = time.perf_counter()
                orc.net_train_epoch(net, x, gt, PATCH, PATCH, npat, MOMENTUM, DECAY, LR)
                tt.append(time.perf_counter() - t0)
            out[key] = {"patches_per_s": npat / min(tt), "sample": "%d patches, 1 epoch, best of 2" % npat}
    if "c5" in wl:
        cfg = NETS["c5"]
        net = NetState(*cfg, synthetic_params(cfg))
        rows = 128
        band = luma_image(rng, rows + 12, C5_W)
        orc.net_forward(net, band, C5_W, rows + 12, 1)
        t0 = time.perf_counter()
        orc.net_forward(net, band, C5_W, rows + 12, 1)
        sec = time.perf_counter() - t0
        frac = rows / float(C5_H - 12)
        out["c5"] = {"mpix": C5_W * C5_H * frac / 1e6 / sec,
                     "sample": "%d of %d output rows of one 1920-wide frame, scaled linearly" % (rows, C5_H - 12)}
    return out


def run_reference(args, rank, world, wl):
    if rank != 0:
        return
    r = reference_numbers(args, wl)
    c3 = r.get("c3", {"mpix": None, "sec_per_step": 0.0, "frac": 1.0, "sample": "not run"})
    mpix = c3["mpix"]
    line = {
        "impl": "reference", "metric": "srcnn_915_inference_mpix_per_s", "value": mpix,
        "unit": "MPix/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * c3["sec_per_step"], "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus, wl),
        "cpu_baseline": {"value": mpix, "unit": "MPix/s", "cores": r["cores"], "kind": r["kind"],
                         "sample": c3["sample"]},
        "e2e": {"value": mpix, "unit": "MPix/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if "c2" in r:
        line["train"] = {"metric": "srcnn_915_train_patches_per_s", "value": r["c2"]["patches_per_s"],
                         "unit": "patches/s", "sample": r["c2"]["sample"]}
    if "c4" in r:
        line["train_c4"] = {"metric": "srcnn_955_train_patches_per_s", "value": r["c4"]["patches_per_s"],
                            "unit": "patches/s", "sample": r["c4"]["sample"]}
    if "c5" in r:
        line["c5"] = {"metric": "srcnn_915_wide_frames_mpix_per_s", "value": r["c5"]["mpix"],
                      "unit": "MPix/s", "sample": r["c5"]["sample"]}
    print(json.dumps(line), flush=True)


# ======================================================================= our arm
def run_ours(args, rank, world, local_rank, wl):
    import torch
    import torch.distributed as dist

    import _pkg
    from helpers import luma_image, patches
    pkg = _pkg.load()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    numa_node = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    stream = torch.cuda.Stream()
    hbm_peak, bf16_peak, peak_kind = peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    res = {}
    dump = bool(args.dump_outputs) and rank == 0
    dumps = {}
    with torch.cuda.stream(stream):
        ctx = pkg.Context(local_rank, stream=stream.cuda_stream)
        if world > 1:
            # the product's own communicator: rank 0 creates the id, torch only carries it over
            uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
            if rank == 0:
                uid.copy_(torch.tensor(list(pkg.Context.comm_unique_id()), dtype=torch.uint8))
            dist.broadcast(uid, 0)
            ctx.comm_init(rank, world, bytes(uid.cpu().tolist()))

        def timed(step_fn, steps, warmup):
            for i in range(warmup):
                step_fn(i)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n0 = ctx.launch_count()
            e0.record(stream)
            for i in range(steps):
                step_fn(warmup + i)
            e1.record(stream)
            barrier()
            ms = e0.elapsed_time(e1)
            return max_over_ranks(ms) / steps, ctx.launch_count() - n0

        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()

        # ---------------------------------------------------------------- PCIe reference rates
        pc_n = 64 << 20
        pc_h, pc_d = pkg.PinnedBuffer((pc_n // 4,)), ctx.alloc(pc_n)

        def copy_rate(fn):
            fn()
            ctx.block()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(4):
                fn()
            e1.record(stream)
            torch.cuda.synchronize()
            return 4 * pc_n / (e0.elapsed_time(e1) / 1e3) / 1e9

        h2d_gbs = copy_rate(lambda: ctx.L.srcnn_write(ctx.h, pc_d, 0, pc_n, pc_h.ptr, 0))
        d2h_gbs = copy_rate(lambda: ctx.L.srcnn_read(ctx.h, pc_d, 0, pc_n, pc_h.ptr, 0))
        ctx.release(pc_d)
        pc_h.free()
        # ... and with BOTH directions busy at once (what a pipelined host-buffer call does most
        # of the time): two torch streams, pinned tensors, 4 x 64 MiB each way
        try:
            hp_a = torch.empty(pc_n, dtype=torch.uint8).pin_memory()
            hp_b = torch.empty(pc_n, dtype=torch.uint8).pin_memory()
            dv_a = torch.empty(pc_n, dtype=torch.uint8, device="cuda")
            dv_b = torch.empty(pc_n, dtype=torch.uint8, device="cuda")
            s_up, s_dn = torch.cuda.Stream(), torch.cuda.Stream()
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            for rep in range(2):            # the first round is the warm-up
                torch.cuda.synchronize()
                ev[0].record(s_up)
                ev[2].record(s_dn)
                for _ in range(4):
                    with torch.cuda.stream(s_up):
                        dv_a.copy_(hp_a, non_blocking=True)
                    with torch.cuda.stream(s_dn):
                        hp_b.copy_(dv_b, non_blocking=True)
                ev[1].record(s_up)
                ev[3].record(s_dn)
                torch.cuda.synchronize()
            h2d_bidir = 4 * pc_n / (ev[0].elapsed_time(ev[1]) / 1e3) / 1e9
            d2h_bidir = 4 * pc_n / (ev[2].elapsed_time(ev[3]) / 1e3) / 1e9
            del hp_a, hp_b, dv_a, dv_b
        except Exception:
            h2d_bidir = d2h_bidir = None

        def pcie_block(h2d, d2h, ms):
            floor = max(h2d / h2d_gbs, d2h / d2h_gbs) / 1e6    # ms, both directions overlapped
            out = {"h2d_gbs_measured": h2d_gbs, "d2h_gbs_measured": d2h_gbs,
                   "floor_ms": floor, "frac_of_floor": floor / ms if ms else None,
                   "note": "floor = max(h2d bytes / measured pinned H2D rate, d2h bytes / D2H rate)"
                           " of this rank: a perfectly overlapped pipeline; 64 MiB srcnn_write / "
                           "srcnn_read copies timed alone in this run"}
            if h2d_bidir and d2h_bidir:
                fb = max(h2d / h2d_bidir, d2h / d2h_bidir) / 1e6
                out.update({"h2d_gbs_both_directions_busy": h2d_bidir,
                            "d2h_gbs_both_directions_busy": d2h_bidir,
                            "floor_ms_both_directions_busy": fb,
                            "frac_of_floor_both_directions_busy": fb / ms if ms else None})
            return out

        windows = {}

        # ---------------------------------------------------------------- C3 inference (primary)
        if "c3" in wl:
            cfg = NETS["c3"]
            pad = net_pad(cfg)
            rng = np.random.default_rng(1234)
            net = pkg.Net(ctx, *cfg, synthetic_params(cfg))
            h3 = w3 = IMG - pad
            r0, r1 = pkg.row_bands(h3, world)[rank]
            band_h = r1 - r0 + pad
            R = 4
            img = pkg.PinnedBuffer((IMG, IMG))
            img.array[:] = luma_image(rng, IMG, IMG)
            out_host = pkg.PinnedBuffer((r1 - r0, w3))
            ins, outs = [], []
            for i in range(R):
                m = ctx.alloc(4 * band_h * IMG)
                ctx.write(m, np.roll(img.array[r0:r0 + band_h], i, axis=1))
                ins.append(m)
                outs.append(ctx.alloc(4 * (r1 - r0) * w3))
            assert net.fused_supported()

            def infer_step(i):
                net.forward_fused(ins[i % R], outs[i % R], IMG, band_h, 1)

            def infer_e2e_step(i):
                net.infer_rows_host(img.array, IMG, IMG, r0, r1, out_host.array)

            windows["c3"] = [time.time(), None]      # clocks: samples of the timed loops only
            inf_ms, inf_launches = timed(infer_step, args.steps, args.warmup)
            if dump:
                last = outs[(args.warmup + args.steps - 1) % R]
                dumps["c3_forward_fused"] = dump_sample(ctx.read(last, (r1 - r0, w3)))
            e2e_ms, _ = timed(infer_e2e_step, args.steps, 3)

            # a STREAM of images through the non-blocking entry: up to two calls in flight, so
            # the download of step i overlaps the upload / first launches of step i+1; every
            # step still uploads its input and downloads its result inside the timed region,
            # which ends after srcnn_block has seen the last result arrive
            out_host2 = pkg.PinnedBuffer((r1 - r0, w3))
            outs_h = [out_host, out_host2]

            def infer_stream(steps, warmup):
                for i in range(warmup):
                    net.infer_rows_host(img.array, IMG, IMG, r0, r1, outs_h[i % 2].array, block=False)
                ctx.block()
                barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for i in range(steps):
                    net.infer_rows_host(img.array, IMG, IMG, r0, r1, outs_h[i % 2].array, block=False)
                ctx.block()
                e1.record(stream)
                barrier()
                return max_over_ranks(e0.elapsed_time(e1)) / steps

            e2e_stream_ms = infer_stream(args.steps, 3)
            assert np.array_equal(out_host.array, out_host2.array)
            if dump:
                dumps["c3_infer_rows_host"] = dump_sample(outs_h[(args.steps - 1) % 2].array)
            out_host2.free()
            res["c3"] = dict(ms=inf_ms, launches=inf_launches, e2e_ms=e2e_ms,
                             e2e_stream_ms=e2e_stream_ms, rows=(r0, r1),
                             band_h=band_h, h2d=4 * band_h * IMG, d2h=4 * (r1 - r0) * w3)
            windows["c3"][1] = time.time()
            for m in ins + outs:
                ctx.release(m)
            img.free()
            out_host.free()

        # ---------------------------------------------------------------- training (C2 weak, C4 strong)
        def train_workload(key, n_loc, n_global):
            cfg = NETS[key]
            grad = torch.zeros(sum(f * f * k * n + n for (k, n, f) in
                                   [(1, cfg[0], cfg[2]), (cfg[0], cfg[1], cfg[3]), (cfg[1], 1, cfg[4])]),
                               device="cuda", dtype=torch.float32)
            gh = ctx.wrap(grad.data_ptr(), grad.numel() * 4)
            net = pkg.Net(ctx, *cfg, synthetic_params(cfg), grad_flat=gh)
            px = pkg.PinnedBuffer((n_loc, PATCH, PATCH))
            pg = pkg.PinnedBuffer((n_loc, PATCH, PATCH))
            rng_r = np.random.default_rng(99 + rank)
            px.array[:], pg.array[:] = patches(rng_r, n_loc, PATCH, PATCH)
            # 9-5-5: 3028 patches = 592 strips of 128 virtual columns = 4 full waves of 148 CTAs (and a
            # multiple of 4 samples, which keeps every chunk of the sample array 16-byte aligned)
            chunk = min(args.chunk if key == "c2" else args.chunk_c4, n_loc)
            d_in, d_gt = ctx.alloc(px.nbytes), ctx.alloc(pg.nbytes)
            ctx.write(d_in, px.array)
            ctx.write(d_gt, pg.array)
            work = ctx.alloc(net.train_workspace_bytes(PATCH, PATCH, chunk))
            bytes_per = 4 * PATCH * PATCH
            base_i, base_g = ctx.mem_ptr(d_in), ctx.mem_ptr(d_gt)
            chunks = []
            for i in range(0, n_loc, chunk):
                S = min(chunk, n_loc - i)
                chunks.append((ctx.wrap(base_i + i * bytes_per, S * bytes_per),
                               ctx.wrap(base_g + i * bytes_per, S * bytes_per), S))
            params_host = pkg.PinnedBuffer((grad.numel(),))

            def train_step(i):
                for (ci, cg, S) in chunks:
                    net.train_chunk(ci, cg, PATCH, PATCH, S, work)
                net.allreduce_grads()       # the ONE exchange step of the path (no-op on 1 rank)
                net.update_all(n_global, MOMENTUM, DECAY, LR)

            def train_e2e_step(i):
                # HOST samples in (pinned), upload of chunk i+1 overlapping the training of chunk i
                net.train_chunks_host(px.array, pg.array, PATCH, PATCH, chunk, work)
                net.allreduce_grads()
                net.update_all(n_global, MOMENTUM, DECAY, LR)
                off = 0
                for l in range(3):     # read the updated parameters back (the step's result)
                    for hnd, cnt in ((net.c.w[l], net.sizes[l][0]), (net.c.b[l], net.sizes[l][1])):
                        ctx.L.srcnn_read(ctx.h, hnd, 0, 4 * cnt, params_host.ptr + 4 * off, 0)
                        off += cnt
                ctx.block()

            windows[key] = [time.time(), None]
            ms, launches = timed(train_step, args.steps, args.warmup)
            if dump:
                p = net.params()
                dumps[key + "_train_chunk_params"] = np.concatenate(
                    [p["%s%d" % (t, l)] for l in (1, 2, 3) for t in ("w", "b")])
            e2e_ms, _ = timed(train_e2e_step, args.steps, 3)
            if dump:
                dumps[key + "_train_chunks_host_params"] = params_host.array.copy()
            windows[key][1] = time.time()
            # per-kernel-id device time of ONE epoch through a profiling context (not the timed run)
            kern = None
            if rank == 0:
                pctx = pkg.Context(local_rank, profile=True)
                pnet = pkg.Net(pctx, *cfg, synthetic_params(cfg))
                pS = chunks[0][2]
                pin_, pgt_ = pctx.upload(px.array[:pS]), pctx.upload(pg.array[:pS])
                pwork = pctx.alloc(pnet.train_workspace_bytes(PATCH, PATCH, pS))
                pnet.train_chunk(pin_, pgt_, PATCH, PATCH, pS, pwork)     # warm-up
                before = pctx.profile()
                pnet.train_chunk(pin_, pgt_, PATCH, PATCH, pS, pwork)
                after = pctx.profile()
                kern = {k: {"ms": (after[k][0] - before[k][0]) / 1e6,
                            "launches": after[k][1] - before[k][1]}
                        for k in after if after[k][1] != before[k][1]}
                kern["_chunk_patches"] = pS
                pctx.close()
            out = dict(ms=ms, launches=launches, e2e_ms=e2e_ms, steps=args.steps, chunk=chunk,
                       n_loc=n_loc, n_global=n_global, grad_floats=grad.numel(), kernels=kern,
                       h2d=2 * n_loc * bytes_per, d2h=4 * grad.numel())
            for m in (d_in, d_gt, work):
                ctx.release(m)
            px.free()
            pg.free()
            params_host.free()
            return out

        if "c2" in wl:
            res["c2"] = train_workload("c2", C2_PATCHES_PER_RANK, C2_PATCHES_PER_RANK * world)
        if "c4" in wl:
            res["c4"] = train_workload("c4", C4_PATCHES_TOTAL // world, C4_PATCHES_TOTAL)

        # ---------------------------------------------------------------- C5 frames
        if "c5" in wl:
            cfg = NETS["c5"]
            pad = net_pad(cfg)
            net = pkg.Net(ctx, *cfg, synthetic_params(cfg))
            n_loc = C5_FRAMES_TOTAL // world
            w3, h3 = C5_W - pad, C5_H - pad
            rng = np.random.default_rng(77 + rank)
            fin = pkg.PinnedBuffer((n_loc, C5_H, C5_W))
            fin.array[:] = frames_like(rng, n_loc, C5_H, C5_W)
            fout = pkg.PinnedBuffer((n_loc, h3, w3))
            G = 4
            d_in = ctx.alloc(fin.nbytes)
            ctx.write(d_in, fin.array)
            d_out = ctx.alloc(fout.nbytes)
            bi, bo = ctx.mem_ptr(d_in), ctx.mem_ptr(d_out)
            groups = []
            for f0 in range(0, n_loc, G):
                S = min(G, n_loc - f0)
                groups.append((ctx.wrap(bi + 4 * f0 * C5_W * C5_H, 4 * S * C5_W * C5_H),
                               ctx.wrap(bo + 4 * f0 * w3 * h3, 4 * S * w3 * h3), S))

            def frames_step(i):
                for gi, go, S in groups:
                    net.forward_fused(gi, go, C5_W, C5_H, S)

            def frames_e2e_step(i):
                net.infer_frames_host(fin.array, C5_W, C5_H, fout.array)

            windows["c5"] = [time.time(), None]
            ms, launches = timed(frames_step, args.steps, args.warmup)
            if dump:
                # into fout, which the host-buffer loop below overwrites: no second 2 GB array
                pkg._check(ctx.L.srcnn_read(ctx.h, d_out, 0, fout.nbytes, fout.ptr, 1))
                dumps["c5_forward_fused"] = dump_sample(fout.array)
            e2e_ms, _ = timed(frames_e2e_step, args.steps, 3)
            if dump:
                dumps["c5_infer_frames_host"] = dump_sample(fout.array)
            windows["c5"][1] = time.time()
            res["c5"] = dict(ms=ms, launches=launches, e2e_ms=e2e_ms, steps=args.steps, n_loc=n_loc,
                             h2d=fin.nbytes, d2h=fout.nbytes)
            ctx.release(d_in)
            ctx.release(d_out)
            fin.free()
            fout.free()

        clocks = sampler.stop() if rank == 0 else None
        wclocks = {k: sampler.summary(v[0], v[1]) for k, v in windows.items()} if rank == 0 else {}
        barrier()
        if world > 1:
            ctx.comm_destroy()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    sm_clock = (clocks or {}).get("sm_mhz") or 1965.0
    fp32_peak = 148 * 128 * 2 * sm_clock * 1e6 / 1e12
    line = {"metric": "srcnn_915_inference_mpix_per_s", "value": None, "unit": "MPix/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": None,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(world, wl)}

    if "c3" in res:
        c = res["c3"]
        cfg = NETS["c3"]
        pad = net_pad(cfg)
        r0, r1 = c["rows"]
        mpix = IMG * IMG / 1e6 / (c["ms"] / 1e3)
        e2e_mpix = IMG * IMG / 1e6 / (c["e2e_ms"] / 1e3)
        # roofline of the dominant kernel of the primary workload: one rank's launch processes
        # 1/world of the image; per-launch duration = the step time (one fused launch + a ~3 us
        # gated fallback launch per step, CUDA events on the launching stream)
        frac_img = (r1 - r0) / float(IMG - pad)
        alg_bytes = 4.0 * (IMG * IMG + (IMG - pad) ** 2) * frac_img
        alg_flop = fwd_flop(cfg, IMG, IMG) * frac_img
        achieved_gbs = alg_bytes / (c["ms"] / 1e3) / 1e9
        achieved_tf = alg_flop / (c["ms"] / 1e3) / 1e12
        impl = os.environ.get("SRCNN_FUSED_IMPL", "hp")
        split = 6.0 if impl == "pl" else 3.0
        traffic, traffic_src = ncu_traffic("forward_fused_hp_kernel<0, 0>")
        if impl == "simt":
            roofline = {"kernel": "forward_fused_kernel (FP32 SIMT)", "bound": "hbm",
                        "achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s",
                        "frac": achieved_gbs / hbm_peak, "traffic": None, "peak_kind": peak_kind,
                        "fp32": {"achieved_tflops": achieved_tf, "peak_tflops": fp32_peak,
                                 "frac": achieved_tf / fp32_peak}}
        else:
            roofline = {
                "kernel": ("forward_fused_hp_kernel (tcgen05 kind::f16, FP16-split operands, all "
                           "three layers)" if split == 3.0 else
                           "forward_fused_pl_kernel (tcgen05 3xTF32, all three layers)"),
                "bound": "tensor", "achieved": achieved_tf, "peak": bf16_peak, "unit": "TFLOP/s",
                "frac": achieved_tf / bf16_peak,
                "traffic": traffic * frac_img if traffic else None, "traffic_source": traffic_src,
                "peak_kind": peak_kind + " dense bf16 (MEASURED_PEAKS.json)",
                "algorithmic_flop_per_launch": alg_flop,
                "precision_ceiling_tflops": bf16_peak / split,
                "frac_of_precision_ceiling": achieved_tf / (bf16_peak / split),
                "note": "algorithmic FP32 FLOPs / launch time against the measured bf16 peak; the "
                        "split-operand scheme the 1e-4 tolerance requires issues 3 tensor-core "
                        "products per FP32 product, so peak/%d is the ceiling at this precision" % split,
                "hbm": {"achieved_gbs": achieved_gbs, "peak_gbs": hbm_peak,
                        "frac": achieved_gbs / hbm_peak,
                        "algorithmic_bytes_per_launch": alg_bytes}}
            if split == 3.0 and world == 1:
                # what the MMA operand traffic of the scheme allows (profiles/r2zb_cta2_probe.txt):
                # per 128-pixel tile 6 x (67 + 51) cycles of shared-memory operand fetch for layer
                # 1 and 12 x 60 cycles of TMEM operand reads for layers 2 and 3
                strips, rows = -(-(IMG - 12) // 124), IMG - 12
                sms = torch.cuda.get_device_properties(0).multi_processor_count
                best = None     # the launcher's band-height rule (fused_forward_pl.cuh: rows_per_cta)
                for nb in range(1, min(512, rows) + 1):
                    r = -(-rows // nb)
                    cost = -(-(strips * -(-rows // r)) // sms) * (r + 4 + 8)
                    if best is None or cost < best[0]:
                        best = (cost, r)
                bands = -(-rows // best[1])
                tiles_per_sm = strips * (rows + 4 * bands) / sms
                mhz = (wclocks.get("c3") or {}).get("sm_mhz") or 1965.0
                cyc = c["ms"] * 1e-3 * mhz * 1e6 / tiles_per_sm
                # tensor-pipe time of a tile's 24 MMA instructions, each timed alone on the B200
                # (tools/probe/ts_probe.cu): A and B in shared memory 67.7 / 51.5 cycles at
                # N = 128 / 64 (operand fetch at 128 B/clk), A in tensor memory 35.9 / 20.5 at
                # N = 64 / 32 (math-bound)
                pipe = 6 * (67.7 + 51.5) + 6 * (35.9 + 20.5)
                roofline["mma_pipe_model"] = {
                    "cycles_per_tile_model": pipe, "cycles_per_tile": cyc,
                    "frac": pipe / cyc, "tiles_per_sm": tiles_per_sm,
                    "source": "profiles/r3d_ts_probe.txt, profiles/r3e_hp_prof_blocks.txt",
                    "note": "the kernel's tile period against the tensor-pipe time of its 24 MMA "
                            "instructions per tile measured in isolation (ncu's sm__pipe_tc_cycles_active "
                            "of the kernel agrees: 61.5 %); the rest of the period is the hand-off "
                            "chain between the roles, not the pipe; launch and prologue time is "
                            "inside cycles_per_tile"}
        line.update({"value": mpix, "ms_per_step": c["ms"], "gpu_launches": int(c["launches"]),
                     "roofline": roofline,
                     "e2e": {"value": e2e_mpix, "unit": "MPix/s", "ms_per_step": c["e2e_ms"],
                             "h2d_bytes_per_step": c["h2d"], "d2h_bytes_per_step": c["d2h"],
                             "mode": "one blocking srcnn_infer_rows_host call per step: pinned "
                                     "host image in, pinned host result out",
                             "stream_of_images": {
                                 "value": IMG * IMG / 1e6 / (c["e2e_stream_ms"] / 1e3),
                                 "ms_per_step": c["e2e_stream_ms"],
                                 "note": "the same steps through srcnn_infer_rows_host_async, two "
                                         "calls in flight and one srcnn_block after the last step: "
                                         "the tail of a call overlaps the head of the next"},
                             "pcie": pcie_block(c["h2d"], c["d2h"], c["e2e_ms"])}})
    # the primary workload's own window (the whole-run record is kept beside it: the training and
    # frame workloads are long tensor-bound runs that can sit at the 1000 W power cap)
    line["clocks"] = wclocks.get("c3") if wclocks.get("c3", {}).get("samples") else clocks
    line["clocks_whole_run"] = clocks
    line["config"]["numa_node_rank0"] = numa_node

    for key, name, metric in (("c2", "train", "srcnn_915_train_patches_per_s"),
                              ("c4", "train_c4", "srcnn_955_train_patches_per_s")):
        if key not in res:
            continue
        t = res[key]
        cfg = NETS[key]
        pps = t["n_global"] / (t["ms"] / 1e3)
        e2e_pps = t["n_global"] / (t["e2e_ms"] / 1e3)
        bpp = train_bytes_per_patch(cfg)
        total_bpp = float(sum(bpp.values()))
        gbs = total_bpp * t["n_loc"] / (t["ms"] / 1e3) / 1e9        # this rank's HBM stream
        flop = train_flop_per_patch(cfg)
        tf = flop * pps / world / 1e12
        tensor_frac = tf / (bf16_peak / 3.0)
        block = {"metric": metric, "value": pps, "unit": "patches/s", "ms_per_step": t["ms"],
                 "steps": t["steps"], "scaling": "weak" if key == "c2" else "strong",
                 "patches_per_step": t["n_global"], "patches_per_gpu": t["n_loc"],
                 "chunk": t["chunk"], "gpu_launches": int(t["launches"]),
                 "allreduce_floats": t["grad_floats"],
                 "roofline": {
                     "bound": "hbm" if key == "c2" else "tensor",
                     "achieved": gbs if key == "c2" else tf,
                     "peak": hbm_peak if key == "c2" else bf16_peak / 3.0,
                     "unit": "GB/s" if key == "c2" else "TFLOP/s",
                     "frac": gbs / hbm_peak if key == "c2" else tensor_frac,
                     "algorithmic_bytes_per_patch": total_bpp,
                     "algorithmic_bytes_per_patch_by_kernel": bpp,
                     "algorithmic_flop_per_patch": flop,
                     "hbm_gbs_per_gpu": gbs, "hbm_frac": gbs / hbm_peak,
                     "tflops_per_gpu": tf, "tensor_frac_of_split_ceiling": tensor_frac,
                     "note": ("whole-step figure per GPU: every activation / delta tensor the "
                              "backward needs written once and read once per consumer kernel, / "
                              "step time, against the measured HBM peak" if key == "c2" else
                              "whole-step figure per GPU: algorithmic FP32 FLOPs / step time against "
                              "bf16 peak / 3 (split operands); the 5x5 layer-2 contractions are "
                              "87% of the FLOPs")},
                 "e2e": {"value": e2e_pps, "unit": "patches/s", "ms_per_step": t["e2e_ms"],
                         "h2d_bytes_per_step": t["h2d"], "d2h_bytes_per_step": t["d2h"],
                         "pcie": pcie_block(t["h2d"], t["d2h"], t["e2e_ms"])}}
        block["clocks"] = wclocks.get(key)
        if t["kernels"]:
            k = dict(t["kernels"])
            pS = k.pop("_chunk_patches")
            block["kernels_one_chunk"] = {"patches": pS, "by_kernel_id": k,
                                          "note": "device time per C-ABI kernel id for one chunk, "
                                                  "cudaEvent pairs in a separate profiling context "
                                                  "(launches serialised); not the timed run"}
        line[name] = block

    if "c5" in res:
        c = res["c5"]
        cfg = NETS["c5"]
        mp = C5_FRAMES_TOTAL * C5_W * C5_H / 1e6
        tf = fwd_flop(cfg, C5_W, C5_H) * c["n_loc"] / (c["ms"] / 1e3) / 1e12
        traffic, traffic_src = ncu_traffic("forward_fused_hpw_kernel<0>")
        line["c5"] = {"metric": "srcnn_915_wide_frames_mpix_per_s", "value": mp / (c["ms"] / 1e3),
                      "unit": "MPix/s", "ms_per_step": c["ms"], "steps": c["steps"],
                      "scaling": "strong", "frames_per_step": C5_FRAMES_TOTAL,
                      "frames_per_gpu": c["n_loc"], "frame": [C5_W, C5_H],
                      "ms_per_frame": c["ms"] / c["n_loc"], "gpu_launches": int(c["launches"]),
                      "roofline": {"kernel": "forward_fused_hpw_kernel (tcgen05 kind::f16, FP16-split)",
                                   "bound": "tensor", "achieved": tf, "peak": bf16_peak,
                                   "unit": "TFLOP/s", "frac": tf / bf16_peak,
                                   "precision_ceiling_tflops": bf16_peak / 3.0,
                                   "frac_of_precision_ceiling": tf / (bf16_peak / 3.0),
                                   "traffic": traffic, "traffic_source": traffic_src},
                      "clocks": wclocks.get("c5"),
                      "e2e": {"value": mp / (c["e2e_ms"] / 1e3), "unit": "MPix/s",
                              "ms_per_step": c["e2e_ms"], "h2d_bytes_per_step": c["h2d"],
                              "d2h_bytes_per_step": c["d2h"],
                              "pcie": pcie_block(c["h2d"], c["d2h"], c["e2e_ms"])}}

    if dump:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumps.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)

    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(args, wl)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def cpu_baseline(args, wl):
    """oracle/_ref (the reference's kernels on the host cores) timed on a bounded sample."""
    a = argparse.Namespace(**vars(args))
    a.steps, a.warmup = 2, 1
    a.ref_rows = min(args.ref_rows, 1024)
    r = reference_numbers(a, wl)
    out = {"value": r.get("c3", {}).get("mpix"), "unit": "MPix/s", "cores": r["cores"],
           "kind": r["kind"], "sample": r.get("c3", {}).get("sample")}
    if "c2" in r:
        out["train_patches_per_s"] = r["c2"]["patches_per_s"]
        out["train_sample"] = r["c2"]["sample"]
    if "c4" in r:
        out["train_c4_patches_per_s"] = r["c4"]["patches_per_s"]
        out["train_c4_sample"] = r["c4"]["sample"]
    if "c5" in r:
        out["c5_mpix_per_s"] = r["c5"]["mpix"]
        out["c5_sample"] = r["c5"]["sample"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workloads", default="c3,c2,c4,c5")
    ap.add_argument("--chunk", type=int, default=2048,
                    help="patches per training chunk (the reference chunks an epoch in two: "
                         "src/Main_cl.cpp:93,128-129)")
    ap.add_argument("--chunk-c4", type=int, default=3028)
    ap.add_argument("--ref-rows", type=int, default=IMG - 12,
                    help="output rows of C3 the reference arm computes per step (default: all)")
    ap.add_argument("--ref-patches", type=int, default=512)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step of each loop to DIR/*.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    wl = [w for w in args.workloads.split(",") if w]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world, wl)
    else:
        run_ours(args, rank, world, local_rank, wl)


if __name__ == "__main__":
    main()
