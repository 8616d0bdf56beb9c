#!/usr/bin/env python
"""Benchmark of the GANet guided-aggregation hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]

A "step" is one pass of the hot path -- SGA forward+backward and LGA2
forward+backward -- over one synthetic batch B x C x D x H x W = 8 x 32 x 192 x
240 x 624 (BASELINE.json; SURVEY.md 8d for the input recipe).  The batch axis is
sharded over the ranks (no data-path collective: SURVEY.md 8e); a rank walks its
shard --chunk samples (default 2) per native call.  Rank 0 prints ONE JSON line.

  value      voxels/s = (B*C*D*H*W + B*D*H*W) * K / max-over-ranks device time,
             inputs resident in HBM, timed with CUDA events on the launch stream
  e2e        the same work through the public nn.Module API starting from pinned
             HOST buffers, results copied back to the host, copies inside the
             timed region
  roofline   algorithmic bytes of the dominant op (SGA fwd+bwd: 22 + 240/D bytes per
             voxel, SURVEY.md 8d) / its device time / measured HBM peak
  cpu_baseline  the reference's own kernel bodies on the host cores (oracle/_ref) on
             a bounded sample; a reported baseline, not the target

`--impl reference` times that CPU reference arm alone on the box's host cores.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "SGA+LGA cost-volume voxels/sec (fwd+bwd) at D=192 HxW=240x624; HBM %peak"
HBM_FALLBACK_GBS = 6650.0      # /opt/skills/guides/B200_PROFILING.md fallback


# ---- arithmetic shared with tests/test_host.py ---------------------------------
def shard_samples(batch, world, rank):
    """Contiguous batch shard of rank `rank` (SURVEY.md 8e: rank r owns [r*B/G, (r+1)*B/G))."""
    lo = batch * rank // world
    hi = batch * (rank + 1) // world
    return list(range(lo, hi))


def samples_per_call(requested, n_mine, fits):
    """Samples handed to one native call: as requested, halved until `fits(count)` says the
    kept-aggregates variant has room (smaller calls beat falling back to the recompute variant)."""
    cs = max(1, min(int(requested), max(1, int(n_mine))))
    while cs > 1 and not fits(cs):
        cs //= 2
    return cs


def sga_bytes_per_voxel(D):
    """SGA fwd (9 + 80/D) + bwd (13 + 160/D) algorithmic bytes per voxel (SURVEY.md 8d)."""
    return 22.0 + 240.0 / D


def lga2_bytes_per_voxel(D):
    """LGA2 fwd (8 + 300/D) + bwd (12 + 600/D) algorithmic bytes per voxel (SURVEY.md 8d)."""
    return 20.0 + 900.0 / D


def dist_setup(backend, device=None):
    """One process per GPU (torchrun env); returns (world, rank, local_rank)."""
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        kw = {"device_id": device} if (backend == "nccl" and device is not None) else {}
        dist.init_process_group(backend, **kw)
    return world, rank, local_rank


def _parse_cpulist(text):
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        lo, _, hi = part.partition("-")
        cpus.update(range(int(lo), int(hi or lo) + 1))
    return cpus


def bind_to_gpu_numa_node(index):
    """Pin this process to the CPUs of the NUMA node its GPU hangs off (PCI bus id ->
    /sys/bus/pci/devices/*/numa_node -> node cpulist), BEFORE any pinned host buffer is allocated, so
    that the buffers are first-touched on that node and the copy threads run next to it.  Without
    this, ranks 4-7 of an 8-GPU box stage through the far socket (round 1: 42 -> 21 GB/s per GPU).
    Returns a small record for the JSON line; any failure leaves the affinity untouched."""
    info = {"gpu": index, "numa_node": None, "cpus": None}
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=pci.bus_id",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=20).stdout
        bus = out.strip().splitlines()[0].strip().lower()          # 00000000:1B:00.0
        dom, rest = bus.split(":", 1)
        path = "/sys/bus/pci/devices/%s:%s/numa_node" % (dom[-4:], rest)
        with open(path) as fh:
            node = int(fh.read().strip())
        info["pci_bus_id"] = bus
        if node < 0:
            return info
        with open("/sys/devices/system/node/node%d/cpulist" % node) as fh:
            cpus = _parse_cpulist(fh.read())
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
            info["numa_node"], info["cpus"] = node, len(allowed)
    except Exception as exc:       # noqa: BLE001
        info["error"] = "%s: %s" % (type(exc).__name__, exc)
    return info


def max_over_ranks(value, world, device="cpu"):
    """Job time = the slowest rank's device time (never a wall clock)."""
    if world == 1:
        return float(value)
    import torch
    import torch.distributed as dist
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(value, world, device="cpu"):
    if world == 1:
        return float(value)
    import torch
    import torch.distributed as dist
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--channels", type=int, default=32)
    ap.add_argument("--depth", type=int, default=192)
    ap.add_argument("--height", type=int, default=240)
    ap.add_argument("--width", type=int, default=624)
    ap.add_argument("--chunk", type=int, default=2,
                    help="samples handed to the SGA/LGA entry points per call")
    ap.add_argument("--config", type=int, default=None, choices=[2, 3, 4],
                    help="BASELINE.json config 2/3/4: the reference's models on the new operators "
                         "(baseline/model_bench.py); default: the headline microbenchmark")
    ap.add_argument("--per-gpu-batch", type=int, default=1, help="--config 2-4: samples per GPU")
    ap.add_argument("--fuse-sga-blocks", action="store_true",
                    help="--config 2-4: also time the model with the fused SGABlock prologue (ganet_b200.fused)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-gpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed to DIR/<name>.npy "
                         "(float32; see dump_positions for the sample kept of a large output)")
    return ap.parse_args()


def load_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


def load_traffic():
    """DRAM bytes per voxel of the dominant op from the committed ncu capture, or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            return json.load(fh)
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, smax, reasons = [], [], set()
        for line in out.splitlines():
            f = [v.strip() for v in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---- the reference's CPU implementation (oracle/_ref, else the oracle port) -------
def physical_cores():
    """Physical cores of the host (unique (package, core) pairs); falls back to os.cpu_count()."""
    try:
        seen, phys, core = set(), None, None
        with open("/proc/cpuinfo") as fh:
            for line in fh:
                if line.startswith("physical id"):
                    phys = line.split(":")[1].strip()
                elif line.startswith("core id"):
                    core = line.split(":")[1].strip()
                elif not line.strip():
                    if phys is not None and core is not None:
                        seen.add((phys, core))
                    phys = core = None
        if seen:
            return len(seen)
    except OSError:
        pass
    return os.cpu_count() or 1


def host_memory_policy(mode):
    """Placement of the CPU arm's arrays on a multi-socket host.  The reference's kernel bodies run under an
    OpenMP loop over all cores, but numpy first-touches every array from ONE thread, i.e. on one NUMA node:
    half the threads then work on remote memory (measured on a 2 x 32-core box: 3.5 s per SGA sample against
    2.2 s for the same 64 threads confined to one socket).  `local` (the default) confines the process to NUMA
    node 0's CPUs; `interleave` spreads the pages over all nodes (set_mempolicy(MPOL_INTERLEAVE), what
    `numactl --interleave=all` does); `default` leaves the kernel's first-touch policy.  Measured on the pool's
    2 x 32-core hosts, whole arm, 64 threads: local 26.4, interleave 16.8, default 16.1 Mvoxel/s (128 threads,
    interleaved: 13.3) -- so the arm runs the configuration that serves the reference best.  Also undoes an
    inherited CPU affinity first, so that the arm measures the same thing standalone and as bench.py's child."""
    info = {"policy": mode}
    try:
        os.sched_setaffinity(0, range(os.cpu_count() or 1))
    except OSError:
        pass
    try:
        nodes = sorted(int(d[4:]) for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit())
    except OSError:
        nodes = [0]
    info["nodes"] = len(nodes)
    if mode == "interleave" and len(nodes) > 1:
        import ctypes
        mask = ctypes.c_ulong(sum(1 << n for n in nodes))
        rc = ctypes.CDLL(None, use_errno=True).syscall(238, 3, ctypes.byref(mask), ctypes.c_ulong(64))   # set_mempolicy, MPOL_INTERLEAVE
        info["set_mempolicy_rc"] = int(rc)
    elif mode == "local" and len(nodes) > 1:
        try:
            with open("/sys/devices/system/node/node%d/cpulist" % nodes[0]) as fh:
                cpus = _parse_cpulist(fh.read())
            os.sched_setaffinity(0, cpus)
            info["cpus"] = len(cpus)
        except OSError:
            pass
    return info


def pin_openmp_env():
    """One OpenMP thread per physical core, bound (OMP_PLACES=cores, OMP_PROC_BIND=close): must be in
    the environment before libgomp initialises, i.e. before numpy / the oracle libraries load.
    Explicit user settings win."""
    os.environ.setdefault("OMP_NUM_THREADS", str(physical_cores()))
    os.environ.setdefault("OMP_PLACES", "cores")
    os.environ.setdefault("OMP_PROC_BIND", "close")


def cpu_reference_sample(depth, height, width):
    """One bounded sample of the workload on the host cores with the reference's own kernel bodies
    (oracle/_ref; the oracle port if the reference was not compiled here): SGA fwd+bwd on
    (1, 2, D, H, W) -- the sample SURVEY.md 8d specifies: two full (n,c) slices, so the scan kernels
    expose 2*H resp. 2*W lines to the host threads -- and LGA2 fwd+bwd on (1, D, H, W).  FIXED shapes
    (no calibration), so every step and every box measures the same thing."""
    import numpy as np
    from oracle import api as port
    from oracle import ref_cpu
    use_ref = ref_cpu.available()
    rng = np.random.default_rng(0)

    def l1(a, axis):
        return (a / np.abs(a).sum(axis=axis, keepdims=True)).astype(np.float32)

    cs = 2
    while cs > 1 and cs * depth * height * width >= 2 ** 31:      # the reference indexes with int
        cs -= 1
    sga_shape = (1, cs, depth, height, width)
    lga_shape = (1, depth, height, width)
    N, C, D, H, W = sga_shape
    x = rng.standard_normal(sga_shape).astype(np.float32)
    g = [l1(rng.standard_normal((N, C, 5, H, W)), 2) for _ in range(4)]
    go = rng.standard_normal(sga_shape).astype(np.float32)
    t0 = time.perf_counter()
    if use_ref:
        out, mask, temp = ref_cpu.sga_forward(x, *g)
        ref_cpu.sga_backward(x, *g, temp, mask, go)
    else:
        out, mask = port.sga_forward(x, *g, fused=False)
        port.sga_backward(x, *g, mask, go, fused=False)
    t_sga = time.perf_counter() - t0
    del x, g, go, out, mask
    xl = rng.standard_normal(lga_shape).astype(np.float32)
    fl = l1(rng.standard_normal((1, 75) + lga_shape[2:]), 1)
    gol = rng.standard_normal(lga_shape).astype(np.float32)
    t0 = time.perf_counter()
    if use_ref:
        y, y1 = ref_cpu.lga2_forward(xl, fl)
        ref_cpu.lga2_backward(xl, fl, y1, gol)
    else:
        y, tmp = port.lga_forward(xl, fl, 2, 2)
        port.lga_backward(xl, fl, tmp, gol, 2, 2)
    t_lga = time.perf_counter() - t0
    return {
        "r_sga": float(np.prod(sga_shape) / t_sga), "r_lga": float(np.prod(lga_shape) / t_lga),
        "t_sga": t_sga, "t_lga": t_lga, "cores": os.cpu_count() or 1,
        "threads": int(os.environ.get("OMP_NUM_THREADS", "0")) or (os.cpu_count() or 1),
        "omp": {k: os.environ.get(k) for k in ("OMP_NUM_THREADS", "OMP_PLACES", "OMP_PROC_BIND")},
        "kind": "reference" if use_ref else "port",
        "sample": "SGA fwd+bwd on %s + LGA2 fwd+bwd on %s per step (fixed shapes), rates combined in "
                  "the workload's voxel proportions" % ("x".join(map(str, sga_shape)),
                                                       "x".join(map(str, lga_shape))),
    }


def cpu_config1():
    """BASELINE.json config 1 -- a single SGA forward on 1x8x48x48x96, the reference's own
    CPU-runnable case -- timed on the host cores with whatever thread count is set."""
    import numpy as np
    from oracle import api as port
    from oracle import ref_cpu
    rng = np.random.default_rng(1)
    shape = (1, 8, 48, 48, 96)
    x = rng.standard_normal(shape).astype(np.float32)
    g = []
    for _ in range(4):
        a = rng.standard_normal((1, 8, 5, 48, 96))
        g.append((a / np.abs(a).sum(axis=2, keepdims=True)).astype(np.float32))
    fwd = ref_cpu.sga_forward if ref_cpu.available() else (lambda *t: port.sga_forward(*t, fused=False))
    fwd(x, *g)
    best = None
    for _ in range(3):
        t0 = time.perf_counter()
        fwd(x, *g)
        dt = time.perf_counter() - t0
        best = dt if best is None or dt < best else best
    return {"workload": "SGA forward on 1x8x48x48x96 (BASELINE.json config 1)", "ms": 1e3 * best,
            "voxels_per_s": float(np.prod(shape) / best)}


def combine_rates(v_sga, v_lga, r_sga, r_lga):
    return (v_sga + v_lga) / (v_sga / r_sga + v_lga / r_lga)


def run_reference_arm(a):
    """`--impl reference`: the reference's own CPU implementation of the path on the
    host cores, K bounded steps after W warm-ups (each step = cpu_reference_sample).  Rank 0 only.
    `value` is the MEDIAN step; `ms_per_step` is what one full-workload step would take at that rate
    (an extrapolation, flagged), `measured_s_per_step` what a bounded step really took."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    B, C, D, H, W = a.batch, a.channels, a.depth, a.height, a.width
    v_sga, v_lga = B * C * D * H * W, B * D * H * W
    vals, secs, info = [], [], None
    t_begin = time.perf_counter()
    for i in range(a.warmup + a.steps):
        info = cpu_reference_sample(D, H, W)
        if i >= a.warmup:
            vals.append(combine_rates(v_sga, v_lga, info["r_sga"], info["r_lga"]))
            secs.append(info["t_sga"] + info["t_lga"])
    wall = time.perf_counter() - t_begin
    value = statistics.median(vals)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "voxels/s",
        "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": 1e3 * (v_sga + v_lga) / value, "ms_per_step_extrapolated": True,
        "measured_s_per_step": statistics.median(secs),
        "value_min_max": [min(vals), max(vals)],
        "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "SGA+LGA2 fwd+bwd, B=%d C=%d D=%d HxW=%dx%d (CPU arm: bounded "
                               "sample per step)" % (B, C, D, H, W)},
        "cpu_baseline": {"value": value, "unit": "voxels/s", "cores": info["cores"],
                         "threads": info["threads"], "omp": info["omp"], "kind": info["kind"],
                         "host_memory": getattr(a, "host_memory", None), "sample": info["sample"]},
        "e2e": {"value": value, "unit": "voxels/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "config1_cpu": cpu_config1(),
        "gpu_launches": 0, "wall_s": wall,
    }
    print(json.dumps(line))
    return 0


def cpu_baseline_leg(a):
    """The cpu_baseline object of our arm's line: the reference arm itself, in a child process so that
    its OpenMP runtime starts with the pinned-thread environment (torch has already initialised
    libgomp in this one), 1 warm-up + 2 bounded steps."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "2", "--warmup", "1",
           "--batch", str(a.batch), "--channels", str(a.channels), "--depth", str(a.depth),
           "--height", str(a.height), "--width", str(a.width)]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
        lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
        ref = json.loads(lines[-1])
        out = dict(ref["cpu_baseline"])
        out["measured_s_per_step"] = ref["measured_s_per_step"]
        out["config1_cpu"] = ref.get("config1_cpu")
        return out
    except Exception as exc:       # noqa: BLE001
        return {"unavailable": "%s: %s" % (type(exc).__name__, exc)}


# ---- our arm ------------------------------------------------------------------------
def make_inputs(torch, dev, samples, C, D, H, W, seed):
    """SURVEY.md 8d recipe, one sample at a time so peak memory stays bounded."""
    import torch.nn.functional as F
    n = len(samples)
    x = torch.empty((n, C, D, H, W), device=dev)
    go = torch.empty_like(x)
    g = [torch.empty((n, C, 5, H, W), device=dev) for _ in range(4)]
    xl = torch.empty((n, D, H, W), device=dev)
    gol = torch.empty_like(xl)
    fl = torch.empty((n, 75, H, W), device=dev)
    gen = torch.Generator(device=dev)
    for i, s in enumerate(samples):
        gen.manual_seed(seed * 100003 + s)
        x[i].normal_(generator=gen)
        go[i].normal_(generator=gen)
        for k in range(4):
            g[k][i].normal_(generator=gen)
            g[k][i] = F.normalize(g[k][i], p=1, dim=1)
        xl[i].normal_(generator=gen)
        gol[i].normal_(generator=gen)
        fl[i].normal_(generator=gen)
        fl[i] = F.normalize(fl[i], p=1, dim=0)
    return x, go, g, xl, gol, fl


# what one call of the timed path returns, in the order one_sample returns it
DUMP_NAMES = ("sga_out", "sga_mask", "sga_grad_x", "sga_grad_g0", "sga_grad_g1", "sga_grad_g2", "sga_grad_g3",
              "lga2_out", "lga2_grad_x", "lga2_grad_f")
DUMP_ELEMENTS = 1 << 20        # per output: 4 MB of float32, so the ten files stay below 64 MB


def dump_positions(per_sample, batch):
    """Flat positions within one sample kept by --dump-outputs: all of them when the whole output fits in
    DUMP_ELEMENTS, else the same fixed, seeded sample in every sample of the batch."""
    k = max(1, DUMP_ELEMENTS // batch)
    if per_sample <= k:
        return None
    import numpy as np
    return np.unique(np.random.default_rng(0).integers(0, per_sample, k))


class OutputDump:
    """Collects, call by call, the outputs of the last timed step on the device and writes them as DIR/<name>.npy.
    Positions and buffers are set up before the timed window, so that inside it the dump adds only asynchronous
    device gathers (ten small launches per call, so that no full-size output outlives its call), and nothing when
    --dump-outputs is not given."""

    def __init__(self, torch, dev, batch, C, D, H, W):
        per_sample = dict(zip(DUMP_NAMES, [(C, D, H, W)] * 3 + [(C, 5, H, W)] * 4 + [(D, H, W)] * 2 + [(75, H, W)]))
        self.bufs, self.shapes, self.pos = {}, {}, {}
        for name, shape in per_sample.items():
            numel = 1
            for d in shape:
                numel *= d
            p = dump_positions(numel, batch)
            self.pos[name] = None if p is None else torch.from_numpy(p).to(dev)
            self.shapes[name] = (batch,) + (shape if p is None else (len(p),))
            self.bufs[name] = torch.empty((batch, numel if p is None else len(p)), dtype=torch.float32, device=dev)

    def keep(self, first, outputs):
        flat = (outputs[0], outputs[1], outputs[2]) + tuple(outputs[3]) + tuple(outputs[4:])
        for name, t in zip(DUMP_NAMES, flat):
            n = t.shape[0]
            t = t.reshape(n, -1)
            pos = self.pos[name]
            self.bufs[name][first:first + n].copy_(t if pos is None else t.index_select(1, pos))

    def write(self, path):
        import numpy as np
        os.makedirs(path, exist_ok=True)
        for name, buf in self.bufs.items():
            np.save(os.path.join(path, name + ".npy"), buf.cpu().numpy().reshape(self.shapes[name]))


def run_ours(a):
    import torch
    import torch.distributed as dist
    from ganet_b200 import ops

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    numa = bind_to_gpu_numa_node(local_rank)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    world, rank, local_rank = dist_setup("nccl", dev)
    if a.dump_outputs and world > 1:
        raise SystemExit("bench.py: --dump-outputs writes one rank's outputs; run it with --gpus 1")
    B, C, D, H, W = a.batch, a.channels, a.depth, a.height, a.width
    mine = shard_samples(B, world, rank)
    v_sga, v_lga = B * C * D * H * W, B * D * H * W
    x, go, g, xl, gol, fl = make_inputs(torch, dev, mine, C, D, H, W, seed=0)

    ev = lambda: torch.cuda.Event(enable_timing=True)   # noqa: E731
    phase_events = []

    # The kept-aggregates variant needs 20 bytes per voxel of the call; the policy is the rule
    # SgaFunction applies under autograd (three times the buffer still free on the device).
    cs = samples_per_call(a.chunk, len(mine), lambda c: ops.keep_aggregates_policy(x[0:c], True))
    keep_flag = [None]

    def one_sample(i, record):
        s = slice(i, min(i + cs, len(mine)))
        e = [ev() for _ in range(5)] if record else None
        if record: e[0].record()
        # forward keeps the four aggregates for backward when the device has room
        # (ops.keep_aggregates_policy: the same rule SgaFunction applies under autograd)
        agg = None
        if keep_flag[0] is None:
            keep_flag[0] = ops.keep_aggregates_policy(x[s], True)
        if keep_flag[0]:
            out, mask, agg = ops.sga_forward(x[s], g[0][s], g[1][s], g[2][s], g[3][s], keep_aggregates=True)
        else:
            out, mask = ops.sga_forward(x[s], g[0][s], g[1][s], g[2][s], g[3][s])
        if record: e[1].record()
        gi, gg = ops.sga_backward(x[s], g[0][s], g[1][s], g[2][s], g[3][s], mask, go[s], aggregates=agg)
        if record: e[2].record()
        y1 = ops.lga_forward(xl[s], fl[s], 2)
        y = ops.lga_forward(y1, fl[s], 2)
        if record: e[3].record()
        g1, gf = ops.lga_backward(y1, fl[s], gol[s], 2)
        gx, gf = ops.lga_backward(xl[s], fl[s], g1, 2, grad_f=gf)
        if record:
            e[4].record()
            phase_events.append(e)
        return out, mask, gi, gg, y, gx, gf

    def step(record, dump=None):
        for i in range(0, len(mine), cs):
            outputs = one_sample(i, record)
            if dump is not None:
                dump.keep(i, outputs)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(a.warmup):
        step(False)
    sync_all()
    dump = OutputDump(torch, dev, len(mine), C, D, H, W) if a.dump_outputs else None   # before the timed window
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    t0, t1 = ev(), ev()
    t0.record()
    for k in range(a.steps):
        step(True, dump if k == a.steps - 1 else None)
    t1.record()
    sync_all()
    ms = t0.elapsed_time(t1)
    clk = clocks.stop() if rank == 0 else None
    if dump is not None:
        dump.write(a.dump_outputs)
    ms = max_over_ranks(ms, world, dev)
    done = sum_over_ranks(len(mine), world, dev)       # every sample processed exactly once
    assert int(done) == B, (done, B)
    value = (v_sga + v_lga) * a.steps / (ms * 1e-3)

    # per-phase device time on this rank (events sit on the launch stream)
    ph = [0.0, 0.0, 0.0, 0.0]
    for e in phase_events:
        for k in range(4):
            ph[k] += e[k].elapsed_time(e[k + 1])
    n_local = len(mine) * a.steps
    local_v_sga = len(mine) * C * D * H * W
    t_sga = (ph[0] + ph[1]) * 1e-3 / a.steps          # seconds per step on this rank
    peak, peak_src = load_peak()
    sga_gbs = sga_bytes_per_voxel(D) * local_v_sga / t_sga / 1e9 if t_sga > 0 else 0.0
    traffic = load_traffic()

    # launches of OUR kernels in the timed region, per native call when the workspace holds the whole
    # call in one chunk.  Horizontal scans in the standard layout (D <= 256, W % 16 == 0): SGA fwd 5
    # (four raw scans + merge) / bwd 4 with kept aggregates, fwd 4 / bwd 8 when recomputing.  Transposed
    # path: fwd 8 / bwd 11 kept, 9 / 16 recomputing.  LGA2 fwd 2, bwd 4.
    from ganet_b200 import _lib
    native = _lib.lib().ganet_sga_aggregate_volumes(*[_lib._i64(v) for v in (1, C, D, H, W)]) == 4
    if native:
        sga_launches = (5 + 4) if keep_flag[0] else (4 + 8)
    else:
        sga_launches = (8 + 11) if keep_flag[0] else (9 + 16)
    calls = a.steps * -(-len(mine) // cs)
    launches = calls * (sga_launches + 2 + 4)

    # ---- roofline of the single hottest kernel family, timed alone ------------------
    # one directional aggregate = ONE launch of the TMA scan kernel in RAW mode: reads x and the
    # guidance once, writes the aggregate once (8 + 20/D algorithmic bytes per voxel)
    kern = None
    if len(mine) > 0:
        s1 = slice(0, min(cs, len(mine)))
        vox = x[s1].numel()
        ops.sga_direction(x[s1], g[0][s1], 0)
        torch.cuda.synchronize()
        k0, k1 = ev(), ev()
        reps = 5
        k0.record()
        for r in range(reps):
            ops.sga_direction(x[s1], g[r % 2][s1], r % 2)       # down / up alternate
        k1.record()
        torch.cuda.synchronize()
        kms = k0.elapsed_time(k1) / reps
        kgbs = (8.0 + 20.0 / D) * vox / (kms * 1e-3) / 1e9
        kern = {"kernel": "sga_tma_fwd_kernel, RAW mode (one scan direction, one launch)",
                "bound": "hbm", "achieved": kgbs, "peak": peak, "unit": "GB/s", "frac": kgbs / peak,
                "ms_per_launch": kms, "voxels_per_launch": vox,
                "algorithmic_bytes_per_voxel": 8.0 + 20.0 / D}

    # ---- end to end through the public modules, from pinned host buffers ---------
    e2e = None
    if not a.no_e2e and len(mine) > 0:
        e2e = run_e2e(torch, dist, world, dev, a, mine, v_sga, v_lga)

    line = None
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "voxels/s", "n_gpus": world,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms / a.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "SGA fwd+bwd on %dx%dx%dx%dx%d + LGA2(r=2) fwd+bwd on %dx%dx%dx%d, "
                                   "batch sharded over ranks, %d samples per call"
                                   % (B, C, D, H, W, B, D, H, W, cs),
                       "global_batch": B, "parallelism": "batch-shard x%d, no data-path collective" % world,
                       "l2": "inputs larger than L2 (3.7 GB per sample, distinct per sample)",
                       "aggregates_kept_for_backward": bool(keep_flag[0])},
            "e2e": e2e, "gpu_launches": launches, "clocks": clk, "numa": numa,
            "roofline": {"bound": "hbm", "kernel": "SGA forward+backward (all launches of the call: four forward scans + merge, four reverse sweeps)",
                         "achieved": sga_gbs, "peak": peak, "unit": "GB/s",
                         "frac": sga_gbs / peak, "peak_source": peak_src,
                         "algorithmic_bytes_per_voxel": sga_bytes_per_voxel(D),
                         "traffic": traffic},
            "roofline_hottest_kernel": kern,
            "phases_ms_per_step": {"sga_fwd": ph[0] / a.steps, "sga_bwd": ph[1] / a.steps,
                                   "lga2_fwd": ph[2] / a.steps, "lga2_bwd": ph[3] / a.steps},
        }
        if world == 1 and not a.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_leg(a)
        if world == 1 and not a.no_ref_gpu:
            del x, go
            torch.cuda.empty_cache()
            line["reference_cuda_on_this_gpu"] = ref_gpu_rate(torch, dev, C, D, H, W)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def run_e2e(torch, dist, world, dev, a, mine, v_sga, v_lga):
    """Same work through the reference-facing nn.Modules with HOST buffers: per sample,
    pinned host -> device copies of every input, forward + autograd backward, results
    (outputs and all gradients) copied back to pinned host memory."""
    import torch.nn.functional as F
    from ganet_b200.modules import SGA, LGA2
    C, D, H, W = a.channels, a.depth, a.height, a.width
    sga, lga2 = SGA(), LGA2(2)
    pin = lambda *s: torch.empty(s, pin_memory=True)    # noqa: E731

    def host_randn(*s, norm_dim=None):      # generated on the device (fast), parked in pinned host memory
        t = torch.randn(*s, device=dev)
        if norm_dim is not None:
            t = F.normalize(t, p=1, dim=norm_dim)
        h = pin(*s)
        h.copy_(t)
        return h

    hx, hgo = host_randn(1, C, D, H, W), host_randn(1, C, D, H, W)
    hg = [host_randn(1, C, 5, H, W, norm_dim=2) for _ in range(4)]
    hxl, hgol = host_randn(1, D, H, W), host_randn(1, D, H, W)
    hfl = host_randn(1, 75, H, W, norm_dim=1)
    r_out, r_gi = pin(1, C, D, H, W), pin(1, C, D, H, W)
    r_gg = [pin(1, C, 5, H, W) for _ in range(4)]
    r_y, r_gx, r_gf = pin(1, D, H, W), pin(1, D, H, W), pin(1, 75, H, W)
    h2d = sum(t.numel() * 4 for t in [hx, hgo, hxl, hgol, hfl] + hg)
    d2h = sum(t.numel() * 4 for t in [r_out, r_gi, r_y, r_gx, r_gf] + r_gg)

    # Three-stage software pipeline over the samples, all through the public modules:
    #   copy-in stream : pinned host -> device inputs (double-buffered)
    #   compute stream : SGA()(...) / LGA2()(...) forward + autograd backward
    #   copy-out stream: outputs and every gradient -> pinned host
    # PCIe is full duplex, so H2D of sample i+1, compute of i and D2H of i-1 overlap.
    s_in, s_comp, s_out = (torch.cuda.Stream(dev) for _ in range(3))
    NB = 2
    dbuf = []
    for _ in range(NB):
        dbuf.append({
            "x": torch.empty(1, C, D, H, W, device=dev).requires_grad_(),
            "g": [torch.empty(1, C, 5, H, W, device=dev).requires_grad_() for _ in range(4)],
            "go": torch.empty(1, C, D, H, W, device=dev),
            "xl": torch.empty(1, D, H, W, device=dev).requires_grad_(),
            "fl": torch.empty(1, 75, H, W, device=dev).requires_grad_(),
            "gol": torch.empty(1, D, H, W, device=dev)})
    free_ev = [None] * NB                  # buffer b may be overwritten after this event
    last_out = [None]

    def run(n_samples):
        for i in range(n_samples):
            bf = dbuf[i % NB]
            with torch.cuda.stream(s_in):
                if free_ev[i % NB] is not None:
                    s_in.wait_event(free_ev[i % NB])
                with torch.no_grad():
                    bf["x"].copy_(hx, non_blocking=True)
                    bf["go"].copy_(hgo, non_blocking=True)
                    for k in range(4):
                        bf["g"][k].copy_(hg[k], non_blocking=True)
                    bf["xl"].copy_(hxl, non_blocking=True)
                    bf["fl"].copy_(hfl, non_blocking=True)
                    bf["gol"].copy_(hgol, non_blocking=True)
                ev_in = torch.cuda.Event()
                ev_in.record(s_in)
            with torch.cuda.stream(s_comp):
                s_comp.wait_event(ev_in)
                for t in [bf["x"], bf["xl"], bf["fl"]] + bf["g"]:
                    t.grad = None
                out = sga(bf["x"], *bf["g"])
                out.backward(bf["go"])
                y = lga2(bf["xl"], bf["fl"])
                y.backward(bf["gol"])
                res = [out.detach(), bf["x"].grad] + [t.grad for t in bf["g"]] + \
                      [y.detach(), bf["xl"].grad, bf["fl"].grad]
                ev_comp = torch.cuda.Event()
                ev_comp.record(s_comp)
                free_ev[i % NB] = ev_comp
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev_comp)
                for dst, src in zip([r_out, r_gi] + r_gg + [r_y, r_gx, r_gf], res):
                    src.record_stream(s_out)
                    dst.copy_(src, non_blocking=True)
                last_out[0] = torch.cuda.Event()
                last_out[0].record(s_out)

    steps = a.steps
    run(2)                                    # warm-up (allocator, both buffers)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    s_in.wait_event(e0)
    for _ in range(steps):
        run(len(mine))
    torch.cuda.current_stream().wait_event(last_out[0])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    wall = time.perf_counter() - t0
    ms = max_over_ranks(ms, world, dev)
    return {"value": (v_sga + v_lga) * steps / (ms * 1e-3), "unit": "voxels/s",
            "h2d_bytes_per_step": h2d * len(mine) * world, "d2h_bytes_per_step": d2h * len(mine) * world,
            "steps": steps, "ms_per_step": ms / steps, "wall_s": wall,
            "api": "ganet_b200.modules.SGA / LGA2 + autograd from pinned host buffers; H2D, compute and "
                   "D2H of consecutive samples overlapped on three streams"}


def ref_gpu_rate(torch, dev, C, D, H, W):
    """The UNMODIFIED reference CUDA kernels (oracle/_ref/GANet*.so) on this same GPU,
    one sample, same inputs recipe -- the number the new kernels have to beat."""
    from oracle import ref_gpu
    if not ref_gpu.available():
        return {"unavailable": "oracle/_ref/GANet*.so not built"}
    import torch.nn.functional as F
    try:
        cc = C
        while cc * D * H * W >= 2 ** 31:      # the reference indexes with int
            cc //= 2
        x = torch.randn(1, cc, D, H, W, device=dev)
        go = torch.randn_like(x)
        g = [F.normalize(torch.randn(1, cc, 5, H, W, device=dev), p=1, dim=2) for _ in range(4)]
        xl = torch.randn(1, D, H, W, device=dev)
        gol = torch.randn_like(xl)
        fl = F.normalize(torch.randn(1, 75, H, W, device=dev), p=1, dim=1)

        def once():
            out, mask, temp = ref_gpu.sga_forward(x, *g)
            ref_gpu.sga_backward(x, *g, temp, mask, go)

        def once_lga():
            y, y1 = ref_gpu.lga2_forward(xl, fl)
            ref_gpu.lga2_backward(xl, fl, y1, gol)

        once(); once_lga()
        torch.cuda.synchronize()
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record(); once(); e[1].record(); once_lga(); e[2].record()
        torch.cuda.synchronize()
        t_sga, t_lga = e[0].elapsed_time(e[1]) * 1e-3, e[1].elapsed_time(e[2]) * 1e-3
        v_sga, v_lga = cc * D * H * W, D * H * W
        r_sga, r_lga = v_sga / t_sga, v_lga / t_lga
        return {"value": combine_rates(C * D * H * W, D * H * W, r_sga, r_lga), "unit": "voxels/s",
                "sga_ms_per_sample": t_sga * 1e3 * C / cc, "lga2_ms_per_sample": t_lga * 1e3,
                "sample": "1x%dx%dx%dx%d SGA fwd+bwd, 1x%dx%dx%d LGA2 fwd+bwd, allocations included "
                          "as in functions/GANet.py" % (cc, D, H, W, D, H, W)}
    except Exception as exc:           # noqa: BLE001
        return {"unavailable": "%s: %s" % (type(exc).__name__, exc)}


def main():
    a = parse_args()
    if a.dump_outputs and (a.config is not None or a.impl != "ours"):
        raise SystemExit("bench.py: --dump-outputs applies to the headline workload of --impl ours")
    if a.config is not None:
        if a.impl == "reference":
            if int(os.environ.get("RANK", "0")) == 0:
                print(json.dumps({"impl": "reference", "config_id": a.config,
                                  "unavailable": "the reference has no CPU path for its models; its CUDA "
                                                 "kernels on this GPU are timed inside `--config %d` "
                                                 "(reference_cuda_on_this_gpu)" % a.config}))
            return 0
        from baseline import model_bench
        return model_bench.run(a)
    if a.impl == "reference":
        pin_openmp_env()              # before numpy / libgomp load
        a.host_memory = host_memory_policy(os.environ.get("GANET_CPU_ARM_MEMORY", "local"))
        return run_reference_arm(a)
    return run_ours(a)


if __name__ == "__main__":
    sys.exit(main())
