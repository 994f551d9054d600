#!/usr/bin/env python
"""bench.py -- whole-job throughput of the B200 baseline-JPEG decode path on BASELINE.json's metric.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torch.distributed.run)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --workload cfg2|cfg3|cfg4|cfg3n ...       (default cfg3 = the configuration the metric is quoted on)
    python bench.py --global-batch 4096 ...                   (strong scaling: BASELINE config 3's batch split over N GPUs)
    python bench.py --dump-outputs DIR ...                    (what the last timed step decoded, as DIR/*.npy)

Workloads (config.workload; tools/bench_inputs.py): the synthetic source images S(w,h,seed) of SURVEY.md 8d encoded by the
REFERENCE ENCODER (oracle/_ref/jpeg, named in config.encoder; the repo's own generator only where that binary is absent),
`--distinct` distinct frames tiled over the batch.
  cfg3 (default): 3840x2160 4:2:0 q75 baseline, DRI = 240.  One step = one pass of the hot path over 840 frames per GPU
        (840 x 135 restart intervals = one full wave of the persistent entropy kernel); cfg3's 4096-frame batch is 4.9 steps
        of one GPU.  Weak scaling (840 frames per GPU per step) unless --global-batch is given.
  cfg2: 1920x1080 4:2:0 q75, DRI = 120, 4096 frames per step on one GPU (BASELINE configs[1]).
  cfg4: 3840x2160 4:2:0 q75 progressive (ten scans), 1024 frames per step on one GPU (BASELINE configs[3]).
  cfg3n: cfg3 without restart markers (DRI-less streams).

value  : frames/s with the compressed bytes AND the restart index already resident in HBM (device-timed, CUDA events on the
         launching stream, max over ranks): K x (unstuff + entropy + reconstruction kernels) on one stream.
         `restart_index_ms` is the once-per-upload restart_index_kernel stated beside it; `value_with_restart_index` folds it in.
pinned_to_device_rgb : SURVEY 8d's primary accounting -- compressed bytes resident in PINNED HOST memory -> RGB resident in
         DEVICE memory: per chunk H2D + restart_index_kernel + all decode kernels, chunks pipelined over three streams, no D2H;
         host marker parsing / packing (b200jpg_batch_create) happened before the timed region.
e2e    : frames/s through the C ABI with HOST buffers, everything inside the timed region: per chunk b200jpg_batch_create
         (host marker parse + packing into pinned memory, one chunk ahead in a second thread) -> H2D -> kernels -> D2H of
         every decoded pixel into pinned host memory -> batch_destroy.
roofline: the dominant stage by time. Reconstruction: algorithmic bytes = 128 B x stored blocks + output bytes (SURVEY 8d)
         over its CUDA-event duration against MEASURED_PEAKS.json hbm_gbs, plus `int32`: the same launches against the
         measured int32 issue rate (b200jpg_microbench_int32), the roofline north_star names for this stage.
         roofline_entropy: stage a (unstuff + entropy kernels), algorithmic bytes = ECS bytes + 128 B x stored blocks.
         `traffic` = DRAM bytes per launch measured by ncu (profiles/), scaled from the per-frame figure of the captured run.
cpu_baseline / --impl reference: the unmodified reference (oracle/_ref/refharness: public API, memory hook, 8-row stripes)
         as forked worker processes on a bounded sample of the same frames; reports the processes used, the physical cores,
         CPU model, affinity and cgroup quota of the box, and the parallelism the box actually delivered.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools import bench_inputs  # noqa: E402

DEFAULT_FRAMES = {"cfg3": 840, "cfg2": 4096, "cfg4": 1024, "cfg3n": 840, "cfg2n": 4096, "cfg1": 8192, "cfg5": 24}
# DRAM bytes per cfg3 frame measured with ncu --set full (dram__bytes_read.sum + dram__bytes_write.sum); see profiles/
NCU_DRAM_BYTES_PER_FRAME = {"cfg3": {"entropy": None, "recon": None}}
try:
    NCU_DRAM_BYTES_PER_FRAME.update(json.load(open(os.path.join(ROOT, "profiles", "dram_bytes_per_frame.json"))))
except Exception:
    pass
INT_OPS_PER_PIXEL_420 = 520e6 / (3840 * 2160)  # SURVEY.md 8d: IDCT 205 M + upsample 133 M + colour 182 M per 4K 4:2:0 frame


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md): NVML polled every 5 ms from a
    thread (nvidia-smi's loop mode needs seconds to deliver its first line -- longer than a timed region of a few steps)."""

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.stop_flag = threading.Event()
        self.thread = None
        self.max_mhz = None

    def _handle(self):
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
        return pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)

    def start(self):
        try:
            nv, h = self._handle()
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        except Exception:
            return
        bits = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}

        def pump():
            while not self.stop_flag.is_set():
                try:
                    self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for name, bit in bits.items():
                        if r & bit:
                            self.reasons.add(name)
                except Exception:
                    pass
                time.sleep(0.005)

        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if not self.thread:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        self.stop_flag.set()
        self.thread.join(timeout=1)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples), "how": "NVML, 5 ms period, during the timed region"}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0}, "fallback"


# ---------------------------------------------------------------------------------------------------------
# host CPU facts for the CPU arm
def cpu_facts():
    """Physical cores, model, what this process may use (affinity, cgroup quota): the denominators of the CPU arm."""
    model, cores, logical = None, set(), 0
    try:
        phys = core = None
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name") and model is None:
                model = ln.split(":", 1)[1].strip()
            elif ln.startswith("processor"):
                logical += 1
            elif ln.startswith("physical id"):
                phys = ln.split(":", 1)[1].strip()
            elif ln.startswith("core id"):
                core = ln.split(":", 1)[1].strip()
                cores.add((phys, core))
    except Exception:
        pass
    try:
        affinity = len(os.sched_getaffinity(0))
    except Exception:
        affinity = None
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                quota = "unlimited" if txt[0] == "max" else round(int(txt[0]) / int(txt[1]), 2)
            else:
                q = int(txt[0])
                period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                quota = "unlimited" if q < 0 else round(q / period, 2)
            break
        except Exception:
            continue
    return {"cpu_model": model, "physical_cores": len(cores) or None, "logical_cpus": logical or os.cpu_count(),
            "affinity_cpus": affinity, "cgroup_cpu_quota": quota}


def run_reference(frames, procs, iters):
    """Unmodified reference through its public API (oracle/_ref/refharness), `procs` forked workers each decoding
    `iters` frames (cycling over the distinct frames). Falls back to the plain-C oracle port when the reference
    binary is not in the snapshot."""
    ref = os.path.join(ROOT, "oracle", "_ref", "refharness")
    with tempfile.TemporaryDirectory() as tmp:
        paths = []
        for i, f in enumerate(frames[:8]):
            p = os.path.join(tmp, "f%d.jpg" % i)
            open(p, "wb").write(f)
            paths.append(p)
        if os.path.exists(ref):
            t0 = time.time()
            r = subprocess.run([ref, "bench", ",".join(paths), str(iters), str(procs)], capture_output=True, text=True)
            if r.returncode == 0:
                d = json.loads(r.stdout.strip().splitlines()[-1])
                d["kind"] = "reference"
                d["wall_total_s"] = time.time() - t0
                return d
    # port: tests/oracle_binding in worker processes
    from concurrent.futures import ProcessPoolExecutor
    t0 = time.time()
    with ProcessPoolExecutor(max_workers=procs) as ex:
        list(ex.map(_oracle_worker, [(frames[:8], iters, p) for p in range(procs)]))
    wall = time.time() - t0
    return {"frames": procs * iters, "procs": procs, "wall_s": wall, "fps": procs * iters / wall, "kind": "port"}


def _oracle_worker(args):
    frames, iters, p = args
    from tests import oracle_binding
    o = oracle_binding.load()
    for i in range(iters):
        rc, _ = o.decode(frames[(p + i) % len(frames)])
        assert rc == 0


def best_reference_config(frames, ncpu, per_frame_s):
    """The reference is single threaded and allocation heavy: beyond a few dozen processes the box's memory system (or a
    CPU quota), not its core count, limits it. Scan the process count (short samples) and keep the fastest: that is the
    CPU arm's best case. Returns (procs, {procs: fps})."""
    cands = sorted(set(max(1, c) for c in (1, ncpu, ncpu // 2, ncpu // 4, ncpu // 8, 3 * ncpu // 8)))  # 1: the per-core rate
    best, scan = None, {}
    for procs in cands:
        iters = max(2, int(round(1.5 / max(per_frame_s, 1e-3)))) if procs == 1 else max(2, int(round(4.0 / max(per_frame_s, 1e-3) / 8)))
        d = run_reference(frames, procs, min(iters, 64))
        scan[procs] = round(d["fps"], 1)
        if best is None or d["fps"] > best[1]:
            best = (procs, d["fps"])
    return best[0], scan


def cpu_arm(frames, ncpu, workload, budget_s=20.0):
    """-> the cpu_baseline object + the fps. A bounded sample: about `budget_s` seconds of wall time on the best process count."""
    w, h = bench_inputs.WORKLOADS[workload][:2]
    per_frame_s = 0.11 * (w * h) / (3840 * 2160)  # about 9 frames/s per process at 4K on this class of host
    procs, scan = best_reference_config(frames, ncpu, per_frame_s)
    iters = max(4, int(budget_s * max(scan[procs], 1.0) / procs))
    cb = run_reference(frames, procs, iters)
    facts = cpu_facts()
    one = scan.get(1) or None
    out = {"value": cb["fps"], "unit": "frames/s", "cores": cb["procs"], "kind": cb["kind"],
           "sample": "%d frames (%d distinct %s frames cycled) in %d worker processes = the fastest of the process counts scanned "
                     "(%s fps); Read + 8-row-striped DisplayRectangle through the reference's public API"
                     % (cb["frames"], min(len(frames), 8), workload, cb["procs"], scan),
           "processes": cb["procs"], "fps_one_process": one,
           "effective_parallelism": round(cb["fps"] / one, 1) if one else None,
           "read_ms_per_frame": cb.get("read_ms_per_frame"), "display_ms_per_frame": cb.get("display_ms_per_frame")}
    out.update(facts)
    return out


def bind_to_gpu_numa_node(index):
    """Pins this rank (and the threads it starts: host packing, pinned-buffer first touch) to the CPUs next to its GPU, so
    the pinned host buffers of the e2e path are NUMA-local to the PCIe root the GPU hangs on. Best effort."""
    if os.environ.get("B200JPG_NO_AFFINITY"):
        return "off"
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = [64 * w + b for w, m in enumerate(words) for b in range(64) if (m >> b) & 1]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return "%d cpus (%d..%d)" % (len(cpus), cpus[0], cpus[-1])
    except Exception as e:  # no NVML, no permission: run unpinned
        return "unavailable: %s" % type(e).__name__
    return "none"


# fixed sample of the decoded frames for --dump-outputs: one 4K frame alone is 25 MB of samples
DUMP_SEED, DUMP_FRAMES, DUMP_SAMPLES_PER_FRAME = 2024, 8, 1 << 20


def dump_outputs(dec, out, directory):
    """Writes what one decode of the batch delivered to its caller, as arrays two builds can be compared on:
    frame_status.npy   float64 [frames]               status of every frame (0 = decoded)
    frame_sums.npy     float64 [frames, components]   sum of every sample of each component of every frame
    frame_samples.npy  float32 [8, 2^20]              the samples at fixed seeded positions of 8 fixed seeded frames
    sample_frames.npy  float64 [8]                    which frames those are"""
    import numpy as np
    import torch
    os.makedirs(directory, exist_ok=True)
    views = [dec.frame_view(out, i) for i in range(dec.n)]
    np.save(os.path.join(directory, "frame_status.npy"), np.array([dec.status(i) for i in range(dec.n)], dtype=np.float64))
    sums = torch.stack([v.reshape(-1, v.shape[-1]).sum(0, dtype=torch.float64) for v in views])
    np.save(os.path.join(directory, "frame_sums.npy"), sums.cpu().numpy())
    rng = np.random.default_rng(DUMP_SEED)
    picked = np.sort(rng.choice(dec.n, size=min(DUMP_FRAMES, dec.n), replace=False))
    n = min([DUMP_SAMPLES_PER_FRAME] + [views[i].numel() for i in picked])
    samples = [views[i].reshape(-1)[torch.from_numpy(rng.integers(0, views[i].numel(), size=n)).to(out.device)] for i in picked]
    np.save(os.path.join(directory, "frame_samples.npy"), torch.stack(samples).float().cpu().numpy())
    np.save(os.path.join(directory, "sample_frames.npy"), picked.astype(np.float64))


# ---------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(DEFAULT_FRAMES))
    ap.add_argument("--frames-per-gpu", type=int, default=0, help="frames per GPU per step (default: per workload)")
    ap.add_argument("--global-batch", type=int, default=0, help="strong scaling: total frames per step, split over the GPUs")
    ap.add_argument("--distinct", type=int, default=0, help="distinct frames cycled through the batch (default 64; cfg5: 2)")
    ap.add_argument("--e2e-chunk", type=int, default=32)
    ap.add_argument("--e2e-producers", type=int, default=0,
                    help="host threads that prepare chunks (b200jpg_batch_create) ahead of the device; 0 = 2 on two to four GPUs, else 1 (measured, see the e2e section)")
    ap.add_argument("--p2d-chunks", type=int, default=2, help="pinned_to_device_rgb: chunks per step (each: H2D + index + kernels on its own stream)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one decoded as DIR/*.npy (rank 0's frames)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    ncpu = os.cpu_count() or 8
    W, H, QUALITY, SUB, DRI, PROG, desc = bench_inputs.WORKLOADS[args.workload]
    if args.distinct <= 0:
        args.distinct = 2 if args.workload == "cfg5" else 64
    strong = args.global_batch > 0
    if strong:
        nf = (args.global_batch + world - 1) // world
        global_batch = args.global_batch
    else:
        nf = args.frames_per_gpu or DEFAULT_FRAMES[args.workload]
        global_batch = nf * max(world, 1)
    mb_codestream = {"cfg2": 0.37, "cfg2n": 0.37, "cfg1": 0.25, "cfg5": 54.0}.get(args.workload, 1.45)
    config = {"workload": desc, "encoder": bench_inputs.encoder_name(args.workload), "frames_per_gpu": nf, "global_batch": global_batch,
              "distinct_frames": args.distinct, "parallelism": "frames sharded over %d GPU(s), no data-path collective" % world,
              "l2": "inputs larger than L2 (no flush needed): about %.1f GB codestreams + %.1f GB coefficients per step vs 126 MB L2"
                    % (nf * mb_codestream * 1e-3, nf * W * H * 3e-9)}

    if args.impl == "reference":
        if rank != 0:
            return 0
        frames = bench_inputs.make_frames(args.workload, 8, min(8, ncpu))
        vals, last = [], None
        # warm-up = the scan over process counts inside cpu_arm; each timed step is a bounded sample of the same workload
        first = cpu_arm(frames, ncpu, args.workload, budget_s=8.0)
        procs = first["processes"]
        iters = max(4, int(12.0 * max(first["value"], 1.0) / procs))
        t0 = time.time()
        for _ in range(args.steps):
            last = run_reference(frames, procs, iters)
            vals.append(last["fps"])
        dt = time.time() - t0
        v = statistics.mean(vals)
        cb = dict(first)
        cb.update({"value": v, "read_ms_per_frame": last.get("read_ms_per_frame"), "display_ms_per_frame": last.get("display_ms_per_frame"),
                   "sample": "%d frames per step (8 distinct %s frames cycled) in %d worker processes; " % (procs * iters, args.workload, procs)
                             + first["sample"]})
        line = {"impl": "reference", "metric": "4K 4:2:0 q75 frames/sec", "value": v, "unit": "frames/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(args.steps, 1), "higher_is_better": True,
                "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic", "config": config,
                "cpu_baseline": cb,
                "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    import torch
    import libjpeg_b200
    from libjpeg_b200 import native
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    config["cpu_affinity"] = bind_to_gpu_numa_node(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    # ---- inputs (untimed): distinct frames of the workload, tiled over this rank's shard of the global batch
    workers = max(1, min(16, ncpu // max(world, 1)))
    base = bench_inputs.make_frames(args.workload, args.distinct, workers)
    from libjpeg_b200 import sharding
    first, last = sharding.shard_range(global_batch, rank, world)
    frames = [base[i % len(base)] for i in range(first, last)]
    nf = len(frames)
    mean_bytes = sum(len(b) for b in base) / len(base)

    dec = libjpeg_b200.BatchDecoder(frames, device=local_rank)
    # ---- the ONE collective of the path: rank 0 broadcasts the shared Huffman/quantisation table blob (NCCL)
    if dist is not None:
        blob = torch.from_numpy(dec.export_tables()).cuda()
        mine = blob.clone()
        dist.broadcast(blob, src=0)
        assert torch.equal(mine, blob), "frames of this rank use tables different from rank 0's"
        dec.import_tables(blob.cpu().numpy())
    out = dec.new_output()
    stream = torch.cuda.Stream()
    dec.upload(stream)
    torch.cuda.synchronize()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        dec.decode(out, stream)
    torch.cuda.synchronize()
    bad = [i for i in range(nf) if dec.status(i) != 0]
    assert not bad, "decode reported errors for frames %s" % bad[:8]

    # ---- value: K steps on one stream, device-timed
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    e0.record(stream)
    for _ in range(args.steps):
        dec.decode(out, stream)
        launches += dec.launches
    e1.record(stream)
    barrier()
    clocks = sampler.stop()
    total_ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(dec, out, args.dump_outputs)
    t = torch.tensor([total_ms], device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    nframes_all = global_batch
    value = nframes_all * args.steps / (total_ms * 1e-3)

    # the once-per-upload restart index, timed alone (idempotent re-run)
    idx_ms = []
    for _ in range(args.steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        dec.reindex(stream)
        b.record(stream)
        torch.cuda.synchronize()
        idx_ms.append(a.elapsed_time(b))
    index_ms = statistics.mean(idx_ms)
    ti = torch.tensor([index_ms], device="cuda")
    if dist is not None:
        dist.all_reduce(ti, op=dist.ReduceOp.MAX)
    index_ms = float(ti.item())

    # per-stage durations for the rooflines: one step at a time, CUDA events recorded by the library on the launching
    # stream around each stage
    ent_ms, rec_ms, uns_ms = [], [], []
    dec.enable_timing(True)
    for _ in range(args.steps):
        dec.decode(out, stream)
        torch.cuda.synchronize()
        a, b = dec.last_timing()
        ent_ms.append(a)
        rec_ms.append(b)
        uns_ms.append(dec.last_unstuff_ms())
    dec.enable_timing(False)
    ent = statistics.mean(ent_ms)
    rec = statistics.mean(rec_ms)
    uns = statistics.mean(uns_ms)

    peaks, peak_kind = measured_peaks()
    ncu = NCU_DRAM_BYTES_PER_FRAME.get(args.workload, {})
    algo_a = dec.ecs_bytes + 128 * dec.stored_blocks
    roof_a = {"bound": "hbm", "kernel": "stage a = unstuff_kernel + %s" % ("pf_dc_kernel + pf_ac_kernel per component (all scans of a block in one pass)" if PROG else
                                                               ("unstuff_long_kernel + spec_sync_kernel + entropy_decode_kernel<indexed>" if args.workload.endswith("n") else "entropy_decode_kernel")),
              "ms_unstuff": uns, "ms_decode": ent - uns,
              "achieved": algo_a / (ent * 1e-3) / 1e9, "peak": peaks["hbm_gbs"],
              "peak_source": peak_kind + " (MEASURED_PEAKS.json hbm_gbs, burst copy)", "unit": "GB/s",
              "traffic": ncu["entropy"] * nf if ncu.get("entropy") else None,
              "algorithmic_bytes_per_launch": algo_a, "ms_per_launch": ent, "share_of_step": ent / (ent + rec)}
    roof_a["frac"] = roof_a["achieved"] / roof_a["peak"]
    import ctypes
    fi, fa, fm = ctypes.c_float(), ctypes.c_float(), ctypes.c_float()
    native.lib.b200jpg_microbench_int32(local_rank, ctypes.byref(fi), ctypes.byref(fa), ctypes.byref(fm))
    int_peak = max(fi.value, fa.value, fm.value)
    int_ops = INT_OPS_PER_PIXEL_420 * W * H * nf
    algo_b = 128 * dec.stored_blocks + dec.out_bytes
    roof_b = {"bound": "hbm", "kernel": ("stage b = idct_planes_kernel<int> of base + residual image, generic_reconstruct_kernel: upsampling + JPEG XT merge + store"
                                         if args.workload == "cfg5" else "stage b = reconstruction kernel(s): IDCT + upsampling + colour + store"),
              "achieved": algo_b / (rec * 1e-3) / 1e9, "peak": peaks["hbm_gbs"],
              "peak_source": peak_kind + " (MEASURED_PEAKS.json hbm_gbs, burst copy)", "unit": "GB/s",
              "traffic": ncu["recon"] * nf if ncu.get("recon") else None,
              "algorithmic_bytes_per_launch": algo_b, "ms_per_launch": rec, "share_of_step": rec / (ent + rec),
              "int32": {"unit": "Gop/s", "achieved": int_ops / (rec * 1e-3) / 1e9, "peak": int_peak,
                        "peak_source": "measured here: b200jpg_microbench_int32 (imad %.0f, alu %.0f, mix %.0f Gop/s; multiply-add = 2 ops)"
                                       % (fi.value, fa.value, fm.value),
                        "algorithmic_ops_per_frame": INT_OPS_PER_PIXEL_420 * W * H}}
    roof_b["frac"] = roof_b["achieved"] / roof_b["peak"]
    roof_b["int32"]["frac"] = roof_b["int32"]["achieved"] / int_peak if int_peak > 0 else None
    roof, roof_other, other_key = (roof_b, roof_a, "roofline_entropy") if rec >= ent else (roof_a, roof_b, "roofline_reconstruction")

    ctx = dec.ctx
    # ---- SURVEY 8d primary accounting: compressed bytes in PINNED host memory -> RGB in DEVICE memory.
    # The batch is cut into chunks that were parsed and packed into pinned memory before the timed region; timed per chunk:
    # H2D + restart_index_kernel + unstuff + entropy + reconstruction, chunks rotating over three streams; no D2H.
    p2d = None
    chunk_frames = max(1, min(nf, max(args.e2e_chunk, (nf + args.p2d_chunks - 1) // args.p2d_chunks)))
    if not args.no_e2e:
        dec.close()
        dec = None
        ctx.trim()  # the whole-batch buffers go back to the driver: the chunk batches allocate their own
        chunks = [frames[c:c + chunk_frames] for c in range(0, nf, chunk_frames)]
        bds = [libjpeg_b200.BatchDecoder(ch, ctx=ctx) for ch in chunks]
        offs, cur = [], 0
        for bd in bds:
            offs.append(cur)
            cur += (bd.out_bytes + 255) // 256 * 256
        big = out if out.numel() >= cur else torch.empty(cur, dtype=torch.uint8, device="cuda")
        streams = [torch.cuda.Stream() for _ in range(min(3, len(bds)))]

        def p2d_step():
            for i, bd in enumerate(bds):
                s = streams[i % len(streams)]
                bd.upload(s)
                bd.decode(big[offs[i]:offs[i] + bd.out_bytes], s)

        for _ in range(2):
            p2d_step()
        barrier()
        psteps = args.steps
        t0 = time.perf_counter()
        for _ in range(psteps):
            p2d_step()
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], device="cuda")
        if dist is not None:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        assert all(bd.status(i) == 0 for bd in bds for i in (0, bd.n - 1))
        p2d = {"value": nframes_all * psteps / dt, "unit": "frames/s", "steps": psteps, "chunk_frames": chunk_frames, "streams": len(streams),
               "h2d_bytes_per_step": int(sum(bd.h2d_bytes for bd in bds)), "d2h_bytes_per_step": 0,
               "timed_region": "per chunk: H2D of the packed codestreams from pinned host memory + restart_index_kernel + unstuff + "
                               "entropy + reconstruction kernels, chunks rotating over the streams; RGB stays in device memory; host "
                               "marker parsing / packing (b200jpg_batch_create) before the timed region; wall clock between barriers"}
        for bd in bds:
            bd.close()
        del bds, big
        ctx.trim()

    # ---- e2e: the calls a user makes, per chunk of frames, all inside the timed region:
    #   b200jpg_batch_create (host: parse markers, pack into pinned memory; a producer thread runs one chunk ahead) -> upload
    #   (H2D + restart index) -> decode -> D2H of every pixel into pinned host memory -> destroy.
    # Chunks rotate over three CUDA streams; device / pinned buffers are recycled by the context's pool.
    e2e = None
    if not args.no_e2e:
        import queue
        chunk = max(1, min(args.e2e_chunk, nf))
        nchunks = (nf + chunk - 1) // chunk
        nslots = min(3, nchunks)
        probe_b = libjpeg_b200.BatchDecoder(frames[:chunk], ctx=ctx)
        ob = probe_b.out_bytes
        probe_b.close()
        slots = [{"stream": torch.cuda.Stream(), "out": torch.empty(ob, dtype=torch.uint8, device="cuda"),
                  "host": torch.empty(ob, dtype=torch.uint8).pin_memory()} for _ in range(nslots)]
        counters = {"h2d": 0, "d2h": 0}

        # measured (profiles/README.md): one GPU 2.13 k frames/s with one thread, 2.05 k with two; four GPUs 4.85 k / 5.73 k; eight GPUs
        # 9.66 k / 9.35 k (eight ranks x two threads x 16 parsing threads oversubscribe the host)
        nprod = args.e2e_producers if args.e2e_producers > 0 else (2 if 2 <= world <= 4 else 1)

        def e2e_step(keep_last=False):
            # host preparation (b200jpg_batch_create: parse + pack into pinned memory) runs ahead of the device in `nprod` threads,
            # thread t building the chunks c = t (mod nprod); the consumer takes them in order
            qs = [queue.Queue(maxsize=2) for _ in range(nprod)]

            def producer(t):
                for c in range(t, nchunks, nprod):
                    qs[t].put(libjpeg_b200.BatchDecoder(frames[c * chunk:(c + 1) * chunk], ctx=ctx))

            ths = [threading.Thread(target=producer, args=(t,), daemon=True) for t in range(nprod)]
            for th in ths:
                th.start()
            inflight = []
            for c in range(nchunks):
                bd = qs[c % nprod].get()
                s = slots[c % nslots]
                with torch.cuda.stream(s["stream"]):
                    bd.upload(s["stream"])
                    bd.decode(s["out"], s["stream"])
                    s["host"][:bd.out_bytes].copy_(s["out"][:bd.out_bytes], non_blocking=True)
                counters["h2d"] += bd.h2d_bytes
                counters["d2h"] += bd.out_bytes
                inflight.append(bd)
                if len(inflight) > nslots:
                    inflight.pop(0).close()
            for s in slots:
                s["stream"].synchronize()
            for bd in inflight[:-1] if keep_last else inflight:
                bd.close()
            for th in ths:
                th.join()
            return inflight[-1] if keep_last else None

        for _ in range(2):
            e2e_step()
        # the host share of a chunk on its own (VERDICT r1 #5): b200jpg_batch_create = marker parse + packing into pinned memory
        tp = []
        for c in range(min(nchunks, 6)):
            t0 = time.perf_counter()
            bd = libjpeg_b200.BatchDecoder(frames[c * chunk:(c + 1) * chunk], ctx=ctx)
            tp.append((time.perf_counter() - t0) * 1e3)
            bd.close()
        host_prepare_ms = statistics.median(tp)
        # ... and the bare copy of a chunk's pixels, pinned, alone on the link: what the D2H leg can at most deliver
        s0 = slots[0]
        t0 = time.perf_counter()
        for _ in range(4):
            s0["host"].copy_(s0["out"], non_blocking=True)
        torch.cuda.synchronize()
        d2h_gbs = 4 * ob / (time.perf_counter() - t0) / 1e9
        barrier()
        counters["h2d"] = counters["d2h"] = 0
        t0 = time.perf_counter()
        esteps = args.steps
        for i in range(esteps):
            last_bd = e2e_step(keep_last=(i == esteps - 1))
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], device="cuda")
        if dist is not None:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        e2e = {"value": nframes_all * esteps / dt, "unit": "frames/s", "h2d_bytes_per_step": int(counters["h2d"] // esteps),
               "d2h_bytes_per_step": int(counters["d2h"] // esteps), "steps": esteps, "chunk_frames": chunk, "streams": nslots, "host_threads_preparing": nprod,
               "host_prepare_ms_per_chunk": host_prepare_ms, "bare_d2h_gbs_this_rank_alone": d2h_gbs,
               "d2h_ceiling_frames_per_s": d2h_gbs * 1e9 / (ob / chunk) * max(world, 1),
               "timed_region": "per chunk: b200jpg_batch_create on the host codestreams (marker parse, packing into pinned memory) -> H2D "
                               "+ restart index -> unstuff + entropy + reconstruction kernels -> D2H of every pixel into pinned host "
                               "memory -> batch_destroy; host preparation runs ahead of the device in its own threads"}
        # sanity: what came back is what the device-resident path produced (frame nf-1 is in `out` from the value run)
        fi_last = last_bd.info(last_bd.n - 1)
        nbytes = fi_last.width * fi_last.height * fi_last.ncomp
        got = last_bd.frame_view(slots[(nchunks - 1) % nslots]["host"], last_bd.n - 1)
        # the value run's buffer holds frame nf-1 at the whole-batch offset: recompute it from the frame sizes (uniform frames)
        stride = (nbytes + 255) // 256 * 256
        want = out[(nf - 1) * stride:(nf - 1) * stride + nbytes].view(fi_last.height, fi_last.width, fi_last.ncomp)
        assert torch.equal(want.cpu(), got), "e2e output differs from the device-resident decode"
        last_bd.close()
        del slots

    if rank == 0:
        line = {"metric": "4K 4:2:0 q75 frames/sec" if args.workload.startswith("cfg3") else "%s frames/sec" % args.workload,
                "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if strong else "weak",
                "vs_baseline": None, "dtype": "int32", "data": "synthetic", "config": dict(config, mean_codestream_bytes=mean_bytes),
                "clocks": clocks, "gpu_launches": launches, "roofline": roof, other_key: roof_other,
                "restart_index_ms": index_ms, "value_with_restart_index": nframes_all / ((ms_per_step + index_ms) * 1e-3),
                "stage_ms": {"entropy": ent, "entropy_unstuff_share": uns, "reconstruction": rec, "restart_index_once_per_upload": index_ms}}
        if p2d:
            line["pinned_to_device_rgb"] = p2d
        if e2e:
            line["e2e"] = e2e
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_arm(base, ncpu, args.workload)
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
