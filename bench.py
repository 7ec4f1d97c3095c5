#!/usr/bin/env python
"""bench.py -- frames/s of the nnnoiseless per-frame denoise path on B200 (driver contract).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--streams B_per_gpu | --total-streams B] [--frames T] [--model PATH] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch: B streams per GPU, each advanced T consecutive
480-sample frames (T frame-steps of 5 kernels each, T = 100 = one second of audio per stream, SURVEY 8(d)).
Default workload:
  * one GPU          : BASELINE.json configs[2] -- batch=65536 streams, synthetic 48 kHz white+sine, built-in model
                       (the largest single-GPU configuration, the one the ncu roofline capture is quoted on);
  * under torchrun   : 32,768 streams per GPU, so that N = 8 IS configs[3] (batch=262144 sharded across 8xB200).
  * --streams 4096   : configs[1];  --model tests/golden/sh.rnnn --total-streams 65536 : configs[4] (strong scaling).
Every rank owns its own streams (no data-path collective; the model image is broadcast once over NCCL).
Input = synthetic white+sine PCM-valued audio, resident in HBM before the timed region; each step reads
T*B*1920 B of input (12.6 GB at the default, >> the 126 MB L2).

--impl reference times the reference's CPU implementation of the same path (the C restatement in
oracle/ -- the Rust crate cannot be built in this image) with all host threads, pinned, on a bounded sample of
the same workload.

--dump-outputs DIR writes what the last timed step returned (see dump_outputs).  The inputs are seeded and the warm-up
steps start from a fresh state, so two builds run with the same arguments can be compared output for output.
"""
import os

# OpenMP placement of the CPU arm must be decided before libgomp initialises (torch loads it too)
os.environ.setdefault("OMP_PROC_BIND", "close")
os.environ.setdefault("OMP_PLACES", "cores")

import argparse  # noqa: E402
import csv  # noqa: E402
import glob  # noqa: E402
import json  # noqa: E402
import re  # noqa: E402
import subprocess  # noqa: E402
import sys  # noqa: E402
import tempfile  # noqa: E402
import time  # noqa: E402

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FRAME = 480
# SURVEY 8(d) / BASELINE.md section 3: algorithmic bytes per stream-frame at T = 1 frame per launch
BYTES_IO = 3844            # 1920 in + 1920 out + 4 vad
BYTES_STATE = 13016        # state round trip (8308 read + 4708 written)
BYTES_PER_FRAME = BYTES_IO + BYTES_STATE  # 16860
# algorithmic bytes of each kernel of the 5-kernel pipeline taken alone (its own compulsory I/O per frame)
KERNEL_BYTES = {
    "hp_filter": 1920 + 8 + 1920 + 8,
    "pitch": 1728 * 4 + 8 + 4 + 8,
    "analysis": 960 * 4 + 960 * 4 + 4 + 704 + 4 + 3848 + 3200 + 3 * 88 + 168 + 4 + 88 + 4,
    "rnn": 168 + 672 + 4 + 672 + 88 + 4,
    "synthesis": 3848 + 3200 + 3 * 88 + 88 + 88 + 88 + 1920 + 1920 + 1920 + 4,
}
KERNEL_PATTERNS = {"hp_filter": "hp_filter_kernel", "pitch": "pitch_kernel", "analysis": "analysis_",
                   "rnn": "rnn_", "synthesis": "synthesis_"}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def measured_traffic():
    """DRAM bytes per stream-frame of every kernel, from the NEWEST committed `ncu --set full` raw page under profiles/
    (rNN_vM_ncu_raw_B<streams>.csv: dram__bytes_read.sum + dram__bytes_write.sum per launch / streams).  Returns
    ({kernel: bytes per stream-frame}, file name) or (None, None)."""
    best = None
    for p in glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_raw_B*.csv")):
        m = re.match(r"r(\d+)_v(\d+)_ncu_raw_B(\d+)\.csv$", os.path.basename(p))
        if m:
            key = (int(m.group(1)), int(m.group(2)))
            if best is None or key > best[0]:
                best = (key, p, int(m.group(3)))
    if best is None:
        return None, None
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    try:
        rows = list(csv.reader(open(best[1])))
        hdr, units = rows[0], rows[1]
        kcol = hdr.index("Kernel Name")
        rd = [i for i, c in enumerate(hdr) if c.endswith("dram__bytes_read.sum")][0]
        wr = [i for i, c in enumerate(hdr) if c.endswith("dram__bytes_write.sum")][0]
        out = {}
        for r in rows[2:]:
            for k, pat in KERNEL_PATTERNS.items():
                if pat in r[kcol]:
                    out[k] = out.get(k, 0.0) + (float(r[rd]) * unit[units[rd]] + float(r[wr]) * unit[units[wr]]) / best[2]
        return (out if len(out) == len(KERNEL_PATTERNS) else None), os.path.basename(best[1])
    except Exception:
        return None, None


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        with open(self.path) as f:
            for line in f:
                c = [x.strip() for x in line.split(",")]
                if len(c) < 9:
                    continue
                try:
                    sm.append(float(c[1])); smax.append(float(c[2]))
                except ValueError:
                    continue
                for n, v in zip(names, c[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
        os.unlink(self.path)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(smax)), "reasons": sorted(reasons),
                "samples": len(sm)}


def synth_on_device(torch, B, T, device, seed):
    """[T][B][480] float32 on `device`: clamp(round(A sin(2 pi f n/48000 + phi) + sigma N(0,1))), per-stream
    f in [100,4000] Hz log-uniform, A in [1000,12000], sigma in [100,3000] (SURVEY 8(d))."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    r = torch.rand(4, B, generator=g, device=device, dtype=torch.float64)
    f = 100.0 * torch.pow(torch.tensor(40.0, dtype=torch.float64, device=device), r[0])
    a = (1000.0 + 11000.0 * r[1]).float()
    sg = (100.0 + 2900.0 * r[2]).float()
    ph = 2 * np.pi * r[3]
    x = torch.empty(T, B, FRAME, device=device, dtype=torch.float32)
    n = torch.arange(FRAME, device=device, dtype=torch.float64)
    for t in range(T):
        arg = 2 * np.pi * f[:, None] * (n[None, :] + t * FRAME) / 48000.0 + ph[:, None]
        arg = torch.remainder(arg, 2 * np.pi).float()
        v = a[:, None] * torch.sin(arg) + sg[:, None] * torch.randn(B, FRAME, generator=g, device=device)
        x[t] = torch.clamp(torch.round(v), -32768.0, 32767.0)
    return x


# BASELINE.json "metric": "48kHz mono frames/sec (480-sample) at 1/2/4/8 B200; %HBM roofline; vs Rust CPU" -- the
# throughput part is the line's value, the other two parts are the `roofline` and `cpu_baseline` objects of the line.
METRIC = "48kHz mono frames/sec (480-sample)"


def load_model_bytes(path):
    """--model: RNNoise text format (.rnnn, e.g. the reference's test_data/sh.rnnn) or nnnoiseless binary -> image bytes."""
    import nnnoiseless_b200 as nb
    data = open(path, "rb").read()
    if data[:7] == b"rnnoise":
        m = nb.RnnModel.from_text(data)
    else:
        m = nb.RnnModel.from_bytes(data)
    if m is None:
        raise SystemExit("bench.py: %s is not a valid model" % path)
    return m.to_bytes()


def resolve_workload(args, world):
    """-> (streams per GPU, scaling, config dict).  The config dict is IDENTICAL for both arms."""
    if args.total_streams > 0:
        B, scaling = max(1, args.total_streams // world), "strong"
    elif args.streams > 0:
        B, scaling = args.streams, "weak"
    else:
        B, scaling = (65536 if world == 1 else 32768), "weak"
    model = "built-in weights.rnn" if not args.model else os.path.basename(args.model)
    total = B * world
    if args.model and total == 65536:
        tag = "configs[4]: batch=65536 streams, custom model %s" % model
    elif not args.model and world == 1 and B == 65536:
        tag = "configs[2]: batch=65536 streams synthetic 48kHz white+sine noise, 1xB200"
    elif not args.model and world == 8 and B == 32768:
        tag = "configs[3]: batch=262144 streams sharded across 8xB200, NCCL weight-broadcast only"
    elif not args.model and B == 4096:
        tag = "configs[1]: batch=4096 independent mono streams per GPU"
    else:
        tag = "batch=%d streams per GPU x %d GPU(s), model %s" % (B, world, model)
    cfg = {"workload": "%s; %d streams per GPU x %d frames per step" % (tag, B, args.frames),
           "streams_per_gpu": B, "frames_per_step": args.frames, "model": model,
           "parallelism": "streams sharded x%d, no data-path collective" % world,
           "l2_policy": "inputs larger than L2: each step streams %.0f MB in + %.0f MB out through HBM per GPU"
                        % (args.frames * B * 1920 / 1e6, args.frames * B * 1920 / 1e6)}
    return B, scaling, cfg


def all_cpus():
    try:
        return sorted(os.sched_getaffinity(0))
    except AttributeError:
        return list(range(os.cpu_count() or 1))


def cgroup_cpu_quota():
    """CPU-time quota of this container in cores (cgroup v2 cpu.max / v1 cfs quota), or None when unlimited: with a quota
    below the affinity count the all-core rate of the CPU arm is bounded by the quota, not by the thread count."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        return None if q == "max" else float(q) / float(per)
    except Exception:
        pass
    try:
        q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        return None if q <= 0 else q / per
    except Exception:
        return None


def usable_threads(cpus):
    """Threads the CPU arm runs: one per CPU of the affinity mask, capped by the container's CPU-time quota (on the GPU
    boxes of this pool: 128 hardware threads visible, cpu.max = 16 cores -- 128 runnable threads only take turns being
    throttled, and calling that "128 cores" would misstate the baseline)."""
    q = cgroup_cpu_quota()
    n = len(cpus)
    if q is not None and q >= 1.0:
        n = min(n, int(q))
    return max(1, n)


def gpu_numa_cpus(torch, local):
    """CPUs of the NUMA node GPU `local` hangs off (sysfs), or None."""
    try:
        p = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read())
        if node < 0:
            return None
        cpus = []
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        return cpus or None
    except Exception:
        return None


def oracle_model(model_bytes):
    import oracle
    import nnnoiseless_b200 as nb
    if model_bytes is None:
        with open(nb.BUILTIN_WEIGHTS_PATH, "rb") as f:
            model_bytes = f.read()
    return oracle.Model(model_bytes)


def cpu_run(m, x_bt, threads):
    """Times the oracle (C restatement of the reference) on [n][T][480] host samples; returns frames/s, threads used."""
    import oracle
    r = oracle.run_batch(m, x_bt, n_threads=threads, want_out=True, want_taps=False)
    return x_bt.shape[0] * x_bt.shape[1] / r["seconds"], r["threads"]


def cpu_side_measurements(m, x_bt, cores, all_core_fps=None):
    """SURVEY 8(d) side figures of the CPU arm: one core, all-zero input (silent fast path), and the benches/sin.rs:9-20
    shape (one second of a 440 Hz sine through a freshly constructed state, construction included); plus what bounds the
    all-core rate on a shared box (container CPU quota, load average, measured all-core / one-core ratio)."""
    import oracle
    one = max(1, min(x_bt.shape[0], 8))
    fps1, _ = cpu_run(m, x_bt[:one], 1)
    zeros = np.zeros_like(x_bt[: max(cores, 1) * 2])
    fps0, _ = cpu_run(m, zeros, cores)
    n = np.arange(48000, dtype=np.float64)
    sine = (np.sin(2 * np.pi * 440.0 * n / 48000.0) * 16384.0).astype(np.float32).reshape(100, FRAME)
    best = None
    for _ in range(5):
        t0 = time.perf_counter()
        st = oracle.State(m)
        lib, h = oracle.lib(), st._h
        out = np.empty(FRAME, np.float32)
        for f in range(100):
            lib.nno_process_frame(h, out.ctypes.data, sine[f].ctypes.data)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return {"one_core_frames_per_s": fps1, "all_core_over_one_core": (all_core_fps / fps1) if all_core_fps else None, "cgroup_cpu_quota_cores": cgroup_cpu_quota(),
            "load_avg_1min": os.getloadavg()[0],
            "silent_input_frames_per_s_all_cores": fps0,
            "sin_1s_440hz_single_stream_ms": 1e3 * best,
            "sin_note": "benches/sin.rs:9-20 shape: 100 frames of a 440 Hz sine incl. state construction, one thread, best of 5"}


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port) on host cores, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    cpus = all_cpus()
    cores = usable_threads(cpus)
    B, scaling, cfg = resolve_workload(args, world)
    T = args.frames
    n = min(B, max(len(cpus) * 8, 8))
    from nnnoiseless_b200.synth import synth_streams  # numpy generator, same signal family as the GPU arm
    x = synth_streams(n, T, seed=1234).reshape(n, T, FRAME)  # n DISTINCT streams of the workload
    m = oracle_model(load_model_bytes(args.model) if args.model else None)
    for _ in range(max(1, min(args.warmup, 2))):
        cpu_run(m, x, cores)       # full-size warm-up: page faults, thread pool, clocks
    t0 = time.perf_counter()
    frames = 0
    threads = 1
    per_step = []
    for _ in range(args.steps):
        fps, threads = cpu_run(m, x, cores)
        per_step.append(fps)
        frames += n * T
    dt = time.perf_counter() - t0
    value = frames / dt
    side = cpu_side_measurements(m, x, cores, value)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": threads, "kind": "port",
                         "per_thread": value / max(threads, 1), "median_step": float(np.median(per_step)),
                         "sample": "%d distinct streams of the workload x %d frames per step (bounded sample of the %d-stream "
                                   "batch), oracle/nno_oracle.c (C restatement; no rustc in image), OpenMP one stream per thread, "
                                   "OMP_PROC_BIND=%s OMP_PLACES=%s" % (n, T, B, os.environ.get("OMP_PROC_BIND"), os.environ.get("OMP_PLACES")),
                         **side},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


DUMP_BYTES = 64_000_000  # --dump-outputs writes at most this much in all


def dump_outputs(torch, path, out, vad):
    """--dump-outputs: what the last timed step returned, as float32 .npy files under `path`.  vad.npy is the [T][B]
    voice probability, whole when it takes at most half of DUMP_BYTES; out.npy is the denoised [n][480] frames of the
    (frame, stream) pairs in a fixed sample (seed 0, in row-major [T][B] order) that fills the other half, or of every
    pair when they fit.  vad.npy is sampled at the same pairs when it is not whole."""
    T, B = vad.shape
    rows = T * B
    n = min(rows, DUMP_BYTES // 2 // (FRAME * 4))
    idx = np.arange(rows) if n == rows else np.sort(np.random.default_rng(0).choice(rows, n, replace=False))
    idx_d = torch.from_numpy(idx).to(out.device)
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "out.npy"), out.reshape(rows, FRAME).index_select(0, idx_d).cpu().numpy())
    v = vad if rows * 4 <= DUMP_BYTES // 2 else vad.reshape(rows).index_select(0, idx_d)
    np.save(os.path.join(path, "vad.npy"), v.cpu().numpy())


def run_b200(args):
    cpus0 = all_cpus()
    # stdout carries exactly ONE JSON line: whatever libraries print on the way (e.g. the NCCL version banner, written by
    # C code straight to fd 1) is diverted to stderr until the line is printed
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist
    import nnnoiseless_b200 as nb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"  # the version banner goes to stdout; stdout carries exactly one JSON line
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # Host side of the e2e leg: run this rank (and allocate its pinned buffers) on the NUMA node its GPU hangs off.
    numa = gpu_numa_cpus(torch, local)
    bound = None
    if numa:
        mine = [c for c in numa if c in cpus0] or None
        if mine and world > 1:
            # ranks that share a node split its CPUs
            try:
                os.sched_setaffinity(0, mine)
                bound = "%d CPUs of the GPU's NUMA node" % len(mine)
            except OSError:
                bound = None
        elif mine:
            try:
                os.sched_setaffinity(0, mine)
                bound = "%d CPUs of the GPU's NUMA node (released for the CPU baseline)" % len(mine)
            except OSError:
                bound = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # model image: rank 0 owns it, everybody else receives it over NCCL (the only collective of the path)
    if rank == 0:
        img = load_model_bytes(args.model) if args.model else nb.RnnModel().to_bytes()
    if world > 1:
        n = torch.zeros(1, dtype=torch.int64, device=dev)
        if rank == 0:
            n[0] = len(img)
        dist.broadcast(n, 0)
        buf = torch.zeros(int(n.item()), dtype=torch.uint8, device=dev)
        if rank == 0:
            buf.copy_(torch.frombuffer(bytearray(img), dtype=torch.uint8))
        dist.broadcast(buf, 0)
        img = buf.cpu().numpy().tobytes()
    model = nb.RnnModel.from_bytes(img)
    assert model is not None

    B, scaling, cfg = resolve_workload(args, world)
    T = args.frames
    batch = nb.DenoiseBatch(B, model, device=local)
    x = synth_on_device(torch, B, T, dev, seed=1234 + rank)
    out = torch.empty_like(x)
    vad = torch.empty(T, B, device=dev)
    stream = torch.cuda.current_stream()
    sp = stream.cuda_stream

    def step():
        batch.process_device(out.data_ptr(), x.data_ptr(), vad.data_ptr(), T, stream_stride=FRAME, frame_stride=B * FRAME,
                             cuda_stream=sp)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        # nvidia-smi needs a moment to start: keep the GPU under the same load until the first sample has arrived
        t_wait = time.time()
        while sampler.proc is not None and os.path.getsize(sampler.path) == 0 and time.time() - t_wait < 5.0:
            step()
            torch.cuda.synchronize()
    barrier()
    # exactly `warmup` steps from a fresh state precede the timed ones: what the last timed step computes depends on the
    # arguments alone, not on how many steps the wait above took
    batch.reset()
    for _ in range(args.warmup):
        step()
    barrier()
    l0 = nb.kernel_launches()
    ps0 = batch.pitch_stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    launches = nb.kernel_launches() - l0
    ps1 = batch.pitch_stats()
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(torch, args.dump_outputs, out, vad)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    frames_total = world * B * T * args.steps
    value = frames_total / (ms_total * 1e-3)

    # ---- per-kernel durations (CUDA events between the kernels, same stream, same workload) ----
    kms = {}
    nprof = min(T, 20)
    for t in range(nprof):
        d = batch.profile_step(out[t].data_ptr(), x[t].data_ptr(), vad[t].data_ptr(), FRAME, sp)
        for k, v in d.items():
            kms.setdefault(k, []).append(v)
    kavg = {k: float(np.mean(v)) for k, v in kms.items()}
    step_ms = sum(kavg.values())
    dom = max(kavg, key=kavg.get)
    peak, peak_src = load_peaks()
    # one launch set = one frame of the rank's B streams; its device time inside the timed region (stages of
    # consecutive frames overlap) is ms_total / (frames per rank) -- all ranks run the same schedule
    launch_ms = ms_total / (T * args.steps)
    path_gbs = BYTES_PER_FRAME * B / (launch_ms * 1e-3) / 1e9
    traffic, traffic_file = measured_traffic()
    nsf = max(1, ps1["stream_frames"] - ps0["stream_frames"])
    roofline = {
        "bound": "hbm", "unit": "GB/s", "peak": peak, "peak_source": peak_src,
        "achieved": path_gbs, "frac": path_gbs / peak, "frame_step_ms_pipelined": launch_ms,
        # DRAM bytes per frame-step: dram__bytes_read.sum + dram__bytes_write.sum of the five kernels from the newest
        # committed `ncu --set full` raw page (per stream-frame, x this B); null until such a page exists
        "traffic": (sum(traffic.values()) * B) if traffic else None,
        "traffic_unit": "bytes per frame-step (ncu --set full, profiles/%s, per stream-frame x B)" % traffic_file if traffic else None,
        "traffic_per_stream_frame": traffic,
        "dominant_kernel_traffic": ({"kernel": dom, "bytes_per_launch": traffic[dom] * B,
                                     "algorithmic_bytes_per_launch": KERNEL_BYTES[dom] * B} if traffic and dom in traffic else None),
        "definition": "16,860 algorithmic B/frame (T=1: 3,844 I/O + 13,016 state round trip, SURVEY 8(d)) x %d frames per "
                      "frame-step / CUDA-event time per frame-step inside the timed region (the five kernels of a frame-step; "
                      "kernels of up to 4 consecutive frames overlap on separate streams)" % B,
        "frame_step_ms_serial_sum": step_ms, "dominant_kernel": dom,
        "kernels": {k: {"ms": v, "share": v / step_ms, "own_bytes_per_frame": KERNEL_BYTES.get(k),
                        "own_gbs": (KERNEL_BYTES.get(k, 0) * B / (v * 1e-3) / 1e9) if v > 0 else None}
                    for k, v in kavg.items()},
        "io_only_frac": (BYTES_IO * B / (launch_ms * 1e-3) / 1e9) / peak,
        "pitch_exact_recomputation": {"coarse_frac": (ps1["coarse_exact"] - ps0["coarse_exact"]) / nsf,
                                      "ladder_frac": (ps1["ladder_exact"] - ps0["ladder_exact"]) / nsf,
                                      "note": "share of stream-frames whose certified FMA pitch sums were recomputed order-exact in-kernel"},
        "compute_note": "path is FP32-issue/latency bound, not HBM bound (SURVEY 8(d)); frac is reported against HBM as asked",
    }

    # ---- e2e: same metric through the public host-buffer API (pinned host memory, copies inside the timed region) ----
    Te = min(T, args.e2e_frames) if args.e2e_frames > 0 else min(T, 16)
    while Te > 1 and Te * B * FRAME * 4 > (2 << 30):  # keep each pinned buffer at or under 2 GiB
        Te //= 2
    hx = torch.empty(Te, B, FRAME, dtype=torch.float32).pin_memory()
    hx.copy_(x[:Te].cpu())
    ho = torch.empty(Te, B, FRAME, dtype=torch.float32).pin_memory()
    hv = torch.empty(Te, B, dtype=torch.float32).pin_memory()
    L = nb.lib()
    import ctypes as C

    def e2e_step():
        rc = L.rnnoise_batch_process_host(batch._h, C.c_void_p(ho.data_ptr()), C.c_void_p(hx.data_ptr()),
                                          C.c_void_p(hv.data_ptr()), Te)
        assert rc == 0, nb.last_error()

    def timed(fn):
        fn()
        barrier()
        t0 = time.perf_counter()
        ne = max(1, min(args.steps, 5))
        for _ in range(ne):
            fn()
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        return world * B * Te * ne / float(dt.item())

    e2e = {"value": timed(e2e_step), "unit": "frames/s", "h2d_bytes_per_step": Te * B * FRAME * 4,
           "d2h_bytes_per_step": Te * B * (FRAME * 4 + 4), "frames_per_call": Te, "host_binding": bound,
           "api": "rnnoise_batch_process_host (pinned host buffers, H2D + 5 kernels/frame + D2H in bounded slices, synchronous)"}
    del hx, ho
    # same through the 16-bit PCM entry point (int16 in/out, conversion fused into the kernels): half the PCIe bytes
    hx16 = torch.empty(Te, B, FRAME, dtype=torch.int16).pin_memory()
    hx16.copy_(x[:Te].to(torch.int16).cpu())
    ho16 = torch.empty(Te, B, FRAME, dtype=torch.int16).pin_memory()

    def e2e16_step():
        rc = L.rnnoise_batch_process_pcm16_host(batch._h, C.c_void_p(ho16.data_ptr()), C.c_void_p(hx16.data_ptr()),
                                                C.c_void_p(hv.data_ptr()), Te)
        assert rc == 0, nb.last_error()

    e2e["pcm16"] = {"value": timed(e2e16_step), "unit": "frames/s", "h2d_bytes_per_step": Te * B * FRAME * 2,
                    "d2h_bytes_per_step": Te * B * (FRAME * 2 + 4), "api": "rnnoise_batch_process_pcm16_host"}
    del hx16, ho16

    # ---- legacy drop-in ABI (src/capi.rs:75-85): one stream, one frame per call, host buffers ----
    legacy = None
    if rank == 0 and world == 1 and not args.no_legacy:
        st = L.rnnoise_create(model._h)
        if st:
            buf = np.ascontiguousarray(x[:50, 0].cpu().numpy())
            for f in range(10):
                L.rnnoise_process_frame(st, buf[f].ctypes.data_as(C.c_void_p), buf[f].ctypes.data_as(C.c_void_p))
            t0 = time.perf_counter()
            nl = 0
            for rep in range(20):
                for f in range(10, 50):
                    L.rnnoise_process_frame(st, buf[f].ctypes.data_as(C.c_void_p), buf[f].ctypes.data_as(C.c_void_p))
                    nl += 1
            dtl = time.perf_counter() - t0
            L.rnnoise_destroy(st)
            legacy = {"frames_per_s": nl / dtl, "us_per_frame": 1e6 * dtl / nl,
                      "api": "rnnoise_process_frame, B = 1, T = 1 per call (ctypes call overhead included)"}

    # ---- CPU baseline (rank 0, N = 1 only): the oracle on a bounded sample of the same workload ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            os.sched_setaffinity(0, cpus0)
        except (OSError, AttributeError):
            pass
        cores = usable_threads(cpus0)
        n = min(B, max(8, 16 * len(cpus0)))
        xs = x[:, :n].permute(1, 0, 2).contiguous().cpu().numpy()  # [n][T][480]
        m = oracle_model(img)
        cpu_run(m, xs, cores)  # full-size warm-up (tables, page faults, thread pool)
        runs = [cpu_run(m, xs, cores) for _ in range(3)]
        fps = float(np.median([r[0] for r in runs]))
        threads = runs[0][1]
        cpu = {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port", "per_thread": fps / max(threads, 1),
               "sample": "first %d streams x %d frames of the GPU workload, median of 3; oracle/nno_oracle.c (C restatement of the "
                         "reference; Rust toolchain absent), -O3 -march=native -ffp-contract=off, OpenMP one stream per thread, "
                         "OMP_PROC_BIND=%s OMP_PLACES=%s" % (n, T, os.environ.get("OMP_PROC_BIND"), os.environ.get("OMP_PLACES")),
               **cpu_side_measurements(m, xs, cores, fps)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg,
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
            "legacy_abi": legacy,
        }
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line))
        sys.stdout.flush()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--streams", type=int, default=0,
                    help="streams per GPU (0 = default: 65536 on one GPU = configs[2], 32768 per GPU under torchrun = configs[3] at N=8)")
    ap.add_argument("--total-streams", type=int, default=0, help="total streams, split over the GPUs (strong scaling; configs[4])")
    ap.add_argument("--frames", type=int, default=100, help="frames per stream per step")
    ap.add_argument("--model", default="", help="custom model: RNNoise text (.rnnn) or nnnoiseless binary")
    ap.add_argument("--e2e-frames", type=int, default=0, help="frames per host-API call in the e2e leg (0 = min(frames, 16))")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-legacy", action="store_true")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed step returned (rank 0) as DIR/out.npy and DIR/vad.npy, at most 64 MB")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
