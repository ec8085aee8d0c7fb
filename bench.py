#!/usr/bin/env python
"""bench.py — registrations/s of the kinematic-icp hot path on B200 (BASELINE.json metric).

A "step" is one full KinematicRegistration::ComputeRobotMotion (prior -> converged or max-iteration pose) of the
OS1-128-shape synthetic scan (~262 k points) against the 1 M-point voxel map (BASELINE.json configs[3], "cfg4").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload 1..4] [--mode sharded|replicas]
                    [--dump-outputs DIR]

N > 1 is launched by torchrun, one rank per GPU.  In `sharded` mode (default, the north-star layout) the scan's
points are split by contiguous index range, the map is replicated, and every IRLS iteration ends with one exchange of
8 doubles (fused into the persistent kernel over NVLink peer memory, or NCCL with --comm nccl): total work is fixed, so
"scaling" is "strong".  The same invocation then also runs BASELINE.json configs[4]'s layout — N independent registrations,
one per GPU — and reports it under "replicas".  Rank 0 prints ONE JSON line.
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
for _p in (ROOT, os.path.join(ROOT, "kinematic-icp_b200", "python")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "scans/sec (full ICP)"
UNIT = "scans/s"
L2_FLUSH_BYTES = 256 << 20  # > 126 MB L2


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", type=int, default=4, help="BASELINE.json config id 1..4 (default 4 = the quoted one)")
    ap.add_argument("--mode", default="sharded", choices=["sharded", "replicas"])
    ap.add_argument("--comm", default="p2p", choices=["p2p", "nccl"],
                    help="N > 1 sharded mode: fused peer-memory exchange inside the persistent kernel (default) or NCCL allreduce")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-replay", action="store_true", help="skip the whole-pipeline replay (kicp_replay) reported under `replay`")
    ap.add_argument("--sustained", type=int, default=1000,
                    help="N = 1: registrations of the back-to-back run reported under `sustained` (0 = skip)")
    ap.add_argument("--no-flush", action="store_true", help="diagnostic only: keep L2 warm between steps")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (float64), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def dump_outputs(d, arrays):
    """One float64 .npy per returned array; the workloads are seeded, so equal arguments give equal inputs."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), np.asarray(a, dtype=np.float64))


def result_arrays(res):
    """The kicp_reg_result of one registration, field by field (per-iteration rows up to `iterations`).  Search windows are handed
    to warps dynamically, so `sums`, `dx` and `last_dx_norm` of two runs agree to rounding, not bit for bit."""
    return {"pose": res.pose_np(), "beta": res.beta, "last_dx_norm": res.last_dx_norm, "iterations": res.iterations,
            "status": res.status, "sums": res.sums_np(), "dx": res.dx_np()}


def workload_config(w, extra=None):
    d = w.describe()
    cfg = {"workload": "%s: %d-pt scan vs %d-pt voxel map (%d voxels), voxel_size %.2f, %d pts/voxel, tau %.4f, "
                       "max_iter 10, conv 1e-3, adaptive regularisation, prior = truth +5%% d +0.01 rad" %
                       (d["name"], d["N"], d["M"], d["voxels"], d["voxel_size"], d["max_points_per_voxel"], d["tau"]),
           "scan_points": d["N"], "map_points": d["M"], "map_voxels": d["voxels"]}
    if extra:
        cfg.update(extra)
    return cfg


# ------------------------------------------------------------------------------------------------ clocks sampler
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.path = tempfile.mktemp(suffix=".csv")
        self.proc = None

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if sm:
            out = {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}
        return out


class NvmlSampler:
    """SM clock and throttle reasons sampled every millisecond by a thread, through NVML (nvidia_ml_py), only while the
    main thread is inside a timed region (`active`): the timed regions of this bench last milliseconds, shorter than one
    nvidia-smi start-up.  Falls back to the nvidia-smi loop above when NVML is unavailable."""
    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, gpu_index, uuid=None):
        import threading
        self.fallback = None
        self.samples, self.active, self.stop_flag = [], False, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = None
            if uuid is not None:
                try:
                    self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(uuid)).encode())
                except Exception:
                    self.h = None
            if self.h is None:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._run, daemon=True)
        except Exception:
            self.nv = None
            self.fallback = ClockSampler(gpu_index)

    def _reasons(self):
        for name in ("nvmlDeviceGetCurrentClocksEventReasons", "nvmlDeviceGetCurrentClocksThrottleReasons"):
            f = getattr(self.nv, name, None)
            if f is not None:
                try:
                    return int(f(self.h))
                except Exception:
                    continue
        return 0

    def _run(self):
        import time as _t
        while not self.stop_flag:
            if self.active:
                try:
                    self.samples.append((float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)), self._reasons()))
                except Exception:
                    pass
            _t.sleep(0.001)

    def start(self):
        if self.fallback is not None:
            self.fallback.start()
        else:
            self.thread.start()

    def stop(self):
        if self.fallback is not None:
            out = self.fallback.stop()
            out["source"] = "nvidia-smi -lms 100 over the whole run"
            return out
        self.stop_flag = True
        self.thread.join(timeout=2)
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": len(self.samples),
               "source": "NVML, 1 ms period, timed regions only"}
        if self.samples:
            out["sm_mhz"] = statistics.median(x[0] for x in self.samples)
            mask = 0
            for _, r in self.samples:
                mask |= r
            out["reasons"] = [name for bit, name in self.REASONS if mask & bit]
        return out


# -------------------------------------------------------------------------------------------------- CPU baseline
def physical_cores():
    """Physical cores of the host (one worker per core: SMT siblings share the units the FP64 search saturates)."""
    seen = set()
    try:
        base = "/sys/devices/system/cpu"
        for d in os.listdir(base):
            path = os.path.join(base, d, "topology", "thread_siblings_list")
            if d.startswith("cpu") and d[3:].isdigit() and os.path.exists(path):
                seen.add(open(path).read().strip())
    except OSError:
        pass
    n = len(seen) if seen else (os.cpu_count() or 1)
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except AttributeError:
        pass
    return max(n, 1)


def cpu_registration_runner(w, threads):
    """Returns (callable running one full registration on `threads` host threads, kind)."""
    from oracle import kicp_oracle_py as ko
    if ko.ref_available():
        _, _, pts = w.map.export_voxels()
        rm = ko.RefMap(w.voxel_size, w.max_range, w.max_points_per_voxel)
        rm.add_points(pts)

        def run():
            return rm.register(w.scan, w.last_pose, w.rel_odom, w.tau, threads=threads)
        return run, "reference"

    def run():
        return w.map.register(w.scan, w.last_pose, w.rel_odom, w.tau, threads=threads)[0]
    return run, "port"


def time_cpu(w, steps, warmup, single_thread_steps=0):
    """The reference's own Registration.cpp (oracle/_ref) on the box's physical cores: a persistent worker pool (oracle/shim/tbb),
    median over `steps` registrations; optionally also T = 1, the reference's online default (pipeline/KinematicICP.hpp:54)."""
    cores = physical_cores()
    run, kind = cpu_registration_runner(w, cores)
    for _ in range(warmup):
        run()
    ts = []
    for _ in range(steps):
        t = time.perf_counter()
        last = run()
        ts.append(time.perf_counter() - t)
    med = statistics.median(ts)
    out = {"value": 1.0 / med, "unit": UNIT, "cores": cores, "kind": kind,
           "sample": "%d full registrations of the same workload (all %d scan points, all iterations), %s, %d host threads "
                     "(one per physical core, persistent pool), median of %.1f s of CPU work" %
                     (steps, w.N, "the reference's own Registration.cpp compiled against header shims (oracle/_ref)"
                      if kind == "reference" else "CPU oracle port", cores, sum(ts)),
           "min_max_ms": [1e3 * min(ts), 1e3 * max(ts)]}
    if single_thread_steps > 0:
        run1, _ = cpu_registration_runner(w, 1)
        t1 = []
        for _ in range(single_thread_steps):
            t = time.perf_counter()
            run1()
            t1.append(time.perf_counter() - t)
        out["value_1_thread"] = 1.0 / statistics.median(t1)
    return out, med, last


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import kicp_oracle_py as ko
    from oracle import workloads as W
    ko.build()
    w = W.Workload(args.workload)
    cb, sec_per_step, last_pose = time_cpu(w, args.steps, max(args.warmup, 1), single_thread_steps=1)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"pose": last_pose})
    line = {"metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sec_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "impl": "reference",
            "config": workload_config(w), "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ------------------------------------------------------------------------------------------------------ GPU arm
def sha256_file(path):
    import hashlib
    h = hashlib.sha256()
    with open(path, "rb") as f:
        h.update(f.read())
    return h.hexdigest()


def measure_l2_bandwidth(ctx):
    """Read bandwidth of an L2-resident buffer on this GPU (the ceiling of a path whose working set lives in L2): 48 MiB read
    40 times by one grid-stride launch with 128-bit loads (kicp_debug_l2_read_bandwidth), CUDA events, best of 3."""
    import ctypes as C
    from kinematic_icp_b200 import _capi
    L = _capi.lib()
    L.kicp_debug_l2_read_bandwidth.argtypes = [C.c_void_p, C.c_uint64, C.c_int32, C.POINTER(C.c_double)]
    out = C.c_double()
    st = L.kicp_debug_l2_read_bandwidth(ctx.h, 48 << 20, 40, C.byref(out))
    return float(out.value) if st == 0 else None


_REAL_STDOUT = None


def quiet_stdout():
    """stdout carries exactly ONE line (the JSON): anything a library prints there meanwhile (NCCL's version banner under
    NCCL_DEBUG=VERSION, compiler chatter) is sent to stderr by pointing fd 1 at fd 2 until emit() restores it."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(line), flush=True)
    if _REAL_STDOUT is not None:
        os.dup2(2, 1)


def run_pipeline_replay(frames=24, beams=64, n_az=2048):
    """Row (f) of SURVEY.md 8 on the record: a synthetic 64-beam drive (BASELINE.json configs[4] shape, one sequence) written as a
    .kseq file and replayed by the product's native harness, kinematic-icp_b200/bin/kicp_replay — every frame through
    kinematic_icp::pipeline::KinematicICP::RegisterFrame of the C++ facade (float32 ingest, de-skew, filters, both down-samples,
    registration, map update on the device), wall clock over the loop, fastest of repetitions 2-5.  Not part of the timed steps."""
    exe = os.path.join(ROOT, "kinematic-icp_b200", "bin", "kicp_replay")
    if not os.path.exists(exe):
        return {"unavailable": "kinematic-icp_b200/bin/kicp_replay not built"}
    from oracle import sequences as S
    with tempfile.TemporaryDirectory() as d:
        seq = S.make_sequence(n_frames=frames, beams=beams, n_az=n_az, seed=4242, deskew=True)
        kseq, tum = os.path.join(d, "drive.kseq"), os.path.join(d, "drive.tum")
        S.write_kseq(seq, kseq)
        out = {}
        for name, extra in (("pinned", []), ("pageable", ["--pageable"])):
            r = subprocess.run([exe, kseq, tum, "--repeat", "5"] + extra, capture_output=True, text=True, timeout=300)
            lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
            if r.returncode != 0 or not lines:
                return {"unavailable": "kicp_replay failed: " + r.stderr.strip()[-200:]}
            out[name] = json.loads(lines[-1])
    # a 24-frame drive lasts ~16 ms of wall clock, so one hiccup of the box halves a single figure: five repetitions, the fastest after
    # the first is the value, all of them are listed
    fps = lambda o: o.get("frames_per_s_best", o["frames_per_s"])
    return {"metric": "frames/s through KinematicICP::RegisterFrame (offline replay, 1 sequence)", "value": fps(out["pinned"]),
            "ms_per_frame": 1e3 / fps(out["pinned"]) if fps(out["pinned"]) > 0 else None, "pageable_host_buffers": fps(out["pageable"]),
            "repetition_seconds": {k: v.get("repetition_seconds") for k, v in out.items()}, "frames": frames,
            "points_per_frame": out["pinned"]["points_per_frame"], "harness": "kinematic-icp_b200/bin/kicp_replay (C++, float32 ingest, de-skew on)",
            "data": "synthetic %d-beam x %d drive" % (beams, n_az)}


def main():
    args = parse_args()
    quiet_stdout()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import ctypes as C

    import numpy as np
    import torch

    import kinematic_icp_b200 as kb
    from kinematic_icp_b200 import _capi
    from oracle import kicp_oracle_py as ko
    from oracle import workloads as W

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus %d needs torchrun --nproc-per-node %d" % (args.gpus, args.gpus))
        args.gpus = world
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    ko.build()
    if rank == 0:
        w = W.Workload(args.workload)  # builds (and caches) once
    if world > 1:
        dist.barrier()
    if rank != 0:
        w = W.Workload(args.workload)

    ctx = kb.Context(local_rank)
    gm = kb.VoxelHashMap(ctx, w.voxel_size, w.max_range, w.max_points_per_voxel)
    gm.load_voxels(*w.map.export_voxels())  # replicated on every GPU
    reg = kb.KinematicRegistration()  # reference defaults: 10 iterations, 1e-3, adaptive regularisation

    if world > 1:
        if args.comm == "nccl":
            if rank == 0:
                uid = torch.tensor(list(kb.comm_unique_id()), dtype=torch.uint8, device=dev)
            else:
                uid = torch.empty(_capi.KICP_UNIQUE_ID_BYTES, dtype=torch.uint8, device=dev)
            dist.broadcast(uid, 0)
            ctx.comm_init(bytes(uid.cpu().tolist()), world, rank)
        else:  # fused exchange over NVLink peer memory: all-gather the CUDA-IPC handles of the mailboxes
            mine = torch.tensor(list(ctx.p2p_handle()), dtype=torch.uint8, device=dev)
            allh = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(allh, mine)
            ctx.p2p_init([bytes(h.cpu().tolist()) for h in allh], world, rank)

    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
    flush_buf = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)

    def flush_l2(i):
        if not args.no_flush:
            with torch.cuda.stream(stream):
                flush_buf.fill_(i & 0xFF)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    try:
        gpu_uuid = torch.cuda.get_device_properties(dev).uuid
    except Exception:
        gpu_uuid = None
    sampler = NvmlSampler(local_rank, gpu_uuid)
    if rank == 0:
        sampler.start()

    def timed_loop(enqueue, steps, warmup, profile=False):
        """W untimed warm-up steps, then K steps each bracketed by CUDA events on the launching stream, with an
        (untimed) L2 flush before every step.  Returns (sum of step ms as max over ranks, kernel profile, step ms)."""
        for i in range(warmup):
            flush_l2(i)
            enqueue(i)
        ctx.synchronize()
        barrier()
        if profile:
            ctx.profile_begin()
        sampler.active = True  # clocks are sampled only inside timed regions
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for i in range(steps):
            flush_l2(i)
            ev[i][0].record(stream)
            enqueue(warmup + i)
            ev[i][1].record(stream)
        prof = ctx.profile_end() if profile else None
        ctx.synchronize()
        sampler.active = False
        barrier()
        step_ms = [a.elapsed_time(b) for a, b in ev]
        return max_over_ranks(sum(step_ms)), prof, step_ms

    params = reg._params()
    last7, odom7 = _capi.as_pose(w.last_pose), _capi.as_pose(w.rel_odom)

    def run_mode(sharded):
        """One layout (whole scan per rank / contiguous index range per rank): HBM-resident `value`, then the e2e variants
        through the synchronous host-pointer calls.  Returns a dict."""
        lo, hi = kb.shard_range(w.N, world, rank) if sharded else (0, w.N)
        shard = np.ascontiguousarray(w.scan[lo:hi])
        scan = kb.Scan(ctx, len(shard))
        scan.upload(shard)
        results = [kb.pinned_result() for _ in range(args.steps + args.warmup)]

        def enqueue_resident(i):
            reg.enqueue(scan, gm, w.last_pose, w.rel_odom, w.tau, results[i], sharded=sharded)

        launches0 = ctx.launch_count
        total_ms, prof, _ = timed_loop(enqueue_resident, args.steps, args.warmup, profile=True)
        launches = int(round((ctx.launch_count - launches0) * args.steps / float(args.steps + args.warmup)))
        timing = ctx.last_timing()  # CTA 0 of this rank, last registration: [pass][windows, barrier wait, reduce(+exchange), solve] ns
        jobs = world if (world > 1 and not sharded) else 1  # replicas: every rank finishes its own registrations
        out = {"value": jobs * args.steps / (total_ms * 1e-3), "ms_per_step": total_ms / args.steps, "prof": prof,
               "launches": launches, "result": results[args.warmup], "last_result": results[-1], "n_local": hi - lo,
               "timing": timing}

        # e2e: host buffers through the public synchronous call, copies inside the timed region
        out_pose = np.empty(7)
        res_host = kb.RegResult()
        L = _capi.lib()

        def make_call(buf, dtype):
            fn = (L.kicp_register_points_sharded if sharded else L.kicp_register_points)

            def call(i):
                st = fn(gm.h, buf.ctypes.data, len(buf), dtype, 0, 0, 0, 0, _capi.dp(last7), _capi.dp(odom7), float(w.tau),
                        C.byref(params), _capi.dp(out_pose), C.byref(res_host))
                assert st == 0, (st, L.kicp_last_error())
            return call

        variants = {}
        shard32 = shard.astype(np.float32)
        for name, src, dtype in (("pinned_f64", shard, _capi.KICP_DTYPE_F64), ("pageable_f64", shard, _capi.KICP_DTYPE_F64),
                                 ("pinned_f32", shard32, _capi.KICP_DTYPE_F32), ("pageable_f32", shard32, _capi.KICP_DTYPE_F32)):
            if name.startswith("pinned"):
                buf = kb.pinned_empty(src.shape, src.dtype)
                buf[:] = src
            else:
                buf = np.array(src, copy=True)  # ordinary (pageable) numpy storage, like std::vector
            ms, _, _ = timed_loop(make_call(buf, dtype), args.steps, args.warmup)
            variants[name] = {"value": jobs * args.steps / (ms * 1e-3), "ms_per_step": ms / args.steps,
                              "h2d_bytes_per_step": int(buf.nbytes) * (world if sharded else jobs)}
            out["e2e_pose_" + name] = out_pose.copy()
        out["e2e"] = variants
        out["d2h_bytes_per_step"] = int(C.sizeof(kb.RegResult)) * world
        scan.close()
        return out

    primary_sharded = world > 1 and args.mode == "sharded"
    main_run = run_mode(primary_sharded)
    replicas_run = run_mode(False) if (world > 1 and primary_sharded) else None
    # ---- sustained load (N = 1): many registrations back to back in ONE timed region, every one behind an L2 flush; the time of the
    # same number of flushes alone is measured right after and subtracted.  The 20-step `value` above keeps the GPU busy for a few
    # milliseconds; this keeps it busy for ~0.4 s (clocks and throttle reasons are sampled through it).
    sustained = None
    if world == 1 and args.sustained > 0:
        try:
            scan_s = kb.Scan(ctx, w.N)
            scan_s.upload(w.scan)
            res_s = kb.pinned_result()

            def back_to_back(k, with_registration):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for i in range(k):
                    flush_l2(i)
                    if with_registration:
                        reg.enqueue(scan_s, gm, w.last_pose, w.rel_odom, w.tau, res_s)
                e1.record(stream)
                ctx.synchronize()
                return e0.elapsed_time(e1)

            back_to_back(10, True)
            sampler.active = True
            t_both = back_to_back(args.sustained, True)
            sampler.active = False
            t_flush = back_to_back(args.sustained, False)
            per_ms = (t_both - t_flush) / args.sustained
            d_s = ko.pose_delta(res_s.pose_np(), main_run["result"].pose_np())
            sustained = {"registrations": args.sustained, "value": 1e3 / per_ms, "unit": UNIT, "ms_per_step": per_ms,
                         "region_ms": t_both, "flushes_alone_ms": t_flush, "pose_delta_vs_timed_run": [d_s[0], d_s[1]],
                         "note": "one CUDA-event pair around %d x (L2 flush + registration) on the library's stream, minus the same number "
                                 "of flushes alone; frame resident in HBM" % args.sustained}
            scan_s.close()
        except Exception as e:  # never let the extra figure take the bench line down
            sustained = {"unavailable": repr(e)[:200]}
    clocks = sampler.stop() if rank == 0 else None

    # ---- cross-rank identity of what the sharded run produced (every rank must hold the same pose and the same sums) ----
    cross_rank_identical = None
    if world > 1 and primary_sharded:
        r = main_run["result"]
        mine = torch.from_numpy(np.concatenate([r.pose_np(), np.ctypeslib.as_array(r.sums).ravel(),
                                                [float(r.iterations)]])).to(dev)
        allv = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allv, mine)
        same = all(torch.equal(allv[0].view(torch.int64), v.view(torch.int64)) for v in allv)
        cross_rank_identical = bool(same)
        assert same, "ranks disagree on the sharded registration result"

    # ---- work counters and per-pass device timings of one extra (untimed) registration --------------------------------
    lo, hi = kb.shard_range(w.N, world, rank) if primary_sharded else (0, w.N)
    scan = kb.Scan(ctx, hi - lo)
    scan.upload(np.ascontiguousarray(w.scan[lo:hi]))
    ctx.set_option("stats", 1)
    res_stats = kb.pinned_result()
    reg.enqueue(scan, gm, w.last_pose, w.rel_odom, w.tau, res_stats, sharded=primary_sharded)
    probes, cands, lines, _ = ctx.last_stats()
    ctx.set_option("stats", 0)
    scan.close()
    # per-rank pass anatomy (max over ranks of each column, median over the passes of the last timed registration)
    tim = main_run["timing"][: max(int(main_run["result"].iterations), 1)] / 1e3  # us
    anatomy = [float(np.median(tim[:, k])) for k in range(6)]
    if world > 1:
        t = torch.tensor(anatomy, dtype=torch.float64, device=dev)
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tmin = t.clone()
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        anatomy_max, anatomy_min = tmax.tolist(), tmin.tolist()
    else:
        anatomy_max = anatomy_min = anatomy

    # ---- parity of what was just timed ------------------------------------------------------------------------
    if rank == 0:
        iters = int(main_run["result"].iterations)
        pose_ref, st_ref = w.map.register(w.scan, w.last_pose, w.rel_odom, w.tau, threads=physical_cores())
        deltas = [ko.pose_delta(main_run["result"].pose_np(), pose_ref)]
        deltas += [ko.pose_delta(main_run["e2e_pose_" + k], pose_ref) for k in main_run["e2e"]]
        if replicas_run is not None:
            deltas.append(ko.pose_delta(replicas_run["result"].pose_np(), pose_ref))
        pose_delta = {"translation_m": max(d[0] for d in deltas), "rotation_rad": max(d[1] for d in deltas),
                      "iterations_gpu": iters, "iterations_cpu": int(st_ref.iterations),
                      "tolerance": "1e-6 m / 1e-7 rad vs the CPU oracle (sequential-order FP64 restatement); float32 uploads "
                                   "included (the workload's coordinates are float32-representable)"}
        assert pose_delta["translation_m"] <= 1e-6 and pose_delta["rotation_rad"] <= 1e-7, pose_delta
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, result_arrays(main_run["last_result"]))
        cpu_baseline = None
        if world == 1 and not args.no_cpu_baseline:
            cpu_baseline, _, _ = time_cpu(w, 5, 1, single_thread_steps=1)

        replay = None
        if world == 1 and args.workload == 4 and not args.no_cpu_baseline and not args.no_replay:
            try:
                replay = run_pipeline_replay()
            except Exception as e:  # the extra figure must never take the bench line down
                replay = {"unavailable": repr(e)[:200]}

        # ---- roofline of the registration kernel ---------------------------------------------------------------
        cbar, kbar = w.map.neighbourhood_stats(w.scan, w.prior)
        a_pt = 16.0 + 27.0 * 16.0 + cbar * 16.0  # SURVEY.md 8(d): logical gather bytes per point per pass
        n_local = main_run["n_local"]
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy)"
        else:
            peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
        prof = main_run["prof"]
        roofline = None
        if prof is not None and prof.assoc_launches > 0:
            passes_per_launch = prof.assoc_iterations / float(prof.assoc_launches)
            t_launch = prof.assoc_ms / prof.assoc_launches * 1e-3
            bytes_per_launch = passes_per_launch * n_local * a_pt
            achieved = bytes_per_launch / t_launch / 1e9
            # what the kernel really moves from L2/HBM into the SMs, from its own counters: two 16-byte hash slots per probe,
            # 128 bytes per line of candidate points, the scan point and the winner's line once per point and pass
            touched_per_pass = (probes * 32.0 + lines * 128.0) / max(iters, 1) + n_local * (24.0 + 128.0)
            l2_peak = measure_l2_bandwidth(ctx)
            t_pass = t_launch / max(passes_per_launch, 1e-9)
            touched_gbs = touched_per_pass / t_pass / 1e9
            traffic, traffic_note = None, "no ncu capture of this build of kicp_register.cu under profiles/ (profiles/ncu_traffic.json)"
            ncu_path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
            src_sha = sha256_file(os.path.join(ROOT, "kinematic-icp_b200", "csrc", "kicp_register.cu"))
            if os.path.exists(ncu_path) and args.workload == 4 and world == 1:
                tj = json.load(open(ncu_path))
                if tj.get("kernel_source_sha256") == src_sha:
                    traffic = tj.get("dram_bytes_per_launch")
                    traffic_note = "dram__bytes_read+write per launch, ncu --set full capture of this very source (%s)" % tj.get("source")
                else:
                    traffic_note = "profiles/ncu_traffic.json was captured for another build of kicp_register.cu: not reported"
            roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                        "traffic": traffic, "traffic_note": traffic_note, "kernel": "k_register<true>",
                        "launch_us": t_launch * 1e6, "passes_per_launch": passes_per_launch, "kernel_us": t_pass * 1e6,
                        "launches_timed": int(prof.assoc_launches), "iterations_timed": int(prof.assoc_iterations),
                        "algorithmic_bytes_per_launch": bytes_per_launch, "algorithmic_bytes_per_point": a_pt,
                        "mean_candidates_per_point": cbar, "mean_occupied_voxels_of_27": kbar, "peak_source": peak_src,
                        "touched": {"bytes_per_pass": touched_per_pass, "achieved_gbs": touched_gbs, "l2_read_peak_gbs": l2_peak,
                                    "frac_of_l2_peak": (touched_gbs / l2_peak) if l2_peak else None, "probes_per_point_per_pass": probes / max(iters, 1) / n_local,
                                    "candidates_per_point_per_pass": cands / max(iters, 1) / n_local,
                                    "lines_per_point_per_pass": lines / max(iters, 1) / n_local,
                                    "note": "bytes the kernel itself requests from L2 per pass, from its device-side counters (option "
                                            "'stats': 32 B per hash probe, 128 B per line of candidate points, the scan point and the "
                                            "winner's line per point), against the L2 read bandwidth measured on this GPU in this run — "
                                            "the physical counterpart of the logical figure above"},
                        "note": "achieved/frac = LOGICAL gather bytes of SURVEY.md 8(d) (16 + 27*16 + c*16 per point and pass, c = all "
                                "%.0f points of the 27 voxels) / CUDA-event duration, against the measured HBM copy peak: the kernel prunes "
                                "the neighbourhood exactly (%.1f of those candidates per point are evaluated) and the map is served from "
                                "L2, so this is not a physical HBM fraction — see `touched` and `traffic` for what moves" %
                                (cbar, cands / max(iters, 1) / n_local)}
        e2e_main = main_run["e2e"]["pinned_f32"]
        line = {
            "metric": METRIC, "value": main_run["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": main_run["ms_per_step"], "higher_is_better": True,
            "scaling": "strong" if (world == 1 or primary_sharded) else "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(w, {
                "parallelism": ("1 GPU" if world == 1 else ("scan sharded by index range over %d GPUs, map replicated, "
                                "per-iteration exchange of 8 doubles: %s" % (world, "fused into the persistent kernel over NVLink peer memory"
                                if args.comm == "p2p" else "NCCL allreduce") if primary_sharded else
                                "%d independent replicas" % world)),
                "l2": "flushed before every timed step (%d MiB write, untimed)" % (L2_FLUSH_BYTES >> 20)
                      if not args.no_flush else "NOT flushed (diagnostic run)",
                "iterations_per_registration": iters}),
            "ms_per_iter": main_run["ms_per_step"] / max(iters, 1),
            "clocks": clocks,
            "e2e": {"value": e2e_main["value"], "unit": UNIT, "h2d_bytes_per_step": e2e_main["h2d_bytes_per_step"],
                    "d2h_bytes_per_step": main_run["d2h_bytes_per_step"], "ms_per_step": e2e_main["ms_per_step"],
                    "host_memory": "pinned float32 xyz — what the reference's callers hold (PointCloud2 FLOAT32 fields, widened to double by "
                                   "RosUtils.cpp:30-39) — through kicp_register_points; the float64 / pageable variants are alongside",
                    "variants": {k: {"value": v["value"], "ms_per_step": v["ms_per_step"], "h2d_bytes_per_step": v["h2d_bytes_per_step"]}
                                 for k, v in main_run["e2e"].items()}},
            "gpu_launches": main_run["launches"],
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "pose_delta_vs_cpu": pose_delta,
            "pass_anatomy_us": {"columns": ["certificate phase", "its grid barrier", "search phase (CTA 0)", "barrier wait", "reduce (+ exchange)", "solve"],
                                "median_over_passes_max_over_ranks": anatomy_max, "min_over_ranks": anatomy_min,
                                "note": "device %globaltimer probes on CTA 0 of every rank, last timed registration"},
            "kernel_time_split_ms_per_step": None if prof is None else {
                "setup launches": prof.prep_ms / max(prof.registrations, 1),
                "registration kernel": prof.assoc_ms / max(prof.registrations, 1),
                "launches_after_convergence": prof.idle_ms / max(prof.registrations, 1)},
        }
        if sustained is not None:
            line["sustained"] = sustained
        if replay is not None:
            line["replay"] = replay
        if cross_rank_identical is not None:
            line["cross_rank_identical"] = cross_rank_identical
        if replicas_run is not None:
            rv = replicas_run["e2e"]["pinned_f32"]
            line["replicas"] = {"value": replicas_run["value"], "unit": UNIT, "e2e": rv["value"], "scaling": "weak",
                                "note": "BASELINE.json configs[4] layout: %d independent registrations, one per GPU, no communication; "
                                        "aggregate scans/s (HBM-resident / pinned-host e2e)" % world}
        emit(line)
    gm.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
