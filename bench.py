#!/usr/bin/env python
"""Headline benchmark: Taylor steps/s (fp64, batch) of outer_ss_long_term_batch on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

The benchmark writes nothing into the source tree: the helpers it compiles at run time (the generated CPU stepper, the
C++ end-to-end tool) go to a temporary directory that is removed at exit.

Workload (BASELINE.json configs[1]): the 6-body outer Solar System of benchmark/outer_ss_long_term_batch.cpp
(model::nbody(6), masses/G/ICs of :60-94, high_accuracy = true, tol = eps -> order 20), 1,048,576 perturbed
initial conditions PER GPU (weak scaling), one bench "step" = propagate_until(t = --tfinal years) of the whole
batch from the same initial conditions. Metric: lane-steps (accepted Taylor steps summed over lanes, the
n_steps field of get_propagate_res()) per second, whole job.

Printed JSON line (see the task contract): value = device-timed whole-job throughput with inputs resident in
HBM; e2e = the same through the host-buffer API (H2D of state/time/t_final from pinned memory + D2H of the
final state and results inside the timed region); roofline = algorithmic bytes (B_tape of SURVEY.md 8(d)) /
propagate-kernel time vs the measured HBM copy bandwidth; cpu_baseline = the oracle's 8-lane CPU port on all
host cores on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

sys.dont_write_bytecode = True  # no __pycache__ in the source tree either
ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

# Lanes of the fixed sample that --dump-outputs writes: 65,536 lanes x 44 float64 values (lane indices included) = 23 MB.
DUMP_LANES = 1 << 16
DUMP_SEED = 2024


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps of every timed leg (>= 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=1 << 20, help="lanes per GPU")
    ap.add_argument("--tfinal", type=float, default=20.0, help="years propagated per bench step")
    ap.add_argument("--perturb", type=float, default=1e-3)
    ap.add_argument("--cpu-lanes", type=int, default=0, help="lanes of the CPU sample (0 = auto)")
    ap.add_argument("--no-cpp-e2e", action="store_true", help="skip the leg through the drop-in C++ class")
    ap.add_argument("--e2e-sub", type=int, default=1, help="sub-batches the end-to-end leg pipelines through the GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--tape", default="auto", choices=["auto", "hbm", "smem", "smem-notmem", "global", "global-cta", "nbody", "nbody-cta"])
    ap.add_argument("--lanes-per-warp", type=int, default=0)
    ap.add_argument("--lanes-per-thread", type=int, default=0)
    ap.add_argument("--block-threads", type=int, default=0)
    ap.add_argument("--blocks-per-sm", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (final state, times, last step size, "
                         "propagate results) for a fixed sample of %d lanes of rank 0 as float64 DIR/<name>.npy"
                         % DUMP_LANES)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 0:
        ap.error("--warmup must not be negative")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    return args


_SCRATCH = None


def scratch_dir():
    """Private temporary directory for what the benchmark compiles at run time (removed at exit)."""
    global _SCRATCH
    if _SCRATCH is None:
        _SCRATCH = tempfile.TemporaryDirectory(prefix="heyoka_b200_bench_")
    return _SCRATCH.name


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


def measured_traffic(kernel_kind, lane_steps_per_launch):
    """DRAM bytes per launch of the dominant kernel from this round's committed `ncu --set full` capture
    (profiles/r2_traffic.json, written by profiles/summarise_ncu.py: dram__bytes_read.sum + dram__bytes_write.sum, the
    lane-steps of the profiled launch and the FP64 pipe utilisation); the kernel's DRAM traffic is proportional to the
    lane-steps. Returns (bytes per launch, capture record) or (None, None)."""
    path = os.path.join(ROOT, "profiles", "r2_traffic.json")
    try:
        with open(path) as f:
            t = json.load(f)[kernel_kind]
        return float(t["dram_bytes"]) / float(t["lane_steps"]) * lane_steps_per_launch, t
    except (OSError, KeyError, ValueError):
        return None, None


def measured_fp64_peak():
    """FP64 peak of the chip, measured by tools/fp64_peak.cu (dependency-free DFMA streams), profiles/r2_fp64_peak.json."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_fp64_peak.json")) as f:
            return float(json.load(f)["dfma_tflops"]), "measured (tools/fp64_peak.cu)"
    except (OSError, KeyError, ValueError):
        return 37.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for k, nm in enumerate(names):
                if len(r) > 5 + k and r[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def workload(args, rank):
    import heyoka_b200 as hb
    from common import outer_ss_batch_state, sys_outer_ss
    sys_ = sys_outer_ss()
    P = hb.Program(sys_, high_accuracy=True)
    st = outer_ss_batch_state(args.batch, perturb=args.perturb, seed=42 + rank)
    return hb, P, st


def cpu_port_run(P, st, tfinal, n_threads, width=8):
    """Time the oracle's driver on `st` (the jet is whatever is installed: the generated straight-line code of
    oracle/codegen.py, or the interpreting port); returns (lane_steps, seconds)."""
    import oracle
    n = st.shape[1]
    o = oracle.OracleIntegrator(P, st, n, mode=oracle.FMA, width=width)
    t0 = time.perf_counter()
    o.propagate_until(tfinal, lockstep=False, n_threads=n_threads)
    dt = time.perf_counter() - t0
    assert np.all(o.t_hi == tfinal)
    return int(o.n_steps.sum()), dt


class CpuBaseline:
    """The CPU arm: generated code (kind "codegen": one straight-line SIMD function per order, gcc -O2 -march=native
    -ffp-contract=fast, the structure of the reference's LLVM-JIT'd stepper, see oracle/codegen.py) in the 4- and
    8-lane variants, the faster of the two on this host; plus the interpreting port as a second figure."""

    def __init__(self, P, cores, perturb):
        import codegen
        import oracle
        from common import outer_ss_batch_state
        self.P, self.cores, self.oracle, self.codegen = P, cores, oracle, codegen
        codegen.BUILD = scratch_dir()
        self.jets = {w: codegen.Jet(P, w) for w in (4, 8)}  # compiled outside of every timed region
        cal = outer_ss_batch_state(8 * cores, perturb=perturb, seed=7)
        self.rates = {}
        for w, j in self.jets.items():
            j.install(oracle.lib)
            cpu_port_run(P, cal, 1.0, cores, w)  # page in
            s, dt = cpu_port_run(P, cal, 4.0, cores, w)
            self.rates[w] = s / dt
        self.width = max(self.rates, key=self.rates.get)
        # The interpreting port (round 1's baseline), for reference.
        codegen.Jet.uninstall(oracle.lib, 8)
        s, dt = cpu_port_run(P, cal, 4.0, cores, 8)
        self.interp_rate = s / dt
        self.jets[8].install(oracle.lib)

    def run(self, st, tfinal):
        return cpu_port_run(self.P, st, tfinal, self.cores, self.width)

    def describe(self, value, sample):
        return {"value": value, "unit": "lane-steps/s", "cores": self.cores, "kind": "codegen", "simd_lanes": self.width,
                "calibration_lane_steps_per_s": {"codegen_w%d" % w: r for w, r in self.rates.items()},
                "interpreting_port_lane_steps_per_s": self.interp_rate,
                "per_core_us_per_lane_step": 1e6 * self.cores / value, "sample": sample}


def cpu_sample_lanes(args, cores, rate_per_core=2.0e5):
    if args.cpu_lanes:
        return args.cpu_lanes
    # ~15 s of CPU work at the calibrated rate (lane-steps/s per core).
    steps_per_lane = max(args.tfinal / 0.38, 1.0)
    lanes = int(15.0 * cores * rate_per_core / steps_per_lane)
    return int(min(max(lanes // (8 * cores), 1) * 8 * cores, args.batch))


def host_cores():
    """Usable host cores: the affinity mask, capped by the cgroup CPU quota (the GPU boxes show 128 logical CPUs
    but run under a 16-CPU quota; oversubscribing it only adds scheduling noise)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except (OSError, ValueError):
        pass
    return n


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path, timed on the host cores. The real
    reference cannot be built in this image (no LLVM/Boost/fmt/spdlog/TBB); its stepper is restated as GENERATED
    straight-line SIMD code (kind: "codegen", see CpuBaseline), on a bounded sample of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    _, P, _ = workload(argparse.Namespace(**{**vars(args), "batch": 8}), 0)
    from common import outer_ss_batch_state
    cores = host_cores()
    cb = CpuBaseline(P, cores, args.perturb)
    lanes = cpu_sample_lanes(args, cores, cb.rates[cb.width] / cores)
    lanes = max(8 * cores, lanes // max(args.steps, 1))
    st = outer_ss_batch_state(lanes, perturb=args.perturb, seed=42)
    for _ in range(min(args.warmup, 1)):
        cb.run(st[:, :8 * cores], min(args.tfinal, 2.0))
    tot_steps, tot_t = 0, 0.0
    for _ in range(args.steps):
        s, dt = cb.run(st, args.tfinal)
        tot_steps += s
        tot_t += dt
    val = tot_steps / tot_t
    sample = "%d lanes x propagate_until(%g yr) per step, %d steps, %d threads" % (lanes, args.tfinal, args.steps, cores)
    print(json.dumps({
        "impl": "reference", "metric": "taylor_lane_steps_per_s", "value": val, "unit": "lane-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "outer_ss_long_term_batch 6-body fp64 order 20 high_accuracy, t_final %g yr" % args.tfinal,
                   "lanes": lanes},
        "cpu_baseline": cb.describe(val, sample),
        "e2e": {"value": val, "unit": "lane-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def dump_outputs(out_dir, n, dev, arrays):
    """Writes the lanes of a fixed sample (DUMP_LANES lanes drawn with DUMP_SEED, ascending; all lanes if the batch is
    smaller) of each device array [..., n] as float64 out_dir/<name>.npy, plus their indices as lanes.npy. The inputs
    depend only on the arguments, so two builds run with the same arguments can be compared file by file."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    lanes = np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=min(n, DUMP_LANES), replace=False))
    idx = torch.from_numpy(lanes).to(dev)
    np.save(os.path.join(out_dir, "lanes.npy"), lanes.astype(np.float64))
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.index_select(t.dim() - 1, idx).double().cpu().numpy())


def cpp_class_e2e(batch, steps, tfinal, perturb):
    """The same workload through the drop-in C++ class (tools/bench_cpp_e2e.cpp): host std::vector buffers in and out,
    the call a heyoka user makes. One line per host_sync mode; an error record if the tool cannot be built."""
    exe = os.path.join(scratch_dir(), "bench_cpp_e2e")
    src = os.path.join(ROOT, "tools", "bench_cpp_e2e.cpp")
    lib = os.path.join(ROOT, "heyoka_b200", "lib")
    try:
        subprocess.run(["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"), src, "-o", exe, "-L" + lib,
                        "-lheyoka_b200", "-Wl,-rpath," + lib], check=True, capture_output=True)
        res = subprocess.run([exe, str(batch), str(steps), repr(float(tfinal)), repr(float(perturb))], capture_output=True,
                             text=True, timeout=600, check=True)
        return [json.loads(line) for line in res.stdout.splitlines() if line.startswith("{")]
    except Exception as e:  # noqa: BLE001 - a reported extra, never fatal for the bench line
        return {"error": "%s: %s" % (type(e).__name__, e)}


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: heyoka_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    hb, P, st_host = workload(args, rank)
    n = args.batch
    b = hb.Batch(P, n, device=local_rank)
    stream = torch.cuda.current_stream()
    b.set_stream(stream.cuda_stream)
    if args.tape != "auto" or args.lanes_per_warp or args.lanes_per_thread or args.block_threads or args.blocks_per_sm:
        b.set_kernel(args.tape, args.lanes_per_warp, args.lanes_per_thread, args.block_threads, args.blocks_per_sm)
    kinfo = b.kernel_info()
    ptrs = b.ptrs()

    # Device-resident inputs: initial state, final times; torch owns these buffers.
    d_state0 = torch.from_numpy(st_host).to(dev)
    d_tf = torch.full((n,), args.tfinal, dtype=torch.float64, device=dev)
    state_bytes = st_host.nbytes

    def as_tensor(ptr, count, dtype=torch.float64):
        # zero-copy view of a library-owned device buffer through the CUDA array interface
        class _W:
            pass
        w = _W()
        w.__cuda_array_interface__ = {"shape": (count,), "typestr": "<f8" if dtype == torch.float64 else "<i8",
                                      "data": (int(ptr), False), "version": 2}
        return torch.as_tensor(w, device=dev)

    t_state = as_tensor(ptrs.state, P.n_eq * n)
    t_thi = as_tensor(ptrs.t_hi, n)
    t_tlo = as_tensor(ptrs.t_lo, n)
    t_nsteps = as_tensor(ptrs.prop_n_steps, n, torch.int64)
    # What the final gather moves (SURVEY.md 8(e)): state, time hi / lo, last_h and the propagate results of every lane,
    # packed into ONE buffer per rank (one all_gather over NVLink).
    small = [t_thi, t_tlo, as_tensor(ptrs.last_h, n), as_tensor(ptrs.prop_min_h, n), as_tensor(ptrs.prop_max_h, n),
             as_tensor(ptrs.prop_outcome, n, torch.int64).view(torch.float64), t_nsteps.view(torch.float64)]
    pack = torch.empty((P.n_eq + len(small)) * n, dtype=torch.float64, device=dev) if world > 1 else None
    gather_buf = torch.empty(world * (P.n_eq + len(small)) * n, dtype=torch.float64, device=dev) if world > 1 else None

    ev_k0, ev_k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kernel_ms = []

    def device_step(timed):
        # inputs already resident in HBM: restore the initial conditions (device-to-device), then propagate
        t_state.copy_(d_state0.reshape(-1))
        t_thi.zero_()
        t_tlo.zero_()
        if timed:
            ev_k0.record(stream)
        flag = b.propagate_until_dev(d_tf.data_ptr())
        if timed:
            ev_k1.record(stream)
        assert flag == 0, "unexpected non-finite state / step limit"
        if world > 1:
            # the only exchange of the path: gather of the final state, times, last_h and propagate results
            pack[:P.n_eq * n].copy_(t_state)
            for k, t in enumerate(small):
                pack[(P.n_eq + k) * n:(P.n_eq + k + 1) * n].copy_(t)
            dist.all_gather_into_tensor(gather_buf, pack)
        if timed:
            torch.cuda.synchronize()
            kernel_ms.append(ev_k0.elapsed_time(ev_k1))

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(args.warmup):
        device_step(False)
    sync_all()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = b.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    ev0.record(stream)
    for _ in range(args.steps):
        device_step(True)
    ev1.record(stream)
    sync_all()
    elapsed_ms = ev0.elapsed_time(ev1)
    lane_steps_rank = int(t_nsteps.sum().item())  # of one bench step (every step repeats the same work)
    if world > 1:
        # The gathered result (after the timed region): every rank's block of the final times is t_final, every state is
        # finite, and this rank's block of the gather is what this rank computed.
        g = gather_buf.view(world, -1)
        assert bool(torch.isfinite(g[:, :P.n_eq * n]).all()), "non-finite state in the gathered result"
        assert bool((g[:, P.n_eq * n:(P.n_eq + 1) * n] == args.tfinal).all()), "a gathered lane is not at t_final"
        assert bool(torch.equal(g[rank, :P.n_eq * n], t_state)), "the gathered block differs from the local state"
    launches = b.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # (Before the end-to-end leg below, which reuses the batch's buffers.)
        dump_outputs(args.dump_outputs, n, dev, {
            "state": t_state.view(P.n_eq, n), "time_hi": t_thi, "time_lo": t_tlo, "last_h": small[2],
            "outcome": small[5].view(torch.int64), "min_h": small[3], "max_h": small[4], "n_steps": t_nsteps})

    # ---- end-to-end through the host-buffer API: pinned host -> device, propagate, device -> pinned host ----
    h_state = torch.from_numpy(st_host).pin_memory()
    h_zero = torch.zeros(n, dtype=torch.float64).pin_memory()
    h_tf = torch.full((n,), args.tfinal, dtype=torch.float64).pin_memory()
    h_out = torch.empty(P.n_eq * n, dtype=torch.float64).pin_memory()
    h_thi = torch.empty(n, dtype=torch.float64).pin_memory()
    h_tlo = torch.empty(n, dtype=torch.float64).pin_memory()
    h_lasth = torch.empty(n, dtype=torch.float64).pin_memory()
    h_oc = torch.empty(n, dtype=torch.int64).pin_memory()
    h_mn = torch.empty(n, dtype=torch.float64).pin_memory()
    h_mx = torch.empty(n, dtype=torch.float64).pin_memory()
    h_ns = torch.empty(n, dtype=torch.int64).pin_memory()
    import ctypes as C
    dp = lambda t: C.cast(C.c_void_p(t.data_ptr()), C.POINTER(C.c_double))  # noqa: E731
    h2d = state_bytes + 3 * 8 * n
    d2h = state_bytes + 3 * 8 * n + 4 * 8 * n

    # One call of the host-buffer entry point (hy_batch_propagate_until_host) on a batch made of E2E_SUB sub-batches on
    # this GPU (the same device listed E2E_SUB times): every sub-batch uploads, runs and downloads on its own stream, so
    # the transfers of one overlap the kernels of the others. Same lanes, same work as the device-timed leg.
    b2 = hb.Batch(P, n, device=[local_rank] * args.e2e_sub) if args.e2e_sub > 1 else b

    def e2e_step():
        hb.check(hb.lib.hy_batch_propagate_until_host(
            b2._h, dp(h_state), None, dp(h_zero), dp(h_zero), dp(h_tf), None, None, 0, dp(h_out), dp(h_thi), dp(h_tlo),
            dp(h_lasth), C.cast(C.c_void_p(h_oc.data_ptr()), C.POINTER(C.c_int64)), dp(h_mn), dp(h_mx),
            C.cast(C.c_void_p(h_ns.data_ptr()), C.POINTER(C.c_uint64))))

    e2e_step()
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_e2e = args.steps
    e0.record(stream)
    t_wall = time.perf_counter()
    for _ in range(n_e2e):
        e2e_step()
    e1.record(stream)
    sync_all()
    e2e_ms = max(e0.elapsed_time(e1), 1e3 * (time.perf_counter() - t_wall))
    e2e_lane_steps = int(h_ns.sum().item())
    assert bool((h_thi == args.tfinal).all())

    # ---- reductions over ranks ----
    if world > 1:
        tt = torch.tensor([elapsed_ms, e2e_ms, float(np.mean(kernel_ms))], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        elapsed_ms, e2e_ms, k_ms = [float(x) for x in tt.tolist()]
        cc = torch.tensor([lane_steps_rank, e2e_lane_steps, launches], dtype=torch.int64, device=dev)
        dist.all_reduce(cc, op=dist.ReduceOp.SUM)
        lane_steps_all, e2e_all, launches_all = [int(x) for x in cc.tolist()]
    else:
        k_ms = float(np.mean(kernel_ms))
        lane_steps_all, e2e_all, launches_all = lane_steps_rank, e2e_lane_steps, launches

    if rank == 0:
        peaks, peak_kind = measured_peaks()
        costs = P.costs()
        value = lane_steps_all * args.steps / (elapsed_ms * 1e-3)
        e2e_val = e2e_all * n_e2e / (e2e_ms * 1e-3)
        # roofline of the dominant kernel (k_propagate) on this rank: algorithmic bytes / launch duration
        ach = lane_steps_rank * costs["b_tape"] / (k_ms * 1e-3) / 1e9
        peak = float(peaks["hbm_gbs"])
        traffic, capture = measured_traffic(kinfo["tape"], lane_steps_rank)
        fp64_peak, fp64_peak_kind = measured_fp64_peak()
        fp64_model = lane_steps_rank * costs["flops"] / (k_ms * 1e-3) / 1e12
        out = {
            "metric": "taylor_lane_steps_per_s", "value": value, "unit": "lane-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {
                "workload": "outer_ss_long_term_batch 6-body fp64 order %d high_accuracy, batch %d per GPU, "
                            "propagate_until(%g yr) per step" % (P.order, n, args.tfinal),
                "n_eq": P.n_eq, "n_uvars": P.n_uvars, "order": P.order, "lanes_per_gpu": n,
                "lane_steps_per_step": lane_steps_all, "perturb": args.perturb,
                "cache": "inputs larger than L2: state %.0f MB + per-warp derivative tapes (GBs) vs 126 MB of L2; ICs "
                         "restored device-to-device before every step" % (state_bytes / 1e6),
                "parallelism": "lanes sharded across %d GPU(s), final-state all_gather" % world,
            },
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "traffic": traffic, "peak_kind": peak_kind,
                         # What really bounds the kernel: it moves ~20 B of DRAM traffic per lane-step (the tape lives
                         # on chip), so the contract's B_tape figure above is an algorithmic equivalent; the binding
                         # resources are the FP64 pipe and instruction issue.
                         "true_bound": "fp64 pipe / instruction issue",
                         "fp64_peak_tflops": fp64_peak, "fp64_peak_kind": fp64_peak_kind,
                         "fp64_frac": fp64_model / fp64_peak,
                         "fp64_pipe_pct": None if capture is None else capture.get("fp64_pipe_pct"),
                         "warp_inst_per_lane_step": None if capture is None else capture.get("warp_inst_per_lane_step"),
                         "dram_bytes_per_lane_step": None if capture is None
                         else capture["dram_bytes"] / capture["lane_steps"],
                         "capture": None if capture is None else capture.get("source"),
                         "kernel": ("k_nb<LT=%d,prop>" % kinfo["lanes_per_warp"]) if kinfo["tape"].startswith("nbody")
                         else ("k_coop<L=%d,N=%d,prop>" % (kinfo["lanes_per_warp"], kinfo["lanes_per_thread"])
                               if kinfo["tape"] == "smem" else "k_hbm<prop>"), "kernel_config": kinfo,
                         "kernel_ms": k_ms, "b_tape_bytes_per_lane_step": costs["b_tape"],
                         "b_min_bytes_per_lane_step": costs["b_min"],
                         "frac_b_min": lane_steps_rank * costs["b_min"] / (k_ms * 1e-3) / 1e9 / peak,
                         "model_flops_per_lane_step": costs["flops"],
                         "fp64_tflops_model": fp64_model},
            "e2e": {"value": e2e_val, "unit": "lane-steps/s", "h2d_bytes_per_step": h2d * world,
                    "d2h_bytes_per_step": d2h * world, "ms_per_step": e2e_ms / n_e2e,
                    "call": "hy_batch_propagate_until_host", "sub_batches_per_gpu": args.e2e_sub},
            "gpu_launches": launches_all,
            "clocks": clocks,
        }
        if world == 1 and not args.no_cpp_e2e:
            out["e2e_cpp_class"] = cpp_class_e2e(n, args.steps, args.tfinal, args.perturb)
        if not args.no_cpu_baseline and world == 1:
            cores = host_cores()
            cb = CpuBaseline(P, cores, args.perturb)
            lanes = cpu_sample_lanes(args, cores, cb.rates[cb.width] / cores)
            s, dt = cb.run(st_host[:, :lanes], args.tfinal)
            out["cpu_baseline"] = cb.describe(
                s / dt, "generated straight-line SIMD stepper (oracle/codegen.py; the reference's LLVM JIT is not "
                        "buildable here): first %d lanes of the same batch, propagate_until(%g yr), %d threads, %.1f s"
                % (lanes, args.tfinal, cores, dt))
        print(json.dumps(out))

    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
