#!/usr/bin/env python
"""bench.py -- gate-applications/s and effective state GB/s of the RustQIP gate-application
hot path on B200 (BASELINE.json metric), next to the reference CPU algorithm.

  python bench.py --gpus N --steps K --warmup W            # this framework (one rank per GPU)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port)

One "step" = one full pass of the synthetic circuit over the 2^n state, starting from |0..0>
(set-basis + the whole gate schedule).  Workload at G GPUs (weak scaling): n = 30 + log2(G)
qubits, f64, layer 0 = H on every qubit then depth-40 layers of random {H,T,CNOT}
(generator G of SURVEY.md section 8d, seed 0x5EED0002): BASELINE.json's "N=30 random circuit"
with configs[1]'s gate set; at 8 GPUs n = 33 = configs[4]'s size.
Rank 0 prints ONE JSON line.
"""
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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# BASELINE.json metric: "gate-apps/sec & state GB/s".  `value` is the state GB/s half --
# effective_state_GBps = gate-apps/s * 2 * 2^N * sizeof(amplitude) (BASELINE.md section 2), the
# whole-job aggregate that grows with the GPU count under weak scaling -- and the gate-apps/s
# half travels beside it in "gate_apps_per_s".
METRIC = "effective_state_GBps (= gate_apps_per_s * 2 * 2^N * sizeof(amplitude))"
UNIT = "GB/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n-local", type=int, default=30, help="qubits per GPU (default 30: 16 GiB f64 shard)")
    ap.add_argument("--depth", type=int, default=40)
    ap.add_argument("--dtype", default="f64", choices=["f64", "f32"])
    ap.add_argument("--gate-set", default="H,T,CNOT")
    ap.add_argument("--seed", type=lambda x: int(x, 0), default=0x5EED0002, help="generator seed of the random workload")
    ap.add_argument("--config5", action="store_true",
                    help="BASELINE configs[4] exactly: depth-30 random {H,CZ,CNOT}, seed 0x5EED0005 (N = n-local + log2 gpus: 33 at 8 GPUs)")
    ap.add_argument("--workload", default="random", choices=["random", "qft", "dense4"],
                    help="random: depth-D random layers (BASELINE metric / configs[1], [4]); qft: configs[2]; dense4: configs[3]")
    ap.add_argument("--dense-k", type=int, default=4, help="qubits per dense block of --workload dense4 (4 = BASELINE configs[3]; 5..10: the wide in-place kernels)")
    ap.add_argument("--no-fusion", action="store_true", help="one kernel sweep per gate")
    ap.add_argument("--no-extras", action="store_true", help="skip the unfused / per-kernel / CPU side measurements")
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the state the last timed step computed (a fixed seeded sample of it) to DIR as .npy files")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm times a sample of the gates, not whole steps")
    return args


def ncu_traffic(kernel, algorithmic_bytes):
    """DRAM traffic per launch from the committed ncu capture (profiles/traffic.json), scaled to this size."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[kernel]
        return {"bytes": t["ratio"] * algorithmic_bytes, "source": t["capture"]}
    except Exception:
        return None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = sorted(sm)[len(sm) // 4:] if sm else []  # drop the idle tail of the samples
        return {"sm_mhz": (float(np.median(busy)) if busy else None), "sm_max_mhz": mx,
                "samples": len(sm), "reasons": sorted(reasons)}


# --dump-outputs: at most 2^21 amplitudes with their indices (48 MB in f64), at the same seeded indices in every run
DUMP_AMPS = 1 << 21
DUMP_SEED = 0x5EED00D0
DUMP_CHUNK = 1 << 24


def dump_outputs(st, out_dir, rank, world):
    """Write what a step hands its caller, the 2^n amplitudes of the state, as state_indices.npy (float64 global
    indices, ascending) and state_amplitudes.npy ([re, im] rows in the state's precision): every amplitude when
    2^n <= DUMP_AMPS, else the amplitudes at a fixed seeded sample of indices.  Collective over the ranks."""
    import torch.distributed as dist
    if st.n < DUMP_AMPS.bit_length():
        idx = np.arange(1 << st.n, dtype=np.int64)
    else:
        idx = np.unique(np.random.default_rng(DUMP_SEED).integers(0, 1 << st.n, size=DUMP_AMPS, dtype=np.int64))
    lo = rank * st.local_len
    mine = idx[(idx >= lo) & (idx < lo + st.local_len)] - lo
    amps = np.empty(mine.size, dtype=st.dtype)
    buf = np.empty(min(DUMP_CHUNK, st.local_len), dtype=st.dtype)
    for off in range(0, st.local_len, buf.size):
        a, b = np.searchsorted(mine, [off, off + buf.size])
        st.download(buf, offset=off)
        amps[a:b] = buf[mine[a:b] - off]
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, amps)
        amps = np.concatenate(parts)
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        np.save(os.path.join(out_dir, "state_indices.npy"), idx.astype(np.float64))
        np.save(os.path.join(out_dir, "state_amplitudes.npy"), amps.view(amps.real.dtype).reshape(-1, 2))


def build_workload(args, world):
    from rustqip_b200 import circuits
    g = (world - 1).bit_length()
    n = args.n_local + g
    if args.workload == "qft":
        ops = circuits.qft(n)
        name = "N=%d %s textbook QFT at MatrixOp level (H, controlled phases, final swaps; BASELINE configs[2]) from |0>" % (n, args.dtype)
    elif args.workload == "dense4":
        ops = circuits.config4(n, blocks=args.depth, k=args.dense_k)
        name = "N=%d %s H^n then %d dense %d-qubit Haar blocks on seeded random qubits (BASELINE configs[3]%s)" % (
            n, args.dtype, args.depth, args.dense_k, "" if args.dense_k == 4 else " with wider blocks")
    else:
        ops = circuits.random_circuit(n, args.depth, args.seed, args.gate_set)
        name = "N=%d %s depth-%d random {%s} from |0>, layer 0 = H^n (SURVEY 8d generator, seed 0x%X)" % (
            n, args.dtype, args.depth, args.gate_set, args.seed)
    return n, ops, name


# ------------------------------------------------------------------------------------------
# reference arm: the reference's CPU algorithm (oracle port, OpenMP over output rows)
# ------------------------------------------------------------------------------------------
def _cpu_threads_env():
    """torchrun exports OMP_NUM_THREADS=1 to its workers: the CPU arm is meant to use every host core, and the
    OpenMP threads must stay where their first-touch pages are (set before libgomp initialises)."""
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
    os.environ.setdefault("OMP_PROC_BIND", "spread")
    os.environ.setdefault("OMP_PLACES", "threads")


class CpuRunner:
    """The reference's CPU algorithm on a bounded sample of the workload: out-of-place
    apply_op_overwrite + buffer swap per gate (qip/src/builder.rs:499,514), all 2^n rows per
    gate, OpenMP over rows on every host core (oracle/qip_oracle.c, a C port: the Rust
    reference cannot be built in this image).

    Sample size: one sample must hold >= `min_gates` consecutive gate applications, or its rate is noise
    (round 1: 2-11 gates per sample, 5.5x spread between boxes).  The per-gate cost is linear in 2^n
    (every gate is one out-of-place sweep, memory-bound far beyond the caches), so when `min_gates` gates at
    the full n do not fit `budget_s` the sample runs the low n_run qubits' gates of the same circuit on a
    2^n_run state and the rate is scaled by 2^-(n - n_run) and labelled EXTRAPOLATED."""

    MAX_BYTES = 80 << 30  # two buffers; keeps first-touch time of a step within seconds
    N_RUN_CAP = 30

    def __init__(self, n, ops, dtype, budget_s=20.0, min_gates=10):
        _cpu_threads_env()
        from oracle import qip_oracle as qo
        self.qo = qo
        qo.set_threads(os.cpu_count() or 1)
        self.cores = qo.max_threads()
        self.n = n
        self.all_ops = ops
        self.dtype = dtype
        amp = np.dtype(dtype).itemsize
        avail = os.sysconf("SC_PAGE_SIZE") * os.sysconf("SC_AVPHYS_PAGES")
        n_run = min(n, self.N_RUN_CAP)
        while 2 * (amp << n_run) > min(0.6 * avail, self.MAX_BYTES) and n_run > 20:
            n_run -= 1
        # calibrate the per-gate time at a small size, then take the largest n_run that still gives min_gates per sample
        n_cal = min(n_run, 24)
        self._setup(n_cal)
        t0 = time.perf_counter()
        for _ in range(4):
            self._gate()
        t_cal = (time.perf_counter() - t0) / 4
        while n_run > n_cal and min_gates * t_cal * float(1 << (n_run - n_cal)) > budget_s:
            n_run -= 1
        if n_run != n_cal:
            self._setup(n_run)

    def _setup(self, n_run):
        n = self.n
        self.n_run = n_run
        sample_ops = [op for op in self.all_ops if all(q >= n - n_run for q in op.indices())]
        if n_run != n:  # gates on the low n_run qubits, renumbered; cost per gate is linear in 2^n
            from rustqip_b200.ops import MatrixOp

            def shift(o):
                return MatrixOp(o.kind, [q - (n - n_run) for q in o.indices()], data=o.data, rows=o.rows,
                                n_control=o.n_control, inner=shift(o.inner) if o.inner is not None else None,
                                swap_n=o.swap_n)
            sample_ops = [shift(op) for op in sample_ops]
        self.ops = sample_ops
        self.state = np.zeros(1 << n_run, dtype=self.dtype)
        self.arena = np.zeros_like(self.state)
        self.state[0] = 1
        self.pos = 0
        self._gate()  # touch every page once: first-touch cost is not part of the gate loop
        self._gate()

    def _gate(self):
        op = self.ops[self.pos % len(self.ops)]
        self.pos += 1
        self.qo.apply_op_overwrite(self.n_run, op, self.state, self.arena)
        self.state, self.arena = self.arena, self.state

    def run(self, budget_s, min_gates=10, max_gates=None):
        """-> (gate-apps/s at the full n, gates done, seconds)"""
        done, t0 = 0, time.perf_counter()
        while True:
            self._gate()
            done += 1
            over = time.perf_counter() - t0 > budget_s
            if (over and done >= min_gates) or (max_gates and done >= max_gates) or time.perf_counter() - t0 > 3 * budget_s:
                break
        dt = time.perf_counter() - t0
        return done / dt / float(1 << (self.n - self.n_run)), done, dt

    def describe(self, done, dt):
        return "%d consecutive gates of the workload after 2 untimed page-touch gates, %.1f s, n=%d, %d OpenMP threads (bound)%s" % (
            done, dt, self.n_run, self.cores,
            "" if self.n_run == self.n else " (a %d-gate sample at n=%d does not fit the step budget / host memory: per-gate cost is "
            "linear in 2^n, value scaled by 2^-%d, EXTRAPOLATED)" % (10, self.n, self.n - self.n_run))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    dtype = np.complex128 if args.dtype == "f64" else np.complex64
    n, ops, name = build_workload(args, max(world, args.gpus))
    # the whole --steps K --warmup W run must end within a few minutes
    per_step = max(2.0, min(20.0, 150.0 / max(1, args.steps + args.warmup)))
    runner = CpuRunner(n, ops, dtype, budget_s=per_step)
    vals, done, dt = [], 0, 0.0
    for i in range(args.warmup + args.steps):
        gps, done, dt = runner.run(per_step)
        if i >= args.warmup:
            vals.append(gps)
    v = float(np.median(vals))
    amp = np.dtype(dtype).itemsize
    line = {
        "impl": "reference", "metric": METRIC, "value": v * 2 * amp * (1 << n) / 1e9, "unit": UNIT,
        "gate_apps_per_s": v, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * len(ops) / v,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.dtype,
        "data": "synthetic",
        "config": {"workload": name, "gates_per_step": len(ops), "fusion": None,
                   "state_bytes_per_gpu": None, "l2_policy": "n/a (CPU arm: two 2^n_run-amplitude buffers far beyond the caches)",
                   "parallelism": "OpenMP over output rows, all host cores"},
        "cpu_baseline": {"value": v * 2 * amp * (1 << n) / 1e9, "unit": UNIT, "gate_apps_per_s": v,
                         "cores": runner.cores, "kind": "port",
                         "sample": "each step: " + runner.describe(done, dt) + "; oracle/qip_oracle.c = C restatement of "
                                   "apply_op_overwrite (the Rust reference cannot be built here), OpenMP static over rows; "
                                   "ms_per_step is the whole circuit at this rate"},
        "e2e": {"value": v * 2 * amp * (1 << n) / 1e9, "unit": UNIT, "gate_apps_per_s": v,
                "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------
# this framework
# ------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist
    from rustqip_b200 import _lib, gates
    from rustqip_b200._abi import marshal_ops, prec_of
    from rustqip_b200.state import Context, State

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus %d needs torchrun (one rank per GPU)" % args.gpus)
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    dtype = np.complex128 if args.dtype == "f64" else np.complex64
    amp = np.dtype(dtype).itemsize
    n, ops, name = build_workload(args, world)
    ctx = Context(local_rank)
    stream = torch.cuda.ExternalStream(ctx.stream_handle(), device=torch.device("cuda", local_rank))
    def map_peers(state):
        a, f = state.ipc_export()
        ta = torch.tensor(list(a), dtype=torch.uint8, device="cuda")
        tf = torch.tensor(list(f), dtype=torch.uint8, device="cuda")
        ga = [torch.empty_like(ta) for _ in range(world)]
        gf = [torch.empty_like(tf) for _ in range(world)]
        dist.all_gather(ga, ta)
        dist.all_gather(gf, tf)
        state.ipc_import(b"".join(bytes(x.cpu().tolist()) for x in ga), b"".join(bytes(x.cpu().tolist()) for x in gf))

    def circuits_mod():
        from rustqip_b200 import circuits
        return circuits

    st = State(n, dtype, ctx, rank=rank, world_size=world)
    if world > 1:
        map_peers(st)
    arr, keep = marshal_ops(ops, st.prec)
    sched_bytes = sum(k.nbytes for k in keep if isinstance(k, np.ndarray)) + C.sizeof(arr)
    fusion = not args.no_fusion

    def step(fus=fusion):
        st.set_basis(0)
        st.apply_marshalled(arr, len(ops), fus)

    def sync_all():
        st.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, reps):
        """device time of `reps` calls on the library's stream, max over ranks (ms)."""
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        st.sync()
        e1.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        sync_all()
        return float(ms.item())

    # Warm-up.  The first step also starts the NVRTC compilation of this schedule's specialised pass kernels on the
    # library's background workers (tiered execution: passes run the generic kernel until theirs is ready); the
    # compile wall time is reported, and the remaining warm-up steps run on the generated kernels like the timed ones.
    t_jit = time.perf_counter()
    step()
    j0 = ctx.jit_stats(wait=True)
    jit_wall_ms = (time.perf_counter() - t_jit) * 1e3
    for _ in range(max(args.warmup - 1, 2)):
        step()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    s0 = ctx.launch_stats()
    ctx.profile(True)   # CUDA-event pairs on the library's stream around every tile pass / exchange
    ctx.profile_read()
    ms = timed(step, args.steps)
    prof = ctx.profile_read()
    ctx.profile(False)
    s1 = ctx.launch_stats()
    j1 = ctx.jit_stats()
    launches = s1["all"] - s0["all"]
    tile_passes = (s1["tile_passes"] - s0["tile_passes"]) / args.steps
    exchanges = (s1["exchanges"] - s0["exchanges"]) / args.steps
    fused_gates = (s1["fused_gates"] - s0["fused_gates"]) / args.steps
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(st, args.dump_outputs, rank, world)
    ms_per_step = ms / args.steps
    gates_total = len(ops)
    gps = gates_total / (ms_per_step / 1e3)
    bytes_alg_gate = 2.0 * amp * (1 << n)  # whole job: read + write every amplitude once per gate
    value = gps * bytes_alg_gate / 1e9
    peak, peak_src = peaks()

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "gate_apps_per_s": gps, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": {"workload": name, "gates_per_step": gates_total, "fusion": fusion,
                   "state_bytes_per_gpu": amp << st.n if world == 1 else amp * st.local_len,
                   "l2_policy": "state (>= 1 GiB per GPU) is far larger than the 126 MB L2; no flush needed",
                   "parallelism": "state sharded by the top log2(G) index bits, NVLink P2P qubit migration" if world > 1 else "single GPU"},
        "effective_frac_of_hbm_peak": value / (peak * world),
        "gpu_launches": int(launches),
        "launches_per_step": {"all": launches / args.steps, "fused_tile_passes": tile_passes,
                              "nvlink_exchanges": exchanges, "gates_in_fused_passes": fused_gates},
        "clocks": clocks,
        "generated_kernels": {"tile_passes_on_generated_kernels_in_timed_region": j1["jit_passes"] - j0["jit_passes"],
                              "tile_passes_in_timed_region": j1["tile_passes"] - j0["tile_passes"],
                              "programs_compiled": j0["programs_compiled"], "nvrtc_ms_sum": j0["compile_ms_total"],
                              "first_step_plus_compile_wall_ms": jit_wall_ms, "note": j1["note"],
                              "mode": os.environ.get("QIPB200_JIT", "async (default)")},
    }
    local_bytes = 2.0 * amp * st.local_len  # one sweep of this rank's shard: read + write every amplitude
    if fusion and tile_passes > 0:
        # dominant kernel of the step = the fused tile pass
        # measured live: CUDA-event pairs around every k_tile_pass launch of the timed region, on the launch stream
        avg_ms = prof["tile_ms"] / max(1, prof["tile_passes"])
        gen = (j1["jit_passes"] - j0["jit_passes"]) == (j1["tile_passes"] - j0["tile_passes"])
        line["roofline"] = {"bound": "hbm", "kernel": "%s (fused shared-memory tile pass, %s, %.1f gates per launch)" % (
                                "qip_pass [NVRTC-generated per pass, rustqip_b200/csrc/jit_codegen.cpp]" if gen else "k_tile_pass<%s> [interpreter]" % (
                                    "double" if args.dtype == "f64" else "float"), args.dtype, fused_gates / tile_passes),
                            "achieved": local_bytes / (avg_ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                            "frac": local_bytes / (avg_ms / 1e3) / 1e9 / peak, "peak_source": peak_src,
                            "traffic": (ncu_traffic("qip_pass" if gen else "k_tile_pass", local_bytes) or {}).get("bytes"),
                            "traffic_source": (ncu_traffic("qip_pass" if gen else "k_tile_pass", local_bytes) or {}).get("source"),
                            "algorithmic_bytes_per_launch": local_bytes, "avg_launch_ms": avg_ms,
                            "frac_of_nominal_8TBps": local_bytes / (avg_ms / 1e3) / 1e9 / 8000.0,
                            "share_of_step": prof["tile_ms"] / max(1e-9, ms),
                            "timing": "CUDA-event pair around each of the %d launches of the timed region (rank %d), on the launch stream" % (
                                prof["tile_passes"], rank),
                            "note": "per launch: every amplitude of the shard read once and written once (SURVEY 8d: 2*2^N*16 B), "
                                    "independent of the number of gates folded into the pass"}
    if world > 1 and prof["exchanges"] > 0:
        xms = prof["exchange_ms"] / prof["exchanges"]
        xbytes = amp * st.local_len / 2.0  # per direction: half a shard leaves, half a shard arrives
        line["exchange"] = {"per_step": prof["exchanges"] / args.steps, "avg_ms": xms,
                            "ms_per_step": prof["exchange_ms"] / args.steps, "share_of_step": prof["exchange_ms"] / max(1e-9, ms),
                            "bytes_per_direction": xbytes, "GBps_per_direction": xbytes / (xms / 1e3) / 1e9,
                            "note": "k_pair_exchange + its two flag barriers, CUDA events on rank 0's stream (waiting for the "
                                    "slowest peer at the barrier is inside)"}
        if os.environ.get("QIPB200_PAIRED_SEND", "0") not in ("", "0"):
            # the transfer happens inside the epoch's last tile pass (paired send): what is timed here is the closing
            # barrier (the drain of the queued NVLink writes) and the stand-in kernel where a pass could not send itself
            line["exchange"]["GBps_per_direction"] = None
            line["exchange"]["note"] = ("QIPB200_PAIRED_SEND: the migration is fused into the epoch's last tile pass (its launches are "
                                        "counted under roofline.avg_launch_ms); avg_ms here = closing flag barrier (+ stand-in kernel)")

    # ---- correctness of the live configuration (VERDICT r1 #1b): (i) the state the timed steps left behind is
    # normalised (whole state, all-reduced over the ranks); (ii) an oracle-sized circuit with every op kind on the
    # rank-held qubits, run on these very ranks through the same schedule path, equals the CPU oracle.
    tolp = 1e-10 if args.dtype == "f64" else 1e-5
    nrm = st.norm2()  # collective on a sharded state: already the whole-state sum, identical on every rank
    pn = 17
    pops = circuits_mod().sharded_parity_circuit(pn, (world - 1).bit_length())
    pst = State(pn, dtype, ctx, rank=rank, world_size=world)
    if world > 1:
        map_peers(pst)
    pst.set_basis(5)
    pst.apply_schedule(pops, fusion=fusion)
    shard = torch.from_numpy(pst.download().view(np.float64 if args.dtype == "f64" else np.float32)).cuda()
    pst.free()
    if world > 1:
        parts = [torch.empty_like(shard) for _ in range(world)]
        dist.all_gather(parts, shard)
        shard = torch.cat(parts)
    perr = None
    if rank == 0:
        from oracle import qip_oracle as qo   # the checker, not the thing measured
        want = qo.run_pipeline(pn, pops, 5, dtype)
        got = shard.cpu().numpy().view(dtype)
        perr = float(np.max(np.abs(got.astype(np.complex128) - want.astype(np.complex128))) / np.max(np.abs(want)))
    line["parity_ok"] = bool(rank != 0 or (perr <= tolp and abs(nrm - 1.0) < (1e-9 if args.dtype == "f64" else 1e-4)))
    line["parity"] = {"norm2_of_timed_state_all_ranks": nrm, "oracle_circuit": "n=%d, %d ops incl. every op kind on the rank-held qubits "
                      "(rustqip_b200.circuits.sharded_parity_circuit), fusion=%s, world=%d" % (pn, len(pops), fusion, world),
                      "max_rel_err_vs_oracle": perr, "tolerance": tolp}

    if not args.no_extras:
        extras = {}
        # (a) unfused schedule: one sweep per gate, as the reference's per-entry loop
        if fusion:
            step(False)
            ms_u = timed(lambda: step(False), 1)
            extras["unfused"] = {"ms_per_step": ms_u, "gate_apps_per_s": gates_total / (ms_u / 1e3),
                                 "effective_state_GBps": gates_total / (ms_u / 1e3) * bytes_alg_gate / 1e9,
                                 "note": "QIPB200_SCHED_NO_FUSION: one in-place kernel sweep per gate, as the reference's per-entry loop"}
        # (b) dominant per-gate kernels, timed alone (CUDA events on the launch stream)
        kern = {}
        g = (world - 1).bit_length()
        probes = {"dense1_H_mid_bit": gates.h(g + (n - g) // 2), "dense1_H_bit0": gates.h(n - 1),
                  "dense1_H_bit5": gates.h(n - 6), "dense1_H_top_local_bit": gates.h(g),
                  "diag_T_mid_bit": gates.t(g + (n - g) // 2), "flip_CNOT": gates.cnot(g + 3, g + (n - g) // 2)}
        for pname, op in probes.items():
            parr, pkeep = marshal_ops([op], st.prec)
            reps = 10
            st.apply_marshalled(parr, 1, False)
            pms = timed(lambda: st.apply_marshalled(parr, 1, False), reps) / reps
            kern[pname] = {"ms": pms, "alg_GBps": local_bytes / (pms / 1e3) / 1e9,
                           "frac_of_peak": local_bytes / (pms / 1e3) / 1e9 / peak}
        extras["kernels_alone"] = kern
        dom = kern["dense1_H_mid_bit"]
        pergate = {"bound": "hbm", "kernel": "k_dense<%s,1,1> (1-qubit dense gate, mid target bit; the unfused per-gate sweep)" % (
                       "double" if args.dtype == "f64" else "float"),
                   "achieved": dom["alg_GBps"], "peak": peak, "unit": "GB/s", "frac": dom["frac_of_peak"],
                   "peak_source": peak_src, "traffic": (ncu_traffic("k_dense", local_bytes) or {}).get("bytes"),
                   "traffic_source": (ncu_traffic("k_dense", local_bytes) or {}).get("source"),
                   "algorithmic_bytes_per_launch": local_bytes, "avg_launch_ms": dom["ms"]}
        if "roofline" in line:
            extras["roofline_per_gate_kernel"] = pergate
        else:
            line["roofline"] = pergate
        # the other single-GPU BASELINE configs, one timed pass each after one warm-up pass
        if world == 1:
            from rustqip_b200 import circuits as _c
            other = {}
            st.free()
            for cname, cn, cdtype, cops in [("configs[1] N=28 f64 depth-40 {H,T,CNOT}", 28, np.complex128, _c.config2()),
                                            ("configs[2] N=30 f32 QFT", 30, np.complex64, _c.qft(30)),
                                            ("configs[3] N=26 f64 200 dense 4-qubit blocks", 26, np.complex128, _c.config4(26, 200))]:
                cst = State(cn, cdtype, ctx)
                carr, ckeep = marshal_ops(cops, cst.prec)
                camp = np.dtype(cdtype).itemsize
                res = {}
                for label, fus in (("fused", True), ("unfused", False)):
                    def cstep():
                        cst.set_basis(0)
                        cst.apply_marshalled(carr, len(cops), fus)
                    cstep()
                    ctx.jit_stats(wait=True)  # generated kernels of this schedule compiled
                    cstep()
                    reps_ms = []
                    for _ in range(3):
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        cst.sync()
                        e0.record(stream)
                        cstep()
                        e1.record(stream)
                        cst.sync()
                        e1.synchronize()
                        reps_ms.append(e0.elapsed_time(e1))
                    cms = float(np.median(reps_ms))
                    res[label] = {"ms": cms, "ms_repeats": reps_ms, "gate_apps_per_s": len(cops) / (cms / 1e3),
                                  "effective_state_GBps": len(cops) / (cms / 1e3) * 2 * camp * (1 << cn) / 1e9}
                res["gates"] = len(cops)
                other[cname] = res
                cst.free()
            extras["other_configs"] = other
            st = State(n, dtype, ctx)  # re-create for the sections below
        line["extras"] = extras

    # end to end through the reference-facing call: LocalBuilder::calculate_state_with_init
    # == qipb200_calculate_state (alloc, |0>, schedule, D2H of all amplitudes into pinned host memory)
    if world == 1:
        st.free()
        host = torch.empty((1 << n) * (2 if True else 1), dtype=torch.float64 if args.dtype == "f64" else torch.float32,
                           pin_memory=True)
        L = _lib.lib()
        flags = _lib.SCHED_DEFAULT if fusion else _lib.SCHED_NO_FUSION

        def e2e_once():
            t0 = time.perf_counter()
            rc = L.qipb200_calculate_state(ctx.handle, st.prec, n, 0, arr, len(ops), flags, C.c_void_p(host.data_ptr()))
            _lib.check(rc, ctx.handle)
            return time.perf_counter() - t0

        e2e_once()
        reps = max(1, min(args.steps, 3))
        dt = sum(e2e_once() for _ in range(reps)) / reps
        line["e2e"] = {"value": gates_total / dt * bytes_alg_gate / 1e9, "unit": UNIT, "gate_apps_per_s": gates_total / dt,
                       "h2d_bytes_per_step": int(sched_bytes),
                       "d2h_bytes_per_step": int(amp << n), "ms_per_step": dt * 1e3,
                       "api": "qipb200_calculate_state (alloc + |0> + schedule + D2H of 2^n amplitudes to pinned host memory), host wall clock"}
        # the downloaded result itself: whole-state norm on the host copy (chunked; it is the D2H'd 16 GiB)
        hn = 0.0
        for lo in range(0, host.numel(), 1 << 28):
            hn += float(torch.sum(host[lo:lo + (1 << 28)].double() ** 2).item())
        line["e2e"]["norm2_of_host_result"] = hn
        line["parity_ok"] = bool(line["parity_ok"] and abs(hn - 1.0) < (1e-9 if args.dtype == "f64" else 1e-4))
    else:
        # sharded: each rank downloads its shard through the same C-ABI calls
        host = torch.empty(st.local_len * 2, dtype=torch.float64 if args.dtype == "f64" else torch.float32, pin_memory=True)

        def e2e_once():
            sync_all()
            t0 = time.perf_counter()
            step()
            st.download_ptr(host.data_ptr(), st.local_len)
            t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())

        e2e_once()
        dt = e2e_once()
        line["e2e"] = {"value": gates_total / dt * bytes_alg_gate / 1e9, "unit": UNIT, "gate_apps_per_s": gates_total / dt,
                       "h2d_bytes_per_step": int(sched_bytes),
                       "d2h_bytes_per_step": int(amp * st.local_len * world), "ms_per_step": dt * 1e3,
                       "api": "state_set_basis + state_apply_schedule + state_download per rank (C ABI), host wall clock, max over ranks"}
        line["exchange_bytes_per_rank_total"] = st.exchange_bytes()
        st.free()

    # CPU baseline beside it (rank 0, N=1 only): bounded sample of the same workload
    if rank == 0 and world == 1 and not args.no_extras:
        try:
            runner = CpuRunner(n, ops, dtype, budget_s=args.cpu_seconds)
            cgps, done, dt = runner.run(args.cpu_seconds)
            line["cpu_baseline"] = {"value": cgps * bytes_alg_gate / 1e9, "unit": UNIT, "gate_apps_per_s": cgps,
                                    "cores": runner.cores, "kind": "port", "sample": runner.describe(done, dt)}
        except Exception as e:  # pragma: no cover
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed: %r" % (e,)}

    if rank == 0:
        print(json.dumps(line), flush=True)
    ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.config5:
        args.gate_set, args.depth, args.seed = "H,CZ,CNOT", 30, 0x5EED0005
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
