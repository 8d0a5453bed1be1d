#!/usr/bin/env python
"""bench.py — candidate assignments / second of the assignment-search hot path on B200.

One "step" = one pass of the hot path over one batch of candidates: ROUNDS search rounds of
ROUND_SIZE candidates each on BASELINE.json's headline topology (config 3: 1000 partitions x 64
brokers x 8 racks, RF 3, synthetic round-robin current assignment).  Every candidate is generated
on-chip from (seed, round, index) and evaluated in full (C1..C7 + objective); each round ends with
an argmin and the winner becomes the next base.

  python bench.py [--gpus N] [--steps K] [--warmup W]            our arm (one JSON line)
  python bench.py --impl reference ...                            the CPU arm: the plain-C restatement
                                                                  of the same path on all host cores
N > 1: launched by torchrun, one rank per GPU; a round of N*ROUND_SIZE candidates is sharded by index
range, the per-round 8-byte minimum travels through NVLink peer mailboxes inside the persistent kernels
(--collective nccl: per-round kernels + one NCCL all-reduce), and every rank applies the same winner.
`e2e` is the same work through the public C-ABI call kao_solve with HOST buffers; at N > 1 rank 0 makes
that one call with kao_options.n_gpus = N (one host thread per GPU inside the library).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# BASELINE.json configs: (P, B, R, RF, brokers removed, fraction re-placed, seed of the re-placement)
CONFIGS = {
    "2": ((256, 32, 4, 3, 0), "config2: 256 partitions x 32 brokers x 4 racks, RF3, round-robin current assignment"),
    "3": ((1000, 64, 8, 3, 0), "config3: 1000 partitions x 64 brokers x 8 racks, RF3, round-robin current assignment"),
    "4": ((1000, 64, 8, 3, 2), "config4: 1000 partitions x 64 brokers x 8 racks, RF3, brokers 62 and 63 removed"),
    "5": ((4096, 256, 16, 3, 0, 0.02, 5), "config5: 4096 partitions x 256 brokers x 16 racks, RF3, 2 % of the replicas re-placed (seed 5)"),
}
ROUNDS, ROUND_SIZE = 32, 1 << 18             # per step and per GPU: 8,388,608 candidates
SEED = 0x5EED
METRIC = "candidate assignments/sec at 1k-partition x 64-broker RF3"
EXACT = {"3": (6962, 38), "4": (6787, 93), "2": (1792, 0), "5": (28401, 141)}      # tests/golden/optima.json (HiGHS): objective, moves


def algo_bytes(P, B):
    """SURVEY.md §8(d): replica bit-plane + leader id + packed result per candidate."""
    return P * ((B + 31) // 32) * 4 + P * (2 if B > 256 else 1) + 8


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region, through NVML (what nvidia-smi reads: its
    own output arrives block-buffered through a pipe, i.e. too late) from a thread of this process every 5 ms
    (start() returns once the first sample is in); only the samples taken between mark_begin() and mark_end()
    count (all of them if there were none)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.samples, self.index, self.thread = [], index, None
        self.t0 = self.t1 = None
        self.running = False
        self.error = None
        self.ready = threading.Event()                       # set after NVML is up and the first sample is in

    def _loop(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.index
            if vis:                                          # NVML counts physical devices
                try:
                    idx = int(vis.split(",")[self.index])
                except (ValueError, IndexError):
                    pass
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            while self.running:
                self.samples.append((time.monotonic(), pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM), mx, int(get_reasons(h))))
                self.ready.set()
                time.sleep(0.005)
        except Exception as e:                               # no NVML: the line says so instead of inventing clocks
            self.error = repr(e)
            self.ready.set()

    def start(self):
        self.running = True
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()
        self.ready.wait(timeout=10.0)                        # nvmlInit can take longer than a whole short bench run

    def mark_begin(self):
        self.t0 = time.monotonic()

    def mark_end(self):
        self.t1 = time.monotonic()

    def stop(self):
        self.running = False
        if self.thread:
            self.thread.join(timeout=2)
        inside = [x for x in self.samples if self.t0 is not None and self.t1 is not None and self.t0 <= x[0] <= self.t1]
        used = inside or self.samples
        sm = sorted(x[1] for x in used)
        reasons = set()
        for x in used:
            for bit, name in self.REASONS.items():
                if x[3] & bit:
                    reasons.add(name)
        out = {"sm_mhz": float(sm[len(sm) // 2]) if sm else None, "sm_max_mhz": float(used[0][2]) if used else None,
               "reasons": sorted(reasons), "samples": len(used), "samples_in_timed_region": len(inside), "source": "NVML, 5 ms period"}
        if self.error:
            out["error"] = self.error
        return out


def host_cpu_info():
    """What the CPU arm could use: affinity, cgroup quota, the CPU model (the CPU arm moved 5.6x between two
    boxes that both reported 128 threads: record enough to tell why)."""
    info = {"nproc": os.cpu_count()}
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
    except AttributeError:
        info["affinity"] = info["nproc"]
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as f:
                info["cgroup_" + os.path.basename(path)] = f.read().strip()
        except OSError:
            pass
    try:
        with open("/proc/cpuinfo") as f:
            for l in f:
                if l.startswith("model name"):
                    info["model"] = l.split(":", 1)[1].strip()
                    break
    except OSError:
        pass
    try:
        info["loadavg_1m"] = os.getloadavg()[0]
    except OSError:
        pass
    return info


def host_threads():
    """All host threads this process may use (torchrun exports OMP_NUM_THREADS=1: not what we want here)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:                                                  # a cgroup quota below the affinity count is the real limit
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
            if quota != "max":
                n = max(1, min(n, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return n


def cpu_port_rate(cfg, seconds_target=10.0):
    """The oracle restatement (plain C + OpenMP, -O3 -march=native, all host cores) on a bounded sample of the
    same workload: whole rounds of the same candidate stream, every candidate evaluated in full, until
    about `seconds_target` seconds of CPU work have been spent."""
    from oracle import model, ref

    pb = model.synthetic_problem(*CONFIGS[cfg][0])
    r = ref.Ref(pb)
    bits, ld = r.init_base()
    threads = host_threads()
    n = ROUND_SIZE - 1
    r.candidate_keys(bits, ld, SEED, 0, ROUND_SIZE, 0, 1 << 14, nthreads=threads)          # warm-up
    total, spent, rnd = 0, 0.0, 0
    while spent < seconds_target and rnd < 64:
        t0 = time.perf_counter()
        r.candidate_keys(bits, ld, SEED, rnd, ROUND_SIZE, 0, n, nthreads=threads)
        spent += time.perf_counter() - t0
        total += n
        rnd += 1
    return total / spent, threads, "%d candidates (%d rounds of the same Philox stream, full evaluation), %.1f s" % (
        total, rnd, spent), r.max_threads(), ref.build_flags()


def exact_solve(cfg, limit_s):
    """The exact 0/1 program of README.md:144-185 solved with HiGHS on the host (the only baseline here that
    resembles the reference's lp_solve call): wall time to the proven optimum, bounded by `limit_s`."""
    from oracle import model

    pb = model.synthetic_problem(*CONFIGS[cfg][0])
    t0 = time.perf_counter()
    sol = model.solve_exact(pb, time_limit=limit_s)
    return {"solver": "HiGHS (scipy.optimize.milp); lp_solve 5.5 is not installed here", "status": sol.status,
            "objective": sol.objective, "moves": sol.moves, "solve_s": round(sol.solve_s, 2), "build_s": round(sol.build_s, 2),
            "wall_s": round(time.perf_counter() - t0, 2), "time_limit_s": limit_s}


def dump_outputs(out_dir, sess, keys, reps, viol, obj, moves):
    """Writes what the last timed step handed its caller as float64 .npy files, so that two builds can be compared
    output for output: the base assignment it left (`replicas`, [P, RF], leader first), that base's
    (violation, objective, moves) (`base_totals`) and, where the path returns them, each round's winning key
    (`round_winners`, [rounds, 3]).  The keys are packed 64-bit words, so they are stored unpacked into
    (violation, objective, candidate index), which float64 holds exactly."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    arrays = {"replicas": reps, "base_totals": [viol, obj, moves]}
    if keys is not None:
        arrays["round_winners"] = [sess.unpack_key(k) for k in keys]
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import model, ref

    pb = model.synthetic_problem(*CONFIGS[args.config][0])
    r = ref.Ref(pb)
    bits, ld = r.init_base()
    threads = host_threads()
    sample = 1 << 20                                        # candidates per step (bounded sample, ~2 s)
    for w in range(args.warmup):
        r.candidate_keys(bits, ld, SEED, w, ROUND_SIZE, 0, 1 << 14, nthreads=threads)
    t0 = time.perf_counter()
    for k in range(args.steps):
        r.candidate_keys(bits, ld, SEED, k, ROUND_SIZE, 0, min(sample, ROUND_SIZE - 1), nthreads=threads)
    dt = time.perf_counter() - t0
    n = args.steps * min(sample, ROUND_SIZE - 1)
    val = n / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "candidates/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32/u32 bitset",
            "data": "synthetic",
            "config": {"workload": CONFIGS[args.config][1], "note": "reference snapshot has no code and lp_solve is not installed: "
                       "this arm is the plain-C restatement of the same generate+evaluate+argmin path"},
            "cpu_baseline": {"value": val, "unit": "candidates/s", "cores": threads, "kind": "port",
                             "sample": "%d candidates per step of the same stream" % min(sample, ROUND_SIZE - 1),
                             "omp_max_threads": r.max_threads(), "build": ref.build_flags(), "host": host_cpu_info()},
            "e2e": {"value": val, "unit": "candidates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=12)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--config", default="3", choices=sorted(CONFIGS), help="BASELINE.json config (3 = the one the metric is quoted on)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the untimed extra keys (other configs, exact solve, time to optimum)")
    ap.add_argument("--probe-schedules", action="store_true", help="time every built variant of the full evaluator and exit")
    ap.add_argument("--device", type=int, default=0, help=argparse.SUPPRESS)
    ap.add_argument("--evaluator", default="auto", choices=["auto", "row", "column"],
                    help="full evaluator of the search kernel: auto = the engine's default (column-major where the layout allows)")
    ap.add_argument("--collective", default="p2p", choices=["p2p", "nccl"],
                    help="N>1: per-round min inside the kernel over NVLink peer memory (p2p) or NCCL all-reduce")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float64; inputs are seeded)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of the GPU path; the reference arm has none to write")
        return reference_arm(args)

    # stdout carries exactly ONE JSON line: whatever libraries print there while the bench runs (NCCL's version
    # banner, for one) goes to stderr instead; the line itself is written to the saved descriptor at the end
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    import numpy as np
    import torch
    import torch.distributed as dist

    import kafka_assignment_optimizer_b200 as kao
    from kafka_assignment_optimizer_b200 import optimizer as kopt, tuning

    cfg_args, workload = CONFIGS[args.config]
    P, B = cfg_args[0], cfg_args[1] - cfg_args[4]
    if args.probe_schedules:
        tuning.probe(kao.synthetic_problem(*cfg_args), args.device, ROUNDS, ROUND_SIZE, SEED,
                     out=lambda l: os.write(json_fd, (l + "\n").encode()))
        return 0

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node %d for --gpus %d" % (args.gpus, args.gpus))
    torch.cuda.set_device(local)
    if world > 1:
        # stdout carries exactly one JSON line: NCCL's own banner / debug output (NCCL_DEBUG) goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        # host-side barriers (gloo): while rank 0 drives ALL GPUs through one kao_solve call (e2e), the other ranks
        # must leave their GPUs idle — an NCCL barrier is a kernel that spins on the GPU, and a cooperative launch
        # of another process on that GPU then has to wait for a time slice (measured: 50 ms instead of 12 ms per solve)
        try:
            host_group = dist.new_group(backend="gloo")
        except Exception as e:                                    # no usable interface for gloo: fall back to NCCL barriers
            print("bench: gloo group unavailable (%s); e2e at N > 1 will see time-slicing" % e, file=sys.stderr)
            host_group = None
    dev = torch.device("cuda", local)

    pb = kao.synthetic_problem(*cfg_args)
    sess = kao.Session(pb, device=local)
    if args.evaluator != "auto" and not sess.set_evaluator(args.evaluator == "column"):
        raise SystemExit("the column-major evaluator does not cover this layout")
    if world > 1 and args.collective == "nccl":
        sess.set_evaluator(False)                            # the NCCL variant runs the per-round kernels (row-major evaluator)
    use_col = sess.stats()["column_major"]
    gsize = ROUND_SIZE * world                               # weak scaling: per-GPU work fixed
    key = torch.full((1,), kopt.KEY_NONE, dtype=torch.int64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2
    stream = torch.cuda.current_stream().cuda_stream

    from kafka_assignment_optimizer_b200 import distributed as kd

    launch_cb, apply_cb = kd.session_callbacks(sess, key, SEED, gsize, stream)
    reduce_cb = (lambda k: dist.all_reduce(k, op=dist.ReduceOp.MIN)) if world > 1 else None

    if world > 1 and args.collective == "p2p":
        sess.p2p_setup_torch(dev)

    def step(k, size=gsize, rounds=ROUNDS):
        """`rounds` rounds; inputs (tables + base) are already resident in HBM."""
        if world == 1:
            return sess.search(SEED, k * rounds, rounds, size)
        if args.collective == "p2p":   # one persistent kernel per rank, keys traded over NVLink peer memory
            return sess.search_sharded(SEED, k * rounds, rounds, size)
        # per-round kernels + one 8-byte NCCL min all-reduce of the packed key per round
        kd.run_rounds(launch_cb, apply_cb, key, k * rounds, rounds, size, rank, world, reduce_cb)
        return None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def host_barrier():
        torch.cuda.synchronize()
        if world > 1:
            if host_group is not None:
                dist.barrier(group=host_group)
            else:
                dist.barrier()

    # N > 1, untimed: the sharded search walks the single-GPU trajectory (VERDICT r1 #5: the 2-GPU pytest is
    # skipped on a 1-GPU box, so the proof travels with the scaling run)
    sharded_equals_single = None
    if world > 1 and args.collective == "p2p":
        chk_rounds, chk_size = 6, 1 << 14
        got, _ = sess.search_sharded(SEED + 1, 0, chk_rounds, chk_size)
        base_sharded = sess.get_base()[0]
        ok = True
        if rank == 0:
            solo = kao.Session(pb, device=local)
            want, _ = solo.search(SEED + 1, 0, chk_rounds, chk_size)
            ok = bool((want == got).all() and (solo.get_base()[0] == base_sharded).all())
            solo.close()
        flag = torch.tensor([1 if ok else 0], device=dev)
        bases = [torch.empty(base_sharded.size, dtype=torch.int32, device=dev) for _ in range(world)]
        dist.all_gather(bases, torch.from_numpy(np.ascontiguousarray(base_sharded).reshape(-1)).to(dev))
        same_everywhere = all(bool((b == bases[0]).all()) for b in bases)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        sharded_equals_single = bool(flag.item()) and same_everywhere
        sess.reset()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                                      # up and sampling by the time the warm-up is through
    for w in range(args.warmup):
        step(w)
    barrier()
    launches0 = sess.stats()["kernel_launches"]
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    sampler.mark_begin()
    for k in range(args.steps):
        flush.fill_(k & 0xFF)                                # L2 flush between timed steps (outside the events)
        ev[k][0].record()
        last = step(args.warmup + k)
        ev[k][1].record()
    barrier()
    sampler.mark_end()
    clocks = sampler.stop() if rank == 0 else None
    ms = sum(a.elapsed_time(b) for a, b in ev)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    launches = sess.stats()["kernel_launches"] - launches0
    n_total = args.steps * ROUNDS * gsize
    value = n_total / (ms * 1e-3)
    reps, viol, obj, moves = sess.get_base()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, sess, None if last is None else last[0], reps, viol, obj, moves)

    # N > 1, untimed: the exchange cost at the small rounds a search for quality uses (32,768 candidates per
    # GPU and round), device-timed, max over ranks
    small_rounds = None
    if world > 1 and args.collective == "p2p" and not args.no_extras:
        sm_size, sm_rounds = (1 << 15) * world, 256
        step(900, sm_size, sm_rounds)
        barrier()
        _, sm_ms = step(901, sm_size, sm_rounds)
        tt = torch.tensor([sm_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        small_rounds = {"round_size_per_gpu": 1 << 15, "rounds": sm_rounds, "ms": float(tt.item()),
                        "value": sm_rounds * sm_size / (float(tt.item()) * 1e-3), "unit": "candidates/s"}

    # N > 1, untimed, p2p: BASELINE configs 4 and 5 sharded over the ranks (configs[3], configs[4])
    other = {}
    if world > 1 and args.collective == "p2p" and not args.no_extras and args.config == "3":
        for c in ("4", "5"):
            pbc = kao.synthetic_problem(*CONFIGS[c][0])
            sc = kao.Session(pbc, device=local)
            sc.p2p_setup_torch(dev)
            rs = (ROUND_SIZE if c == "4" else 1 << 14) * world
            rn = 32 if c == "4" else 16
            sc.search_sharded(SEED, 0, 2, rs)
            barrier()
            _, c_ms = sc.search_sharded(SEED, 100, rn, rs)
            tt = torch.tensor([c_ms], dtype=torch.float64, device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            st = sc.stats()
            other["config" + c] = {"workload": CONFIGS[c][1], "rounds": rn, "round_size": rs, "ms": float(tt.item()),
                                   "value": rn * rs / (float(tt.item()) * 1e-3), "unit": "candidates/s",
                                   "evaluator": "column-major" if st["column_major"] else "row-major",
                                   "algorithmic_bytes_per_candidate": algo_bytes(pbc.P, pbc.B),
                                   "roofline_frac_per_gpu": rn * rs / world / (float(tt.item()) * 1e-3) * algo_bytes(pbc.P, pbc.B) / 1e9 / measured_peak()[0]}
            sc.close()
            barrier()

    # end to end through the public C-ABI call with HOST buffers (tables up, winner down, every step).  At
    # N > 1 rank 0 makes ONE kao_solve call with n_gpus = N; the other ranks wait at the barrier.
    e2e = None
    barrier()
    host_barrier()                                                # every GPU idle from here until rank 0 is through
    if rank == 0:
        import dataclasses

        e2e_steps = max(3, min(args.steps, 6))
        pinned = {f.name: torch.from_numpy(np.ascontiguousarray(getattr(pb, f.name))).pin_memory()
                  for f in dataclasses.fields(pb) if isinstance(getattr(pb, f.name), np.ndarray)}
        pb_host = dataclasses.replace(pb, **{k: v.numpy() for k, v in pinned.items()})
        row = args.evaluator == "row"
        kopt.solve(pb_host, SEED, 2, 1 << 12, 0, n_gpus=world, row_major=row)        # warm the contexts / modules
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k in range(e2e_steps):
            res = kopt.solve(pb_host, SEED + k, ROUNDS, gsize, 0, n_gpus=world, row_major=row)
        e2e_s = time.perf_counter() - t0
        h2d = (pb.rack_of.nbytes + pb.wF.nbytes + pb.wL.nbytes + 4 * 4 * pb.B + 2 * 4 * pb.R + pb.cur.nbytes) * world
        d2h = pb.P * pb.RF * 4 + ROUNDS * 8 + 16
        e2e = {"value": e2e_steps * ROUNDS * gsize / e2e_s, "unit": "candidates/s",
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "api": "kao_solve(n_gpus=%d): pinned host buffers; create + upload + %d rounds x %d candidates + download + destroy per step" % (
                   world, ROUNDS, gsize),
               "n_gpus": int(res.n_gpus),
               "last_result": {"violation": int(res.violation), "objective": int(res.objective), "moves": int(res.moves),
                               "objective_bound": int(res.objective_bound), "proven_optimal": bool(res.optimal)}}
        if not args.no_extras and args.config in EXACT:
            def time_to_solution():
                # the call a user makes to SOLVE: small rounds, early stop; must end feasible at the exact optimum
                kw = dict(rounds=2000, round_size=1 << 14, patience=100, n_gpus=1)
                if args.config == "4":                          # local optima of the 3-row neighbourhood: many short searches
                    kw = dict(rounds=400, round_size=1 << 12, patience=150, restarts=12, n_gpus=1)
                if args.config == "5":
                    kw.update(delta=True, rounds=20000, round_size=1 << 15, patience=3000)
                r2 = kopt.solve(pb_host, SEED, device=0, **kw)
                r3 = kopt.solve(pb_host, SEED, device=0, tight_bound=True, **kw)   # + the flow bound (host): optimality certificate
                return {
                    "ms": r2.total_ms, "device_ms": r2.device_ms, "rounds_run": int(r2.rounds), "candidates": int(r2.n_candidates),
                    "violation": int(r2.violation), "objective": int(r2.objective), "moves": int(r2.moves),
                    "exact_objective": EXACT[args.config][0], "exact_moves": EXACT[args.config][1],
                    "reached_exact_optimum": bool(r2.violation == 0 and r2.objective == EXACT[args.config][0]),
                    "with_flow_bound": {"ms": r3.total_ms, "objective": int(r3.objective), "objective_bound": int(r3.objective_bound),
                                        "proven_optimal": bool(r3.optimal)},
                    "call": "kao_solve(%s), 1 GPU, host buffers" % ", ".join("%s=%s" % kv for kv in sorted(kw.items()))}

            try:                                                  # an extra key must never cost the line itself
                e2e["time_to_solution"] = time_to_solution()
            except Exception as e:
                e2e["time_to_solution"] = {"error": repr(e)}
    host_barrier()
    barrier()

    line = None
    if rank == 0:
        # dominant kernel = the persistent multi-round search kernel (one cooperative launch per step):
        # timed alone with CUDA events on the launching stream (kao_search brackets it)
        prof_steps = 4
        solo = sess if world == 1 else kao.Session(pb, device=local)
        if world > 1 and args.evaluator != "auto":
            solo.set_evaluator(args.evaluator == "column")
        s_ms = sum(solo.search(SEED, 10_000 + i * ROUNDS, ROUNDS, ROUND_SIZE)[1] for i in range(prof_steps)) / prof_steps
        col_solo = solo.stats()["column_major"]
        peak, peak_src = measured_peak()
        ab = algo_bytes(P, B)
        achieved = ab * ROUND_SIZE * ROUNDS / (s_ms * 1e-3) / 1e9
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                traffic = json.load(f).get("search_persistent_kernel_column_major_dram_bytes_per_launch" if col_solo
                                           else "search_persistent_kernel_dram_bytes_per_launch")
        except Exception:
            pass
        sched = solo.stats()["schedule"]
        roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": traffic,
                    "kernel": ("search_persistent_kernel<EvalCfgT<W=%d,sync=%d,pop=%05x,threads=%d>> (column-major evaluator)"
                               % ((solo.stats()["words_per_row"],) + tuple(sched)) if col_solo else
                               "search_persistent_kernel<EvalCfg<W=%d,NPH=5,...>> (row-major evaluator)" % solo.stats()["words_per_row"]),
                    "algorithmic_bytes_per_candidate": ab, "candidates_per_launch": ROUND_SIZE * ROUNDS,
                    "kernel_ms_per_launch": s_ms,
                    "peak_source": peak_src,
                    "note": "candidates are generated and consumed on-chip (shared memory): the measured DRAM traffic "
                            "(`traffic`, ncu dram__bytes_read+write per launch) is far below the algorithmic bytes by "
                            "design; the physical bounds are the ALU / XU pipes (profiles/)"}
        extras = {}
        if not args.no_extras:
            def collect_extras():
                solo.profile_rounds(SEED, 19_000, 1, ROUND_SIZE)                      # load the per-round kernels (lazy module load)
                pr_ms, ap_ms = solo.profile_rounds(SEED, 20_000, 8, ROUND_SIZE)       # per-round kernels (NCCL path)
                roofline["per_round_kernels_ms"] = {"search_round_kernel": pr_ms / 8, "apply_winner_kernel": ap_ms / 8}
                # SURVEY 8(f)3, reported separately: the same search with delta evaluation (NOT the headline metric)
                if solo.stats()["words_per_row"] <= 2:
                    solo.search_delta(SEED, 30_000, ROUNDS, ROUND_SIZE)
                    _, d_ms = solo.search_delta(SEED, 31_000, ROUNDS, ROUND_SIZE)
                    extras["delta_evaluation"] = {
                        "value": ROUNDS * ROUND_SIZE / (d_ms * 1e-3), "unit": "candidates/s", "kernel_ms_per_launch": d_ms,
                        "note": "same candidate stream and keys, scored from base totals + patched rows (one thread per "
                                "candidate); not a full evaluation per candidate, so not comparable with `value`"}
                # the other single-GPU BASELINE configs as extra keys (device-timed, same kernel family)
                if world == 1 and args.config == "3":
                    for c, rs, rn in (("2", 1 << 16, 32), ("4", ROUND_SIZE, 32), ("5", 1 << 14, 16)):
                        pbc = kao.synthetic_problem(*CONFIGS[c][0])
                        sc = kao.Session(pbc, device=local)
                        sc.search(SEED, 0, 2, rs)
                        _, c_ms = sc.search(SEED, 100, rn, rs)
                        st = sc.stats()
                        cab = algo_bytes(pbc.P, pbc.B)
                        extras.setdefault("other_configs", {})["config" + c] = {
                            "workload": CONFIGS[c][1], "rounds": rn, "round_size": rs, "kernel_ms": c_ms,
                            "value": rn * rs / (c_ms * 1e-3), "unit": "candidates/s",
                            "evaluator": "column-major" if st["column_major"] else "row-major",
                            "algorithmic_bytes_per_candidate": cab,
                            "roofline_frac": rn * rs / (c_ms * 1e-3) * cab / 1e9 / peak}
                        sc.close()

            try:                                                  # extra keys must never cost the line itself
                collect_extras()
            except Exception as e:
                extras["extras_error"] = repr(e)
        if solo is not sess:
            solo.close()
        cpu = None
        if not args.no_cpu_baseline and world == 1:         # reported at N=1 only
            try:
                v, threads, sample, omp, port_build = cpu_port_rate(args.config)
                cpu = {"value": v, "unit": "candidates/s", "cores": threads, "kind": "port", "sample": sample,
                       "omp_max_threads": omp, "build": port_build, "host": host_cpu_info(),
                       "note": "lp_solve (the reference's solver) is not installed here and cannot be timed; "
                               "this is the plain-C/OpenMP restatement of the same path"}
                if not args.no_extras and args.config in ("2", "3", "4"):
                    cpu["exact_solve"] = exact_solve(args.config, 150.0)
            except Exception as e:
                cpu = dict(cpu or {}, error=repr(e))
        line = {"metric": METRIC, "value": value, "unit": "candidates/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "u32 bitset / int32",
                "data": "synthetic",
                "config": {"workload": workload, "rounds_per_step": ROUNDS, "round_size_per_gpu": ROUND_SIZE,
                           "candidates_per_step": ROUNDS * gsize, "seed": SEED,
                           "evaluator": ("column-major" if use_col else "row-major") + (" (engine default)" if args.evaluator == "auto" else " (forced)"),
                           "l2": "flushed between timed steps (256 MiB write); working set is shared-memory resident",
                           "parallelism": ("single GPU" if world == 1 else
                                           "index-range sharding over %d ranks; per-round 8-byte min %s" % (
                                               world, "inside the persistent kernel over NVLink peer mailboxes"
                                               if args.collective == "p2p" else "by NCCL all-reduce"))},
                "search_state": {"violation": int(viol), "objective": int(obj), "moves": int(moves),
                                 "exact_optimum": {"objective": EXACT[args.config][0], "moves": EXACT[args.config][1],
                                                   "source": "tests/golden/optima.json (HiGHS)"},
                                 "sharded_equals_single": sharded_equals_single},
                "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches),
                "clocks": clocks}
        line.update(extras)
        if small_rounds:
            line["small_rounds"] = small_rounds
        if other:
            line["other_configs"] = other
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    sess.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
