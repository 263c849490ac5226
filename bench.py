#!/usr/bin/env python
"""bench.py — simulated node·rounds/sec of the SWIM per-round hot path on B200.

  python bench.py --gpus N --steps K --warmup W          # CUDA path (this repo)
  python bench.py --impl reference --steps K --warmup W  # CPU arm: the restated oracle, all host threads

A "step" is ONE protocol round over all N simulated nodes of BASELINE config C3
(N = 1,048,576, D = 32 uniform-random views, k = 3, piggyback fan-out 4, B = 8, S = 5,
0.1 % of the nodes crash at round 10). For --gpus G > 1 the node set is sharded G ways
(weak scaling: 1,048,576 nodes per GPU, config C4 at G = 4) with one all-to-all of cross-shard
piggyback envelopes per round.

Prints ONE JSON line (rank 0). `value` = node·rounds/s with state resident in HBM, timed with
CUDA events on the stream the kernels run on, max over ranks. `e2e` = the same metric through
the C ABI one round per call with host buffers: every step uploads that round's event trace,
runs one round and reads the counters and the convergence count back
(swim_sim_inject + swim_sim_step_async(1) + swim_sim_observe, one synchronisation per round).

`--dump-outputs DIR` writes, after the timed windows, what the last of them left on the handle (write_outputs) as
DIR/<name>.npy: the inputs depend on the arguments alone, so two builds run with the same arguments can be compared
file by file (and the CUDA arm with `--impl reference`).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from swim_b200 import _abi as A  # noqa: E402

def usable_cpus():
    """CPUs this process may actually use (affinity mask and cgroup quota), for the CPU arm."""
    n = len(os.sched_getaffinity(0))
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(int(q) / int(per))))
    except (OSError, ValueError):
        pass
    return n


# host-side OpenMP code (the library's in-edge index build, the oracle): torchrun exports OMP_NUM_THREADS=1 to its workers,
# which would make every rank build its index serially; give each local rank its share of the host cores instead
_local_world = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))
if _local_world > 1:
    os.environ["OMP_NUM_THREADS"] = str(max(1, usable_cpus() // _local_world))
else:
    os.environ.setdefault("OMP_NUM_THREADS", str(usable_cpus()))

# (two seams for tests/test_bench_dryrun.py, which runs this file's CUDA arm on the emulator, several ranks as threads of one
# process: where the launcher's environment is read, and where the tensors of the host-side reductions live)
_ENV = os.environ
_TENSOR_DEVICE = "cuda"

N_PER_GPU = 1 << 20
CRASH_ROUND = 10
CRASH_PPM = 1000  # 0.1 %
SEED = 0x5EED0001 + 3


def workload(n_gpus, nodes_per_gpu=N_PER_GPU):
    from swim_b200.sim import crash_events, default_config, generate_topology
    n = nodes_per_gpu * n_gpus
    cfg_kw = dict(n_nodes=n, view_cap=32, k_indirect=3, fanout=4, pb_cap=8, suspicion_rounds=5, retransmit=8,
                  loss_ppm=0, seed=SEED)
    nbr = generate_topology("random", n, 32, 32, seed=3)
    rng = np.random.default_rng(3)
    crashed = np.sort(rng.choice(n, size=n * CRASH_PPM // 1000000, replace=False)).astype(np.uint32)
    return cfg_kw, nbr, crash_events(CRASH_ROUND, crashed), n


def algorithmic_bytes(cfg_kw, n_nodes, rounds, ctr_delta):
    """SURVEY.md §8(d): AB = 7·D + 16·B + 4·F + 8 + 2·(8 + 8·b̄)·m̄ bytes per node·round, canonical
    widths (state 1 B, incarnation 4 B, timer 2 B, record 8 B). Returns (AB per node·round, tick share)."""
    D, B, F = 32, cfg_kw["pb_cap"], cfg_kw["fanout"]
    msgs = float(ctr_delta[A.CTR_MSGS])
    recs = float(ctr_delta[A.CTR_RECS_SENT])
    m_bar = msgs / (n_nodes * rounds)
    b_bar = recs / msgs if msgs else 0.0
    floor = 7 * D + 16 * B + 4 * F + 8
    msg_side = (8 + 8 * b_bar) * m_bar  # written once (tick) and read once (receive)
    return floor + 2 * msg_side, floor + msg_side, m_bar, b_bar


DUMP_NODES = 32768  # rows written by --dump-outputs: a fixed sample of node ids (C3's full state is 0.5 GB per GPU)
DUMP_SEED = 0xD0
DUMP_MAX_BYTES = 64 << 20


def write_outputs(h, out_dir, n_nodes, rank=0, world=1):
    """What a caller of the timed path reads back after its last step, as float64 arrays in out_dir/<name>.npy:
    counters (A.CTR_NAMES order, summed over ranks), mismatches (the convergence count), digest (the 64-bit state digest
    as [high, low] 32-bit halves), and every state array of A.ARRAY_NAMES — the piggyback records field by field as
    pb_<field> — at the rows of sample_nodes, DUMP_NODES node ids drawn with a fixed seed. `h` is a Simulator or an
    Oracle. With world > 1 every rank must call this (it gathers) and rank 0 writes."""
    nodes = np.sort(np.random.default_rng(DUMP_SEED).choice(n_nodes, size=min(n_nodes, DUMP_NODES), replace=False))
    own = nodes[(nodes >= h.first) & (nodes < h.first + h.n_local)]
    part = {}
    for a in range(A.ARR_COUNT):
        full = a in A.REPLICATED_ARRAYS  # [N] on every rank; the other arrays hold this rank's rows only
        x = h.get_array(a).reshape(n_nodes if full else h.n_local, -1)[own if full else own - h.first]
        if a == A.ARR_PB:
            for f in ("member", "incarnation", "from", "kind", "ttl"):
                part["pb_" + f] = x[f]
        else:
            part[A.ARRAY_NAMES[a]] = x if x.shape[1] > 1 else x[:, 0]
    if world > 1:
        import torch.distributed as dist
        from swim_b200 import dist as sdist
        parts = [None] * world
        dist.all_gather_object(parts, part)
        part = {k: np.concatenate([p[k] for p in parts]) for k in part}  # ranks own ascending node ranges
        ctr, mm, dg = sdist.global_sum(h.counters()), sdist.global_sum([h.mismatches()]), sdist.global_digest(h.digest())
        if rank != 0:
            return
    else:
        ctr, mm, dg = h.counters(), [h.mismatches()], h.digest()
    out = dict(part, sample_nodes=nodes, counters=ctr, mismatches=mm, digest=[dg >> 32, dg & 0xFFFFFFFF])
    out = {k: np.asarray(v).astype(np.float64) for k, v in out.items()}
    total = sum(v.nbytes for v in out.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes (limit {DUMP_MAX_BYTES})")
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def timed_kernel_name(steps, world):
    """Which fused kernel runs the timed rounds: round_kernel_x (one grid barrier per round) for launches of >= 32 rounds on
    a single shard, the two-phase round_kernel otherwise (swim_sim.cu: kXModeMinRounds); SWIM_XMODE=1 / 0 forces one."""
    x = os.environ.get("SWIM_XMODE")
    if x is not None:
        return "round_kernel_x<1>" if x != "0" else "round_kernel<1>"
    longest = steps - max(0, CRASH_ROUND - 1 - 5)  # the launch behind the crash events (warm-up 5: rounds 6..9 come first)
    return "round_kernel_x<1>" if world == 1 and longest >= 32 else "round_kernel<1>"


def summarize_timeline(tl, warmup):
    """tl: [rounds, 8] ns stamps of round_kernel's phase boundaries (CTA 0; swim_sim_get_timeline). Per-phase means over
    the rounds that ran the phase; a round committed by a batched quiet scan shares its batch's stamps."""
    scan, work, recv, busy_total, quiet_total, bar3 = [], [], [], [], [], []
    last_scan, last_work, rel1, rel2 = [], [], [], []  # slowest CTA's phase time; release latency of the two barriers
    x_own, x_last = [], []  # one-barrier rounds: CTA 0's / the slowest CTA's interval
    own = {"scan": [], "work": [], "recv": []}  # CTA 0's own share of a phase (the rest is waiting at the barrier)
    n_busy = n_quiet = 0
    r = 0
    R = len(tl)
    while r < R:
        t = tl[r]
        if t[0] == 0:
            r += 1
            continue
        if t[4] == 0:  # ended after the first barrier: a quiescent round, or a committed batch of them
            span = int(t[7]) if t[7] > 0 else 1
            quiet_total.append((t[2] - t[0]) / span)
            n_quiet += span
            r += span
            continue
        n_busy += 1
        if t[3] == 0 and t[4] == 1:  # round_kernel_x: ONE interval and one barrier per round (slot 4 holds the busy flag)
            busy_total.append(t[2] - t[0]); x_own.append(t[1] - t[0])
            if t[5]:
                x_last.append(t[5] - t[0]); rel1.append(t[2] - t[5])
            r += 1
            continue
        scan.append(t[2] - t[0]); own["scan"].append(t[1] - t[0])
        work.append(t[4] - t[2]); own["work"].append(t[3] - t[2])
        busy_total.append(t[4] - t[0])  # (the receive pass of a round runs inside the next round's scan phase)
        if t[5] and t[6]:
            last_scan.append(t[5] - t[0]); rel1.append(t[2] - t[5])
            last_work.append(t[6] - t[2]); rel2.append(t[4] - t[6])
        r += 1
    f = lambda v: float(np.mean(v)) / 1e3 if len(v) else None
    return {"busy_rounds": n_busy, "quiet_rounds": n_quiet, "busy_us": f(busy_total), "quiet_us": f(quiet_total),
            "scan_us": f(scan), "work_us": f(work), "recv_us": f(recv), "recv_rounds": len(recv),
            "cta0_scan_us": f(own["scan"]), "cta0_work_us": f(own["work"]), "cta0_recv_us": f(own["recv"]),
            "busy_us_max": float(np.max(busy_total)) / 1e3 if busy_total else None,
            "barriers_per_busy_round": 1 if x_own else 2,
            "cta0_interval_us": f(x_own), "slowest_cta_interval_us": f(x_last),
            "slowest_cta_scan_us": f(last_scan), "slowest_cta_work_us": f(last_work),
            "barrier1_release_us": f(rel1), "barrier2_release_us": f(rel2),
            "what": "in-kernel %globaltimer stamps of CTA 0 at round_kernel's phase boundaries over the timed rounds; a phase "
                    "runs from one grid barrier to the next: scan (+ the receive pass of the round before, on otherwise idle "
                    "warps) | work = K1b; cta0_* is CTA 0's own part of it, slowest_cta_* the arrival of the LAST CTA at the phase's "
                    "barrier, barrierN_release_us what the barrier itself adds after that. round_kernel_x (default) has ONE "
                    "interval per round — mail of the round before + K1b + the next round's scan — and one barrier: "
                    "busy_us / cta0_interval_us / slowest_cta_interval_us / barrier1_release_us describe it, the scan_ / "
                    "work_ keys stay empty"}


def make_roofline(cfg_kw, n_local, ms_per_round, ab_round, m_bar, b_bar, peak, measured_peak, prof, rounds_p, timeline,
                  ctr_delta, steps, world):
    """SURVEY 8(d) as written: the kernel in the timed path (round_kernel<W>: scan, tick work and receive of every round
    of a launch), achieved = canonical algorithmic bytes per round / its CUDA-event time per round."""
    achieved = ab_round * n_local / (ms_per_round * 1e-3) / 1e9
    traffic = dram_gbs = None
    tp = os.path.join(ROOT, "profiles", "round_traffic.json")
    if os.path.exists(tp):
        t = json.load(open(tp))
        traffic = t.get("dram_bytes_per_round")
    if traffic:
        dram_gbs = traffic / (ms_per_round * 1e-3) / 1e9
    # what the implementation has to move per round: one 16-byte record per node (scan) + the rows it opens
    msgs = float(ctr_delta[A.CTR_MSGS]) / steps / max(1, world)
    impl = 16.0 * n_local + 1024.0 * msgs + 900.0 * msgs / max(1.0, cfg_kw["fanout"] * 0.97)
    calib = None
    cp = os.path.join(ROOT, "profiles", "calibration.json")
    if os.path.exists(cp):
        calib = json.load(open(cp))
    floor = None
    if calib and timeline and timeline.get("busy_rounds"):
        # a busy round: 2 grid barriers + the dependent-load chains, each warp walking its items one after the other
        nwarps = calib.get("resident_warps", 4736)
        items_w = max(1.0, msgs / max(1.0, cfg_kw["fanout"] * 0.97) / nwarps)
        items_r = max(1.0, msgs / nwarps)
        hop = calib["hbm_load_ns"] / 1e3
        n_bar = timeline.get("barriers_per_busy_round", 2)
        floor_busy = n_bar * calib["grid_barrier_ns"] / 1e3 + hop * (1 + 2 * items_w)
        floor = {"busy_round_us": floor_busy, "measured_busy_round_us": timeline["busy_us"],
                 "frac_of_floor": floor_busy / timeline["busy_us"] if timeline["busy_us"] else None,
                 "grid_barrier_us": calib["grid_barrier_ns"] / 1e3, "hbm_dependent_load_us": hop,
                 "l2_dependent_load_us": calib.get("l2_load_ns", 0) / 1e3,
                 "barriers_per_busy_round": n_bar,
                 "model": "grid barriers of a busy round (1 with round_kernel_x, 2 with the two-phase round_kernel) + "
                          "dependent-load hops (1 for the scan's records, 2 per K1b item: list entry -> row -> recipients' "
                          "filters) x K1b items per warp, mean items of the timed rounds; the receive pass overlaps"}
    return {"bound": "hbm", "kernel": ("round_kernel_x<1>" if timeline.get("barriers_per_busy_round") == 1 else "round_kernel<1>")
                      if timeline and timeline.get("busy_rounds") else timed_kernel_name(steps, world), "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak,
            "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if measured_peak else "6650 GB/s (of fallback)",
            "traffic": traffic, "dram_gbs": dram_gbs, "dram_frac": dram_gbs / peak if dram_gbs else None,
            "algorithmic_bytes_per_round": ab_round * n_local,
            "ab_per_node_round": {"round": ab_round, "m_bar": m_bar, "b_bar": b_bar},
            "impl_bytes_per_round_model": impl,
            "latency_floor": floor, "timeline": timeline,
            "split_kernels_us": {"tick_scan": prof["tick_scan"] / rounds_p * 1e3, "tick_work": prof["tick_work"] / rounds_p * 1e3,
                                 "recv": prof["recv"] / rounds_p * 1e3, "exchange": prof["exchange"] / rounds_p * 1e3,
                                 "events_total": prof["events"] * 1e3},
            "note": "achieved = SURVEY 8(d)'s canonical bytes per round (376 B/node quiescent floor + message terms) / the "
                    "CUDA-event time per round of the kernel in the timed path. The implementation moves far fewer bytes (a "
                    "16-byte derived record per node in the scan, full rows only for nodes with work): `traffic` (ncu dram "
                    "bytes per round) and dram_frac say how much of HBM it really uses; at C3's size the round is bound by "
                    "grid barriers and dependent-load chains (latency_floor), not by bandwidth — the HBM-regime point is "
                    "profiles/r02_hbm_regime.md"}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for nm, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.f.name)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons),
                       samples=len(sm))
        return out


def cpu_arm(cfg_kw, nbr, events, n_nodes, steps, warmup):
    """The CPU arm: the restated oracle (oracle/swim_oracle.c, OpenMP over nodes) on the same config, with all the
    host threads this process may use (torchrun exports OMP_NUM_THREADS=1 to its workers: override it before the
    default through omp_set_num_threads; SWIM_CPU_THREADS pins a number)."""
    from oracle.oracle import Oracle, num_threads, set_num_threads
    set_num_threads(int(os.environ.get("SWIM_CPU_THREADS", usable_cpus())))
    from swim_b200.sim import default_config
    orc = Oracle(default_config(**cfg_kw))
    orc.set_view(nbr)
    orc.inject(events)
    orc.step(warmup)
    t0 = time.perf_counter()
    orc.step(steps)
    dt = time.perf_counter() - t0
    return n_nodes * steps / dt, dt, num_threads(), orc


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    cfg_kw, nbr, events, n = workload(args.gpus, args.nodes_per_gpu)  # the same N as the CUDA arm at --gpus G (one shard: all on the host)
    val, dt, threads, orc = cpu_arm(cfg_kw, nbr, events, n, args.steps, args.warmup)
    if args.dump_outputs:
        write_outputs(orc, args.dump_outputs, n)
    line = {
        "impl": "reference", "metric": "simulated node-rounds/sec", "value": val, "unit": "node-rounds/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3 / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/u32", "data": "synthetic",
        "config": config_dict(cfg_kw, n, args.gpus),
        "cpu_baseline": {"value": val, "unit": "node-rounds/s", "cores": threads, "kind": "port",
                         "sample": f"all {n} nodes of C3 x{args.gpus}, rounds {args.warmup + 1}..{args.warmup + args.steps} "
                                   "(restated C oracle, OpenMP; the Haskell reference cannot be built here)"},
        "e2e": {"value": val, "unit": "node-rounds/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    return line


def config_dict(cfg_kw, n, n_gpus, exchange_mode="single"):
    return {"workload": f"C3 x{n_gpus}: N={n} simulated nodes ({n // n_gpus}/GPU), D=32 uniform-random views, k=3, "
                        f"fanout=4, B=8, S=5, T=8, {CRASH_PPM / 1e4:.1f}% crash at round {CRASH_ROUND}; step = 1 round",
            "n_nodes": n, "view_degree": 32, "k_indirect": 3, "fanout": 4, "pb_cap": 8, "suspicion_rounds": 5,
            "retransmit": 8, "crash_round": CRASH_ROUND, "seed": SEED,
            "parallelism": f"shard{n_gpus}" if n_gpus > 1 else "single", "exchange": exchange_mode,
            # rounds decided per batched quiet scan of round_kernel (single shard; 0 = off), DESIGN.md section 5
            "quiet_batch": (min(8, max(0, int(os.environ.get("SWIM_QUIET_BATCH", "4")))) if n_gpus == 1 else 0),
            "launch_switches": {k: os.environ[k] for k in ("SWIM_PIPELINE", "SWIM_SPLIT", "SWIM_ROUND_KERNEL", "SWIM_XMODE",
                                                            "SWIM_ONE_ROUND_PER_LAUNCH", "SWIM_WPB", "SWIM_QUIET_BATCH") if k in os.environ},
            "l2": "no flush between rounds: consecutive rounds of one simulation share state by definition; "
                  "state arrays total 0.5 GB/GPU (> 126 MB L2), the per-round hot set (packed state rows 32 MB "
                  "+ flags) is L2-resident by design"}


def run_cuda(args):
    import torch
    import torch.distributed as dist

    rank = int(_ENV.get("RANK", "0"))
    world = int(_ENV.get("WORLD_SIZE", "1"))
    local = int(_ENV.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node N for --gpus N")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the swim_b200 compute path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from swim_b200 import dist as sdist
    from swim_b200.sim import Simulator, default_config
    cfg_kw, nbr, events, n = workload(world, args.nodes_per_gpu)

    exchange = {"mode": "single"}

    def fresh(inject=True, flags=0):
        sim = Simulator(default_config(rank=rank, world=world, device=local, flags=flags, **cfg_kw))
        sim.set_view(nbr)
        exchange["mode"] = sdist.connect(sim, args.exchange)
        if inject:
            sim.inject(events)
        return sim

    def barrier():
        # Drain this rank's streams BEFORE the NCCL barrier: a sharded round kernel is one resident wave that waits on the
        # device for its peers; an NCCL kernel slipping onto the GPU between two of its launches could take a CTA slot and
        # wait for a peer whose own NCCL kernel is queued behind a round kernel that waits for us (DESIGN.md section 9).
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    t_bench0 = time.perf_counter()

    def log(msg):  # progress on stderr (stdout carries exactly one JSON line)
        if rank == 0:
            print(f"[bench +{time.perf_counter() - t_bench0:7.2f}s] {msg}", file=sys.stderr, flush=True)

    # ------------------------------------------------ device-resident timing (value)
    # One handle, one device-resident checkpoint (swim_sim_save at round 0): every timing window starts from the same state
    # and runs the same rounds, so the windows differ only by the machine.
    log(f"workload built: {n} nodes, world {world}")
    # ONE handle serves every leg below (the host-side index build of swim_sim_set_view is the expensive part of a handle,
    # tens of seconds per rank at 8 x C3): the checkpoint is taken at round 0 WITHOUT pending events; a leg that runs the
    # event trace from the queue does load() + inject(events), the end-to-end leg injects round by round instead.
    sim = fresh(inject=False)
    # a non-default torch stream: its handle is what the library launches on, so the torch events
    # below bracket the kernels (handle 0 would mean "the handle's private stream" to the C ABI)
    stream = torch.cuda.Stream()
    assert stream.cuda_stream != 0
    sim.set_stream(stream.cuda_stream)
    sim.save()

    def restart(flags=0, inject=True):
        # swim_sim_load moves the round counter back and re-arms the cross-GPU handshake words of THIS rank: it is a collective
        # — no rank may step before every rank has loaded (a peer's first publication would be wiped out by a late load and
        # its owner would wait for it until the watchdog fires), so: barrier, load, barrier.
        barrier()
        sim.load()
        if sim.cfg.flags != flags:
            sim.set_params(flags=flags)
        if inject:
            sim.inject(events)
        barrier()

    restart()
    clocks = ClockSampler(local) if rank == 0 else None  # runs until the end of the e2e region
    # clock spin-up: a fresh process finds the GPU at its idle clock (~1 GHz on this pool) and a 2 ms window is over
    # before the governor reacts; run real rounds for a while first, then go back to the checkpoint. (Not part of the
    # W warm-up rounds: those are rounds 1..W of the workload and precede every window.)
    barrier()
    t_spin = time.perf_counter()
    while args.spinup > 0:
        sim.step(256)
        go = time.perf_counter() - t_spin < args.spinup
        if world > 1:  # every rank must issue the same steps (a shard's kernel waits for its peers): one decision for all
            t = torch.tensor([int(go)], device=_TENSOR_DEVICE)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            go = bool(t.item())
        if not go:
            break
    windows = []
    ctr_delta, launches = None, 0
    for w in range(args.windows):
        restart()
        sim.step(args.warmup)
        c0, l0 = sim.counters(), sim.launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record(stream)
        sim.step_async(args.steps)
        ev1.record(stream)
        barrier()
        ms_w = ev0.elapsed_time(ev1)
        sim.sync()
        if sim.round != args.warmup + args.steps:
            raise RuntimeError(f"timed window ended at round {sim.round}, not {args.warmup} + {args.steps}")
        c1, l1 = sim.counters(), sim.launch_count()
        if world > 1:
            t = torch.tensor([ms_w], device=_TENSOR_DEVICE)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_w = float(t.item())
        windows.append(ms_w)
        if ctr_delta is None:
            if world > 1:
                cd = torch.tensor((c1 - c0).astype(np.int64), device=_TENSOR_DEVICE)
                dist.all_reduce(cd)
                ctr_delta = cd.cpu().numpy().astype(np.uint64)
            else:
                ctr_delta = c1 - c0
            launches = int(l1 - l0)
        if args.dump_outputs and w == args.windows - 1:
            write_outputs(sim, args.dump_outputs, n, rank, world)
    ms = float(np.median(windows))
    log(f"timed windows done: {windows}")
    value = n * args.steps / (ms * 1e-3)

    # ------------------------------------------------ phase timeline of the same rounds (fused kernel, in-kernel timer)
    timeline = None
    if True:  # (sharded runs: stamps exist only on the fused-kernel path, SWIM_ROUND_KERNEL; each rank reports its own CTA 0)
        restart()
        sim.step(args.warmup)
        sim.set_timeline(args.steps)
        sim.step(args.steps)
        tl = sim.timeline(args.steps).astype(np.int64)
        sim.set_timeline(0)
        timeline = summarize_timeline(tl, args.warmup)

    log("timeline done")
    # ------------------------------------------------ per-kernel timing of the same rounds (split launches)
    restart()
    sim.step(args.warmup)
    sim.set_profile(True)
    sim.step(args.steps)
    prof = sim.profile_ms()
    sim.set_profile(False)

    log("split-kernel profile done")
    # ------------------------------------------------ parity leg: the rounds just timed, against the oracle on the same N
    # (the checker, outside every timed region): global digest (shard digests add up), counters and convergence count
    # after W + K rounds (at most 40: through the crash burst) from the same checkpoint
    parity = None
    if not args.no_parity:
        rounds_chk = min(args.warmup + args.steps, 40)
        restart()
        sim.step(rounds_chk)
        dg = sdist.global_digest(sim.digest())
        gc = sdist.global_sum(sim.counters())
        gm = int(sdist.global_sum([sim.mismatches()])[0])
        if rank == 0:
            from oracle.oracle import Oracle, set_num_threads
            set_num_threads(int(os.environ.get("SWIM_CPU_THREADS", usable_cpus())))
            orc = Oracle(default_config(**cfg_kw))
            orc.set_view(nbr)
            orc.inject(events)
            orc.step(rounds_chk)
            bad = []
            if dg != orc.digest():
                bad.append("digest")
            if [int(x) for x in gc] != [int(x) for x in orc.counters()]:
                bad.append("counters")
            if gm != orc.mismatches():
                bad.append("mismatches")
            parity = {"status": "ok" if not bad else "FAILED: " + ",".join(bad), "rounds": rounds_chk, "n_nodes": n,
                      "digest": f"{dg:016x}", "what": "global state digest + all counters + convergence count of the CUDA run "
                      f"(all {world} shard(s)) == restated C oracle on the same N, seed and event trace"}
            del orc
    log(f"parity leg done: {parity['status'] if parity else None}")
    ab_round, ab_tick, m_bar, b_bar = algorithmic_bytes(cfg_kw, n, args.steps, ctr_delta)
    peaks = {}
    pk_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk_path):
        peaks = json.load(open(pk_path))
    peak = float(peaks.get("hbm_gbs", 6650.0))
    n_local = n // world
    rounds_p = max(1.0, prof["rounds"])
    roofline = make_roofline(cfg_kw, n_local, ms / args.steps, ab_round, m_bar, b_bar, peak, bool(peaks), prof, rounds_p,
                             timeline, ctr_delta, args.steps, world)

    # ------------------------------------------------ end to end through the C ABI, host buffers
    e2e = None
    if True:
        by_round = {}
        for e in events:
            by_round.setdefault(int(e["round"]), []).append(e)
        by_round = {r: np.array(v, dtype=A.EVENT_DTYPE) for r, v in by_round.items()}
        h2d = d2h = 0

        def one_round(r):
            nonlocal h2d, d2h
            arr = by_round.get(r)
            if arr is not None:
                sim.inject(arr)  # host buffer -> library (pinned staging) -> device, uploaded by the step below
                h2d += arr.nbytes
            # one round, and its result as a convergence study reads it — the cumulative counters and the convergence
            # count — in ONE C-ABI call (swim_sim_step_observe): the device writes them into mapped pinned host memory
            # behind the round and the call polls a sequence number there (the state digest is a parity tool: 370 MB of
            # reads per call, not part of the metric)
            if use_step_observe[0]:
                try:
                    c, mm = sim.step_observe(1)
                    d2h += c.nbytes + 24
                    return c, None, mm
                except Exception as exc:  # noqa: BLE001 — fall back to the two-call form, and say so in the JSON line
                    use_step_observe[0] = False
                    e2e_notes.append(f"swim_sim_step_observe failed ({exc}); fell back to step_async + observe")
                    raise
            sim.step_async(1)
            c, dg, mm = sim.observe(digest=False)
            d2h += c.nbytes + 8
            return c, dg, mm

        e2e_windows = []
        use_step_observe, e2e_notes = [True], []
        restart(inject=False)
        try:  # one probe round outside every timed window: the mapped-memory read-back must work on this box
            one_round(1)
        except Exception:  # noqa: BLE001
            if world > 1:  # (a fallback taken by one rank alone would desynchronise the ranks' collectives: fail loudly)
                raise
            sim.close()
            sim = fresh(inject=False)
            sim.set_stream(stream.cuda_stream)
            sim.save()
        for w in range(args.windows):
            restart(inject=False)
            for r in range(1, args.warmup + 1):
                one_round(r)
            h2d = d2h = 0
            barrier()
            t0 = time.perf_counter()
            for r in range(args.warmup + 1, args.warmup + args.steps + 1):
                one_round(r)
            sim.sync()  # surfaces a watchdog report, if any; the stream is already idle
            barrier()
            dt = time.perf_counter() - t0
            if world > 1:
                t = torch.tensor([dt], device=_TENSOR_DEVICE)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t.item())
            e2e_windows.append(dt)
        dt = float(np.median(e2e_windows))
        e2e = {"value": n * args.steps / dt, "unit": "node-rounds/s", "h2d_bytes_per_step": h2d / args.steps,
               "d2h_bytes_per_step": d2h / args.steps,
               "windows_ms": [round(x * 1e3, 4) for x in e2e_windows], "notes": e2e_notes,
               "api": "swim_sim_step_observe" if use_step_observe[0] else "swim_sim_step_async + swim_sim_observe",
               "what": "per round: swim_sim_inject(host events, when the round has any) + swim_sim_step_observe(1): one round, then "
                       "the counters and the convergence count written by the device into mapped pinned host memory — host "
                       "wall clock, max over ranks, median of the windows"}
    clk = clocks.stop() if clocks else None
    log("e2e done")

    # ------------------------------------------------ convergence metric (second half of BASELINE's metric)
    conv = None
    if rank == 0 or world > 1:
        def rounds_to_convergence(flags):
            restart(flags=flags)
            sim.step(CRASH_ROUND)
            r = CRASH_ROUND
            mm = None
            stride = 8  # coarse while thousands of view entries are wrong, exact (every round) in the tail
            while r < args.converge_limit:
                sim.step(stride)
                r += stride
                mm = sim.mismatches()
                if world > 1:
                    t = torch.tensor([mm], device=_TENSOR_DEVICE, dtype=torch.int64)
                    dist.all_reduce(t)
                    mm = int(t.item())
                if mm == 0:
                    break
                if mm < 64:
                    stride = 1
            return (r if mm == 0 else None), mm

        r0, mm0 = rounds_to_convergence(0)
        # the same workload with the paper's round-robin probe order (SWIM_F_ROUND_ROBIN, `-- FIXME: move from random to
        # robust scheme`, Core.hs:232): every observer reaches the crashed member within 2 view_cap - 1 rounds
        r1, mm1 = rounds_to_convergence(A.F_ROUND_ROBIN)
        conv = {"rounds_to_convergence": r0, "checked_every": "8 rounds, every round once fewer than 64 view entries are wrong", "limit": args.converge_limit, "mismatches_at_end": mm0,
                "crash_round": CRASH_ROUND, "rounds_to_convergence_round_robin": r1, "mismatches_at_end_round_robin": mm1}

    log(f"convergence done: {conv}")
    if sim.cfg.flags:
        sim.set_params(flags=0)
    sim.close()
    # ------------------------------------------------ second workload: the state machine under load (ring-lattice views)
    # C3's uniformly random views almost never let a receiver know the member a record is about (32 of 2^20), so its
    # dissemination path idles. With ring-lattice views (each node knows its 32 nearest ids) records reach nodes that know
    # the member: every delivered record runs through suspectOrDeadNode' (Core.hs:142-187) and many change state. Same N,
    # k, fanout, B, S, T, crash set and window; reported beside the headline workload, not instead of it.
    ring = None
    if world == 1 and not args.no_ring:
        from swim_b200.sim import generate_topology
        nbr_ring = generate_topology("ring", n, 32, 32, seed=3)
        sim = Simulator(default_config(rank=rank, world=world, device=local, **cfg_kw))
        sim.set_view(nbr_ring)
        sim.inject(events)
        sim.set_stream(stream.cuda_stream)
        sim.save()
        wins = []
        cdelta = None
        for w in range(args.windows):
            sim.load()
            sim.step(args.warmup)
            c0 = sim.counters()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            ev0.record(stream)
            sim.step_async(args.steps)
            ev1.record(stream)
            torch.cuda.synchronize()
            wins.append(ev0.elapsed_time(ev1))
            sim.sync()
            cdelta = sim.counters() - c0
        sim.load()
        sim.step(args.warmup)
        sim.set_timeline(args.steps)
        sim.step(args.steps)
        tl_ring = summarize_timeline(sim.timeline(args.steps).astype(np.int64), args.warmup)
        sim.set_timeline(0)
        # rounds to convergence, checked every round
        sim.load()
        sim.step(CRASH_ROUND)
        r_conv = None
        for r in range(CRASH_ROUND + 1, min(args.converge_limit, 400) + 1):
            sim.step(1)
            if sim.mismatches() == 0:
                r_conv = r
                break
        # parity of this workload too (the oracle, outside every timed region)
        ring_parity = None
        if not args.no_parity:
            from oracle.oracle import Oracle
            rounds_chk = min(args.warmup + args.steps, 40)
            sim.load()
            sim.step(rounds_chk)
            orc = Oracle(default_config(**cfg_kw))
            orc.set_view(nbr_ring)
            orc.inject(events)
            orc.step(rounds_chk)
            ring_parity = "ok" if (sim.digest() == orc.digest() and sim.counters().tolist() == orc.counters().tolist()) else "FAILED"
            del orc
        sim.close()
        ms_r = float(np.median(wins))
        cd = dict(zip(A.CTR_NAMES, [int(x) for x in cdelta]))
        ring = {"workload": f"ring-lattice views: node i knows i-16..i+16, N={n}, otherwise C3 (k=3, fanout=4, B=8, S=5, T=8, "
                            f"{CRASH_PPM / 1e4:.1f}% crash at round {CRASH_ROUND})",
                "value": n * args.steps / (ms_r * 1e-3), "unit": "node-rounds/s", "ms_per_step": ms_r / args.steps,
                "windows_ms": [round(x, 5) for x in wins], "rounds_to_convergence": r_conv,
                "recs_applied_over_recs_sent": cd["recs_applied"] / max(1, cd["recs_sent"]),
                "msgs_delivered_to_k2_note": "ring views: nearly every envelope passes the recipient's membership filter",
                "counters_timed_region": cd, "timeline": tl_ring, "parity_check": ring_parity}

    log("ring workload done" if ring else "ring workload skipped")
    # ------------------------------------------------ CPU baseline (rank 0, N=1 only): bounded sample
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        rounds = 512  # a bounded sample of roughly 10-30 s of CPU work on the box's host cores
        val, dt, threads, _ = cpu_arm(cfg_kw, nbr, events, n, rounds, 3)
        cpu = {"value": val, "unit": "node-rounds/s", "cores": threads, "kind": "port",
               "sample": f"all {n} nodes of C3, rounds 4..{3 + rounds} ({dt:.1f} s of CPU wall time; restated C "
                         "oracle with OpenMP; the Haskell reference cannot be built here: no GHC)"}

    if rank == 0:
        line = {"metric": "simulated node-rounds/sec", "value": value, "unit": "node-rounds/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/u32",
                "data": "synthetic", "config": config_dict(cfg_kw, n, world, exchange["mode"]), "clocks": clk, "e2e": e2e,
                "timing": {"windows_ms": [round(x, 5) for x in windows], "stat": "median", "min_ms": min(windows),
                           "max_ms": max(windows), "spinup_s": args.spinup,
                           "how": "every window: swim_sim_load (device checkpoint of round 0) -> W warm-up rounds -> "
                                  "K timed rounds between CUDA events on the launching stream, max over ranks"},
                "gpu_launches": launches,
                "gpu_launches_note": "round_kernel<1> runs K1a, K1b and K2 of every consecutive event-free round of a call "
                                     "in ONE launch (grid barriers between phases), so the timed region of K rounds is a "
                                     "handful of launches, not 3K",
                "parity_check": parity["status"] if parity else None, "parity": parity,
                "roofline": roofline, "cpu_baseline": cpu, "convergence": conv, "state_machine_workload": ring,
                "counters_timed_region": dict(zip(A.CTR_NAMES, [int(x) for x in ctr_delta]))}
    else:
        line = None
    if world > 1:
        dist.destroy_process_group()
    return line


class StdoutToStderr:
    """Everything third parties print on fd 1 during the run (e.g. NCCL's version banner) goes to stderr, so that
    stdout carries exactly ONE line: the JSON result."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=448, help="rounds in each timed window")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--nodes-per-gpu", type=int, default=N_PER_GPU)
    ap.add_argument("--converge-limit", type=int, default=1200)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the post-run parity leg against the oracle")
    ap.add_argument("--no-ring", action="store_true", help="skip the second (ring-lattice) workload")
    ap.add_argument("--windows", type=int, default=5, help="timed windows of --steps rounds each; the median is reported")
    ap.add_argument("--spinup", type=float, default=0.5, help="seconds of untimed rounds before the first window (GPU clocks)")
    ap.add_argument("--exchange", default=None, choices=[None, "p2p", "nccl"],
                    help="cross-shard exchange: fused peer-memory (default) or staged NCCL all-to-all")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the state the last timed window computed to DIR/<name>.npy (float64, a seeded node sample)")
    args = ap.parse_args()
    if args.steps < 1 or args.windows < 1:
        ap.error("--steps and --windows must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    with StdoutToStderr():
        line = run_reference(args) if args.impl == "reference" else run_cuda(args)
    if line is not None:
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
