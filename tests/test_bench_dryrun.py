"""bench.py's CUDA arm end to end WITHOUT a GPU: the library is the emulator build (tests/emu: the CUDA sources compiled for
the CPU), `torch.cuda` is replaced by a handful of stand-ins (streams and events are wall-clock stamps). Not a measurement
— the numbers mean nothing — but every leg of the single-GPU flow runs: the one shared handle with its checkpoint, the timed
windows, the phase timeline parser, the split-kernel profile, the parity leg against the oracle, the end-to-end loop through
swim_sim_step_observe, both convergence legs (parameter change on the live handle), the ring-lattice workload and the CPU arm.
What the driver runs on hardware must at least be free of Python-level mistakes."""
import argparse
import json
import os
import sys
import time

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _Stream:
    cuda_stream = 0x1000  # any non-zero handle: the emulated runtime never looks inside a stream


class _Event:
    def __init__(self, enable_timing=False):
        self.t = None

    def record(self, stream=None):
        self.t = time.perf_counter()

    def elapsed_time(self, other):
        return max(1e-3, (other.t - self.t) * 1e3)


@pytest.fixture()
def emulated_bench(monkeypatch):
    import torch
    import swim_b200._lib as L
    sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
    import build_emu
    saved = (L.SO_PATH, L._lib)
    L.SO_PATH, L._lib = build_emu.build(), None
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(torch.cuda, "set_device", lambda *_a, **_k: None)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *_a, **_k: None)
    monkeypatch.setattr(torch.cuda, "Stream", _Stream)
    monkeypatch.setattr(torch.cuda, "Event", _Event)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "LOCAL_WORLD_SIZE"):
        monkeypatch.delenv(k, raising=False)
    sys.path.insert(0, ROOT)
    import bench
    yield bench
    L.SO_PATH, L._lib = saved


@pytest.mark.parametrize("steps,xmode", [(20, None), (40, None), (12, "1")])
def test_cuda_arm_runs_every_leg_on_the_emulator(emulated_bench, steps, xmode, monkeypatch, capsys):
    bench = emulated_bench
    if xmode is not None:
        monkeypatch.setenv("SWIM_XMODE", xmode)
    args = argparse.Namespace(gpus=1, steps=steps, warmup=5, impl="cuda", nodes_per_gpu=8192, converge_limit=160, no_cpu=False,
                              no_parity=False, no_ring=False, windows=2, spinup=0.0, exchange=None, dump_outputs=None)
    line = bench.run_cuda(args)
    json.dumps(line)  # serialisable
    assert line["metric"] == "simulated node-rounds/sec" and line["n_gpus"] == 1 and line["steps"] == steps
    assert line["value"] > 0 and line["ms_per_step"] > 0 and line["higher_is_better"] is True
    assert line["parity_check"] == "ok", line["parity"]
    assert line["gpu_launches"] >= 1
    e = line["e2e"]
    assert e["value"] > 0 and e["api"] == "swim_sim_step_observe" and not e["notes"] and len(e["windows_ms"]) == 2
    assert e["d2h_bytes_per_step"] > 0  # counters + convergence count every round
    r = line["roofline"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic", "kernel", "latency_floor", "split_kernels_us"):
        assert k in r
    assert r["kernel"].startswith("round_kernel")
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["value"] > 0
    c = line["convergence"]
    assert c["crash_round"] == bench.CRASH_ROUND and "rounds_to_convergence_round_robin" in c
    g = line["state_machine_workload"]
    assert g["parity_check"] == "ok" and g["value"] > 0
    assert line["config"]["n_nodes"] == 8192 and "workload" in line["config"]


def _check_dump(bench, out_dir, n_nodes, rounds, tmp_path):
    """What --dump-outputs wrote is the state the oracle reaches after the same rounds of the same workload, file for file."""
    import numpy as np
    from oracle.oracle import Oracle
    from swim_b200.sim import default_config
    cfg_kw, nbr, events, n = bench.workload(1, n_nodes)
    orc = Oracle(default_config(**cfg_kw))
    orc.set_view(nbr)
    orc.inject(events)
    orc.step(rounds)
    want = tmp_path / "oracle_outputs"
    bench.write_outputs(orc, str(want), n)
    names = sorted(os.listdir(out_dir))
    assert names == sorted(os.listdir(want))
    assert {"counters.npy", "digest.npy", "mismatches.npy", "sample_nodes.npy", "nbr.npy", "pb_member.npy"} <= set(names)
    for f in names:
        got = np.load(os.path.join(out_dir, f))
        assert got.dtype == np.float64 and np.array_equal(got, np.load(want / f)), f
    assert np.load(want / "counters.npy").tolist() == [float(x) for x in orc.counters()]
    assert len(np.load(want / "sample_nodes.npy")) == min(n, bench.DUMP_NODES)


def test_dump_outputs_on_the_emulator(emulated_bench, tmp_path, monkeypatch):
    """--dump-outputs: the state of the last timed round (warm-up + steps), sampled when the node set is larger than
    DUMP_NODES, equals the oracle's."""
    bench = emulated_bench
    monkeypatch.setattr(bench, "DUMP_NODES", 1000)
    out = tmp_path / "outputs"
    args = argparse.Namespace(gpus=1, steps=12, warmup=5, impl="cuda", nodes_per_gpu=4096, converge_limit=40, no_cpu=True,
                              no_parity=True, no_ring=True, windows=2, spinup=0.0, exchange=None, dump_outputs=str(out))
    line = bench.run_cuda(args)
    assert line["steps"] == 12
    _check_dump(bench, out, 4096, 5 + 12, tmp_path)


# ---------------------------------------------------------------- the sharded flow: ranks as threads of one process
class _ThreadDist:
    """The few torch.distributed calls bench.py and swim_b200/dist.py make, for `world` ranks that are threads of this
    process (rank = a thread-local): every collective is two passes through one threading.Barrier."""

    def __init__(self, world):
        import threading
        self.world = world
        self.bar = threading.Barrier(world, timeout=120)
        self.tl = threading.local()
        self.slots = [None] * world

    def _exchange(self, value):
        self.slots[self.tl.rank] = value
        self.bar.wait()
        got = list(self.slots)
        self.bar.wait()  # everybody has read before the slots are written again
        return got

    def init_process_group(self, *_a, **_k): pass
    def destroy_process_group(self, *_a, **_k): pass
    def is_initialized(self): return True
    def get_world_size(self, *_a): return self.world
    def get_rank(self, *_a): return self.tl.rank
    def get_backend(self, *_a): return "gloo"
    def barrier(self, *_a, **_k): self.bar.wait()

    def all_reduce(self, t, op=None):
        import torch
        vals = torch.stack([v for v in self._exchange(t.clone())])
        is_max = op is not None and "MAX" in str(op).upper()
        t.copy_(vals.max(dim=0).values if is_max else vals.sum(dim=0))

    def all_gather_object(self, out, obj):
        out[:] = self._exchange(obj)

    def broadcast_object_list(self, lst, src=0):
        got = self._exchange(list(lst))
        lst[:] = got[src]


@pytest.mark.parametrize("world,steps", [(2, 20), (3, 12)])
def test_sharded_cuda_arm_on_the_emulator(emulated_bench, world, steps, monkeypatch, tmp_path):
    """bench.py --gpus N with the ranks as threads (each with its own handle on the emulated device, connected through raw
    peer pointers exactly as ranks of one process are on hardware): the collective structure of every leg — load as a
    collective, the spin-up that ends on one decision for all ranks, streams drained before barriers, the end-to-end loop
    one round per call with in-kernel handshakes, parameter change for the round-robin convergence leg. A rank that steps
    out of line dead-locks here (the barrier times out after 120 s) instead of on the driver's 8-GPU box."""
    import threading
    import torch
    bench = emulated_bench
    fake = _ThreadDist(world)
    for name in ("init_process_group", "destroy_process_group", "is_initialized", "get_world_size", "get_rank", "get_backend",
                 "barrier", "all_reduce", "all_gather_object", "broadcast_object_list"):
        monkeypatch.setattr(torch.distributed, name, getattr(fake, name))
    monkeypatch.setattr(bench, "_TENSOR_DEVICE", "cpu")
    monkeypatch.setenv("SWIM_ROUND_KERNEL", "1")

    class _Env:
        def get(self, key, default=None):
            r = fake.tl.rank
            return {"RANK": str(r), "LOCAL_RANK": str(r), "WORLD_SIZE": str(world), "LOCAL_WORLD_SIZE": str(world)}.get(key, os.environ.get(key, default))

    monkeypatch.setattr(bench, "_ENV", _Env())
    # ranks never arrive together on a real box: every rank is late by its own amount at the calls that move the round
    # counter (the race bench.py once lost: a late swim_sim_load wiping out a peer's first publication)
    from swim_b200.sim import Simulator
    real_load = Simulator.load

    def late_load(self):
        time.sleep(0.03 * fake.tl.rank)
        real_load(self)

    monkeypatch.setattr(Simulator, "load", late_load)
    lines, errs = [None] * world, []

    def rank_main(r):
        fake.tl.rank = r
        args = argparse.Namespace(gpus=world, steps=steps, warmup=5, impl="cuda", nodes_per_gpu=2048, converge_limit=120, no_cpu=True,
                                  no_parity=False, no_ring=True, windows=2, spinup=0.05, exchange=None,
                                  dump_outputs=str(tmp_path / "outputs"))
        try:
            lines[r] = bench.run_cuda(args)
        except BaseException as e:  # noqa: BLE001
            errs.append((r, repr(e)))
            fake.bar.abort()

    ts = [threading.Thread(target=rank_main, args=(r,), daemon=True) for r in range(world)]
    for t in ts:
        t.start()
    for t in ts:
        t.join(timeout=600)
    assert not errs, errs
    assert not any(t.is_alive() for t in ts), "a rank is stuck"
    line = lines[0]
    assert all(ln is None for ln in lines[1:])  # rank 0 alone reports
    json.dumps(line)
    assert line["n_gpus"] == world and line["config"]["n_nodes"] == 2048 * world and line["config"]["exchange"] == "p2p"
    assert line["parity_check"] == "ok", line["parity"]
    assert line["value"] > 0 and line["e2e"]["value"] > 0 and line["e2e"]["api"] == "swim_sim_step_observe"
    assert line["convergence"] is not None and line["state_machine_workload"] is None and line["cpu_baseline"] is None
    _check_dump(bench, tmp_path / "outputs", 2048 * world, 5 + steps, tmp_path)  # the shards' rows, gathered by rank 0
