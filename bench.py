#!/usr/bin/env python
"""bench.py — AppendEntries/sec across Raft groups on B200 (BASELINE.json metric).

Unit of work = one AppendEntries ack consumed by the leader path (ack -> Leadership.State update -> quorum index ->
commitIndex).  One engine LAUNCH drains one batch: ROWS ticks x G groups, each tick one group op (SUBMIT / heartbeat) and
one ack per follower lane.  One bench STEP = one pass over a recorded WINDOW of L consecutive batches of the synthetic
stream (L x ROWS ticks: at N=1, 128 x 16 = 2 048 ticks, twice the 1 024 timed ticks SURVEY.md §8(d) names for config #2), so
that K = 20 steps give a timed region of >= 100 ms.  The window is generated closed-loop on the device (the peers are workload.cu), recorded in HBM
and replayed bit-exactly; each replay starts by rolling the tables back to the window's start (a 22 MB device copy
enqueued on the step stream, inside the timed region, < 0.5 % of it).

  N == 1   BASELINE config #2: 64K groups, 3 replicas, one B200.
  N  > 1   BASELINE config #4: 1 M groups (same total at N = 2, 4, 8: strong scaling), contiguous gid blocks per rank, one
           ncclAllGather of commitIndex[G/N] after EVERY launch; the last gathered vector of the timed region is
           checked against the ranks' own commit columns (config.gather_verified).

  value     device-resident inputs, CUDA events on the engine's stream, max over ranks.
  e2e       the same stream through the C-ABI host path (rafting_step_begin_host / rafting_step_wait_slot): pinned host
            inbox -> H2D -> kernel -> D2H of the outbox, every launch inside the timed region.
  roofline  algorithmic bytes per ack (192 B at R=3, SURVEY.md §8d) x acks per launch / mean kernel time, against
            MEASURED_PEAKS.json's HBM copy bandwidth.
  cpu_baseline / --impl reference
            the CPU restatement of the reference's EventLoop path (oracle/, "port": the reference is Java and neither
            this image nor the GPU box has a JDK) on every host core, on a bounded sample of the same stream.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

SEED2, SEED4 = 0x5EED0002, 0x5EED0004
WORKLOAD2 = "64K RaftContext groups, 3 replicas, synthetic AppendEntries stream on 1xB200"
WORKLOAD4 = "1M groups, 3 replicas, sharded across {n}xB200 with NCCL commitIndex all-gather"
G_CONFIG2, G_CONFIG4 = 65536, 1 << 20
METRIC = "AppendEntries/sec across Raft groups"


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--groups", type=int, default=0, help="groups per GPU (default: 65536 at N=1, 1M/N at N>1)")
    p.add_argument("--replicas", type=int, default=3)
    p.add_argument("--rows", type=int, default=16, help="ticks per launch")
    p.add_argument("--launches", type=int, default=0, help="launches per step = length of the recorded window (default: sized to ~7 GB of inboxes)")
    p.add_argument("--cpu-groups", type=int, default=65536, help="groups in the CPU sample")
    p.add_argument("--cpu-launches", type=int, default=4, help="oracle passes (rows ticks each) per CPU step")
    p.add_argument("--cpu-steps", type=int, default=12, help="timed steps of the in-line cpu_baseline leg")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-cpu", action="store_true")
    p.add_argument("--no-secondary", action="store_true", help="skip the vote / follower-request rates (configs #3, #5)")
    p.add_argument("--no-bind", action="store_true", help="do not bind the process to the GPU's NUMA node")
    p.add_argument("--log-appends", action="store_true",
                   help="experiment (SURVEY 8(f)-1): a second host thread appends entry payloads to the HBM entry buffer "
                        "(rafting_log_append, its own stream) during the whole timed region; the line gains run.log_appends")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="after the timed steps, write the outbox of the last launch of the last timed step as DIR/<column>.npy "
                        "(float64, at most 64 MB in all: a fixed sample of groups, listed in gids.npy), so that two builds can be "
                        "compared output for output")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    return args


def b_ack(R):                      # SURVEY.md §8(d): B_ack(R) = 184 + 8 (R - 2)
    return 184 + 8 * (R - 2)


def measured_traffic(G, R, rows):
    """DRAM bytes per launch from the committed ncu --set full capture (only valid for the profiled shape)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        if (G, R, rows) == (65536, 3, 16):
            return float(t["traffic_bytes_per_launch"]), t["source"]
    except Exception:
        pass
    return None, None


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def inbox_bytes_per_launch(G, rows, F):
    """op_meta 8 + op_nr 16 per (row, group); ev_meta 8 + ev_tn 16 + ev_el 16 per (row, group, lane)."""
    return rows * G * (24 + 40 * F)


def window_launches(args, G):
    """launches per step = length of the recorded window: up to ~14 GB of distinct inboxes in HBM, 4..128 launches."""
    return args.launches or int(max(4, min(128, 14.0e9 // inbox_bytes_per_launch(G, args.rows, args.replicas - 1))))


def workload_config(args, world, G):
    """The `config` object: the workload definition, identical in the engine arm and in the reference arm."""
    if world == 1:
        name, total, seed = WORKLOAD2, G, SEED2
    else:
        name, total, seed = WORKLOAD4.format(n=world), G * world, SEED4
    L = window_launches(args, G)
    return {"workload": name, "groups_total": total, "groups_per_gpu": G, "replicas": args.replicas, "rows_per_launch": args.rows,
            "launches_per_step": L, "ticks_per_step": L * args.rows, "seed": hex(seed),
            "step": "one pass over a window of consecutive batches of the stream (ticks per step = launches x rows); the CPU arm "
                    "times a bounded sample of it (cpu_baseline.sample)"}


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons sampled while `armed` (NVML in-process every ~2 ms; nvidia-smi subprocess as a fallback)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.armed = index, False, False
        self.sm, self.mx, self.reasons, self.power = [], [], set(), []
        self.nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = (pynvml, pynvml.nvmlDeviceGetHandleByIndex(index))
        except Exception:
            self.nv = None

    def sample_nvml(self):
        nv, h = self.nv
        sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        try:
            bits = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
            bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        try:
            self.power.append(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)
        except Exception:
            pass
        self.sm.append(float(sm)); self.mx.append(float(mx))
        for bit, name in self.REASONS.items():
            if bits & bit:
                self.reasons.add(name)

    def sample_smi(self):
        out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        r = [x.strip() for x in out.split(",")]
        if len(r) > 8 and r[1].replace(".", "").isdigit():
            self.sm.append(float(r[1])); self.mx.append(float(r[2]))
            for k, nm in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
                if r[5 + k].lower().startswith("active"):
                    self.reasons.add(nm)

    def run(self):
        while not self.stop_flag:
            if self.armed:
                try:
                    self.sample_nvml() if self.nv else self.sample_smi()
                except Exception:
                    pass
                time.sleep(0.002)
            else:
                time.sleep(0.0005)

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                "reasons": sorted(self.reasons), "samples": len(self.sm), "power_w_max": max(self.power) if self.power else None,
                "source": "nvml" if self.nv else "nvidia-smi"}


# ------------------------------------------------------------------------------------------------
# host placement: a rank runs on the CPUs of the NUMA node its GPU hangs off, so that its pinned staging buffers are
# first-touched there and every H2D / D2H copy stays off the socket interconnect
# ------------------------------------------------------------------------------------------------
def parse_cpulist(txt):
    cpus = set()
    for part in txt.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        cpus.update(range(int(a), int(b or a) + 1))
    return cpus


def bind_to_gpu_numa(local_rank):
    try:
        bus = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(local_rank)],
                             capture_output=True, text=True, timeout=10).stdout.strip().lower()
        if bus.startswith("00000000:"):
            bus = bus[4:]
        path = f"/sys/bus/pci/devices/{bus}/local_cpulist"
        cpus = parse_cpulist(open(path).read()) & os.sched_getaffinity(0)
        node = open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip()
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"numa_node": int(node), "cpus": len(cpus), "pci": bus}
    except Exception as ex:            # no sysfs entry (container without the topology): stay unbound
        return {"numa_node": None, "error": str(ex)[:80]}
    return {"numa_node": None}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle (port of the reference's EventLoop path) on a bounded sample of the same stream
# ------------------------------------------------------------------------------------------------
def interleave_host_memory():
    """MPOL_INTERLEAVE over every NUMA node for this thread's future allocations (the recorded inboxes of the CPU arm): the loop
    threads of both sockets then stream their inputs at the same bandwidth.  Best effort (raw syscall, no libnuma here)."""
    try:
        nodes = [int(d[4:]) for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()]
        if len(nodes) < 2:
            return False
        mask = C.c_ulong(sum(1 << n for n in nodes))
        libc = C.CDLL(None, use_errno=True)
        return libc.syscall(238, 3, C.byref(mask), C.c_ulong(max(nodes) + 2)) == 0        # set_mempolicy(MPOL_INTERLEAVE)
    except Exception:
        return False


def run_cpu_sample(args, threads, steps, warmup, launches, seed):
    """steps x (launches oracle passes of rows ticks over cpu_groups groups), RECORD then REPLAY like the GPU arm: a first
    oracle instance runs the closed loop (oracle pass -> simulated peers -> next inbox) untimed and keeps every inbox; a
    second, fresh instance then replays the recorded inboxes back to back with nothing between the passes, so the loop
    threads never park on the single-threaded generator.  Only orc_step of the replay is inside the clock; outboxes are
    preallocated and touched once; the two instances must end with identical commit columns."""
    from oracle import binding
    from rafting_b200 import abi, workload
    G, R, rows = args.cpu_groups, args.replicas, args.rows
    cfg = abi.make_cfg(replicas=R, max_groups=G, max_rows=rows)
    interleaved = interleave_host_memory()
    init = np.zeros(G, dtype=abi.GROUP_INIT_DTYPE)
    init["ballot"] = -1; init["first_index"] = 1; init["now_ms"] = workload.T0_MS - 2000
    init["term"] = np.arange(G) % 7
    w1 = workload.make_wl(seed, 1, G, R - 1)
    w = workload.make_wl(seed, rows, G, R - 1)
    L = binding.lib()
    outs = [abi.Outbox(rows, G, R - 1, G) for _ in range(2)]
    for ob in outs:                                         # touch every page once, outside the clock
        for name, _, _ in abi.Outbox.ROW_COLS:
            getattr(ob, name)[...] = 0
        for name, _ in abi.Outbox.GROUP_COLS:
            getattr(ob, name)[...] = 0
    n_pass = (warmup + steps) * launches

    def fresh():
        o = binding.Oracle(cfg)
        o.open_bulk(0, init)
        out, elect = None, []
        for ph in (0, 1, 2):
            ib = workload.election_inbox_host(w1, ph, out)
            out = o.step(ib, threads=threads)
            elect.append(ib)
        return o

    # ---- record (untimed) ----
    o = fresh()
    inboxes, acks, prev = [], [], None
    for k in range(n_pass):
        ib = workload.leader_inbox_host(w, k, prev)
        acks.append(int(((ib.ev_meta & np.uint64(0xF)) != 0).sum()))
        ob = outs[k % 2]
        ic, oc = ib.as_c(), ob.as_c()
        if L.orc_step(o._h, C.byref(ic), C.byref(oc), threads):
            raise RuntimeError("orc_step failed")
        inboxes.append(ib); prev = ob
    commit_a = prev.commit_index.copy()
    o.close()
    # ---- replay (timed) ----
    o = fresh()
    ics = [ib.as_c() for ib in inboxes]
    ocs = [outs[k % 2].as_c() for k in range(n_pass)]
    step_s, step_acks = [], []
    k = 0
    for s in range(warmup + steps):
        t0 = time.perf_counter()
        for _ in range(launches):
            if L.orc_step(o._h, C.byref(ics[k]), C.byref(ocs[k]), threads):
                raise RuntimeError("orc_step failed")
            k += 1
        dt = time.perf_counter() - t0
        if s >= warmup:
            step_s.append(dt); step_acks.append(sum(acks[k - launches:k]))
    replay_ok = bool(np.array_equal(commit_a, outs[(n_pass - 1) % 2].commit_index))
    o.close()
    total_s, total_acks = float(np.sum(step_s)), int(np.sum(step_acks))
    rates = np.array(step_acks) / np.array(step_s)
    return {"value": total_acks / total_s, "acks": total_acks, "seconds": total_s, "steps": len(step_s),
            "ms_per_step": 1e3 * total_s / len(step_s), "replay_ok": replay_ok, "last_outbox": outs[(n_pass - 1) % 2],
            "median_rate": float(np.median(rates)), "min_rate": float(rates.min()), "max_rate": float(rates.max()),
            "sample": f"{G} groups x {rows} ticks x {launches} passes per step x {len(step_s)} steps of the same keyed stream "
                      f"(first {G} group ids, {total_acks} acks, {total_s:.1f} s of CPU wall time), in-memory log, {threads} pinned loop "
                      f"threads taking 64-group chunks from a shared queue; recorded closed-loop by one oracle instance, replayed back "
                      f"to back by a fresh one (only orc_step is timed; inbox pages interleaved over NUMA nodes: {interleaved}; "
                      f"replay == record: {replay_ok})"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    cores = len(os.sched_getaffinity(0))
    seed = SEED2 if world == 1 else SEED4
    G = args.groups or (G_CONFIG2 if world == 1 else G_CONFIG4 // world)
    res = run_cpu_sample(args, threads=cores, steps=args.steps, warmup=max(args.warmup, 1), launches=args.cpu_launches, seed=seed)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res["last_outbox"])
    cfg = workload_config(args, world, G)
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": "acks/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"],
        "higher_is_better": True, "scaling": "weak" if world == 1 else "strong", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": res["value"], "unit": "acks/s", "cores": cores, "kind": "port", "sample": res["sample"],
                         "median_step_rate": res["median_rate"], "min_step_rate": res["min_rate"], "max_step_rate": res["max_rate"]},
        "e2e": {"value": res["value"], "unit": "acks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference is Java; no JDK in this image or on the GPU box -> oracle/ (C port of the reference's EventLoop path) is timed; "
                "this process loads liboracle.so and the stream generator librafting_workload.so, not the product library",
    }
    emit(line)


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def run_engine(args):
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    all_cpus = os.sched_getaffinity(0)
    placement = {"numa_node": None, "bound": False}
    if not args.no_bind:
        placement = bind_to_gpu_numa(local)
        placement["bound"] = placement.get("numa_node") is not None
    import torch
    import torch.distributed as dist
    from rafting_b200 import abi, devbatch, engine, workload

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()

    R, rows = args.replicas, args.rows
    G = args.groups or (G_CONFIG2 if world == 1 else G_CONFIG4 // world)
    seed = SEED2 if world == 1 else SEED4
    F = R - 1
    K, W = args.steps, max(args.warmup, 3)
    cfg = abi.make_cfg(replicas=R, max_groups=G, max_rows=rows, device=local)
    e = engine.Engine(cfg)
    gid_base = rank * G
    init = np.zeros(G, dtype=abi.GROUP_INIT_DTYPE)
    init["ballot"] = -1; init["first_index"] = 1; init["now_ms"] = workload.T0_MS - 2000
    init["term"] = (gid_base + np.arange(G)) % 7
    e.open_bulk(0, init)
    if world > 1:
        box = [engine.Engine.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        e.comm_init(rank, world, box[0])
    else:
        e.comm_init(0, 1, None)
    stream_ptr = e.stream()
    ext = torch.cuda.ExternalStream(stream_ptr, device=dev)

    # ---- election warm-up + settle, all on the device ------------------------------------------
    w1 = workload.make_wl(seed, 1, G, F, gid_base=gid_base)
    w = workload.make_wl(seed, rows, G, F, gid_base=gid_base)
    in1, out1 = devbatch.DevInbox(1, G, F, dev), devbatch.DevOutbox(1, G, F, G, dev)
    prev_c = None
    for ph in (0, 1, 2):
        ic = in1.as_c()
        workload.election_step(w1, ph, prev_c, ic, on_device=True, stream=stream_ptr)
        oc = out1.as_c()
        e.step_device(ic, oc, stream_ptr)
        prev_c = oc
    outs = [devbatch.DevOutbox(rows, G, F, G, dev) for _ in range(2)]
    # the leader stream never marks a follower unavailable: the op_ab column (its only field used by SUBMIT / TIMEOUT)
    # is omitted from the batch, as a shim would do
    probe = devbatch.DevInbox(rows, G, F, dev, unavail=False)
    inbox_bytes, outbox_bytes = probe.nbytes(), outs[0].nbytes()
    L = window_launches(args, G)
    assert inbox_bytes == inbox_bytes_per_launch(G, rows, F)
    inboxes = [probe] + [devbatch.DevInbox(rows, G, F, dev, unavail=False) for _ in range(L - 1)]
    settle = devbatch.DevInbox(rows, G, F, dev, unavail=False)
    SETTLE = 8                                # 128 ticks: every follower has acknowledged once, the stream is in steady state
    prev_out = None
    for k in range(SETTLE):
        ic = settle.as_c()
        workload.leader_step(w, k, None if prev_out is None else prev_out.as_c(), ic, on_device=True, stream=stream_ptr)
        prev_out = outs[k % 2]
        e.step_device(ic, prev_out.as_c(), stream_ptr)
    torch.cuda.synchronize()
    # keep the outbox the recorded window starts from, then checkpoint the tables
    start_out = devbatch.DevOutbox(rows, G, F, G, dev)
    for name in start_out.t:
        start_out.t[name].copy_(prev_out.t[name])
    torch.cuda.synchronize()
    e.checkpoint()

    # ---- phase A: generate + record the window closed-loop (untimed) ------------------------------
    prev_out = start_out
    for k in range(L):
        ic = inboxes[k].as_c()
        workload.leader_step(w, SETTLE + k, prev_out.as_c(), ic, on_device=True, stream=stream_ptr)
        prev_out = outs[k % 2]
        e.step_device(ic, prev_out.as_c(), stream_ptr)
    torch.cuda.synchronize()
    acks_per_launch = [int(((inboxes[k].t["ev_meta"].view(torch.int64) & 0xF) != 0).sum().item()) for k in range(L)]
    acks_window = sum(acks_per_launch)
    digest_a = e.digest(0, G)
    del start_out

    # ---- phase B: timed replay, inputs resident in HBM ---------------------------------------------
    ics = (abi.InboxC * L)(*[ib.as_c() for ib in inboxes])
    ocs = (abi.OutboxC * L)(*[outs[k % 2].as_c() for k in range(L)])
    gather = world > 1

    def window():
        e.restore(sync=False)
        e.step_device_seq(ics, ocs, L, gather=gather, stream=0)

    def warm():
        for _ in range(W):
            window()
        e.allgather_join()
        torch.cuda.synchronize(); barrier()

    sampler = ClockSampler(local); sampler.start()
    warm()
    appender = None
    if args.log_appends:
        import threading
        e.log_config(segment_bytes=1 << 22, hbm_segments=1024, ring_slots=64)        # 4 GiB arena: no spill during the run
        n_ref, payload = 16384, 256
        a_refs = np.zeros(n_ref, dtype=engine.Engine.ENTRY_REF)
        a_refs["gid"] = np.arange(n_ref, dtype=np.uint32) % G
        a_refs["len"] = payload
        a_refs["term"] = 1
        a_refs["blob_off"] = np.arange(n_ref, dtype=np.uint64) * payload
        a_blob = np.random.default_rng(5).integers(0, 256, size=n_ref * payload, dtype=np.uint8)
        a_state = {"stop": False, "calls": 0, "bytes": 0, "rc": 0, "t0": 0.0, "t1": 0.0}

        def _append_loop():
            torch.cuda.set_device(local)
            Lb = engine.lib()
            idx = 1
            a_state["t0"] = time.perf_counter()
            while not a_state["stop"]:
                a_refs["index"] = idx
                rc = Lb.rafting_log_append(e._h, a_refs.ctypes.data, n_ref, a_blob.ctypes.data, a_blob.nbytes)
                if rc:
                    a_state["rc"] = rc
                    break
                idx += 1
                a_state["calls"] += 1
                a_state["bytes"] += a_blob.nbytes
            a_state["t1"] = time.perf_counter()
        appender = threading.Thread(target=_append_loop, daemon=True)
        appender.start()
        time.sleep(0.05)
    sampler.armed = True
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(ext)
    for _ in range(K):
        window()
    e.allgather_join()                      # the timed region ends when the last summary has been gathered
    ev1.record(ext)
    torch.cuda.synchronize(); barrier()
    log_appends = None
    if appender is not None:
        a_state["stop"] = True
        appender.join(timeout=30)
        secs = max(1e-9, a_state["t1"] - a_state["t0"])
        log_appends = {"calls": a_state["calls"], "payload_bytes": a_state["bytes"], "GB_per_s": a_state["bytes"] / secs / 1e9,
                       "status": a_state["rc"], "records_per_call": n_ref, "payload": payload,
                       "what": "rafting_log_append from a second host thread during the whole timed region (entry buffer's own stream)"}
    sampler.armed = False                   # clocks are sampled only while the GPU is under the timed load
    total_ms = ev0.elapsed_time(ev1)
    digest_b = e.digest(0, G)
    replay_ok = bool((digest_a == digest_b).all())
    if args.dump_outputs:                   # copied now: the passes below reuse the outbox buffers
        last = abi.Outbox(rows, G, F, G)
        for name, t in outs[(L - 1) % 2].t.items():
            getattr(last, name).view(np.uint8).reshape(-1)[:] = t.cpu().numpy()
        dump_outputs(args.dump_outputs, last, DUMP_BYTES // world, f"rank{rank}_" if world > 1 else "")

    # ---- the gathered vector of the timed region's LAST launch against the ranks' own commit columns ----
    gather_ok = None
    if world > 1:
        got = torch.from_numpy(e.allgather_last()).to(dev)
        mine = outs[(L - 1) % 2].t["commit_index"].view(torch.int64).clone()
        parts = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(parts, mine)                       # torch.distributed's own all-gather of the same column
        table = torch.from_numpy(np.array([s.commit_index for s in e.export_bulk(0, min(G, 4096))], dtype=np.int64)).to(dev)
        ok = bool(torch.equal(got, torch.cat(parts))) and bool(torch.equal(mine[:table.numel()], table)) and int(got.max().item()) > 0
        flag = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        gather_ok = bool(flag.item())

    # pass 2 — one window with an event pair around every kernel (roofline of the dominant kernel)
    warm()
    sampler.armed = True
    NK = min(L, 32)
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(2 * NK)]
    e.restore(sync=False)
    for j in range(NK):
        evs[2 * j].record(ext)
        e.step_device(ics[j], ocs[j], stream_ptr)
        evs[2 * j + 1].record(ext)
    torch.cuda.synchronize(); barrier()
    kern_ms = [evs[2 * j].elapsed_time(evs[2 * j + 1]) for j in range(NK)]
    sampler.armed = False

    # ---- e2e: the same stream through the C-ABI host path, HOST buffers in, HOST buffers out ---------
    e2e = None
    e2e_dense = None
    e2e_frames = None
    lat_ms = []
    if not args.no_e2e:
        from rafting_b200 import compact
        NSL = 4                                           # launches in flight on the host path (RAFTING_HOST_SLOTS)

        def pinned_like(a):
            t = torch.empty(a.nbytes, dtype=torch.uint8).pin_memory()
            v = t.numpy().view(a.dtype).reshape(a.shape)
            v[...] = a
            return t, v

        def host_inbox(k):                                # numpy views of launch k's recorded dense inbox
            ib = abi.Inbox(rows, G, F, with_ops=False, with_events=False)
            for name, dt, lane in (("op_meta", np.uint64, 0), ("op_nr", abi.I64X2, 0), ("ev_meta", np.uint64, 1), ("ev_tn", abi.I64X2, 1), ("ev_el", abi.I64X2, 1)):
                setattr(ib, name, inboxes[k].t[name].cpu().numpy().view(dt).reshape((rows, G, F) if lane else (rows, G)))
            ib.flags = abi.INBOX_NO_REQUESTS
            return ib

        # (A) the COMPACT host path (include/rafting_b200.h): narrow wire columns, the (epochAtSend, lastIndexAtSend) echo kept in HBM.
        # The transport's pinned receive buffers are filled before the clock starts, as the transport would have decoded
        # them.  Launch 0 of the window answers RPCs that were planned on the device path (no tags): it runs untimed,
        # every one of its acks an escape record, and the state right after it is the starting point of every timed pass.
        K2 = int(max(4, min(L, 25)))
        e.restore(); e.checkpoint()                       # (the in-flight table, created by the first compact call, joins the checkpoint)
        ESC_CAP = max(1 << 16, rows * G * F // 16)        # escape records a launch may produce before the dense fallback is needed
        cout0 = compact.CompactOutbox(rows, G, F, esc_cap=ESC_CAP)
        e.step_compact(compact.encode_inbox(host_inbox(0), None, None), cout0)
        e.checkpoint()
        tags, sent_term, sent_inc = cout0.tags(), cout0.current_term.copy(), cout0.incarnation.copy()
        cins, keep = [], []
        couts = []
        esc_out_max = 0
        # every launch's wire columns live in ONE pinned block per direction, laid out by rafting_compact_layout: one copy up,
        # one copy down per launch
        in_off0, out_off = engine.Engine.compact_layout(rows, G, F, 0, ESC_CAP)
        for sl in range(NSL):
            t = torch.zeros(int(out_off[11]), dtype=torch.uint8).pin_memory(); keep.append(t)
            couts.append(compact.outbox_in_block(t.numpy(), out_off, rows, G, F, ESC_CAP))
        for k in range(1, K2):                            # record pass (untimed): the tags the engine hands out are replayed below
            ci = compact.encode_inbox(host_inbox(k), tags, sent_term, sent_inc)
            in_off, _ = engine.Engine.compact_layout(rows, G, F, len(ci.esc), ESC_CAP)
            t = torch.zeros(int(in_off[5]), dtype=torch.uint8).pin_memory(); keep.append(t)
            ci = compact.inbox_in_block(t.numpy(), in_off, ci)
            e.step_compact(ci, couts[0])
            esc_out_max = max(esc_out_max, int(couts[0].counts[0]))
            tags, sent_term, sent_inc = couts[0].tags(), couts[0].current_term.copy(), couts[0].incarnation.copy()
            cins.append(ci)
        digest_c = e.digest(0, G)
        cin_c = [ci.as_c() for ci in cins]
        cout_c = [co.as_c() for co in couts]
        # bytes that actually cross PCIe per launch: the single copy up (row_base .. ev_c, or .. the escape records) and the single
        # copy down (plan_c .. counters + the 256 escape records that always travel with them), alignment padding included
        h2d = int(np.mean([(in_off0[4] + len(ci.esc) * abi.CESC_IN.itemsize) if len(ci.esc) else (in_off0[3] + ci.ev_c.nbytes) for ci in cins]))   # in_off: row_base, op_c, op_unavail, ev_c, esc, total
        d2h = int(out_off[10] + min(ESC_CAP, 256) * abi.CESC_OUT.itemsize)
        esc_in = int(np.mean([len(ci.esc) for ci in cins]))
        acks_pass = sum(acks_per_launch[1:K2])
        n_pass_launch = K2 - 1

        def compact_pass():
            for j in range(n_pass_launch):
                sl = j % NSL
                if j >= NSL:
                    e.step_wait_compact(sl)               # outbox of launch j-NSL is readable on the host
                e.step_begin_compact(sl, cin_c[j], cout_c[sl])
            for sl in range(NSL):
                e.step_wait_compact(sl)

        e.restore(); compact_pass()                       # untimed: every slot's device staging exists before the clock starts
        e2e_exact = bool((e.digest(0, G) == digest_c).all())
        reps = int(max(2, min(40, 0.15 / (0.8e-3 * (G / 65536) * n_pass_launch) + 1)))
        barrier()
        sampler.armed = True
        t0 = time.perf_counter()
        for _ in range(reps):
            e.restore(sync=False)
            compact_pass()
        spent = time.perf_counter() - t0
        sampler.armed = False
        # latency: one launch at a time, host ack in -> commit record readable out
        e.restore()
        for j in range(min(n_pass_launch, 12)):
            t1 = time.perf_counter()
            e.step_begin_compact(0, cin_c[j], cout_c[0])
            e.step_wait_compact(0)
            lat_ms.append((time.perf_counter() - t1) * 1e3)
        # the device path over the same launches ends in the same state
        e.restore()
        e.step_device_seq((abi.InboxC * n_pass_launch)(*[inboxes[k].as_c() for k in range(1, K2)]),
                          (abi.OutboxC * n_pass_launch)(*[outs[k % 2].as_c() for k in range(1, K2)]), n_pass_launch, gather=False, stream=0)
        torch.cuda.synchronize()
        e2e_exact = e2e_exact and bool((e.digest(0, G) == digest_c).all())
        t = torch.tensor([spent], dtype=torch.float64, device=dev)
        ae = torch.tensor([float(acks_pass * reps)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(ae, op=dist.ReduceOp.SUM)
        if esc_out_max > ESC_CAP:
            raise SystemExit(f"bench.py: a launch produced {esc_out_max} escape records (> {ESC_CAP}): the compact e2e number would need the dense fallback")
        e2e = {"spent": float(t.item()), "h2d": h2d, "d2h": d2h, "acks": float(ae.item()), "launches": n_pass_launch * reps,
               "launches_per_pass": n_pass_launch, "passes": reps, "exact": e2e_exact, "esc_in": esc_in, "esc_out_max": esc_out_max}

        # (A') the same launches arriving as FRAMES (SURVEY §8(f)-2, include/rafting_ingest.h): each launch's wire columns sit in ONE
        # pinned receive buffer as frames of the reference's layout |SOH|TYPE|STX|HEAD_LEN|HEAD|BODY_LEN|BODY|ETX| (type 0x1A, head =
        # column name); the timed loop cuts the buffer with rafting_frame_scan and hands the body addresses to the engine
        e2e_frames = None
        if world == 1:
            from rafting_b200 import ingest
            IL = ingest.lib()
            rx = []
            for ci in cins:
                blob = b"".join(ingest.encode(ingest.BATCH, name.encode(), getattr(ci, name).tobytes())
                                for name in ("row_base", "op_c", "ev_c", "esc") if getattr(ci, name) is not None and len(getattr(ci, name)))
                tt = torch.frombuffer(bytearray(blob), dtype=torch.uint8).pin_memory()
                rx.append((tt, tt.data_ptr(), len(blob)))
            frames = np.zeros(8, dtype=ingest.FRAME)
            nfr, used, transparent = C.c_uint32(), C.c_size_t(), C.c_int()
            cinf = [abi.CInboxC() for _ in range(NSL)]

            def frame_pass():
                for j in range(n_pass_launch):
                    sl = j % NSL
                    if j >= NSL:
                        e.step_wait_compact(sl)
                    _, base, ln = rx[j]
                    if IL.rafting_frame_scan(base, ln, frames.ctypes.data, 8, C.byref(nfr), C.byref(used), C.byref(transparent)) or used.value != ln:
                        raise RuntimeError("frame scan failed")
                    ci = cinf[sl]
                    ci.rows, ci.n_esc, ci.op_c, ci.ev_c, ci.esc, ci.op_unavail = rows, 0, None, None, None, None
                    for fr in frames[:nfr.value]:
                        head = tt_bytes(base + int(fr["head_off"]), int(fr["head_len"]))
                        addr = base + int(fr["body_off"])
                        if head == b"row_base":
                            ci.row_base = addr
                        elif head == b"op_c":
                            ci.op_c = addr
                        elif head == b"ev_c":
                            ci.ev_c = addr
                        elif head == b"esc":
                            ci.esc, ci.n_esc = addr, int(fr["body_len"]) // abi.CESC_IN.itemsize
                    e.step_begin_compact(sl, ci, cout_c[sl])
                for sl in range(NSL):
                    e.step_wait_compact(sl)

            def tt_bytes(addr, n):
                return C.string_at(addr, n)

            e.restore(); frame_pass()
            frames_exact = bool((e.digest(0, G) == digest_c).all())
            t0 = time.perf_counter()
            for _ in range(reps):
                e.restore(sync=False)
                frame_pass()
            fspent = time.perf_counter() - t0
            e2e_frames = {"value": acks_pass * reps / fspent, "unit": "acks/s", "launches": n_pass_launch * reps,
                          "rx_bytes_per_launch": int(np.mean([r[2] for r in rx])), "same_end_state_as_device_path": frames_exact,
                          "what": "the compact launches as frames of the reference's wire layout in one pinned receive buffer per launch; "
                                  "rafting_frame_scan + pointer hand-over inside the timed loop"}
            del rx
        del cins, keep, couts

        # (B) the DENSE host path of round 1 on a few launches of the same window, for the before / after of the byte cut
        if world == 1:
            K3 = int(max(3, min(L, 6)))
            host_in = []
            for k in range(K3):
                cols = {name: t.cpu().pin_memory() for name, t in inboxes[k].t.items()}
                ic = abi.InboxC()
                ic.rows, ic.n_active, ic.flags = rows, 0, abi.INBOX_NO_REQUESTS
                for name, t in cols.items():
                    setattr(ic, name, t.data_ptr())
                host_in.append((cols, ic))
            host_out = []
            for sl in range(NSL):
                cols = {name: torch.zeros(t.numel(), dtype=torch.uint8).pin_memory() for name, t in outs[0].t.items()}
                oc = abi.OutboxC()
                for name, t in cols.items():
                    setattr(oc, name, t.data_ptr())
                host_out.append((cols, oc))
            sparse = ("rep_term", "ballot_term", "ballot_last")
            dh2d = sum(t.numel() for t in host_in[0][0].values())
            dd2h = sum(t.numel() for name, t in host_out[0][0].items() if name not in sparse) + 16

            def dense_pass():
                for j in range(K3):
                    sl = j % NSL
                    if j >= NSL:
                        e.step_wait_slot(sl)
                    e.step_begin_host(sl, host_in[j][1], host_out[sl][1])
                for sl in range(NSL):
                    e.step_wait_slot(sl)
            e.restore(); dense_pass()
            t0 = time.perf_counter()
            for _ in range(6):
                e.restore(sync=False); dense_pass()
            dspent = time.perf_counter() - t0
            e2e_dense = {"value": sum(acks_per_launch[:K3]) * 6 / dspent, "unit": "acks/s", "h2d_bytes_per_launch": int(dh2d),
                         "d2h_bytes_per_launch": int(dd2h), "launches": 6 * K3}
            del host_in, host_out
    sampler.stop_flag = True

    # ---- reduce over ranks ------------------------------------------------------------------------
    tt = torch.tensor([total_ms, float(np.mean(kern_ms))], dtype=torch.float64, device=dev)
    aa = torch.tensor([float(acks_window * K)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(aa, op=dist.ReduceOp.SUM)
    total_ms_max, kern_ms_max = float(tt[0].item()), float(tt[1].item())
    acks_all = float(aa.item())

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        os.sched_setaffinity(0, all_cpus)                   # the CPU leg may use every host core, not just the GPU's node
        cores = len(all_cpus)
        cpu = run_cpu_sample(args, threads=cores, steps=args.cpu_steps, warmup=1, launches=args.cpu_launches, seed=seed)
        cpu3 = run_cpu_sample(args, threads=3, steps=2, warmup=1, launches=2, seed=seed)
        cpu["cores"] = cores; cpu["t3"] = cpu3["value"]

    # SURVEY §8(d): vote replies (config #3) and follower-side AppendEntries requests (config #5) are separate rates,
    # device-resident at full size; reported next to the headline, not part of `value`
    secondary = None
    if rank == 0 and world == 1 and not args.no_secondary and not args.no_e2e:
        del inboxes, ics
        torch.cuda.empty_cache()
        import importlib.util
        spec = importlib.util.spec_from_file_location("bench_secondary", os.path.join(ROOT, "tools", "bench_secondary.py"))
        mod = importlib.util.module_from_spec(spec); spec.loader.exec_module(mod)
        secondary = []
        for r in mod.run_all(quiet=True, steps5=64):
            secondary.append({"config": r["config"], "groups": r["groups"], "replicas": r["replicas"], "rows_per_step": r["rows_per_step"],
                              "steps": r["steps"], "kernel_ms_per_step": r["kernel_ms_per_step_median"],
                              "rates_per_s": r["rates_per_s"], "roofline_frac": r["roofline"]["frac"]})

    if rank == 0:
        peak, peak_src = measured_peak()
        launches = K * L
        acks_launch = acks_window / L
        # dominant kernel's launch duration: at N=1 the timed region holds the K*L step kernels and K table roll-backs
        # (22 MB device copies), so region time / launches is the (slightly pessimistic) unperturbed figure; with N>1 the
        # region also holds the gathers, so the per-kernel event pairs of pass 2 are used
        k_ms = total_ms / launches if world == 1 else float(np.mean(kern_ms))
        achieved = acks_launch * b_ack(R) / (k_ms * 1e-3) / 1e9
        traffic, traffic_src = measured_traffic(G, R, rows)
        value = acks_all / (total_ms_max * 1e-3)
        cfgd = workload_config(args, world, G)
        run = {
            "acks_per_launch_per_gpu": acks_launch,
            "inputs": f"each launch reads its own pre-generated inbox resident in HBM ({inbox_bytes / 1e6:.0f} MB inbox + "
                      f"{outbox_bytes / 1e6:.0f} MB outbox per launch, window {L * inbox_bytes / 1e9:.1f} GB >> L2), no L2 flush needed",
            "collective": ("ncclAllGather of commitIndex[G/N] after every launch, source = the launch's outbox commit column, on its "
                           "own stream; the step stream waits for the gather issued one launch earlier") if world > 1 else "none (1 GPU)",
            "bit_exact_replay": replay_ok, "host_placement": placement}
        if log_appends is not None:
            run["log_appends"] = log_appends
        if world > 1:
            cfgd["gather_verified"] = gather_ok            # SURVEY §8(d) #4's pass criterion, checked on every rank
        line = {
            "metric": METRIC, "value": value, "unit": "acks/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": total_ms_max / K,
            "higher_is_better": True, "scaling": "weak" if world == 1 else "strong", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": cfgd, "run": run,
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "bytes_per_ack": b_ack(R), "algorithmic_bytes_per_launch": acks_launch * b_ack(R),
                         "kernel_ms": k_ms, "kernel_ms_event_pair_per_launch": float(np.mean(kern_ms)),
                         "kernel": "rafting::unrolled::step_kernel<FT=R-1,NST=3>"},
            "clocks": sampler.summary(),
            "timed_region_ms": total_ms_max,
        }
        if e2e:
            ev = e2e["acks"] / e2e["spent"]
            line["e2e"] = {"value": ev, "unit": "acks/s", "h2d_bytes_per_step": e2e["h2d"] * L, "d2h_bytes_per_step": e2e["d2h"] * L,
                           "h2d_bytes_per_launch": e2e["h2d"], "d2h_bytes_per_launch": e2e["d2h"],
                           "h2d_bytes_per_ack": e2e["h2d"] / acks_launch, "d2h_bytes_per_ack": e2e["d2h"] / acks_launch,
                           "launches": e2e["launches"], "timed_region_ms": e2e["spent"] * 1e3, "same_end_state_as_device_path": e2e["exact"],
                           "escape_records_per_launch_up": e2e["esc_in"], "escape_records_per_launch_down_max": e2e["esc_out_max"],
                           "path": "compact (rafting_step_begin_compact / rafting_step_wait_compact)",
                           "note": "wall clock around the compact host path with caller-owned pinned buffers, three launches in flight (H2D / "
                                   "unpack + step + pack kernels / D2H of successive launches overlap); every launch's wire columns cross PCIe up "
                                   "and down inside the timed region; lossless: the end state equals the device path's, bit for bit; "
                                   "bytes_per_step = per launch x the launches of one step"}
            if e2e_dense:
                line["e2e_dense_path"] = e2e_dense
            if e2e_frames:
                line["e2e_from_frames"] = e2e_frames
            line["commit_latency_ms"] = {"p50": float(np.percentile(lat_ms, 50)), "p99": float(np.percentile(lat_ms, 99)),
                                         "what": "one synchronous launch: host ack in pinned inbox -> commit record readable in pinned outbox"}
        if cpu:
            line["cpu_baseline"] = {"value": cpu["value"], "unit": "acks/s", "cores": cpu["cores"], "kind": "port",
                                    "sample": cpu["sample"], "median_step_rate": cpu["median_rate"], "min_step_rate": cpu["min_rate"],
                                    "max_step_rate": cpu["max_rate"], "t3_loop_threads_value": cpu["t3"]}
        if secondary:
            line["secondary_rates"] = secondary
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# --dump-outputs: what the timed path hands its caller, so that two builds can be compared output for output
# ------------------------------------------------------------------------------------------------
DUMP_BYTES, DUMP_SEED = 60 << 20, 0x5EED00D0       # array bytes; with the .npy headers the files stay under 64 MB


def as_float64(a):
    """A column as float64 without loss: (x, y) pairs and the bit-packed 64-bit meta words (as 32-bit halves, low
    first) gain a last axis of 2; terms, indices and clocks are converted whole and checked to round-trip."""
    from rafting_b200 import abi
    if a.dtype == abi.I64X2:
        a = np.stack([a["x"], a["y"]], axis=-1)
    elif a.dtype == np.uint64:
        a = np.stack([a & np.uint64(0xFFFFFFFF), a >> np.uint64(32)], axis=-1)
    f = a.astype(np.float64)
    if not np.array_equal(f.astype(a.dtype), a):
        raise SystemExit("bench.py --dump-outputs: an output value has no exact float64 form")
    return f


def dump_outputs(out_dir, ob, budget=DUMP_BYTES, prefix=""):
    """Writes the host outbox `ob` as <out_dir>/<prefix><column>.npy for a sample of groups drawn with a fixed seed (all
    groups when they fit `budget`); <prefix>gids.npy lists them.  Row columns are [rows, groups(, F)(, 2)], group columns
    [groups(, 2)].  Payload slots that their meta column marks empty are written as 0: the engine leaves them
    unwritten, so their bytes are not part of what it computed."""
    masks = ob.payload_masks()

    def columns(gids):
        for name, _, _ in ob.ROW_COLS:
            col = getattr(ob, name)[:, gids]
            if name in masks:
                col[~masks[name][:, gids]] = 0
            yield name, as_float64(col)
        for name, _ in ob.GROUP_COLS:
            yield name, as_float64(getattr(ob, name)[gids])

    per_group = 8 + sum(a.nbytes for _, a in columns(np.arange(1)))
    n = min(ob.n, budget // per_group)
    gids = np.arange(ob.n) if n == ob.n else np.sort(np.random.default_rng(DUMP_SEED).choice(ob.n, n, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, prefix + "gids.npy"), gids.astype(np.float64))
    for name, a in columns(gids):
        np.save(os.path.join(out_dir, prefix + name + ".npy"), a)


_REAL_STDOUT = None


def emit(line: dict):
    """The one JSON line, on the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    # stdout carries exactly one JSON line: anything libraries print on fd 1 while the bench runs (NCCL prints its
    # version banner there) is diverted to stderr
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_engine(args)


if __name__ == "__main__":
    main()
