#!/usr/bin/env python
"""bench.py -- committed entries/sec across N Raft groups; HBM GB/s vs roofline.

One "step" = one pass of the hot path (one raft_step launch) over every member row of the
workload: all RPC records sent in the previous step are evaluated, every leader appends
`cmds` client commands, every follower handles its AppendEntries / written events, quorum
is evaluated, replies and new AppendEntries are emitted for the next step.

 value      committed entries/s (sum of commit_index advances on leaders / device time), inputs
            (mailboxes, log views, SoA) resident in HBM: ra_engine_flood, CUDA events on the
            engine's stream, max over ranks.
 e2e        the same flood driven through the public C ABI (ra_engine_step with pinned HOST
            buffers; H2D of the step's events and D2H of its notes inside every step).
 roofline   algorithmic bytes (SURVEY.md §8d: B_commit(5) = 2884 B, B_commit(7) = 4282 B per
            committed entry) / duration of the raft_step launches / measured HBM peak.
 cpu_baseline  the CPU restatement of ra_server (oracle/, kind "port": the reference is Erlang
            and no OTP toolchain exists on the box) on a bounded sample of the same workload.

 --impl reference times that CPU port with all host threads (see DESIGN.md "reference arm").
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B_COMMIT = {3: 40 + 104 * 3 + 2 * (169 + 185) + (128 + 8 * 3) + 2 * (145 + 8 * 3),
            5: 2884, 7: 4282}
METRIC = "committed entries/sec across N Raft groups; HBM GB/s vs roofline"
# dram__bytes_read.sum + dram__bytes_write.sum of raft_step_kernel per launch: read from the committed ncu summary
# of the shipped build (tools/ncu_summary.py output of one `ncu --set full` capture of this workload)
TRAFFIC_FILE = os.path.join(ROOT, "profiles", "r02_raft_step_ncu_full.txt")


def traffic_bytes():
    """-> (bytes per launch or None, source)"""
    try:
        rd = wr = None
        for ln in open(TRAFFIC_FILE):
            f = ln.split()
            if len(f) >= 3 and f[0] == "dram__bytes_read.sum":
                rd = float(f[1]) * {"[Mbyte]": 1e6, "[Gbyte]": 1e9, "[Kbyte]": 1e3, "[byte]": 1.0}[f[2]]
            if len(f) >= 3 and f[0] == "dram__bytes_write.sum":
                wr = float(f[1]) * {"[Mbyte]": 1e6, "[Gbyte]": 1e9, "[Kbyte]": 1e3, "[byte]": 1.0}[f[2]]
        if rd is not None and wr is not None:
            return int(rd + wr), os.path.relpath(TRAFFIC_FILE, ROOT)
    except (OSError, KeyError, ValueError):
        pass
    return None, "no ncu summary found"


DUMP_BYTES = 64 * 10**6      # --dump-outputs: ceiling on what one dump writes, .npy headers included
DUMP_SEED = 0xD0             # the fixed row sample of --dump-outputs when all rows would not fit in DUMP_BYTES


def dump_outputs(out_dir: str, eng) -> dict:
    """What the flood leaves its caller, as float64 arrays out_dir/<name>.npy:

    counters.npy  the ra_counters fields in include/ra_engine.h order, totals over the whole run
    row.npy       the rows dumped: all of them, or a fixed sample (seed DUMP_SEED) when all would pass DUMP_BYTES
    <field>.npy   each ra_row_state field of those rows, shape (rows,) or (rows, k); the peers' fields as
                  peer_<field>.npy, one column per member.  Entries RaRowState.key() does not compare (runs past
                  n_runs, peers past n_members, the cond_reply_* fields while flags bit 1 is clear) are zero, so
                  two builds compare the way the parity diff does.
    Every value is an integer below 2^53 (checked), so float64 holds it exactly."""
    import numpy as np
    from ra_b200 import abi
    dt = np.dtype(abi.RaRowState)
    peer_fields = [f for f in dt["peers"].base.names if not f.startswith("_")]
    n, m = eng.n_rows, eng.n_members
    cols = sum(int(np.prod(dt[f].shape)) for f in dt.names if f != "peers") + len(peer_fields) * m
    k = min(n, (DUMP_BYTES - 2**20) // (8 * cols))       # 1 MiB left for the counters and the .npy headers
    ids = np.arange(n) if k == n else np.sort(np.random.default_rng(DUMP_SEED).choice(n, k, replace=False))
    rows = np.frombuffer(b"".join(bytes(r) for r in eng.read_rows(ids.tolist())), dtype=dt)
    out = {"counters": np.array(list(eng.counters().values()), dtype=np.uint64)}
    out.update((f, rows[f]) for f in dt.names if f != "peers")
    run_live = np.arange(abi.RA_MAX_RUNS) < rows["n_runs"][:, None]
    for f in ("run_start", "run_term"):
        out[f] = np.where(run_live, rows[f], 0)
    cond_live = (rows["flags"] & 2) != 0
    for f in ("cond_reply_term", "cond_reply_next_index", "cond_reply_last_index", "cond_reply_last_term"):
        out[f] = np.where(cond_live, rows[f], 0)
    peer_live = np.arange(m) < rows["n_members"][:, None]
    for f in peer_fields:
        out["peer_" + f] = np.where(peer_live, rows["peers"][f][:, :m], 0)
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, a in out.items():
        if a.size and int(a.max()) >= 2**53:
            raise ValueError("--dump-outputs: %s holds %d, which float64 cannot hold exactly" % (name, int(a.max())))
        path = os.path.join(out_dir, name + ".npy")
        np.save(path, a.astype(np.float64))
        total += os.path.getsize(path)
    return {"dir": out_dir, "rows": int(k), "of_rows": n, "sample_seed": None if k == n else DUMP_SEED,
            "files": len(out), "bytes": total}


def b_commit(m: int) -> int:
    return (40 + 104 * m) + (m - 1) * (169 + 185) + (128 + 8 * m) + (m - 1) * (145 + 8 * m)


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region.

    Primary source: NVML polled from a thread (~500 Hz, so a 20 ms region still gets samples);
    secondary: an `nvidia-smi -lms` child (its first line can take longer than the region)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    MASKS = (("sw_power_cap", 0x4), ("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40))

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.lines = []
        self.nv = []            # (sm_mhz, max_mhz, reasons bitmask)
        self._stop = threading.Event()
        self._nvt = None
        self._nvml = None       # (module, handle, max clock, reasons fn): set up BEFORE the timed region
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            try:
                import torch
                uuid = getattr(torch.cuda.get_device_properties(self.idx), "uuid", None)
                if uuid is not None:
                    u = "GPU-" + str(uuid)
                    try:
                        h = pynvml.nvmlDeviceGetHandleByUUID(u)
                    except Exception:
                        h = pynvml.nvmlDeviceGetHandleByUUID(u.encode())
            except Exception:
                h = None
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.idx)
            mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            fn = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                getattr(pynvml, "nvmlDeviceGetCurrentClocksThrottleReasons")
            pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)          # make sure the query works
            self._nvml = (pynvml, h, float(mx), fn)
        except Exception:
            self._nvml = None

    def _nvml_loop(self):
        try:
            pynvml, h, mx, reasons_fn = self._nvml
            while not self._stop.is_set():
                sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                try:
                    rs = int(reasons_fn(h))
                except Exception:
                    rs = 0
                self.nv.append((float(sm), mx, rs))
                time.sleep(0.002)          # ~500 Hz: plenty for a 20 ms region, negligible GIL pressure
        except Exception:
            return

    def start(self):
        try:
            if self._nvml is not None:
                self._nvt = threading.Thread(target=self._nvml_loop, daemon=True)
                self._nvt.start()
        except Exception:
            self._nvt = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self) -> dict:
        self._stop.set()                                       # NVML samples end with the timed region
        if self._nvt is not None:
            self._nvt.join(timeout=1.0)
        if self.nv:
            sm = sorted(x[0] for x in self.nv)
            bits = 0
            for x in self.nv:
                bits |= x[2]
            if self.proc:
                self.proc.terminate()
            return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(x[1] for x in self.nv),
                    "reasons": sorted(n for n, m in self.MASKS if bits & m), "samples": len(sm), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def dist_init(n_gpus: int):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local


def barrier_sync(world: int, local: int):
    import torch
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize(local)


def reduce_max_sum(world: int, local, ms: float, commits: float, events: float):
    """MAX of the per-rank time, SUM of the per-rank work (local=None: CPU tensors, gloo)."""
    if world == 1:
        return ms, commits, events
    import torch
    import torch.distributed as dist
    dev = "cpu" if local is None else "cuda:%d" % local
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    s = torch.tensor([commits, events], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dist.all_reduce(s, op=dist.ReduceOp.SUM)
    return float(t.item()), float(s[0].item()), float(s[1].item())


def run_engine(args):
    from ra_b200 import abi
    from ra_b200.engine import Engine, HostFlood
    import torch

    rank, world, local = dist_init(args.gpus)
    G, M = args.groups, args.members
    dev = local
    spread = world > 1 and args.placement == "spread"
    peer = False
    if spread:
        # members of a group on different GPUs; cross-shard RPC records by NCCL all-to-all
        from ra_b200.sharded import NcclTransport, NvlinkPeerTransport, Shard, ShardedFlood
        torch.cuda.set_device(dev)
        peer = args.transport == "peer" and world <= 8
        sh = Shard(G, M, world, rank, device=dev, buckets=not peer)
        eng = sh.eng
        fl = ShardedFlood(NvlinkPeerTransport(sh) if peer else NcclTransport(sh))
        fl.bootstrap()
        seed = args.seed                                         # one global host model
        flood = lambda n: fl.run(n, args.cmds, args.permille, seed, faults=args.faults)
    else:
        eng = Engine(G, M, device=dev, route_on_device=True)
        eng.reset_empty()
        eng.step([abi.ev_simple(eng.row_of(g, 0), abi.EV_ELECTION_TIMEOUT) for g in range(G)])
        seed = args.seed + rank
        flood = lambda n: eng.flood(n, args.cmds, args.permille, seed=seed, sync=False, faults=args.faults)
    flood(args.settle)                                           # elect leaders, fill the pipeline
    flood(args.warmup)                                           # W untimed warm-up steps
    torch.cuda.synchronize(dev)
    eng.sync()
    c0 = eng.counters()
    sampler = ClockSampler(dev)
    sampler.start()
    barrier_sync(world, local)
    if spread:
        # the engine runs on torch's current stream in this mode: time with torch CUDA events on it
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        flood(args.steps)
        t1.record()
        torch.cuda.synchronize(dev)
        ms, launches = t0.elapsed_time(t1), 3 * args.steps
    else:
        flood(args.steps)
        eng.sync()
        ms, launches = eng.last_kernel_ms()                      # CUDA events on the engine's stream
    barrier_sync(world, local)
    clocks = sampler.stop()
    c1 = eng.counters()
    dump = dump_outputs(args.dump_outputs, eng) if args.dump_outputs else None
    commits = c1["commits"] - c0["commits"]
    events = c1["events"] - c0["events"]
    dropped = c1["msgs_dropped"] - c0["msgs_dropped"]
    ms_max, commits_all, events_all = reduce_max_sum(world, local, ms, commits, events)
    value = commits_all / (ms_max * 1e-3)

    # parity of THIS run (the rows the timed region left): every `stride`-th global group is replayed by the CPU
    # oracle (checker only; groups are independent and the flood host model is keyed by global ids), and every
    # rank diffs the members of those groups that live on it, field by field
    parity = None
    if not args.no_parity:
        parity = parity_sample(args, eng, world, rank, spread, seed, args.settle + args.warmup + args.steps)
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([parity["rows_checked"], parity["rows_bad"]], dtype=torch.int64, device="cuda:%d" % local)
            dist.all_reduce(t)
            parity["rows_checked"], parity["rows_bad"] = int(t[0]), int(t[1])
        # the oracle replays a LOSSLESS transport: records dropped for capacity (counted, Raft tolerates them) make the
        # two runs legitimately different
        parity["msgs_dropped_in_run"] = int(c1["msgs_dropped"])

    # e2e: the same flood through ra_engine_step with pinned host buffers (rank-local engine)
    e2e = None
    if not args.no_e2e:
        # host-model threads: the CPUs this job may really use, shared by the ranks of the node
        os.environ.setdefault("RA_HOSTSIM_THREADS", str(max(1, min(16, effective_cpus() // max(1, world)))))
        if True:
            # K engines (disjoint sets of groups) driven by ONE host thread through the split-phase calls
            # ra_engine_submit_host / ra_engine_collect: while the notes of one partition travel device->host and
            # its host model runs, another partition's batch travels host->device and its kernels run.  Every
            # step of every partition still goes through the public C ABI with host buffers.
            K = max(1, min(args.e2e_engines, G))
            engs = [Engine(G // K + (1 if i < G % K else 0), M, device=dev, route_on_device=True) for i in range(K)]
            for e_ in engs:
                e_.reset_empty()
            hf = HostFlood(engs)
            hf.run(0, args.cmds, args.permille, seed=seed, bootstrap=True)

            def host_steps(n):
                return hf.run(n, args.cmds, args.permille, seed=seed)

            class _Multi:                                   # counters / close over all K engines
                def counters(self):
                    tot = {}
                    for e_ in engs:
                        for k_, v_ in e_.counters().items():
                            tot[k_] = tot.get(k_, 0) + v_
                    return tot
                def close(self):
                    for e_ in engs: e_.close()
            eng2 = _Multi()
        host_steps(args.settle)
        host_steps(min(args.warmup, 10))
        # three timed blocks of e2e_steps steps, the MEDIAN block is reported (a block is ~70 ms of wall time on 16
        # shared host cores: one scheduling hiccup would otherwise decide the number); all three are listed
        blocks = []
        for _b in range(3):
            d0 = eng2.counters()
            barrier_sync(world, local)
            st_b = host_steps(args.e2e_steps)
            barrier_sync(world, local)
            d1 = eng2.counters()
            sec_b, ec_b, _ = reduce_max_sum(world, local, st_b["seconds"], d1["commits"] - d0["commits"], 0)
            blocks.append((ec_b / sec_b, sec_b, ec_b, st_b))
        _, sec, ec, st = sorted(blocks, key=lambda b: b[0])[1]
        e2e = {"value": ec / sec, "unit": "commits/s",
               "blocks_commits_per_s": [round(b[0], 1) for b in blocks], "reported": "median of 3 blocks",
               "h2d_bytes_per_step": st["h2d_bytes"] // args.e2e_steps,
               "d2h_bytes_per_step": st["d2h_bytes"] // args.e2e_steps,
               "steps": args.e2e_steps, "ms_per_step": sec * 1e3 / args.e2e_steps,
               "engine_call_ms_per_step": st.get("step_seconds", 0.0) * 1e3 / args.e2e_steps,
               "host_model_ms_per_step": st.get("model_seconds", 0.0) * 1e3 / args.e2e_steps,
               "gpu_launches_per_step": 6 * max(1, min(args.e2e_engines, G)),
               "engines": max(1, min(args.e2e_engines, G)),
               "notes_format": ("16-byte units (ra_note16: one per note, extension entries for the rare note that does "
                                "not fit; decoded by the host model)" if os.environ.get("RA_HOSTSIM_COMPACT", "1") != "0"
                                else "32-byte ra_note records"),
               "placement": "every rank drives %d engines holding disjoint groups of its own (all members of a group on "
                            "one GPU, records routed on that GPU); no cross-rank traffic on this leg" % max(1, min(args.e2e_engines, G))}
        hf.close()
        eng2.close()

    latency = None
    if world == 1 and args.latency:
        try:
            latency = latency_probe(dev)
        except Exception as ex:
            latency = {"error": repr(ex)[:200]}
    extras = {}
    if args.extra_configs and args.config == 3:
        eng.close()
        ks = [2, 4, 5] if world == 1 else [4]
        for k in ks:
            try:
                extras["config%d" % k] = extra_config(k, world, rank, local)
            except Exception as ex:                      # an extra must never take the headline down with it
                extras["config%d" % k] = {"error": repr(ex)[:200]}
    if rank != 0:
        return
    peak, peak_src = hbm_peak()
    traffic, traffic_src = traffic_bytes()
    bc = b_commit(M)
    achieved = (commits / (ms * 1e-3)) * bc / 1e9               # this rank, GB/s
    par = ("members of a group on different GPUs ((group+slot) mod N); " +
           ("RPC records are stored by the step kernels straight into the destination GPU's mailbox planes "
            "over NVLink (CUDA IPC peer mappings); " +
            ("a device-side flag barrier over the same mappings closes every step (no collective, no host in the loop)"
             if os.environ.get("RA_PEER_BARRIER", "device") == "device" else
             "one 1-element NCCL all-reduce per step keeps the shards in lock step")
            if spread and peer else
            "cross-shard RPC records by NCCL all_to_all_single (bucket counts + equal-size buckets) every step")
           if spread else
           "groups sharded by rank, every member of a group on one GPU, no data-path collective")
    out = {
        "metric": METRIC, "value": value, "unit": "commits/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": workload_config(args),
        "run": {"parallelism": par, "placement": "spread" if spread else ("group" if world > 1 else "single GPU"),
                "events_per_step": events_all / args.steps, "commits_per_step": commits_all / args.steps,
                "msgs_dropped": dropped},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     # SURVEY 8d: also against the nominal HBM3e figure; and what the kernel really moves
                     "peak_nominal": 8000.0, "frac_nominal": achieved / 8000.0,
                     "achieved_traffic": (traffic / 1e9) / (ms * 1e-3 / args.steps) if (traffic and world == 1 and args.config == 3) else None,
                     "frac_traffic": ((traffic / 1e9) / (ms * 1e-3 / args.steps) / peak) if (traffic and world == 1 and args.config == 3) else None,
                     "bytes_per_commit": bc, "algorithmic_bytes_per_launch": bc * commits / args.steps,
                     "kernel": "raft_step_kernel (+ raft_general_kernel for the rows that leave the fast paths)"},
    }
    if parity:
        out["parity"] = parity
    if extras:
        out["configs"] = extras
    if latency:
        out["latency"] = latency
    if e2e:
        out["e2e"] = e2e
    if dump:
        out["dump"] = dump
    if world == 1 and not args.no_cpu:
        out["cpu_baseline"] = cpu_baseline(args, sample_groups=min(G, args.cpu_groups), steps=args.cpu_steps)
    print(json.dumps(out))


CONFIGS = {
    # BASELINE.json configs[1..4] as flood parameters (groups are per GPU unless "total")
    2: dict(groups=10_000, members=5, cmds=1, permille=0, faults=None,
            what="configs[1]: 10k groups x 5, steady-state AppendEntries, 1 entry/RPC (20 MB of state: L2-resident)"),
    3: dict(groups=100_000, members=5, cmds=1, permille=10, faults=None,
            what="configs[2]: 100k groups x 5, AppendEntries + 1 % election timeouts per step"),
    4: dict(groups=100_000, members=5, cmds=64, permille=10, faults=None, total=True,
            what="configs[3]: 100k groups x 5 IN TOTAL over the GPUs (strong scaling), 64-entry pipelined AppendEntries"),
    5: dict(groups=10_000, members=7, cmds=1, permille=0, faults=(5, 20, 10, 32),
            what="configs[4]: 10k groups x 7, 0.5 % AppendEntries lost, 2 % lagging fsync, 1 % of groups partitioned "
                 "per 32-step window (next_index back-off, term-conflict / truncate paths)"),
}


def extra_config(k: int, world: int, rank: int, local: int, steps: int = 100, warmup: int = 10, settle: int = 40) -> dict:
    """One more configuration on the device-resident flood path, timed like the headline (CUDA events, max over
    ranks).  Single GPU: one engine; N > 1 (config 4): members spread over the ranks, peer-store transport."""
    import torch
    from ra_b200 import abi
    from ra_b200.engine import Engine
    c = CONFIGS[k]
    G, M = c["groups"], c["members"]
    if world > 1:
        from ra_b200.sharded import NvlinkPeerTransport, Shard, ShardedFlood
        gl = G // world if c.get("total") else G
        sh = Shard(gl, M, world, rank, device=local, buckets=False)
        eng = sh.eng
        fl = ShardedFlood(NvlinkPeerTransport(sh))
        fl.bootstrap()
        flood = lambda n: fl.run(n, c["cmds"], c["permille"], 0xA00 + k, faults=c["faults"])
    else:
        gl = G
        eng = Engine(G, M, device=local, route_on_device=True)
        eng.reset_empty()
        eng.step([abi.ev_simple(eng.row_of(g, 0), abi.EV_ELECTION_TIMEOUT) for g in range(G)])
        flood = lambda n: eng.flood(n, c["cmds"], c["permille"], seed=0xA00 + k, sync=False, faults=c["faults"])
    flood(settle); flood(warmup)
    torch.cuda.synchronize(local); eng.sync()
    c0 = eng.counters()
    barrier_sync(world, local)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        t0.record(); flood(steps); t1.record()
        torch.cuda.synchronize(local)
        ms = t0.elapsed_time(t1)
    else:
        flood(steps); eng.sync()
        ms, _ = eng.last_kernel_ms()
    barrier_sync(world, local)
    c1 = eng.counters()
    ms_max, commits, events = reduce_max_sum(world, local, ms, c1["commits"] - c0["commits"], c1["events"] - c0["events"])
    out = {"what": c["what"], "groups_per_gpu": gl, "members": M, "cmds_per_step": c["cmds"], "election_permille": c["permille"],
           "faults": c["faults"], "value": commits / (ms_max * 1e-3), "unit": "commits/s", "ms_per_step": ms_max / steps,
           "steps": steps, "events_per_step": events / steps, "msgs_dropped": c1["msgs_dropped"] - c0["msgs_dropped"],
           "fatal_rows": c1["fatal_rows"], "scaling": "strong" if c.get("total") and world > 1 else "n/a"}
    if c["cmds"] == 1:
        out["roofline_frac"] = out["value"] / world * b_commit(M) / 1e9 / hbm_peak()[0]
    eng.close()
    return out


def latency_probe(dev: int, groups: int = 100_000, members: int = 5) -> dict:
    """Round trip of ONE ra_engine_step_host call (what a batching process pays per batch) on a 500k-row engine,
    for batches of 1 / 1k / 100k command events, host buffers pinned (ra_engine_alloc_host) and pageable.
    p50 / p99 over repeated calls; every call also evaluates what the previous calls left in the mailboxes."""
    import ctypes as C
    from ra_b200 import abi
    from ra_b200.engine import Engine, lib
    eng = Engine(groups, members, device=dev, route_on_device=True)
    eng.reset_empty()
    eng.step([abi.ev_simple(eng.row_of(g, 0), abi.EV_ELECTION_TIMEOUT) for g in range(groups)])
    eng.flood(40, 1, 0, seed=1)                      # leaders = slot 0 of every group (rows 0 .. groups-1)
    l = lib()
    f = l.ra_engine_step_host
    sz = C.c_size_t
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_void_p, sz, C.c_void_p, sz, C.POINTER(sz), C.c_void_p, sz, C.POINTER(sz)]
    l.ra_engine_alloc_host.restype = C.c_void_p
    l.ra_engine_alloc_host.argtypes = [sz]
    l.ra_engine_free_host.argtypes = [C.c_void_p]
    notes_cap, msgs_cap = groups * members * 3, 1024
    nm, nn = sz(0), sz(0)
    out = {}
    for kind in ("pinned", "pageable"):
        nbytes_ev, nbytes_n, nbytes_m = 100_000 * 32, notes_cap * 32, msgs_cap * 64
        if kind == "pinned":
            pev, pn, pm = (l.ra_engine_alloc_host(b) for b in (nbytes_ev, nbytes_n, nbytes_m))
            keep = None
        else:
            keep = [C.create_string_buffer(b) for b in (nbytes_ev, nbytes_n, nbytes_m)]
            pev, pn, pm = (C.addressof(k) for k in keep)
        evs = (abi.RaHostEvent * 100_000).from_address(pev)
        for i in range(100_000):
            evs[i].row = i; evs[i].type = abi.EV_COMMAND; evs[i].flags = 0; evs[i].n = 1
        for _ in range(6):                                # drain what the flood left in flight
            eng._check(f(eng._h, pev, 0, pm, msgs_cap, C.byref(nm), pn, notes_cap, C.byref(nn)), "step_host")
        for n, reps in ((1, 60), (1000, 60), (100_000, 15)):
            ts = []
            for _ in range(reps + 3):
                t0 = time.perf_counter()
                eng._check(f(eng._h, pev, n, pm, msgs_cap, C.byref(nm), pn, notes_cap, C.byref(nn)), "step_host")
                ts.append((time.perf_counter() - t0) * 1e3)
            ts = sorted(ts[3:])
            out["%s_%d" % (kind, n)] = {"p50_ms": ts[len(ts) // 2], "p99_ms": ts[min(len(ts) - 1, int(len(ts) * 0.99))],
                                       "notes_out": int(nn.value)}
        if kind == "pinned":
            for q in (pev, pn, pm):
                l.ra_engine_free_host(q)
    eng.close()
    out["how"] = ("one ra_engine_step_host call per sample: n COMMAND events to n leaders of a %d-row engine "
                  "(route_on_device), wall clock around the call" % (groups * members))
    return out


def workload_config(args) -> dict:
    """The `config` object of BOTH arms (engine and --impl reference): the workload, nothing measured."""
    G, M = args.groups, args.members
    return {"workload": "%d groups x %d members per GPU, steady-state AppendEntries flood, %d command(s) per leader per "
                        "step, %.1f%% election timeouts per step (BASELINE.json configs[%d])%s"
                        % (G, M, args.cmds, args.permille / 10.0, args.config - 1,
                           (", faults %s" % (args.faults,)) if args.faults else ""),
            "groups_per_gpu": G, "members": M, "cmds_per_step": args.cmds, "election_permille": args.permille,
            "l2": "working set (SoA %.0f MB + mailboxes) %s the 126 MB L2; no explicit flush"
                  % (G * M * 392 / 1e6, "exceeds" if G * M * 392 > 126e6 else "fits in")}


def parity_sample(args, eng, world: int, rank: int, spread: bool, seed: int, flood_steps: int, stride: int = 97) -> dict:
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_lib import Oracle
    from ra_b200 import abi
    G, M = args.groups, args.members
    total = G * world if spread else G                      # groups of the global run this rank belongs to
    n = (total + stride - 1) // stride
    while n > 1 and (n - 1) * stride >= total:
        n -= 1
    o = Oracle(n, M, route_on_device=True)
    o.set_sample(stride, 0, total)
    o.reset_empty()
    o.step([abi.ev_simple(o.row_of(g, 0), abi.EV_ELECTION_TIMEOUT) for g in range(n)])
    o.flood(flood_steps, args.cmds, args.permille, seed=seed, threads=max(1, min(8, effective_cpus() // max(1, world))),
            faults=args.faults)
    want = o.read_rows(range(o.n_rows))
    ids, exp = [], []
    for i in range(n):
        gg = i * stride
        for s in range(M):
            if spread:
                if (gg + s) % world != rank:
                    continue
                ids.append(s * G + gg // world)
            else:
                ids.append(s * G + gg)
            exp.append(want[s * n + i])
    got = eng.read_rows(ids)
    bad = sum(1 for a, b in zip(got, exp) if a.key()[1:] != b.key()[1:])
    o.close()
    return {"rows_checked": len(ids), "rows_bad": bad, "stride": stride,
            "how": "every %d-th global group replayed by the CPU oracle for all %d steps of this run; each rank "
                   "diffs its members of those groups (all ra_row_state fields)" % (stride, flood_steps + 1)}


def effective_cpus() -> int:
    """Host cores this process may actually use: min(online CPUs, affinity mask, cgroup CPU quota)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, -(-int(txt[0]) // int(txt[1]))))
            else:
                q = int(txt[0])
                per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if q > 0:
                    n = min(n, max(1, -(-q // per)))
            break
        except (OSError, ValueError, IndexError):
            continue
    return max(1, n)


def cpu_model() -> str:
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def cpu_baseline(args, sample_groups: int, steps: int, threads: int | None = None, min_seconds: float = 2.0) -> dict:
    """The oracle (CPU port of ra_server's hot path) on the same workload: all host cores, then one core.

    The timed region is whole floods of `chunk` steps repeated until it is at least `min_seconds` long, after a
    warm-up flood (thread start-up, page faults and the first growth steps of the log arrays happen before it),
    so the figure does not depend on the step count asked for."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_lib import Oracle
    from ra_b200 import abi
    cores = threads or effective_cpus()
    o = Oracle(sample_groups, args.members, route_on_device=True)
    o.reset_empty()
    o.step([abi.ev_simple(o.row_of(g, 0), abi.EV_ELECTION_TIMEOUT) for g in range(sample_groups)])
    o.flood(args.settle, args.cmds, args.permille, seed=args.seed, threads=cores, faults=args.faults)
    chunk = max(5, min(20, steps))
    o.flood(chunk, args.cmds, args.permille, seed=args.seed, threads=cores, faults=args.faults)      # warm-up
    c0 = o.counters()
    t0 = time.perf_counter()
    done = 0
    while True:
        o.flood(chunk, args.cmds, args.permille, seed=args.seed, threads=cores, faults=args.faults)
        done += chunk
        dt = time.perf_counter() - t0
        if dt >= min_seconds or done >= 2000:
            break
    c1 = o.counters()
    # one core, same rows (a few steps are enough: ~10x slower per step)
    s1 = max(2, min(5, chunk // 4))
    t1 = time.perf_counter()
    o.flood(s1, args.cmds, args.permille, seed=args.seed, threads=1, faults=args.faults)
    dt1 = time.perf_counter() - t1
    c2 = o.counters()
    o.close()
    return {"value": (c1["commits"] - c0["commits"]) / dt, "unit": "commits/s", "cores": cores, "kind": "port",
            "cpu_model": cpu_model(),
            "sample": "%d groups x %d members (the full workload), %d steps of the same flood in %.1f s after a "
                      "warm-up flood; C restatement of ra_server.erl, not BEAM" % (sample_groups, args.members, done, dt),
            "seconds": dt, "ms_per_step": dt * 1e3 / done, "steps": done,
            "one_core": {"value": (c2["commits"] - c1["commits"]) / dt1, "unit": "commits/s", "steps": s1, "seconds": dt1}}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    G, M = args.groups, args.members
    # the full workload (cpu_groups caps it for small hosts); whole floods repeated for >= 2 s, see cpu_baseline
    sg = min(G, args.cpu_groups)
    cb = cpu_baseline(args, sample_groups=sg, steps=args.steps)
    out = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "commits/s",
           "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"],
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
           "config": workload_config(args),
           "run": {"groups": sg, "threads": cb["cores"], "steps_timed": cb["steps"], "seconds": cb["seconds"]},
           "cpu_baseline": cb,
           "e2e": {"value": cb["value"], "unit": "commits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--groups", type=int, default=100_000, help="groups per GPU")
    ap.add_argument("--members", type=int, default=5)
    ap.add_argument("--cmds", type=int, default=1)
    ap.add_argument("--permille", type=int, default=10, help="election timeouts per step per 1000 groups")
    ap.add_argument("--settle", type=int, default=40, help="untimed steps to elect leaders and fill the pipeline")
    ap.add_argument("--seed", type=int, default=0xA00)
    ap.add_argument("--e2e-steps", type=int, default=100)
    ap.add_argument("--e2e-engines", type=int, default=4,
                    help="e2e leg at N=1: partitions (engines holding disjoint groups) one host thread pipelines "
                         "through ra_engine_submit_host / ra_engine_collect")
    ap.add_argument("--cpu-groups", type=int, default=100_000, help="groups of the CPU legs (default: the full workload)")
    ap.add_argument("--cpu-steps", type=int, default=300)
    ap.add_argument("--placement", default="spread", choices=["spread", "group"],
                    help="N>1: spread = members of a group on different GPUs + NCCL all-to-all of RPC records; "
                         "group = whole groups per GPU, no collective")
    ap.add_argument("--transport", default="peer", choices=["peer", "a2a"],
                    help="spread placement: peer = NVLink peer stores from inside the step kernels; "
                         "a2a = per-destination buckets + NCCL all_to_all_single + deliver kernel")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--config", type=int, default=3, choices=[2, 3, 4, 5],
                    help="BASELINE.json configs[config-1] as the headline workload (default 3 = configs[2])")
    ap.add_argument("--no-extra-configs", dest="extra_configs", action="store_false",
                    help="skip the keyed entries for the other configs (N=1: 2, 4, 5; N>1: 4 strong-scaled)")
    ap.add_argument("--no-latency", dest="latency", action="store_false", help="skip the per-call latency probe (N=1)")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle replay of every 97th group of this run")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the engine's counters and rows as DIR/<name>.npy (float64, "
                         "at most 64 MB: a fixed sample of the rows when all would not fit); one process only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "engine" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs needs --impl engine in one process")
    args.faults = None
    if args.config != 3:
        c = CONFIGS[args.config]
        args.groups, args.members, args.cmds, args.permille, args.faults = c["groups"], c["members"], c["cmds"], c["permille"], c["faults"]
        if c.get("total"):
            args.groups = c["groups"] // max(1, int(os.environ.get("WORLD_SIZE", "1")))
    if args.warmup < 3:
        args.warmup = 3
    try:
        if args.impl == "reference":
            run_reference(args)
        else:
            run_engine(args)
    finally:
        sys.stdout.flush()
        try:                                   # no "destroy_process_group() was not called" noise after the JSON line
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized():
                dist.destroy_process_group()
        except Exception:
            pass


if __name__ == "__main__":
    main()
