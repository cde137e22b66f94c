#!/usr/bin/env python
"""bench.py -- commit-index recomputes/s on synthetic AppendResponse streams.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # CPU baseline arm (the oracle port)
    python bench.py --workload cfg4|cfg5 ...                 # the other BASELINE.json configs

One "step" = one pass of the hot path over one batch: apply ONE round of synthetic
AppendResponses (about 3.5 records per group, SURVEY 8(d)) to a 1M-group x 5-peer arena and
recompute the commit index of every group (Raft::maybe_commit).

  value            groups recomputed per second over all GPUs, records already resident in HBM
                   (fused tile kernel, one launch per step; CUDA events on the launching stream)
  e2e              the same step through the reference-facing C-ABI from what the reference's
                   handle_append_response consumes: 24-byte records (raftgpu_append_resp) in pinned
                   HOST memory -> raftgpu_step_begin_records (the library's staging threads pack
                   them into the compact stream, H2D) -> kernels -> raftgpu_step_wait (D2H of the
                   advanced bitmap + new commit indexes).  Everything after the records exist is
                   inside the timed region.  This is the number to hold against the reference arm.
  e2e_prepacked    the step for a caller that already holds its batch as the compact stream
                   (raftgpu_step_begin_compact): the pack is NOT timed -- PCIe-bound floor
  e2e_wire         the step from serialized eraftpb.Message bytes (raftgpu_step_begin_wire)
  recompute_only   Raft::maybe_commit alone (BASELINE.md 3: rate x 74 B), back-to-back passes
  scatter          the general two-kernel path (scatter apply + recompute) for unordered arrival

Multi-GPU: groups shard across ranks, no data-path collective; NCCL only reduces the per-rank
counters and times.
"""
from __future__ import annotations

import argparse
import gc
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "commit_index_recomputes_per_s"
UNIT = "recomputes/s"
K_PEERS = 5
B_ALG_APPLY = 76                      # SURVEY 8(d): bytes per applied AppendResponse
N_ARENAS = 4                          # rotated so consecutive steps never share L2 contents
DUMP_MAX_GROUPS = 1_500_000           # --dump-outputs writes 32 B per group in all: at most 48 MB

# BASELINE.json configs: groups per GPU, peer slots in the voter union, joint?, seed
WORKLOADS = {
    "cfg2": dict(groups=100_000, peers=5, joint=False, seed=0x5EED0002,
                 text="cfg2: 100K raft groups x 5 peers per GPU"),
    "cfg3": dict(groups=1_000_000, peers=5, joint=False, seed=0x5EED0003,
                 text="cfg3: 1M raft groups x 5 peers per GPU"),
    "cfg4": dict(groups=1_000_000, peers=7, joint=True, seed=0x5EED0004,
                 text="cfg4: 1M raft groups x 7 peer slots per GPU under joint consensus (two 5-voter majorities)"),
    "cfg5": dict(groups=1_250_000, peers=5, joint=False, seed=0x5EED0005,
                 text="cfg5: 10M raft groups x 5 peers sharded over 8 GPUs = 1.25M groups per GPU"),
}


def config_of(args) -> dict:
    """The workload description both arms print (identical for --impl reference)."""
    w = WORKLOADS[args.workload]
    return {"workload": w["text"] + ", one synthetic AppendResponse round per step (apply + recompute)",
            "groups_per_gpu": args.groups or w["groups"], "peers": w["peers"], "seed": hex(w["seed"]),
            "l2": f"inputs larger than L2: {N_ARENAS} arenas rotated, fresh records every step",
            "parallelism": "groups sharded over the GPUs, no data-path collective"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the measured phases run."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int, cpus=None):
        self.gpu, self.proc, self.path = gpu_index, None, f"/tmp/raftgpu_clocks_{os.getpid()}.csv"
        self.cpus = cpus    # where the poller may run: NOT on the staging threads' cores (it wakes every 50 ms and
        #                     a pinned staging thread that loses its CPU for a time slice stalls the whole step)

    def start(self):
        try:
            self.f = open(self.path, "w")
            cpus = self.cpus
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-i", str(self.gpu), "-lms", "50"], stdout=self.f, stderr=subprocess.DEVNULL,
                preexec_fn=(lambda: os.sched_setaffinity(0, cpus)) if cpus else None)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.proc:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        with open(self.path) as f:
            for line in f:
                parts = [x.strip() for x in line.split(",")]
                if len(parts) < 8:
                    continue
                try:
                    sm.append(float(parts[1]))
                    mx.append(float(parts[2]))
                except ValueError:
                    continue
                for nm, v in zip(names, parts[4:8]):
                    if v == "Active":
                        reasons.add(nm)
        try:
            os.remove(self.path)
        except OSError:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons),
                       samples=len(sm))
        return out


def gpu_local_cpus(torch, device: int):
    """CPUs on the NUMA node the GPU's PCIe root hangs off (sysfs local_cpulist)."""
    try:
        pr = torch.cuda.get_device_properties(device)
        path = f"/sys/bus/pci/devices/{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0/local_cpulist"
        cpus = set()
        for tok in open(path).read().strip().split(","):
            lo, _, hi = tok.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        return cpus & os.sched_getaffinity(0)
    except Exception:
        return set()


def _siblings(cpu: int):
    try:
        txt = open(f"/sys/devices/system/cpu/cpu{cpu}/topology/thread_siblings_list").read().strip()
        out = set()
        for tok in txt.split(","):
            lo, _, hi = tok.partition("-")
            out.update(range(int(lo), int(hi or lo) + 1))
        return out
    except Exception:
        return {cpu}


def dump_outputs(path, n, steps):
    """steps: {leg: (advanced bitmap u32[], commit index u64[])} of one step.  Writes groups.npy (the group ids, float64:
    all of them, or a fixed seeded sample of DUMP_MAX_GROUPS), and per leg <leg>_advanced.npy (float32, 1 where the group
    advanced) and <leg>_commit_index.npy (float64, the group's new commit index; -1 where it did not advance, since the
    API leaves those entries unspecified)."""
    os.makedirs(path, exist_ok=True)
    groups = np.arange(n)
    if n > DUMP_MAX_GROUPS:
        groups = np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_GROUPS, replace=False))
    np.save(os.path.join(path, "groups.npy"), groups.astype(np.float64))
    for leg, (bm, com) in steps.items():
        adv = np.unpackbits(bm.view(np.uint8), bitorder="little")[groups].astype(bool)
        com = com[groups]
        if np.any(com[adv] >= 1 << 53):
            raise ValueError(f"{leg}: a commit index is not exact in float64")
        np.save(os.path.join(path, f"{leg}_advanced.npy"), adv.astype(np.float32))
        np.save(os.path.join(path, f"{leg}_commit_index.npy"), np.where(adv, com.astype(np.float64), -1.0))


def cpu_leg(n_groups, seed, rounds_wanted, threads, budget_s=20.0, joint=False):
    """The oracle (oracle/raft_oracle.c: apply + recompute, range-partitioned over `threads`
    pthreads) on a bounded sample of the same workload.  Only used as the CPU baseline."""
    B = importlib.import_module("raft-rs_b200").binding
    from oracle import oracle as O
    synth = B.Synth(n_groups, seed, k_peers=K_PEERS, joint=joint)
    cols = O.copy_columns(synth.initial)
    total, done = 0.0, 0
    for _ in range(rounds_wanted):
        recs = synth.next_round()
        secs, _ = O.bench_step(cols, recs, threads, fast=True)
        total += secs
        done += 1
        if total > budget_s:
            break
    return n_groups * done / total, done


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path.  raft-rs is Rust and
    this image has no rustc/cargo, so the arm runs the pinned C port (oracle/) with every host
    thread, on the same config / metric as the GPU arm: it consumes the same 24-byte records the
    GPU arm's `e2e` starts from."""
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    t0 = time.perf_counter()
    B = importlib.import_module("raft-rs_b200").binding
    from oracle import oracle as O
    w = WORKLOADS[args.workload]
    n = args.groups or w["groups"]
    synth = B.Synth(n, w["seed"], k_peers=K_PEERS, joint=w["joint"])
    cols = O.copy_columns(synth.initial)
    for _ in range(args.warmup):   # warmup rounds are part of the same stream
        O.bench_step(cols, synth.next_round(), threads, fast=True)
    total = 0.0
    for _ in range(args.steps):
        secs, _ = O.bench_step(cols, synth.next_round(), threads, fast=True)
        total += secs
    value = n * args.steps / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
        "data": "synthetic", "config": config_of(args),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{args.steps} rounds of the {args.workload} stream ({n} groups), {threads} pthreads, "
                                   "oracle/raft_oracle.c tuned path (ro_bench_step_fast, == the literal port), "
                                   "input = 24-byte records in host memory"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="graft", choices=["graft", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS),
                    help="BASELINE.json config: cfg3 (default, the headline) 1M groups x 5 peers per GPU; cfg4 1M groups "
                         "x 7 peer slots under joint consensus (90 B per recompute); cfg5 10M groups over 8 GPUs "
                         "(1.25M per GPU); cfg2 100K groups")
    ap.add_argument("--groups", type=int, default=0, help="override the groups per GPU of the workload")
    ap.add_argument("--e2e-threads", type=int, default=0, help="library staging threads (default: from the GPU-local cores)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="timed e2e steps (default: --steps)")
    ap.add_argument("--e2e-chunk", type=int, default=0,
                    help="pipelined e2e steps per timed chunk (default: all timed steps in one chunk, at most 32, for `e2e`; "
                         "8 for the secondary legs)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sublegs", action="store_true", help="skip recompute_only / scatter / secondary e2e legs")
    ap.add_argument("--profile", action="store_true",
                    help="device-resident loop only (for ncu): no clock warm loop, no e2e, no CPU leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step of the fused leg and of `e2e` returned "
                         "(advanced flag and new commit index per group) as DIR/<name>.npy; DIR/rank<r>/ under several "
                         "ranks.  Inputs are seeded: the same arguments give the same outputs on every build")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch
    import torch.distributed as dist

    B = importlib.import_module("raft-rs_b200").binding
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback (use --impl reference "
                         "for the CPU baseline arm)")
    torch.cuda.set_device(local_rank)
    all_cpus = os.sched_getaffinity(0)
    local_cpus = gpu_local_cpus(torch, local_rank)
    if local_cpus:
        # like `numactl --cpunodebind`: host staging threads and their buffers next to the GPU
        os.sched_setaffinity(0, local_cpus)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    wl = WORKLOADS[args.workload]
    n = args.groups or wl["groups"]
    K, W = args.steps, args.warmup
    joint = wl["joint"]
    k_union = wl["peers"]
    seed0 = wl["seed"]
    b_alg_recompute = 8 * k_union + 34    # SURVEY 8(d): 74 B per recompute at K = 5, 90 B at 7
    peak_gbs, peak_src = peaks()
    sublegs = not (args.no_sublegs or args.profile)
    rec_slots = (7 if joint else 5) * n + 64

    # ---- synthetic inputs: N_ARENAS independent stores; W+K rounds for the fused leg and, after
    # them in the same streams, W+K rounds for the scatter leg.  HBM holds all rounds; host memory
    # is one reused record buffer per generator.
    n_legs = 2 if sublegs else 1
    total_rounds = n_legs * (W + K)
    per_arena = [(total_rounds + N_ARENAS - 1 - a) // N_ARENAS for a in range(N_ARENAS)]
    arenas, round_len, d_recs, d_offs, d_outs = [], [], [], [], []
    pack_buf = np.empty((7 * n + 64, 2), dtype=np.uint64)
    for a in range(N_ARENAS):
        seed = seed0 + 0x100 * a + 0x10000 * rank
        s = B.Synth(n, seed, k_peers=K_PEERS, joint=joint)
        ar = B.Arena(n, device=local_rank, n_rings=1, ring_records=4096)
        assert ar.group_alloc_range(n) == 0
        ar.load_columns(s.initial)
        ptrs, lens, offs = [], [], []
        for _ in range(per_arena[a]):
            recs = s.next_round()
            k = ar.pack_records(recs, pack_buf)      # the packed 16-byte form, in group order
            p = ar.device_alloc(16 * k)
            ar.h2d(p, pack_buf[:k])
            lens.append((k, len(recs)))
            off = B.tile_index(pack_buf, k, n)       # first record of every 256-group tile
            po = ar.device_alloc(off.nbytes)
            ar.h2d(po, off)
            offs.append(po)
            ptrs.append(p)
        # the step's outputs in HBM: the advanced bitmap and the new commit index of every advanced group
        d_outs.append((ar.device_alloc(4 * ((n + 31) // 32 + 1)), ar.device_alloc(8 * n)))
        arenas.append(ar)
        round_len.append(lens)
        d_recs.append(ptrs)
        d_offs.append(offs)
        del s
    schedule = [(i % N_ARENAS, i // N_ARENAS) for i in range(total_rounds)]  # (arena, round) per step

    stream = torch.cuda.Stream()
    sh = stream.cuda_stream

    def step_fused(i):
        a, r = schedule[i]
        arenas[a].step_sorted_device(d_recs[a][r], round_len[a][r][0], d_offs[a][r], stream=sh,
                                     d_adv=d_outs[a][0], d_commit=d_outs[a][1])

    def step_scatter(i, ev=None):
        a, r = schedule[i]
        arenas[a].apply_device_packed(d_recs[a][r], round_len[a][r][0], stream=sh)
        if ev:
            ev.record(stream)
        arenas[a].recompute(0, n, stream=sh, d_adv=d_outs[a][0], d_commit=d_outs[a][1])

    def timed(fn, first, count, per_launch=True):
        """count back-to-back steps under CUDA events on the launching stream -> (ms total, ms in kernels).
        per_launch: an event pair around every launch (the fused kernel: 70 us, the pair costs nothing
        visible); without it the launches are captured into ONE CUDA graph and replayed, so that short
        kernels (the 14 us recompute pass) run back to back instead of at the pace Python issues them."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        graph = None
        if not per_launch:
            try:
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=stream):
                    for i in range(count):
                        fn(first + i)
            except Exception as e:   # capture refused: time the plain launches
                print(f"[bench] CUDA graph capture failed ({e}); timing direct launches", file=sys.stderr)
                graph = None
                torch.cuda.synchronize()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(count)] \
            if per_launch else []
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0.record(stream)
        if graph is not None:
            graph.replay()
        else:
            for i in range(count):
                if per_launch:
                    evs[i][0].record(stream)
                fn(first + i)
                if per_launch:
                    evs[i][1].record(stream)
        e1.record(stream)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        total = e0.elapsed_time(e1)
        return total, (sum(a_.elapsed_time(b_) for a_, b_ in evs) if per_launch else total)

    sampler = ClockSampler(local_rank, (all_cpus - local_cpus) or None)   # the poller runs on the other socket
    sampler.start()
    with torch.cuda.stream(stream):
        # clocks up: the recompute pass is idempotent on unchanged progress
        t_end = time.perf_counter() + (0.0 if args.profile else 0.3)
        while time.perf_counter() < t_end:
            for a in arenas:
                a.recompute(0, n, stream=sh)
            stream.synchronize()
        for i in range(W):
            step_fused(i)
        # the K timed steps are captured into ONE CUDA graph and replayed: the kernels run back to back, so their
        # average duration is the timed region / K (no per-launch event pairs, no Python launch pacing in between)
        ms_total, ms_kernel = timed(step_fused, W, K, per_launch=False)
        n_records = sum(round_len[a][r][1] for a, r in schedule[W:W + K])
        dumps = {}
        if args.dump_outputs:    # read now: the scatter and recompute legs reuse the output buffers
            a = schedule[W + K - 1][0]
            bm, com = np.empty((n + 31) // 32, dtype=np.uint32), np.empty(n, dtype=np.uint64)
            arenas[a].d2h(bm, d_outs[a][0])
            arenas[a].d2h(com, d_outs[a][1])
            dumps["fused"] = (bm, com)
        sc = ro = None
        if sublegs:
            # scatter: the same streams continue through the general path (no group order needed)
            base = W + K
            for i in range(W):
                step_scatter(base + i)
            ev_mid = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for i in range(K):
                evs[i][0].record(stream)
                step_scatter(base + W + i, ev_mid[i])
                evs[i][1].record(stream)
            e1.record(stream)
            torch.cuda.synchronize()
            sc_records = sum(round_len[a][r][1] for a, r in schedule[base + W:base + W + K])
            sc = {"ms_total": e0.elapsed_time(e1),
                  "ms_apply": sum(evs[i][0].elapsed_time(ev_mid[i]) for i in range(K)),
                  "ms_recompute": sum(ev_mid[i].elapsed_time(evs[i][1]) for i in range(K)), "records": sc_records}
            # recompute only: Raft::maybe_commit over every group, arenas rotated (4 x 74 MB > L2 hit window)
            for i in range(W):
                arenas[i % N_ARENAS].recompute(0, n, stream=sh)
            ro_total, _ = timed(lambda i: arenas[i % N_ARENAS].recompute(0, n, stream=sh, d_adv=d_outs[i % N_ARENAS][0],
                                                                          d_commit=d_outs[i % N_ARENAS][1]), 0, K, per_launch=False)
            ro = {"ms_total": ro_total}

    # ---- e2e: host buffers -> C-ABI -> results in host memory, on a fresh arena ------------------
    # staging threads per rank: one per physical GPU-local core, shared with the other ranks whose
    # GPU hangs off the same socket (two sockets per host)
    # ranks whose GPU hangs off the same socket share its cores: every rank takes its share (RAFTGPU_CPU_SHARE = k/R)
    same_node = [r for r in range(world) if gpu_local_cpus(torch, r) == local_cpus] if local_cpus else list(range(world))
    ranks_per_node = max(1, len(same_node))
    if ranks_per_node > 1:
        os.environ.setdefault("RAFTGPU_CPU_SHARE", f"{same_node.index(local_rank)}/{ranks_per_node}")
    # three quarters of the rank's share of the GPU-local logical CPUs: every physical core plus half of the SMT
    # siblings (measured at N = 1: 32 threads 0.91e9/s, 48 threads 1.06e9/s, 56 threads stall -- the caller's and the
    # submitter's threads need CPUs too)
    e2e_threads = args.e2e_threads or max(4, min(48, (3 * (len(local_cpus) or 64)) // (4 * ranks_per_node)))
    os.environ.setdefault("RAFTGPU_HOST_THREADS", str(e2e_threads))
    e2e_steps = 0 if args.profile else (args.e2e_steps or K)
    chunk = max(2, args.e2e_chunk or min(32, e2e_steps))    # `e2e`: one pinned record buffer per step of a chunk
    chunk2 = max(2, args.e2e_chunk or 8)                    # secondary legs
    es = B.Synth(n, seed0 + 0x10000 * rank, k_peers=K_PEERS, joint=joint)
    ea = B.Arena(n, device=local_rank, n_rings=e2e_threads)
    if local_cpus:
        # the caller's thread keeps off the CPUs the staging threads are pinned to (staging_cpu_order in
        # abi_staging.inc: the rank's share of the socket's physical cores, then of their SMT siblings)
        prim = sorted(c for c in local_cpus if c == min(_siblings(c)))
        sibs = sorted(local_cpus - set(prim))
        k = same_node.index(local_rank) if ranks_per_node > 1 else 0
        share = prim[k::ranks_per_node] + sibs[k::ranks_per_node]
        rest = set(share[e2e_threads:])
        if rest:
            os.sched_setaffinity(0, rest)
    assert ea.group_alloc_range(n) == 0
    ea.load_columns(es.initial)
    flags = B.STEP_READ_COMMITTED
    # the caller's 24-byte records live in pinned, GPU-local host memory (raftgpu_host_alloc)
    rec_bytes = rec_slots * B.APPEND_RESP_DTYPE.itemsize
    bufs = [ea.host_alloc_bytes(rec_bytes).view(B.APPEND_RESP_DTYPE) for _ in range(chunk)] if e2e_steps else []

    def pipelined_leg(prepare, begin, chunk=chunk2):
        """`chunk` steps at a time: prepare(j) builds batch j (UNTIMED: the generation of the inputs);
        then, timed: begin(batch 0); for each j: begin(batch j+1) while step j is in flight; wait(j).
        Wall clock around the chunk, barrier + synchronize on both sides."""
        secs, done, dma, first = 0.0, 0, [0, 0], True
        phase = [0.0, 0.0]    # host seconds inside begin / inside wait
        while done < e2e_steps:
            m = min(chunk, e2e_steps - done)
            batches = [prepare(j) for j in range(m)]
            if first:                       # untimed warm-up steps (pool threads, first-touch, clocks)
                for j in range(m):
                    begin(batches[j])
                    ea.step_wait()
                first = False
                continue
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            gc.collect()
            gc.disable()      # no collector pause inside the timed region
            t0 = time.perf_counter()
            begin(batches[0])
            phase[0] += time.perf_counter() - t0
            for j in range(m):
                ta = time.perf_counter()
                if j + 1 < m:
                    begin(batches[j + 1])
                tb = time.perf_counter()
                sr = ea.step_wait()
                tc = time.perf_counter()
                phase[0] += tb - ta
                phase[1] += tc - tb
                dma[0] += sr.h2d_bytes
                dma[1] += sr.d2h_bytes
                # the step really did the work it is credited with: every group recomputed, a full round applied
                assert sr.n_groups == n and sr.n_records > n, (sr.n_groups, sr.n_records)
                if os.environ.get("RAFTGPU_TRACE"):
                    print(f"[bench] step {j}: begin {1e6 * (tb - ta):.0f} us, wait {1e6 * (tc - tb):.0f} us", file=sys.stderr)
            secs += time.perf_counter() - t0
            gc.enable()
            done += m
        d = max(1, done)
        return {"seconds": secs, "steps": done, "h2d": dma[0] / d, "d2h": dma[1] / d,
                "host_ms": {"begin": 1e3 * phase[0] / d, "wait": 1e3 * phase[1] / d}}

    legs = {}
    if e2e_steps:
        # e2e: 24-byte records (pinned host memory) -> raftgpu_step_begin_records -> raftgpu_step_wait
        # (RAFTGPU_STEP_ASYNC: the call returns once the staging threads have the batch; the records stay untouched
        # in their pinned buffer until the step's raftgpu_step_wait, which is what this loop does anyway)
        # With a small CPU share (several GPUs per socket) packing is the bottleneck: the records then cross PCIe as
        # they are (RAFTGPU_STEP_RAW: 3.7x the bytes, no host work at all).  Crossover ~12 staging threads (DESIGN 5).
        # Default: HYBRID -- the library packs the head of the batch while the DMA engine ships the tail as it is,
        # split so that the staging threads and PCIe finish together (include/raftgpu.h RAFTGPU_STEP_HYBRID).
        e2e_mode = os.environ.get("BENCH_E2E_MODE") or "hybrid"
        e2e_flags = flags | {"raw": B.STEP_RAW, "packed": B.STEP_ASYNC, "hybrid": B.STEP_ASYNC | B.STEP_HYBRID}[e2e_mode]
        legs["e2e"] = pipelined_leg(lambda j: es.next_round(bufs[j]),
                                    lambda recs: ea.step_begin_records(recs, e2e_flags), chunk)
        if args.dump_outputs:
            dumps["e2e"] = tuple(x.copy() for x in ea.step_results(n))
    if e2e_steps and sublegs:
        # e2e_prepacked: the caller already holds the compact stream (pack untimed)
        cap_b = B.compact_bound(rec_slots)
        pk = [ea.host_alloc_bytes(cap_b) for _ in range(chunk2)]
        legs["e2e_prepacked"] = pipelined_leg(
            lambda j: (pk[j], B.pack_compact(es.next_round(bufs[j]), pk[j])[0]),
            lambda b: ea.step_begin_compact(b[0], b[1], flags))
        for b_ in pk:
            ea.host_free(b_)
        if hasattr(ea, "step_begin_wire"):
            # e2e_wire: serialized eraftpb.Message frames (pinned) -> device-side varint decode -> the same step
            W_ = importlib.import_module("raft-rs_b200").wire
            wb = [W_.WireBuffers(ea, rec_slots) for _ in range(chunk2)]
            legs["e2e_wire"] = pipelined_leg(
                lambda j: wb[j].encode(es.next_round(bufs[j])),
                lambda w_: ea.step_begin_wire(w_, flags))
            for w_ in wb:
                w_.free()
    clocks = sampler.stop()

    # ---- aggregate over ranks (NCCL: counters and times only) -----------------------------------
    cnt = [a.counters() for a in arenas]
    S = importlib.import_module("raft-rs_b200.shard")
    times = {"ms_total": ms_total}
    for name, lg in legs.items():
        times[name] = lg["seconds"]
    if sc:
        times["sc_ms"] = sc["ms_total"]
        times["ro_ms"] = ro["ms_total"]
    sums, maxes = S.aggregate(
        dist if world > 1 else None, torch,
        {"recomputes": sum(c["recomputes"] for c in cnt), "advanced": sum(c["advanced"] for c in cnt),
         "records": sum(c["records"] for c in cnt)},
        times, device="cuda")
    value = world * n * K / (maxes["ms_total"] * 1e-3)

    if rank == 0:
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                traffic = json.load(f)
        except Exception:
            traffic = {}
        alg_bytes = n_records * B_ALG_APPLY + n * K * b_alg_recompute
        gbs = alg_bytes / (ms_kernel * 1e-3) / 1e9
        tkey = "step_tile_kernel" + ("" if args.workload in ("cfg3", "cfg5", "cfg2") else "_" + args.workload)
        tr = traffic.get(tkey)
        if tr and n != 1_000_000:
            tr = int(tr * n / 1_000_000)   # the captures are of 1M-group launches; the kernel's traffic is linear in the groups
        dom = {"kernel": "step_tile_kernel", "avg_us": 1e3 * ms_kernel / K, "share": ms_kernel / ms_total,
               "alg_bytes_per_launch": alg_bytes / K, "achieved": gbs, "frac": gbs / peak_gbs, "traffic": tr}
        if tr:   # the honest bandwidth fraction: DRAM bytes the kernel really moves (ncu) / its duration
            dom["dram_gbs"] = tr / (dom["avg_us"] * 1e-6) / 1e9
            dom["dram_frac"] = dom["dram_gbs"] / peak_gbs
        cfg = config_of(args)    # identical to the reference arm's
        details = {"records_per_step": n_records / K, "record_format": "16 B packed (raftgpu_pack_records), group order",
                   "device_path": "fused tile kernel (raftgpu_step_sorted_device, group-ordered batch + tile index)",
                   "outputs": "advanced bitmap + new commit index per advanced group written to HBM inside the timed launches",
                   "prepared_outside": "packed records and the tile index (4 B per 256 groups) are device resident before the timed "
                                       "region; the `scatter` object is the same step for any arrival order with no index"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": maxes["ms_total"] / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": cfg, "details": details,
            "roofline": {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["achieved"],
                         "peak": peak_gbs, "unit": "GB/s", "frac": dom["frac"], "traffic": dom["traffic"],
                         "dram_frac": dom.get("dram_frac"), "peak_source": peak_src,
                         "note": "achieved = SURVEY 8(d) algorithmic bytes (76 B per record + 8K+34 B per group) / the kernel's "
                                 "average duration (CUDA events); dram_frac = ncu DRAM bytes per launch (profiles/traffic.json) / "
                                 "the same duration: the fused kernel reads `matched` once, so it moves fewer bytes than the "
                                 "two-pass algorithmic count"},
            "kernels": [dom],
            "gpu_launches": K,
            "clocks": clocks,
            "counters": {"recomputes": sums["recomputes"], "advanced": sums["advanced"], "records": sums["records"]},
        }
        if sc:
            line["scatter"] = {
                "value": world * n * K / (maxes["sc_ms"] * 1e-3), "unit": UNIT, "ms_per_step": maxes["sc_ms"] / K,
                "apply_us": 1e3 * sc["ms_apply"] / K, "recompute_us": 1e3 * sc["ms_recompute"] / K,
                "apply_frac": sc["records"] * B_ALG_APPLY / (sc["ms_apply"] * 1e-3) / 1e9 / peak_gbs,
                "api": "raftgpu_apply_device_packed + raftgpu_recompute: the general path, any arrival order (one record per "
                       "cell per call), no tile index"}
            ro_gbs = world * n * K * b_alg_recompute / (maxes["ro_ms"] * 1e-3) / 1e9
            rkey = "recompute_kernel" + ("" if args.workload in ("cfg3", "cfg5", "cfg2") else "_" + args.workload)
            line["recompute_only"] = {
                "value": world * n * K / (maxes["ro_ms"] * 1e-3), "unit": UNIT, "us_per_pass": 1e3 * maxes["ro_ms"] / K,
                "bytes_per_recompute": b_alg_recompute, "achieved_gbs_per_gpu": ro_gbs / world,
                "frac": ro_gbs / world / peak_gbs, "traffic": (int(traffic[rkey] * n / 1_000_000) if traffic.get(rkey) else None),
                "api": "raftgpu_recompute: Raft::maybe_commit for every group, nothing applied (BASELINE.md 3: rate x (8K+34) B)"}
        apis = {
            "e2e": "raftgpu_step_begin_records(READ_COMMITTED | ASYNC | HYBRID) + raftgpu_step_wait (`mode`: hybrid; packed = "
                   "without HYBRID, raw = RAFTGPU_STEP_RAW): the step's 24-byte records (raftgpu_append_resp, what "
                   "handle_append_response consumes) sit in pinned host memory (raftgpu_host_alloc); timed: the library's "
                   "staging threads pack the head of the batch into the compact stream while the DMA engine ships the tail "
                   "as it is (split so that both finish together), H2D, scatter apply of the raw part, tile index + fused "
                   "apply/recompute kernel, D2H of the advanced bitmap and the commit indexes; two steps in flight",
            "e2e_prepacked": "raftgpu_step_begin_compact + raftgpu_step_wait: the caller already holds the batch as the "
                             "compact stream (raftgpu_pack_compact NOT timed): the PCIe-bound floor of the step",
            "e2e_wire": "raftgpu_step_begin_wire + raftgpu_step_wait: serialized eraftpb.Message frames in pinned host "
                        "memory, varint decode on the GPU, then the same step",
        }
        for name, lg in legs.items():
            if not lg["steps"]:
                continue
            line[name] = {"value": world * n * lg["steps"] / maxes[name], "unit": UNIT,
                          "ms_per_step": 1e3 * maxes[name] / lg["steps"], "steps": lg["steps"],
                          "h2d_bytes_per_step": lg["h2d"], "d2h_bytes_per_step": lg["d2h"],
                          "host_ms_per_step": lg["host_ms"], "pipelined_chunk": chunk if name == "e2e" else chunk2,
                          "api": apis[name]}
        if "e2e" in line:
            line["e2e"].update({"caller_record_bytes_per_step": 24.0 * n_records / K, "host_threads": e2e_threads, "mode": e2e_mode,
                                "host_cpus_bound": len(local_cpus) or None})
        if world == 1 and not args.no_cpu_baseline and not args.profile:
            os.sched_setaffinity(0, all_cpus)   # the CPU baseline gets every host core
            threads = len(all_cpus)
            v, done = cpu_leg(n, seed0, 64, threads, budget_s=15.0, joint=joint)
            line["cpu_baseline"] = {
                "value": v, "unit": UNIT, "cores": threads, "kind": "port",
                "sample": f"{done} rounds of the same {args.workload} stream (apply + recompute), {threads} "
                          "pthreads, oracle/raft_oracle.c tuned path (ro_bench_step_fast, == the literal port)"}
        print(json.dumps(line), flush=True)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs if world == 1 else os.path.join(args.dump_outputs, f"rank{rank}"), n, dumps)
    for a in arenas:
        a.close()
    ea.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
