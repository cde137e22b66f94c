"""Micro-benchmark of the read-index passes: 1M groups x 5 voters, one MsgReadIndex per leader group per tick, 4 heartbeat
acknowledgements per request, 4 arenas rotated so the working set exceeds L2; CUDA-event timing of every pass over many
launches after a warm-up, the existing heartbeat_resp pass beside them for context.  Prints the card and its power limit,
then one line for DESIGN.md.  Algorithmic bytes are computed here, not measured; the peak is the project's measured HBM
rate (DESIGN.md 5)."""
import importlib
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
B = importlib.import_module("raft-rs_b200").binding

PEAK_GBS = 6555.8
n, A, P, K = 1_000_000, 4, 8, 20
# bytes per item, from the kernels' loads and stores (k_read.cuh, k_control.cuh)
BYTES = {
    # request 16 + status 1 + index 8; meta 4, committed / term_start / last_index 24, rd_meta 4 + 4, the new entry 20
    "request": 16 + 1 + 8 + 4 + 24 + 8 + 20,
    # record 24; meta 4, rd_meta 4, the entry's ctx 8, its word read and written 8
    "ack": 24 + 4 + 4 + 8 + 8,
    # per group: rd_meta 4 + 4, meta 4, the word 4, the released entry's ctx + index 16 read and its 24-byte state written
    "release": 4 + 4 + 4 + 4 + 16 + 24,
    # record 24 + result 1; meta 4, touched 4, pflags 2, peer_committed 16, matched 8, last_index 8, pending_req_snapshot 8
    "heartbeat_resp": 24 + 1 + 4 + 4 + 2 + 16 + 8 + 8 + 8,
}

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()
print(f"card: {gpu[0] if gpu else 'unknown'}")

stream = torch.cuda.Stream()
rng = np.random.default_rng(7)
arenas = []
for k in range(A):
    a = B.Arena(n)
    a.enable_read_index(P)
    a.group_alloc_range(n)
    a.column_write(B.COL_META, 0, 0, np.full(n, B.make_meta(0x1F, self_slot=0), dtype=np.uint32))
    a.column_write(B.COL_LAST_INDEX, 0, 0, np.full(n, 100, dtype=np.uint64))
    a.column_write(B.COL_COMMITTED, 0, 0, np.full(n, 100, dtype=np.uint64))
    a.column_write(B.COL_TERM_START, 0, 0, np.full(n, 50, dtype=np.uint64))
    reqs = np.zeros(n, dtype=B.READ_REQ_DTYPE)
    reqs["group"], reqs["from_slot"], reqs["ctx"] = np.arange(n), rng.integers(1, 5, n), rng.integers(0, 1 << 40, n)
    recs = np.zeros(4 * n, dtype=B.APPEND_RESP_DTYPE)
    recs["group"], recs["peer_slot"] = np.repeat(np.arange(n), 4), np.tile([1, 2, 3, 4], n)
    recs["flags"], recs["index"], recs["commit"] = B.REC_HEARTBEAT | B.REC_READ_CTX, np.repeat(reqs["ctx"], 4), 100
    d = {name: a.device_alloc(size) for name, size in (("req", reqs.nbytes), ("st", n), ("idx", 8 * n), ("rec", recs.nbytes),
                                                       ("res", 4 * n), ("out", 24 * n), ("cnt", 16))}
    a.h2d(d["req"], reqs)
    a.h2d(d["rec"], recs)
    arenas.append((a, d))

PASSES = ("request", "ack", "release", "heartbeat_resp")


def run(a, d, name):
    s = stream.cuda_stream
    if name == "request":
        a.read_index_device(d["req"], n, d["st"], d["idx"], stream=s)
    elif name == "ack":
        a.read_ack_device(d["rec"], 4 * n, stream=s)
    elif name == "release":
        a.read_release_device(0, n, d["out"], n, d["cnt"], stream=s)
    else:
        a._ck(a._L.raftgpu_heartbeat_resp_device(a._h, s, d["rec"], 4 * n, d["res"], None), "heartbeat_resp_device")


for k in range(2 * A):                                   # warm-up: every pass on every arena
    for name in PASSES:
        run(*arenas[k % A], name)
torch.cuda.synchronize()
ms = dict.fromkeys(PASSES, 0.0)
for k in range(K):
    a, d = arenas[k % A]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(PASSES) + 1)]
    ev[0].record(stream)
    for i, name in enumerate(PASSES):
        run(a, d, name)
        ev[i + 1].record(stream)
    torch.cuda.synchronize()
    for i, name in enumerate(PASSES):
        ms[name] += ev[i].elapsed_time(ev[i + 1])
# every tick released every request: check the last one
a, d = arenas[(K - 1) % A]
cnt, st = np.zeros(2, dtype=np.uint64), np.zeros(n, dtype=np.uint8)
a.d2h(cnt, d["cnt"])
a.d2h(st, d["st"])
assert cnt[0] == cnt[1] == n and np.all(st == B.READ_QUEUED), (cnt, np.bincount(st))
items = {"request": n, "ack": 4 * n, "release": n, "heartbeat_resp": 4 * n}
parts = []
for name in PASSES:
    us = 1e3 * ms[name] / K
    mb = BYTES[name] * items[name] / 1e6
    bound_us = mb / PEAK_GBS * 1e3
    parts.append(f"{name} {us:.1f} us ({mb:.0f} MB, >= {bound_us:.1f} us, {bound_us / us:.0%} of {PEAK_GBS} GB/s)")
print(f"read index, 1M groups x 5 voters, 1 request + 4 acks per group, {A} arenas rotated, max_pending {P}: " + "; ".join(parts))
for a, _ in arenas:
    a.close()
