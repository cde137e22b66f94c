"""Micro-benchmark of the fused tile kernel (step_tile_kernel): 1M groups x 5 peers, 4 arenas rotated (inputs larger
than L2), R rounds each, one CUDA graph of all launches, CUDA events.  With RAFTGPU_TILE_DEBUG=1 the kernel's phase
cycle counters are printed.  CONFIGS="K=V K=V;K=V;..." lists the knob settings to run after the default
(RAFTGPU_TILE_DEBUG / _SKIP), all in this one process."""
import importlib, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

os.environ["RAFTGPU_TILE_TUNE"] = "1"      # the library re-reads its RAFTGPU_TILE_* knobs on every launch
KNOBS = ("RAFTGPU_TILE_DEBUG", "RAFTGPU_TILE_SKIP")
CONFIGS = [{}, {"RAFTGPU_TILE_DEBUG": "1"}] + [dict(kv.split("=") for kv in c.split()) for c in os.environ.get("CONFIGS", "").split(";") if c.strip()]

import numpy as np, torch
B = importlib.import_module("raft-rs_b200").binding
n = int(os.environ.get("N", 1_000_000))
R = int(os.environ.get("R", 6))
joint = os.environ.get("JOINT", "0") == "1"
NA = 4
arenas, rounds = [], []
pack_buf = np.empty((7 * n + 64, 2), dtype=np.uint64)
for a in range(NA):
    s = B.Synth(n, 0x5EED0003 + 0x100 * a, k_peers=5, joint=joint)
    ar = B.Arena(n, n_rings=1, ring_records=4096)
    ar.group_alloc_range(n); ar.load_columns(s.initial)
    rr = []
    for _ in range(R):
        recs = s.next_round()
        k = ar.pack_records(recs, pack_buf)
        p = ar.device_alloc(16 * k); ar.h2d(p, pack_buf[:k])
        off = B.tile_index(pack_buf, k, n)
        po = ar.device_alloc(off.nbytes); ar.h2d(po, off)
        rr.append((p, k, po))
    arenas.append(ar); rounds.append(rr)
st = torch.cuda.Stream(); sh = st.cuda_stream
sched = [(i % NA, i // NA) for i in range(NA * R)]
warm = NA          # the first round of every arena, untimed
k = len(sched) - warm
snapshots = [ar.read_columns(n) for ar in arenas]


def run(cfg):
    for name in KNOBS:
        os.environ.pop(name, None)
    os.environ.update(cfg)
    for ar, snap in zip(arenas, snapshots):
        ar.load_columns(snap)                  # every configuration sees the same states
    with torch.cuda.stream(st):
        for a, r in sched[:warm]:
            arenas[a].step_sorted_device(*rounds[a][r], stream=sh)
        torch.cuda.synchronize()
        d0 = sum(ar.debug_read().astype(np.float64) for ar in arenas)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=st):
            for a, r in sched[warm:]:
                arenas[a].step_sorted_device(*rounds[a][r], stream=sh)
        best = 1e9
        for rep in range(3):
            if rep:
                for ar, snap in zip(arenas, snapshots):
                    ar.load_columns(snap)
                for a, r in sched[:warm]:
                    arenas[a].step_sorted_device(*rounds[a][r], stream=sh)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record(st); g.replay(); e1.record(st)
            torch.cuda.synchronize()
            best = min(best, 1e3 * e0.elapsed_time(e1) / k)
    msg = f"{best:.2f} us per launch (best of 3 x {k} launches)"
    if cfg.get("RAFTGPU_TILE_DEBUG"):
        d = sum(ar.debug_read().astype(np.float64) for ar in arenas) - d0
        tiles = max(d[4], 1)
        msg += "; cycles per tile (tid 0 of the consumer group): wait %.0f, A %.0f, B %.0f, C %.0f; tiles %d" % (
            d[0] / tiles, d[1] / tiles, d[2] / tiles, d[3] / tiles, tiles)
    print(cfg or "default", "->", msg, flush=True)


for cfg in CONFIGS:
    run(cfg)
