"""Micro-benchmark: back-to-back recompute passes over rotated arenas (idempotent), CUDA events."""
import importlib, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
B = importlib.import_module("raft-rs_b200").binding
n = int(os.environ.get("N", 1_000_000)); joint = os.environ.get("JOINT", "0") == "1"
A = 4
arenas = []
for a in range(A):
    s = B.Synth(n, 0x5EED0003 + a, joint=joint)
    ar = B.Arena(n, n_rings=1, ring_records=4096)
    ar.group_alloc_range(n); ar.load_columns(s.initial); arenas.append(ar)
st = torch.cuda.Stream(); sh = st.cuda_stream
with torch.cuda.stream(st):
    for _ in range(20):
        for ar in arenas: ar.recompute(0, n, stream=sh)
    torch.cuda.synchronize()
    reps = 100
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(reps):
        for ar in arenas: ar.recompute(0, n, stream=sh)
    e1.record(st); torch.cuda.synchronize()
us = 1e3 * e0.elapsed_time(e1) / (reps * A)
k = 7 if joint else 5
print(f"recompute n={n} joint={joint}: {us:.2f} us/pass  {n*(8*k+34)/us/1e3:.0f} GB/s alg")
