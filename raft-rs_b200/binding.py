"""ctypes binding of libraftgpu.so (include/raftgpu.h) for the tests and bench.py.

This is plumbing around the C-ABI: it never computes a quorum, a Progress
transition or a commit index itself -- every such call goes to the CUDA library
and raises when that fails (RAFTGPU_ERR_NO_DEVICE on a box without a GPU: there
is no CPU fallback).
"""
from __future__ import annotations

import ctypes as C
import os
import re
import types

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RAFTGPU_LIB") or os.path.join(_HERE, "libraftgpu.so")   # (RAFTGPU_LIB: experimental builds)
SYNTH_LIB_PATH = os.path.join(_HERE, "libraftgpu_synth.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "raftgpu.h")
SYNTH_HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "raftgpu_synth.h")

SLOTS = 8
U64_MAX = (1 << 64) - 1
NO_TERM_START = U64_MAX

OK, ERR_INVALID, ERR_CUDA, ERR_NOMEM, ERR_NO_DEVICE, ERR_RANGE, ERR_FULL, ERR_PEER_NOT_FOUND, \
    ERR_COMMIT_RANGE, ERR_BUSY, ERR_TOO_MANY_PEERS = 0, -1, -2, -3, -4, -5, -6, -7, -8, -9, -10

STATE_PROBE, STATE_REPLICATE, STATE_SNAPSHOT = 0, 1, 2
VOTE_PENDING, VOTE_LOST, VOTE_WON = 0, 1, 2
PF_STATE_MASK, PF_PAUSED, PF_RECENT_ACTIVE, PF_INS_FULL = 0x03, 0x04, 0x08, 0x10
META_HAS_SELF, META_GROUP_COMMIT = 0x08000000, 0x10000000
REC_REJECT, REC_LOCAL, REC_HEARTBEAT, REC_EXT = 0x01, 0x02, 0x04, 0x80
RES_OK, RES_OLD_PAUSED, RES_NO_PROGRESS, RES_SEND = 0x01, 0x02, 0x04, 0x08
STEP_READ_COMMITTED, STEP_READ_RESULTS, STEP_ASYNC, STEP_RAW, STEP_HYBRID = 0x1, 0x2, 0x4, 0x8, 0x10
BULK_SORTED = 0x1
(POP_MAYBE_UPDATE, POP_MAYBE_DECR_TO, POP_UPDATE_COMMITTED, POP_OPTIMISTIC_UPDATE, POP_BECOME_PROBE,
 POP_BECOME_REPLICATE, POP_BECOME_SNAPSHOT, POP_SNAPSHOT_FAILURE, POP_MAYBE_SNAPSHOT_ABORT, POP_IS_PAUSED,
 POP_RESUME, POP_PAUSE, POP_UPDATE_STATE, POP_RESET, POP_INS_ADD, POP_INS_FREE_TO, POP_INS_FREE_FIRST_ONE,
 POP_INS_RESET, POP_INS_FULL) = range(19)

(COL_MATCHED, COL_NEXT_IDX, COL_PEER_COMMITTED, COL_PENDING_SNAPSHOT, COL_PENDING_REQ_SNAPSHOT,
 COL_COMMIT_GROUP_ID, COL_PFLAGS, COL_VOTES, COL_META, COL_COMMITTED, COL_TERM_START,
 COL_LAST_INDEX, COL_TERM, COL_INS_META) = range(14)
WIRE_OK, WIRE_SKIP_TYPE, WIRE_TERM, WIRE_NEEDS_LOG, WIRE_MALFORMED, WIRE_DUP = range(6)

APPEND_RESP_DTYPE = np.dtype(
    [("group", "<u4"), ("peer_slot", "u1"), ("flags", "u1"), ("reserved", "<u2"),
     ("index", "<u8"), ("commit", "<u8")]
)
assert APPEND_RESP_DTYPE.itemsize == 24
SEND_ENTRY_DTYPE = np.dtype([("group", "<u4"), ("peer_slot", "u1"), ("flags", "u1"), ("reserved", "<u2"),
                             ("next_idx", "<u8")])
assert SEND_ENTRY_DTYPE.itemsize == 16
SEND_SNAPSHOT = 0x1
READ_REQ_DTYPE = np.dtype([("group", "<u4"), ("from_slot", "u1"), ("flags", "u1"), ("reserved", "<u2"), ("ctx", "<u8")])
assert READ_REQ_DTYPE.itemsize == 16
READ_STATE_DTYPE = np.dtype([("group", "<u4"), ("to_slot", "u1"), ("flags", "u1"), ("reserved", "<u2"),
                             ("index", "<u8"), ("ctx", "<u8")])
assert READ_STATE_DTYPE.itemsize == 24
READ_LOCAL, READ_LEASE = 0x1, 0x2
READ_DROPPED, READ_READY, READ_QUEUED, READ_ALREADY_PENDING, READ_FULL, READ_SPLIT, READ_INVALID = range(7)
REC_READ_CTX = 0x08
READ_WORD_LOCAL, READ_WORD_ACKED = 0x01000000, 0x02000000
NO_READ_CTX = U64_MAX

# host column name -> (column id, numpy dtype, per-peer?)
COLUMNS = {
    "matched": (COL_MATCHED, np.uint64, True),
    "next_idx": (COL_NEXT_IDX, np.uint64, True),
    "peer_committed": (COL_PEER_COMMITTED, np.uint64, True),
    "pending_snapshot": (COL_PENDING_SNAPSHOT, np.uint64, True),
    "pending_request_snapshot": (COL_PENDING_REQ_SNAPSHOT, np.uint64, True),
    "commit_group_id": (COL_COMMIT_GROUP_ID, np.uint64, True),
    "pflags": (COL_PFLAGS, np.uint8, True),
    "meta": (COL_META, np.uint32, False),
    "committed": (COL_COMMITTED, np.uint64, False),
    "term_start": (COL_TERM_START, np.uint64, False),
    "last_index": (COL_LAST_INDEX, np.uint64, False),
}
# (the term column, COL_TERM, is written separately: only the wire path reads it)


class RaftGpuError(RuntimeError):
    def __init__(self, status, what, detail=""):
        self.status = status
        super().__init__(f"{what}: {strerror(status)} ({status}){': ' + detail if detail else ''}")


class Progress(C.Structure):
    _fields_ = [("matched", C.c_uint64), ("next_idx", C.c_uint64),
                ("pending_snapshot", C.c_uint64), ("pending_request_snapshot", C.c_uint64),
                ("commit_group_id", C.c_uint64), ("committed_index", C.c_uint64),
                ("state", C.c_uint8), ("paused", C.c_uint8), ("recent_active", C.c_uint8),
                ("ins_full", C.c_uint8), ("present", C.c_uint8), ("reserved", C.c_uint8 * 3)]


class GroupState(C.Structure):
    _fields_ = [("meta", C.c_uint32), ("reserved", C.c_uint32), ("committed", C.c_uint64),
                ("term_start", C.c_uint64), ("last_index", C.c_uint64)]


class Info(C.Structure):
    _fields_ = [("abi_version", C.c_uint32), ("device", C.c_int32), ("cap", C.c_uint32),
                ("slots", C.c_uint32), ("n_alloc", C.c_uint32), ("hi", C.c_uint32),
                ("sm_count", C.c_uint32), ("reserved", C.c_uint32), ("l2_bytes", C.c_uint64),
                ("device_bytes", C.c_uint64), ("pinned_bytes", C.c_uint64)]


class Counters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("recomputes", "advanced", "records", "updates", "rejects",
                                          "decrements", "no_progress", "votes_tallied")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


class StepResult(C.Structure):
    _fields_ = [("n_records", C.c_uint64), ("n_waves", C.c_uint32), ("n_groups", C.c_uint32),
                ("n_advanced", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("n_duplicates", C.c_uint64)]


class WireBatch(C.Structure):
    _fields_ = [("bytes", C.c_void_p), ("n_bytes", C.c_uint64), ("offsets", C.c_void_p), ("n", C.c_uint64),
                ("records", C.c_void_p), ("n_records", C.c_uint64)]


class SynthColumns(C.Structure):
    _fields_ = [("cap", C.c_uint32), ("n_groups", C.c_uint32)] + \
        [(n, C.c_void_p) for n in ("matched", "next_idx", "peer_committed", "pflags", "meta",
                                   "committed", "term_start", "last_index", "term", "sim_acked",
                                   "sim_last", "sim_flags")]


def compact_bound(n_records: int) -> int:
    return int(lib().raftgpu_compact_bound(n_records))


def pack_compact(recs: np.ndarray, out: np.ndarray, want_units: bool = False):
    """records -> compact stream blob in `out` (u8, 16-byte aligned).  Returns (bytes, unit_of_record|None)."""
    assert recs.dtype == APPEND_RESP_DTYPE and recs.flags.c_contiguous and out.dtype == np.uint8
    nb = C.c_uint64()
    units = np.empty(len(recs), dtype=np.uint32) if want_units else None
    rc = lib().raftgpu_pack_compact(recs.ctypes.data, len(recs), out.ctypes.data, out.nbytes, C.byref(nb),
                                    units.ctypes.data if want_units else None)
    if rc != 0:
        raise RuntimeError(f"raftgpu_pack_compact failed: {rc}")
    return nb.value, units


COMPACT_HDR_DTYPE = np.dtype([("magic", "<u4"), ("n_units", "<u4"), ("n_blocks", "<u4"), ("n_side", "<u4"),
                              ("n_records", "<u8"), ("off_blocks", "<u8"), ("off_units", "<u8"),
                              ("off_side", "<u8"), ("total_bytes", "<u8"), ("flags", "<u4"), ("reserved", "<u4")])
COMPACT_TILEABLE, COMPACT_ONE_WAVE = 0x1, 0x2


def unpack_compact(blob: np.ndarray) -> np.ndarray:
    """Decode a compact stream back to public records (tests; mirrors load_compact in kernels.cuh)."""
    h = blob[:COMPACT_HDR_DTYPE.itemsize].view(COMPACT_HDR_DTYPE)[0]
    assert h["magic"] == 0x31434752
    nu, ns = int(h["n_units"]), int(h["n_side"])
    units = blob[int(h["off_units"]):int(h["off_units"]) + 4 * nu].view(np.uint32)
    g_base = blob[int(h["off_blocks"]):int(h["off_blocks"]) + 4 * int(h["n_blocks"])].view(np.uint32)
    side = blob[int(h["off_side"]):int(h["off_side"]) + 24 * ns].view(APPEND_RESP_DTYPE)
    out = []
    for i in range(nu):
        u = int(units[i])
        kind = u & 3
        if kind == 3:
            k = u >> 2
            if k < 0x1fffffff and k < ns:     # (payload units and padding carry no record of their own)
                out.append(tuple(side[k]))
                if (side[k]["flags"] & REC_REJECT) and k + 1 < ns and (side[k + 1]["flags"] & REC_EXT):
                    out.append(tuple(side[k + 1]))
            continue
        if kind != 0:
            continue
        back = (u >> 3) & 7
        hpos = i - back - 2
        ha, hb = int(units[hpos]), int(units[hpos + 1])
        assert ha & 3 == 1 and hb & 3 == 2
        g = int(g_base[hpos // 2048]) + ((hb >> 2) & 0xfff)
        base = (ha >> 2) | ((hb >> 14) << 30)
        index = base + ((u >> 10) & 0x3fff)
        cd = u >> 24
        local, reject = bool(u & 4), bool(u & (1 << 9))
        commit = (0 if cd == 255 else index + cd) if local else index - cd
        out.append((g, (u >> 6) & 7, REC_LOCAL if local else (REC_REJECT if reject else 0), 0, index, commit))
        if reject:
            pl = int(units[i + 1])
            assert pl & 3 == 3 and (pl >> 2) & (1 << 29)
            d = (pl >> 2) & ((1 << 29) - 1)
            if d >= 1 << 28:
                d -= 1 << 29
            out.append((g, (u >> 6) & 7, REC_EXT, 0, (index + d) & ((1 << 64) - 1), 0))
    return np.array(out, dtype=APPEND_RESP_DTYPE)


def declared_symbols() -> list[str]:
    """Every function include/raftgpu.h declares (parsed from the header text)."""
    with open(HEADER_PATH, encoding="utf-8") as f:
        text = f.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(raftgpu_[a-z0-9_]+)\s*\(", text)))


_lib = None


def lib() -> C.CDLL:
    """Load libraftgpu.so; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: run __graft_entry__.build() / make -C raft-rs_b200")
        L = C.CDLL(LIB_PATH)
        vp, u32, i32, u64 = C.c_void_p, C.c_uint32, C.c_int32, C.c_uint64
        sig = {
            "raftgpu_strerror": ([i32], C.c_char_p),
            "raftgpu_abi_version": ([], u32),
            "raftgpu_arena_create": ([i32, u32, u32, u32, u32, C.POINTER(vp)], i32),
            "raftgpu_arena_destroy": ([vp], i32),
            "raftgpu_arena_info": ([vp, C.POINTER(Info)], i32),
            "raftgpu_last_error": ([vp], C.c_char_p),
            "raftgpu_group_alloc": ([vp, C.POINTER(u32)], i32),
            "raftgpu_group_alloc_range": ([vp, u32, C.POINTER(u32)], i32),
            "raftgpu_group_alloc_wide": ([vp, C.POINTER(u32)], i32),
            "raftgpu_group_free": ([vp, u32], i32),
            "raftgpu_group_set_conf": ([vp, u32, u32, u32, u32, i32, u64], i32),
            "raftgpu_group_reset": ([vp, u32, u64, u64, u64, u64], i32),
            "raftgpu_group_become_leader": ([vp, u32], i32),
            "raftgpu_group_set_log_bounds": ([vp, u32, u64, u64], i32),
            "raftgpu_group_commit_to": ([vp, u32, u64], i32),
            "raftgpu_group_get": ([vp, u32, C.POINTER(GroupState)], i32),
            "raftgpu_progress_get": ([vp, u32, u32, C.POINTER(Progress)], i32),
            "raftgpu_progress_set": ([vp, u32, u32, C.POINTER(Progress)], i32),
            "raftgpu_progress_op": ([vp, u32, u32, i32, u64, u64, u64, C.POINTER(i32)], i32),
            "raftgpu_has_quorum": ([vp, u32, u32, C.POINTER(i32)], i32),
            "raftgpu_quorum_recently_active": ([vp, u32, u32, C.POINTER(i32)], i32),
            "raftgpu_group_maybe_commit_to": ([vp, u32, u64, C.POINTER(i32)], i32),
            "raftgpu_set_group_commit": ([vp, u32, i32], i32),
            "raftgpu_assign_commit_group": ([vp, u32, u32, u64], i32),
            "raftgpu_column_write": ([vp, i32, u32, u32, u32, vp], i32),
            "raftgpu_column_read": ([vp, i32, u32, u32, u32, vp], i32),
            "raftgpu_maximal_committed_index": ([vp, u32, C.POINTER(u64), C.POINTER(i32)], i32),
            "raftgpu_maybe_commit": ([vp, u32, C.POINTER(i32), C.POINTER(u64)], i32),
            "raftgpu_recompute": ([vp, vp, u32, u32, vp, vp, vp, vp], i32),
            "raftgpu_apply_device": ([vp, vp, vp, u64, vp], i32),
            "raftgpu_apply_device_packed": ([vp, vp, vp, u64, vp], i32),
            "raftgpu_step_sorted_device": ([vp, vp, vp, u64, vp, vp, vp, vp], i32),
            "raftgpu_tile_index": ([vp, u64, u32, vp, u64], i32),
            "raftgpu_tile_groups": ([], u32),
            "raftgpu_enqueue_append_resp": ([vp, u32, vp, u64], i32),
            "raftgpu_enqueue_bulk": ([vp, vp, u64, u32], i32),
            "raftgpu_step_begin": ([vp, u32], i32),
            "raftgpu_step_begin_packed": ([vp, vp, u64, u32], i32),
            "raftgpu_pack_records": ([vp, u64, vp, u64, C.POINTER(u64)], i32),
            "raftgpu_compact_bound": ([u64], u64),
            "raftgpu_pack_compact": ([vp, u64, vp, u64, C.POINTER(u64), vp], i32),
            "raftgpu_step_begin_compact": ([vp, vp, u64, u32], i32),
            "raftgpu_step_begin_records": ([vp, vp, u64, u32], i32),
            "raftgpu_step_slot_results": ([vp, C.POINTER(vp), C.POINTER(u64)], i32),
            "raftgpu_compact_tile_index_device": ([vp, vp, vp, vp, vp, vp], i32),
            "raftgpu_step_compact_device": ([vp, vp, vp, vp, vp, vp, vp, vp, vp, u32], i32),
            "raftgpu_host_alloc": ([vp, u64, C.POINTER(vp)], i32),
            "raftgpu_host_free": ([vp, vp], i32),
            "raftgpu_step_wait": ([vp, C.POINTER(StepResult)], i32),
            "raftgpu_step": ([vp, u32, C.POINTER(StepResult)], i32),
            "raftgpu_step_results": ([vp, C.POINTER(vp), C.POINTER(vp)], i32),
            "raftgpu_step_record_results": ([vp, u32, vp, u64, C.POINTER(u64)], i32),
            "raftgpu_reset_votes": ([vp, u32], i32),
            "raftgpu_record_vote": ([vp, u32, u32, i32], i32),
            "raftgpu_tally_votes": ([vp, vp, u32, u32, vp], i32),
            "raftgpu_send_list_device": ([vp, vp, u32, u32, vp, vp, u64, vp], i32),
            "raftgpu_heartbeat_commits_device": ([vp, vp, u32, u32, vp], i32),
            "raftgpu_step_send_list": ([vp, vp, u64, C.POINTER(u64)], i32),
            "raftgpu_vote_result": ([vp, u32, C.POINTER(i32), C.POINTER(u32), C.POINTER(u32)], i32),
            "raftgpu_group_set_term": ([vp, u32, u64], i32),
            "raftgpu_arena_enable_inflights": ([vp, u32], i32),
            "raftgpu_inflights_get": ([vp, u32, u32, C.POINTER(u32), C.POINTER(u32), vp, u32], i32),
            "raftgpu_heartbeat_resp_device": ([vp, vp, vp, u64, vp, vp], i32),
            "raftgpu_heartbeat_resp": ([vp, vp, u64, vp], i32),
            "raftgpu_update_state_device": ([vp, vp, vp, u64, vp], i32),
            "raftgpu_update_state": ([vp, vp, u64, vp], i32),
            "raftgpu_wire_apply_device": ([vp, vp, vp, u64, vp, u64, vp], i32),
            "raftgpu_step_begin_wire": ([vp, C.POINTER(WireBatch), u32], i32),
            "raftgpu_step_wire_status": ([vp, C.POINTER(vp), C.POINTER(u64)], i32),
            "raftgpu_arena_enable_read_index": ([vp, u32], i32),
            "raftgpu_read_index_device": ([vp, vp, vp, u64, vp, vp], i32),
            "raftgpu_read_index": ([vp, vp, u64, vp, vp], i32),
            "raftgpu_read_ack_device": ([vp, vp, vp, u64], i32),
            "raftgpu_read_release_device": ([vp, vp, u32, u32, vp, u64, vp], i32),
            "raftgpu_read_release": ([vp, vp, u64, C.POINTER(u64)], i32),
            "raftgpu_heartbeat_resp_read": ([vp, vp, u64, vp, vp, u64, C.POINTER(u64)], i32),
            "raftgpu_read_index_last_ctx_device": ([vp, vp, u32, u32, vp], i32),
            "raftgpu_group_read_index_conf_changed": ([vp, u32, vp, u64, C.POINTER(u64)], i32),
            "raftgpu_read_index_get": ([vp, u32, vp, vp, vp, u32, C.POINTER(u32)], i32),
            "raftgpu_counters_read": ([vp, C.POINTER(Counters)], i32),
            "raftgpu_synchronize": ([vp], i32),
            "raftgpu_debug_read": ([vp, vp], i32),
            "raftgpu_device_alloc": ([vp, u64, C.POINTER(vp)], i32),
            "raftgpu_device_free": ([vp, vp], i32),
            "raftgpu_memcpy_h2d": ([vp, vp, vp, u64], i32),
            "raftgpu_memcpy_d2h": ([vp, vp, vp, u64], i32),
        }
        for name, (args, res) in sig.items():
            f = getattr(L, name)
            f.argtypes, f.restype = args, res
        L._signatures = sig
        _lib = L
    return _lib


_synth_lib = None


def synth_lib() -> C.CDLL:
    """libraftgpu_synth.so: the synthetic workload generator (include/raftgpu_synth.h), a
    separate library so the product .so carries no bench infrastructure."""
    global _synth_lib
    if _synth_lib is None:
        if not os.path.exists(SYNTH_LIB_PATH):
            raise RuntimeError(f"{SYNTH_LIB_PATH} is missing: run __graft_entry__.build() / make -C raft-rs_b200")
        L = C.CDLL(SYNTH_LIB_PATH)
        vp, u32, i32, u64 = C.c_void_p, C.c_uint32, C.c_int32, C.c_uint64
        L.raftgpu_synth_init.argtypes, L.raftgpu_synth_init.restype = [C.POINTER(SynthColumns), u64, u32, i32], i32
        L.raftgpu_synth_round.argtypes = [C.POINTER(SynthColumns), u64, u32, u32, vp, u64, C.POINTER(u64)]
        L.raftgpu_synth_round.restype = i32
        L.raftgpu_synth_wire_encode.argtypes = [vp, u64, vp, vp, u64, vp, C.POINTER(u64), C.POINTER(u64), vp, C.POINTER(u64)]
        L.raftgpu_synth_wire_encode.restype = i32
        _synth_lib = L
    return _synth_lib


def strerror(status: int) -> str:
    return lib().raftgpu_strerror(status).decode()


TILE_GROUPS = 256


def tile_groups() -> int:
    return int(lib().raftgpu_tile_groups())


def tile_index(packed: np.ndarray, n_packed: int, n_groups: int) -> np.ndarray:
    """raftgpu_tile_index: first packed record of every 256-group tile (+ the end)."""
    tg = int(lib().raftgpu_tile_groups())
    n_tiles = (n_groups + tg - 1) // tg
    out = np.zeros(n_tiles + 1, dtype=np.uint32)
    rc = lib().raftgpu_tile_index(packed.ctypes.data, n_packed, n_groups, out.ctypes.data, len(out))
    if rc != OK:
        raise RaftGpuError(rc, "raftgpu_tile_index")
    return out


# --------------------------------------------------------------------------- host columns

def new_columns(cap: int, n_groups: int | None = None):
    """Zeroed host-side SoA columns in the arena's layout ([SLOTS][cap] / [cap])."""
    c = types.SimpleNamespace(cap=int(cap), n_groups=int(cap if n_groups is None else n_groups))
    for name, (_, dt, per_peer) in COLUMNS.items():
        setattr(c, name, np.zeros((SLOTS, cap) if per_peer else cap, dtype=dt))
    c.term = np.zeros(cap, dtype=np.uint64)  # only the oracle's literal-log check reads it
    return c


def copy_columns(c):
    d = types.SimpleNamespace(cap=c.cap, n_groups=c.n_groups)
    for name in list(COLUMNS) + ["term"]:
        setattr(d, name, getattr(c, name).copy())
    return d


def make_meta(incoming, outgoing=0, learners=0, self_slot=0, group_commit=False) -> int:
    m = (incoming & 0xFF) | ((outgoing & 0xFF) << 8) | ((learners & 0xFF) << 16)
    if self_slot is not None:
        m |= ((self_slot & 7) << 24) | META_HAS_SELF
    if group_commit:
        m |= META_GROUP_COMMIT
    return m


# --------------------------------------------------------------------------- synthetic workload

class Synth:
    """Deterministic AppendResponse workload (SURVEY 8(d)); see csrc/synth.cpp."""

    def __init__(self, n_groups: int, seed: int, k_peers: int = 5, joint: bool = False,
                 cap: int | None = None):
        self.n_groups, self.seed, self.joint = n_groups, seed, joint
        self.k_union = 7 if joint else k_peers
        cap = n_groups if cap is None else cap
        self.cols = new_columns(cap, n_groups)
        self.sim_acked = np.zeros((SLOTS, cap), dtype=np.uint64)
        self.sim_last = np.zeros(cap, dtype=np.uint64)
        self.sim_flags = np.zeros((SLOTS, cap), dtype=np.uint8)
        self._sc = SynthColumns()
        self._sc.cap, self._sc.n_groups = cap, n_groups
        c = self.cols
        for name, arr in [("matched", c.matched), ("next_idx", c.next_idx),
                          ("peer_committed", c.peer_committed), ("pflags", c.pflags),
                          ("meta", c.meta), ("committed", c.committed),
                          ("term_start", c.term_start), ("last_index", c.last_index),
                          ("term", c.term), ("sim_acked", self.sim_acked),
                          ("sim_last", self.sim_last), ("sim_flags", self.sim_flags)]:
            setattr(self._sc, name, arr.ctypes.data)
        rc = synth_lib().raftgpu_synth_init(C.byref(self._sc), seed, k_peers, int(joint))
        if rc != OK:
            raise RaftGpuError(rc, "raftgpu_synth_init")
        # what an arena / the oracle is loaded with (rounds only advance the sim_* state)
        self.initial = self.cols
        self.round_no = 0
        self._buf = None

    def max_records_per_round(self) -> int:
        return self.n_groups * (2 * (self.k_union - 1) + 1)

    def next_round(self, out: np.ndarray | None = None) -> np.ndarray:
        """Returns a VIEW into a buffer that the next call overwrites (copy it to keep it):
        fresh host pages are expensive on the GPU boxes' VMs, so one buffer is reused."""
        if out is None:
            if self._buf is None:
                cap = min(self.max_records_per_round(), (7 if self.joint else 5) * self.n_groups + 64)
                self._buf = np.empty(cap, dtype=APPEND_RESP_DTYPE)
            out = self._buf
        n = C.c_uint64()
        rc = synth_lib().raftgpu_synth_round(C.byref(self._sc), self.seed, self.round_no, self.k_union,
                                       out.ctypes.data, len(out), C.byref(n))
        if rc != OK:
            raise RaftGpuError(rc, "raftgpu_synth_round")
        self.round_no += 1
        return out[: n.value]


# --------------------------------------------------------------------------- the arena

class Arena:
    """Thin owner of a raftgpu_arena*; every method is one C-ABI call."""

    def __init__(self, max_groups: int, device: int = 0, n_rings: int = 0, ring_records: int = 0):
        self._L = lib()
        self._h = C.c_void_p()
        rc = self._L.raftgpu_arena_create(device, max_groups, SLOTS, n_rings, ring_records,
                                          C.byref(self._h))
        if rc != OK:
            detail = self._L.raftgpu_last_error(None)
            self._h = C.c_void_p()
            raise RaftGpuError(rc, "raftgpu_arena_create", detail.decode() if detail else "")
        self.info = self.get_info()
        self.cap = self.info.cap

    # -- plumbing
    def _ck(self, rc, what):
        if rc != OK:
            detail = self._L.raftgpu_last_error(self._h)
            raise RaftGpuError(rc, what, detail.decode() if detail else "")

    def close(self):
        if self._h:
            self._L.raftgpu_arena_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def get_info(self) -> Info:
        i = Info()
        self._ck(self._L.raftgpu_arena_info(self._h, C.byref(i)), "arena_info")
        return i

    def debug_read(self) -> np.ndarray:
        out = np.zeros(8, dtype=np.uint64)
        self._ck(self._L.raftgpu_debug_read(self._h, out.ctypes.data), "debug_read")
        return out

    def synchronize(self):
        self._ck(self._L.raftgpu_synchronize(self._h), "synchronize")

    def counters(self) -> dict:
        c = Counters()
        self._ck(self._L.raftgpu_counters_read(self._h, C.byref(c)), "counters_read")
        return c.as_dict()

    def device_alloc(self, nbytes: int) -> int:
        p = C.c_void_p()
        self._ck(self._L.raftgpu_device_alloc(self._h, nbytes, C.byref(p)), "device_alloc")
        return p.value

    def device_free(self, ptr: int):
        self._ck(self._L.raftgpu_device_free(self._h, ptr), "device_free")

    def h2d(self, dptr: int, arr: np.ndarray):
        arr = np.ascontiguousarray(arr)
        self._ck(self._L.raftgpu_memcpy_h2d(self._h, dptr, arr.ctypes.data, arr.nbytes), "memcpy_h2d")

    def d2h(self, arr: np.ndarray, dptr: int):
        assert arr.flags.c_contiguous
        self._ck(self._L.raftgpu_memcpy_d2h(self._h, arr.ctypes.data, dptr, arr.nbytes), "memcpy_d2h")

    # -- group lifecycle
    def group_alloc(self) -> int:
        g = C.c_uint32()
        self._ck(self._L.raftgpu_group_alloc(self._h, C.byref(g)), "group_alloc")
        return g.value

    def group_alloc_wide(self) -> int:
        """A group of up to 16 peers = group slots g (even) and g + 1 (include/raftgpu.h)."""
        g = C.c_uint32()
        self._ck(self._L.raftgpu_group_alloc_wide(self._h, C.byref(g)), "group_alloc_wide")
        return g.value

    def group_alloc_range(self, n: int) -> int:
        g = C.c_uint32()
        self._ck(self._L.raftgpu_group_alloc_range(self._h, n, C.byref(g)), "group_alloc_range")
        return g.value

    def group_free(self, g):
        self._ck(self._L.raftgpu_group_free(self._h, g), "group_free")

    def group_set_conf(self, g, incoming, outgoing=0, learners=0, self_slot=0, next_idx=1):
        self._ck(self._L.raftgpu_group_set_conf(self._h, g, incoming, outgoing, learners,
                                                -1 if self_slot is None else self_slot, next_idx),
                 "group_set_conf")

    def group_reset(self, g, term_start, last_index, committed, persisted):
        self._ck(self._L.raftgpu_group_reset(self._h, g, term_start, last_index, committed, persisted),
                 "group_reset")

    def group_become_leader(self, g):
        self._ck(self._L.raftgpu_group_become_leader(self._h, g), "group_become_leader")

    def group_set_log_bounds(self, g, term_start, last_index):
        self._ck(self._L.raftgpu_group_set_log_bounds(self._h, g, term_start, last_index),
                 "group_set_log_bounds")

    def group_commit_to(self, g, to_commit) -> int:
        return self._L.raftgpu_group_commit_to(self._h, g, to_commit)

    def group_get(self, g) -> GroupState:
        s = GroupState()
        self._ck(self._L.raftgpu_group_get(self._h, g, C.byref(s)), "group_get")
        return s

    def progress_get(self, g, slot) -> Progress:
        p = Progress()
        self._ck(self._L.raftgpu_progress_get(self._h, g, slot, C.byref(p)), "progress_get")
        return p

    def progress_set(self, g, slot, p: Progress):
        self._ck(self._L.raftgpu_progress_set(self._h, g, slot, C.byref(p)), "progress_set")

    def progress_op(self, g, slot, op: int, a0=0, a1=0, a2=0) -> int:
        r = C.c_int32()
        self._ck(self._L.raftgpu_progress_op(self._h, g, slot, op, a0, a1, a2, C.byref(r)), "progress_op")
        return r.value

    def has_quorum(self, g, slot_mask: int) -> bool:
        r = C.c_int32()
        self._ck(self._L.raftgpu_has_quorum(self._h, g, slot_mask, C.byref(r)), "has_quorum")
        return bool(r.value)

    def quorum_recently_active(self, g, perspective_of_slot: int) -> bool:
        r = C.c_int32()
        self._ck(self._L.raftgpu_quorum_recently_active(self._h, g, perspective_of_slot, C.byref(r)),
                 "quorum_recently_active")
        return bool(r.value)

    def group_maybe_commit_to(self, g, max_index: int) -> bool:
        r = C.c_int32()
        self._ck(self._L.raftgpu_group_maybe_commit_to(self._h, g, max_index, C.byref(r)),
                 "group_maybe_commit_to")
        return bool(r.value)

    def set_group_commit(self, g, enable: bool):
        self._ck(self._L.raftgpu_set_group_commit(self._h, g, int(enable)), "set_group_commit")

    def assign_commit_group(self, g, slot, gid):
        self._ck(self._L.raftgpu_assign_commit_group(self._h, g, slot, gid), "assign_commit_group")

    # -- bulk columns
    def column_write(self, col: int, slot: int, first: int, arr: np.ndarray):
        arr = np.ascontiguousarray(arr)
        self._ck(self._L.raftgpu_column_write(self._h, col, slot, first, arr.shape[0], arr.ctypes.data),
                 "column_write")

    def column_read(self, col: int, slot: int, first: int, n: int, dtype) -> np.ndarray:
        out = np.zeros(n, dtype=dtype)
        self._ck(self._L.raftgpu_column_read(self._h, col, slot, first, n, out.ctypes.data), "column_read")
        return out

    def load_columns(self, c, first: int = 0):
        """Upload host columns (groups [0, c.n_groups)) to arena groups [first, ...)."""
        n = c.n_groups
        for name, (col, dt, per_peer) in COLUMNS.items():
            arr = getattr(c, name)
            if per_peer:
                for s in range(SLOTS):
                    self.column_write(col, s, first, arr[s, :n])
            else:
                self.column_write(col, 0, first, arr[:n])

    def read_columns(self, n: int, first: int = 0):
        c = new_columns(n, n)
        for name, (col, dt, per_peer) in COLUMNS.items():
            arr = getattr(c, name)
            if per_peer:
                for s in range(SLOTS):
                    arr[s, :] = self.column_read(col, s, first, n, dt)
            else:
                arr[:] = self.column_read(col, 0, first, n, dt)
        return c

    # -- hot path
    def maximal_committed_index(self, g):
        idx, gc = C.c_uint64(), C.c_int32()
        self._ck(self._L.raftgpu_maximal_committed_index(self._h, g, C.byref(idx), C.byref(gc)),
                 "maximal_committed_index")
        return idx.value, bool(gc.value)

    def maybe_commit(self, g):
        adv, com = C.c_int32(), C.c_uint64()
        self._ck(self._L.raftgpu_maybe_commit(self._h, g, C.byref(adv), C.byref(com)), "maybe_commit")
        return bool(adv.value), com.value

    def recompute(self, first, n, stream=None, d_adv=None, d_commit=None, d_mci=None, d_gc=None):
        self._ck(self._L.raftgpu_recompute(self._h, stream, first, n, d_adv, d_commit, d_mci, d_gc),
                 "recompute")

    def apply_device(self, d_recs, n, stream=None, d_results=None):
        self._ck(self._L.raftgpu_apply_device(self._h, stream, d_recs, n, d_results), "apply_device")

    def apply_device_packed(self, d_packed, n_packed, stream=None, d_results=None):
        self._ck(self._L.raftgpu_apply_device_packed(self._h, stream, d_packed, n_packed, d_results),
                 "apply_device_packed")

    def step_sorted_device(self, d_packed, n_packed, d_tile_off, stream=None, d_results=None, d_adv=None,
                           d_commit=None):
        self._ck(self._L.raftgpu_step_sorted_device(self._h, stream, d_packed, n_packed, d_tile_off, d_results,
                                                    d_adv, d_commit), "step_sorted_device")

    def enqueue(self, recs: np.ndarray, ring: int = 0):
        assert recs.dtype == APPEND_RESP_DTYPE and recs.flags.c_contiguous
        self._ck(self._L.raftgpu_enqueue_append_resp(self._h, ring, recs.ctypes.data, len(recs)),
                 "enqueue_append_resp")

    def enqueue_bulk(self, recs: np.ndarray, sorted_by_group: bool = False):
        assert recs.dtype == APPEND_RESP_DTYPE and recs.flags.c_contiguous
        self._ck(self._L.raftgpu_enqueue_bulk(self._h, recs.ctypes.data, len(recs),
                                              BULK_SORTED if sorted_by_group else 0), "enqueue_bulk")

    def host_alloc_packed(self, n_records: int) -> np.ndarray:
        """NUMA-local pinned buffer of packed 16-byte records (u64 pairs), owned by the arena."""
        p = C.c_void_p()
        self._ck(self._L.raftgpu_host_alloc(self._h, 16 * n_records, C.byref(p)), "host_alloc")
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint64)), shape=(n_records, 2))

    def pack_records(self, recs: np.ndarray, out: np.ndarray) -> int:
        assert recs.dtype == APPEND_RESP_DTYPE and recs.flags.c_contiguous and out.dtype == np.uint64
        n = C.c_uint64()
        self._ck(self._L.raftgpu_pack_records(recs.ctypes.data, len(recs), out.ctypes.data, out.shape[0],
                                              C.byref(n)), "pack_records")
        return n.value

    def step_begin_packed(self, packed: np.ndarray, n_packed: int, flags=0):
        self._ck(self._L.raftgpu_step_begin_packed(self._h, packed.ctypes.data, n_packed, flags),
                 "step_begin_packed")

    def host_alloc_bytes(self, n_bytes: int) -> np.ndarray:
        """NUMA-local pinned byte buffer owned by the arena (16-byte aligned)."""
        p = C.c_void_p()
        self._ck(self._L.raftgpu_host_alloc(self._h, n_bytes, C.byref(p)), "host_alloc")
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(n_bytes,))

    def compact_tile_index_device(self, d_blob, hdr_blob: np.ndarray, d_tile_off, d_bad, stream=None):
        """hdr_blob: host bytes that start with the blob's raftgpu_compact_hdr."""
        self._ck(self._L.raftgpu_compact_tile_index_device(self._h, stream, d_blob, hdr_blob.ctypes.data, d_tile_off,
                                                           d_bad), "compact_tile_index_device")

    def step_compact_device(self, d_blob, hdr_blob: np.ndarray, d_tile_off, stream=None, d_results=None, d_adv=None,
                            d_commit=None, d_dup=None, ordered=False):
        self._ck(self._L.raftgpu_step_compact_device(self._h, stream, d_blob, hdr_blob.ctypes.data, d_tile_off,
                                                     d_results, d_adv, d_commit, d_dup, 1 if ordered else 0),
                 "step_compact_device")

    def host_free(self, buf: np.ndarray):
        self._ck(self._L.raftgpu_host_free(self._h, buf.ctypes.data), "host_free")

    def step_begin_records(self, recs: np.ndarray, flags=0):
        assert recs.dtype == APPEND_RESP_DTYPE and recs.flags.c_contiguous
        self._ck(self._L.raftgpu_step_begin_records(self._h, recs.ctypes.data, len(recs), flags), "step_begin_records")

    def step_begin_compact(self, blob: np.ndarray, n_bytes: int, flags=0):
        self._ck(self._L.raftgpu_step_begin_compact(self._h, blob.ctypes.data, n_bytes, flags),
                 "step_begin_compact")

    def step_begin(self, flags=0):
        self._ck(self._L.raftgpu_step_begin(self._h, flags), "step_begin")

    # -- Inflights on the device (SURVEY 8(f) rank 2)
    def enable_inflights(self, max_inflight: int):
        self._ck(self._L.raftgpu_arena_enable_inflights(self._h, max_inflight), "arena_enable_inflights")
        self.ins_cap = max_inflight

    def inflights_get(self, g, slot):
        """(start, count, ring u64[cap]) of one peer's window."""
        st, cnt = C.c_uint32(), C.c_uint32()
        buf = np.zeros(self.ins_cap, dtype=np.uint64)
        self._ck(self._L.raftgpu_inflights_get(self._h, g, slot, C.byref(st), C.byref(cnt), buf.ctypes.data, self.ins_cap),
                 "inflights_get")
        return st.value, cnt.value, buf

    # -- heartbeat responses / update_state (SURVEY 8(f) ranks 3 and 2)
    def heartbeat_resp(self, recs: np.ndarray) -> np.ndarray:
        """raftgpu_heartbeat_resp: REC_HEARTBEAT records -> result bytes (RES_OK | RES_SEND | RES_NO_PROGRESS)."""
        assert recs.dtype == APPEND_RESP_DTYPE and recs.flags.c_contiguous
        res = np.zeros(len(recs), dtype=np.uint8)
        self._ck(self._L.raftgpu_heartbeat_resp(self._h, recs.ctypes.data, len(recs), res.ctypes.data), "heartbeat_resp")
        return res

    def update_state(self, entries: np.ndarray) -> np.ndarray:
        """raftgpu_update_state: send entries with next_idx = last -> result bytes."""
        assert entries.dtype == SEND_ENTRY_DTYPE and entries.flags.c_contiguous
        res = np.zeros(len(entries), dtype=np.uint8)
        self._ck(self._L.raftgpu_update_state(self._h, entries.ctypes.data, len(entries), res.ctypes.data), "update_state")
        return res

    # -- wire path (SURVEY 8(f4))
    def group_set_term(self, g, term):
        self._ck(self._L.raftgpu_group_set_term(self._h, g, term), "group_set_term")

    def step_begin_wire(self, batch, flags=0):
        """batch: anything with .bytes (u8 array), .n_bytes, .offsets (u32 array), .n, .records (24-byte records or
        None), .n_records -- e.g. wire.WireBuffers.  The arrays must stay alive and untouched until step_wait."""
        wb = WireBatch(batch.bytes.ctypes.data, batch.n_bytes, batch.offsets.ctypes.data, batch.n,
                       batch.records.ctypes.data if batch.n_records else None, batch.n_records)
        self._ck(self._L.raftgpu_step_begin_wire(self._h, C.byref(wb), flags), "step_begin_wire")

    def wire_status(self) -> np.ndarray:
        """Status bytes (RAFTGPU_WIRE_* << 4 | RAFTGPU_RES_*) of the last completed wire step (a view)."""
        p, n = C.c_void_p(), C.c_uint64()
        self._ck(self._L.raftgpu_step_wire_status(self._h, C.byref(p), C.byref(n)), "step_wire_status")
        if n.value == 0:
            return np.zeros(0, dtype=np.uint8)
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(n.value,))

    def wire_apply_device(self, d_bytes, n_bytes, d_offsets, n, d_status, stream=None):
        self._ck(self._L.raftgpu_wire_apply_device(self._h, stream, d_bytes, n_bytes, d_offsets, n, d_status), "wire_apply_device")

    def step_wait(self, check: bool = True) -> StepResult:
        r = StepResult()
        rc = self._L.raftgpu_step_wait(self._h, C.byref(r))
        if check:
            self._ck(rc, "step_wait")
        r.status = rc
        return r

    def step(self, flags=0) -> StepResult:
        r = StepResult()
        self._ck(self._L.raftgpu_step(self._h, flags, C.byref(r)), "step")
        return r

    def step_results(self, n_groups: int):
        """(adv_bitmap u32[], committed u64[] | None) views into the arena's pinned results."""
        pa, pc = C.c_void_p(), C.c_void_p()
        self._ck(self._L.raftgpu_step_results(self._h, C.byref(pa), C.byref(pc)), "step_results")
        words = (n_groups + 31) // 32
        bm = np.ctypeslib.as_array(C.cast(pa, C.POINTER(C.c_uint32)), shape=(words,))
        com = np.ctypeslib.as_array(C.cast(pc, C.POINTER(C.c_uint64)), shape=(n_groups,)) if pc.value else None
        return bm, com

    def slot_results(self) -> np.ndarray:
        """Result bytes of the last zero-copy step, one per packed record / compact unit (a view)."""
        p, n = C.c_void_p(), C.c_uint64()
        self._ck(self._L.raftgpu_step_slot_results(self._h, C.byref(p), C.byref(n)), "step_slot_results")
        if n.value == 0:
            return np.zeros(0, dtype=np.uint8)
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(n.value,))

    def record_results(self, ring: int = 0) -> np.ndarray:
        """Result bytes of the records enqueued on `ring` in the last step, in enqueue order."""
        n = C.c_uint64()
        self._ck(self._L.raftgpu_step_record_results(self._h, ring, None, 0, C.byref(n)),
                 "step_record_results")
        out = np.zeros(n.value, dtype=np.uint8)
        if n.value:
            self._ck(self._L.raftgpu_step_record_results(self._h, ring, out.ctypes.data, n.value,
                                                         C.byref(n)), "step_record_results")
        return out

    # -- ReadIndex (ReadOnly queues in HBM)
    def enable_read_index(self, max_pending: int):
        self._ck(self._L.raftgpu_arena_enable_read_index(self._h, max_pending), "arena_enable_read_index")
        self.rd_cap = max_pending

    def read_index(self, reqs: np.ndarray, check: bool = True):
        """raftgpu_read_index: requests -> (status bytes, read indexes).  check=False returns a SPLIT batch's results
        instead of raising."""
        assert reqs.dtype == READ_REQ_DTYPE and reqs.flags.c_contiguous
        st, idx = np.zeros(len(reqs), dtype=np.uint8), np.zeros(len(reqs), dtype=np.uint64)
        rc = self._L.raftgpu_read_index(self._h, reqs.ctypes.data, len(reqs), st.ctypes.data, idx.ctypes.data)
        if check or rc != ERR_INVALID:
            self._ck(rc, "read_index")
        return st, idx

    def read_release(self, capacity: int):
        """raftgpu_read_release -> (states, complete: False when groups did not fit and wait for the next call)."""
        out, n = np.zeros(capacity, dtype=READ_STATE_DTYPE), C.c_uint64()
        rc = self._L.raftgpu_read_release(self._h, out.ctypes.data if capacity else None, capacity, C.byref(n))
        if rc != ERR_FULL:
            self._ck(rc, "read_release")
        return out[: n.value], rc == OK

    def heartbeat_resp_read(self, recs: np.ndarray, capacity: int):
        """raftgpu_heartbeat_resp_read -> (result bytes, released states, complete)."""
        assert recs.dtype == APPEND_RESP_DTYPE and recs.flags.c_contiguous
        res, out, n = np.zeros(len(recs), dtype=np.uint8), np.zeros(capacity, dtype=READ_STATE_DTYPE), C.c_uint64()
        rc = self._L.raftgpu_heartbeat_resp_read(self._h, recs.ctypes.data, len(recs), res.ctypes.data,
                                                 out.ctypes.data if capacity else None, capacity, C.byref(n))
        if rc != ERR_FULL:
            self._ck(rc, "heartbeat_resp_read")
        return res, out[: n.value], rc == OK

    def read_index_device(self, d_reqs, n, d_status, d_index=None, stream=None):
        self._ck(self._L.raftgpu_read_index_device(self._h, stream, d_reqs, n, d_status, d_index), "read_index_device")

    def read_ack_device(self, d_records, n, stream=None):
        self._ck(self._L.raftgpu_read_ack_device(self._h, stream, d_records, n), "read_ack_device")

    def read_release_device(self, first, n, d_out, capacity, d_count, stream=None):
        self._ck(self._L.raftgpu_read_release_device(self._h, stream, first, n, d_out, capacity, d_count),
                 "read_release_device")

    def read_index_last_ctx_device(self, first, n, d_out, stream=None):
        self._ck(self._L.raftgpu_read_index_last_ctx_device(self._h, stream, first, n, d_out), "read_index_last_ctx_device")

    def read_index_conf_changed(self, g, capacity: int = 64) -> np.ndarray:
        out, n = np.zeros(capacity, dtype=READ_STATE_DTYPE), C.c_uint64()
        self._ck(self._L.raftgpu_group_read_index_conf_changed(self._h, g, out.ctypes.data, capacity, C.byref(n)),
                 "group_read_index_conf_changed")
        return out[: n.value]

    def read_index_get(self, g):
        """One group's pending requests in queue order: (ctx u64[], index u64[], word u32[])."""
        cap = self.rd_cap
        ctx, idx, word, n = (np.zeros(cap, dtype=np.uint64), np.zeros(cap, dtype=np.uint64),
                             np.zeros(cap, dtype=np.uint32), C.c_uint32())
        self._ck(self._L.raftgpu_read_index_get(self._h, g, ctx.ctypes.data, idx.ctypes.data, word.ctypes.data, cap,
                                                C.byref(n)), "read_index_get")
        return ctx[: n.value], idx[: n.value], word[: n.value]

    # -- votes
    def reset_votes(self, g):
        self._ck(self._L.raftgpu_reset_votes(self._h, g), "reset_votes")

    def record_vote(self, g, slot, vote: bool):
        self._ck(self._L.raftgpu_record_vote(self._h, g, slot, int(vote)), "record_vote")

    def send_list_device(self, first, n, d_adv, d_out, capacity, d_count, stream=None):
        self._ck(self._L.raftgpu_send_list_device(self._h, stream, first, n, d_adv, d_out, capacity, d_count),
                 "send_list_device")

    def heartbeat_commits_device(self, first, n, d_out, stream=None):
        self._ck(self._L.raftgpu_heartbeat_commits_device(self._h, stream, first, n, d_out), "heartbeat_commits_device")

    def step_send_list(self, capacity: int) -> np.ndarray:
        """Post-commit send decisions of the last completed step (raftgpu_step_send_list)."""
        out = np.zeros(capacity, dtype=SEND_ENTRY_DTYPE)
        n = C.c_uint64()
        self._ck(self._L.raftgpu_step_send_list(self._h, out.ctypes.data, capacity, C.byref(n)), "step_send_list")
        return out[: n.value]

    def tally_votes(self, first, n, d_out, stream=None):
        self._ck(self._L.raftgpu_tally_votes(self._h, stream, first, n, d_out), "tally_votes")

    def vote_result(self, g):
        r, gr, rj = C.c_int32(), C.c_uint32(), C.c_uint32()
        self._ck(self._L.raftgpu_vote_result(self._h, g, C.byref(r), C.byref(gr), C.byref(rj)),
                 "vote_result")
        return gr.value, rj.value, r.value
