"""ReadIndex on the device (raftgpu_arena_enable_read_index): the reference's read-index tests replayed through the C-ABI,
random traffic against the arena-form oracle (tests/read_index_oracle.py, itself checked against the literal restatement
of read_only.rs), the release pass's capacity contract, and that enabling read index changes nothing else."""
import ctypes as C
import types

import numpy as np
import pytest

import read_index_oracle as R
from helpers import B, O, assert_columns_equal

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------- scenarios

class GpuDriver:
    """One leader group of a real arena, driven through the C-ABI: the host forms for requests and releases, the
    device form for acks (a batch may ack one cell twice, which the tracker part of raftgpu_heartbeat_resp_read
    refuses)."""

    def __init__(self, max_pending=64):
        self.a = B.Arena(256)
        self.a.enable_read_index(max_pending)
        self.g = self.a.group_alloc()
        self.d_recs = self.a.device_alloc(24 * 64)

    def set_conf(self, incoming, outgoing=0, learners=0, self_slot=0):
        self.a.group_set_conf(self.g, incoming, outgoing, learners, self_slot)

    def set_log(self, committed, term_start, last_index):
        self.a.group_set_log_bounds(self.g, term_start, last_index)
        self.a.column_write(B.COL_COMMITTED, 0, self.g, np.array([committed], dtype=np.uint64))

    def reset(self):
        s = self.a.group_get(self.g)
        self.a.group_reset(self.g, s.term_start, s.last_index, s.committed, s.last_index)

    def request(self, ctx, from_slot=None, lease=False):
        r = np.zeros(1, dtype=B.READ_REQ_DTYPE)
        r["group"], r["ctx"], r["from_slot"] = self.g, ctx, 0 if from_slot is None else from_slot
        r["flags"] = (B.READ_LOCAL if from_slot is None else 0) | (B.READ_LEASE if lease else 0)
        st, idx = self.a.read_index(r)
        return int(st[0]), int(idx[0])

    def acks(self, pairs):
        recs = np.zeros(len(pairs), dtype=B.APPEND_RESP_DTYPE)
        for i, (slot, ctx) in enumerate(pairs):
            recs[i]["group"], recs[i]["peer_slot"], recs[i]["index"] = self.g, slot, ctx
            recs[i]["flags"] = B.REC_HEARTBEAT | B.REC_READ_CTX
        if len(recs):
            self.a.h2d(self.d_recs, recs)
        self.a.read_ack_device(self.d_recs, len(recs))
        st, complete = self.a.read_release(64)
        assert complete
        return R.states_to_list(st)

    def conf_changed(self):
        return R.states_to_list(self.a.read_index_conf_changed(self.g))

    def pending(self):
        return [int(c) for c in self.a.read_index_get(self.g)[0]]


@pytest.mark.parametrize("name", sorted(R.SCENARIOS))
def test_reference_scenario_on_gpu(name):
    d = GpuDriver()
    try:
        R.SCENARIOS[name](d)
    finally:
        d.a.close()


def test_heartbeat_resp_read_runs_the_whole_handler():
    """raftgpu_heartbeat_resp_read = the tracker part (same result bytes and columns as raftgpu_heartbeat_resp), recv_ack,
    release; and the last pending context is what bcast_heartbeat attaches."""
    d = GpuDriver()
    a, g = d.a, d.g
    a.group_set_conf(g, 0b11111, 0, 0, 0, 1)
    d.set_log(7, 3, 9)
    assert [d.request(c, 1)[0] for c in (5, 6)] == [R.QUEUED, R.QUEUED]
    d_last = a.device_alloc(8)
    a.read_index_last_ctx_device(g, 1, d_last)
    last = np.zeros(1, dtype=np.uint64)
    a.d2h(last, d_last)
    assert last.tolist() == [6]
    recs = np.zeros(3, dtype=B.APPEND_RESP_DTYPE)
    recs["group"], recs["peer_slot"], recs["commit"] = g, [1, 2, 3], 7
    recs["flags"] = B.REC_HEARTBEAT | B.REC_READ_CTX
    recs["index"] = [5, 6, 5]
    res, states, complete = a.heartbeat_resp_read(recs, 8)
    assert complete and res.tolist() == [B.RES_OK | B.RES_SEND] * 3
    # ctx 5 has {0, 1, 3}: a quorum of five, released; ctx 6 only {0, 2}
    assert R.states_to_list(states) == [(1, 7, 5)]
    assert d.pending() == [6]
    for s in (1, 2, 3):
        assert a.progress_get(g, s).committed_index == 7 and a.progress_get(g, s).recent_active
    a.close()


# ---------------------------------------------------------------------------------------------- random traffic

def _snapshot(a, hi):
    """The per-group columns the read passes look at, as they are on the device."""
    c = types.SimpleNamespace(meta=np.zeros(a.cap, dtype=np.uint32))
    c.meta[:hi] = a.column_read(B.COL_META, 0, 0, hi, np.uint32)
    for name, col in (("committed", B.COL_COMMITTED), ("term_start", B.COL_TERM_START), ("last_index", B.COL_LAST_INDEX)):
        setattr(c, name, np.zeros(a.cap, dtype=np.uint64))
        getattr(c, name)[:hi] = a.column_read(col, 0, 0, hi, np.uint64)
    return c


def _lo_key(states, meta):
    g = states["group"].astype(np.int64)
    return np.where((meta[g] & R.WIDE_HI) != 0, g - 1, g)


def _check_release(got, want, meta, what):
    """Same states; each group's states contiguous and in queue order; groups in any order."""
    key = _lo_key(got, meta)
    runs = 1 + int(np.count_nonzero(key[1:] != key[:-1])) if len(key) else 0
    assert runs == len(np.unique(key)), f"{what}: a group's states are not contiguous"
    order = np.argsort(key, kind="stable")
    assert np.array_equal(got[order], want), what


def _build_mixed(n, P, rng):
    """n plain groups (5 voters, 5 % joint over 7 slots, 5 % with learners, self slot random) and n / 1000 wide groups
    (peers on both halves, the self slot on either).  Returns (arena, oracle, logical groups, wide lows)."""
    a = B.Arena(n + 2 * (n // 1000) + 256)
    a.enable_read_index(P)
    assert a.group_alloc_range(n) == 0
    meta = np.array([B.make_meta(0x1F, self_slot=int(s)) for s in range(5)], dtype=np.uint32)[rng.integers(0, 5, n)]
    kind = rng.random(n)
    meta[kind < 0.05] = B.make_meta(0x1F, 0b1110001, 0, 0)
    meta[(kind >= 0.05) & (kind < 0.10)] = B.make_meta(0x1F, 0, 0x60, 1)
    a.column_write(B.COL_META, 0, 0, meta)
    wides = []
    for k in range(n // 1000):
        g = a.group_alloc_wide()
        a.group_set_conf(g, 0x0307, 0x0C03 if k % 3 == 0 else 0, 0x0400, 9 if k % 2 else 0)
        wides.append(g)
    hi = a.get_info().hi
    li = rng.integers(10, 1000, hi).astype(np.uint64)
    cm = li - rng.integers(0, 3, hi).astype(np.uint64)
    u = rng.random(hi)
    ts = np.where(u < 0.8, rng.integers(1, 10, hi).astype(np.uint64), np.uint64(R.U64_MAX))
    ts = np.where((u >= 0.8) & (u < 0.85), cm + np.uint64(1), ts)              # nothing committed in the term yet
    for g in wides:
        li[g + 1], cm[g + 1], ts[g + 1] = li[g], cm[g], ts[g]
    a.column_write(B.COL_LAST_INDEX, 0, 0, li)
    a.column_write(B.COL_COMMITTED, 0, 0, cm)
    a.column_write(B.COL_TERM_START, 0, 0, ts)
    ar = R.ArenaReads(a.cap, P)
    ar.alloc(0, hi)
    return a, ar, np.concatenate([np.arange(n), np.array(wides, dtype=np.int64)]), np.array(wides, dtype=np.int64)


def _requests(rng, groups, wides, hi, ar, snap):
    k = len(groups) // 2
    sel = rng.permutation(groups)[:k]
    reps = np.where(rng.random(k) < 0.7, 1, rng.integers(2, 4, k))
    g = np.repeat(sel, reps)
    m = len(g)
    r = np.zeros(m + 4, dtype=B.READ_REQ_DTYPE)
    local = rng.random(m) < 0.3
    frm = rng.integers(1, 5, m)
    is_wide = np.isin(g, wides)
    wslot = np.array([1, 2, 8, 9, 10])[rng.integers(0, 5, m)]
    frm = np.where(is_wide, wslot, frm)
    r["group"][:m] = np.where(is_wide & ~local & (frm >= 8), g + 1, g)
    r["from_slot"][:m] = np.where(local, 0, frm % 8)
    r["flags"][:m] = np.where(local, B.READ_LOCAL, 0) | np.where(rng.random(m) < 0.05, B.READ_LEASE, 0)
    r["ctx"][:m] = rng.integers(0, 6, m)
    r["group"][m:] = [hi + 3, 0, hi + 100, 1]          # unallocated groups, slot 9: INVALID
    r["from_slot"][m:] = [1, 9, 1, 2]
    return r


def _acks(rng, groups, wides, ar):
    k = len(groups) // 2
    sel = rng.permutation(groups)[:k]
    is_wide = np.isin(sel, wides)
    slots = rng.random((k, 7)).argsort(axis=1)[:, :4] + 1                  # 4 distinct peers of 1..7
    wslots = np.array([0, 1, 2, 8, 9, 10, 11])[rng.random((k, 7)).argsort(axis=1)[:, :4]]
    slots = np.where(is_wide[:, None], wslots, slots).ravel()
    g = np.repeat(sel, 4)
    head, cnt = ar.head_count(g)
    u = rng.random(len(g))
    live_last = ar.ctx[ar.pos(head, np.maximum(cnt - 1, 0)), g]
    live_first = ar.ctx[head % ar.P, g]
    ctx = np.where(u < 0.7, live_last, np.where(u < 0.85, live_first, rng.integers(0, 6, len(g)).astype(np.uint64)))
    recs = np.zeros(len(g), dtype=B.APPEND_RESP_DTYPE)
    recs["group"] = g + slots // 8
    recs["peer_slot"] = slots % 8
    recs["flags"] = B.REC_HEARTBEAT | np.where(rng.random(len(g)) < 0.9, B.REC_READ_CTX, 0)
    recs["index"] = ctx
    return recs


@pytest.mark.parametrize("n,P", [(100_000, 2), (1_000_000, 4)])
def test_random_traffic_vs_arena_oracle(n, P):
    """Ticks of: the log moving (committed / term_start / last_index columns), requests (local, forwarded, lease,
    duplicate tokens, non-leaders, unallocated groups; max_pending small enough to hit FULL), heartbeat responses acking
    live and stale contexts from voters, learners and absent slots (some without a context), then occasional
    set_conf + conf_changed and reset.  Compared after every tick: status bytes, read indexes, the release list,
    last_ctx of every group and sampled queues."""
    rng = np.random.default_rng(n + P)
    a, ar, groups, wides = _build_mixed(n, P, rng)
    hi = a.get_info().hi
    cap_out = 2 * hi
    d_req = a.device_alloc(16 * (hi + 8))
    d_st, d_idx = a.device_alloc(hi + 8), a.device_alloc(8 * (hi + 8))
    d_rec = a.device_alloc(24 * 4 * hi)
    d_out, d_cnt, d_last = a.device_alloc(24 * cap_out), a.device_alloc(16), a.device_alloc(8 * hi)
    seen = {s: 0 for s in range(7)}
    n_released = 0
    for tick in range(3):
        move = rng.choice(groups, len(groups) // 10, replace=False)
        snap = _snapshot(a, hi)
        cm = snap.committed[:hi].copy()
        cm[move] = np.minimum(cm[move] + np.uint64(1), snap.last_index[move])
        for g in wides:
            cm[g + 1] = cm[g]
        a.column_write(B.COL_COMMITTED, 0, 0, cm)
        snap = _snapshot(a, hi)
        reqs = _requests(rng, groups, wides, hi, ar, snap)
        a.h2d(d_req, reqs)
        a.read_index_device(d_req, len(reqs), d_st, d_idx)
        st, idx = np.zeros(len(reqs), dtype=np.uint8), np.zeros(len(reqs), dtype=np.uint64)
        a.d2h(st, d_st)
        a.d2h(idx, d_idx)
        want_st, want_idx = ar.read_index(reqs, snap, hi)
        assert np.array_equal(st, want_st), (tick, np.flatnonzero(st != want_st)[:5])
        assert np.array_equal(idx, want_idx), tick
        for s in range(7):
            seen[s] += int(np.count_nonzero(st == s))
        recs = _acks(rng, groups, wides, ar)
        a.h2d(d_rec, recs)
        a.read_ack_device(d_rec, len(recs))
        a.read_release_device(0, hi, d_out, cap_out, d_cnt)
        cnt = np.zeros(2, dtype=np.uint64)
        a.d2h(cnt, d_cnt)
        assert cnt[0] == cnt[1] <= cap_out
        got = np.zeros(int(cnt[1]), dtype=B.READ_STATE_DTYPE)
        if len(got):
            a.d2h(got, d_out)
        ar.ack(recs, snap)
        want = ar.release(snap, 0, hi)
        _check_release(got, want, snap.meta, f"release tick {tick}")
        n_released += len(got)
        # configuration changes + the post_conf_change tail, resets
        for g in rng.choice(n, 4, replace=False):
            g = int(g)
            old = int(snap.meta[g])
            self_slot = (old >> 24) & 7
            incoming = (1 << self_slot) | int(rng.integers(0, 32))
            a.group_set_conf(g, incoming, 0, 0, self_slot)
            was = (old & 0xFF) | ((old >> 8) & 0xFF) | ((old >> 16) & 0xFF)
            ar.clear_slots(g, was & ~incoming)
            snap.meta[g] = B.make_meta(incoming, 0, 0, self_slot)
            assert np.array_equal(a.read_index_conf_changed(g), ar.conf_changed(snap, g)), (tick, g)
        for g in rng.choice(n, 4, replace=False):
            g = int(g)
            a.group_reset(g, int(snap.term_start[g]), int(snap.last_index[g]), int(snap.committed[g]), 0)
            ar.reset(g)
        a.read_index_last_ctx_device(0, hi, d_last)
        last = np.zeros(hi, dtype=np.uint64)
        a.d2h(last, d_last)
        assert np.array_equal(last, ar.last_ctx(0, hi)), tick
        for g in rng.choice(groups, 30, replace=False):
            got_q, want_q = a.read_index_get(int(g)), ar.queue(int(g))
            for x, y in zip(got_q, want_q):
                assert np.array_equal(x, y), (tick, int(g))
    assert n_released > n // 10
    assert all(seen[s] for s in (R.DROPPED, R.READY, R.QUEUED, R.ALREADY_PENDING, R.FULL, R.INVALID)), seen
    a.close()


# ---------------------------------------------------------------------------------------------- capacity

def test_release_into_a_small_buffer_loses_nothing():
    n = 8192
    a = B.Arena(n)
    a.enable_read_index(4)
    a.group_alloc_range(n)
    meta = np.full(n, B.make_meta(0b111, self_slot=0), dtype=np.uint32)
    a.column_write(B.COL_META, 0, 0, meta)
    for col in (B.COL_COMMITTED, B.COL_TERM_START, B.COL_LAST_INDEX):
        a.column_write(col, 0, 0, np.full(n, 5, dtype=np.uint64))
    snap = _snapshot(a, n)
    ar = R.ArenaReads(a.cap, 4)
    ar.alloc(0, n)
    reqs = np.zeros(2 * n, dtype=B.READ_REQ_DTYPE)
    reqs["group"] = np.repeat(np.arange(n), 2)
    reqs["from_slot"], reqs["ctx"] = 1, np.tile([10, 11], n)
    st, _ = a.read_index(reqs)
    assert np.array_equal(st, ar.read_index(reqs, snap, n)[0]) and np.all(st == R.QUEUED)
    recs = np.zeros(n, dtype=B.APPEND_RESP_DTYPE)
    recs["group"], recs["peer_slot"], recs["index"] = np.arange(n), 2, 11
    recs["flags"] = B.REC_HEARTBEAT | B.REC_READ_CTX
    d_rec, d_out, d_cnt = a.device_alloc(24 * n), a.device_alloc(24 * 2 * n), a.device_alloc(16)
    a.h2d(d_rec, recs)
    a.read_ack_device(d_rec, n)
    ar.ack(recs, snap)
    want = ar.release(snap, 0, n)
    assert len(want) == 2 * n
    parts, cnt = [], np.zeros(2, dtype=np.uint64)
    a.read_release_device(0, n, d_out, 1000, d_cnt)
    a.d2h(cnt, d_cnt)
    assert cnt[0] > 1000 >= cnt[1] > 0
    part = np.zeros(int(cnt[1]), dtype=B.READ_STATE_DTYPE)
    a.d2h(part, d_out)
    parts.append(part)
    # the host form: a small buffer again (ERR_FULL = call again), then the rest
    states, complete = a.read_release(3000)
    assert not complete and 0 < len(states) <= 3000
    parts.append(states)
    states, complete = a.read_release(2 * n)
    assert complete
    parts.append(states)
    assert a.read_release(2 * n)[0].size == 0
    got = np.concatenate(parts)
    _check_release(got[np.argsort(got["group"], kind="stable")], want, snap.meta, "union of the partial releases")
    a.close()


# ---------------------------------------------------------------------------------------------- nothing else changes

def test_enabling_read_index_changes_nothing_else():
    """Heartbeat records with and without REC_READ_CTX through raftgpu_heartbeat_resp give the same result bytes and
    columns on an enabled arena as plain records on a plain arena; a step on an enabled arena still runs the fused tile
    kernel (raftgpu_step_sorted_device, which refuses arenas that cannot) and computes the same columns."""
    n = 4096
    synth = B.Synth(n, seed=0x2EAD, k_peers=5)
    plain, rd = B.Arena(n), B.Arena(n)
    rd.enable_read_index(8)
    for a in (plain, rd):
        a.group_alloc_range(n)
        a.load_columns(synth.initial)
    ref = O.copy_columns(synth.initial)
    rng = np.random.default_rng(3)
    pk = np.zeros((2 * 6 * n + 8, 2), dtype=np.uint64)
    for rnd in range(2):
        recs = synth.next_round().copy()
        k = plain.pack_records(recs, pk)
        off = B.tile_index(pk, k, n)
        O.arena_apply(ref, recs, mode=0)
        O.arena_recompute(ref)
        for a in (plain, rd):
            d_pk, d_off = a.device_alloc(pk.nbytes), a.device_alloc(off.nbytes)
            a.h2d(d_pk, pk)
            a.h2d(d_off, off)
            a.step_sorted_device(d_pk, k, d_off)
            a.synchronize()
            assert_columns_equal(a.read_columns(n), ref, n, f"fused step {rnd}")
        g = rng.integers(0, n, n // 2).astype(np.uint32)
        s = rng.integers(1, 5, n // 2).astype(np.uint8)
        _, first = np.unique(g.astype(np.uint64) * 8 + s, return_index=True)
        hb = np.zeros(len(first), dtype=B.APPEND_RESP_DTYPE)
        hb["group"], hb["peer_slot"], hb["commit"] = g[first], s[first], ref.committed[g[first]]
        hb["flags"] = B.REC_HEARTBEAT
        hb_ctx = hb.copy()
        hb_ctx["flags"][::2] |= B.REC_READ_CTX
        hb_ctx["index"][::2] = 77
        want = O.arena_apply_heartbeat(ref, hb)
        assert np.array_equal(plain.heartbeat_resp(hb), want)
        assert np.array_equal(rd.heartbeat_resp(hb_ctx), want)
        for a in (plain, rd):
            assert_columns_equal(a.read_columns(n), ref, n, f"heartbeats {rnd}")
    plain.close()
    rd.close()


def test_every_read_entry_point_refuses_a_plain_arena():
    a = B.Arena(256)
    g = a.group_alloc()
    L, h = a._L, a._h
    n = C.c_uint64()
    n32 = C.c_uint32()
    buf = a.device_alloc(4096)
    calls = [
        L.raftgpu_read_index_device(h, None, buf, 1, buf, buf),
        L.raftgpu_read_index(h, buf, 0, None, None),
        L.raftgpu_read_ack_device(h, None, buf, 1),
        L.raftgpu_read_release_device(h, None, 0, 1, buf, 1, buf),
        L.raftgpu_read_release(h, None, 0, C.byref(n)),
        L.raftgpu_heartbeat_resp_read(h, None, 0, None, None, 0, C.byref(n)),
        L.raftgpu_read_index_last_ctx_device(h, None, 0, 1, buf),
        L.raftgpu_group_read_index_conf_changed(h, g, None, 0, C.byref(n)),
        L.raftgpu_read_index_get(h, g, None, None, None, 0, C.byref(n32)),
    ]
    assert calls == [B.ERR_INVALID] * len(calls)
    # enabling is refused after groups exist, and outside 1..64
    assert L.raftgpu_arena_enable_read_index(h, 8) == B.ERR_INVALID
    b = B.Arena(256)
    assert b._L.raftgpu_arena_enable_read_index(b._h, 0) == B.ERR_INVALID
    assert b._L.raftgpu_arena_enable_read_index(b._h, 65) == B.ERR_INVALID
    info0 = b.get_info().device_bytes
    b.enable_read_index(8)
    assert b.get_info().device_bytes - info0 == b.cap * (20 * 8 + 4 + 4)
    a.close()
    b.close()


def test_struct_layouts_match_the_header():
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scripts"))
    import gen_rust_stub as G
    lay = G.struct_layouts()
    for name, dt in (("raftgpu_read_req", B.READ_REQ_DTYPE), ("raftgpu_read_state", B.READ_STATE_DTYPE)):
        size, offs = lay[name]
        assert size == dt.itemsize
        assert [o for _, o, _ in offs] == [dt.fields[f][1] for f in dt.names], name
