"""Oracle of the read-index path (ReadOnly, src/read_only.rs, and the parts of raft.rs that drive it), in two forms.

* The LITERAL form restates the reference: an unbounded queue of contexts, each pending request with its index, its
  `from` and an ack set keyed by peer ID (read_only.rs:63-134); the MsgReadIndex branch of step_leader
  (raft.rs:2056-2091, commit_to_current_term through the log's term of the committed index), the read tail of
  handle_heartbeat_response (raft.rs:1805-1818) and of post_conf_change (raft.rs:2648-2664).  Quorum is
  ProgressTracker::has_quorum (tracker.rs:367-372) = JointConfig::vote_result (joint.rs:56-67) over
  MajorityConfig::vote_result (majority.rs:130-154).
* The ARENA form keeps the device's bounded layout (columns [max_pending][cap] by ring position, a head | count word
  per group, acks by peer slot) and the batch rules of include/raftgpu.h, vectorised with numpy so that it runs at a
  million groups.  test_oracle_read_index.py checks it against the literal form on random traffic.

The reference's read-index tests are restated as SCENARIOS over a small driver interface (one leader group, peers
as slots), which the literal form, the arena form and the GPU (tests/test_gpu_read_index.py) all implement.
"""
from __future__ import annotations

import collections
import importlib

import numpy as np

B = importlib.import_module("raft-rs_b200").binding

DROPPED, READY, QUEUED, ALREADY_PENDING, FULL, SPLIT, INVALID = range(7)
ALLOC = 0x80000000
WORD_LOCAL, WORD_ACKED = 0x01000000, 0x02000000
WIDE_LO, WIDE_HI = 0x20000000, 0x40000000
U64_MAX = (1 << 64) - 1


# ============================================================================ literal form

def majority_vote_won(voters: set, yes: set) -> bool:
    """MajorityConfig::vote_result(..) == Won with `yes` the granted votes and nobody rejecting (majority.rs:130-154)."""
    if not voters:
        return True                                   # :131-136
    return len(voters & yes) >= len(voters) // 2 + 1  # util.rs:118-120 majority()


def ro_joint_vote_result(incoming: set, outgoing: set, acks: set) -> bool:
    """ProgressTracker::has_quorum (tracker.rs:367-372) -> JointConfig::vote_result (joint.rs:56-67)."""
    return majority_vote_won(incoming, acks) and majority_vote_won(outgoing, acks)


class ReadIndexStatus:                        # read_only.rs:57-61
    def __init__(self, req_from, index, acks):
        self.req_from, self.index, self.acks = req_from, index, acks


class ReadOnly:                               # read_only.rs:63-135
    def __init__(self):
        self.pending_read_index = {}
        self.read_index_queue = collections.deque()

    def add_request(self, index, ctx, req_from, self_id):          # :86-99
        if ctx in self.pending_read_index:
            return False
        self.pending_read_index[ctx] = ReadIndexStatus(req_from, index, {self_id})
        self.read_index_queue.append(ctx)
        return True

    def recv_ack(self, id_, ctx):                                    # :104-109
        rs = self.pending_read_index.get(ctx)
        if rs is None:
            return None
        rs.acks.add(id_)
        return rs.acks

    def advance(self, ctx):                                          # :114-129
        out = []
        if ctx in self.read_index_queue:
            i = list(self.read_index_queue).index(ctx)
            for _ in range(i + 1):
                c = self.read_index_queue.popleft()
                out.append((c, self.pending_read_index.pop(c)))
        return out

    def last_pending_request_ctx(self):                              # :132-134
        return self.read_index_queue[-1] if self.read_index_queue else None


class LiteralLeader:
    """One Raft node's read-index state as the reference keeps it.  Peers are ids; `slot_id` maps the engine's peer
    slots to ids, and a slot that becomes present again gets a fresh id (the engine clears a removed slot's acks)."""
    INVALID_ID = 0

    def __init__(self):
        self.ro = ReadOnly()
        self.slot_id, self.id_slot, self.next_id = {}, {}, 1
        self.incoming = self.outgoing = self.learners = frozenset()
        self.self_id = None
        self.term, self.term_start, self.committed, self.last_index = 2, U64_MAX, 0, 0

    def set_conf(self, incoming, outgoing=0, learners=0, self_slot=0):
        now = incoming | outgoing | learners
        for s in list(self.slot_id):
            if not (now >> s) & 1:
                del self.slot_id[s]
        for s in range(16):
            if (now >> s) & 1 and s not in self.slot_id:
                self.slot_id[s] = self.next_id
                self.id_slot[self.next_id] = s
                self.next_id += 1
        ids = lambda m: frozenset(self.slot_id[s] for s in range(16) if (m >> s) & 1)
        self.incoming, self.outgoing, self.learners = ids(incoming), ids(outgoing), ids(learners)
        self.self_id = self.slot_id.get(self_slot) if self_slot is not None else None

    def set_log(self, committed, term_start, last_index):
        self.committed, self.term_start, self.last_index = committed, term_start, last_index

    def reset(self):                                                  # raft.rs:957
        self.ro = ReadOnly()

    def log_term(self, i):
        """RaftLog::term: entries [term_start, last_index] carry the leader's term, earlier ones an older term."""
        return self.term if self.term_start <= i <= self.last_index else self.term - 1

    def commit_to_current_term(self):                                 # raft.rs:2527-2531
        return self.log_term(self.committed) == self.term

    def is_singleton(self):                                           # joint.rs:77-79
        return not self.outgoing and len(self.incoming) == 1

    def step_read_index(self, ctx, from_slot=None, lease=False):
        """step_leader's MsgReadIndex branch (raft.rs:2056-2091) -> (status, index)."""
        from_id = self.self_id if from_slot is None else self.slot_id.get(from_slot, -from_slot - 1)
        if not self.commit_to_current_term():                         # :2057-2061
            return DROPPED, 0
        if self.is_singleton() or lease:                              # :2063-2069, :2083-2088
            return READY, self.committed
        if not self.ro.add_request(self.committed, ctx, from_id, self.self_id):
            return ALREADY_PENDING, 0
        return QUEUED, self.committed

    def _ready(self, released):
        """handle_ready_read_index (raft.rs:2790-2806): (to_slot | None for a local ReadState, index, ctx)."""
        out = []
        for ctx, rs in released:
            local = rs.req_from in (self.INVALID_ID, self.self_id)
            out.append((None if local else self.id_slot.get(rs.req_from, -1), rs.index, ctx))
        return out

    def heartbeat_response(self, from_slot, ctx):
        """raft.rs:1805-1818 (the peer has a Progress: :1779-1789)."""
        if from_slot not in self.slot_id or ctx is None:
            return []
        acks = self.ro.recv_ack(self.slot_id[from_slot], ctx)
        if acks is None or not ro_joint_vote_result(self.incoming, self.outgoing, acks):
            return []
        return self._ready(self.ro.advance(ctx))

    def post_conf_change(self):                                       # raft.rs:2648-2664
        ctx = self.ro.last_pending_request_ctx()
        if ctx is None:
            return []
        acks = self.ro.recv_ack(self.self_id, ctx)
        if acks is None or not ro_joint_vote_result(self.incoming, self.outgoing, acks):
            return []
        return self._ready(self.ro.advance(ctx))

    def pending(self):
        return list(self.ro.read_index_queue)


# ============================================================================ arena form

def _popc(x):
    return np.bitwise_count(np.asarray(x, dtype=np.uint32)).astype(np.int64)


def _won(mask, acks):
    """majority_vote(mask, acks, 0) == Won, vectorised."""
    mask, acks = np.asarray(mask, dtype=np.uint32), np.asarray(acks, dtype=np.uint32)
    return (mask == 0) | (_popc(acks & mask) >= _popc(mask) // 2 + 1)


class ArenaReads:
    """The device's read-index columns and passes.  `cols` arguments carry the arena's meta / committed / term_start /
    last_index columns (numpy, indexed by group slot) as they are when the pass runs."""

    def __init__(self, cap: int, max_pending: int):
        self.cap, self.P = cap, max_pending
        self.ctx = np.zeros((max_pending, cap), dtype=np.uint64)
        self.index = np.zeros((max_pending, cap), dtype=np.uint64)
        self.word = np.zeros((max_pending, cap), dtype=np.uint32)
        self.rmeta = np.zeros(cap, dtype=np.uint32)

    # -- control-plane hooks
    def alloc(self, first, n, allocated=True):
        self.rmeta[first:first + n] = ALLOC if allocated else 0

    def reset(self, g):
        self.rmeta[g] &= np.uint32(ALLOC)

    def clear_slots(self, lo, removed16):
        """raftgpu_group_set_conf: the removed peer slots (16-bit mask over the whole group) lose their acks."""
        self.word[:, lo] &= np.uint32(~removed16 & 0xFFFFFFFF)

    # -- helpers
    def head_count(self, g):
        m = self.rmeta[g]
        return (m & 0xFF).astype(np.int64), ((m >> 16) & 0xFF).astype(np.int64)

    def pos(self, head, k):
        return (head + k) % self.P

    @staticmethod
    def conf(cols, lo):
        lo = np.asarray(lo, dtype=np.int64)
        m = cols.meta[lo].astype(np.uint32)
        wide = (m & WIDE_LO) != 0
        mh = np.where(wide, cols.meta[np.minimum(lo + 1, len(cols.meta) - 1)], 0).astype(np.uint32)
        inn = (m & 0xFF) | ((mh & 0xFF) << 8)
        out = ((m >> 8) & 0xFF) | (((mh >> 8) & 0xFF) << 8)
        has = (m & B.META_HAS_SELF) != 0
        has_h = (mh & B.META_HAS_SELF) != 0
        self_bit = np.where(has, np.uint32(1) << ((m >> 24) & 7),
                            np.where(has_h, np.uint32(1) << (8 + ((mh >> 24) & 7)), 0)).astype(np.uint32)
        return inn.astype(np.uint32), out.astype(np.uint32), self_bit

    def quorum(self, cols, lo, acks):
        inn, out, _ = self.conf(cols, lo)
        return _won(inn, acks) & _won(out, acks)

    # -- the request pass
    def read_index(self, reqs, cols, hi):
        n = len(reqs)
        status = np.zeros(n, dtype=np.uint8)
        index = np.zeros(n, dtype=np.uint64)
        if n == 0:
            return status, index
        g = reqs["group"].astype(np.int64)
        gi = np.minimum(g, self.cap - 1)
        local = (reqs["flags"] & B.READ_LOCAL) != 0
        lease = (reqs["flags"] & B.READ_LEASE) != 0
        frm = np.where(local, 0, reqs["from_slot"]).astype(np.int64)
        valid = (g < hi) & ((self.rmeta[gi] & ALLOC) != 0) & (local | (frm < 8))
        whi = (cols.meta[gi] & WIDE_HI) != 0
        key = np.where(whi, g - 1, g)
        frm = np.where(whi & ~local, frm + 8, frm)
        key = np.where(valid, key, -1)
        status[~valid] = INVALID
        start = np.ones(n, dtype=bool)
        start[1:] = key[1:] != key[:-1]
        run = np.cumsum(start) - 1
        run_first = np.flatnonzero(start)
        run_key = key[run_first]
        ok_runs = np.flatnonzero(run_key >= 0)
        _, first_of_key = np.unique(run_key[ok_runs], return_index=True)
        is_first = np.zeros(len(run_first), dtype=bool)
        is_first[ok_runs[first_of_key]] = True
        split = valid & ~is_first[run]
        status[split] = SPLIT
        act = valid & is_first[run]
        posn = np.arange(n) - run_first[run]
        for r in range(int(posn[act].max()) + 1 if act.any() else 0):
            sel = np.flatnonzero(act & (posn == r))
            k = key[sel]
            committed = cols.committed[k]
            current = (cols.term_start[k] <= committed) & (committed <= cols.last_index[k])
            inn, out, self_bit = self.conf(cols, k)
            singleton = (out == 0) & (_popc(inn) == 1)
            head, cnt = self.head_count(k)
            dup = np.zeros(len(sel), dtype=bool)
            for j in range(self.P):
                p = self.pos(head, j)
                dup |= (j < cnt) & (self.ctx[p, k] == reqs["ctx"][sel])
            st = np.where(~current, DROPPED,
                          np.where(singleton | lease[sel], READY,
                                   np.where(dup, ALREADY_PENDING, np.where(cnt == self.P, FULL, QUEUED))))
            status[sel] = st
            index[sel] = np.where((st == READY) | (st == QUEUED), committed, 0)
            q = st == QUEUED
            kq, p = k[q], self.pos(head[q], cnt[q])
            self.ctx[p, kq] = reqs["ctx"][sel][q]
            self.index[p, kq] = committed[q]
            self.word[p, kq] = self_bit[q] | (frm[sel][q].astype(np.uint32) << 16) | \
                np.where(local[sel][q], WORD_LOCAL, 0).astype(np.uint32)
            self.rmeta[kq] = (self.rmeta[kq] & ~np.uint32(0x00FF0000)) | ((cnt[q] + 1).astype(np.uint32) << 16)
        return status, index

    # -- recv_ack
    def ack(self, recs, cols):
        want = B.REC_HEARTBEAT | B.REC_READ_CTX
        g = recs["group"].astype(np.int64)
        slot = recs["peer_slot"].astype(np.int64)
        ok = ((recs["flags"] & want) == want) & (g < self.cap) & (slot < 8)
        gi = np.where(ok, g, 0)
        m = cols.meta[gi].astype(np.uint32)
        present = (m & 0xFF) | ((m >> 8) & 0xFF) | ((m >> 16) & 0xFF)
        ok &= ((present >> np.where(ok, slot, 0).astype(np.uint32)) & 1) != 0
        whi = (m & WIDE_HI) != 0
        lo = np.where(whi, gi - 1, gi)[ok]
        bit = (np.uint32(1) << np.where(whi, slot + 8, slot)[ok].astype(np.uint32)) | np.uint32(WORD_ACKED)
        tok = recs["index"][ok]
        head, cnt = self.head_count(lo)
        found = np.zeros(len(lo), dtype=bool)
        for j in range(self.P):
            p = self.pos(head, j)
            hit = ~found & (j < cnt) & (self.ctx[p, lo] == tok)
            np.bitwise_or.at(self.word, (p[hit], lo[hit]), bit[hit])
            found |= hit

    # -- advance behind has_quorum
    def release(self, cols, first, n):
        """-> READ_STATE_DTYPE array sorted by (group of the low half, queue position)."""
        g = np.arange(first, first + n, dtype=np.int64)
        head, cnt = self.head_count(g)
        rel = np.zeros(n, dtype=np.int64)
        for j in range(self.P):
            p = self.pos(head, j)
            w = self.word[p, g]
            hit = (j < cnt) & ((w & WORD_ACKED) != 0) & self.quorum(cols, g, w & 0xFFFF)
            rel = np.where(hit, j + 1, rel)
        rows = []
        for j in range(self.P):
            sel = np.flatnonzero(rel > j)
            if not len(sel):
                continue
            gg, p = g[sel], self.pos(head[sel], j)
            rows.append((gg, np.full(len(sel), j), p))
        out = self._emit(rows)
        for j in range(self.P):                                      # the marks go, the released requests leave
            p = self.pos(head, j)
            live = j < cnt
            self.word[p[live], g[live]] &= np.uint32(~WORD_ACKED & 0xFFFFFFFF)
        nh = (head + rel) % self.P
        self.rmeta[g] = (self.rmeta[g] & np.uint32(ALLOC)) | nh.astype(np.uint32) | ((cnt - rel).astype(np.uint32) << 16)
        return out

    def _emit(self, rows):
        if not rows:
            return np.zeros(0, dtype=B.READ_STATE_DTYPE)
        gg = np.concatenate([r[0] for r in rows])
        kk = np.concatenate([r[1] for r in rows])
        pp = np.concatenate([r[2] for r in rows])
        order = np.lexsort((kk, gg))
        gg, pp = gg[order], pp[order]
        w = self.word[pp, gg]
        frm = (w >> 16) & 0xFF
        local = (w & WORD_LOCAL) != 0
        out = np.zeros(len(gg), dtype=B.READ_STATE_DTYPE)
        out["group"] = np.where(~local & (frm >= 8), gg + 1, gg)
        out["to_slot"] = np.where(local, 0, frm & 7)
        out["flags"] = np.where(local, B.READ_LOCAL, 0)
        out["index"] = self.index[pp, gg]
        out["ctx"] = self.ctx[pp, gg]
        return out

    def last_ctx(self, first, n):
        g = np.arange(first, first + n, dtype=np.int64)
        head, cnt = self.head_count(g)
        p = self.pos(head, np.maximum(cnt - 1, 0))
        return np.where(cnt > 0, self.ctx[p, g], np.uint64(U64_MAX)).astype(np.uint64)

    def conf_changed(self, cols, g):
        head, cnt = self.head_count(np.array([g]))
        head, cnt = int(head[0]), int(cnt[0])
        if not cnt:
            return self._emit([])
        _, _, self_bit = self.conf(cols, np.array([g]))
        p = (head + cnt - 1) % self.P
        self.word[p, g] |= self_bit[0]
        if not self.quorum(cols, np.array([g]), np.array([self.word[p, g] & 0xFFFF]))[0]:
            return self._emit([])
        out = self._emit([(np.full(cnt, g), np.arange(cnt), (head + np.arange(cnt)) % self.P)])
        self.rmeta[g] = (self.rmeta[g] & np.uint32(ALLOC)) | np.uint32((head + cnt) % self.P)
        return out

    def queue(self, g):
        """(ctx, index, word) of group g's pending requests, in queue order (raftgpu_read_index_get)."""
        head, cnt = self.head_count(np.array([g]))
        p = (int(head[0]) + np.arange(int(cnt[0]))) % self.P
        return self.ctx[p, g].copy(), self.index[p, g].copy(), self.word[p, g].copy()


# ============================================================================ scenarios

class ArenaDriver:
    """One leader group (group slot 0) of an ArenaReads, driven like the reference's tests drive a Raft."""

    def __init__(self, max_pending=64):
        self.ar = ArenaReads(128, max_pending)
        self.cols = B.new_columns(128, 1)
        self.cols.term_start[:] = U64_MAX
        self.ar.alloc(0, 1)

    def set_conf(self, incoming, outgoing=0, learners=0, self_slot=0):
        was = int(self.cols.meta[0]) & 0xFF
        was = was | ((int(self.cols.meta[0]) >> 8) & 0xFF) | ((int(self.cols.meta[0]) >> 16) & 0xFF)
        self.cols.meta[0] = B.make_meta(incoming, outgoing, learners, self_slot)
        now = incoming | outgoing | learners
        self.ar.clear_slots(0, was & ~now)

    def set_log(self, committed, term_start, last_index):
        self.cols.committed[0], self.cols.term_start[0], self.cols.last_index[0] = committed, term_start, last_index

    def reset(self):
        self.ar.reset(0)

    def request(self, ctx, from_slot=None, lease=False):
        r = np.zeros(1, dtype=B.READ_REQ_DTYPE)
        r["ctx"], r["from_slot"] = ctx, 0 if from_slot is None else from_slot
        r["flags"] = (B.READ_LOCAL if from_slot is None else 0) | (B.READ_LEASE if lease else 0)
        st, idx = self.ar.read_index(r, self.cols, 1)
        return int(st[0]), int(idx[0])

    def acks(self, pairs):
        recs = np.zeros(len(pairs), dtype=B.APPEND_RESP_DTYPE)
        for i, (slot, ctx) in enumerate(pairs):
            recs[i]["peer_slot"], recs[i]["index"] = slot, ctx
            recs[i]["flags"] = B.REC_HEARTBEAT | B.REC_READ_CTX
        self.ar.ack(recs, self.cols)
        return states_to_list(self.ar.release(self.cols, 0, 1))

    def conf_changed(self):
        return states_to_list(self.ar.conf_changed(self.cols, 0))

    def pending(self):
        return [int(c) for c in self.ar.queue(0)[0]]


class LiteralDriver:
    def __init__(self, max_pending=None):
        self.l = LiteralLeader()

    def set_conf(self, incoming, outgoing=0, learners=0, self_slot=0):
        self.l.set_conf(incoming, outgoing, learners, self_slot)

    def set_log(self, committed, term_start, last_index):
        self.l.set_log(committed, term_start, last_index)

    def reset(self):
        self.l.reset()

    def request(self, ctx, from_slot=None, lease=False):
        return self.l.step_read_index(ctx, from_slot, lease)

    def acks(self, pairs):
        """One batch of heartbeat responses, delivered one at a time as the reference does."""
        out = []
        for slot, ctx in pairs:
            out += self.l.heartbeat_response(slot, ctx)
        return out

    def conf_changed(self):
        return self.l.post_conf_change()

    def pending(self):
        return self.l.pending()


def states_to_list(st):
    """READ_STATE_DTYPE rows -> [(to_slot | None for a local ReadState, index, ctx)] (single 8-slot group)."""
    return [(None if r["flags"] & B.READ_LOCAL else int(r["to_slot"]), int(r["index"]), int(r["ctx"])) for r in st]


# Leader in slot 0; a committed entry of the current term unless a scenario says otherwise.
def _leader(d, incoming, learners=0, committed=11, term_start=2):
    d.set_conf(incoming, 0, learners, 0)
    d.set_log(committed, term_start, committed)


def sc_raft_frees_read_only_mem(d):            # test_raft.rs:1442-1479
    _leader(d, 0b11, committed=2)
    assert d.request(101, from_slot=1) == (QUEUED, 2)
    assert d.pending() == [101]
    assert d.acks([(1, 101)]) == [(1, 2, 101)]
    assert d.pending() == []


def sc_read_only_option_safe(d):               # test_raft.rs:2230-2318
    _leader(d, 0b111)
    for i, (slot, wri, c1, c2, pending) in enumerate([
            (0, 11, 1, 11, False), (1, 21, 2, 22, False), (2, 31, 3, 33, False),
            (0, 41, 4, 44, True), (1, 51, 5, 55, True), (2, 61, 6, 66, True)]):
        d.set_log(wri, 2, wri)                                       # `proposals` committed entries of the term
        frm = None if slot == 0 else slot
        want_to = None if slot == 0 else slot
        # msg1, msg1 (duplicate), msg2 all reach the leader before any heartbeat response
        assert d.request(c1, frm) == (QUEUED, wri)
        assert d.request(c1, frm) == (ALREADY_PENDING, 0)
        assert d.request(c2, frm) == (QUEUED, wri)
        if pending:
            # heartbeat responses dropped; msg2 again: already pending, its heartbeats' acks release both
            assert d.request(c2, frm) == (ALREADY_PENDING, 0)
            got = d.acks([(1, c2), (2, c2)])
        else:
            got = d.acks([(1, c1), (2, c1), (1, c1), (2, c1), (1, c2), (2, c2)])
        assert got == [(want_to, wri, c1), (want_to, wri, c2)], (i, got)
        assert d.pending() == []


def sc_read_only_with_learner(d):              # test_raft.rs:2321-2391 (voter 0 = leader, learner 1)
    _leader(d, 0b01, learners=0b10)
    for i, (slot, wri, ctx) in enumerate([(0, 11, 1), (1, 21, 2), (0, 31, 3), (1, 41, 4)]):
        d.set_log(wri, 2, wri)
        frm = None if slot == 0 else slot
        # a singleton voter set answers at once, for the learner's forwarded request too
        assert d.request(ctx, frm) == (READY, wri), i
        assert d.pending() == []


def sc_read_only_option_lease(d):              # test_raft.rs:2394-2468
    _leader(d, 0b111)
    for i, (slot, wri, ctx) in enumerate([(0, 11, 1), (1, 21, 2), (2, 31, 3), (0, 41, 4)]):
        d.set_log(wri, 2, wri)
        assert d.request(ctx, None if slot == 0 else slot, lease=True) == (READY, wri), i
        assert d.pending() == []


def sc_read_only_for_new_leader(d):            # test_raft.rs:2503-2578
    # the new leader (term 2) has entries 1..2 of term 1, committed 1, and its empty entry 3 not yet committed
    d.set_conf(0b111, 0, 0, 0)
    d.set_log(1, 3, 3)
    assert d.request(7) == (DROPPED, 0)
    assert d.pending() == []
    d.set_log(4, 3, 4)                         # the proposal at 4 commits: the term has a committed entry
    assert d.request(7) == (QUEUED, 4)
    assert d.acks([(1, 7), (2, 7)]) == [(None, 4, 7)]


def sc_read_when_quorum_becomes_less(d):       # test_raft.rs:5380-5415
    _leader(d, 0b11, committed=1, term_start=1)
    assert d.request(0xABC) == (QUEUED, 1)
    assert d.acks([]) == []                    # peer 2's heartbeat response is dropped
    d.set_conf(0b01, 0, 0, 0)                  # remove_node(2) -> post_conf_change
    assert d.conf_changed() == [(None, 1, 0xABC)]


def sc_raw_node_read_index(d):                 # test_raw_node.rs:573-608: a single node answers at once
    _leader(d, 0b1, committed=1, term_start=1)
    assert d.request(0x6161) == (READY, 1)
    assert d.pending() == []


def sc_read_only_direct(d):                    # read_only.rs: recv_ack / advance / last_pending_request_ctx
    _leader(d, 0b11111)
    for c in (1, 2, 3, 4):
        assert d.request(c, 1)[0] == QUEUED
    assert d.acks([(1, 99)]) == []             # an ack for an unknown ctx is ignored
    assert d.pending() == [1, 2, 3, 4]
    assert d.acks([(1, 3)]) == []              # {self, 1}: no quorum of 5
    assert d.acks([(2, 3)]) == [(1, 11, 1), (1, 11, 2), (1, 11, 3)]   # advance pops up to and including ctx 3
    assert d.pending() == [4]
    assert d.acks([(1, 3), (2, 3), (3, 3)]) == []                     # acks for a popped ctx change nothing
    assert d.pending() == [4]
    d.reset()
    assert d.pending() == []


SCENARIOS = {f.__name__[3:]: f for f in (
    sc_raft_frees_read_only_mem, sc_read_only_option_safe, sc_read_only_with_learner, sc_read_only_option_lease,
    sc_read_only_for_new_leader, sc_read_when_quorum_becomes_less, sc_raw_node_read_index, sc_read_only_direct)}
