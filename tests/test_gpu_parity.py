"""GPU parity tests proper: the CUDA path, through the C-ABI, against the oracle.

Bit-exact (integer / index work): golden vectors replayed THROUGH the GPU, the
reference's table tests, full element-wise comparison of every column on the
synthetic streams (BASELINE configs 2-4), and size-independent properties at the
full sizes.  Run with ``-m gpu`` on a B200.
"""
import ctypes as C
import os
import random

import numpy as np
import pytest

from helpers import B, O, assert_columns_equal, bitmap_to_bool, checksum
from oracle import datadriven as dd

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def small():
    a = B.Arena(4096)
    yield a
    a.close()


# --------------------------------------------------------------------------- goldens via GPU

class GpuQuorum:
    """Evaluates the quorum functions on the GPU: voter ids are mapped to peer slots of one
    arena group, acked indexes become its matched / commit_group_id columns."""

    def __init__(self, arena):
        self.a = arena
        self.g = arena.group_alloc()

    def _setup(self, incoming, outgoing, lookup, gc):
        ids = []
        for i in list(incoming) + list(outgoing):
            if i not in ids:
                ids.append(i)
        assert len(ids) <= B.SLOTS
        slot = {i: s for s, i in enumerate(ids)}
        m_in = sum(1 << slot[i] for i in set(incoming))
        m_out = sum(1 << slot[i] for i in set(outgoing))
        self.a.group_set_conf(self.g, 0, 0, 0, None, 1)            # drop every Progress
        self.a.group_set_conf(self.g, m_in, m_out, 0, None, 1)
        self.a.set_group_commit(self.g, gc)
        for i, s in slot.items():
            p = self.a.progress_get(self.g, s)
            p.matched, p.commit_group_id = lookup.get(i, (0, 0))   # missing voter == (0, 0)
            self.a.progress_set(self.g, s, p)
        return slot

    def joint(self, incoming, outgoing, lookup, gc):
        self._setup(incoming, outgoing, lookup, gc)
        return self.a.maximal_committed_index(self.g)

    def majority(self, voters, lookup, gc):
        return self.joint(voters, [], lookup, gc)

    def joint_vote(self, incoming, outgoing, votes):
        slot = self._setup(incoming, outgoing, {}, False)
        self.a.reset_votes(self.g)
        for i, v in votes.items():
            if i in slot:
                self.a.record_vote(self.g, slot[i], v)
        return self.a.vote_result(self.g)[2]

    def majority_vote(self, voters, votes):
        return self.joint_vote(voters, [], votes)

    def impl(self):
        return dd.Impl(self.majority, self.joint, self.majority_vote, self.joint_vote)


@pytest.mark.parametrize("name,count", [("majority_commit.txt", 16), ("joint_commit.txt", 50),
                                        ("joint_group_commit.txt", 14), ("majority_vote.txt", 22),
                                        ("joint_vote.txt", 39)])
def test_golden_vectors_through_the_gpu(small, golden_dir, name, count):
    q = GpuQuorum(small)
    cases = dd.replay_file(os.path.join(golden_dir, "quorum", name), q.impl())
    assert len(cases) == count
    for d, actual in cases:
        assert actual == d.expected, f"{d.pos}\n--- gpu\n{actual}--- expected\n{d.expected}"
    small.group_free(q.g)


# --------------------------------------------------------------------------- table tests via GPU

def load_one(arena, cols):
    g = arena.group_alloc()
    for name, (col, dt, per_peer) in B.COLUMNS.items():
        arr = getattr(cols, name)
        if per_peer:
            for s in range(B.SLOTS):
                arena.column_write(col, s, g, arr[s, :1])
        else:
            arena.column_write(col, 0, g, arr[:1])
    return g


def read_one(arena, g):
    return arena.read_columns(1, first=g)


def apply_recs(arena, recs, g):
    recs = recs.copy()
    recs["group"] = g
    arena.enqueue(recs)
    r = arena.step(B.STEP_READ_COMMITTED | B.STEP_READ_RESULTS)
    return r, arena.record_results(0)


def progress_cols(state, matched, next_idx, pending_snapshot=0, paused=False):
    c = O.new_columns(1, 1)
    c.meta[0] = O.make_meta(0b11, 0, 0, 0)
    c.matched[1, 0], c.next_idx[1, 0], c.pending_snapshot[1, 0] = matched, next_idx, pending_snapshot
    c.pflags[1, 0] = state | (O.PF_PAUSED if paused else 0)
    c.pflags[0, 0] = O.STATE_REPLICATE
    c.term_start[0] = O.U64_MAX
    return c


def rec(slot, index, commit=0, reject=False, hint=0, request_snapshot=0, local=False):
    if reject:
        r = np.zeros(2, dtype=B.APPEND_RESP_DTYPE)
        r[0] = (0, slot, B.REC_REJECT, 0, index, commit)
        r[1] = (0, slot, B.REC_EXT, 0, hint, request_snapshot)
        return r
    r = np.zeros(1, dtype=B.APPEND_RESP_DTYPE)
    r[0] = (0, slot, B.REC_LOCAL if local else 0, 0, index, commit)
    return r


# src/tracker/progress.rs:351-373 test_progress_update
@pytest.mark.parametrize("update,wm,wn,wok", [(2, 3, 5, False), (3, 3, 5, False), (4, 4, 5, True),
                                               (5, 5, 6, True)])
def test_progress_update_on_gpu(small, update, wm, wn, wok):
    g = load_one(small, progress_cols(O.STATE_REPLICATE, 3, 5))
    _, res = apply_recs(small, rec(1, update), g)
    got = read_one(small, g)
    assert (int(got.matched[1, 0]), int(got.next_idx[1, 0])) == (wm, wn)
    assert bool(res[0] & B.RES_OK) == wok
    small.group_free(g)


# src/tracker/progress.rs:375-412 test_progress_maybe_decr
@pytest.mark.parametrize("state,m,n,rejected,last,w,wn", [
    (1, 5, 10, 5, 5, False, 10), (1, 5, 10, 4, 4, False, 10), (1, 5, 10, 9, 9, True, 6),
    (0, 0, 0, 0, 0, False, 0), (0, 0, 10, 5, 5, False, 10), (0, 0, 10, 9, 9, True, 9),
    (0, 0, 2, 1, 1, True, 1), (0, 0, 1, 0, 0, True, 1), (0, 0, 10, 9, 2, True, 3),
    (0, 0, 10, 9, 0, True, 1)])
def test_progress_maybe_decr_on_gpu(small, state, m, n, rejected, last, w, wn):
    cols = progress_cols(state, m, n, paused=True)
    g = load_one(small, cols)
    _, res = apply_recs(small, rec(1, rejected, reject=True, hint=last), g)
    got = read_one(small, g)
    assert bool(res[0] & B.RES_OK) == w
    assert (int(got.matched[1, 0]), int(got.next_idx[1, 0])) == (m, wn)
    want = O.copy_columns(cols)
    O.arena_apply(want, rec(1, rejected, reject=True, hint=last), mode=0)
    assert_columns_equal(got, want, 1)
    small.group_free(g)


def one_group(matches, gids=None, group_commit=False, committed=0, term_start=1, last_index=None):
    n = len(matches)
    c = O.new_columns(1, 1)
    for s, m in enumerate(matches):
        c.matched[s, 0], c.next_idx[s, 0] = m, m + 1
        if gids:
            c.commit_group_id[s, 0] = gids[s]
    c.meta[0] = O.make_meta((1 << n) - 1, 0, 0, 0, group_commit)
    c.committed[0], c.term_start[0] = committed, term_start
    c.last_index[0] = max(matches) if last_index is None else last_index
    return c


# harness/tests/integration_cases/test_raft.rs:1145-1240 test_commit
@pytest.mark.parametrize("matches,logs,sm_term,want", [
    ([1], [(1, 1)], 1, 1), ([1], [(1, 1)], 2, 0), ([2], [(1, 1), (2, 2)], 2, 2),
    ([1], [(2, 1)], 2, 1),
    ([2, 1, 1], [(1, 1), (2, 2)], 1, 1), ([2, 1, 1], [(1, 1), (1, 2)], 2, 0),
    ([2, 1, 2], [(1, 1), (2, 2)], 2, 2), ([2, 1, 2], [(1, 1), (1, 2)], 2, 0),
    ([2, 1, 1, 1], [(1, 1), (2, 2)], 1, 1), ([2, 1, 1, 1], [(1, 1), (1, 2)], 2, 0),
    ([2, 1, 1, 2], [(1, 1), (2, 2)], 1, 1), ([2, 1, 1, 2], [(1, 1), (1, 2)], 2, 0),
    ([2, 1, 2, 2], [(1, 1), (2, 2)], 2, 2), ([2, 1, 2, 2], [(1, 1), (1, 2)], 2, 0)])
def test_commit_on_gpu(small, matches, logs, sm_term, want):
    own = [i for t, i in logs if t == sm_term]
    g = load_one(small, one_group(matches, term_start=min(own) if own else O.U64_MAX,
                                  last_index=logs[-1][1]))
    adv, committed = small.maybe_commit(g)
    assert committed == want and adv == (want > 0)
    small.group_free(g)


# test_raft.rs:5092-5163 test_group_commit
@pytest.mark.parametrize("matches,gids,g_w,q_w", [
    ([1], [0], 1, 1), ([1], [1], 1, 1),
    ([2, 2, 1], [1, 2, 1], 2, 2), ([2, 2, 1], [1, 1, 2], 1, 2), ([2, 2, 1], [1, 0, 1], 1, 2),
    ([2, 2, 1], [0, 0, 0], 1, 2),
    ([4, 2, 1, 3], [0, 0, 0, 0], 1, 2), ([4, 2, 1, 3], [1, 0, 0, 0], 1, 2),
    ([4, 2, 1, 3], [0, 1, 0, 2], 2, 2), ([4, 2, 1, 3], [0, 2, 1, 0], 1, 2),
    ([4, 2, 1, 3], [1, 1, 1, 1], 2, 2), ([4, 2, 1, 3], [1, 1, 2, 1], 1, 2),
    ([4, 2, 1, 3], [1, 2, 1, 1], 2, 2), ([4, 2, 1, 3], [4, 3, 2, 1], 2, 2)])
def test_group_commit_on_gpu(small, matches, gids, g_w, q_w):
    g = load_one(small, one_group(matches, term_start=min(matches)))
    for s, gid in enumerate(gids):
        if gid:
            small.assign_commit_group(g, s, gid)
    small.set_group_commit(g, True)
    assert small.maybe_commit(g)[1] == g_w
    small.set_group_commit(g, False)
    assert small.maybe_commit(g)[1] == q_w
    small.group_free(g)


def test_group_commit_random_vs_oracle(small):
    rng = random.Random(2024)
    g = small.group_alloc()
    for _ in range(300):
        inc, out = rng.randrange(1, 256), rng.choice([0, rng.randrange(0, 256)])
        c = O.new_columns(1, 1)
        c.meta[0] = O.make_meta(inc, out, 0, None, True)
        for s in range(8):
            c.matched[s, 0] = rng.randrange(0, 12)
            c.commit_group_id[s, 0] = rng.randrange(0, 4)
        for name, (col, dt, per_peer) in B.COLUMNS.items():
            arr = getattr(c, name)
            if per_peer:
                for s in range(B.SLOTS):
                    small.column_write(col, s, g, arr[s, :1])
            else:
                small.column_write(col, 0, g, arr[:1])
        assert small.maximal_committed_index(g) == O.arena_mci(c, 0), (inc, out)
    small.group_free(g)


def test_progress_ops_vs_oracle(small):
    """raftgpu_progress_op: every Progress method (progress.rs:75-243) on the device cell vs the
    oracle's restatement, on random states and arguments."""
    L = O.lib()
    rng = random.Random(77)
    g = small.group_alloc()
    small.group_set_conf(g, 0b11, 0, 0, 0, 1)
    ops = [
        (B.POP_MAYBE_UPDATE, lambda p, a: L.ro_progress_maybe_update(p, a[0]), 1),
        (B.POP_MAYBE_DECR_TO, lambda p, a: L.ro_progress_maybe_decr_to(p, a[0], a[1], a[2]), 3),
        (B.POP_UPDATE_COMMITTED, lambda p, a: L.ro_progress_update_committed(p, a[0]) or 0, 1),
        (B.POP_OPTIMISTIC_UPDATE, lambda p, a: L.ro_progress_optimistic_update(p, a[0]) or 0, 1),
        (B.POP_BECOME_PROBE, lambda p, a: L.ro_progress_become_probe(p) or 0, 0),
        (B.POP_BECOME_REPLICATE, lambda p, a: L.ro_progress_become_replicate(p) or 0, 0),
        (B.POP_BECOME_SNAPSHOT, lambda p, a: L.ro_progress_become_snapshot(p, a[0]) or 0, 1),
        (B.POP_SNAPSHOT_FAILURE, lambda p, a: L.ro_progress_snapshot_failure(p) or 0, 0),
        (B.POP_MAYBE_SNAPSHOT_ABORT, lambda p, a: L.ro_progress_maybe_snapshot_abort(p), 0),
        (B.POP_IS_PAUSED, lambda p, a: L.ro_progress_is_paused(p), 0),
        (B.POP_RESUME, lambda p, a: L.ro_progress_resume(p) or 0, 0),
        (B.POP_PAUSE, lambda p, a: L.ro_progress_pause(p) or 0, 0),
        (B.POP_UPDATE_STATE, lambda p, a: L.ro_progress_update_state(p, a[0]), 1),
        (B.POP_RESET, lambda p, a: L.ro_progress_reset(p, a[0]) or 0, 1),
    ]
    fields = ("matched", "next_idx", "pending_snapshot", "pending_request_snapshot", "commit_group_id",
              "committed_index", "state", "paused", "recent_active", "ins_full")
    for _ in range(400):
        want = O.Progress()
        want.matched, want.next_idx = rng.randrange(0, 12), rng.randrange(0, 14)
        want.pending_snapshot = rng.choice([0, 0, rng.randrange(1, 14)])
        want.pending_request_snapshot = rng.choice([0, 0, rng.randrange(1, 14)])
        want.commit_group_id, want.committed_index = rng.randrange(0, 3), rng.randrange(0, 12)
        want.state, want.paused = rng.randrange(0, 3), rng.randrange(0, 2)
        want.recent_active, want.ins_full = rng.randrange(0, 2), rng.randrange(0, 2)
        got = small.progress_get(g, 1)
        for f in fields:
            setattr(got, f, getattr(want, f))
        small.progress_set(g, 1, got)
        code, fn, nargs = rng.choice(ops)
        args = [rng.choice([0, rng.randrange(0, 14)]) for _ in range(3)]
        want_ret = fn(C.byref(want), args)
        got_ret = small.progress_op(g, 1, code, *args)
        after = small.progress_get(g, 1)
        assert got_ret == want_ret, (code, args)
        for f in fields:
            assert getattr(after, f) == getattr(want, f), (code, args, f)
    small.group_free(g)


def test_has_quorum_and_recently_active_vs_oracle(small):
    rng = random.Random(3)
    g = small.group_alloc()
    for _ in range(100):
        inc, out = rng.randrange(0, 256), rng.choice([0, rng.randrange(0, 256)])
        learners = rng.randrange(0, 256) & ~(inc | out)
        small.group_set_conf(g, 0, 0, 0, None, 1)
        small.group_set_conf(g, inc, out, learners, None, 1)
        active = rng.randrange(0, 256)
        a = [s + 1 for s in range(8) if inc >> s & 1]
        b = [s + 1 for s in range(8) if out >> s & 1]
        want = O.joint_vote_result(a, b, {s + 1: True for s in range(8) if active >> s & 1}) == O.VOTE_WON
        assert small.has_quorum(g, active) == want           # tracker.rs:367-372
        present = inc | out | learners
        if present:
            me = rng.choice([s for s in range(8) if present >> s & 1])
            flags = {}
            for s in range(8):
                if present >> s & 1:
                    p = small.progress_get(g, s)
                    p.recent_active = rng.randrange(0, 2)
                    flags[s] = p.recent_active
                    small.progress_set(g, s, p)
            act = {s + 1: True for s, f in flags.items() if f or s == me}
            want = O.joint_vote_result(a, b, act) == O.VOTE_WON
            assert small.quorum_recently_active(g, me) == want  # tracker.rs:346-361
            for s in flags:
                assert small.progress_get(g, s).recent_active == (1 if s == me else 0)
    small.group_free(g)


# --------------------------------------------------------------------------- lifecycle

def test_group_lifecycle_mirrors_raft_new_reset_become_leader(small):
    g = small.group_alloc()
    # Raft::new: confchange::restore adds three voters with next_idx = last_index + 1 = 1
    small.group_set_conf(g, 0b111, 0, 0, 0, 1)
    for s in range(3):
        p = small.progress_get(g, s)
        assert (p.matched, p.next_idx, p.state, p.recent_active, p.present) == (0, 1, 0, 1, 1)
    with pytest.raises(B.RaftGpuError) as e:
        small.progress_get(g, 5)
    assert e.value.status == B.ERR_PEER_NOT_FOUND
    # Raft::reset at last_index 7, committed 4, persisted 7  (raft.rs:942-971)
    small.group_reset(g, B.NO_TERM_START, 7, 4, 7)
    p0, p1 = small.progress_get(g, 0), small.progress_get(g, 1)
    assert (p0.matched, p0.next_idx, p0.committed_index, p0.recent_active) == (7, 8, 4, 0)
    assert (p1.matched, p1.next_idx, p1.state) == (0, 8, B.STATE_PROBE)
    assert small.maybe_commit(g) == (False, 4)                  # follower: no quorum commit
    # become_leader (raft.rs:1162-1203): self Replicate, noop appended at 8 = term_start
    small.group_become_leader(g)
    st = small.group_get(g)
    assert (st.term_start, st.last_index, st.committed) == (8, 8, 4)
    assert small.progress_get(g, 0).state == B.STATE_REPLICATE
    # leader persists the noop, one follower acks it -> commit 8
    recs = np.concatenate([rec(0, 8, commit=8, local=True), rec(1, 8, commit=4)])
    r, res = apply_recs(small, recs, g)
    assert small.group_get(g).committed == 8 and r.n_advanced >= 1
    # RaftLog::commit_to (raft_log.rs:286-300)
    assert small.group_commit_to(g, 3) == B.OK and small.group_get(g).committed == 8
    assert small.group_commit_to(g, 9) == B.ERR_COMMIT_RANGE
    # apply_conf removing a voter drops its Progress
    small.group_set_conf(g, 0b011, 0, 0, 0, 9)
    with pytest.raises(B.RaftGpuError):
        small.progress_get(g, 2)
    small.group_free(g)


def test_enqueue_splits_duplicate_cells_into_waves(small):
    """Several responses of one peer in one batch keep their arrival order
    (raft.rs:1559: messages are stepped one at a time)."""
    cols = one_group([20, 2, 2], term_start=1, last_index=20)
    cols.pflags[1, 0], cols.pending_snapshot[1, 0] = O.STATE_SNAPSHOT, 8
    cols.pflags[0, 0] = cols.pflags[2, 0] = O.STATE_REPLICATE
    g = load_one(small, cols)
    # Snapshot peer: 9 aborts the snapshot (-> Probe), 12 then flips Probe -> Replicate;
    # in the other order the result differs, so order must be preserved.
    recs = np.concatenate([rec(1, 9), rec(1, 12), rec(2, 5), rec(1, 3), rec(2, 5, reject=True, hint=5)])
    want = O.copy_columns(cols)
    want_res = O.arena_apply(want, recs, mode=0)
    O.arena_recompute(want)
    r, res = apply_recs(small, recs, g)
    assert r.n_waves == 3 and r.n_records == len(recs)
    got = read_one(small, g)
    assert_columns_equal(got, want, 1)
    assert int(got.pflags[1, 0]) & 3 == O.STATE_REPLICATE and int(got.committed[0]) == 12
    # results come back per ring in ENQUEUE order, whichever wave a record ran in
    assert np.array_equal(res, want_res)
    small.group_free(g)


# --------------------------------------------------------------------------- synthetic streams

CONFIGS = {
    "cfg2_100k_x5": dict(n=100_000, seed=0x5EED0002, joint=False, rounds=12),
    "cfg3_1m_x5": dict(n=1_000_000, seed=0x5EED0003, joint=False, rounds=4),
    "cfg4_1m_x7_joint": dict(n=1_000_000, seed=0x5EED0004, joint=True, rounds=4),
}


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_synthetic_stream_elementwise(name):
    cfg = CONFIGS[name]
    n = cfg["n"]
    synth = B.Synth(n, cfg["seed"], joint=cfg["joint"])
    arena = B.Arena(n)
    assert arena.group_alloc_range(n) == 0
    arena.load_columns(synth.initial)
    ref = O.copy_columns(synth.initial)
    total_adv = 0
    for rnd in range(cfg["rounds"]):
        recs = synth.next_round().copy()
        half = len(recs) // 2
        while recs[half]["flags"] & B.REC_EXT:
            half += 1
        arena.enqueue(recs[:half], ring=0)          # two rings, as two caller threads would
        arena.enqueue(recs[half:], ring=1)
        r = arena.step(B.STEP_READ_COMMITTED | B.STEP_READ_RESULTS)
        bm, com = arena.step_results(n)
        res = np.concatenate([arena.record_results(0), arena.record_results(1)])
        want_res = O.arena_apply(ref, recs, mode=0)
        want_adv, want_bm, _, _ = O.arena_recompute(ref)
        assert r.n_waves == 1 and r.n_records == len(recs)
        assert r.n_advanced == want_adv
        assert np.array_equal(res, want_res), f"{name} round {rnd}: per-record results differ"
        assert np.array_equal(bm, want_bm[: len(bm)])
        adv = bitmap_to_bool(bm, n)
        assert np.array_equal(com[adv], ref.committed[:n][adv])
        total_adv += want_adv
        got = arena.read_columns(n)
        assert_columns_equal(got, ref, n, f"{name} round {rnd}")
    assert total_adv > n  # the stream really advances commit indexes
    cnt = arena.counters()
    assert cnt["recomputes"] == n * cfg["rounds"] and cnt["advanced"] == total_adv
    arena.close()


def test_enqueue_bulk_sorted_unsorted_and_order_check():
    """raftgpu_enqueue_bulk: the library's own staging threads; same results as the oracle for
    a sorted batch (fast path), for the same batch shuffled (atomic bookkeeping) and a loud
    error when SORTED is promised but not true."""
    n = 200_000
    synth = B.Synth(n, 0x5EED0002)
    for shuffled in (False, True):
        arena = B.Arena(n)
        arena.group_alloc_range(n)
        arena.load_columns(synth.initial)
        ref = O.copy_columns(synth.initial)
        s2 = B.Synth(n, 0x5EED0002)
        for rnd in range(3):
            recs = s2.next_round().copy()
            if shuffled:
                # permute whole records but keep each REJECT glued to its EXT
                main = np.nonzero((recs["flags"] & B.REC_EXT) == 0)[0]
                perm = np.random.default_rng(rnd).permutation(main)
                idx = []
                for i in perm:
                    idx.append(i)
                    if recs[i]["flags"] & B.REC_REJECT:
                        idx.append(i + 1)
                sub = np.ascontiguousarray(recs[np.array(idx)])
                arena.enqueue_bulk(sub, sorted_by_group=False)
            else:
                arena.enqueue_bulk(recs, sorted_by_group=True)
            r = arena.step(B.STEP_READ_COMMITTED)
            O.arena_apply(ref, recs, mode=0)      # one wave: order inside it does not matter
            want_adv, want_bm, _, _ = O.arena_recompute(ref)
            assert r.n_waves == 1 and r.n_records == len(recs) and r.n_advanced == want_adv
            assert_columns_equal(arena.read_columns(n), ref, n, f"bulk shuffled={shuffled} round {rnd}")
        if not shuffled:
            bad = s2.next_round().copy()[::-1].copy()
            with pytest.raises(B.RaftGpuError) as e:
                arena.enqueue_bulk(bad, sorted_by_group=True)
            assert e.value.status == B.ERR_INVALID
        arena.close()


def test_zero_copy_packed_submission_and_duplicate_detection():
    """raftgpu_step_begin_packed: the caller's pinned packed buffer goes to the GPU with no staging
    copy; results equal the oracle; a batch that breaks the one-record-per-cell promise is
    detected ON THE DEVICE and the step fails loudly."""
    n = 100_000
    synth = B.Synth(n, 0x5EED0002)
    arena = B.Arena(n)
    arena.group_alloc_range(n)
    arena.load_columns(synth.initial)
    ref = O.copy_columns(synth.initial)
    bufs = [arena.host_alloc_packed(5 * n + 64) for _ in range(2)]
    for rnd in range(4):
        recs = synth.next_round().copy()
        k = arena.pack_records(recs, bufs[rnd % 2])
        assert len(recs) <= k <= len(recs) + np.count_nonzero(recs["flags"] & B.REC_REJECT)
        arena.step_begin_packed(bufs[rnd % 2], k, B.STEP_READ_COMMITTED)
        r = arena.step_wait()
        O.arena_apply(ref, recs, mode=0)
        want_adv, want_bm, _, _ = O.arena_recompute(ref)
        assert r.n_advanced == want_adv and r.n_duplicates == 0 and r.h2d_bytes == 16 * k
        bm, com = arena.step_results(n)
        assert np.array_equal(bm, want_bm[: len(bm)])
        adv = bitmap_to_bool(bm, n)
        assert np.array_equal(com[adv], ref.committed[:n][adv])
        assert_columns_equal(arena.read_columns(n), ref, n, f"zero-copy round {rnd}")
    # wide commits (commit > index, huge deltas) survive packing
    wide = np.zeros(3, dtype=B.APPEND_RESP_DTYPE)
    wide[0] = (5, 1, 0, 0, 10, 1 << 40)                 # commit far above index
    wide[1] = (6, 2, 0, 0, (1 << 50) + 7, 3)            # delta does not fit 24 bits
    wide[2] = (7, 0, B.REC_LOCAL, 0, 9, 4)              # LOCAL with commit < index
    k = arena.pack_records(wide, bufs[0])
    assert k == 6
    arena.step_begin_packed(bufs[0], k, 0)
    arena.step_wait()
    O.arena_apply(ref, wide, mode=0)
    O.arena_recompute(ref)
    assert_columns_equal(arena.read_columns(n), ref, n, "wide commits")
    # two records for one cell in one zero-copy batch: detected by the kernel
    dup = np.zeros(2, dtype=B.APPEND_RESP_DTYPE)
    dup[0] = (11, 1, 0, 0, int(ref.matched[1, 11]) + 5, 0)
    dup[1] = (11, 1, 0, 0, int(ref.matched[1, 11]) + 9, 0)
    k = arena.pack_records(dup, bufs[1])
    arena.step_begin_packed(bufs[1], k, 0)
    r = arena.step_wait(check=False)
    assert r.status == B.ERR_INVALID and r.n_duplicates == 1
    arena.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n,joint,shuffle", [(100_003, False, False), (40_000, True, False), (50_000, False, True)])
def test_compact_stream_submission_vs_oracle(n, joint, shuffle):
    """raftgpu_step_begin_compact: the 4-byte-unit stream (group runs + ESC side table) goes over PCIe
    as is.  A tileable stream (groups ascending) takes the fused tile kernel; with the groups in
    random order (`shuffle`) it is not tileable and apply_compact_kernel + the recompute pass run
    instead.  Either way columns, bitmap, committed and the per-record result bytes equal the
    oracle's; hostile values take the ESC path; a second record for a cell is applied in order by
    the fused kernel and refused (on the device) by the scatter kernel."""
    synth = B.Synth(n, 0x5EED0009, joint=joint)
    rank = np.random.default_rng(3).permutation(n + 1)

    def arrange(recs):
        if not shuffle:
            return recs
        return np.ascontiguousarray(recs[np.argsort(rank[recs["group"]], kind="stable")])

    arena = B.Arena(n)
    arena.group_alloc_range(n)
    arena.load_columns(synth.initial)
    ref = O.copy_columns(synth.initial)
    cap_bytes = B.compact_bound(8 * n)
    bufs = [arena.host_alloc_bytes(cap_bytes) for _ in range(2)]
    for rnd in range(4):
        recs = arrange(synth.next_round().copy())
        nb, units = B.pack_compact(recs, bufs[rnd % 2], want_units=True)
        assert shuffle or nb < 0.45 * 16 * len(recs)
        hdr = bufs[rnd % 2][:64].view(B.COMPACT_HDR_DTYPE)[0]
        assert bool(hdr["flags"] & B.COMPACT_TILEABLE) == (not shuffle)
        arena.step_begin_compact(bufs[rnd % 2], nb, B.STEP_READ_COMMITTED | B.STEP_READ_RESULTS)
        r = arena.step_wait()
        want_res = O.arena_apply(ref, recs, mode=0)
        want_adv, want_bm, _, _ = O.arena_recompute(ref)
        main = (recs["flags"] & B.REC_EXT) == 0
        assert r.n_advanced == want_adv and r.n_duplicates == 0 and r.h2d_bytes == nb
        assert r.n_records == np.count_nonzero(main)
        bm, com = arena.step_results(n)
        assert np.array_equal(bm, want_bm[: len(bm)])
        adv = bitmap_to_bool(bm, n)
        assert np.array_equal(com[adv], ref.committed[:n][adv])
        res = arena.slot_results()
        assert np.array_equal(res[units[main]], want_res[main]), "per-record results differ"
        other = np.ones(len(res), dtype=bool)
        other[units[main]] = False
        assert not res[other].any()
        assert_columns_equal(arena.read_columns(n), ref, n, f"compact round {rnd}")
    # hostile values: huge indices, commit above index, lagging peers, LOCAL with commit < index
    odd = np.zeros(8, dtype=B.APPEND_RESP_DTYPE)
    odd[0] = (5, 1, 0, 0, 10, 1 << 40)
    odd[1] = (6, 2, 0, 0, (1 << 50) + 7, 3)
    odd[2] = (6, 3, 0, 0, (1 << 50) + 7 - 40000, (1 << 50))
    odd[3] = (7, 0, B.REC_LOCAL, 0, 9, 4)
    odd[4] = (8, 1, 0, 0, (1 << 63) + 11, (1 << 63) + 2)
    odd[5] = (9, 9, 0, 0, 77, 70)                         # no such peer slot: NO_PROGRESS
    odd[6] = (12, 1, 0, 0, int(ref.matched[1, 12]) + 300, int(ref.matched[1, 12]))   # commit delta 300
    odd[7] = (n - 1, 7, 0, 0, 77, 70)                     # a slot the group has no peer in
    odd = arrange(odd)
    nb, units = B.pack_compact(odd, bufs[0], want_units=True)
    arena.step_begin_compact(bufs[0], nb, B.STEP_READ_RESULTS)
    arena.step_wait()
    want_res = O.arena_apply(ref, odd, mode=0)
    O.arena_recompute(ref)
    assert np.array_equal(arena.slot_results()[units], want_res)
    assert_columns_equal(arena.read_columns(n), ref, n, "hostile values")
    # an empty batch still recomputes
    nb, _ = B.pack_compact(np.zeros(0, dtype=B.APPEND_RESP_DTYPE), bufs[1])
    arena.step_begin_compact(bufs[1], nb, 0)
    r = arena.step_wait()
    assert r.n_records == 0 and r.n_advanced == 0
    # two records for one cell in one batch
    dup = np.zeros(3, dtype=B.APPEND_RESP_DTYPE)
    dup[0] = (11, 1, 0, 0, int(ref.matched[1, 11]) + 5, 0)
    dup[1] = (11, 1, 0, 0, int(ref.matched[1, 11]) + 9, 0)
    dup[2] = (3, 1, 0, 0, int(ref.matched[1, 3]) + 1, 0)       # descending after group 11: scatter path when shuffled
    if not shuffle:
        dup = dup[[2, 0, 1]]
    nb, units = B.pack_compact(dup, bufs[1], want_units=True)
    arena.step_begin_compact(bufs[1], nb, B.STEP_READ_RESULTS)
    r = arena.step_wait(check=False)
    if shuffle:    # the scatter kernel has one thread per record: a second record for a cell is refused
        assert r.status == B.ERR_INVALID and r.n_duplicates == 1
    else:          # the fused kernel walks a group's records in order: applied one after the other
        assert r.status == B.OK and r.n_duplicates == 0
        want_res = O.arena_apply(ref, dup, mode=0)
        O.arena_recompute(ref)
        assert np.array_equal(arena.slot_results()[units], want_res)
        assert_columns_equal(arena.read_columns(n), ref, n, "two records for one cell, in order")
    # a mangled header is refused before anything is submitted
    bad = bufs[0]
    bad[:4] = 0
    with pytest.raises(RuntimeError):
        arena.step_begin_compact(bad, 64, 0)
    arena.close()


def _fused_round(arena, n, recs, ref, pk, d_bufs):
    """One fused step (raftgpu_step_sorted_device) on `recs` (group order) checked against the oracle."""
    k = arena.pack_records(recs, pk)
    off = B.tile_index(pk, k, n)
    d_pk, d_off, d_res, d_bm, d_com = d_bufs
    arena.h2d(d_pk, pk[:k])
    arena.h2d(d_off, off)
    arena.h2d(d_bm, np.zeros(arena.cap // 32, dtype=np.uint32))   # bits past n_groups are left untouched
    arena.step_sorted_device(d_pk, k, d_off, d_results=d_res, d_adv=d_bm, d_commit=d_com)
    res = np.zeros(k, dtype=np.uint8)
    bm = np.zeros(arena.cap // 32, dtype=np.uint32)
    arena.d2h(res, d_res)
    arena.d2h(bm, d_bm)
    want_res = O.arena_apply(ref, recs, mode=0)
    want_adv, want_bm, _, _ = O.arena_recompute(ref)
    main_pk = (pk[:k, 0] & np.uint64(1 << 37)) == 0           # packed records that are not EXT payloads
    main_orig = (recs["flags"] & B.REC_EXT) == 0
    assert np.array_equal(res[main_pk], want_res[main_orig]), "per-record results differ"
    assert not res[~main_pk].any()
    words = (n + 31) // 32
    assert np.array_equal(bm[:words], want_bm[:words])
    assert_columns_equal(arena.read_columns(n), ref, n, "fused step")
    return want_adv


@pytest.mark.parametrize("n,joint", [(100_003, False), (70_001, True), (1_000_000, False)])
def test_fused_tile_step_vs_oracle(n, joint):
    """raftgpu_step_sorted_device: the fused apply + recompute kernel on group-ordered batches,
    including a ragged last tile, the general (joint, hint 0x7f) instantiation and 1M groups."""
    synth = B.Synth(n, 0x5EED0007, joint=joint)
    arena = B.Arena(n)
    arena.group_alloc_range(n)
    arena.load_columns(synth.initial)
    ref = O.copy_columns(synth.initial)
    pk = np.zeros((9 * n + 64, 2), dtype=np.uint64)
    d_bufs = (arena.device_alloc(pk.nbytes), arena.device_alloc(4 * (n // 256 + 2)),
              arena.device_alloc(9 * n + 64), arena.device_alloc(arena.cap // 8), arena.device_alloc(8 * arena.cap))
    total = 0
    for _ in range(3 if n >= 1_000_000 else 6):
        total += _fused_round(arena, n, synth.next_round().copy(), ref, pk, d_bufs)
    assert total > n // 2
    cnt = arena.counters()
    assert cnt["recomputes"] % n == 0 and cnt["advanced"] == total
    arena.close()


def test_fused_tile_step_learners_group_commit_and_crowded_tiles():
    """Fused kernel corner cases: peers outside the voter hint (learners -> HBM path), group commit
    groups (general kernel), a tile crowded with rejections (about 128 per warp: more than the per-warp
    deferral list holds, so the rest are applied inside the record loop), and a record that is not in
    its tile."""
    n = 2000
    synth = B.Synth(n, 0x5EED0009)
    cols = synth.initial
    rng = np.random.default_rng(5)
    learners = rng.random(n) < 0.3                      # slot 6 is a learner in 30 % of the groups
    cols.meta[:n] |= (learners.astype(np.uint32) << np.uint32(16 + 6))
    cols.next_idx[6, :n] = np.where(learners, cols.matched[0, :n] - 5, 0)
    cols.pflags[6, :n] = np.where(learners, O.STATE_PROBE, 0)
    gc = rng.random(n) < 0.2                            # 20 % of the groups use group commit
    cols.meta[:n] |= np.where(gc, O.META_GROUP_COMMIT, 0).astype(np.uint32)
    cols.commit_group_id[:5, :n] = rng.integers(0, 3, (5, n))
    arena = B.Arena(n)
    arena.group_alloc_range(n)
    arena.load_columns(cols)
    ref = O.copy_columns(cols)
    pk = np.zeros((20 * n, 2), dtype=np.uint64)
    d_bufs = (arena.device_alloc(pk.nbytes), arena.device_alloc(4 * (n // 256 + 2)),
              arena.device_alloc(20 * n), arena.device_alloc(arena.cap // 8), arena.device_alloc(8 * arena.cap))
    for rnd in range(3):
        base = synth.next_round().copy()
        # add learner responses (slot 6) and make tile 1 (groups 256..511) crowded with rejects:
        extra = []
        for g in np.nonzero(learners)[0]:
            extra.append((g, 6, 0, 0, int(ref.matched[0, g]) - 3 + rnd, 0))
        recs = np.concatenate([base, np.array(extra, dtype=B.APPEND_RESP_DTYPE)])
        if rnd == 1:   # every follower of tile 1 rejects: 3 packed records each (reject, hint, snapshot)
            keep = ~((recs["group"] >= 256) & (recs["group"] < 512) & (recs["peer_slot"] >= 1) & (recs["peer_slot"] <= 4))
            recs = recs[keep]
            crowd = []
            for g in range(256, 512):
                for s in range(1, 5):
                    crowd.append((g, s, B.REC_REJECT, 0, int(ref.next_idx[s, g]) - 1, 0))
                    crowd.append((g, s, B.REC_EXT, 0, int(ref.matched[s, g]), 77))
            recs = np.concatenate([recs, np.array(crowd, dtype=B.APPEND_RESP_DTYPE)])
        order = np.argsort(recs["group"], kind="stable")   # group order, arrival order kept inside a group
        recs = np.ascontiguousarray(recs[order])
        adv = _fused_round(arena, n, recs, ref, pk, d_bufs)
    # a record filed under the wrong tile is not applied
    bad = np.zeros(2, dtype=B.APPEND_RESP_DTYPE)
    bad[0] = (10, 1, 0, 0, int(ref.matched[1, 10]) + 1, int(ref.matched[1, 10]))
    bad[1] = (900, 1, 0, 0, int(ref.matched[1, 900]) + 1, int(ref.matched[1, 900]))
    k = arena.pack_records(bad, pk)
    assert k == 2
    off = B.tile_index(pk, k, n)
    off[1:4] = 2                                            # claim both records belong to tile 0
    arena.h2d(d_bufs[0], pk[:k])
    arena.h2d(d_bufs[1], off)
    arena.step_sorted_device(d_bufs[0], k, d_bufs[1], d_results=d_bufs[2])
    res = np.zeros(k, dtype=np.uint8)
    arena.d2h(res, d_bufs[2])
    assert res[1] == B.RES_NO_PROGRESS and res[0] & B.RES_OK
    with pytest.raises(B.RaftGpuError):
        B.tile_index(np.ascontiguousarray(pk[:k][::-1]), k, n)   # not in group order
    arena.close()


@pytest.mark.parametrize("n,joint,mode", [(100_003, False, "sorted"), (40_000, True, "sorted"), (50_000, False, "shuffled"),
                                          (30_000, False, "pipelined"), (900, False, "sorted")])
def test_step_begin_records_vs_oracle(n, joint, mode):
    """raftgpu_step_begin_records: 24-byte records in pageable memory, packed into the compact stream
    by the library's staging threads (one slice each, stitched at unit-block boundaries), one step.
    Sorted batches take the fused kernel; `shuffled` group order the scatter kernel; `pipelined`
    adds several acks per cell, which the fused kernel applies in order."""
    synth = B.Synth(n, 0x5EED000D, joint=joint)
    arena = B.Arena(n)
    arena.group_alloc_range(n)
    arena.load_columns(synth.initial)
    ref = O.copy_columns(synth.initial)
    rank = np.random.default_rng(4).permutation(n + 1)
    for rnd in range(4):
        recs = synth.next_round().copy()
        if mode == "shuffled":
            recs = np.ascontiguousarray(recs[np.argsort(rank[recs["group"]], kind="stable")])
        if mode == "pipelined":
            extra = []
            for g in range(rnd, n, 5):
                m = int(ref.matched[2, g])
                for d_ in (3, 1, 6):
                    extra.append((g, 2, 0, 0, m + d_, m))
            recs = np.concatenate([recs, np.array(extra, dtype=B.APPEND_RESP_DTYPE)])
            recs = np.ascontiguousarray(recs[np.argsort(recs["group"], kind="stable")])
        arena.step_begin_records(recs, B.STEP_READ_COMMITTED)
        if rnd % 2 == 0:        # two steps in flight every other round
            recs2 = synth.next_round().copy()
            if mode == "shuffled":
                recs2 = np.ascontiguousarray(recs2[np.argsort(rank[recs2["group"]], kind="stable")])
            arena.step_begin_records(recs2, B.STEP_READ_COMMITTED)
        r = arena.step_wait()
        O.arena_apply(ref, recs, mode=0)
        want_adv, want_bm, _, _ = O.arena_recompute(ref)
        assert r.n_advanced == want_adv and r.n_duplicates == 0
        if mode != "shuffled":     # (the fallback path counts packed records, EXT payloads included)
            assert r.n_records == np.count_nonzero((recs["flags"] & B.REC_EXT) == 0)
            assert r.h2d_bytes < 12 * len(recs)
        bm, com = arena.step_results(n)
        assert np.array_equal(bm, want_bm[: len(bm)])
        adv = bitmap_to_bool(bm, n)
        assert np.array_equal(com[adv], ref.committed[:n][adv])
        if rnd % 2 == 0:
            r = arena.step_wait()
            O.arena_apply(ref, recs2, mode=0)
            want_adv, want_bm, _, _ = O.arena_recompute(ref)
            assert r.n_advanced == want_adv
            bm, com = arena.step_results(n)
            assert np.array_equal(bm, want_bm[: len(bm)])
        assert_columns_equal(arena.read_columns(n), ref, n, f"step_begin_records {mode} round {rnd}")
    # empty batch; then mixing with enqueued records is refused
    arena.step_begin_records(np.zeros(0, dtype=B.APPEND_RESP_DTYPE), 0)
    assert arena.step_wait().n_records == 0
    one = np.zeros(1, dtype=B.APPEND_RESP_DTYPE)
    one[0] = (3, 1, 0, 0, int(ref.matched[1, 3]) + 1, 0)
    arena.enqueue(one)
    with pytest.raises(B.RaftGpuError):
        arena.step_begin_records(one, 0)
    arena.step(0)
    O.arena_apply(ref, one, mode=0)
    O.arena_recompute(ref)
    assert_columns_equal(arena.read_columns(n), ref, n, "after the refused mix")
    arena.close()


def _compact_round(arena, n, recs, ref, blob, d_bufs, ordered=False):
    """One fused compact step (raftgpu_step_compact_device) on `recs` (group order) vs the oracle."""
    nb, units = B.pack_compact(recs, blob, want_units=True)
    hdr = blob[:64].view(B.COMPACT_HDR_DTYPE)[0]
    assert hdr["flags"] & B.COMPACT_TILEABLE
    d_blob, d_off, d_res, d_bm, d_com, d_bad = d_bufs
    nu = int(hdr["n_units"])
    arena.h2d(d_blob, blob[:nb])
    arena.h2d(d_bm, np.zeros(arena.cap // 32, dtype=np.uint32))
    arena.h2d(d_res, np.zeros(max(nu, 1), dtype=np.uint8))
    arena.h2d(d_bad, np.zeros(1, dtype=np.uint32))
    arena.compact_tile_index_device(d_blob, blob, d_off, d_bad)
    arena.step_compact_device(d_blob, blob, d_off, d_results=d_res, d_adv=d_bm, d_commit=d_com, d_dup=d_bad,
                              ordered=ordered)
    res = np.zeros(max(nu, 1), dtype=np.uint8)
    bm = np.zeros(arena.cap // 32, dtype=np.uint32)
    bad = np.zeros(1, dtype=np.uint32)
    arena.d2h(res, d_res)
    arena.d2h(bm, d_bm)
    arena.d2h(bad, d_bad)
    assert bad[0] == 0
    want_res = O.arena_apply(ref, recs, mode=0)
    want_adv, want_bm, _, _ = O.arena_recompute(ref)
    main = (recs["flags"] & B.REC_EXT) == 0
    assert np.array_equal(res[units[main]], want_res[main]), "per-record results differ"
    other = np.ones(len(res), dtype=bool)
    other[units[main]] = False
    assert not res[other].any()
    words = (n + 31) // 32
    assert np.array_equal(bm[:words], want_bm[:words])
    assert_columns_equal(arena.read_columns(n), ref, n, "fused compact step")
    return want_adv


def _compact_bufs(arena, n, per_group):
    cap_b = B.compact_bound(per_group * n + 64)
    blob = np.zeros(cap_b, dtype=np.uint8)
    d = (arena.device_alloc(cap_b), arena.device_alloc(4 * (3 * (arena.cap // B.tile_groups() + 2) + 2)),
         arena.device_alloc(3 * per_group * n + 64), arena.device_alloc(arena.cap // 8),
         arena.device_alloc(8 * arena.cap), arena.device_alloc(4))
    return blob, d


@pytest.mark.gpu
@pytest.mark.parametrize("n,joint,ordered", [(100_003, False, False), (100_003, False, True), (70_001, True, False),
                                             (70_001, True, True), (1_000_000, False, False)])
def test_fused_compact_step_vs_oracle(n, joint, ordered):
    """raftgpu_step_compact_device: the fused kernel on compact streams -- one thread per unit, or
    (`ordered`) the per-group walk -- including a ragged last tile, the general (joint, hint 0x7f)
    instantiation and 1M groups."""
    synth = B.Synth(n, 0x5EED000A, joint=joint)
    arena = B.Arena(n)
    arena.group_alloc_range(n)
    arena.load_columns(synth.initial)
    ref = O.copy_columns(synth.initial)
    blob, d_bufs = _compact_bufs(arena, n, 9)
    total = 0
    for _ in range(3 if n >= 1_000_000 else 6):
        total += _compact_round(arena, n, synth.next_round().copy(), ref, blob, d_bufs, ordered=ordered)
    assert total > n // 2
    cnt = arena.counters()
    assert cnt["recomputes"] % n == 0 and cnt["advanced"] == total
    arena.close()


@pytest.mark.gpu
def test_fused_compact_step_corner_cases():
    """Learners outside the voter hint (HBM path), group-commit groups, a tile with more units than
    the shared-memory staging holds, groups with more than 8 records (several runs), several records
    for one cell (applied in stream order), Snapshot-state peers, sparse batches with empty tiles."""
    n = 3000
    synth = B.Synth(n, 0x5EED000B)
    cols = synth.initial
    rng = np.random.default_rng(8)
    learners = rng.random(n) < 0.3
    cols.meta[:n] |= (learners.astype(np.uint32) << np.uint32(16 + 6))
    cols.next_idx[6, :n] = np.where(learners, cols.matched[0, :n] - 5, 0)
    cols.pflags[6, :n] = np.where(learners, O.STATE_PROBE, 0)
    gc = rng.random(n) < 0.2
    cols.meta[:n] |= np.where(gc, O.META_GROUP_COMMIT, 0).astype(np.uint32)
    cols.commit_group_id[:5, :n] = rng.integers(0, 3, (5, n))
    snap = rng.random(n) < 0.1                           # slot 2 is in Snapshot state in 10 % of the groups
    cols.pflags[2, :n] = np.where(snap, O.STATE_SNAPSHOT, cols.pflags[2, :n])
    cols.pending_snapshot[2, :n] = np.where(snap, cols.matched[2, :n] + 3, 0)
    arena = B.Arena(n)
    arena.group_alloc_range(n)
    arena.load_columns(cols)
    ref = O.copy_columns(cols)
    blob, d_bufs = _compact_bufs(arena, n, 40)
    tg = B.tile_groups()
    for rnd in range(4):
        base = synth.next_round().copy()
        extra = []
        for g in np.nonzero(learners)[0]:
            extra.append((g, 6, 0, 0, int(ref.matched[0, g]) - 3 + rnd, 0))
        if rnd == 1:   # tile 1 crowded: every follower rejects (ESC units + side table) and acks twice more
            for g in range(tg, 2 * tg):
                for s_ in range(1, 5):
                    extra.append((g, s_, B.REC_REJECT, 0, int(ref.next_idx[s_, g]) - 1, 0))
                    extra.append((g, s_, B.REC_EXT, 0, int(ref.matched[s_, g]), 77 if s_ == 1 else 0))
                    extra.append((g, s_, 0, 0, int(ref.matched[s_, g]) + 2, int(ref.matched[s_, g])))
                    extra.append((g, s_, 0, 0, int(ref.matched[s_, g]) + 7, int(ref.matched[s_, g]) + 1))
        if rnd == 2:   # pipelined acks: the same cell several times, out of order too
            for g in range(0, n, 7):
                m = int(ref.matched[1, g])
                for d_ in (4, 2, 9, 9, 1):
                    extra.append((g, 1, 0, 0, m + d_, m))
        recs = np.concatenate([base, np.array(extra, dtype=B.APPEND_RESP_DTYPE)]) if extra else base
        if rnd == 3:   # a sparse batch: most tiles get no units at all
            recs = recs[(recs["group"] % 700) < 3]
        # group order; inside a group arrival order, with each EXT right behind its REJECT
        order = np.argsort(recs["group"], kind="stable")
        _compact_round(arena, n, np.ascontiguousarray(recs[order]), ref, blob, d_bufs)
    # empty stream
    _compact_round(arena, n, np.zeros(0, dtype=B.APPEND_RESP_DTYPE), ref, blob, d_bufs)
    # a stream that claims ONE_WAVE but holds two records for one cell: the per-unit kernel applies
    # the first it sees, refuses the other and counts it
    dup = np.zeros(2, dtype=B.APPEND_RESP_DTYPE)
    m = int(ref.matched[1, 40])
    dup[0] = (40, 1, 0, 0, m + 5, m)
    dup[1] = (40, 1, 0, 0, m + 5, m)
    nb, _ = B.pack_compact(dup, blob)
    hdr = blob[:64].view(B.COMPACT_HDR_DTYPE)
    assert not (hdr[0]["flags"] & B.COMPACT_ONE_WAVE)
    hdr[0]["flags"] |= B.COMPACT_ONE_WAVE
    d_blob, d_off, d_res, d_bm, d_com, d_bad = d_bufs
    arena.h2d(d_blob, blob[:nb])
    arena.h2d(d_bad, np.zeros(1, dtype=np.uint32))
    arena.compact_tile_index_device(d_blob, blob, d_off, d_bad)
    arena.step_compact_device(d_blob, blob, d_off, d_dup=d_bad)
    bad = np.zeros(1, dtype=np.uint32)
    arena.d2h(bad, d_bad)
    assert bad[0] == 1
    O.arena_apply(ref, dup[:1], mode=0)
    O.arena_recompute(ref)
    assert_columns_equal(arena.read_columns(n), ref, n, "duplicate refused")
    arena.close()


def _random_state(n, rng):
    """Arbitrary configurations (joint, learners, group commit, no self) and per-peer states."""
    c = O.new_columns(n, n)
    for g in range(n):
        inc = int(rng.integers(1, 256))
        out = int(rng.integers(0, 256)) if rng.random() < 0.3 else 0
        learners = int(rng.integers(0, 256)) & ~(inc | out) if rng.random() < 0.4 else 0
        voters = [s_ for s_ in range(8) if (inc | out) >> s_ & 1]
        self_slot = int(rng.choice(voters)) if rng.random() < 0.9 else None
        c.meta[g] = O.make_meta(inc, out, learners, self_slot, group_commit=bool(rng.random() < 0.15))
        base = int(rng.integers(100, 1 << 40))
        c.last_index[g] = base + int(rng.integers(0, 10))
        c.term_start[g] = (1 << 64) - 1 if rng.random() < 0.05 else max(1, base - int(rng.integers(0, 30)))
        c.committed[g] = base - int(rng.integers(0, 40))
        c.term[g] = int(rng.integers(1, 1000))
        for s_ in range(8):
            m = base - int(rng.integers(0, 50))
            c.matched[s_, g] = m
            c.next_idx[s_, g] = m + 1 + int(rng.integers(0, 5))
            c.peer_committed[s_, g] = m - int(rng.integers(0, 5))
            state = int(rng.choice([O.STATE_PROBE, O.STATE_REPLICATE, O.STATE_REPLICATE, O.STATE_SNAPSHOT]))
            c.pflags[s_, g] = state | (O.PF_PAUSED if rng.random() < 0.3 else 0) | (O.PF_INS_FULL if rng.random() < 0.2 else 0) | \
                (O.PF_RECENT_ACTIVE if rng.random() < 0.5 else 0)
            c.pending_snapshot[s_, g] = m + int(rng.integers(0, 6)) if state == O.STATE_SNAPSHOT else 0
            c.pending_request_snapshot[s_, g] = int(rng.integers(1, 100)) if rng.random() < 0.05 else 0
            c.commit_group_id[s_, g] = int(rng.integers(0, 4))
    return c


def _random_batch(ref, n, rng, per_cell):
    """Group-ordered batch; `per_cell` > 1 lets a (group, peer) cell receive several records."""
    rows = []
    for g in range(n):
        if rng.random() < 0.3:
            continue
        meta = int(ref.meta[g])
        has_self, self_slot = bool(meta & O.META_HAS_SELF), (meta >> 24) & 7
        slots = rng.permutation(8)[: int(rng.integers(1, 6))]
        for s_ in slots:
            s_ = int(s_)
            for _ in range(int(rng.integers(1, per_cell + 1))):
                m, nx = int(ref.matched[s_, g]), int(ref.next_idx[s_, g])
                kind = rng.random()
                if has_self and s_ == self_slot:
                    idx = m + int(rng.integers(0, 8))
                    rows.append((g, s_, B.REC_LOCAL, 0, idx, 0 if rng.random() < 0.2 else idx + int(rng.integers(0, 5))))
                elif kind < 0.7:
                    idx = max(0, m + int(rng.integers(-6, 12)))
                    commit = idx + 3 if rng.random() < 0.03 else max(0, idx - int(rng.integers(0, 300 if rng.random() < 0.05 else 6)))
                    rows.append((g, s_, 0, 0, idx, commit))
                else:
                    idx = int(rng.choice([nx - 1, m, m + 1, m + 3, max(0, m - 2)]))
                    rows.append((g, s_, B.REC_REJECT, 0, idx, max(0, m - int(rng.integers(0, 4)))))
                    if rng.random() < 0.85:
                        rows.append((g, s_, B.REC_EXT, 0, max(0, idx + int(rng.integers(-5, 3))),
                                     int(rng.integers(1, 1 << 30)) if rng.random() < 0.2 else 0))
    return np.array(rows, dtype=B.APPEND_RESP_DTYPE) if rows else np.zeros(0, dtype=B.APPEND_RESP_DTYPE)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_every_ingest_path_agrees_with_the_oracle_on_random_states(seed):
    """Differential test: arbitrary configurations / peer states, random group-ordered batches (accepts,
    stale acks, commits above the index, leader-local records, rejections with and without hint and
    snapshot request, peers the group does not have), through EVERY way of handing a batch to the
    engine -- rings + waves, bulk staging, zero-copy packed, zero-copy compact (fused), the records
    API, the device-resident fused kernels -- each compared with the oracle column by column."""
    rng = np.random.default_rng(seed)
    n = 2500
    init = _random_state(n, rng)
    ref = O.copy_columns(init)
    names = ["enqueue", "bulk", "packed", "compact", "records", "fused16", "fusedc"]
    arenas = {}
    for name in names:
        # (the wave-splitting paths keep later waves in an overflow area sized from the arena capacity)
        a = B.Arena(32 * n if name in ("enqueue", "bulk") else n)
        a.group_alloc_range(n)
        a.load_columns(init)
        arenas[name] = a
    pk_host = arenas["packed"].host_alloc_packed(40 * n)
    blob_host = arenas["compact"].host_alloc_bytes(B.compact_bound(40 * n))
    pk = np.zeros((40 * n, 2), dtype=np.uint64)
    f16 = arenas["fused16"]
    d16 = (f16.device_alloc(pk.nbytes), f16.device_alloc(4 * (n // B.tile_groups() + 2)))
    blob, dc = _compact_bufs(arenas["fusedc"], n, 40)
    for rnd in range(5):
        per_cell = 3 if rnd >= 3 else 1          # the last rounds: several records per (group, peer)
        recs = _random_batch(ref, n, rng, per_cell)
        O.arena_apply(ref, recs, mode=0)
        want_adv, want_bm, _, _ = O.arena_recompute(ref)
        words = (n + 31) // 32
        for name in names:
            a = arenas[name]
            if per_cell > 1 and name in ("packed", "fused16"):
                continue                          # these promise one record per cell
            if name == "enqueue":
                a.enqueue(recs)
                r = a.step(0)
            elif name == "bulk":
                a.enqueue_bulk(recs, sorted_by_group=True)
                r = a.step(0)
            elif name == "packed":
                k = a.pack_records(recs, pk_host)
                a.step_begin_packed(pk_host, k, 0)
                r = a.step_wait()
            elif name == "compact":
                nb, _ = B.pack_compact(recs, blob_host)
                a.step_begin_compact(blob_host, nb, 0)
                r = a.step_wait()
            elif name == "records":
                a.step_begin_records(recs, 0)
                r = a.step_wait()
            elif name == "fused16":
                k = a.pack_records(recs, pk)
                a.h2d(d16[0], pk[:max(k, 1)])
                a.h2d(d16[1], B.tile_index(pk, k, n))
                a.step_sorted_device(d16[0], k, d16[1])
                r = None
            else:
                _compact_round_nocheck(a, recs, blob, dc)
                r = None
            if r is not None:
                assert r.n_advanced == want_adv and r.n_duplicates == 0, (name, rnd)
                bm, _ = a.step_results(n)
                assert np.array_equal(bm[:words], want_bm[:words]), (name, rnd)
            assert_columns_equal(a.read_columns(n), ref, n, f"{name}, round {rnd}, seed {seed}")
        if per_cell == 1:     # fused16 / packed skipped the multi-record rounds: keep them in step
            continue
        for name in ("packed", "fused16"):
            arenas[name].load_columns(ref)
    for a in arenas.values():
        a.close()


def _compact_round_nocheck(arena, recs, blob, d_bufs):
    nb, _ = B.pack_compact(recs, blob)
    d_blob, d_off, d_res, d_bm, d_com, d_bad = d_bufs
    arena.h2d(d_blob, blob[:nb])
    arena.h2d(d_bad, np.zeros(1, dtype=np.uint32))
    arena.compact_tile_index_device(d_blob, blob, d_off, d_bad)
    arena.step_compact_device(d_blob, blob, d_off, d_dup=d_bad)
    bad = np.zeros(1, dtype=np.uint32)
    arena.d2h(bad, d_bad)
    assert bad[0] == 0


def test_mci_and_properties_at_full_size():
    """1M x 7 joint: maximal_committed_index for every group vs the oracle, plus
    size-independent properties: idempotence, monotone commit, joint = min of halves."""
    n = 1_000_000
    synth = B.Synth(n, 0x5EED0004, joint=True)
    arena = B.Arena(n)
    arena.group_alloc_range(n)
    arena.load_columns(synth.initial)
    d_mci, d_gc = arena.device_alloc(8 * arena.cap), arena.device_alloc(arena.cap)
    d_bm = arena.device_alloc(arena.cap // 8)
    arena.recompute(0, n, d_adv=d_bm, d_mci=d_mci, d_gc=d_gc)
    mci = np.zeros(arena.cap, dtype=np.uint64)
    bm1 = np.zeros(arena.cap // 32, dtype=np.uint32)
    arena.d2h(mci, d_mci)
    arena.d2h(bm1, d_bm)
    ref = O.copy_columns(synth.initial)
    want_adv, want_bm, want_mci, _ = O.arena_recompute(ref, want_mci=True)
    assert np.array_equal(mci[:n], want_mci[:n])
    assert checksum(mci[:n]) == checksum(want_mci[:n])
    assert np.array_equal(bm1[: len(want_bm)], want_bm)
    committed1 = arena.column_read(B.COL_COMMITTED, 0, 0, n, np.uint64)
    assert np.array_equal(committed1, ref.committed[:n])
    assert np.all(committed1 >= synth.initial.committed[:n])          # never decreases
    # idempotence: a second pass over unchanged progress advances nothing
    arena.recompute(0, n, d_adv=d_bm)
    arena.d2h(bm1, d_bm)
    assert not bm1.any()
    assert np.array_equal(arena.column_read(B.COL_COMMITTED, 0, 0, n, np.uint64), committed1)
    # joint = min(incoming-only, outgoing-only): re-run with each half as a plain majority
    meta = synth.initial.meta[:n].copy()
    halves = []
    for shift in (0, 8):
        m = ((meta >> shift) & 0xFF) | (meta & 0xFF000000)
        arena.column_write(B.COL_META, 0, 0, m.astype(np.uint32))
        arena.recompute(0, n, d_mci=d_mci)
        arena.d2h(mci, d_mci)
        halves.append(mci[:n].copy())
    assert np.array_equal(np.minimum(halves[0], halves[1]), want_mci[:n])
    arena.close()


def test_partial_ranges_and_bitmap_edges():
    n = 10_000
    synth = B.Synth(n, 0x5EED0002)
    arena = B.Arena(n)
    arena.group_alloc_range(n)
    arena.load_columns(synth.initial)
    ref = O.copy_columns(synth.initial)
    d_bm = arena.device_alloc(arena.cap // 8)
    bm = np.full(arena.cap // 32, 0xFFFFFFFF, dtype=np.uint32)
    arena.h2d(d_bm, bm)
    first, cnt = 37, 4321   # neither end on a 32-group boundary
    arena.recompute(first, cnt, d_adv=d_bm)
    arena.d2h(bm, d_bm)
    want_bm = np.full(arena.cap // 32, 0xFFFFFFFF, dtype=np.uint32)
    for g in range(first, first + cnt):
        if not O.arena_maybe_commit(ref, g):
            want_bm[g >> 5] &= ~np.uint32(1 << (g & 31))
    assert np.array_equal(bm, want_bm)
    assert np.array_equal(arena.column_read(B.COL_COMMITTED, 0, 0, n, np.uint64), ref.committed[:n])
    arena.close()


def test_send_list_vs_oracle():
    """SURVEY 8(f) rank 2: the post-commit send decisions (bcast_append over the groups whose commit
    advanced, gated by Progress::is_paused) as a stream-compaction kernel; the same entries as the
    oracle's loop, as a set (the reference iterates a HashMap: no order is promised)."""
    n = 60_001
    synth = B.Synth(n, 0x5EED000C)
    cols = synth.initial
    rng = np.random.default_rng(12)
    learners = rng.random(n) < 0.3                      # a learner in slot 6: gets appends too
    cols.meta[:n] |= (learners.astype(np.uint32) << np.uint32(16 + 6))
    cols.next_idx[6, :n] = np.where(learners, cols.matched[0, :n] - 5, 0)
    cols.pflags[6, :n] = np.where(learners, O.STATE_REPLICATE, 0)
    # every pause reason: paused probes, full inflight windows, snapshot state, pending snapshot requests
    cols.pflags[1, :n] |= np.where(rng.random(n) < 0.2, O.PF_INS_FULL, 0).astype(np.uint8)
    cols.pflags[2, :n] = np.where(rng.random(n) < 0.1, O.STATE_SNAPSHOT, cols.pflags[2, :n])
    cols.pflags[3, :n] = np.where(rng.random(n) < 0.1, O.STATE_PROBE | O.PF_PAUSED, cols.pflags[3, :n])
    cols.pending_request_snapshot[4, :n] = np.where(rng.random(n) < 0.05, 77, 0)
    arena = B.Arena(n)
    arena.group_alloc_range(n)
    arena.load_columns(cols)
    ref = O.copy_columns(cols)

    def as_set(e):
        return sorted(zip(e["group"].tolist(), e["peer_slot"].tolist(), e["flags"].tolist(), e["next_idx"].tolist()))

    for rnd in range(3):
        recs = synth.next_round().copy()
        arena.enqueue(recs)
        arena.step(0)
        O.arena_apply(ref, recs, mode=0)
        _, want_bm, _, _ = O.arena_recompute(ref)
        want = O.arena_send_list(ref, want_bm)
        got = arena.step_send_list(8 * n)
        assert len(got) == len(want) > n // 10
        assert as_set(got) == as_set(want), f"send list differs in round {rnd}"
        assert not np.any(got["peer_slot"] == 0)                      # never to the leader itself
    # a plain bcast_append (no bitmap) over a sub-range, through the device entry point
    d_out, d_cnt = arena.device_alloc(16 * 8 * n), arena.device_alloc(8)
    first, cnt = 1000, 40_003
    arena.send_list_device(first, cnt, None, d_out, 8 * n, d_cnt)
    total = np.zeros(1, dtype=np.uint64)
    arena.d2h(total, d_cnt)
    want = O.arena_send_list(ref, None, first, cnt)
    assert total[0] == len(want)
    got = np.zeros(len(want), dtype=B.SEND_ENTRY_DTYPE)
    arena.d2h(got, d_out)
    assert as_set(got) == as_set(want)
    # too small a buffer: the count still says how many there are
    arena.send_list_device(first, cnt, None, d_out, 10, d_cnt)
    arena.d2h(total, d_cnt)
    assert total[0] == len(want)
    with pytest.raises(B.RaftGpuError):
        arena.step_send_list(5)
    arena.close()


def test_heartbeat_commits_vs_oracle():
    """SURVEY 8(f) rank 3, leader side: bcast_heartbeat's per-peer commit = min(matched, committed)
    (raft.rs:838-840, 875-889) as one dense pass, on arbitrary configurations."""
    rng = np.random.default_rng(21)
    n = 5000
    init = _random_state(n, rng)
    arena = B.Arena(n)
    arena.group_alloc_range(n)
    arena.load_columns(init)
    d_out = arena.device_alloc(8 * 8 * n)
    for first, cnt in ((0, n), (37, 3001)):
        arena.heartbeat_commits_device(first, cnt, d_out)
        got = np.zeros((8, cnt), dtype=np.uint64)
        arena.d2h(got, d_out)
        assert np.array_equal(got, O.arena_heartbeat_commits(init, first, cnt))
    arena.close()


def test_vote_tally_batched_vs_oracle():
    n = 50_000
    rng = np.random.default_rng(7)
    arena = B.Arena(n)
    arena.group_alloc_range(n)
    c = O.new_columns(arena.cap, n)
    inc = rng.integers(0, 256, n, dtype=np.uint32)
    out = np.where(rng.random(n) < 0.5, 0, rng.integers(0, 256, n)).astype(np.uint32)
    c.meta[:n] = inc | (out << 8)
    votes = rng.integers(0, 3, (B.SLOTS, arena.cap), dtype=np.uint8)
    arena.column_write(B.COL_META, 0, 0, c.meta[:n])
    for s in range(B.SLOTS):
        arena.column_write(B.COL_VOTES, s, 0, votes[s, :n])
    d_out = arena.device_alloc(4 * arena.cap)
    arena.tally_votes(0, n, d_out)
    got = np.zeros(arena.cap, dtype=np.uint32)
    arena.d2h(got, d_out)
    for g in range(n):      # every group
        gr, rj, r = O.arena_vote_result(c, votes, g)
        assert int(got[g]) == r | (gr << 8) | (rj << 16), g
    arena.close()


def test_concurrent_enqueue_from_eight_threads():
    """The threading contract of SURVEY 8(b): raftgpu_enqueue_append_resp from several caller threads at once,
    one ring each, different groups on different threads (raw_node.rs:284 / raft.rs:292-294).  Eight threads
    enqueue TWO rounds each in small, ragged calls (so every cell gets two records -> two waves); columns,
    advanced bitmap, commit indexes and the per-ring results against the oracle, three steps in a row."""
    import threading
    n, T = 40_000, 8
    synth = B.Synth(n, 0x7E57, k_peers=5)
    arena = B.Arena(n, n_rings=T)
    assert arena.group_alloc_range(n) == 0
    arena.load_columns(synth.initial)
    ref = O.copy_columns(synth.initial)
    rng = np.random.default_rng(99)
    for step in range(3):
        r1, r2 = synth.next_round().copy(), synth.next_round().copy()
        per_thread = []
        for t in range(T):
            # thread t owns the groups g % T == t; its records keep their arrival order: round 1, then (for one
            # group in sixteen: the later waves share a small overflow buffer) round 2
            second = r2[(r2["group"] % T == t) & ((r2["group"] // T) % 16 == 0)]
            mine = np.concatenate([r1[r1["group"] % T == t], second])
            per_thread.append(mine)
        errors = []
        start = threading.Barrier(T)

        def work(t):
            try:
                recs = per_thread[t]
                start.wait()
                i = 0
                while i < len(recs):
                    k = int(rng.integers(1, 700))
                    j = min(len(recs), i + k)
                    while j < len(recs) and (recs[j]["flags"] & B.REC_EXT):   # never separate a REJECT from its EXT
                        j += 1
                    arena.enqueue(recs[i:j], ring=t)      # ctypes releases the GIL: the calls really overlap
                    i = j
            except Exception as e:   # noqa: BLE001
                errors.append(e)

        th = [threading.Thread(target=work, args=(t,)) for t in range(T)]
        for x in th:
            x.start()
        for x in th:
            x.join()
        assert not errors, errors
        r = arena.step(B.STEP_READ_COMMITTED | B.STEP_READ_RESULTS)
        assert r.n_waves == 2 and r.n_records == sum(len(x) for x in per_thread)
        want_adv = None
        for t in range(T):   # cells of different threads are disjoint: any interleaving of the threads is the same
            want_res = O.arena_apply(ref, per_thread[t], mode=0)
            assert np.array_equal(arena.record_results(t), want_res), (step, t)
        want_adv, want_bm, _, _ = O.arena_recompute(ref)
        bm, com = arena.step_results(n)
        assert r.n_advanced == want_adv and np.array_equal(bm, want_bm[: len(bm)])
        adv = bitmap_to_bool(bm, n)
        assert np.array_equal(com[adv], ref.committed[:n][adv])
        assert_columns_equal(arena.read_columns(n), ref, n, f"concurrent enqueue step {step}")
    arena.close()


# --------------------------------------------------------------------------- heartbeat responses / update_state

def random_arena_state(n, seed):
    """Arbitrary configurations and peer states for n groups (joint, learners, every ProgressState, pause /
    inflights-full bits, snapshot requests), as host columns."""
    rng = np.random.default_rng(seed)
    c = O.new_columns(n + 128 - n % 128 if n % 128 else n, n)
    inc = rng.integers(0, 256, n, dtype=np.uint32)
    out = np.where(rng.random(n) < 0.5, 0, rng.integers(0, 256, n)).astype(np.uint32)
    lrn = rng.integers(0, 256, n, dtype=np.uint32) & ~(inc | out)
    c.meta[:n] = inc | (out << 8) | (lrn << 16)
    base = rng.integers(1000, 1 << 40, n, dtype=np.uint64)
    c.last_index[:n] = base
    c.committed[:n] = base - rng.integers(0, 50, n).astype(np.uint64)
    for s in range(B.SLOTS):
        c.matched[s, :n] = base - rng.integers(0, 3, n).astype(np.uint64) * rng.integers(0, 100, n).astype(np.uint64)
        c.next_idx[s, :n] = c.matched[s, :n] + 1 + rng.integers(0, 5, n).astype(np.uint64)
        c.peer_committed[s, :n] = c.matched[s, :n] - rng.integers(0, 20, n).astype(np.uint64)
        c.pflags[s, :n] = rng.integers(0, 3, n) | (rng.integers(0, 2, n) << 2) | (rng.integers(0, 2, n) << 3) | (rng.integers(0, 2, n) << 4)
        c.pending_request_snapshot[s, :n] = np.where(rng.random(n) < 0.1, rng.integers(1, 1 << 30, n), 0)
    return c, rng


def test_heartbeat_responses_vs_oracle():
    """handle_heartbeat_response (raft.rs:1777-1804) as a batch: every column and every result byte, on arbitrary
    configurations; an unknown peer, a record without the flag, and the one-record-per-cell rule."""
    n = 30_000
    c, rng = random_arena_state(n, 41)
    a = B.Arena(n)
    assert a.group_alloc_range(n) == 0
    a.load_columns(c)
    ref = O.copy_columns(c)
    for rnd in range(3):
        k = 60_000
        g = rng.integers(0, n, k, dtype=np.uint32)
        s = rng.integers(0, 9, k).astype(np.uint8)          # slot 8: no such slot
        cells, first = np.unique(g.astype(np.uint64) * 16 + s, return_index=True)
        recs = np.zeros(len(first), dtype=B.APPEND_RESP_DTYPE)
        recs["group"], recs["peer_slot"] = g[first], s[first]
        recs["flags"] = np.where(rng.random(len(first)) < 0.97, B.REC_HEARTBEAT, 0)
        recs["commit"] = ref.committed[recs["group"]] - rng.integers(0, 30, len(first)).astype(np.uint64)
        got = a.heartbeat_resp(recs)
        want = O.arena_apply_heartbeat(ref, recs)
        assert np.array_equal(got, want), rnd
        assert_columns_equal(a.read_columns(n), ref, n, f"heartbeat round {rnd}")
        assert np.count_nonzero(want & B.RES_SEND) > 1000 and np.count_nonzero(want == B.RES_NO_PROGRESS) > 1000
    dup = np.zeros(2, dtype=B.APPEND_RESP_DTYPE)
    slot = int(np.flatnonzero([(int(ref.meta[5]) >> b) & 1 for b in range(8)] + [1])[0]) % 8
    dup["group"], dup["peer_slot"], dup["flags"] = 5, slot, B.REC_HEARTBEAT
    if (int(ref.meta[5]) | int(ref.meta[5]) >> 8 | int(ref.meta[5]) >> 16) >> slot & 1:
        with pytest.raises(B.RaftGpuError):
            a.heartbeat_resp(dup)
    a.close()


def test_update_state_vs_oracle_and_probe_peers_are_sent_to_once():
    """Progress::update_state over a send list (progress.rs:231-243).  Then the property the ADVICE item is about:
    after update_state a probing peer is paused, so the NEXT send list does not name it again."""
    n = 20_000
    c, rng = random_arena_state(n, 43)
    a = B.Arena(n)
    assert a.group_alloc_range(n) == 0
    a.load_columns(c)
    ref = O.copy_columns(c)
    d_cnt = a.device_alloc(8)
    cap = 8 * n
    d_out = a.device_alloc(16 * cap)
    a.send_list_device(0, n, None, d_out, cap, d_cnt)       # bcast_append over every group
    cnt = np.zeros(1, dtype=np.uint64)
    a.d2h(cnt, d_cnt)
    entries = np.zeros(int(cnt[0]), dtype=B.SEND_ENTRY_DTYPE)
    a.d2h(entries, d_out)
    entries = entries[np.lexsort((entries["peer_slot"], entries["group"]))]
    want_list = O.arena_send_list(ref)
    assert np.array_equal(entries, want_list)
    sent = entries.copy()
    sent["next_idx"] = ref.last_index[sent["group"]]          # everything up to last_index went out
    got = a.update_state(sent)
    want = O.arena_update_state(ref, sent)
    assert np.array_equal(got, want) and set(np.unique(want)) <= {1}      # the list never names Snapshot peers
    assert_columns_equal(a.read_columns(n), ref, n, "update_state")
    a.send_list_device(0, n, None, d_out, cap, d_cnt)
    a.d2h(cnt, d_cnt)
    again = np.zeros(int(cnt[0]), dtype=B.SEND_ENTRY_DTYPE)
    a.d2h(again, d_out)
    probe_cells = {(int(g), int(s)) for g, s in zip(sent["group"], sent["peer_slot"]) if (c.pflags[s, g] & 3) == O.STATE_PROBE}
    assert probe_cells and not probe_cells & {(int(g), int(s)) for g, s in zip(again["group"], again["peer_slot"])}
    # a Snapshot-state peer is a panic in the reference: reported, not applied
    snap = np.zeros(1, dtype=B.SEND_ENTRY_DTYPE)
    gs = np.argwhere((ref.pflags[:, :n] & 3) == O.STATE_SNAPSHOT)
    gs = [(s, g) for s, g in gs if ((int(ref.meta[g]) | int(ref.meta[g]) >> 8 | int(ref.meta[g]) >> 16) >> s) & 1]
    snap["peer_slot"], snap["group"], snap["next_idx"] = gs[0][0], gs[0][1], 5
    assert a.update_state(snap).tolist() == [0xFF] == O.arena_update_state(ref, snap).tolist()
    a.close()


def test_async_record_steps_keep_two_ticks_in_flight():
    """RAFTGPU_STEP_ASYNC: raftgpu_step_begin_records returns once the staging threads have the batch; the submitter
    thread packs / copies / launches.  Tick j+1 is begun before tick j is waited for, six ticks in a row: every
    step's advanced bitmap and commit indexes and the final columns against the oracle."""
    n = 300_000
    synth = B.Synth(n, 0xA51C, k_peers=5)
    os.environ.setdefault("RAFTGPU_HOST_THREADS", "8")
    arena = B.Arena(n, n_rings=8)
    assert arena.group_alloc_range(n) == 0
    arena.load_columns(synth.initial)
    ref = O.copy_columns(synth.initial)
    rounds = [synth.next_round().copy() for _ in range(6)]
    flags = B.STEP_READ_COMMITTED | B.STEP_ASYNC
    arena.step_begin_records(rounds[0], flags)
    for j in range(len(rounds)):
        if j + 1 < len(rounds):
            arena.step_begin_records(rounds[j + 1], flags)      # waits for submission j, then returns at once
        r = arena.step_wait()
        O.arena_apply(ref, rounds[j], mode=0)
        want_adv, want_bm, _, _ = O.arena_recompute(ref)
        bm, com = arena.step_results(n)
        assert r.n_advanced == want_adv and r.n_records == int(np.count_nonzero((rounds[j]["flags"] & B.REC_EXT) == 0))
        assert np.array_equal(bm, want_bm[: len(bm)]), j
        adv = bitmap_to_bool(bm, n)
        assert np.array_equal(com[adv], ref.committed[:n][adv])
    assert_columns_equal(arena.read_columns(n), ref, n, "async steps")
    # an ordinary call right after an asynchronous one first lets the submission finish
    e1, e2 = synth.next_round().copy(), synth.next_round().copy()
    arena.step_begin_records(e1, flags)
    arena.step_begin_records(e2, B.STEP_READ_COMMITTED)      # synchronous form: two steps in flight, in order
    for e in (e1, e2):
        arena.step_wait()
        O.arena_apply(ref, e, mode=0)
        O.arena_recompute(ref)
    assert_columns_equal(arena.read_columns(n), ref, n, "async then sync")
    arena.close()


def test_raw_record_steps_match_the_packed_ones():
    """RAFTGPU_STEP_RAW: the 24-byte records cross PCIe as they are (no host packing) and go through the scatter
    kernel.  Same rounds as the packed form on a second arena: identical results, result bytes per record; a
    second record for a cell is refused (one wave, verified on the GPU)."""
    n = 200_000
    synth = B.Synth(n, 0x0AB1, k_peers=5)
    a1, a2 = B.Arena(n), B.Arena(n)
    for a in (a1, a2):
        assert a.group_alloc_range(n) == 0
        a.load_columns(synth.initial)
    ref = O.copy_columns(synth.initial)
    buf = a2.host_alloc_bytes(24 * (5 * n + 64)).view(B.APPEND_RESP_DTYPE)
    for rnd in range(3):
        recs = synth.next_round().copy()
        a1.step_begin_records(recs, B.STEP_READ_COMMITTED)
        r1 = a1.step_wait()
        buf[: len(recs)] = recs
        a2.step_begin_records(buf[: len(recs)], B.STEP_READ_COMMITTED | B.STEP_READ_RESULTS | B.STEP_RAW)
        r2 = a2.step_wait()
        want_res = O.arena_apply(ref, recs, mode=0)
        want_adv, want_bm, _, _ = O.arena_recompute(ref)
        assert r1.n_advanced == r2.n_advanced == want_adv and r2.n_duplicates == 0
        assert r2.h2d_bytes == 24 * len(recs)
        assert np.array_equal(a2.slot_results()[: len(recs)], want_res)
        b2, c2 = a2.step_results(n)
        assert np.array_equal(b2, want_bm[: len(b2)])
        adv = bitmap_to_bool(b2, n)
        assert np.array_equal(c2[adv], ref.committed[:n][adv])
    assert_columns_equal(a2.read_columns(n), ref, n, "raw steps")
    assert_columns_equal(a1.read_columns(n), ref, n, "packed steps")
    dup = np.concatenate([recs[:1000], recs[:1]])
    dup = dup[(dup["flags"] & (B.REC_EXT | B.REC_REJECT)) == 0]
    a2.step_begin_records(np.ascontiguousarray(np.concatenate([dup, dup[:1]])), B.STEP_RAW)
    r = a2.step_wait(check=False)
    assert r.status == B.ERR_INVALID and r.n_duplicates >= 1
    a1.close()
    a2.close()


def test_hybrid_record_steps_split_between_packer_and_dma(monkeypatch):
    """RAFTGPU_STEP_HYBRID: the head of the batch through the host packer + fused kernel, the tail over PCIe as it is
    + scatter kernel, for several splits (0 % = everything raw, 100 % = nothing), synchronous and asynchronous: results
    identical to the oracle's; the bytes that crossed PCIe add up; a batch that is not in group order is refused on the
    device (the two parts must not share a group); pageable records ignore the flag."""
    n = 200_000
    synth = B.Synth(n, 0x0AB2, k_peers=5)
    a = B.Arena(n)
    assert a.group_alloc_range(n) == 0
    a.load_columns(synth.initial)
    ref = O.copy_columns(synth.initial)
    buf = a.host_alloc_bytes(24 * (5 * n + 64)).view(B.APPEND_RESP_DTYPE)       # pinned
    seen_split = 0
    for rnd, (pct, extra) in enumerate([("40", 0), ("0", 0), ("100", 0), ("75", B.STEP_ASYNC), (None, B.STEP_ASYNC), ("55", 0)]):
        if pct is None:
            monkeypatch.delenv("RAFTGPU_HYBRID_PACK_PCT", raising=False)      # the library's own model
        else:
            monkeypatch.setenv("RAFTGPU_HYBRID_PACK_PCT", pct)
        recs = synth.next_round()
        k = len(recs)
        buf[:k] = recs
        a.step_begin_records(buf[:k], B.STEP_READ_COMMITTED | B.STEP_HYBRID | extra)
        r = a.step_wait()
        O.arena_apply(ref, recs, mode=0)
        want_adv, want_bm, _, _ = O.arena_recompute(ref)
        assert r.n_advanced == want_adv and r.n_duplicates == 0, (rnd, pct)
        assert np.count_nonzero((recs["flags"] & B.REC_EXT) == 0) <= r.n_records <= k, (rnd, r.n_records, k)
        if pct == "0":
            assert r.h2d_bytes >= 24 * k
        elif pct == "100":
            assert r.h2d_bytes < 8 * k
        elif pct is not None:
            raw = (1 - int(pct) / 100) * 24 * k
            assert 0.9 * raw < r.h2d_bytes < raw + 8 * k, (pct, r.h2d_bytes, k)
            seen_split += 1
        bm, com = a.step_results(n)
        assert np.array_equal(bm, want_bm[: len(bm)]), (rnd, pct)
        adv = bitmap_to_bool(bm, n)
        assert np.array_equal(com[adv], ref.committed[:n][adv])
        assert_columns_equal(a.read_columns(n), ref, n, f"hybrid round {rnd} ({pct} % packed)")
    assert seen_split == 3
    # pageable records: the flag is ignored, the step is the ordinary one
    monkeypatch.setenv("RAFTGPU_HYBRID_PACK_PCT", "50")
    recs = synth.next_round().copy()
    a.step_begin_records(recs, B.STEP_HYBRID)
    r = a.step_wait()
    O.arena_apply(ref, recs, mode=0)
    O.arena_recompute(ref)
    assert r.h2d_bytes < 8 * len(recs)
    assert_columns_equal(a.read_columns(n), ref, n, "pageable + hybrid")
    # the two halves of the batch swapped: the raw part now holds groups below the packed part's -> refused
    recs = synth.next_round()
    k = len(recs)
    h = k // 2
    while recs["group"][h] == recs["group"][h - 1] or recs["flags"][h] & B.REC_EXT:
        h += 1
    buf[: k - h] = recs[h:]
    buf[k - h: k] = recs[:h]
    a.step_begin_records(buf[:k], B.STEP_HYBRID)
    r = a.step_wait(check=False)
    assert r.status == B.ERR_INVALID and r.n_duplicates >= 1
    a.close()


def test_batches_that_cover_only_some_groups_at_full_size():
    """A tick in which only part of the store's groups have traffic -- the first 5 % of the groups, every seventh tile,
    a random 2 % -- at 1M groups, through both fused kernels (records API -> compact stream, and packed records + tile
    index, device resident).  Light (record-less) tiles finish early and their loads land out of order with the heavy
    ones: the consumers of the TMA ring must still pair every stage with its own tile (this hung / corrupted results
    before the consumers checked the previous use of a stage, wait_stage in k_tile.cuh).  Several rounds each: the failure was intermittent."""
    n = 1_000_000
    synth = B.Synth(n, 0x5A7E, k_peers=5)
    arenas = [B.Arena(n), B.Arena(n)]
    for a in arenas:
        assert a.group_alloc_range(n) == 0
        a.load_columns(synth.initial)
    ref = O.copy_columns(synth.initial)
    rng = np.random.default_rng(5)
    pk = np.zeros((6 * n, 2), dtype=np.uint64)
    d_pk, d_off = arenas[1].device_alloc(pk.nbytes), arenas[1].device_alloc(4 * (n // B.tile_groups() + 2))
    d_bm = arenas[1].device_alloc(4 * (n // 32 + 1))
    words = (n + 31) // 32
    for rnd in range(8):
        recs = synth.next_round()
        g = recs["group"]
        if rnd % 4 == 0:
            keep = g < n // 20
        elif rnd % 4 == 1:
            keep = (g // 256) % 7 == 0
        elif rnd % 4 == 2:
            chosen = rng.random(n) < 0.02
            keep = chosen[g]
        else:
            keep = g >= n - n // 50
        part = np.ascontiguousarray(recs[keep])
        O.arena_apply(ref, part, mode=0)
        want_adv, want_bm, _, _ = O.arena_recompute(ref)
        a = arenas[0]
        a.step_begin_records(part, B.STEP_READ_COMMITTED)
        r = a.step_wait()
        assert r.n_advanced == want_adv and r.n_duplicates == 0, rnd
        bm, com = a.step_results(n)
        assert np.array_equal(bm[:words], want_bm[:words]), rnd
        adv = bitmap_to_bool(bm, n)
        assert np.array_equal(com[adv], ref.committed[:n][adv])
        a = arenas[1]
        k = a.pack_records(part, pk)
        a.h2d(d_pk, pk[: max(k, 1)])
        a.h2d(d_off, B.tile_index(pk, k, n))
        a.step_sorted_device(d_pk, k, d_off, d_adv=d_bm)
        got_bm = np.zeros(words, dtype=np.uint32)
        a.d2h(got_bm, d_bm)
        assert np.array_equal(got_bm, want_bm[:words]), rnd
        for a, name in zip(arenas, ("records api", "packed device")):
            got = a.read_columns(n)
            for col in ("matched", "next_idx", "peer_committed", "pflags", "committed", "last_index"):
                assert checksum(getattr(got, col)) == checksum(getattr(ref, col)[..., :n]), (name, rnd, col)
    for a in arenas:
        a.close()
