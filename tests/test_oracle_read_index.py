"""The read-index oracle (tests/read_index_oracle.py) pinned by the reference's read-index tests, and its arena form (the
device's bounded layout and batch rules) against its literal form on random traffic."""
import numpy as np
import pytest

import read_index_oracle as R
from helpers import B


@pytest.mark.parametrize("form", ["literal", "arena"])
@pytest.mark.parametrize("name", sorted(R.SCENARIOS))
def test_reference_scenario(name, form):
    R.SCENARIOS[name](R.LiteralDriver() if form == "literal" else R.ArenaDriver())


def test_read_only_advance_and_last_ctx_literal():
    ro = R.ReadOnly()
    assert ro.last_pending_request_ctx() is None
    assert ro.add_request(5, b"a", 2, 1) and ro.add_request(6, b"b", 2, 1) and ro.add_request(7, b"c", 3, 1)
    assert not ro.add_request(8, b"a", 3, 1)                          # read_only.rs:88-90
    assert ro.recv_ack(2, b"zz") is None                              # unknown ctx
    assert ro.recv_ack(2, b"b") == {1, 2}
    assert ro.last_pending_request_ctx() == b"c"
    assert [(c, s.index) for c, s in ro.advance(b"b")] == [(b"a", 5), (b"b", 6)]
    assert ro.advance(b"b") == [] and ro.last_pending_request_ctx() == b"c"


def test_arena_full_and_split_and_invalid():
    """The bounds the reference does not have: FULL at max_pending, SPLIT for a group whose requests are not contiguous,
    INVALID for an unallocated group or a slot >= 8."""
    ar = R.ArenaReads(128, 2)
    cols = B.new_columns(128, 4)
    ar.alloc(0, 3)
    for g in range(3):
        cols.meta[g] = B.make_meta(0b111, self_slot=0)
        cols.committed[g] = cols.term_start[g] = cols.last_index[g] = 9
    r = np.zeros(8, dtype=B.READ_REQ_DTYPE)
    r["group"] = [0, 0, 0, 1, 0, 2, 3, 2]
    r["ctx"] = [1, 2, 3, 1, 4, 1, 1, 2]
    r["from_slot"] = [1, 1, 1, 1, 1, 9, 1, 2]
    st, idx = ar.read_index(r, cols, 4)
    assert st.tolist() == [R.QUEUED, R.QUEUED, R.FULL, R.QUEUED, R.SPLIT, R.INVALID, R.INVALID, R.QUEUED]
    assert idx.tolist() == [9, 9, 0, 9, 0, 0, 0, 9]
    assert ar.last_ctx(0, 4).tolist() == [2, 1, 2, R.U64_MAX]


def _random_conf(rng):
    incoming = 1 | int(rng.integers(0, 256)) & 0b11111110 if rng.random() < 0.8 else 1
    outgoing = (1 | int(rng.integers(0, 256))) if rng.random() < 0.25 else 0
    learners = int(rng.integers(0, 256)) & ~(incoming | outgoing) & 0xFF if rng.random() < 0.3 else 0
    return incoming, outgoing, learners


def test_arena_form_matches_literal_form_on_random_traffic():
    """48 groups (joint configurations, learners, non-leaders, singletons) over 60 ticks of requests (local,
    forwarded, lease, duplicates), heartbeat responses acking random contexts (pending, released, unknown; absent
    slots, learners), configuration changes with the post_conf_change tail, and resets.  max_pending is never reached."""
    rng = np.random.default_rng(0x5EAD)
    G = 48
    ar = R.ArenaReads(128, 64)
    ar.alloc(0, G)
    cols = B.new_columns(128, G)
    cols.term_start[:] = R.U64_MAX          # not a leader until a tick says otherwise
    lit = [R.LiteralLeader() for _ in range(G)]
    confs = []
    for g in range(G):
        c = _random_conf(rng)
        confs.append(c)
        cols.meta[g] = B.make_meta(*c, self_slot=0)
        lit[g].set_conf(*c, self_slot=0)
    n_released = n_queued = 0
    for tick in range(60):
        for g in range(G):
            if rng.random() < 0.3:
                li = int(rng.integers(5, 50))
                ts = R.U64_MAX if rng.random() < 0.1 else int(rng.integers(1, li + 1))
                cm = int(rng.integers(0, li + 1))
                cols.committed[g], cols.term_start[g], cols.last_index[g] = cm, ts, li
                lit[g].set_log(cm, ts, li)
        # requests: a contiguous run per chosen group, groups in random order
        reqs = []
        for g in rng.permutation(G)[: G // 2]:
            present = [s for s in range(8) if ((confs[g][0] | confs[g][1] | confs[g][2]) >> s) & 1 and s != 0]
            for _ in range(int(rng.integers(1, 4))):
                local = not present or rng.random() < 0.4
                reqs.append((g, 0 if local else int(rng.choice(present)),
                             (B.READ_LOCAL if local else 0) | (B.READ_LEASE if rng.random() < 0.1 else 0),
                             int(rng.integers(0, 8))))
        r = np.array(reqs, dtype=[("group", "<u4"), ("from_slot", "u1"), ("flags", "u1"), ("ctx", "<u8")])
        rq = np.zeros(len(r), dtype=B.READ_REQ_DTYPE)
        for f in ("group", "from_slot", "flags", "ctx"):
            rq[f] = r[f]
        st, idx = ar.read_index(rq, cols, G)
        for i, (g, s, f, c) in enumerate(reqs):
            want = lit[g].step_read_index(c, None if f & B.READ_LOCAL else s, bool(f & B.READ_LEASE))
            assert (int(st[i]), int(idx[i])) == want, (tick, i, reqs[i])
        n_queued += int(np.count_nonzero(st == R.QUEUED))
        # one batch of heartbeat responses
        recs, want = [], {}
        for g in range(G):
            pend = lit[g].pending()
            for s in range(8):
                if rng.random() < 0.5:
                    c = int(rng.choice(pend)) if pend and rng.random() < 0.8 else int(rng.integers(0, 8))
                    recs.append((g, s, B.REC_HEARTBEAT | B.REC_READ_CTX, 0, c, 0))
                    want.setdefault(g, []).extend(lit[g].heartbeat_response(s, c))
        hb = np.array(recs, dtype=B.APPEND_RESP_DTYPE)
        ar.ack(hb, cols)
        got = ar.release(cols, 0, G)
        assert _by_group(got) == {g: v for g, v in want.items() if v}, tick
        n_released += len(got)
        # configuration changes (then post_conf_change) and resets
        for g in rng.choice(G, 3, replace=False):
            g = int(g)
            if rng.random() < 0.5:
                old = confs[g]
                confs[g] = _random_conf(rng)
                was, now = old[0] | old[1] | old[2], confs[g][0] | confs[g][1] | confs[g][2]
                cols.meta[g] = B.make_meta(*confs[g], self_slot=0)
                ar.clear_slots(g, was & ~now)
                lit[g].set_conf(*confs[g], self_slot=0)
                assert R.states_to_list(ar.conf_changed(cols, g)) == lit[g].post_conf_change(), (tick, g)
            else:
                ar.reset(g)
                lit[g].reset()
        for g in range(G):
            assert [int(c) for c in ar.queue(g)[0]] == lit[g].pending(), (tick, g)
        assert ar.last_ctx(0, G).tolist() == [(lit[g].pending() or [R.U64_MAX])[-1] for g in range(G)]
    assert n_released > 200 and n_queued > 200


def _by_group(states):
    out = {}
    for r in states:
        out.setdefault(int(r["group"]), []).append((None if r["flags"] & B.READ_LOCAL else int(r["to_slot"]),
                                                    int(r["index"]), int(r["ctx"])))
    return out
