// k_control.cuh -- send_list_kernel, tally_kernel and the single-group control-plane kernels.
// Part of kernels.cuh (included there, inside namespace raftgpu; not a standalone header).

// ---------------------------------------------------------------------------
// send_list_kernel: bcast_append (raft.rs:857-865) behind Raft::maybe_commit (raft.rs:1745-1748) as a
// stream compaction.  One lane per group, a warp per 32 groups = one word of the advanced bitmap;
// a selected group contributes one entry per present peer other than itself that is not paused
// (progress.rs:210-216).  Lanes count their entries, a warp scan turns the counts into offsets, ONE
// global atomic per warp reserves the range, each lane writes its 16-byte entries.
// Algorithmic bytes: 4 per 32 groups (bitmap) + per advanced group 4 (meta) + K x 17 (pflags,
// next_idx, pending_request_snapshot of its peers) read, 16 written per entry.
__global__ void __launch_bounds__(256)
send_list_kernel(Columns c, uint32_t first, uint32_t n, const uint32_t *__restrict__ adv_bitmap,
                 raftgpu_send_entry *__restrict__ out, unsigned long long capacity, unsigned long long *__restrict__ count,
                 bool has_wide) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t base = first & ~31u;
    const uint32_t n_tiles = static_cast<uint32_t>((static_cast<uint64_t>(first - base) + n + 31) >> 5);
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t tile = warp; tile < n_tiles; tile += n_warps) {
        const uint32_t g = base + tile * 32u + lane;
        const uint32_t word = adv_bitmap ? adv_bitmap[g >> 5] : 0xffffffffu;
        const bool in_range = g >= first && g < first + n;
        // the high half of a wide group (odd slot, RAFTGPU_META_WIDE_HI) follows the low half's bit: its entries name
        // (g, slot) = the wide group's peer 8 + slot
        const uint32_t bit = (has_wide && in_range && (lane & 1u) && (c.meta[g] & RAFTGPU_META_WIDE_HI)) ? lane - 1 : lane;
        const bool sel = in_range && ((word >> bit) & 1u);
        uint32_t send = 0;
        uint64_t nx[kSlots], prs[kSlots];  // loaded together with the flag bytes: one round trip, not one per entry
        if (sel) {
            const uint32_t meta = c.meta[g];
            uint32_t peers = RAFTGPU_META_IN(meta) | RAFTGPU_META_OUT(meta) | RAFTGPU_META_LEARN(meta);
            if (meta & RAFTGPU_META_HAS_SELF) peers &= ~(1u << RAFTGPU_META_SELF(meta));  // raft.rs:863 id != self_id
            uint32_t f[kSlots];
#pragma unroll
            for (int s = 0; s < kSlots; s++) {
                f[s] = RAFTGPU_STATE_SNAPSHOT;
                nx[s] = 0;
                prs[s] = 0;
                if ((peers >> s) & 1u) {
                    const size_t cell = static_cast<size_t>(s) * c.cap + g;
                    f[s] = c.pflags[cell];
                    nx[s] = c.next_idx[cell];
                    prs[s] = c.pending_req_snapshot[cell];
                }
            }
#pragma unroll
            for (int s = 0; s < kSlots; s++) {
                const uint32_t state = f[s] & RAFTGPU_PF_STATE_MASK;
                const bool paused = state == RAFTGPU_STATE_PROBE ? (f[s] & RAFTGPU_PF_PAUSED) != 0
                                                                 : (state == RAFTGPU_STATE_REPLICATE ? (f[s] & RAFTGPU_PF_INS_FULL) != 0 : true);
                if (((peers >> s) & 1u) && !paused) send |= 1u << s;
            }
        }
        const uint32_t cnt = __popc(send);
        uint32_t incl = cnt;  // inclusive warp scan
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= static_cast<uint32_t>(d)) incl += v;
        }
        const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
        if (total == 0) continue;
        unsigned long long pos = 0;
        if (lane == 31) pos = atomicAdd(count, static_cast<unsigned long long>(total));
        pos = __shfl_sync(0xffffffffu, pos, 31) + (incl - cnt);
#pragma unroll
        for (int s = 0; s < kSlots; s++) {
            if (!((send >> s) & 1u)) continue;
            if (pos < capacity) {
                const uint64_t w0 = static_cast<uint64_t>(g) | (static_cast<uint64_t>(s) << 32) |
                                    (static_cast<uint64_t>(prs[s] != RAFTGPU_INVALID_INDEX ? RAFTGPU_SEND_SNAPSHOT : 0u) << 40);
                reinterpret_cast<ulonglong2 *>(out)[pos] = make_ulonglong2(w0, nx[s]);
            }
            pos++;
        }
    }
}

// ---------------------------------------------------------------------------
// heartbeat_commit_kernel: bcast_heartbeat (raft.rs:875-889) -> send_heartbeat's
// commit = min(pr.matched, raft_log.committed) (raft.rs:838-840) for every peer but the group's own.
// One thread per group, coalesced rows; algorithmic bytes per group: 4 (meta) + 8 (committed) +
// 8K (matched) read, 8 x 8 written.
__global__ void __launch_bounds__(256)
heartbeat_commit_kernel(Columns c, uint32_t first, uint32_t n, uint64_t *__restrict__ out) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint32_t g = first + i;
        const uint32_t meta = c.meta[g];
        uint32_t peers = RAFTGPU_META_IN(meta) | RAFTGPU_META_OUT(meta) | RAFTGPU_META_LEARN(meta);
        if (meta & RAFTGPU_META_HAS_SELF) peers &= ~(1u << RAFTGPU_META_SELF(meta));  // raft.rs:887 id != self_id
        const uint64_t committed = c.committed[g];
        uint64_t v[kSlots];
#pragma unroll
        for (int s = 0; s < kSlots; s++) v[s] = ((peers >> s) & 1u) ? c.matched[static_cast<size_t>(s) * c.cap + g] : 0ull;
#pragma unroll
        for (int s = 0; s < kSlots; s++)
            out[static_cast<size_t>(s) * n + i] = ((peers >> s) & 1u) ? umin64(v[s], committed) : RAFTGPU_NO_HEARTBEAT;
    }
}

// ---------------------------------------------------------------------------
// heartbeat_resp_kernel: the tracker part of Raft::handle_heartbeat_response (raft.rs:1777-1804), one
// thread per RAFTGPU_REC_HEARTBEAT record (commit = m.commit): update_committed, recent_active = true,
// resume(); a Replicate peer whose inflights window is full frees its first entry (:1796-1798 -- the
// window is then no longer full: INS_FULL clears); RAFTGPU_RES_SEND where the reference calls send_append:
// pr.matched < last_index || pending_request_snapshot != INVALID_INDEX (:1800-1803).  A scatter pass by
// nature (the records name the cells); one record per cell, verified through `touched` like the other
// zero-copy paths (a second record for a cell is not applied and bumps *dup_count).
__global__ void __launch_bounds__(256)
heartbeat_resp_kernel(Columns c, const raftgpu_append_resp *__restrict__ recs, uint64_t n, uint8_t *__restrict__ results,
                      uint32_t *__restrict__ touched, uint32_t *__restrict__ dup_count) {
    const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
    for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint64_t *p = reinterpret_cast<const uint64_t *>(recs + i);
        const uint64_t w0 = p[0], commit = p[2];
        const uint32_t g = static_cast<uint32_t>(w0), slot = static_cast<uint32_t>(w0 >> 32) & 0xffu;
        const uint32_t rflags = static_cast<uint32_t>(w0 >> 40) & 0xffu;
        uint32_t res = 0;
        if (rflags & RAFTGPU_REC_HEARTBEAT) {
            const bool in_range = g < c.cap && slot < kSlots;
            const uint32_t meta = in_range ? c.meta[g] : 0u;
            const uint32_t present = RAFTGPU_META_IN(meta) | RAFTGPU_META_OUT(meta) | RAFTGPU_META_LEARN(meta);
            if (!in_range || !((present >> slot) & 1u)) {
                res = RAFTGPU_RES_NO_PROGRESS;  // raft.rs:1779-1789
            } else {
                const uint32_t bit = 1u << (8 * (g & 3u) + slot);
                if (touched && (atomicOr(&touched[g >> 2], bit) & bit)) {
                    if (dup_count) atomicAdd(dup_count, 1u);
                } else {
                    const size_t cell = static_cast<size_t>(slot) * c.cap + g;
                    const uint32_t f0 = c.pflags[cell];
                    uint32_t f = (f0 | RAFTGPU_PF_RECENT_ACTIVE) & ~RAFTGPU_PF_PAUSED;          // :1792-1793
                    if ((f0 & RAFTGPU_PF_STATE_MASK) == RAFTGPU_STATE_REPLICATE) {  // :1796-1798
                        if (!c.ins_cap)
                            f &= ~RAFTGPU_PF_INS_FULL;  // host-side windows: a full one that loses an entry is not full
                        else if (f0 & RAFTGPU_PF_INS_FULL)
                            ins_free_first_one(c, cell, f);
                    }
                    if (commit > c.peer_committed[cell]) c.peer_committed[cell] = commit;      // :1791
                    if (f != f0) c.pflags[cell] = static_cast<uint8_t>(f);
                    res = RAFTGPU_RES_OK;
                    if (c.matched[cell] < c.last_index[g] || c.pending_req_snapshot[cell] != RAFTGPU_INVALID_INDEX)
                        res |= RAFTGPU_RES_SEND;                                                // :1800-1803
                }
            }
        }
        if (results) results[i] = static_cast<uint8_t>(res);
    }
}

// ---------------------------------------------------------------------------
// update_state_kernel: Progress::update_state(last) (progress.rs:231-243) for a list of sends, i.e. what
// send_append does once it has built a MsgAppend for the entry (raft.rs:753-760): Replicate ->
// optimistic_update(last): next_idx = last + 1 (the ins.add(last) that goes with it is the host's Inflights);
// Probe -> pause().  Without it a probing peer is never paused and every later send list names it again.
// entries: raftgpu_send_entry with next_idx = `last` (the index of the last entry sent).  results[i]: 1 done,
// 0xff where the reference panics (Snapshot state), RAFTGPU_RES_NO_PROGRESS for an unknown peer.
__global__ void __launch_bounds__(256)
update_state_kernel(Columns c, const raftgpu_send_entry *__restrict__ e, uint64_t n, uint8_t *__restrict__ results) {
    const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
    for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint32_t g = e[i].group, slot = e[i].peer_slot;
        const uint64_t last = e[i].next_idx;
        uint32_t res;
        const bool in_range = g < c.cap && slot < kSlots;
        const uint32_t meta = in_range ? c.meta[g] : 0u;
        const uint32_t present = RAFTGPU_META_IN(meta) | RAFTGPU_META_OUT(meta) | RAFTGPU_META_LEARN(meta);
        if (!in_range || !((present >> slot) & 1u)) {
            res = RAFTGPU_RES_NO_PROGRESS;
        } else {
            const size_t cell = static_cast<size_t>(slot) * c.cap + g;
            const uint32_t f0 = c.pflags[cell];
            const uint32_t state = f0 & RAFTGPU_PF_STATE_MASK;
            res = 1;
            if (state == RAFTGPU_STATE_REPLICATE) {
                uint32_t f = f0;
                if (c.ins_cap && !ins_add(c, cell, last, f)) {
                    res = 0xffu;                                                  // ins.add on a full window panics
                } else {
                    c.next_idx[cell] = last + 1;                                  // :233-236 optimistic_update
                    if (f != f0) c.pflags[cell] = static_cast<uint8_t>(f);
                }
            } else if (state == RAFTGPU_STATE_PROBE)
                c.pflags[cell] = static_cast<uint8_t>(f0 | RAFTGPU_PF_PAUSED);    // :237 pause()
            else
                res = 0xffu;                                                      // :238-241 panic!
        }
        if (results) results[i] = static_cast<uint8_t>(res);
    }
}

// ---------------------------------------------------------------------------
// tally_kernel: ProgressTracker::tally_votes (tracker.rs:313-340) per group:
// granted / rejected over voters, JointConfig::vote_result (joint.rs:56-67) over
// MajorityConfig::vote_result (majority.rs:130-154).
__device__ __forceinline__ uint32_t majority_vote(uint32_t mask, uint32_t yes, uint32_t no) {
    if (mask == 0) return RAFTGPU_VOTE_WON;  // majority.rs:131-136
    const uint32_t n = __popc(mask), q = (n >> 1) + 1;
    const uint32_t y = __popc(yes & mask), missing = n - y - __popc(no & mask);
    if (y >= q) return RAFTGPU_VOTE_WON;
    if (y + missing >= q) return RAFTGPU_VOTE_PENDING;
    return RAFTGPU_VOTE_LOST;
}

__global__ void __launch_bounds__(256)
tally_kernel(Columns c, uint32_t first, uint32_t n, uint32_t *__restrict__ out,
             unsigned long long *__restrict__ counters) {
    const uint64_t t = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    const bool active = t < n;
    if (active) {
        const uint32_t g = first + static_cast<uint32_t>(t);
        uint32_t meta = c.meta[g];
        uint32_t in = RAFTGPU_META_IN(meta), outm = RAFTGPU_META_OUT(meta);
        uint32_t yes = 0, no = 0;
#pragma unroll
        for (int s = 0; s < kSlots; s++) {
            const uint32_t v = c.votes[static_cast<size_t>(s) * c.cap + g];
            yes |= (v == 2u) << s;
            no |= (v == 1u) << s;
        }
        if (meta & (RAFTGPU_META_WIDE_LO | RAFTGPU_META_WIDE_HI)) {  // a wide group: both halves get the result over 16 peers
            const uint32_t other = (meta & RAFTGPU_META_WIDE_LO) ? g + 1 : g - 1, sh_me = (meta & RAFTGPU_META_WIDE_LO) ? 0u : 8u;
            const uint32_t mo = c.meta[other];
            uint32_t yo = 0, no2 = 0;
            for (int s = 0; s < kSlots; s++) {
                const uint32_t v = c.votes[static_cast<size_t>(s) * c.cap + other];
                yo |= (v == 2u) << s;
                no2 |= (v == 1u) << s;
            }
            in = (in << sh_me) | (RAFTGPU_META_IN(mo) << (8u - sh_me));
            outm = (outm << sh_me) | (RAFTGPU_META_OUT(mo) << (8u - sh_me));
            yes = (yes << sh_me) | (yo << (8u - sh_me));
            no = (no << sh_me) | (no2 << (8u - sh_me));
        }
        const uint32_t i = majority_vote(in, yes, no), o = majority_vote(outm, yes, no);
        uint32_t r;
        if (i == RAFTGPU_VOTE_WON && o == RAFTGPU_VOTE_WON)
            r = RAFTGPU_VOTE_WON;
        else if (i == RAFTGPU_VOTE_LOST || o == RAFTGPU_VOTE_LOST)
            r = RAFTGPU_VOTE_LOST;
        else
            r = RAFTGPU_VOTE_PENDING;
        const uint32_t voters = in | outm;  // tracker.rs:320-322
        out[g] = r | (__popc(yes & voters) << 8) | (__popc(no & voters) << 16);
    }
    const uint32_t local[1] = {active ? 1u : 0u};
    const int which[1] = {kCntVotes};
    block_flush_counts<1>(local, which, counters, nullptr);
}

// ---------------------------------------------------------------------------
// Control-plane helpers (single thread; launched <<<1,1>>>).

// ProgressTracker::apply_conf (tracker.rs:380-397)
__global__ void conf_kernel(Columns c, uint32_t g, uint32_t new_meta, uint32_t added,
                            uint32_t removed, uint64_t next_idx) {
    for (int s = 0; s < kSlots; s++) {
        const size_t cell = static_cast<size_t>(s) * c.cap + g;
        if (((added | removed) >> s) & 1u) {
            const bool add = (added >> s) & 1u;
            c.matched[cell] = 0;
            c.next_idx[cell] = add ? next_idx : 0;  // Progress::new(next_idx, ..), progress.rs:60-73
            c.peer_committed[cell] = 0;
            c.pending_snapshot[cell] = 0;
            c.pending_req_snapshot[cell] = 0;
            c.commit_group_id[cell] = 0;
            c.pflags[cell] = add ? RAFTGPU_PF_RECENT_ACTIVE : 0;  // tracker.rs:385-389
            c.votes[cell] = 0;
            ins_reset(c, cell);  // Inflights::new(max_inflight), progress.rs:70
        }
    }
    rd_clear_slots(c, g, new_meta, removed);  // acks are by peer id: a later occupant of the slot must not inherit them
    c.meta[g] = new_meta;
}

// Raft::reset (raft.rs:942-971) for the tracker + log bookkeeping of one group.
__global__ void reset_kernel(Columns c, uint32_t g, uint64_t term_start, uint64_t last_index,
                             uint64_t committed, uint64_t persisted) {
    const uint32_t meta = c.meta[g];
    const uint32_t present = RAFTGPU_META_IN(meta) | RAFTGPU_META_OUT(meta) | RAFTGPU_META_LEARN(meta);
    for (int s = 0; s < kSlots; s++) {
        if (!((present >> s) & 1u)) continue;
        const size_t cell = static_cast<size_t>(s) * c.cap + g;
        // Progress::reset(last_index + 1), progress.rs:82-92
        c.matched[cell] = 0;
        c.next_idx[cell] = last_index + 1;
        c.pending_snapshot[cell] = 0;
        c.pending_req_snapshot[cell] = RAFTGPU_INVALID_INDEX;
        c.pflags[cell] = RAFTGPU_STATE_PROBE;
        ins_reset(c, cell);  // progress.rs:91 ins.reset()
        c.votes[cell] = 0;  // prs.reset_votes(), raft.rs:953
        if ((meta & RAFTGPU_META_HAS_SELF) && RAFTGPU_META_SELF(meta) == static_cast<uint32_t>(s)) {
            c.matched[cell] = persisted;         // raft.rs:967
            c.peer_committed[cell] = committed;  // raft.rs:968
        }
    }
    rd_empty(c, g);  // raft.rs:957 read_only = ReadOnly::new(..)
    c.committed[g] = committed;
    c.term_start[g] = term_start;
    c.last_index[g] = last_index;
}

// Raft::become_leader's tracker side (raft.rs:1176-1192): self.become_replicate(),
// then the empty entry of the new term is appended at last_index + 1.
__global__ void become_leader_kernel(Columns c, uint32_t g) {
    const uint32_t meta = c.meta[g];
    if (meta & RAFTGPU_META_HAS_SELF) {
        const size_t cell = static_cast<size_t>(RAFTGPU_META_SELF(meta)) * c.cap + g;
        c.pflags[cell] = static_cast<uint8_t>(
            (c.pflags[cell] & ~(RAFTGPU_PF_PAUSED | RAFTGPU_PF_INS_FULL | RAFTGPU_PF_STATE_MASK)) |
            RAFTGPU_STATE_REPLICATE);
        c.pending_snapshot[cell] = 0;
        ins_reset(c, cell);
        c.next_idx[cell] = c.matched[cell] + 1;  // progress.rs:110-114
    }
    const uint64_t li = c.last_index[g] + 1;  // raft.rs:1192 append_entry(&mut [Entry::default()])
    c.last_index[g] = li;
    c.term_start[g] = li;
}

__global__ void progress_get_kernel(Columns c, uint32_t g, uint32_t s, raftgpu_progress *out) {
    const size_t cell = static_cast<size_t>(s) * c.cap + g;
    const uint32_t f = c.pflags[cell];
    const uint32_t meta = c.meta[g];
    raftgpu_progress p{};
    p.matched = c.matched[cell];
    p.next_idx = c.next_idx[cell];
    p.pending_snapshot = c.pending_snapshot[cell];
    p.pending_request_snapshot = c.pending_req_snapshot[cell];
    p.commit_group_id = c.commit_group_id[cell];
    p.committed_index = c.peer_committed[cell];
    p.state = f & RAFTGPU_PF_STATE_MASK;
    p.paused = (f & RAFTGPU_PF_PAUSED) != 0;
    p.recent_active = (f & RAFTGPU_PF_RECENT_ACTIVE) != 0;
    p.ins_full = (f & RAFTGPU_PF_INS_FULL) != 0;
    p.present = ((RAFTGPU_META_IN(meta) | RAFTGPU_META_OUT(meta) | RAFTGPU_META_LEARN(meta)) >> s) & 1u;
    *out = p;
}

__global__ void progress_set_kernel(Columns c, uint32_t g, uint32_t s, raftgpu_progress p) {
    const size_t cell = static_cast<size_t>(s) * c.cap + g;
    c.matched[cell] = p.matched;
    c.next_idx[cell] = p.next_idx;
    c.pending_snapshot[cell] = p.pending_snapshot;
    c.pending_req_snapshot[cell] = p.pending_request_snapshot;
    c.commit_group_id[cell] = p.commit_group_id;
    c.peer_committed[cell] = p.committed_index;
    const bool full = c.ins_cap ? (c.ins_meta[cell] >> 16) == c.ins_cap : p.ins_full != 0;  // device windows: derived
    c.pflags[cell] = static_cast<uint8_t>((p.state & RAFTGPU_PF_STATE_MASK) |
                                          (p.paused ? RAFTGPU_PF_PAUSED : 0) |
                                          (p.recent_active ? RAFTGPU_PF_RECENT_ACTIVE : 0) |
                                          (full ? RAFTGPU_PF_INS_FULL : 0));
}

__device__ __forceinline__ uint32_t majority_vote(uint32_t mask, uint32_t yes, uint32_t no);

// Every method of Progress (src/tracker/progress.rs:75-243) on one cell, literally, for the
// host mirror's ProgressRef: op codes are RAFTGPU_POP_*.  *out gets the bool / status result.
__global__ void progress_op_kernel(Columns c, uint32_t g, uint32_t s, int op, uint64_t a0, uint64_t a1,
                                   uint64_t a2, int32_t *out) {
    const size_t cell = static_cast<size_t>(s) * c.cap + g;
    uint64_t matched = c.matched[cell], next = c.next_idx[cell];
    uint32_t f = c.pflags[cell];
    const uint32_t state = f & RAFTGPU_PF_STATE_MASK;
    int32_t ret = 0;
    auto reset_st = [&](uint32_t st) {  // progress.rs:75-80
        f = (f & ~(RAFTGPU_PF_PAUSED | RAFTGPU_PF_INS_FULL | RAFTGPU_PF_STATE_MASK)) | st;
        c.pending_snapshot[cell] = 0;
        ins_reset(c, cell);
    };
    switch (op) {
    case RAFTGPU_POP_MAYBE_UPDATE:  // progress.rs:138-150
        if (matched < a0) {
            matched = a0;
            f &= ~RAFTGPU_PF_PAUSED;
            ret = 1;
        }
        if (next < a0 + 1) next = a0 + 1;
        break;
    case RAFTGPU_POP_MAYBE_DECR_TO: {  // progress.rs:168-206 (a0 rejected, a1 match_hint, a2 request_snapshot)
        if (state == RAFTGPU_STATE_REPLICATE) {
            if (a0 < matched || (a0 == matched && a2 == RAFTGPU_INVALID_INDEX)) break;
            if (a2 == RAFTGPU_INVALID_INDEX)
                next = matched + 1;
            else
                c.pending_req_snapshot[cell] = a2;
            ret = 1;
            break;
        }
        if ((next == 0 || next - 1 != a0) && a2 == RAFTGPU_INVALID_INDEX) break;
        if (a2 == RAFTGPU_INVALID_INDEX) {
            next = umin64(a0, a1 + 1);
            if (next < 1) next = 1;
        } else if (c.pending_req_snapshot[cell] == RAFTGPU_INVALID_INDEX) {
            c.pending_req_snapshot[cell] = a2;
        }
        f &= ~RAFTGPU_PF_PAUSED;
        ret = 1;
        break;
    }
    case RAFTGPU_POP_UPDATE_COMMITTED:  // progress.rs:153-157
        if (a0 > c.peer_committed[cell]) c.peer_committed[cell] = a0;
        break;
    case RAFTGPU_POP_OPTIMISTIC_UPDATE:  // progress.rs:160-163
        next = a0 + 1;
        break;
    case RAFTGPU_POP_BECOME_PROBE:  // progress.rs:95-107
        if (state == RAFTGPU_STATE_SNAPSHOT) {
            const uint64_t pending = c.pending_snapshot[cell];
            reset_st(RAFTGPU_STATE_PROBE);
            next = umax64(matched + 1, pending + 1);
        } else {
            reset_st(RAFTGPU_STATE_PROBE);
            next = matched + 1;
        }
        break;
    case RAFTGPU_POP_BECOME_REPLICATE:  // progress.rs:110-114
        reset_st(RAFTGPU_STATE_REPLICATE);
        next = matched + 1;
        break;
    case RAFTGPU_POP_BECOME_SNAPSHOT:  // progress.rs:117-121
        reset_st(RAFTGPU_STATE_SNAPSHOT);
        c.pending_snapshot[cell] = a0;
        break;
    case RAFTGPU_POP_SNAPSHOT_FAILURE:  // progress.rs:124-127
        c.pending_snapshot[cell] = 0;
        break;
    case RAFTGPU_POP_MAYBE_SNAPSHOT_ABORT:  // progress.rs:131-134
        ret = state == RAFTGPU_STATE_SNAPSHOT && matched >= c.pending_snapshot[cell];
        break;
    case RAFTGPU_POP_IS_PAUSED:  // progress.rs:210-216
        ret = state == RAFTGPU_STATE_PROBE ? (f & RAFTGPU_PF_PAUSED) != 0
              : state == RAFTGPU_STATE_REPLICATE ? (f & RAFTGPU_PF_INS_FULL) != 0 : 1;
        break;
    case RAFTGPU_POP_RESUME:  // progress.rs:219-222
        f &= ~RAFTGPU_PF_PAUSED;
        break;
    case RAFTGPU_POP_PAUSE:  // progress.rs:225-228
        f |= RAFTGPU_PF_PAUSED;
        break;
    case RAFTGPU_POP_UPDATE_STATE:  // progress.rs:231-243 (a0 = last); -1 where the reference panics
        if (state == RAFTGPU_STATE_REPLICATE) {
            if (c.ins_cap && !ins_add(c, cell, a0, f))
                ret = -1;       // ins.add on a full window panics (inflights.rs:66-68)
            else
                next = a0 + 1;  // optimistic_update (without device windows ins.add(last) is the host's)
        } else if (state == RAFTGPU_STATE_PROBE)
            f |= RAFTGPU_PF_PAUSED;
        else
            ret = -1;
        break;
    case RAFTGPU_POP_RESET:  // progress.rs:82-92 (a0 = next_idx)
        matched = 0;
        next = a0;
        f = RAFTGPU_STATE_PROBE;
        c.pending_snapshot[cell] = 0;
        c.pending_req_snapshot[cell] = RAFTGPU_INVALID_INDEX;
        ins_reset(c, cell);
        break;
    // Inflights (src/tracker/inflights.rs) on the cell's window; -3 when the arena keeps no windows
    case RAFTGPU_POP_INS_ADD:  // :65-82 (a0 = inflight); -1 where the reference panics
        ret = !c.ins_cap ? -3 : (ins_add(c, cell, a0, f) ? 0 : -1);
        break;
    case RAFTGPU_POP_INS_FREE_TO:  // :85-110
        if (c.ins_cap) ins_free_to(c, cell, a0, f); else ret = -3;
        break;
    case RAFTGPU_POP_INS_FREE_FIRST_ONE:  // :113-116
        if (c.ins_cap) ins_free_first_one(c, cell, f); else ret = -3;
        break;
    case RAFTGPU_POP_INS_RESET:  // :119-123
        if (c.ins_cap) { ins_reset(c, cell); f &= ~RAFTGPU_PF_INS_FULL; } else ret = -3;
        break;
    case RAFTGPU_POP_INS_FULL:  // :54-56
        ret = !c.ins_cap ? -3 : ((c.ins_meta[cell] >> 16) == c.ins_cap);
        break;
    default:
        ret = -2;
    }
    c.matched[cell] = matched;
    c.next_idx[cell] = next;
    c.pflags[cell] = static_cast<uint8_t>(f);
    *out = ret;
}

// ProgressTracker::has_quorum (tracker.rs:367-372): vote_result(|id| set.get(id).map(|_| true)) == Won,
// and quorum_recently_active (tracker.rs:346-361), which also clears recent_active.
__global__ void quorum_kernel(Columns c, uint32_t g, int op, uint32_t arg, int32_t *out) {
    const uint32_t meta = c.meta[g];
    const bool wide = (meta & RAFTGPU_META_WIDE_LO) != 0;  // peers 8..15 live in group g + 1
    const uint32_t meta_hi = wide ? c.meta[g + 1] : 0u;
    const uint32_t in = RAFTGPU_META_IN(meta) | (RAFTGPU_META_IN(meta_hi) << 8);
    const uint32_t outm = RAFTGPU_META_OUT(meta) | (RAFTGPU_META_OUT(meta_hi) << 8);
    uint32_t active = arg;
    if (op == 1) {  // quorum_recently_active(perspective_of = slot arg)
        const uint32_t present = in | outm | RAFTGPU_META_LEARN(meta) | (RAFTGPU_META_LEARN(meta_hi) << 8);
        active = 0;
        for (int s = 0; s < (wide ? 2 * kSlots : kSlots); s++) {
            if (!((present >> s) & 1u)) continue;
            uint8_t *f = &c.pflags[static_cast<size_t>(s & 7) * c.cap + g + (s >> 3)];
            if (static_cast<uint32_t>(s) == arg) {
                *f |= RAFTGPU_PF_RECENT_ACTIVE;  // tracker.rs:350-352
                active |= 1u << s;
            } else if (*f & RAFTGPU_PF_RECENT_ACTIVE) {
                active |= 1u << s;  // tracker.rs:353-358
                *f &= ~RAFTGPU_PF_RECENT_ACTIVE;
            }
        }
    }
    // members of the set vote yes, everyone else is missing (None)
    const uint32_t i = majority_vote(in, active, 0), o = majority_vote(outm, active, 0);
    *out = (i == RAFTGPU_VOTE_WON && o == RAFTGPU_VOTE_WON) ? 1 : 0;
}

// The two halves of a wide group share the group's log / commit columns: make them agree (a LOCAL record or a
// single-half control-plane call may have touched one half only).
__global__ void wide_sync_kernel(Columns c, uint32_t g) {
    const uint64_t li = umax64(c.last_index[g], c.last_index[g + 1]);
    const uint64_t cm = umax64(c.committed[g], c.committed[g + 1]);
    c.last_index[g] = c.last_index[g + 1] = li;
    c.committed[g] = c.committed[g + 1] = cm;
    c.term_start[g + 1] = c.term_start[g];
    c.term[g + 1] = c.term[g];
}

__global__ void group_get_kernel(Columns c, uint32_t g, raftgpu_group_state *out) {
    raftgpu_group_state s{};
    s.meta = c.meta[g];
    s.committed = c.committed[g];
    s.term_start = c.term_start[g];
    s.last_index = c.last_index[g];
    *out = s;
}

// op 0: set_log_bounds; op 1: commit_to (status in *out: 0 ok, 1 out of range);
// op 2: meta bit set/clear (a = mask, b = enable); op 3: assign commit group (a = slot, b = id);
// op 4: reset votes; op 5: record vote (a = slot, b = vote+1), first vote wins (tracker.rs:308-310)
__global__ void group_op_kernel(Columns c, uint32_t g, int op, uint64_t a, uint64_t b,
                                uint32_t *out) {
    switch (op) {
    case 0:
        c.term_start[g] = a;
        c.last_index[g] = b;
        break;
    case 1:  // RaftLog::commit_to, raft_log.rs:286-300
        if (c.committed[g] >= a) {
            *out = 0;
        } else if (c.last_index[g] < a) {
            *out = 1;
        } else {
            c.committed[g] = a;
            *out = 0;
        }
        break;
    case 2:
        c.meta[g] = b ? (c.meta[g] | static_cast<uint32_t>(a)) : (c.meta[g] & ~static_cast<uint32_t>(a));
        break;
    case 3:
        c.commit_group_id[static_cast<size_t>(a) * c.cap + g] = b;
        break;
    case 4:
        for (int s = 0; s < kSlots; s++) c.votes[static_cast<size_t>(s) * c.cap + g] = 0;
        break;
    case 5: {
        uint8_t *v = &c.votes[static_cast<size_t>(a) * c.cap + g];
        if (*v == 0) *v = static_cast<uint8_t>(b);  // entry(id).or_insert(vote)
        break;
    }
    case 6:  // RaftLog::maybe_commit(max_index = a, term = the leader's), raft_log.rs:487-499, range form
        if (a > c.committed[g] && a >= c.term_start[g] && a <= c.last_index[g]) {
            c.committed[g] = a;
            *out = 1;
        } else {
            *out = 0;
        }
        break;
    }
}
