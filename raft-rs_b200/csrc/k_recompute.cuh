// k_recompute.cuh -- the recompute pass: Raft::maybe_commit per group.
// Part of kernels.cuh (included there, inside namespace raftgpu; not a standalone header).

// ---------------------------------------------------------------------------
// The recompute pass: one Raft::maybe_commit (raft.rs:893-904) per group.
//   mci  = ProgressTracker::maximal_committed_index      tracker.rs:294-298
//        = min(incoming.committed_index, outgoing.committed_index)   joint.rs:47-51
//   if mci > committed && term(mci) == term              raft_log.rs:487-499
//        committed = mci; prs[self].update_committed      raft.rs:896-900
// term(mci) == term is the range test term_start <= mci <= last_index (DESIGN.md).
// Algorithmic bytes per group: 8K (matched) + 4 (meta) + 24 (committed,
// term_start, last_index) read, 8 written when advanced.
//
// Two specialisations.  kSimple5 = the host has verified
// from its mirror of the meta column that EVERY group in the range is the plain
// 5-voter configuration in slots 0..4 (no joint half, no group commit): the
// kernel then carries no mask logic and no general selection network, which
// roughly halves its instructions and registers.  The general form handles any
// configuration; `hint` is a superset guess of the voter slots in the range (the
// host keeps the union of all voter masks) so that the matched loads of the
// hinted slots are issued together with meta / committed / term_start /
// last_index -- ONE round trip to HBM instead of two.  Voter slots outside the
// hint are fetched after meta arrives: correct for any hint, fast for a tight one.

// maximal_committed_index of one group from its matched values v[].
template <bool kSimple5>
__device__ __forceinline__ void eval_mci(const Columns &c, uint32_t g, uint32_t meta, uint64_t (&v)[kSlots],
                                         uint32_t hint, uint64_t &mci, bool &use_gc) {
    if constexpr (kSimple5) {
        mci = median5(v[0], v[1], v[2], v[3], v[4]);  // 5 voters: q = 3 = the median
        use_gc = false;
    } else {
        const uint32_t in = RAFTGPU_META_IN(meta), out = RAFTGPU_META_OUT(meta);
        const uint32_t voters = in | out;
        const uint32_t missing = voters & ~hint;
        if (missing) {  // hint was too small for this group: second trip for the rest
#pragma unroll
            for (int s = 0; s < kSlots; s++)
                if ((missing >> s) & 1u) v[s] = c.matched[static_cast<size_t>(s) * c.cap + g];
        }
        if ((meta & (0xffffu | RAFTGPU_META_GROUP_COMMIT | RAFTGPU_META_WIDE_LO | RAFTGPU_META_WIDE_HI)) == 0x1fu) {
            mci = median5(v[0], v[1], v[2], v[3], v[4]);
            use_gc = false;
        } else if (!(meta & RAFTGPU_META_GROUP_COMMIT)) {
            uint64_t i_idx, o_idx;
            quorum_index_joint(v, in, out, i_idx, o_idx);  // both halves from one comparison pass; empty => u64::MAX
            mci = umin64(i_idx, o_idx);                    // joint.rs:50
            use_gc = (in == 0) && (out == 0);              // majority.rs:71-75 vs :99-101
        } else {
            // (a COPY of v goes to the out-of-line group-commit routine: taking v's own address would put it in local
            //  memory for the common path too)
            uint64_t vv[kSlots], gid[kSlots];
            for (int s = 0; s < kSlots; s++) {
                vv[s] = v[s];
                gid[s] = ((voters >> s) & 1u) ? c.commit_group_id[static_cast<size_t>(s) * c.cap + g] : 0ull;
            }
            uint64_t i_idx, o_idx;
            bool i_gc, o_gc;
            majority_group_commit(vv, gid, in, &i_idx, &i_gc);
            majority_group_commit(vv, gid, out, &o_idx, &o_gc);
            mci = umin64(i_idx, o_idx);
            use_gc = i_gc && o_gc;
        }
    }
}

// RaftLog::maybe_commit (raft_log.rs:487-499, range form) + raft.rs:896-900.
__device__ __forceinline__ bool commit_group(const Columns &c, uint32_t g, uint32_t meta, uint64_t mci,
                                             bool use_gc, uint64_t committed, uint64_t term_start,
                                             uint64_t last_index, uint64_t *commit_out, uint64_t *mci_out,
                                             uint8_t *gc_out) {
    if (mci_out) mci_out[g] = mci;
    if (gc_out) gc_out[g] = use_gc ? 1 : 0;
    const bool advanced = mci > committed && mci >= term_start && mci <= last_index;
    if (advanced) {
        c.committed[g] = mci;  // commit_to: mci <= last_index, never the fatal! branch
        if (commit_out) commit_out[g] = mci;
        if (meta & RAFTGPU_META_HAS_SELF) {  // raft.rs:896-900
            const size_t cell = static_cast<size_t>(RAFTGPU_META_SELF(meta)) * c.cap + g;
            if (mci > c.peer_committed[cell]) c.peer_committed[cell] = mci;
        }
    }
    return advanced;
}

// Raft::maybe_commit for the wide group whose low half is g: maximal_committed_index over both halves' peers, the
// term / range test against the group's log bounds (a LOCAL record writes last_index on the half that holds the
// leader's own slot: the halves are merged here -- last_index only grows between control-plane resets), and the new
// commit index on BOTH halves (heartbeat commits and heartbeat responses read their own half's columns).
__device__ __noinline__ bool commit_wide_group(const Columns &c, uint32_t g, uint32_t meta_lo, uint64_t *commit_out,
                                               uint64_t *mci_out, uint8_t *gc_out) {
    uint64_t mci;
    bool use_gc;
    wide_mci(c, g, meta_lo, mci, use_gc);
    if (mci_out) mci_out[g] = mci;
    if (gc_out) gc_out[g] = use_gc ? 1 : 0;
    const uint64_t li = umax64(c.last_index[g], c.last_index[g + 1]);
    if (c.last_index[g] != li) c.last_index[g] = li;
    if (c.last_index[g + 1] != li) c.last_index[g + 1] = li;
    const uint64_t committed = c.committed[g];
    const bool advanced = mci > committed && mci >= c.term_start[g] && mci <= li;  // raft_log.rs:487-499
    if (advanced) {
        c.committed[g] = mci;
        c.committed[g + 1] = mci;
        if (commit_out) commit_out[g] = mci;
        const uint32_t meta_hi = c.meta[g + 1];  // raft.rs:896-900: the leader's own Progress, in whichever half it lives
        if (meta_lo & RAFTGPU_META_HAS_SELF) {
            const size_t cell = static_cast<size_t>(RAFTGPU_META_SELF(meta_lo)) * c.cap + g;
            if (mci > c.peer_committed[cell]) c.peer_committed[cell] = mci;
        } else if (meta_hi & RAFTGPU_META_HAS_SELF) {
            const size_t cell = static_cast<size_t>(RAFTGPU_META_SELF(meta_hi)) * c.cap + g + 1;
            if (mci > c.peer_committed[cell]) c.peer_committed[cell] = mci;
        }
    }
    return advanced;
}

// One word of the advanced bitmap per warp-tile.
__device__ __forceinline__ void publish_tile(uint32_t *adv_bitmap, uint64_t g64, uint32_t lane, bool active,
                                             bool advanced, uint32_t (&local)[2]) {
    const unsigned act = __ballot_sync(0xffffffffu, active);
    const unsigned adv = __ballot_sync(0xffffffffu, advanced);
    if (lane == 0 && act != 0 && adv_bitmap) {
        uint32_t *word = &adv_bitmap[g64 >> 5];
        if (act == 0xffffffffu) {
            *word = adv;
        } else {  // range starts / ends inside this word: leave the other bits alone
            atomicAnd(word, ~act);
            if (adv) atomicOr(word, adv);
        }
    }
    local[0] += active ? 1u : 0u;
    local[1] += advanced ? 1u : 0u;
}

// Persistent grid, each warp walks 32-group tiles with a grid stride.
template <bool kSimple5>
__global__ void __launch_bounds__(256, kSimple5 ? 6 : 4)
recompute_kernel(Columns c, uint32_t first, uint32_t n, uint32_t hint_arg,
                 uint32_t *__restrict__ adv_bitmap, uint64_t *__restrict__ commit_out,
                 uint64_t *__restrict__ mci_out, uint8_t *__restrict__ gc_out,
                 uint32_t *__restrict__ step_advanced, unsigned long long *__restrict__ counters) {
    const uint32_t hint = kSimple5 ? 0x1fu : hint_arg;
    const uint32_t base = first & ~31u;
    const uint32_t n_tiles = static_cast<uint32_t>((static_cast<uint64_t>(first - base) + n + 31) >> 5);
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t n_warps = (gridDim.x * blockDim.x) >> 5;
    const uint64_t end = static_cast<uint64_t>(first) + n;
    uint32_t local[2] = {0, 0};  // recomputes, advanced

    for (uint32_t tile = warp; tile < n_tiles; tile += n_warps) {
        const uint64_t g64 = static_cast<uint64_t>(base) + (static_cast<uint64_t>(tile) << 5) + lane;
        const bool active = g64 >= first && g64 < end;
        const uint32_t g = static_cast<uint32_t>(g64);
        bool advanced = false, wide_hi = false;
        if (active) {
            // one batch of independent loads
            const uint32_t meta = c.meta[g];
            uint64_t v[kSlots];
#pragma unroll
            for (int s = 0; s < kSlots; s++)
                v[s] = ((hint >> s) & 1u) ? c.matched[static_cast<size_t>(s) * c.cap + g] : 0ull;
            const uint64_t committed = c.committed[g];
            const uint64_t term_start = c.term_start[g];
            const uint64_t last_index = c.last_index[g];
            uint64_t mci;
            bool use_gc;
            if (!kSimple5 && (meta & (RAFTGPU_META_WIDE_LO | RAFTGPU_META_WIDE_HI))) {
                // a wide group is evaluated once, on its low half, over both halves' peers; the high half is not a
                // group of its own (its bit of the bitmap stays 0, it is not counted)
                if (meta & RAFTGPU_META_WIDE_LO) advanced = commit_wide_group(c, g, meta, commit_out, mci_out, gc_out);
                wide_hi = (meta & RAFTGPU_META_WIDE_HI) != 0;
            } else {
                eval_mci<kSimple5>(c, g, meta, v, hint, mci, use_gc);
                advanced = commit_group(c, g, meta, mci, use_gc, committed, term_start, last_index, commit_out,
                                        mci_out, gc_out);
            }
        }
        publish_tile(adv_bitmap, g64, lane, active, advanced, local);
        if (wide_hi) local[0]--;  // publish_tile counted the lane as a recompute
    }
    const int which[2] = {kCntRecomputes, kCntAdvanced};
    block_flush_counts<2>(local, which, counters, step_advanced);
}
