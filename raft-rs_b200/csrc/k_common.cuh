// k_common.cuh -- the arena columns, counters, the quorum selection (MajorityConfig / JointConfig::committed_index), block-level counter flush.
// Part of kernels.cuh (included there, inside namespace raftgpu; not a standalone header).

constexpr int kSlots = RAFTGPU_SLOTS;

// Device view of the arena: per-peer columns are [kSlots][cap], per-group [cap].
struct Columns {
    uint32_t cap;
    uint64_t *matched;
    uint64_t *next_idx;
    uint64_t *peer_committed;
    uint64_t *pending_snapshot;
    uint64_t *pending_req_snapshot;
    uint64_t *commit_group_id;
    uint8_t *pflags;
    uint8_t *votes;
    uint32_t *meta;
    uint64_t *committed;
    uint64_t *term_start;
    uint64_t *last_index;
    uint64_t *term;  // Raft::term, 0 = unknown (wire path only)
    // Inflights on the device (raftgpu_arena_enable_inflights; SURVEY 8(f) rank 2): ins_cap = window size
    // (Config::max_inflight_msgs), 0 = off (INS_FULL is then the host's to report); ins_meta [kSlots][cap] =
    // start | count << 16 (inflights.rs:21-23); ins_buf [kSlots][cap][ins_cap] the rings
    uint32_t ins_cap;
    uint32_t *ins_meta;
    uint64_t *ins_buf;
    // ReadOnly queues (raftgpu_arena_enable_read_index; k_read.cuh): rd_cap = max_pending, 0 = off; rd_meta [cap] =
    // head | count << 16 | kRdAlloc; rd_ctx / rd_index / rd_word [rd_cap][cap] by ring position; rd_first [cap] the
    // request pass's scratch (UINT32_MAX between passes)
    uint32_t rd_cap;
    uint32_t *rd_meta;
    uint64_t *rd_ctx;
    uint64_t *rd_index;
    uint32_t *rd_word;
    uint32_t *rd_first;
};

enum Counter : int {
    kCntRecomputes = 0,
    kCntAdvanced,
    kCntRecords,
    kCntUpdates,
    kCntRejects,
    kCntDecrements,
    kCntNoProgress,
    kCntVotes,
    kCntCount
};

// Fire-and-forget L2 prefetch: costs no destination register, so it deepens the memory pipeline
// beyond what registers x occupancy allow (the kernels here are long-scoreboard bound).
__device__ __forceinline__ void prefetch_l2(const void *p) {
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}

__device__ __forceinline__ uint64_t umin64(uint64_t a, uint64_t b) { return a < b ? a : b; }
__device__ __forceinline__ uint64_t umax64(uint64_t a, uint64_t b) { return a > b ? a : b; }

// ---------------------------------------------------------------------------
// Inflights (src/tracker/inflights.rs) of one cell, when the arena keeps the windows on the device.  The flag bit
// RAFTGPU_PF_INS_FULL mirrors ins.full() (what Progress::is_paused reads, progress.rs:213): every function
// takes the caller's copy of the flag byte and keeps the bit right.
__device__ __forceinline__ void ins_reset(const Columns &c, size_t cell) {  // :119-123
    if (c.ins_cap) c.ins_meta[cell] = 0;
}
// :85-110 free_to
__device__ __noinline__ void ins_free_to(const Columns &c, size_t cell, uint64_t to, uint32_t &flags) {
    const uint32_t m = c.ins_meta[cell];
    uint32_t start = m & 0xffffu, count = m >> 16;
    const uint64_t *ring = c.ins_buf + cell * c.ins_cap;
    if (count == 0 || to < ring[start]) return;  // out of the left side of the window
    uint32_t i = 0, idx = start;
    while (i < count) {
        if (to < ring[idx]) break;  // found the first large inflight
        idx += 1;
        if (idx >= c.ins_cap) idx -= c.ins_cap;
        i += 1;
    }
    c.ins_meta[cell] = idx | ((count - i) << 16);
    if (i) flags &= ~RAFTGPU_PF_INS_FULL;
}
// :113-116 free_first_one
__device__ __forceinline__ void ins_free_first_one(const Columns &c, size_t cell, uint32_t &flags) {
    const uint32_t m = c.ins_meta[cell];
    if ((m >> 16) == 0) return;
    ins_free_to(c, cell, c.ins_buf[cell * c.ins_cap + (m & 0xffffu)], flags);
}
// :65-82 add; false where the reference panics (the window is full)
__device__ __forceinline__ bool ins_add(const Columns &c, size_t cell, uint64_t inflight, uint32_t &flags) {
    const uint32_t m = c.ins_meta[cell];
    const uint32_t start = m & 0xffffu, count = m >> 16;
    if (count == c.ins_cap) return false;
    uint32_t next = start + count;
    if (next >= c.ins_cap) next -= c.ins_cap;
    c.ins_buf[cell * c.ins_cap + next] = inflight;
    c.ins_meta[cell] = start | ((count + 1) << 16);
    if (count + 1 == c.ins_cap) flags |= RAFTGPU_PF_INS_FULL;
    return true;
}

// ---------------------------------------------------------------------------
// ReadOnly queues (k_read.cuh): the layout constants and the two control-plane hooks, no-ops on arenas without queues.
constexpr uint32_t kRdAlloc = 0x80000000u;  // rd_meta: the group slot is allocated (a request for any other is INVALID)
constexpr uint32_t kRdAckMask = 0xffffu;    // rd_word: acks over peer slots 0..15
constexpr uint32_t kRdFromShift = 16;       // rd_word: from slot (0..15) in bits 16..23
__device__ __forceinline__ uint32_t rd_head(uint32_t m) { return m & 0xffu; }
__device__ __forceinline__ uint32_t rd_count(uint32_t m) { return (m >> 16) & 0xffu; }
// apply_conf removed peer slots `removed` of the half `g` whose new meta word is `meta`: their acks leave every pending
// request of the group (the queue lives on the low half of a wide group, where peer 8 + s is ack bit 8 + s)
__device__ __forceinline__ void rd_clear_slots(const Columns &c, uint32_t g, uint32_t meta, uint32_t removed) {
    if (!c.rd_cap || !removed) return;
    const bool hi = (meta & RAFTGPU_META_WIDE_HI) != 0;
    const uint32_t lo = hi ? g - 1 : g, clear = removed << (hi ? 8 : 0);
    for (uint32_t p = 0; p < c.rd_cap; p++) {
        uint32_t *w = &c.rd_word[static_cast<size_t>(p) * c.cap + lo];
        if (*w & clear) *w &= ~clear;
    }
}
// Raft::reset replaces the ReadOnly (raft.rs:957)
__device__ __forceinline__ void rd_empty(const Columns &c, uint32_t g) {
    if (c.rd_cap) c.rd_meta[g] &= kRdAlloc;
}

// ---------------------------------------------------------------------------
// MajorityConfig::committed_index without group commit (majority.rs:70-101):
// the q-th largest acked index of the voters in `mask`, q = n/2 + 1
// (util.rs:118-120); the empty config yields u64::MAX (majority.rs:71-75).

// General form (any masks, joint configurations): quorum_index_joint in quorum_select.h -- the 8 slots are ordered
// once as predecessor bit masks (28 compares) and the q-th largest member of each half is the member with q - 1
// predecessors inside its mask.  (Until round 2 each half sorted the zero-padded slots with a 19-comparator network.)

// The common 5-voter case (q = 3): the median, by the classic 10 min/max form
// med5(a..e) = med3(e, max(min(a,b),min(c,d)), min(max(a,b),max(c,d))).
__device__ __forceinline__ uint64_t median5(uint64_t a, uint64_t b, uint64_t c, uint64_t d,
                                            uint64_t e) {
    const uint64_t lo = umax64(umin64(a, b), umin64(c, d));
    const uint64_t hi = umin64(umax64(a, b), umax64(c, d));
    return umax64(umin64(lo, hi), umin64(umax64(lo, hi), e));
}

// MajorityConfig::committed_index WITH group commit (majority.rs:70-124), the
// literal algorithm: gather, stable descending sort, then the scan of :102-123.
// Rare path (ProgressTracker::group_commit is off by default), kept out of line
// so its local arrays do not cost the common path registers.
__device__ __noinline__ void majority_group_commit(const uint64_t *v, const uint64_t *gid,
                                                   uint32_t mask, uint64_t *out_index,
                                                   bool *out_use_gc) {
    if (mask == 0) {  // :71-75
        *out_index = UINT64_MAX;
        *out_use_gc = true;
        return;
    }
    uint64_t idx[kSlots], grp[kSlots];
    int n = 0;
    for (int s = 0; s < kSlots; s++) {
        if ((mask >> s) & 1u) {  // :77-85 (voters without progress do not occur in a tracker)
            idx[n] = v[s];
            grp[n] = gid[s];
            n++;
        }
    }
    for (int i = 1; i < n; i++) {  // :95 stable sort, descending by index
        uint64_t xi = idx[i], xg = grp[i];
        int j = i;
        while (j > 0 && idx[j - 1] < xi) {
            idx[j] = idx[j - 1];
            grp[j] = grp[j - 1];
            j--;
        }
        idx[j] = xi;
        grp[j] = xg;
    }
    const int quorum = n / 2 + 1;  // :97
    const uint64_t quorum_commit_index = idx[quorum - 1];
    uint64_t checked_group_id = grp[quorum - 1];
    bool single_group = true;
    for (int i = 0; i < n; i++) {  // :105-118
        if (grp[i] == 0) {
            single_group = false;
            continue;
        }
        if (checked_group_id == 0) {
            checked_group_id = grp[i];
            continue;
        }
        if (checked_group_id == grp[i]) continue;
        *out_index = umin64(idx[i], quorum_commit_index);
        *out_use_gc = true;
        return;
    }
    *out_index = single_group ? quorum_commit_index : idx[n - 1];  // :119-123
    *out_use_gc = false;
}

// ProgressTracker::maximal_committed_index (tracker.rs:294-298) of group g:
// JointConfig::committed_index (joint.rs:47-51) over both majority halves, reading
// matched / commit_group_id through the ProgressMap AckedIndexer (tracker.rs:183-190).
__device__ __forceinline__ void group_mci(const Columns &c, uint32_t g, uint32_t meta, uint64_t &mci,
                                          bool &use_gc) {
    const uint32_t in = RAFTGPU_META_IN(meta), out = RAFTGPU_META_OUT(meta);
    const uint32_t voters = in | out;
    uint64_t v[kSlots];
#pragma unroll
    for (int s = 0; s < kSlots; s++)
        v[s] = ((voters >> s) & 1u) ? c.matched[static_cast<size_t>(s) * c.cap + g] : 0ull;
    if (!(meta & RAFTGPU_META_GROUP_COMMIT)) {
        uint64_t i_idx, o_idx;
        quorum_index_joint(v, in, out, i_idx, o_idx);  // quorum_select.h; empty outgoing => u64::MAX
        mci = umin64(i_idx, o_idx);                    // joint.rs:50
        // a non-empty half reports false (majority.rs:99-101), an empty one true (:71-75)
        use_gc = (in == 0) && (out == 0);
    } else {
        uint64_t gid[kSlots];
        for (int s = 0; s < kSlots; s++)
            gid[s] = ((voters >> s) & 1u) ? c.commit_group_id[static_cast<size_t>(s) * c.cap + g] : 0ull;
        uint64_t i_idx, o_idx;
        bool i_gc, o_gc;
        majority_group_commit(v, gid, in, &i_idx, &i_gc);
        majority_group_commit(v, gid, out, &o_idx, &o_gc);
        mci = umin64(i_idx, o_idx);
        use_gc = i_gc && o_gc;  // joint.rs:50
    }
}

// ---------------------------------------------------------------------------
// WIDE groups (RAFTGPU_META_WIDE_LO / _HI): up to 16 peers over two consecutive group slots.  Rare (a joint change of
// a large configuration with learners), so the code is the literal algorithm on 16 values, out of line.

// MajorityConfig::committed_index over up to 16 voters: gather, stable descending insertion sort (majority.rs:95), the
// quorum element, then -- with group commit -- the scan of majority.rs:102-123.
__device__ __noinline__ void majority_committed_index16(const uint64_t *v, const uint64_t *gid, uint32_t mask, bool group_commit,
                                                        uint64_t *out_index, bool *out_use_gc) {
    if (mask == 0) {  // majority.rs:71-75
        *out_index = UINT64_MAX;
        *out_use_gc = true;
        return;
    }
    uint64_t idx[16], grp[16];
    int n = 0;
    for (int s = 0; s < 16; s++)
        if ((mask >> s) & 1u) {
            idx[n] = v[s];
            grp[n] = gid ? gid[s] : 0;
            n++;
        }
    for (int i = 1; i < n; i++) {
        const uint64_t xi = idx[i], xg = grp[i];
        int j = i;
        while (j > 0 && idx[j - 1] < xi) {
            idx[j] = idx[j - 1];
            grp[j] = grp[j - 1];
            j--;
        }
        idx[j] = xi;
        grp[j] = xg;
    }
    const int quorum = n / 2 + 1;  // util.rs:118-120
    const uint64_t quorum_commit_index = idx[quorum - 1];
    if (!group_commit) {  // majority.rs:99-101
        *out_index = quorum_commit_index;
        *out_use_gc = false;
        return;
    }
    uint64_t checked_group_id = grp[quorum - 1];
    bool single_group = true;
    for (int i = 0; i < n; i++) {  // :105-118
        if (grp[i] == 0) {
            single_group = false;
            continue;
        }
        if (checked_group_id == 0) {
            checked_group_id = grp[i];
            continue;
        }
        if (checked_group_id == grp[i]) continue;
        *out_index = umin64(idx[i], quorum_commit_index);
        *out_use_gc = true;
        return;
    }
    *out_index = single_group ? quorum_commit_index : idx[n - 1];  // :119-123
    *out_use_gc = false;
}

// maximal_committed_index of the wide group whose low half is g (tracker.rs:294-298, joint.rs:47-51)
__device__ __noinline__ void wide_mci(const Columns &c, uint32_t g, uint32_t meta_lo, uint64_t &mci, bool &use_gc) {
    const uint32_t meta_hi = c.meta[g + 1];
    const uint32_t in = RAFTGPU_META_IN(meta_lo) | (RAFTGPU_META_IN(meta_hi) << 8);
    const uint32_t out = RAFTGPU_META_OUT(meta_lo) | (RAFTGPU_META_OUT(meta_hi) << 8);
    const uint32_t voters = in | out;
    const bool gc = (meta_lo & RAFTGPU_META_GROUP_COMMIT) != 0;
    uint64_t v[16], gid[16];
    for (int s = 0; s < 16; s++) {
        const size_t cell = static_cast<size_t>(s & 7) * c.cap + g + (s >> 3);
        const bool member = (voters >> s) & 1u;
        v[s] = member ? c.matched[cell] : 0ull;
        gid[s] = (member && gc) ? c.commit_group_id[cell] : 0ull;
    }
    uint64_t i_idx, o_idx;
    bool i_gc, o_gc;
    majority_committed_index16(v, gid, in, gc, &i_idx, &i_gc);
    majority_committed_index16(v, gid, out, gc, &o_idx, &o_gc);
    mci = umin64(i_idx, o_idx);  // joint.rs:50
    use_gc = i_gc && o_gc;
}

// Side-effect-free single-group query (thread 0 of one warp).
__global__ void mci_kernel(Columns c, uint32_t g, uint64_t *out_mci, uint8_t *out_gc) {
    if (threadIdx.x != 0) return;
    uint64_t mci;
    bool use_gc;
    const uint32_t meta = c.meta[g];
    if (meta & RAFTGPU_META_WIDE_LO)
        wide_mci(c, g, meta, mci, use_gc);
    else
        group_mci(c, g, meta, mci, use_gc);
    *out_mci = mci;
    *out_gc = use_gc ? 1 : 0;
}

// Block-level counter flush: per-thread tallies -> warp shuffle reduce -> shared
// -> ONE global atomic per counter per block.  (v1 issued one atomic per warp per
// counter; ~10^5 same-address atomics serialise in L2 and dominated both kernels.)
template <int kN>
__device__ __forceinline__ void block_flush_counts(const uint32_t (&local)[kN], const int (&which)[kN],
                                                   unsigned long long *counters,
                                                   uint32_t *extra_u32 /* nullable, gets local[1] */) {
    __shared__ uint32_t s_cnt[kN];
    if (threadIdx.x < kN) s_cnt[threadIdx.x] = 0;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kN; k++) {
        const uint32_t w = __reduce_add_sync(0xffffffffu, local[k]);
        if ((threadIdx.x & 31) == 0 && w) atomicAdd(&s_cnt[k], w);
    }
    __syncthreads();
    if (threadIdx.x < kN && s_cnt[threadIdx.x]) {
        atomicAdd(&counters[which[threadIdx.x]], static_cast<unsigned long long>(s_cnt[threadIdx.x]));
        if (extra_u32 && threadIdx.x == 1) atomicAdd(extra_u32, s_cnt[1]);
    }
}
