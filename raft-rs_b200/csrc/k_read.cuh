// k_read.cuh -- ReadOnly (src/read_only.rs) on the device: the MsgReadIndex branch of step_leader, recv_ack for heartbeat
// responses, advance as a stream compaction, last_pending_request_ctx and the read tail of post_conf_change.
// Part of kernels.cuh (included there, inside namespace raftgpu; not a standalone header).
//
// Per group a bounded ring of pending requests (raftgpu_arena_enable_read_index): columns [rd_cap][cap] indexed by
// ring position -- ctx (the caller's 64-bit token of the context), index (raft_log.committed when queued), and one word
// of ack bits over peer slots 0..15, the from slot, LOCAL and the "acknowledged since the last release pass" mark --
// plus rd_meta [cap] = head | count << 16.  A wide group's queue lives on its low half.  The reference keys acks by
// peer id; here by slot, so raftgpu_group_set_conf clears a removed slot's bits (rd_clear_slots, k_common.cuh).
//
// Quorum is ProgressTracker::has_quorum (tracker.rs:367-372): both halves of the joint configuration Won with the acks
// as yes votes and everyone else missing -- majority_vote (k_control.cuh), the same function the vote tally uses.
// Learner acks are in the set but count for nothing, as in the reference.

constexpr uint32_t kRdInvalid = 0xffffffffu;

// The group a request / record belongs to (the low half of a wide group) and the peer slot 0..15 it names.
__device__ __forceinline__ uint32_t rd_lo(const Columns &c, uint32_t g, uint32_t &slot) {
    if (c.meta[g] & RAFTGPU_META_WIDE_HI) {
        slot += RAFTGPU_SLOTS;
        return g - 1;
    }
    return g;
}

// Voter masks over 16 slots and the self slot (kRdInvalid: none) of the group whose low half is `lo`.
__device__ __forceinline__ void rd_conf(const Columns &c, uint32_t lo, uint32_t &in, uint32_t &out, uint32_t &self) {
    const uint32_t m = c.meta[lo];
    const uint32_t mh = (m & RAFTGPU_META_WIDE_LO) ? c.meta[lo + 1] : 0u;
    in = RAFTGPU_META_IN(m) | (RAFTGPU_META_IN(mh) << 8);
    out = RAFTGPU_META_OUT(m) | (RAFTGPU_META_OUT(mh) << 8);
    self = (m & RAFTGPU_META_HAS_SELF) ? RAFTGPU_META_SELF(m)
           : (mh & RAFTGPU_META_HAS_SELF) ? RAFTGPU_SLOTS + RAFTGPU_META_SELF(mh) : kRdInvalid;
}

// ProgressTracker::has_quorum(acks) (tracker.rs:367-372) through JointConfig::vote_result (joint.rs:56-67)
__device__ __forceinline__ bool rd_quorum(uint32_t in, uint32_t out, uint32_t acks) {
    return majority_vote(in, acks, 0) == RAFTGPU_VOTE_WON && majority_vote(out, acks, 0) == RAFTGPU_VOTE_WON;
}

// Request i -> its group's low half (kRdInvalid: not allocated, or a non-LOCAL request from slot >= 8); w0 / from out.
__device__ __forceinline__ uint32_t rd_req_key(const Columns &c, const raftgpu_read_req *reqs, uint64_t i, uint32_t hi,
                                               uint64_t &w0, uint32_t &from) {
    w0 = reinterpret_cast<const uint64_t *>(reqs + i)[0];
    const uint32_t g = static_cast<uint32_t>(w0), flags = static_cast<uint32_t>(w0 >> 40) & 0xffu;
    from = static_cast<uint32_t>(w0 >> 32) & 0xffu;
    if (g >= hi || !(c.rd_meta[g] & kRdAlloc)) return kRdInvalid;
    if (flags & RAFTGPU_READ_LOCAL) {  // the from slot is not used: stored as 0
        uint32_t unused = 0;
        from = 0;
        return rd_lo(c, g, unused);
    }
    if (from >= RAFTGPU_SLOTS) return kRdInvalid;
    return rd_lo(c, g, from);
}

// Pass 1 of the request batch: the first run of every group, by atomicMin over its requests' positions.
__global__ void __launch_bounds__(256)
read_scan_kernel(Columns c, const raftgpu_read_req *__restrict__ reqs, uint64_t n, uint32_t hi, uint8_t *__restrict__ status) {
    const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
    for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
        uint64_t w0;
        uint32_t from;
        const uint32_t key = rd_req_key(c, reqs, i, hi, w0, from);
        if (key == kRdInvalid)
            status[i] = RAFTGPU_READ_INVALID;
        else
            atomicMin(&c.rd_first[key], static_cast<uint32_t>(i));
    }
}

// Pass 2: the thread at the head of a group's first run walks the run in batch order (the step_leader branch,
// raft.rs:2056-2091, per request); the head of any later run marks it SPLIT.  The first run's head puts rd_first back.
__global__ void __launch_bounds__(256)
read_apply_kernel(Columns c, const raftgpu_read_req *__restrict__ reqs, uint64_t n, uint32_t hi, uint8_t *__restrict__ status,
                  uint64_t *__restrict__ out_index) {
    const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
    for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
        uint64_t w0, w0p;
        uint32_t from, fromp;
        const uint32_t key = rd_req_key(c, reqs, i, hi, w0, from);
        if (key == kRdInvalid) {
            if (out_index) out_index[i] = 0;
            continue;
        }
        if (i > 0 && rd_req_key(c, reqs, i - 1, hi, w0p, fromp) == key) continue;  // not the head of a run
        if (c.rd_first[key] != static_cast<uint32_t>(i)) {
            for (uint64_t j = i; j < n && rd_req_key(c, reqs, j, hi, w0p, fromp) == key; j++) {
                status[j] = RAFTGPU_READ_SPLIT;
                if (out_index) out_index[j] = 0;
            }
            continue;
        }
        // commit_to_current_term (raft.rs:2057) in range form: the committed entry is of the leader's term
        const uint64_t committed = c.committed[key], ts = c.term_start[key], li = c.last_index[key];
        const bool current = ts <= committed && committed <= li;
        uint32_t in, out, self;
        rd_conf(c, key, in, out, self);
        const bool singleton = out == 0 && __popc(in) == 1;  // JointConfig::is_singleton, joint.rs:77-79
        const uint32_t m0 = c.rd_meta[key];
        const uint32_t head = rd_head(m0);
        uint32_t count = rd_count(m0);
        for (uint64_t j = i; j < n; j++) {
            if (j > i && rd_req_key(c, reqs, j, hi, w0, from) != key) break;
            const uint32_t flags = static_cast<uint32_t>(w0 >> 40) & 0xffu;
            const uint64_t ctx = reinterpret_cast<const uint64_t *>(reqs + j)[1];
            uint32_t st;
            uint64_t idx = 0;
            if (!current) {
                st = RAFTGPU_READ_DROPPED;                                   // :2057-2061
            } else if (singleton || (flags & RAFTGPU_READ_LEASE)) {
                st = RAFTGPU_READ_READY;                                     // :2063-2069, :2083-2088
                idx = committed;
            } else {
                st = RAFTGPU_READ_QUEUED;
                for (uint32_t k = 0; k < count; k++) {                       // read_only.rs:88-90
                    uint32_t p = head + k;
                    if (p >= c.rd_cap) p -= c.rd_cap;
                    if (c.rd_ctx[static_cast<size_t>(p) * c.cap + key] == ctx) {
                        st = RAFTGPU_READ_ALREADY_PENDING;
                        break;
                    }
                }
                if (st == RAFTGPU_READ_QUEUED && count == c.rd_cap) st = RAFTGPU_READ_FULL;
                if (st == RAFTGPU_READ_QUEUED) {                             // read_only.rs:91-98, acks = {self}
                    uint32_t p = head + count;
                    if (p >= c.rd_cap) p -= c.rd_cap;
                    const size_t cell = static_cast<size_t>(p) * c.cap + key;
                    c.rd_ctx[cell] = ctx;
                    c.rd_index[cell] = committed;
                    c.rd_word[cell] = (self != kRdInvalid ? 1u << self : 0u) | (from << kRdFromShift) |
                                      ((flags & RAFTGPU_READ_LOCAL) ? RAFTGPU_READ_WORD_LOCAL : 0u);
                    count++;
                    idx = committed;
                }
            }
            status[j] = static_cast<uint8_t>(st);
            if (out_index) out_index[j] = idx;
        }
        if (count != rd_count(m0)) c.rd_meta[key] = (m0 & ~0x00ff0000u) | (count << 16);
        c.rd_first[key] = kRdInvalid;
    }
}

// recv_ack (read_only.rs:104-109) for every HEARTBEAT | READ_CTX record whose peer has a Progress (raft.rs:1779-1789).
__global__ void __launch_bounds__(256)
read_ack_kernel(Columns c, const raftgpu_append_resp *__restrict__ recs, uint64_t n) {
    const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
    const uint32_t want = RAFTGPU_REC_HEARTBEAT | RAFTGPU_REC_READ_CTX;
    for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint64_t *p = reinterpret_cast<const uint64_t *>(recs + i);
        const uint64_t w0 = p[0], ctx = p[1];
        const uint32_t g = static_cast<uint32_t>(w0);
        uint32_t slot = static_cast<uint32_t>(w0 >> 32) & 0xffu;
        if (((static_cast<uint32_t>(w0 >> 40) & want) != want) || g >= c.cap || slot >= kSlots) continue;
        const uint32_t meta = c.meta[g];
        if (!(((RAFTGPU_META_IN(meta) | RAFTGPU_META_OUT(meta) | RAFTGPU_META_LEARN(meta)) >> slot) & 1u)) continue;
        const uint32_t lo = rd_lo(c, g, slot);
        const uint32_t m = c.rd_meta[lo];
        const uint32_t head = rd_head(m), count = rd_count(m);
        for (uint32_t k = 0; k < count; k++) {
            uint32_t q = head + k;
            if (q >= c.rd_cap) q -= c.rd_cap;
            const size_t cell = static_cast<size_t>(q) * c.cap + lo;
            if (c.rd_ctx[cell] == ctx) {  // tokens are unique within a group's pending set
                atomicOr(&c.rd_word[cell], (1u << slot) | RAFTGPU_READ_WORD_ACKED);
                break;
            }
        }
    }
}

// Write released request `cell` of group lo as a raftgpu_read_state (24 bytes: three u64 stores).
__device__ __forceinline__ void rd_emit(const Columns &c, uint32_t lo, size_t cell, raftgpu_read_state *out, uint64_t pos) {
    const uint32_t w = c.rd_word[cell];
    const uint32_t from = (w >> kRdFromShift) & 0xffu;
    const uint32_t local = (w & RAFTGPU_READ_WORD_LOCAL) ? RAFTGPU_READ_LOCAL : 0u;
    const uint32_t g = (!local && from >= RAFTGPU_SLOTS) ? lo + 1 : lo;  // a wide group's peer 8 + s is (g + 1, s)
    uint64_t *o = reinterpret_cast<uint64_t *>(out + pos);
    o[0] = static_cast<uint64_t>(g) | (static_cast<uint64_t>(local ? 0u : (from & 7u)) << 32) | (static_cast<uint64_t>(local) << 40);
    o[1] = c.rd_index[cell];
    o[2] = c.rd_ctx[cell];
}

// advance (read_only.rs:114-129) behind has_quorum for a batch of acks, as a stream compaction in the send_list_kernel
// pattern: one lane per group, each lane counts the requests it releases (up to the last acked-and-quorate one), a warp
// scan turns counts into offsets, ONE global atomic per warp reserves the range.  A warp whose range does not fit in
// `capacity` changes nothing (its groups keep queues and marks for the next call); count[0] counts it anyway,
// count[1] only what was written -- the warps that fit hold a prefix of the reservations.
// Algorithmic bytes per group: 4 (rd_meta) + 4 per pending request (rd_word) + 4 (meta) read; per released request
// 16 (ctx, index) read and 24 written, 4 (rd_meta) written.
__global__ void __launch_bounds__(256)
read_release_kernel(Columns c, uint32_t first, uint32_t n, raftgpu_read_state *__restrict__ out, unsigned long long capacity,
                    unsigned long long *__restrict__ count) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t base = first & ~31u;
    const uint32_t n_tiles = static_cast<uint32_t>((static_cast<uint64_t>(first - base) + n + 31) >> 5);
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t tile = warp; tile < n_tiles; tile += n_warps) {
        const uint32_t g = base + tile * 32u + lane;
        const bool in_range = g >= first && g < first + n;
        const uint32_t m = in_range ? c.rd_meta[g] : 0u;
        const uint32_t head = rd_head(m), pend = rd_count(m);
        uint32_t rel = 0, marked = 0;  // marked: a request of this group carries the ACKED mark
        if (pend) {
            uint32_t in, outm, self;
            rd_conf(c, g, in, outm, self);
            for (uint32_t k = 0; k < pend; k++) {
                uint32_t q = head + k;
                if (q >= c.rd_cap) q -= c.rd_cap;
                const uint32_t w = c.rd_word[static_cast<size_t>(q) * c.cap + g];
                if (!(w & RAFTGPU_READ_WORD_ACKED)) continue;
                marked = 1;
                if (rd_quorum(in, outm, w & kRdAckMask)) rel = k + 1;
            }
        }
        uint32_t incl = rel;  // inclusive warp scan
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= static_cast<uint32_t>(d)) incl += v;
        }
        const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
        if (!__any_sync(0xffffffffu, marked)) continue;
        unsigned long long pos = 0;
        if (lane == 31 && total) pos = atomicAdd(&count[0], static_cast<unsigned long long>(total));
        pos = __shfl_sync(0xffffffffu, pos, 31);
        if (pos + total > capacity) continue;  // does not fit: nothing changes for these 32 groups
        if (lane == 31 && total) atomicAdd(&count[1], static_cast<unsigned long long>(total));
        pos += incl - rel;
        if (!marked) continue;
        for (uint32_t k = 0; k < rel; k++) {
            uint32_t q = head + k;
            if (q >= c.rd_cap) q -= c.rd_cap;
            rd_emit(c, g, static_cast<size_t>(q) * c.cap + g, out, pos + k);
        }
        for (uint32_t k = rel; k < pend; k++) {  // the marks of the requests that stay
            uint32_t q = head + k;
            if (q >= c.rd_cap) q -= c.rd_cap;
            uint32_t *w = &c.rd_word[static_cast<size_t>(q) * c.cap + g];
            if (*w & RAFTGPU_READ_WORD_ACKED) *w &= ~RAFTGPU_READ_WORD_ACKED;
        }
        if (rel) {
            uint32_t h = head + rel;
            if (h >= c.rd_cap) h -= c.rd_cap;
            c.rd_meta[g] = (m & kRdAlloc) | h | ((pend - rel) << 16);
        }
    }
}

// last_pending_request_ctx (read_only.rs:132-134) of groups [first, first + n)
__global__ void __launch_bounds__(256)
read_last_ctx_kernel(Columns c, uint32_t first, uint32_t n, uint64_t *__restrict__ out) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint32_t g = first + i, m = c.rd_meta[g], pend = rd_count(m);
        uint32_t q = rd_head(m) + pend - 1;
        if (q >= c.rd_cap) q -= c.rd_cap;
        out[i] = pend ? c.rd_ctx[static_cast<size_t>(q) * c.cap + g] : RAFTGPU_NO_READ_CTX;
    }
}

// post_conf_change's read tail (raft.rs:2648-2664), one group: recv_ack(self, last ctx), then -- when that set is a
// quorum of the new configuration -- advance(last ctx) releases the whole queue.  res[0] = requests released (or
// needed, when they do not fit in `capacity`: then nothing is released), res[1] = 1 when they did not fit.
__global__ void read_conf_changed_kernel(Columns c, uint32_t g, raftgpu_read_state *out, uint64_t capacity,
                                         unsigned long long *res) {
    res[0] = res[1] = 0;
    const uint32_t m = c.rd_meta[g], head = rd_head(m), pend = rd_count(m);
    if (!pend) return;
    uint32_t in, outm, self;
    rd_conf(c, g, in, outm, self);
    uint32_t q = head + pend - 1;
    if (q >= c.rd_cap) q -= c.rd_cap;
    uint32_t *w = &c.rd_word[static_cast<size_t>(q) * c.cap + g];
    if (self != kRdInvalid) *w |= 1u << self;
    if (!rd_quorum(in, outm, *w & kRdAckMask)) return;
    res[0] = pend;
    if (pend > capacity) {
        res[1] = 1;
        return;
    }
    for (uint32_t k = 0; k < pend; k++) {
        uint32_t p = head + k;
        if (p >= c.rd_cap) p -= c.rd_cap;
        rd_emit(c, g, static_cast<size_t>(p) * c.cap + g, out, k);
    }
    c.rd_meta[g] = (m & kRdAlloc) | ((head + pend) % c.rd_cap);
}

// raftgpu_read_index_get: the queue of one group in order
__global__ void read_get_kernel(Columns c, uint32_t g, uint64_t *ctx, uint64_t *index, uint32_t *word, uint32_t *n) {
    const uint32_t m = c.rd_meta[g], pend = rd_count(m);
    for (uint32_t k = 0; k < pend; k++) {
        uint32_t p = rd_head(m) + k;
        if (p >= c.rd_cap) p -= c.rd_cap;
        const size_t cell = static_cast<size_t>(p) * c.cap + g;
        ctx[k] = c.rd_ctx[cell];
        index[k] = c.rd_index[cell];
        word[k] = c.rd_word[cell];
    }
    *n = pend;
}

// group alloc / free: the queue of [first, first + n) is empty, and marked allocated or not
__global__ void read_alloc_kernel(Columns c, uint32_t first, uint32_t n, uint32_t value) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) c.rd_meta[first + i] = value;
}
