// k_apply.cuh -- record formats (public, packed, compact stream), apply_one (raft.rs:1663-1743), the scatter apply kernels.
// Part of kernels.cuh (included there, inside namespace raftgpu; not a standalone header).

// ---------------------------------------------------------------------------
// Progress state helpers on a register copy of one cell.
struct Cell {
    uint64_t matched, next_idx;
    uint32_t flags;  // pflags byte
};

// progress.rs:75-80 reset_state: paused = false, pending_snapshot = 0, state, ins.reset()
__device__ __forceinline__ void reset_state(const Columns &c, size_t cell, Cell &p, uint32_t state, uint64_t *pending_snapshot) {
    p.flags &= ~(RAFTGPU_PF_PAUSED | RAFTGPU_PF_INS_FULL | RAFTGPU_PF_STATE_MASK);
    p.flags |= state;
    ins_reset(c, cell);  // ins.reset()
    // a plain store, not "if non-zero then clear": the cold column would otherwise cost a dependent
    // HBM read on every state transition (and, in the fused kernel, stall the tile's barrier)
    *pending_snapshot = 0;
}

// apply_kernel: the per-message prefix of Raft::handle_append_response
// (raft.rs:1663-1743) for one wave of records, one thread per record, persistent
// grid-stride loop.  Within a wave every (group, peer) cell is touched by at most
// one record, so threads never race on a cell and no atomics are needed on the
// columns.
//
// The loop is software-pipelined three deep, because the work is two dependent
// HBM round trips (the record names the cell; the cell decides the update):
//   iteration k issues   the record load of element k+2,
//                        the cell loads (meta, matched, next_idx, pflags,
//                        committed_index) of element k+1,
//   and computes / stores element k,
// so every load has a whole iteration to land.  (An extra L2-prefetch stage was
// measured and does not help: at ~12 MB in flight the kernel is limited by the DRAM
// efficiency of sector-granular scattered accesses, not by latency -- profiles/.)
// Algorithmic bytes per record: 24 (record) + RMW of matched, next_idx,
// committed_index (48) + flag byte and meta (~4) = 76.
struct RecRegs {
    uint64_t w0, index, commit;
};
struct CellRegs {
    uint32_t meta;
    uint32_t flags;
    uint64_t matched, next_idx, peer_committed;
};
// Where one cell's hot fields live: HBM (scatter kernel) or a shared-memory tile (fused kernel).
// The cold columns (pending_snapshot, pending_request_snapshot) are always addressed in HBM.
struct CellPtrs {
    uint64_t *matched, *next_idx, *peer_committed, *last_index;
    uint8_t *pflags;
};

// PackedRec and the kPk* / kCu* bit layouts: wire_format.h

template <bool kPacked>
__device__ __forceinline__ RecRegs load_rec(const void *recs_v, uint64_t i, uint64_t n) {
    RecRegs r;
    if (i >= n) {  // past the end: a no-op (EXT) record
        r.w0 = static_cast<uint64_t>(RAFTGPU_REC_EXT) << 40;
        r.index = 0;
        r.commit = 0;
        return r;
    }
    if constexpr (!kPacked) {
        const uint64_t *p = reinterpret_cast<const uint64_t *>(static_cast<const raftgpu_append_resp *>(recs_v) + i);
        r.w0 = p[0];
        r.index = p[1];
        r.commit = p[2];
    } else {
        const ulonglong2 q = reinterpret_cast<const ulonglong2 *>(recs_v)[i];  // one 128-bit load
        const uint64_t w0 = q.x;
        const uint32_t delta = static_cast<uint32_t>(w0 >> 40);
        const uint32_t flags = ((w0 & kPkReject) ? RAFTGPU_REC_REJECT : 0u) | ((w0 & kPkLocal) ? RAFTGPU_REC_LOCAL : 0u) |
                               ((w0 & kPkExt) ? RAFTGPU_REC_EXT : 0u);
        // the public layout: group | slot << 32 | flags << 40
        r.w0 = (w0 & 0xffffffffull) | (((w0 >> 32) & 7ull) << 32) | (static_cast<uint64_t>(flags) << 40);
        r.index = q.y;
        if (w0 & kPkLocal)
            r.commit = delta == kPkNoCommit ? 0 : q.y + delta;
        else
            r.commit = q.y - delta;
        if ((w0 & kPkWide) && !(w0 & kPkExt)) {  // rare: the exact commit follows in an EXT of kind 3
            for (uint64_t j = i + 1; j < n && j <= i + 3; j++) {
                const ulonglong2 e = reinterpret_cast<const ulonglong2 *>(recs_v)[j];
                if (!(e.x & kPkExt)) break;
                if ((e.x >> 40) == 3) r.commit = e.y;
            }
        }
    }
    return r;
}

// next_probe_index / request_snapshot of the REJECT at position i (raft.rs:1560-1661, 1709)
template <bool kPacked>
__device__ __forceinline__ void load_reject_ext(const void *recs_v, uint64_t i, uint64_t n, uint64_t &hint,
                                                uint64_t &request_snapshot) {
    hint = 0;
    request_snapshot = RAFTGPU_INVALID_INDEX;
    if constexpr (!kPacked) {
        if (i + 1 < n) {
            const uint64_t *e = reinterpret_cast<const uint64_t *>(static_cast<const raftgpu_append_resp *>(recs_v) + i + 1);
            if ((e[0] >> 40) & RAFTGPU_REC_EXT) {
                hint = e[1];
                request_snapshot = e[2];
            }
        }
    } else {
        for (uint64_t j = i + 1; j < n && j <= i + 3; j++) {
            const ulonglong2 e = reinterpret_cast<const ulonglong2 *>(recs_v)[j];
            if (!(e.x & kPkExt)) break;
            const uint32_t kind = static_cast<uint32_t>(e.x >> 40);
            if (kind == 1) hint = e.y;
            if (kind == 2) request_snapshot = e.y;
        }
    }
}

__device__ __forceinline__ CellPtrs global_cell_ptrs(const Columns &c, const RecRegs &r) {
    const uint32_t g = static_cast<uint32_t>(r.w0);
    const uint32_t slot = static_cast<uint32_t>(r.w0 >> 32) & 0xffu;
    const bool ok = g < c.cap && slot < kSlots;
    const size_t cell = ok ? static_cast<size_t>(slot) * c.cap + g : 0;
    return CellPtrs{c.matched + cell, c.next_idx + cell, c.peer_committed + cell, c.last_index + (ok ? g : 0),
                    c.pflags + cell};
}

__device__ __forceinline__ CellRegs load_cell(const Columns &c, const RecRegs &r) {
    const uint32_t g = static_cast<uint32_t>(r.w0);
    const uint32_t slot = static_cast<uint32_t>(r.w0 >> 32) & 0xffu;
    // cell 0 / group 0 is a harmless stand-in for EXT and out-of-range records
    // (nothing is written for them)
    const bool ok = !((r.w0 >> 40) & RAFTGPU_REC_EXT) && g < c.cap && slot < kSlots;
    const size_t cell = ok ? static_cast<size_t>(slot) * c.cap + g : 0;
    CellRegs d;
    d.meta = c.meta[ok ? g : 0];
    d.matched = c.matched[cell];
    d.next_idx = c.next_idx[cell];
    d.flags = c.pflags[cell];
    d.peer_committed = c.peer_committed[cell];
    return d;
}

// One record against its cell: raft.rs:1663-1743.  Returns the result byte.
// kFmt: 0 = records in the public 24-byte layout, 1 = packed 16-byte records (a REJECT's EXT is
// looked up behind position i in either), 2 = the caller has decoded them already (compact
// streams) and hands them in through the two integer arguments: n = next_probe_index hint,
// i = request_snapshot (recs unused) -- registers only, no stack traffic.
template <int kFmt>
__device__ __forceinline__ uint32_t apply_one(const Columns &c, const void *recs, uint64_t n, uint64_t i,
                                              const RecRegs &rec, const CellRegs &cd, const CellPtrs &ptr,
                                              uint32_t *local) {
    const uint64_t index = rec.index, commit = rec.commit;
    const uint32_t g = static_cast<uint32_t>(rec.w0);
    const uint32_t slot = static_cast<uint32_t>(rec.w0 >> 32) & 0xffu;
    const uint32_t rflags = static_cast<uint32_t>(rec.w0 >> 40) & 0xffu;
    if (rflags & RAFTGPU_REC_EXT) return 0;
    local[0]++;
    const bool in_range = g < c.cap && slot < kSlots;
    const uint32_t present =
        RAFTGPU_META_IN(cd.meta) | RAFTGPU_META_OUT(cd.meta) | RAFTGPU_META_LEARN(cd.meta);
    if (!in_range || !((present >> slot) & 1u)) {
        // raft.rs:1663-1673: no progress available for m.from
        local[4]++;
        return RAFTGPU_RES_NO_PROGRESS;
    }
    const size_t cell = static_cast<size_t>(slot) * c.cap + g;
    Cell pr;
    pr.matched = cd.matched;
    pr.next_idx = cd.next_idx;
    pr.flags = cd.flags;
    const uint32_t state = pr.flags & RAFTGPU_PF_STATE_MASK;
    uint32_t res = 0;

    if (rflags & RAFTGPU_REC_LOCAL) {
        // raft.rs:974-991 append_entry: last_index grew
        if (commit != 0) *ptr.last_index = commit;
        // raft.rs:1010-1014 on_persist_entries: prs[self].maybe_update(index)
        if (pr.matched < index) {  // progress.rs:138-150
            pr.matched = index;
            pr.flags &= ~RAFTGPU_PF_PAUSED;
            local[1]++;
            res = RAFTGPU_RES_OK;
        }
        if (pr.next_idx < index + 1) pr.next_idx = index + 1;
    } else {
        pr.flags |= RAFTGPU_PF_RECENT_ACTIVE;  // raft.rs:1674
        // raft.rs:1677 pr.update_committed(m.commit), progress.rs:153-157
        if (commit > cd.peer_committed) *ptr.peer_committed = commit;

        if (rflags & RAFTGPU_REC_REJECT) {
            local[2]++;
            uint64_t hint, request_snapshot;
            if constexpr (kFmt == 2) {
                hint = n;
                request_snapshot = i;
            } else {
                load_reject_ext<(kFmt == 1)>(recs, i, n, hint, request_snapshot);
            }
            // Progress::maybe_decr_to, progress.rs:168-206
            bool ok;
            if (state == RAFTGPU_STATE_REPLICATE) {
                if (index < pr.matched || (index == pr.matched && request_snapshot == RAFTGPU_INVALID_INDEX)) {
                    ok = false;  // :173-177 stale
                } else {
                    if (request_snapshot == RAFTGPU_INVALID_INDEX)
                        pr.next_idx = pr.matched + 1;  // :178-179
                    else
                        c.pending_req_snapshot[cell] = request_snapshot;  // :181
                    ok = true;
                }
            } else if ((pr.next_idx == 0 || pr.next_idx - 1 != index) &&
                       request_snapshot == RAFTGPU_INVALID_INDEX) {
                ok = false;  // :188-192 stale
            } else {
                if (request_snapshot == RAFTGPU_INVALID_INDEX) {  // :195-199
                    pr.next_idx = umin64(index, hint + 1);
                    if (pr.next_idx < 1) pr.next_idx = 1;
                } else if (c.pending_req_snapshot[cell] == RAFTGPU_INVALID_INDEX) {
                    c.pending_req_snapshot[cell] = request_snapshot;  // :200-203
                }
                pr.flags &= ~RAFTGPU_PF_PAUSED;  // :204 resume()
                ok = true;
            }
            if (ok) {
                local[3]++;
                res = RAFTGPU_RES_OK | RAFTGPU_RES_SEND;
                if (state == RAFTGPU_STATE_REPLICATE) {
                    // raft.rs:1716-1718 become_probe (progress.rs:95-107, not Snapshot)
                    reset_state(c, cell, pr, RAFTGPU_STATE_PROBE, &c.pending_snapshot[cell]);
                    pr.next_idx = pr.matched + 1;
                }
            }
        } else {
            // raft.rs:1724 old_paused = pr.is_paused(), progress.rs:210-216
            const bool old_paused =
                state == RAFTGPU_STATE_PROBE
                    ? (pr.flags & RAFTGPU_PF_PAUSED) != 0
                    : (state == RAFTGPU_STATE_REPLICATE ? (pr.flags & RAFTGPU_PF_INS_FULL) != 0 : true);
            // raft.rs:1725 pr.maybe_update(m.index), progress.rs:138-150
            const bool need_update = pr.matched < index;
            if (need_update) {
                pr.matched = index;
                pr.flags &= ~RAFTGPU_PF_PAUSED;
            }
            if (pr.next_idx < index + 1) pr.next_idx = index + 1;
            if (need_update) {
                local[1]++;
                res = RAFTGPU_RES_OK | (old_paused ? RAFTGPU_RES_OLD_PAUSED : 0u);
                if (state == RAFTGPU_STATE_PROBE) {
                    // raft.rs:1730 become_replicate, progress.rs:110-114
                    reset_state(c, cell, pr, RAFTGPU_STATE_REPLICATE, &c.pending_snapshot[cell]);
                    pr.next_idx = pr.matched + 1;
                } else if (state == RAFTGPU_STATE_SNAPSHOT) {
                    // raft.rs:1731-1741 maybe_snapshot_abort -> become_probe
                    const uint64_t pending = c.pending_snapshot[cell];
                    if (pr.matched >= pending) {  // progress.rs:131-134
                        reset_state(c, cell, pr, RAFTGPU_STATE_PROBE, &c.pending_snapshot[cell]);
                        pr.next_idx = umax64(pr.matched + 1, pending + 1);  // :99-102
                    }
                } else if (c.ins_cap) {
                    ins_free_to(c, cell, index, pr.flags);  // raft.rs:1742 Replicate: pr.ins.free_to(m.index)
                }  // (without device-side windows the Inflights ring is the host's)
            }
        }
    }
    if (pr.matched != cd.matched) *ptr.matched = pr.matched;
    if (pr.next_idx != cd.next_idx) *ptr.next_idx = pr.next_idx;
    if (pr.flags != cd.flags) *ptr.pflags = static_cast<uint8_t>(pr.flags);
    return res;
}

// kCheckDup (zero-copy submissions, where no host code has seen the records): every record marks
// its cell in `touched` ([cap] bytes, one bit per peer slot, cleared by the caller beforehand)
// with an L2 atomic; a cell marked twice breaks the one-wave precondition -- the record is NOT
// applied and *dup_count is bumped so the step can fail loudly.
template <bool kPacked, bool kCheckDup = false>
__global__ void __launch_bounds__(256, 4)
apply_kernel(Columns c, const void *__restrict__ recs, uint64_t n, uint8_t *__restrict__ results,
             unsigned long long *__restrict__ counters, uint32_t *__restrict__ touched = nullptr,
             uint32_t *__restrict__ dup_count = nullptr, uint32_t min_group = 0) {
    // (kCheckDup: a record of a group below min_group is refused like a duplicate -- the hybrid step promises that
    //  its raw part only holds groups above its packed part)
    const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
    uint32_t local[5] = {0, 0, 0, 0, 0};  // records, updates, rejects, decrements, no_progress
    uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    // prologue: fill the pipeline
    RecRegs rec_a = load_rec<kPacked>(recs, i, n);
    RecRegs rec_b = load_rec<kPacked>(recs, i + stride, n);
    CellRegs cell_a = load_cell(c, rec_a);
    for (; i < n; i += stride) {
        const RecRegs rec_c = load_rec<kPacked>(recs, i + 2 * stride, n);  // element k+2: record
        const CellRegs cell_b = load_cell(c, rec_b);               // element k+1: cell -> registers
        if constexpr (kCheckDup) {
            const uint32_t g = static_cast<uint32_t>(rec_a.w0), slot = static_cast<uint32_t>(rec_a.w0 >> 32) & 0xffu;
            if (!((rec_a.w0 >> 40) & RAFTGPU_REC_EXT) && g < c.cap && slot < kSlots) {
                const uint32_t bit = 1u << (8 * (g & 3u) + slot);
                if (g < min_group || (atomicOr(&touched[g >> 2], bit) & bit)) {  // second record for this cell in one wave
                    atomicAdd(dup_count, 1u);
                    if (results) results[i] = 0;
                    rec_a = rec_b;
                    cell_a = cell_b;
                    rec_b = rec_c;
                    continue;
                }
            }
        }
        const CellPtrs gp = global_cell_ptrs(c, rec_a);
        const uint32_t res = apply_one<(kPacked ? 1 : 0)>(c, recs, n, i, rec_a, cell_a, gp, local);  // element k
        if (results) results[i] = static_cast<uint8_t>(res);
        rec_a = rec_b;
        cell_a = cell_b;
        rec_b = rec_c;
    }
    const int which[5] = {kCntRecords, kCntUpdates, kCntRejects, kCntDecrements, kCntNoProgress};
    block_flush_counts<5>(local, which, counters, nullptr);
}

// ---------------------------------------------------------------------------
// The compact stream (raftgpu.h "compact stream"): 4-byte units, group runs with a header.
struct CompactSrc {
    const uint32_t *units;
    const uint32_t *g_base;              // one per block of RAFTGPU_COMPACT_BLOCK units
    const raftgpu_append_resp *side;     // ESC targets, public layout (a REJECT is followed by its EXT)
    uint32_t n_units, n_side;
};

// A REJECT's payload unit (the one behind it): hint = index + signed 29-bit delta.
__device__ __forceinline__ uint64_t compact_hint(uint64_t index, uint32_t payload_unit) {
    const int32_t d = static_cast<int32_t>(payload_unit << 1) >> 3;  // bits [2,31), sign-extended
    return index + static_cast<uint64_t>(static_cast<int64_t>(d));
}

// Unit i as a record in the public register layout.  Headers, payload units, padding and
// malformed units come back as EXT (a no-op).
__device__ __forceinline__ RecRegs load_compact(const CompactSrc &s, uint64_t i) {
    RecRegs r;
    r.w0 = static_cast<uint64_t>(RAFTGPU_REC_EXT) << 40;
    r.index = 0;
    r.commit = 0;
    if (i >= s.n_units) return r;
    const uint32_t u = s.units[i];
    const uint32_t kind = u & 3u;
    if (kind == kCuEsc) {
        const uint32_t k = u >> 2;
        if (k < s.n_side && k < kCuPad) {
            const uint64_t *p = reinterpret_cast<const uint64_t *>(s.side + k);
            r.w0 = p[0];
            r.index = p[1];
            r.commit = p[2];
        }
        return r;
    }
    if (kind != kCuRec) return r;
    const uint32_t back = (u >> 3) & 7u;
    if (i < back + 2u) return r;
    const uint64_t h = i - back - 2u;
    const uint32_t ha = s.units[h], hb = s.units[h + 1];
    if ((ha & 3u) != kCuHdrA || (hb & 3u) != kCuHdrB) return r;
    const uint32_t g = s.g_base[h / RAFTGPU_COMPACT_BLOCK] + ((hb >> 2) & 0xfffu);
    const uint64_t base = static_cast<uint64_t>(ha >> 2) | (static_cast<uint64_t>(hb >> 14) << 30);
    const uint32_t slot = (u >> 6) & 7u;
    const uint64_t index = base + ((u >> 10) & 0x3fffu);
    const uint32_t cd = u >> 24;
    const bool local = (u & kCuLocal) != 0;
    uint32_t flags = local ? RAFTGPU_REC_LOCAL : 0u;
    r.index = index;
    r.commit = local ? (cd == kCuNoCommit ? 0 : index + cd) : (index >= cd ? index - cd : 0);
    if (u & kCuReject) flags = RAFTGPU_REC_REJECT;
    r.w0 = static_cast<uint64_t>(g) | (static_cast<uint64_t>(slot) << 32) | (static_cast<uint64_t>(flags) << 40);
    return r;
}

// {next_probe_index hint, request_snapshot} of the REJECT that unit i decoded to (rare: looked up
// when the record is applied, not carried through the pipeline).
__device__ __forceinline__ void compact_reject_ext(const CompactSrc &s, uint64_t i, uint64_t index, uint64_t (&ext)[2]) {
    ext[0] = 0;
    ext[1] = RAFTGPU_INVALID_INDEX;
    const uint32_t u = s.units[i];
    if ((u & 3u) == kCuEsc) {
        load_reject_ext<false>(s.side, u >> 2, s.n_side, ext[0], ext[1]);
    } else {
        const uint32_t pl = i + 1 < s.n_units ? s.units[i + 1] : 0u;
        if ((pl & 3u) == kCuEsc && ((pl >> 2) & kCuPayload)) ext[0] = compact_hint(index, pl);
    }
}

// apply_kernel for a compact stream: the same three-deep pipeline, one thread per UNIT (header
// units idle).  A run's header sits in the cache lines its records' neighbours load, so the
// decode adds L1/L2 hits, not HBM trips.  REJECTs only arrive through ESC units, whose payload
// (and EXT continuation) is read from the side table in the public layout.
template <bool kCheckDup>
__global__ void __launch_bounds__(256, 4)
apply_compact_kernel(Columns c, CompactSrc src, uint8_t *__restrict__ results, unsigned long long *__restrict__ counters,
                     uint32_t *__restrict__ touched, uint32_t *__restrict__ dup_count) {
    const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
    const uint64_t n = src.n_units;
    uint32_t local[5] = {0, 0, 0, 0, 0};  // records, updates, rejects, decrements, no_progress
    uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    RecRegs rec_a = load_compact(src, i);
    RecRegs rec_b = load_compact(src, i + stride);
    CellRegs cell_a = load_cell(c, rec_a);
    for (; i < n; i += stride) {
        const RecRegs rec_c = load_compact(src, i + 2 * stride);
        const CellRegs cell_b = load_cell(c, rec_b);
        bool skip = false;
        if constexpr (kCheckDup) {
            const uint32_t g = static_cast<uint32_t>(rec_a.w0), slot = static_cast<uint32_t>(rec_a.w0 >> 32) & 0xffu;
            if (!((rec_a.w0 >> 40) & RAFTGPU_REC_EXT) && g < c.cap && slot < kSlots) {
                const uint32_t bit = 1u << (8 * (g & 3u) + slot);
                if (atomicOr(&touched[g >> 2], bit) & bit) {  // second record for this cell in one wave
                    atomicAdd(dup_count, 1u);
                    skip = true;
                }
            }
        }
        uint32_t res = 0;
        if (!skip) {
            const CellPtrs gp = global_cell_ptrs(c, rec_a);
            uint64_t ext[2] = {0, RAFTGPU_INVALID_INDEX};
            if ((rec_a.w0 >> 40) & RAFTGPU_REC_REJECT) compact_reject_ext(src, i, rec_a.index, ext);
            res = apply_one<2>(c, nullptr, ext[0], ext[1], rec_a, cell_a, gp, local);
        }
        if (results) results[i] = static_cast<uint8_t>(res);
        rec_a = rec_b;
        cell_a = cell_b;
        rec_b = rec_c;
    }
    const int which[5] = {kCntRecords, kCntUpdates, kCntRejects, kCntDecrements, kCntNoProgress};
    block_flush_counts<5>(local, which, counters, nullptr);
}
