// k_tile.cuh -- step_tile_kernel: the fused apply + recompute tile kernel on packed records (the headline kernel), and
// the machinery it shares with step_tile_compact_kernel (k_tile_compact.cuh): the stage layout, the load and store
// warps, the barrier set-up, the commit phase, the hand-over, the general record path and the counter flush.
// Part of kernels.cuh (included there, inside namespace raftgpu; not a standalone header).

// ---------------------------------------------------------------------------
// step_tile_kernel: apply + recompute FUSED, for batches whose records are in group order.
//
// The scatter apply kernel above moves ~12 MB in flight but tops out near 3.7 TB/s: its cell
// accesses are sector-granular (8 useful bytes per 32-byte sector request, several rows per
// record), which HBM serves at roughly half the efficiency of dense bursts.  When the batch is
// ordered by group, a tile of kFTile consecutive groups owns a CONTIGUOUS record range, so the
// whole step becomes dense traffic: per tile the load warp (tile_load_warp) bulk-loads (TMA, cp.async.bulk)
// the tile's rows of matched / next_idx / committed_index / pflags / meta / committed /
// term_start / last_index into one shared-memory stage (TileStage); the consumers
//   A. apply every record of the tile, read straight from HBM / L2, to the shared-memory rows (one thread per record;
//      distinct cells per wave, so no conflicts),
//   B. recompute the commit index of the tile's groups from the same shared-memory rows (tile_commit;
//      matched is read from HBM once per step instead of twice),
//   C. hand the stage to the store warp (tile_handoff), which bulk-stores the rows back (tile_store_warp).
// Peer slots outside `hint` (learners) and the cold columns are handled through HBM directly.
// tile_off[t] = index of the first packed record of tile t (raftgpu_tile_index builds it).
constexpr int kFTile = RAFTGPU_TILE_GROUPS;  // groups per tile = threads per consumer group
// consumer groups per CTA: tile i of a CTA is handled by group i % kFGroups, so the phases of kFGroups tiles overlap
// inside one CTA (DESIGN 3.4: why three)
constexpr int kFGroups = 3;
constexpr int kFMaxStages = 8;
// Row strides inside a stage.  Records arrive in group order, so the ~3.5 records of one group sit
// in neighbouring lanes and touch the SAME column index of DIFFERENT rows: with a 256-element row
// stride they would all fall on the same shared-memory banks (4-way conflicts on every access).
// 258 u64 (= 2064 B, still 16-byte aligned for TMA) shifts consecutive rows by 4 banks.
constexpr uint32_t kFRow64 = (kFTile + 2) * 8;   // bytes per u64 row
constexpr uint32_t kFRow8 = kFTile + 16;         // bytes per u8 (pflags) row
constexpr uint32_t kFDefer = 32;                 // deferred (rare-path) records per warp per tile; more are handled inline
// units step_tile_compact_kernel stages per tile (a multiple of 4); the rest of a crowded tile is read from HBM
constexpr uint32_t kCUnitCap = 1536;

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// 1-D TMA: global -> shared, completion counted in bytes on `bar`
__device__ __forceinline__ void tma_load_1d(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
// 1-D TMA store: shared -> global, tracked by the per-thread bulk async-group
__device__ __forceinline__ void tma_store_1d(void *dst, const void *src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int n_threads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n_threads) : "memory");
}
// A consumer's wait for "the loads of MY tile have landed in this stage".  A consumer group sees only every kFGroups-th
// tile, so on one stage's `full` barrier it skips phases -- and a parity wait is only exact while the waiter is at
// most ONE phase ahead.  With uniform tiles that always holds; with a batch that covers only part of the groups it
// does not (record-less tiles are done in a microsecond, loads of light and heavy tiles land out of order): a group
// could pass the barrier of a stage still armed for the PREVIOUS tile and work on half-landed rows.  So it first
// waits for the previous use of the stage to be DONE (`done` barrier, previous phase).  That wait is exact: the
// group's own previous tile was loaded, hence the tile n_stages before IT was stored, stores happen in tile order,
// and with n_stages >= kFGroups that covers the previous user of this stage; and once the previous user is done, the
// `full` barrier is in this tile's phase, so the second wait is exact too.
__device__ __forceinline__ void wait_stage(uint64_t *full_bar, uint64_t *done_bar, uint32_t parity) {
    mbar_wait(done_bar, parity ^ 1u);  // (first use of a stage: the parity-1 wait on a fresh barrier passes at once)
    mbar_wait(full_bar, parity);
}

// The peer slot of the r-th hinted row of a stage.
__device__ __forceinline__ uint32_t hinted_slot(uint32_t hint, uint32_t r) {
    uint32_t slot = 0, seen = 0;
    for (uint32_t s2 = 0; s2 < kSlots; s2++)
        if ((hint >> s2) & 1u) {
            if (seen == r) slot = s2;
            seen++;
        }
    return slot;
}

// One stage of the ring, as both fused kernels lay it out: H rows each of matched, next_idx and committed_index (u64,
// kFRow64 apart, one per hinted peer slot), then the tile's rows of committed, term_start and last_index (u64), meta
// (u32), and H pflags rows (u8, kFRow8 apart).  tile_stage_bytes(H) is its size; the compact kernel stages its units
// behind it.
__host__ __device__ constexpr uint32_t tile_stage_bytes(uint32_t H) {
    return 3u * H * kFRow64 + 3u * kFRow64 + kFTile * 4u + H * kFRow8;
}
struct TileStage {
    uint64_t *matched, *next, *pc, *committed, *ts, *li;
    uint32_t *meta;
    uint8_t *flags;
    uint32_t *units;  // step_tile_compact_kernel: the tile's staged units
    __device__ __forceinline__ TileStage(uint8_t *smem, int st, uint32_t stage_bytes, uint32_t H) {
        uint8_t *sb = smem + static_cast<size_t>(st) * stage_bytes;
        const uint32_t o_next = H * kFRow64, o_pc = 2u * H * kFRow64, o_committed = 3u * H * kFRow64,
                       o_ts = o_committed + kFRow64, o_li = o_ts + kFRow64, o_meta = o_li + kFRow64,
                       o_flags = o_meta + kFTile * 4u;
        matched = reinterpret_cast<uint64_t *>(sb);
        next = reinterpret_cast<uint64_t *>(sb + o_next);
        pc = reinterpret_cast<uint64_t *>(sb + o_pc);
        committed = reinterpret_cast<uint64_t *>(sb + o_committed);
        ts = reinterpret_cast<uint64_t *>(sb + o_ts);
        li = reinterpret_cast<uint64_t *>(sb + o_li);
        meta = reinterpret_cast<uint32_t *>(sb + o_meta);
        flags = sb + o_flags;
        units = reinterpret_cast<uint32_t *>(sb + tile_stage_bytes(H));
    }
};

// Row j of a stage and the HBM row it mirrors, for the tile of groups from g0 (ng16 of them, rounded up to 16 bytes
// for every row; inside the padded stride): j < 4H the hinted rows of matched, next_idx, committed_index and pflags,
// then committed, last_index, term_start and meta.  The load warp copies all 4H + 4 in; the store warp writes the
// first 4H + 2 back.
struct TileRow {
    void *smem, *hbm;
    uint32_t bytes;
};
__device__ __forceinline__ TileRow tile_row(const Columns &c, const TileStage &s, uint32_t j, uint32_t hint, uint32_t H,
                                            uint32_t g0, uint32_t ng16) {
    constexpr uint32_t R64 = kFRow64 / 8;
    if (j < 4u * H) {
        const uint32_t col = j / H, r = j % H;
        const size_t cell = static_cast<size_t>(hinted_slot(hint, r)) * c.cap + g0;
        if (col == 0) return {s.matched + r * R64, c.matched + cell, ng16 * 8u};
        if (col == 1) return {s.next + r * R64, c.next_idx + cell, ng16 * 8u};
        if (col == 2) return {s.pc + r * R64, c.peer_committed + cell, ng16 * 8u};
        return {s.flags + r * kFRow8, c.pflags + cell, ng16};
    }
    if (j == 4u * H) return {s.committed, c.committed + g0, ng16 * 8u};
    if (j == 4u * H + 1u) return {s.li, c.last_index + g0, ng16 * 8u};
    if (j == 4u * H + 2u) return {s.ts, c.term_start + g0, ng16 * 8u};
    return {s.meta, c.meta + g0, ng16 * 4u};
}

struct TileBarriers {
    uint64_t full[kFMaxStages];   // loads landed            (load warp -> consumers)
    uint64_t done[kFMaxStages];   // rows final in smem      (consumers -> store warp)
    uint64_t empty[kFMaxStages];  // rows read by the stores (store warp -> load warp)
};
__device__ __forceinline__ void tile_init_barriers(TileBarriers &bar, int n_stages) {
    if (threadIdx.x == 0) {
        for (int s = 0; s < n_stages; s++) {
            mbar_init(&bar.full[s], 1);
            mbar_init(&bar.done[s], 1);
            mbar_init(&bar.empty[s], 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
}

// What both fused kernels take besides their records.
struct FusedArgs {
    const uint32_t *tile_off;  // [n_tiles + 1]: where tile t's records start
    uint32_t n_groups;         // groups [0, n_groups)
    uint32_t hint;
    int n_stages;
    uint8_t *results;          // nullable, one byte per packed record / compact unit
    uint32_t *adv_bitmap;      // nullable
    uint64_t *commit_out;      // nullable
    uint32_t *step_advanced;   // nullable
    unsigned long long *counters;
    unsigned long long *dbg;   // nullable: [8] cycle totals per phase (diagnostics, RAFTGPU_TILE_DEBUG=1)
};

struct TileArgs : FusedArgs {
    const PackedRec *recs;     // packed records in group order
    uint32_t skip;             // diagnostics only (RAFTGPU_TILE_SKIP, results are WRONG): 1 no records, 2 no recompute, 4 no stores
};

// The load warp of both fused kernels: once the store warp has released a stage, the tile's rows (tile_row) and,
// given `units` (the compact kernel), up to kCUnitCap of its units from the 16-byte boundary below its first one
// arrive in it by TMA.  The `full` barrier expects the byte total of the same copies.
__device__ __forceinline__ void tile_load_warp(const Columns &c, const FusedArgs &a, uint8_t *smem, uint32_t stage_bytes,
                                               uint32_t hint, uint32_t H, TileBarriers &bar, const uint32_t *units) {
    const uint32_t n_tiles = (a.n_groups + kFTile - 1) / kFTile;
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t n_rows = 4u * H + 4u;
    uint32_t it = 0;
    uint32_t nx_u0 = 0, nx_u1 = 0;
    if (units && blockIdx.x < n_tiles) {
        nx_u0 = a.tile_off[blockIdx.x];
        nx_u1 = a.tile_off[blockIdx.x + 1];
    }
    for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, it++) {
        const int st = it % a.n_stages;
        const uint32_t ph = (it / a.n_stages) & 1u;
        const uint32_t g0 = tile * kFTile;
        const uint32_t ng = a.n_groups - g0 < kFTile ? a.n_groups - g0 : kFTile;
        const uint32_t ng16 = (ng + 15u) & ~15u;
        uint32_t ua = 0, staged = 0;
        if (units) {
            const uint32_t u0 = nx_u0, u1 = nx_u1;
            if (tile + gridDim.x < n_tiles) {  // next tile's index: fetched while this one is being issued
                nx_u0 = a.tile_off[tile + gridDim.x];
                nx_u1 = a.tile_off[tile + gridDim.x + 1];
            }
            ua = u0 & ~3u;
            const uint32_t cnt4 = (u1 - ua + 3u) & ~3u;
            staged = u1 > u0 ? (cnt4 < kCUnitCap ? cnt4 : kCUnitCap) : 0u;
        }
        const TileStage s(smem, st, stage_bytes, H);
        // copy j < n_rows: row j; copy n_rows: the units (read only)
        const uint32_t n_copies = n_rows + (staged ? 1u : 0u);
        auto copy = [&](uint32_t j) -> TileRow {
            return j < n_rows ? tile_row(c, s, j, hint, H, g0, ng16)
                              : TileRow{s.units, const_cast<uint32_t *>(units + ua), staged * 4u};
        };
        uint32_t bytes = 0;
        for (uint32_t j = lane; j < n_copies; j += 32) bytes += copy(j).bytes;
        bytes = __reduce_add_sync(0xffffffffu, bytes);
        if (lane == 0) {
            mbar_wait(&bar.empty[st], ph ^ 1u);
            mbar_expect_tx(&bar.full[st], bytes);
        }
        __syncwarp();
        for (uint32_t j = lane; j < n_copies; j += 32) {
            const TileRow row = copy(j);
            tma_load_1d(row.smem, row.hbm, row.bytes, &bar.full[st]);
        }
    }
}

// The store warp of both fused kernels: once the consumers are done with a stage, its rows go back to HBM (and the
// `committed` row to commit_out as well: one dense copy, not 8-byte scatters), then the stage is free for the load
// warp.  no_stores: diagnostics only (RAFTGPU_TILE_SKIP, results are WRONG).
__device__ __forceinline__ void tile_store_warp(const Columns &c, const FusedArgs &a, uint8_t *smem, uint32_t stage_bytes,
                                                uint32_t hint, uint32_t H, bool no_stores, TileBarriers &bar) {
    const uint32_t n_tiles = (a.n_groups + kFTile - 1) / kFTile;
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t n_out = 4u * H + 2u + (a.commit_out ? 1u : 0u);
    uint32_t it = 0;
    for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, it++) {
        const int st = it % a.n_stages;
        const uint32_t ph = (it / a.n_stages) & 1u;
        const uint32_t g0 = tile * kFTile;
        const uint32_t ng = a.n_groups - g0 < kFTile ? a.n_groups - g0 : kFTile;
        const uint32_t ng16 = (ng + 15u) & ~15u;
        const TileStage s(smem, st, stage_bytes, H);
        mbar_wait(&bar.done[st], ph);  // every lane waits: the barrier's completion orders the consumers' writes
        for (uint32_t j = lane; j < (no_stores ? 0u : n_out); j += 32) {
            const TileRow row = j < 4u * H + 2u ? tile_row(c, s, j, hint, H, g0, ng16)
                                                : TileRow{s.committed, a.commit_out + g0, ng16 * 8u};
            tma_store_1d(row.hbm, row.smem, row.bytes);
        }
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // shared memory has been read
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar.empty[st]);
    }
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // all stores have landed
}

// A record that is not on a kernel's fast path (Snapshot state, a REJECT / hostile value, a peer slot outside the
// hint): the literal apply_one against the shared-memory cell, or against HBM for a slot the tile does not stage.
// kFmt, recs, n, i: where apply_one finds a REJECT's next_probe_index hint and request_snapshot (k_apply.cuh) --
// behind position i of the packed records (1), or handed in as n and i (2, compact streams).
template <int kFmt>
__device__ __forceinline__ uint32_t tile_general_apply(const Columns &c, const RecRegs &rec, const void *recs, uint64_t n,
                                                       uint64_t i, uint32_t gl, uint32_t hint, const TileStage &t,
                                                       uint32_t *local) {
    constexpr uint32_t R64 = kFRow64 / 8;
    const uint32_t slot = static_cast<uint32_t>(rec.w0 >> 32) & 0xffu;
    if (slot < kSlots && ((hint >> slot) & 1u)) {
        const uint32_t r = __popc(hint & ((1u << slot) - 1u));
        CellRegs cd;
        cd.meta = t.meta[gl];
        cd.matched = t.matched[r * R64 + gl];
        cd.next_idx = t.next[r * R64 + gl];
        cd.flags = t.flags[r * kFRow8 + gl];
        cd.peer_committed = t.pc[r * R64 + gl];
        const CellPtrs sp{&t.matched[r * R64 + gl], &t.next[r * R64 + gl], &t.pc[r * R64 + gl], &t.li[gl],
                          &t.flags[r * kFRow8 + gl]};
        return apply_one<kFmt>(c, recs, n, i, rec, cd, sp, local);
    }
    CellRegs cd = load_cell(c, rec);
    cd.meta = t.meta[gl];
    CellPtrs gp = global_cell_ptrs(c, rec);
    gp.last_index = &t.li[gl];
    return apply_one<kFmt>(c, recs, n, i, rec, cd, gp, local);
}

// Raft::maybe_commit (raft.rs:893-904) for group g = g0 + gl of a tile from its staged rows, by thread gl of the
// consumer group (all of them call it: the advanced bitmap is published per warp).
template <bool kSimple5>
__device__ __forceinline__ void tile_commit(const Columns &c, const TileStage &s, uint32_t gl, uint32_t g, uint32_t ng,
                                            uint32_t hint, uint32_t lane, uint32_t *adv_bitmap, uint32_t *local) {
    constexpr uint32_t R64 = kFRow64 / 8;
    const bool active = gl < ng;
    bool advanced = false;
    if (active) {
        const uint32_t meta = s.meta[gl];
        uint64_t v[kSlots];
        uint32_t r = 0;
#pragma unroll
        for (int s2 = 0; s2 < kSlots; s2++) {
            v[s2] = 0;
            if ((hint >> s2) & 1u) {
                v[s2] = s.matched[r * R64 + gl];
                r++;
            }
        }
        uint64_t mci;
        bool use_gc;
        eval_mci<kSimple5>(c, g, meta, v, hint, mci, use_gc);
        advanced = mci > s.committed[gl] && mci >= s.ts[gl] && mci <= s.li[gl];  // raft_log.rs:488
        if (advanced) {
            s.committed[gl] = mci;  // (the store warp copies the row to commit_out too)
            if (meta & RAFTGPU_META_HAS_SELF) {  // raft.rs:896-900
                const uint32_t self = RAFTGPU_META_SELF(meta);
                uint64_t *pc = ((hint >> self) & 1u) ? &s.pc[__popc(hint & ((1u << self) - 1u)) * R64 + gl]
                                                     : &c.peer_committed[static_cast<size_t>(self) * c.cap + g];
                if (mci > *pc) *pc = mci;
            }
        }
    }
    uint32_t lc[2] = {0, 0};
    publish_tile(adv_bitmap, g, lane, active, advanced, lc);
    local[5] += lc[0];
    local[6] += lc[1];
}

// Hand the stage to the store warp: the consumers' generic writes -> async proxy (fence), the whole consumer group
// done (named barrier), then one arrive on the stage's `done` barrier.
__device__ __forceinline__ void tile_handoff(uint64_t *done_bar, int bar_id, uint32_t tid) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    named_bar_sync(bar_id, kFTile);
    if (tid == 0) mbar_arrive(done_bar);
}

// RAFTGPU_TILE_DEBUG=1: thread 0 of a consumer group adds the intervals between its stamps t[0..3] and now to
// dbg[0..3] (what each kernel's phases are: at its stamps) and counts the tile in dbg[4].
__device__ __forceinline__ void tile_debug(unsigned long long *dbg, uint32_t tid, const long long (&clk)[4]) {
    if (dbg && tid == 0) {
        const long long now = clock64();
        atomicAdd(&dbg[0], static_cast<unsigned long long>(clk[1] - clk[0]));
        atomicAdd(&dbg[1], static_cast<unsigned long long>(clk[2] - clk[1]));
        atomicAdd(&dbg[2], static_cast<unsigned long long>(clk[3] - clk[2]));
        atomicAdd(&dbg[3], static_cast<unsigned long long>(now - clk[3]));
        atomicAdd(&dbg[4], 1ull);
    }
}

// Every thread's tallies: records, updates, rejects, decrements, no_progress | recomputes, advanced.
__device__ __forceinline__ void tile_flush(const uint32_t (&local)[7], const FusedArgs &a) {
    const int which[7] = {kCntRecords, kCntUpdates, kCntRejects, kCntDecrements, kCntNoProgress, kCntRecomputes, kCntAdvanced};
    block_flush_counts<7>(local, which, a.counters, nullptr);
    if (a.step_advanced) {
        const uint32_t w = __reduce_add_sync(0xffffffffu, local[6]);
        if ((threadIdx.x & 31) == 0 && w) atomicAdd(a.step_advanced, w);
    }
}

template <bool kSimple5>
__global__ void __launch_bounds__(kFTile *kFGroups + 64, 1) step_tile_kernel(Columns c, TileArgs a) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ __align__(8) TileBarriers bar;
    __shared__ uint32_t s_defer[32][kFDefer];                 // per warp: tile-relative indexes of its rare-path records
    __shared__ uint32_t s_ndefer[32];

    const uint32_t hint = kSimple5 ? 0x1fu : (a.hint & 0xffu);
    const uint32_t H = kSimple5 ? 5u : static_cast<uint32_t>(__popc(hint));
    const uint32_t stage_bytes = tile_stage_bytes(H);
    const uint32_t n_tiles = (a.n_groups + kFTile - 1) / kFTile;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    tile_init_barriers(bar, a.n_stages);

    uint32_t local[7] = {0, 0, 0, 0, 0, 0, 0};  // records, updates, rejects, decrements, no_progress | recomputes, advanced
    if (warp == kFGroups * kFTile / 32 + 1) {
        tile_store_warp(c, a, smem, stage_bytes, hint, H, (a.skip & 4u) != 0, bar);
    } else if (warp == kFGroups * kFTile / 32) {
        tile_load_warp(c, a, smem, stage_bytes, hint, H, bar, nullptr);
    } else {
        // ===================== consumers: group cg takes every kFGroups-th tile of this CTA =====================
        const uint32_t cg = warp / (kFTile / 32);
        const uint32_t tid = threadIdx.x - cg * kFTile;
        const int bar_id = 1 + static_cast<int>(cg);
        constexpr uint32_t R64 = kFRow64 / 8;  // row stride in u64 elements
        uint32_t it = 0;
        const uint32_t first_tile = blockIdx.x + cg * gridDim.x, tile_step = kFGroups * gridDim.x;
        uint32_t nx_beg = first_tile < n_tiles ? a.tile_off[first_tile] : 0u, nx_end = first_tile < n_tiles ? a.tile_off[first_tile + 1] : 0u;
        it = cg;
        for (uint32_t tile = first_tile; tile < n_tiles; tile += tile_step, it += kFGroups) {

            const int st = it % a.n_stages;
            const uint32_t ph = (it / a.n_stages) & 1u;
            const uint32_t g0 = tile * kFTile;
            const uint32_t ng = a.n_groups - g0 < kFTile ? a.n_groups - g0 : kFTile;
            const uint32_t rbeg = nx_beg, rend = nx_end;
            if (tile + tile_step < n_tiles) {  // next tile of this consumer group: fetched during this one
                nx_beg = a.tile_off[tile + tile_step];
                nx_end = a.tile_off[tile + tile_step + 1];
            }
            const uint32_t cnt = rend - rbeg;
            const TileStage s(smem, st, stage_bytes, H);
            const ulonglong2 *g_recs = reinterpret_cast<const ulonglong2 *>(a.recs + rbeg);
            // this thread's first record is requested BEFORE the wait for the stage (its address does
            // not depend on it); the loop then fetches one record ahead.  (Two ahead measured 11 % SLOWER -- 83.5 vs
            // 75.0 us, scripts/micro_tile.py: the kernel sits at its 72-register ceiling and the consumers are bound by
            // issue latency, not by the record reads.)
            ulonglong2 q_next = make_ulonglong2(kPkExt, 0ull);
            if (tid < cnt) q_next = g_recs[tid];
            long long clk[4] = {0, 0, 0, 0};
            if (a.dbg && tid == 0) clk[0] = clock64();
            wait_stage(&bar.full[st], &bar.done[st], ph);
            if (a.dbg && tid == 0) clk[1] = clock64();

            // ---- A: the tile's records against the shared-memory rows (raft.rs:1663-1743)
            // Records are read straight from HBM / L2: the stage holds rows only, which buys a fifth stage (staging
            // the records too measured equal, DESIGN 3.4); the records of a tile were prefetched into L2 while the
            // previous tile was processed, and the loop fetches each record one iteration ahead.
            auto rec_at = [&](uint32_t j) -> ulonglong2 {
                return j < cnt ? g_recs[j] : make_ulonglong2(kPkExt, 0ull);
            };
            // The main loop handles the records that make up ~98 % of the traffic -- an accept or a leader-local
            // record for a staged cell of a peer in Replicate or Probe state -- straight on the packed words and the
            // shared-memory cell.  Whatever else turns up (a rejection, a WIDE commit, a Snapshot-state peer, a learner
            // outside the hint, a record that is not this tile's) is put on the WARP's deferred list and handled after
            // the loop with all the warp's lanes working on such records at once, instead of one lane at a time
            // inside the loop (half of all warp-iterations contain a rejection): a wave has at most one record per
            // cell, so the order between the two passes does not matter.
            uint32_t *my_defer = s_defer[warp];
            if (lane == 0) s_ndefer[warp] = 0;
            __syncwarp();
            // A record the straight-line form does not take: a rejection without a snapshot request on a staged
            // Replicate / Probe cell directly (maybe_decr_to, progress.rs:168-206), the rest through apply_one.
            auto slow_record = [&](const uint32_t k) {
                const ulonglong2 q = rec_at(k);
                const uint64_t w0 = q.x;
                const uint32_t slot = static_cast<uint32_t>(w0 >> 32) & 7u;
                const uint32_t g = static_cast<uint32_t>(w0);
                const uint32_t gl = g - g0;
                if (!(w0 & kPkWide) && (w0 & kPkReject) && gl < ng && ((hint >> slot) & 1u)) {
                    const uint32_t r = kSimple5 ? slot : static_cast<uint32_t>(__popc(hint & ((1u << slot) - 1u)));
                    const uint32_t ci = r * R64 + gl;
                    const uint32_t f0 = s.flags[r * kFRow8 + gl];
                    const uint32_t state = f0 & RAFTGPU_PF_STATE_MASK;
                    const bool present = kSimple5 || (((RAFTGPU_META_IN(s.meta[gl]) | RAFTGPU_META_OUT(s.meta[gl]) |
                                                        RAFTGPU_META_LEARN(s.meta[gl])) >> slot) & 1u);
                    if (present && state != RAFTGPU_STATE_SNAPSHOT) {
                        // its EXT payloads: [kind 1 hint] [kind 2 snapshot request]
                        uint64_t hint_idx = 0;
                        bool snapshot_req = false;
                        const ulonglong2 e1 = rec_at(k + 1);   // (past the end: a padding EXT of kind 0)
                        const ulonglong2 e2 = rec_at(k + 2);
                        const bool x1 = (e1.x & kPkExt) != 0, x2 = x1 && (e2.x & kPkExt) != 0;
                        if (x1 && (e1.x >> 40) == 1) hint_idx = e1.y;
                        if ((x1 && (e1.x >> 40) == 2) || (x2 && (e2.x >> 40) == 2)) snapshot_req = true;
                        if (!snapshot_req) {
                            const uint64_t index = q.y;
                            const uint32_t delta = static_cast<uint32_t>(w0 >> 40);
                            uint64_t m = s.matched[ci], nx = s.next[ci];
                            const uint64_t nx0 = nx;
                            uint32_t f = f0 | RAFTGPU_PF_RECENT_ACTIVE, res = 0;         // raft.rs:1674
                            local[0]++;
                            local[2]++;
                            const uint64_t commit = index - delta;
                            if (commit > s.pc[ci]) s.pc[ci] = commit;                   // raft.rs:1677
                            bool ok;
                            if (state == RAFTGPU_STATE_REPLICATE) {
                                ok = index > m;                                          // :173-177 stale otherwise
                                if (ok) nx = m + 1;                                      // :178-179
                            } else if (nx == 0 || nx - 1 != index) {
                                ok = false;                                              // :188-192 stale
                            } else {
                                nx = umin64(index, hint_idx + 1);                        // :195-199
                                if (nx < 1) nx = 1;
                                f &= ~RAFTGPU_PF_PAUSED;                                 // :204
                                ok = true;
                            }
                            if (ok) {
                                local[3]++;
                                res = RAFTGPU_RES_OK | RAFTGPU_RES_SEND;
                                if (state == RAFTGPU_STATE_REPLICATE) {                  // raft.rs:1716-1718 become_probe
                                    f = (f & ~(RAFTGPU_PF_PAUSED | RAFTGPU_PF_INS_FULL | RAFTGPU_PF_STATE_MASK)) | RAFTGPU_STATE_PROBE;
                                    c.pending_snapshot[static_cast<size_t>(slot) * c.cap + g] = 0;
                                    nx = m + 1;
                                }
                            }
                            if (nx != nx0) s.next[ci] = nx;
                            if (f != f0) s.flags[r * kFRow8 + gl] = static_cast<uint8_t>(f);
                            if (a.results) a.results[rbeg + k] = static_cast<uint8_t>(res);
                            return;
                        }
                    }
                }
                // General path.
                const PackedRec *base = a.recs + rbeg;
                const RecRegs rec = load_rec<true>(base, k, cnt);
                uint32_t res = 0;
                if (!((rec.w0 >> 40) & RAFTGPU_REC_EXT)) {
                    const uint32_t gl2 = static_cast<uint32_t>(rec.w0) - g0;
                    if (gl2 >= ng) {  // not this tile's group: the batch is not in group order / bad index
                        local[0]++;
                        local[4]++;
                        res = RAFTGPU_RES_NO_PROGRESS;
                    } else {
                        res = tile_general_apply<1>(c, rec, base, cnt, k, gl2, hint, s, local);
                    }
                }
                if (a.results) a.results[rbeg + k] = static_cast<uint8_t>(res);
            };
            for (uint32_t k = tid; k < ((a.skip & 1u) ? 0u : cnt); k += kFTile) {
                const ulonglong2 q = q_next;
                q_next = rec_at(k + kFTile);
                const uint64_t w0 = q.x;
                if (w0 & kPkExt) {
                    if (a.results) a.results[rbeg + k] = 0;
                    continue;
                }
                const uint32_t slot = static_cast<uint32_t>(w0 >> 32) & 7u;
                const uint32_t g = static_cast<uint32_t>(w0);
                const uint32_t gl = g - g0;
                bool done = false;
                if (!(w0 & (kPkWide | kPkReject)) && gl < ng && ((hint >> slot) & 1u)) {
                    const uint32_t r = kSimple5 ? slot : static_cast<uint32_t>(__popc(hint & ((1u << slot) - 1u)));
                    const uint32_t ci = r * R64 + gl;
                    const uint32_t f0 = s.flags[r * kFRow8 + gl];
                    const uint32_t state = f0 & RAFTGPU_PF_STATE_MASK;
                    const bool present = kSimple5 || (((RAFTGPU_META_IN(s.meta[gl]) | RAFTGPU_META_OUT(s.meta[gl]) |
                                                        RAFTGPU_META_LEARN(s.meta[gl])) >> slot) & 1u);
                    if (present && state != RAFTGPU_STATE_SNAPSHOT) {
                        // accept / leader-local: maybe_update (progress.rs:138-150), shared by the accept path
                        // (raft.rs:1674-1677, 1724-1730) and the leader-local path (raft.rs:974-991, 1010-1014);
                        // only an accept looks at is_paused() and may move a probing peer to Replicate.
                        const uint64_t index = q.y;
                        const uint32_t delta = static_cast<uint32_t>(w0 >> 40);
                        const bool is_local = (w0 & kPkLocal) != 0;
                        const uint64_t m = s.matched[ci], nx = s.next[ci], pcv = s.pc[ci];
                        local[0]++;
                        if (is_local && delta != kPkNoCommit) s.li[gl] = index + delta;   // raft.rs:974-991
                        const uint64_t commit = index - delta;
                        if (!is_local && commit > pcv) s.pc[ci] = commit;                 // raft.rs:1677
                        const bool probe = state == RAFTGPU_STATE_PROBE;
                        const bool need = m < index;
                        const bool old_paused = !is_local && (f0 & (probe ? RAFTGPU_PF_PAUSED : RAFTGPU_PF_INS_FULL)) != 0;
                        const bool trans = need && !is_local && probe;                    // raft.rs:1730 become_replicate
                        uint32_t f = is_local ? f0 : (f0 | RAFTGPU_PF_RECENT_ACTIVE);     // raft.rs:1674
                        if (need) f &= ~RAFTGPU_PF_PAUSED;
                        if (trans)
                            f = (f & ~(RAFTGPU_PF_PAUSED | RAFTGPU_PF_INS_FULL | RAFTGPU_PF_STATE_MASK)) | RAFTGPU_STATE_REPLICATE;
                        uint64_t nnx = nx < index + 1 ? index + 1 : nx;
                        if (trans) {
                            nnx = index + 1;                                              // next_idx = matched + 1
                            c.pending_snapshot[static_cast<size_t>(slot) * c.cap + g] = 0;
                        }
                        local[1] += need ? 1u : 0u;
                        if (need) s.matched[ci] = index;
                        if (nnx != nx) s.next[ci] = nnx;
                        if (f != f0) s.flags[r * kFRow8 + gl] = static_cast<uint8_t>(f);
                        if (a.results)
                            a.results[rbeg + k] = static_cast<uint8_t>(need ? (RAFTGPU_RES_OK | (old_paused ? RAFTGPU_RES_OLD_PAUSED : 0u)) : 0u);
                        done = true;
                    }
                }
                if (!done) {   // the rare kinds: onto the warp's list, handled after the loop by all its lanes together
                    const uint32_t at = atomicAdd(&s_ndefer[warp], 1u);
                    if (at < kFDefer)
                        my_defer[at] = k;
                    else
                        slow_record(k);  // the list is full: here and now (correct, only slower)
                }
            }
            __syncwarp();
            {
                const uint32_t nd = s_ndefer[warp] < kFDefer ? s_ndefer[warp] : kFDefer;
                for (uint32_t j = lane; j < nd; j += 32) slow_record(my_defer[j]);
            }
            named_bar_sync(bar_id, kFTile);
            if (a.dbg && tid == 0) clk[2] = clock64();

            // ---- B: Raft::maybe_commit for the tile's groups
            if (!(a.skip & 2u)) tile_commit<kSimple5>(c, s, tid, g0 + tid, ng, hint, lane, a.adv_bitmap, local);

            // ---- C: hand the stage to the store warp, then the next tile's record range -> L2 (one line = 8 records)
            tile_handoff(&bar.done[st], bar_id, tid);
            if (a.dbg && tid == 0) clk[3] = clock64();
            if (tile + tile_step < n_tiles) {
                const uint32_t nn = nx_end - nx_beg;
                for (uint32_t k = tid * 8u; k < nn; k += kFTile * 8u) prefetch_l2(a.recs + nx_beg + k);
            }
            // dbg: waiting for the TMA loads, A: records, B: recompute (+ fence, barrier), C: stores + drain
            tile_debug(a.dbg, tid, clk);
        }
    }
    tile_flush(local, a);
}
