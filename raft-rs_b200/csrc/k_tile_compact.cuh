// k_tile_compact.cuh -- step_tile_compact_kernel (+ its tile index kernels): the fused step on the compact stream.
// Part of kernels.cuh (included there, inside namespace raftgpu; not a standalone header).

// step_tile_compact_kernel: the fused step for a TILEABLE compact stream (groups ascending, every
// run headed -- raftgpu_compact_hdr.flags & RAFTGPU_COMPACT_TILEABLE).  Everything but the record
// loop is step_tile_kernel's (k_tile.cuh): stage ring and layout, load warp (which also stages the
// tile's units behind the rows), store warp, commit phase, hand-over, general record path and counter
// flush.  The consumers work per GROUP instead of per record:
//   0. a unit-parallel pre-pass finds, for every group of the tile, the first unit of its first
//      run (shared-memory atomicMin on the run headers),
//   1. thread gl then walks the runs of group g0+gl SEQUENTIALLY -- header decoded once, each
//      record a handful of instructions against the shared-memory cells -- so the records of one
//      cell apply in stream order (no one-wave restriction) and
//   2. goes straight on to the group's Raft::maybe_commit (tile_commit): its cells were written by
//      this very thread, so no barrier separates apply and recompute.
// Against the per-record form this is ~2.5x fewer warp instructions per tile (no per-record
// header/cell address arithmetic, no three-way divergence on the record kind) and a third of the
// record bytes.  tile_off[t] = unit position of the first run header of tile t.
struct CTileArgs : FusedArgs {  // (tile_off: unit positions; results: one byte per unit)
    CompactSrc src;
    const uint2 *tile_gb;      // [n_tiles]: g_base of the unit block tile t starts in, and of the next block
    uint32_t *dup_count;       // nullable (!kOrdered): bumped for a second record on one cell, which is not applied
};

// shared memory besides the stages: one u32 run index per group per consumer group
constexpr uint32_t kCRunBytes = static_cast<uint32_t>(kFGroups) * kFTile * 4u;

// The common records -- accept, leader-local, rejection without a snapshot request -- for a peer
// in Replicate or Probe state whose cell is staged in shared memory: statement for statement the
// branches of apply_one (raft.rs:1674-1677, 1709-1730, 974-991, 1010-1014; progress.rs:95-114,
// 138-157, 168-206).  Returns false (nothing touched) when the record needs the general path.
template <bool kSimple5>
__device__ __forceinline__ bool tile_fast_apply(const Columns &c, const TileStage &t, uint32_t gl, uint32_t g, uint32_t slot,
                                                uint64_t index, uint64_t commit, bool is_local, bool is_reject,
                                                uint64_t ext_hint, uint32_t hint, uint32_t present_mask, uint32_t *local,
                                                uint32_t &res) {
    constexpr uint32_t R64 = kFRow64 / 8;
    if (!((hint >> slot) & 1u)) return false;
    const uint32_t r = kSimple5 ? slot : static_cast<uint32_t>(__popc(hint & ((1u << slot) - 1u)));
    const uint32_t ci = r * R64 + gl;
    const uint32_t f0 = t.flags[r * kFRow8 + gl];
    const uint32_t state = f0 & RAFTGPU_PF_STATE_MASK;
    if (!((present_mask >> slot) & 1u) || state == RAFTGPU_STATE_SNAPSHOT) return false;
    uint64_t m = t.matched[ci], nx = t.next[ci];
    const uint64_t m0 = m, nx0 = nx;
    uint32_t f = f0;
    local[0]++;
    if (is_local) {
        if (commit != 0) t.li[gl] = commit;
    } else {
        f |= RAFTGPU_PF_RECENT_ACTIVE;
        if (commit > t.pc[ci]) t.pc[ci] = commit;
    }
    if (is_reject) {  // maybe_decr_to without a snapshot request
        local[2]++;
        bool ok;
        if (state == RAFTGPU_STATE_REPLICATE) {
            ok = index > m;                              // progress.rs:173-177 stale otherwise
            if (ok) nx = m + 1;                          // :178-179
        } else if (nx == 0 || nx - 1 != index) {
            ok = false;                                  // :188-192 stale
        } else {
            nx = umin64(index, ext_hint + 1);            // :195-199
            if (nx < 1) nx = 1;
            f &= ~RAFTGPU_PF_PAUSED;                     // :204
            ok = true;
        }
        if (ok) {
            local[3]++;
            res = RAFTGPU_RES_OK | RAFTGPU_RES_SEND;
            if (state == RAFTGPU_STATE_REPLICATE) {      // raft.rs:1716-1718 become_probe
                f = (f & ~(RAFTGPU_PF_PAUSED | RAFTGPU_PF_INS_FULL | RAFTGPU_PF_STATE_MASK)) | RAFTGPU_STATE_PROBE;
                c.pending_snapshot[static_cast<size_t>(slot) * c.cap + g] = 0;
                nx = m + 1;
            }
        }
    } else {
        const bool old_paused = !is_local && (state == RAFTGPU_STATE_PROBE ? (f & RAFTGPU_PF_PAUSED) != 0
                                                                           : (f & RAFTGPU_PF_INS_FULL) != 0);
        const bool need = m < index;
        if (need) {
            m = index;
            f &= ~RAFTGPU_PF_PAUSED;
            local[1]++;
            res = RAFTGPU_RES_OK | (old_paused ? RAFTGPU_RES_OLD_PAUSED : 0u);
        }
        if (nx < index + 1) nx = index + 1;
        if (need && !is_local && state == RAFTGPU_STATE_PROBE) {
            f = (f & ~(RAFTGPU_PF_PAUSED | RAFTGPU_PF_INS_FULL | RAFTGPU_PF_STATE_MASK)) | RAFTGPU_STATE_REPLICATE;
            c.pending_snapshot[static_cast<size_t>(slot) * c.cap + g] = 0;
            nx = m + 1;
        }
    }
    if (m != m0) t.matched[ci] = m;
    if (nx != nx0) t.next[ci] = nx;
    if (f != f0) t.flags[r * kFRow8 + gl] = static_cast<uint8_t>(f);
    return true;
}

// kOrdered: per-group walk (records of a cell apply in stream order; any number per cell).
// !kOrdered: one thread per unit (faster; at most one record per (group, peer) cell per batch --
// checked on the fly in a shared-memory bitmap when a.dup_count is given).
template <bool kSimple5, bool kOrdered>
__global__ void __launch_bounds__(kFTile *kFGroups + 64, 1) step_tile_compact_kernel(Columns c, CTileArgs a) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ __align__(8) TileBarriers bar;

    const uint32_t hint = kSimple5 ? 0x1fu : (a.hint & 0xffu);
    const uint32_t H = kSimple5 ? 5u : static_cast<uint32_t>(__popc(hint));
    const uint32_t stage_bytes = tile_stage_bytes(H) + kCUnitCap * 4u;  // the rows, then the tile's units
    const uint32_t n_tiles = (a.n_groups + kFTile - 1) / kFTile;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t *s_run_all = reinterpret_cast<uint32_t *>(smem + static_cast<size_t>(a.n_stages) * stage_bytes);
    if (threadIdx.x < kFGroups * kFTile) s_run_all[threadIdx.x] = kOrdered ? 0xffffffffu : 0u;
    tile_init_barriers(bar, a.n_stages);

    uint32_t local[7] = {0, 0, 0, 0, 0, 0, 0};  // records, updates, rejects, decrements, no_progress | recomputes, advanced
    if (warp == kFGroups * kFTile / 32 + 1) {
        tile_store_warp(c, a, smem, stage_bytes, hint, H, false, bar);
    } else if (warp == kFGroups * kFTile / 32) {
        tile_load_warp(c, a, smem, stage_bytes, hint, H, bar, a.src.units);
    } else {
        // ===================== consumers: thread gl of group cg owns group g0 + gl of its tiles =====================
        const uint32_t cg = warp / (kFTile / 32);
        const uint32_t tid = threadIdx.x - cg * kFTile;
        const int bar_id = 1 + static_cast<int>(cg);
        uint32_t *s_run = s_run_all + cg * kFTile;
        uint32_t it = 0;
        // tile index and g_base words of this consumer group's NEXT tile are fetched during the current
        // one (tile_gb[t] = the g_base words of the two unit blocks tile t starts in)
        const uint32_t first_tile = blockIdx.x + cg * gridDim.x, tile_step = kFGroups * gridDim.x;
        uint32_t nx_u0 = 0, nx_u1 = 0;
        uint2 nx_gb = make_uint2(0u, 0u);
        if (first_tile < n_tiles) {
            nx_u0 = a.tile_off[first_tile];
            nx_u1 = a.tile_off[first_tile + 1];
            nx_gb = a.tile_gb[first_tile];
        }
        it = cg;
        for (uint32_t tile = first_tile; tile < n_tiles; tile += tile_step, it += kFGroups) {

            const int st = it % a.n_stages;
            const uint32_t ph = (it / a.n_stages) & 1u;
            const uint32_t g0 = tile * kFTile;
            const uint32_t ng = a.n_groups - g0 < kFTile ? a.n_groups - g0 : kFTile;
            const uint32_t u0 = nx_u0, u1 = nx_u1;
            const uint32_t gb0 = nx_gb.x, gb1 = nx_gb.y;
            if (tile + tile_step < n_tiles) {
                nx_u0 = a.tile_off[tile + tile_step];
                nx_u1 = a.tile_off[tile + tile_step + 1];
                nx_gb = a.tile_gb[tile + tile_step];
            }
            const uint32_t ua = u0 & ~3u;
            const uint32_t lead = u0 - ua, cnt = u1 - ua;  // local unit positions [lead, cnt)
            const uint32_t cnt4 = (cnt + 3u) & ~3u;
            const uint32_t staged = u1 > u0 ? (cnt4 < kCUnitCap ? cnt4 : kCUnitCap) : 0u;
            const TileStage t(smem, st, stage_bytes, H);
            const uint32_t *s_units = t.units;
            const uint32_t *g_units = a.src.units + ua;
            const uint32_t blk0 = ua / RAFTGPU_COMPACT_BLOCK;
            long long clk[4] = {0, 0, 0, 0};
            if (a.dbg && tid == 0) clk[0] = clock64();
            wait_stage(&bar.full[st], &bar.done[st], ph);  // (k_tile.cuh: exact although this group skips phases)
            if (a.dbg && tid == 0) clk[1] = clock64();

            // ---- 0: first run header of every group of the tile.  The g_base words of the (at most
            // two, unless the tile is crowded) unit blocks the tile spans were fetched before the wait.
            auto group_of = [&](uint32_t p, uint32_t hb) -> uint32_t {
                const uint32_t blk = (ua + p) / RAFTGPU_COMPACT_BLOCK;
                const uint32_t gb = blk == blk0 ? gb0 : (blk == blk0 + 1u ? gb1 : a.src.g_base[blk]);
                return gb + ((hb >> 2) & 0xfffu);
            };
            const uint32_t gl = tid;
            const bool active = gl < ng;
            const uint32_t g = g0 + gl;
            if constexpr (kOrdered) {
                for (uint32_t p = lead + tid; p < cnt; p += kFTile) {
                    const uint32_t u = p < staged ? s_units[p] : g_units[p];
                    const uint32_t kind = u & 3u;
                    if (kind == kCuEsc) {  // a side-table record: start pulling it towards L1 for the walk below
                        const uint32_t k = u >> 2;
                        if (k < kCuPad && k < a.src.n_side) {
                            asm volatile("prefetch.global.L1 [%0];" ::"l"(a.src.side + k));
                            asm volatile("prefetch.global.L1 [%0];" ::"l"(reinterpret_cast<const uint8_t *>(a.src.side + k) + 40));
                        }
                        continue;
                    }
                    if (kind != kCuHdrA || p + 1u >= cnt) continue;
                    const uint32_t hb = p + 1u < staged ? s_units[p + 1u] : g_units[p + 1u];
                    if ((hb & 3u) != kCuHdrB) continue;
                    const uint32_t gt = group_of(p, hb) - g0;
                    if (gt < ng) atomicMin(&s_run[gt], p);
                }
                named_bar_sync(bar_id, kFTile);
                if (a.dbg && tid == 0) clk[2] = clock64();

                // ---- 1: the runs of group g, record by record (raft.rs:1663-1743)
                uint32_t p = s_run[gl];
                s_run[gl] = 0xffffffffu;  // ready for this consumer group's next tile
                if (active && p != 0xffffffffu) {
                    const uint32_t meta = t.meta[gl];
                    const uint32_t present_mask = kSimple5 ? 0x1fu
                                                           : (RAFTGPU_META_IN(meta) | RAFTGPU_META_OUT(meta) | RAFTGPU_META_LEARN(meta));
                    uint64_t base = 0;
                    while (p < cnt) {
                        const uint32_t u = p < staged ? s_units[p] : g_units[p];
                        const uint32_t kind = u & 3u;
                        if (kind == kCuHdrA) {  // a run header: ours (the first, or a continuation) or the next group's
                            if (p + 1u >= cnt) break;
                            const uint32_t hb = p + 1u < staged ? s_units[p + 1u] : g_units[p + 1u];
                            if ((hb & 3u) != kCuHdrB) break;
                            if (group_of(p, hb) != g) break;
                            base = static_cast<uint64_t>(u >> 2) | (static_cast<uint64_t>(hb >> 14) << 30);
                            p += 2u;
                            continue;
                        }
                        if (kind == kCuHdrB) break;  // malformed
                        uint32_t res = 0;
                        RecRegs rec;
                        uint64_t ext_hint = 0, ext_snapshot = RAFTGPU_INVALID_INDEX;
                        bool general = false;
                        uint32_t step = 1;
                        if (kind == kCuRec) {
                            const uint32_t slot = (u >> 6) & 7u;
                            const uint64_t index = base + ((u >> 10) & 0x3fffu);
                            const uint32_t cd = u >> 24;
                            const bool is_local = (u & kCuLocal) != 0;
                            const bool is_reject = (u & kCuReject) != 0;
                            const uint64_t commit = is_local ? (cd == kCuNoCommit ? 0 : index + cd) : (index >= cd ? index - cd : 0);
                            if (is_reject && p + 1u < cnt) {  // its hint rides in the next unit
                                const uint32_t pl = p + 1u < staged ? s_units[p + 1u] : g_units[p + 1u];
                                if ((pl & 3u) == kCuEsc && ((pl >> 2) & kCuPayload)) {
                                    ext_hint = compact_hint(index, pl);
                                    step = 2;
                                }
                            }
                            const bool fast = tile_fast_apply<kSimple5>(c, t, gl, g, slot, index, commit, is_local, is_reject, ext_hint,
                                                                        hint, present_mask, local, res);
                            if (!fast) {
                                general = true;
                                rec.w0 = static_cast<uint64_t>(g) | (static_cast<uint64_t>(slot) << 32) |
                                         (static_cast<uint64_t>(is_reject ? RAFTGPU_REC_REJECT : (is_local ? RAFTGPU_REC_LOCAL : 0u)) << 40);
                                rec.index = index;
                                rec.commit = commit;
                            }
                        } else {  // ESC: the full record sits in the side table (a stray payload unit: nothing)
                            const uint32_t k = u >> 2;
                            if (k == kCuPad) break;  // padding only ever follows the last run of a slice
                            if (k < kCuPad && k < a.src.n_side) {
                                const uint64_t *sp = reinterpret_cast<const uint64_t *>(a.src.side + k);
                                rec.w0 = sp[0];
                                rec.index = sp[1];
                                rec.commit = sp[2];
                                if ((rec.w0 >> 40) & RAFTGPU_REC_EXT) {
                                    // a continuation by itself carries nothing
                                } else if (static_cast<uint32_t>(rec.w0) != g) {  // not this run's group: the stream lied
                                    local[0]++;
                                    local[4]++;
                                    res = RAFTGPU_RES_NO_PROGRESS;
                                } else {
                                    general = true;
                                    if ((rec.w0 >> 40) & RAFTGPU_REC_REJECT)
                                        load_reject_ext<false>(a.src.side, k, a.src.n_side, ext_hint, ext_snapshot);
                                }
                            }
                        }
                        if (general) res = tile_general_apply<2>(c, rec, nullptr, ext_hint, ext_snapshot, gl, hint, t, local);
                        if (a.results) a.results[ua + p] = static_cast<uint8_t>(res);
                        p += step;
                    }
                }
            } else {
                // ---- 1': one thread per unit; a record finds its run header `back` units behind it
                uint32_t *s_touch = s_run;  // 2048 bits: (group, peer slot) cells seen in this tile
                for (uint32_t k = lead + tid; k < cnt; k += kFTile) {
                    const uint32_t u = k < staged ? s_units[k] : g_units[k];
                    const uint32_t kind = u & 3u;
                    if (kind == kCuHdrA || kind == kCuHdrB) continue;
                    uint32_t res = 0, gt = 0, slot = 0;
                    RecRegs rec;
                    uint64_t ext_hint = 0, ext_snapshot = RAFTGPU_INVALID_INDEX;
                    bool general = false, fast_ok = false, is_local = false, is_reject = false;
                    if (kind == kCuRec) {
                        const uint32_t back = (u >> 3) & 7u;
                        if (k < lead + back + 2u) continue;  // malformed
                        const uint32_t hp = k - back - 2u;
                        const uint32_t ha = hp < staged ? s_units[hp] : g_units[hp];
                        const uint32_t hb = hp + 1u < staged ? s_units[hp + 1u] : g_units[hp + 1u];
                        if ((ha & 3u) != kCuHdrA || (hb & 3u) != kCuHdrB) continue;
                        gt = group_of(hp, hb) - g0;
                        slot = (u >> 6) & 7u;
                        rec.index = (static_cast<uint64_t>(ha >> 2) | (static_cast<uint64_t>(hb >> 14) << 30)) + ((u >> 10) & 0x3fffu);
                        const uint32_t cd = u >> 24;
                        is_local = (u & kCuLocal) != 0;
                        is_reject = (u & kCuReject) != 0;
                        rec.commit = is_local ? (cd == kCuNoCommit ? 0 : rec.index + cd) : (rec.index >= cd ? rec.index - cd : 0);
                        if (is_reject && k + 1u < cnt) {  // its hint rides in the next unit
                            const uint32_t pl = k + 1u < staged ? s_units[k + 1u] : g_units[k + 1u];
                            if ((pl & 3u) == kCuEsc && ((pl >> 2) & kCuPayload)) ext_hint = compact_hint(rec.index, pl);
                        }
                        rec.w0 = static_cast<uint64_t>(g0 + gt) | (static_cast<uint64_t>(slot) << 32) |
                                 (static_cast<uint64_t>(is_reject ? RAFTGPU_REC_REJECT : (is_local ? RAFTGPU_REC_LOCAL : 0u)) << 40);
                        fast_ok = true;
                    } else {  // ESC: the full record sits in the side table (payload units / padding: nothing)
                        const uint32_t k2 = u >> 2;
                        if (k2 >= kCuPad || k2 >= a.src.n_side) continue;
                        const uint64_t *sp = reinterpret_cast<const uint64_t *>(a.src.side + k2);
                        rec.w0 = sp[0];
                        rec.index = sp[1];
                        rec.commit = sp[2];
                        if ((rec.w0 >> 40) & RAFTGPU_REC_EXT) continue;  // a continuation by itself carries nothing
                        gt = static_cast<uint32_t>(rec.w0) - g0;
                        slot = static_cast<uint32_t>(rec.w0 >> 32) & 0xffu;
                        if ((rec.w0 >> 40) & RAFTGPU_REC_REJECT)
                            load_reject_ext<false>(a.src.side, k2, a.src.n_side, ext_hint, ext_snapshot);
                    }
                    if (gt >= ng) {  // not this tile's group: the stream lied
                        local[0]++;
                        local[4]++;
                        res = RAFTGPU_RES_NO_PROGRESS;
                    } else {
                        bool dup = false;
                        if (a.dup_count && slot < kSlots) {
                            const uint32_t bit = 1u << (8u * (gt & 3u) + slot);
                            dup = (atomicOr(&s_touch[gt >> 2], bit) & bit) != 0;
                            if (dup) atomicAdd(a.dup_count, 1u);
                        }
                        if (!dup) {
                            const uint32_t present_mask =
                                kSimple5 ? 0x1fu
                                         : (RAFTGPU_META_IN(t.meta[gt]) | RAFTGPU_META_OUT(t.meta[gt]) | RAFTGPU_META_LEARN(t.meta[gt]));
                            general = !(fast_ok && tile_fast_apply<kSimple5>(c, t, gt, g0 + gt, slot, rec.index, rec.commit, is_local,
                                                                             is_reject, ext_hint, hint, present_mask, local, res));
                            if (general) res = tile_general_apply<2>(c, rec, nullptr, ext_hint, ext_snapshot, gt, hint, t, local);
                        }
                    }
                    if (a.results) a.results[ua + k] = static_cast<uint8_t>(res);
                }
                named_bar_sync(bar_id, kFTile);
                if (a.dup_count && tid < kFTile / 4) s_touch[tid] = 0;  // clean for this consumer group's next tile
                if (a.dbg && tid == 0) clk[2] = clock64();
            }
            __syncwarp();
            if (a.dbg && tid == 0) clk[3] = clock64();

            // ---- 2: Raft::maybe_commit for this thread's group, 3: hand the stage to the store warp
            tile_commit<kSimple5>(c, t, gl, g, ng, hint, lane, a.adv_bitmap, local);
            tile_handoff(&bar.done[st], bar_id, tid);
            // dbg: waiting for the TMA loads, 0: run index, 1: records, 2 + 3: recompute, fence, barrier
            tile_debug(a.dbg, tid, clk);
        }
    }
    tile_flush(local, a);
}

// Tile index of a tileable compact stream, on the device (the zero-copy step has no host pass
// over the units): tile_off[t] = position of the first run header whose group is >= t * kFTile.
// One thread per unit; a header finds the previous run's group by looking back over at most one
// run (2 + 8 units).  *bad is bumped when groups do not ascend or an ESC unit has no run.
__global__ void __launch_bounds__(256)
compact_tile_index_kernel(CompactSrc src, uint32_t n_groups, uint32_t *__restrict__ tile_off, uint32_t *__restrict__ bad) {
    const uint32_t n_tiles = (n_groups + kFTile - 1) / kFTile;
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < src.n_units; i += stride) {
        const uint32_t u = src.units[i];
        if ((u & 3u) == kCuEsc && (u >> 2) < kCuPad) {  // a side-table record must sit inside a run
            bool headed = false;
            for (uint32_t b = 1; b <= 8u && b <= i; b++) {
                const uint32_t k = src.units[i - b] & 3u;
                if (k == kCuHdrB) {
                    headed = true;
                    break;
                }
            }
            if (!headed) atomicAdd(bad, 1u);
            continue;
        }
        if ((u & 3u) != kCuHdrA || i + 1 >= src.n_units) continue;
        const uint32_t hb = src.units[i + 1];
        if ((hb & 3u) != kCuHdrB) continue;
        const uint32_t g = src.g_base[i / RAFTGPU_COMPACT_BLOCK] + ((hb >> 2) & 0xfffu);
        // previous run header, if any: at most one run (2 + 8 units) back, not counting the padding
        // that fills a staging slice up to its block boundary (raftgpu_step_begin_records)
        bool have_prev = false;
        uint32_t gp = 0;
        for (uint32_t b = 2, real = 0; b <= i && real <= 10u; b++) {
            const uint32_t ua = src.units[i - b];
            if (ua == (kCuEsc | (kCuPad << 2))) continue;
            real++;
            if ((ua & 3u) == kCuHdrA && (src.units[i - b + 1] & 3u) == kCuHdrB) {
                gp = src.g_base[(i - b) / RAFTGPU_COMPACT_BLOCK] + ((src.units[i - b + 1] >> 2) & 0xfffu);
                have_prev = true;
                break;
            }
        }
        if (!have_prev) {  // the first run of the stream: everything before it must be padding
            for (uint32_t b = 1; b <= i && b <= 12u; b++)
                if (src.units[i - b] != (kCuEsc | (kCuPad << 2))) {
                    atomicAdd(bad, 1u);
                    break;
                }
        }
        if (have_prev && gp > g) atomicAdd(bad, 1u);       // groups must ascend
        if (g >= n_groups) {
            atomicAdd(bad, 1u);
            continue;
        }
        const uint32_t t_hi = g / kFTile;
        const uint32_t t_lo = have_prev ? (gp / kFTile) + 1u : 0u;  // tiles (prev tile, this tile] start here
        if (!have_prev || gp / kFTile != t_hi)
            for (uint32_t t2 = t_lo; t2 <= t_hi; t2++) tile_off[t2] = i;
    }
    // tiles behind the last run are filled by the host-side launch (tile_off pre-set to n_units)
    (void)n_tiles;
}

// tile_gb[t] = the g_base words of the unit block tile t's (16-byte aligned) first unit lies in and of
// the block after it, so that the fused kernel decodes group ids without dependent global loads.
__global__ void __launch_bounds__(256)
compact_tile_gb_kernel(CompactSrc src, uint32_t n_tiles, const uint32_t *__restrict__ tile_off, uint2 *__restrict__ tile_gb) {
    const uint32_t n_blk = (src.n_units + RAFTGPU_COMPACT_BLOCK - 1) / RAFTGPU_COMPACT_BLOCK;
    for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < n_tiles; t += gridDim.x * blockDim.x) {
        const uint32_t blk0 = (tile_off[t] & ~3u) / RAFTGPU_COMPACT_BLOCK;
        tile_gb[t] = make_uint2(blk0 < n_blk ? src.g_base[blk0] : 0u, blk0 + 1u < n_blk ? src.g_base[blk0 + 1u] : 0u);
    }
}
