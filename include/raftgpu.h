/*
 * raftgpu.h -- C-ABI boundary of the B200 batched multi-raft commit-index engine.
 *
 * raft-rs (pingcap/raft-rs, crate `raft` 0.6.0 @ 7c21f8d) has no FFI/plugin
 * interface for this path: the boundary is the Rust method surface of
 * ProgressTracker / Progress / quorum::{MajorityConfig,JointConfig} /
 * RaftLog::maybe_commit / Raft::maybe_commit.  Each entry point below names the
 * reference interface (file:line, relative to the reference checkout) it
 * replaces; the Rust-side binding a maintainer would add is in INTEGRATION.md.
 *
 * Conventions
 *  - plain C: pointers and sizes only, no C++/torch types;
 *  - every function returns an int32_t status (RAFTGPU_OK or a negative
 *    RAFTGPU_ERR_*); nothing throws or aborts across the boundary.  The hot-path
 *    functions of the reference are infallible (they return bool / tuples);
 *    the codes here cover misuse and CUDA failures, plus the two places the
 *    reference itself errors: StepPeerNotFound (raw_node.rs:402-411) and the
 *    `fatal!` in RaftLog::commit_to (raft_log.rs:291-298);
 *  - there is NO CPU fallback: without a CUDA device every compute entry point
 *    returns RAFTGPU_ERR_NO_DEVICE;
 *  - `stream` parameters are a cudaStream_t passed as void* (NULL = the arena's
 *    own compute stream);
 *  - threading follows the reference (raw_node.rs:284 "RawNode is a
 *    thread-unsafe Node", raft.rs:292-294 `Raft: Send`): calls that touch ONE
 *    group may run concurrently for DIFFERENT groups; raftgpu_step* and the
 *    arena lifecycle calls need exclusive access.
 *
 * Data layout in HBM (struct-of-arrays, see DESIGN.md): per-peer columns are
 * [RAFTGPU_SLOTS][cap] u64 / u8, per-group columns are [cap]; a "group" is one
 * raft group (one ProgressTracker), a "peer slot" one Progress of that group.
 */
#ifndef RAFTGPU_H
#define RAFTGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RAFTGPU_ABI_VERSION 1
#define RAFTGPU_SLOTS 8 /* peer slots per group (voters + learners, both halves of a joint config) */

/* ---- status codes ------------------------------------------------------- */
#define RAFTGPU_OK 0
#define RAFTGPU_ERR_INVALID (-1)        /* bad argument */
#define RAFTGPU_ERR_CUDA (-2)           /* CUDA runtime error; see raftgpu_last_error */
#define RAFTGPU_ERR_NOMEM (-3)          /* host / device allocation failed, or arena full */
#define RAFTGPU_ERR_NO_DEVICE (-4)      /* no CUDA device: there is no CPU fallback */
#define RAFTGPU_ERR_RANGE (-5)          /* group / peer slot out of range or not allocated */
#define RAFTGPU_ERR_FULL (-6)           /* staging ring full: call raftgpu_step first */
#define RAFTGPU_ERR_PEER_NOT_FOUND (-7) /* Error::StepPeerNotFound, raw_node.rs:402-411 */
#define RAFTGPU_ERR_COMMIT_RANGE (-8)   /* RaftLog::commit_to fatal!, raft_log.rs:291-298 */
#define RAFTGPU_ERR_BUSY (-9)           /* a step is still in flight on this buffer */
/* A group would need more peer slots than it has: 8 (RAFTGPU_SLOTS) for an ordinary group, 16 for a wide one
 * (raftgpu_group_alloc_wide).  Peers = voters of both halves of a joint configuration + learners + learners_next
 * (tracker.rs:37-92).  The reference has no limit (majority.rs:86-93 sorts any number of voters on the heap); 16
 * covers two disjoint 7-voter sets in a joint change plus learners.  Beyond that the caller keeps the group on the
 * stock ProgressTracker (arena groups are independent). */
#define RAFTGPU_ERR_TOO_MANY_PEERS (-10)

const char *raftgpu_strerror(int32_t status);
uint32_t raftgpu_abi_version(void);

/* ---- constants shared with the reference -------------------------------- */
/* ProgressState, src/tracker/state.rs:22-29 */
#define RAFTGPU_STATE_PROBE 0
#define RAFTGPU_STATE_REPLICATE 1
#define RAFTGPU_STATE_SNAPSHOT 2
/* INVALID_INDEX, src/raft.rs:81 */
#define RAFTGPU_INVALID_INDEX 0ull
/* VoteResult, src/quorum.rs:12-20 (declaration order) */
#define RAFTGPU_VOTE_PENDING 0
#define RAFTGPU_VOTE_LOST 1
#define RAFTGPU_VOTE_WON 2
/* "not a leader": no index is of the current term */
#define RAFTGPU_NO_TERM_START UINT64_MAX

/* per-peer flag byte (column RAFTGPU_COL_PFLAGS) */
#define RAFTGPU_PF_STATE_MASK 0x03u
#define RAFTGPU_PF_PAUSED 0x04u        /* Progress::paused, progress.rs:24 */
#define RAFTGPU_PF_RECENT_ACTIVE 0x08u /* Progress::recent_active, progress.rs:41 */
#define RAFTGPU_PF_INS_FULL 0x10u      /* Inflights::full(), inflights.rs:54-56: reported by the host, or (with
                                          raftgpu_arena_enable_inflights) kept by the device */

/* per-group meta word (column RAFTGPU_COL_META): the tracker::Configuration
 * (tracker.rs:37-92) as bit masks over peer slots. */
#define RAFTGPU_META_IN(m) ((m) & 0xffu)            /* voters.incoming, joint.rs:13 */
#define RAFTGPU_META_OUT(m) (((m) >> 8) & 0xffu)    /* voters.outgoing, joint.rs:14 */
#define RAFTGPU_META_LEARN(m) (((m) >> 16) & 0xffu) /* learners | learners_next */
#define RAFTGPU_META_SELF(m) (((m) >> 24) & 0x7u)   /* slot of Raft::id */
#define RAFTGPU_META_HAS_SELF 0x08000000u
#define RAFTGPU_META_GROUP_COMMIT 0x10000000u       /* ProgressTracker::group_commit, tracker.rs:207 */
/* A WIDE group (raftgpu_group_alloc_wide: up to 16 peers) occupies two consecutive group slots: `g` (even) holds
 * peers 0..7 and carries WIDE_LO, `g + 1` holds peers 8..15 and carries WIDE_HI.  Each half's masks describe its own
 * eight peers; quorum / votes / commit are evaluated once, on the low half, over both. */
#define RAFTGPU_META_WIDE_LO 0x20000000u
#define RAFTGPU_META_WIDE_HI 0x40000000u

/* ---- plain data types --------------------------------------------------- */
typedef struct raftgpu_arena raftgpu_arena; /* opaque; owns all device + pinned memory */

/* One Progress (src/tracker/progress.rs:8-56) minus `ins` (Inflights stays host-side). */
typedef struct {
    uint64_t matched;                  /* progress.rs:10 */
    uint64_t next_idx;                 /* progress.rs:12 */
    uint64_t pending_snapshot;         /* progress.rs:31 */
    uint64_t pending_request_snapshot; /* progress.rs:35 */
    uint64_t commit_group_id;          /* progress.rs:52 */
    uint64_t committed_index;          /* progress.rs:55 */
    uint8_t state;                     /* progress.rs:22 */
    uint8_t paused;                    /* progress.rs:25 */
    uint8_t recent_active;             /* progress.rs:41 */
    uint8_t ins_full;                  /* Inflights::full() as last reported by the host */
    uint8_t present;                   /* 1 when the slot holds a Progress */
    uint8_t reserved[3];
} raftgpu_progress;

/* Per-group log / commit bookkeeping: the part of RaftLog (raft_log.rs:33-59)
 * RaftLog::maybe_commit needs, in range form (DESIGN.md "term test"). */
typedef struct {
    uint32_t meta;
    uint32_t reserved;
    uint64_t committed;  /* RaftLog::committed, raft_log.rs:45 */
    uint64_t term_start; /* first index whose entry carries the leader's current term */
    uint64_t last_index; /* RaftLog::last_index() */
} raftgpu_group_state;

/* One MsgAppendResponse as handle_append_response consumes it (raft.rs:1559-1775,
 * eraftpb.proto:71-92): 24 bytes.  A REJECT record is followed by ONE EXT record
 * with the same group/peer_slot whose `index` is next_probe_index (m.reject_hint,
 * or find_conflict_by_term(..).0 when m.log_term > 0 -- that lookup needs the
 * leader's log and is done by the caller, raft.rs:1560-1661) and whose `commit`
 * is m.request_snapshot. */
typedef struct {
    uint32_t group;     /* group slot */
    uint8_t peer_slot;  /* slot of m.from */
    uint8_t flags;      /* RAFTGPU_REC_* */
    uint16_t reserved;
    uint64_t index;     /* m.index */
    uint64_t commit;    /* m.commit */
} raftgpu_append_resp;
#define RAFTGPU_REC_REJECT 0x01u /* m.reject */
/* Leader-local record (not a message): `commit`, when non-zero, is the new
 * last_index after Raft::append_entry (raft.rs:974-991); `index` is the newly
 * persisted index of Raft::on_persist_entries (raft.rs:994-1016), which runs
 * prs[self].maybe_update(index); peer_slot is the leader's own slot. */
#define RAFTGPU_REC_LOCAL 0x02u
#define RAFTGPU_REC_EXT 0x80u    /* extension record of the preceding REJECT */
/* A MsgHeartbeatResponse (raft.rs:1777-1819): `commit` = m.commit, `index` unused.  Only
 * raftgpu_heartbeat_resp[_device] takes such records; the append-response paths ignore them. */
#define RAFTGPU_REC_HEARTBEAT 0x04u

/* The packed 16-byte wire form of a record (raftgpu_pack_records); layout in DESIGN.md 2. */
typedef struct {
    uint64_t w0, w1;
} raftgpu_packed_rec;

/* per-record result byte */
#define RAFTGPU_RES_OK 0x01u          /* maybe_update / maybe_decr_to returned true */
#define RAFTGPU_RES_OLD_PAUSED 0x02u  /* pr.is_paused() before maybe_update, raft.rs:1724 */
#define RAFTGPU_RES_NO_PROGRESS 0x04u /* prs.get_mut(m.from) == None, raft.rs:1663-1673 */
#define RAFTGPU_RES_SEND 0x08u        /* reject path reached self.send_append(m.from), raft.rs:1719 */

/* column ids for bulk IO */
enum {
    RAFTGPU_COL_MATCHED = 0,              /* u64 [SLOTS][cap] */
    RAFTGPU_COL_NEXT_IDX = 1,             /* u64 [SLOTS][cap] */
    RAFTGPU_COL_PEER_COMMITTED = 2,       /* u64 [SLOTS][cap]  Progress::committed_index */
    RAFTGPU_COL_PENDING_SNAPSHOT = 3,     /* u64 [SLOTS][cap] */
    RAFTGPU_COL_PENDING_REQ_SNAPSHOT = 4, /* u64 [SLOTS][cap] */
    RAFTGPU_COL_COMMIT_GROUP_ID = 5,      /* u64 [SLOTS][cap] */
    RAFTGPU_COL_PFLAGS = 6,               /* u8  [SLOTS][cap] */
    RAFTGPU_COL_VOTES = 7,                /* u8  [SLOTS][cap]  0 missing, 1 no, 2 yes */
    RAFTGPU_COL_META = 8,                 /* u32 [cap] */
    RAFTGPU_COL_COMMITTED = 9,            /* u64 [cap] */
    RAFTGPU_COL_TERM_START = 10,          /* u64 [cap] */
    RAFTGPU_COL_LAST_INDEX = 11,          /* u64 [cap] */
    RAFTGPU_COL_TERM = 12,                /* u64 [cap]  Raft::term (raft.rs:227), 0 = unknown; only the wire path reads it */
    RAFTGPU_COL_INS_META = 13,            /* u32 [SLOTS][cap]  Inflights start | count << 16 (raftgpu_arena_enable_inflights) */
    RAFTGPU_COL__COUNT = 14
};

typedef struct {
    uint32_t abi_version;
    int32_t device;
    uint32_t cap;          /* max groups */
    uint32_t slots;        /* RAFTGPU_SLOTS */
    uint32_t n_alloc;      /* groups currently allocated */
    uint32_t hi;           /* allocated groups live in [0, hi) */
    uint32_t sm_count;
    uint32_t reserved;
    uint64_t l2_bytes;
    uint64_t device_bytes; /* HBM held by this arena */
    uint64_t pinned_bytes;
} raftgpu_info;

/* monotonically increasing device-side counters (what the multi-GPU run gathers) */
typedef struct {
    uint64_t recomputes;      /* per-group Raft::maybe_commit evaluations */
    uint64_t advanced;        /* of which advanced `committed` */
    uint64_t records;         /* AppendResponse records applied */
    uint64_t updates;         /* maybe_update returned true */
    uint64_t rejects;         /* reject records seen */
    uint64_t decrements;      /* maybe_decr_to returned true */
    uint64_t no_progress;     /* records for an unknown responder */
    uint64_t votes_tallied;   /* per-group vote_result evaluations */
} raftgpu_counters;

typedef struct {
    uint64_t n_records;  /* records submitted in this step (EXT records included) */
    uint32_t n_waves;    /* kernel waves the records were split into (see raftgpu_enqueue_append_resp) */
    uint32_t n_groups;   /* groups recomputed */
    uint64_t n_advanced; /* groups whose committed index advanced */
    uint64_t h2d_bytes;  /* bytes DMAed host -> device for this step (packed staging records) */
    uint64_t d2h_bytes;  /* bytes DMAed device -> host (advanced bitmap, commit indexes, results) */
    uint64_t n_duplicates; /* zero-copy steps: records dropped because their cell already had one */
} raftgpu_step_result;

/* ---- arena lifecycle ---------------------------------------------------- */

/* ProgressTracker::with_capacity (tracker.rs:217-236) for `max_groups` trackers
 * at once: allocates every column in HBM plus the pinned staging buffers.
 * slots_per_group must be RAFTGPU_SLOTS (8): the unit of the arena is the 8-slot group, and a group that needs up
 * to 16 peers takes two of them (raftgpu_group_alloc_wide); any other value is RAFTGPU_ERR_TOO_MANY_PEERS.  ring_records = capacity of each of
 * the `n_rings` host staging rings (0 = default). */
int32_t raftgpu_arena_create(int32_t device, uint32_t max_groups, uint32_t slots_per_group,
                             uint32_t n_rings, uint32_t ring_records, raftgpu_arena **out);
int32_t raftgpu_arena_destroy(raftgpu_arena *arena);
int32_t raftgpu_arena_info(const raftgpu_arena *arena, raftgpu_info *out);
/* Last CUDA / argument error text for this arena (never NULL). */
const char *raftgpu_last_error(const raftgpu_arena *arena);

/* ---- group lifecycle (control plane; synchronous, small copies) --------- */

/* Raft::new (raft.rs:318-400) / drop: one slot per ProgressTracker. */
int32_t raftgpu_group_alloc(raftgpu_arena *arena, uint32_t *out_group);
int32_t raftgpu_group_alloc_range(raftgpu_arena *arena, uint32_t n, uint32_t *out_first);
/* A WIDE group: up to 16 peer slots (a joint configuration of large voter sets with learners; the reference has no
 * limit, majority.rs:86-93).  It occupies two consecutive group slots: *out_group (even) and *out_group + 1.  Every
 * single-group call takes the group id with peer slots 0..15 and 16-bit masks; in RECORDS (and send-list entries,
 * wire frames, column IO) peer 8 + s of wide group g is addressed as (group g + 1, slot s) -- the per-cell paths do
 * not know about wide groups at all.  Quorum, votes and Raft::maybe_commit are evaluated once, on the low half, over
 * both halves' peers; the advanced bit and the commit index are the low half's.  While an arena holds wide groups its
 * steps run through the scatter + recompute kernels (the fused tile kernel evaluates 8-slot groups); a 17th peer is
 * RAFTGPU_ERR_TOO_MANY_PEERS. */
int32_t raftgpu_group_alloc_wide(raftgpu_arena *arena, uint32_t *out_group);
int32_t raftgpu_group_free(raftgpu_arena *arena, uint32_t group);

/* ProgressTracker::apply_conf (tracker.rs:380-397) / confchange::restore
 * (confchange/restore.rs:91-107): replace the Configuration.  Slots that become
 * present get Progress::new(next_idx, ..) with recent_active = true
 * (tracker.rs:385-390); slots that disappear are removed (tracker.rs:392-394). */
int32_t raftgpu_group_set_conf(raftgpu_arena *arena, uint32_t group, uint32_t incoming_mask,
                               uint32_t outgoing_mask, uint32_t learner_mask, int32_t self_slot,
                               uint64_t next_idx);

/* Raft::reset (raft.rs:942-971) followed by become_leader's bookkeeping
 * (raft.rs:1162-1203): every Progress is reset(last_index + 1); the self slot
 * gets matched = persisted, committed_index = committed (raft.rs:964-970).
 * term_start = RAFTGPU_NO_TERM_START for a non-leader. */
int32_t raftgpu_group_reset(raftgpu_arena *arena, uint32_t group, uint64_t term_start,
                            uint64_t last_index, uint64_t committed, uint64_t persisted);

/* The tracker side of Raft::become_leader (raft.rs:1162-1203), after
 * raftgpu_group_reset: prs[self].become_replicate() (raft.rs:1180), then the
 * empty entry of the new term is appended (raft.rs:1192), so last_index += 1 and
 * term_start = that index. */
int32_t raftgpu_group_become_leader(raftgpu_arena *arena, uint32_t group);

/* Raft::append_entry (raft.rs:974-991): the log grew; entries of the current
 * term are [term_start, last_index]. */
int32_t raftgpu_group_set_log_bounds(raftgpu_arena *arena, uint32_t group, uint64_t term_start,
                                     uint64_t last_index);
/* RaftLog::commit_to (raft_log.rs:286-300): never decreases; RAFTGPU_ERR_COMMIT_RANGE
 * where the reference `fatal!`s (to_commit > last_index). */
int32_t raftgpu_group_commit_to(raftgpu_arena *arena, uint32_t group, uint64_t to_commit);
int32_t raftgpu_group_get(raftgpu_arena *arena, uint32_t group, raftgpu_group_state *out);

/* ProgressTracker::get / get_mut (tracker.rs:267-275): Progress has pub fields,
 * so the Rust shim reads a copy and writes it back. */
int32_t raftgpu_progress_get(raftgpu_arena *arena, uint32_t group, uint32_t peer_slot,
                             raftgpu_progress *out);
int32_t raftgpu_progress_set(raftgpu_arena *arena, uint32_t group, uint32_t peer_slot,
                             const raftgpu_progress *in);

/* Any single method of Progress (src/tracker/progress.rs:75-243) on one peer, executed on the
 * device columns; a0..a2 are the method's arguments, *out_result its bool (or -1 where the
 * reference panics: update_state in Snapshot).  This is what the host mirror's ProgressRef
 * calls; batches of maybe_update / maybe_decr_to go through raftgpu_enqueue_* instead. */
enum {
    RAFTGPU_POP_MAYBE_UPDATE = 0,         /* (n)                                  progress.rs:138-150 */
    RAFTGPU_POP_MAYBE_DECR_TO = 1,        /* (rejected, match_hint, request_snapshot)     :168-206 */
    RAFTGPU_POP_UPDATE_COMMITTED = 2,     /* (committed_index)                            :153-157 */
    RAFTGPU_POP_OPTIMISTIC_UPDATE = 3,    /* (n)                                          :160-163 */
    RAFTGPU_POP_BECOME_PROBE = 4,         /*                                              :95-107  */
    RAFTGPU_POP_BECOME_REPLICATE = 5,     /*                                              :110-114 */
    RAFTGPU_POP_BECOME_SNAPSHOT = 6,      /* (snapshot_idx)                               :117-121 */
    RAFTGPU_POP_SNAPSHOT_FAILURE = 7,     /*                                              :124-127 */
    RAFTGPU_POP_MAYBE_SNAPSHOT_ABORT = 8, /*                                              :131-134 */
    RAFTGPU_POP_IS_PAUSED = 9,            /*                                              :210-216 */
    RAFTGPU_POP_RESUME = 10,              /*                                              :219-222 */
    RAFTGPU_POP_PAUSE = 11,               /*                                              :225-228 */
    RAFTGPU_POP_UPDATE_STATE = 12,        /* (last)                                       :231-243 */
    RAFTGPU_POP_RESET = 13,               /* (next_idx)                                   :82-92   */
    /* Inflights (src/tracker/inflights.rs) of the peer's window, arenas with raftgpu_arena_enable_inflights only
     * (*out_result = -3 otherwise) */
    RAFTGPU_POP_INS_ADD = 14,             /* (inflight); -1 where the reference panics    inflights.rs:65-82 */
    RAFTGPU_POP_INS_FREE_TO = 15,         /* (to)                                         :85-110  */
    RAFTGPU_POP_INS_FREE_FIRST_ONE = 16,  /*                                              :113-116 */
    RAFTGPU_POP_INS_RESET = 17,           /*                                              :119-123 */
    RAFTGPU_POP_INS_FULL = 18             /*                                              :54-56   */
};
int32_t raftgpu_progress_op(raftgpu_arena *arena, uint32_t group, uint32_t peer_slot, int32_t op,
                            uint64_t a0, uint64_t a1, uint64_t a2, int32_t *out_result);

/* ProgressTracker::has_quorum (tracker.rs:367-372) for a set of peer slots, and
 * quorum_recently_active (tracker.rs:346-361; clears recent_active like the reference). */
int32_t raftgpu_has_quorum(raftgpu_arena *arena, uint32_t group, uint32_t slot_mask, int32_t *out);
int32_t raftgpu_quorum_recently_active(raftgpu_arena *arena, uint32_t group, uint32_t perspective_of_slot,
                                       int32_t *out);

/* RaftLog::maybe_commit(max_index, term) (raft_log.rs:487-499) for term == the leader's
 * current term, i.e. the range test on [term_start, last_index]. */
int32_t raftgpu_group_maybe_commit_to(raftgpu_arena *arena, uint32_t group, uint64_t max_index,
                                      int32_t *out_advanced);

/* ProgressTracker::enable_group_commit (tracker.rs:238-241) and
 * Raft::assign_commit_groups / clear_commit_group (raft.rs:531-552). */
int32_t raftgpu_set_group_commit(raftgpu_arena *arena, uint32_t group, int32_t enable);
int32_t raftgpu_assign_commit_group(raftgpu_arena *arena, uint32_t group, uint32_t peer_slot,
                                    uint64_t commit_group_id);

/* Bulk column IO for [first_group, first_group + n) of one column (peer_slot is
 * ignored for per-group columns): restoring / inspecting many groups at once. */
int32_t raftgpu_column_write(raftgpu_arena *arena, int32_t column, uint32_t peer_slot,
                             uint32_t first_group, uint32_t n, const void *host_src);
int32_t raftgpu_column_read(raftgpu_arena *arena, int32_t column, uint32_t peer_slot,
                            uint32_t first_group, uint32_t n, void *host_dst);

/* ---- the hot path ------------------------------------------------------- */

/* ProgressTracker::maximal_committed_index (tracker.rs:294-298) for one group:
 * JointConfig::committed_index (joint.rs:47-51) over MajorityConfig::committed_index
 * (majority.rs:70-124).  Runs the batched kernel on a 1-group range. */
int32_t raftgpu_maximal_committed_index(raftgpu_arena *arena, uint32_t group, uint64_t *out_index,
                                        int32_t *out_use_group_commit);

/* Raft::maybe_commit (raft.rs:893-904) for one group: maximal_committed_index ->
 * RaftLog::maybe_commit (raft_log.rs:487-499) -> prs[self].update_committed. */
int32_t raftgpu_maybe_commit(raftgpu_arena *arena, uint32_t group, int32_t *out_advanced,
                             uint64_t *out_committed);

/* Batched Raft::maybe_commit over groups [first, first + n): ONE kernel pass.
 * Asynchronous on `stream`.  d_adv_bitmap (device, u32 words indexed by
 * group >> 5 from group 0; may be NULL) gets bit g set iff group g advanced;
 * d_commit_out (device u64 [cap], may be NULL) gets the new committed index of
 * advanced groups (entries of other groups are unspecified: the fused step kernels
 * copy every group's commit index there, this pass only the advanced ones); d_mci_out / d_gc_out (may be NULL) get maximal_committed_index
 * for every group. */
int32_t raftgpu_recompute(raftgpu_arena *arena, void *stream, uint32_t first, uint32_t n,
                          uint32_t *d_adv_bitmap, uint64_t *d_commit_out, uint64_t *d_mci_out,
                          uint8_t *d_gc_out);

/* Batched handle_append_response prefix (raft.rs:1663-1743: recent_active,
 * update_committed, maybe_decr_to | maybe_update + state transition) over `n`
 * records ALREADY IN HBM.  Precondition: at most one non-EXT record per
 * (group, peer_slot) in the range -- one "wave"; raftgpu_enqueue_append_resp
 * builds waves for arbitrary streams.  d_results (device, n bytes) may be NULL.
 * Asynchronous on `stream`. */
int32_t raftgpu_apply_device(raftgpu_arena *arena, void *stream,
                             const raftgpu_append_resp *d_records, uint64_t n, uint8_t *d_results);

/* Same, for records that are already in the packed 16-byte wire form (raftgpu_pack_records,
 * the format the staging path ships over PCIe) in HBM: a third less record traffic. */
int32_t raftgpu_apply_device_packed(raftgpu_arena *arena, void *stream, const void *d_packed_records,
                                    uint64_t n_packed, uint8_t *d_results);

/* The FUSED step for batches in group order: apply + recompute in one kernel whose HBM traffic is
 * all dense bulk transfers (DESIGN.md 3.4).  d_packed_records are packed records in
 * non-decreasing group order (EXT payloads directly behind their record); d_tile_off[t] is the
 * index of the first record whose group is >= t * RAFTGPU_TILE_GROUPS, for t = 0..n_tiles
 * (raftgpu_tile_index builds and validates it on the host).  One wave per call, like
 * raftgpu_apply_device; processes all allocated groups [0, hi).  A record found outside its tile
 * is not applied and reported as RAFTGPU_RES_NO_PROGRESS.  Asynchronous on `stream`. */
#define RAFTGPU_TILE_GROUPS 256
uint32_t raftgpu_tile_groups(void); /* RAFTGPU_TILE_GROUPS, as the library sees it */
int32_t raftgpu_step_sorted_device(raftgpu_arena *arena, void *stream, const void *d_packed_records,
                                   uint64_t n_packed, const uint32_t *d_tile_off, uint8_t *d_results,
                                   uint32_t *d_adv_bitmap, uint64_t *d_commit_out);
/* Host helper: out[t] for t = 0..n_tiles where n_tiles = ceil(n_groups / RAFTGPU_TILE_GROUPS)
 * (out has n_tiles + 1 entries).  RAFTGPU_ERR_INVALID if the records are not in group order,
 * RAFTGPU_ERR_RANGE if one names a group >= n_groups (no tile would visit it). */
int32_t raftgpu_tile_index(const raftgpu_packed_rec *packed, uint64_t n_packed, uint32_t n_groups,
                           uint32_t *out, uint64_t out_capacity);

/* Stage host records for the next step (RawNode::step -> Raft::step ->
 * handle_append_response, raw_node.rs:402-411 / raft.rs:1559).  Records for one
 * (group, peer) keep their arrival order: a second record for a cell that
 * already has one in the pending step is placed in a later wave.  `ring`
 * selects one of the arena's staging rings; different threads use different
 * rings (and, as in the reference, different groups). */
int32_t raftgpu_enqueue_append_resp(raftgpu_arena *arena, uint32_t ring,
                                    const raftgpu_append_resp *records, uint64_t n);

/* Bulk form of the above for a caller that already holds a whole batch in host memory:
 * the library splits it over its own staging threads (pinned to the GPU-local CPUs; count
 * from RAFTGPU_HOST_THREADS, default 16, at most the arena's ring count), one ring each.
 * The records of one (group, peer) cell keep their arrival order when the group's records are contiguous in
 * the batch (what a ready loop produces); a cell whose records are scattered through an unordered batch
 * belongs on one ring through raftgpu_enqueue_append_resp.
 * RAFTGPU_BULK_SORTED: the caller promises records are in non-decreasing group order, which
 * lets the threads skip atomics on the per-cell bookkeeping; the order is verified and
 * RAFTGPU_ERR_INVALID returned (nothing is applied; call raftgpu_step to discard) if not. */
#define RAFTGPU_BULK_SORTED 0x1u
int32_t raftgpu_enqueue_bulk(raftgpu_arena *arena, const raftgpu_append_resp *records, uint64_t n,
                             uint32_t flags);

/* ---- zero-copy submission ---------------------------------------------------
 * For callers that build their batch directly in DMA-able memory: raftgpu_host_alloc returns
 * pinned memory on the GPU-local NUMA node, raftgpu_pack_records converts public records to
 * the 16-byte packed wire form (a REJECT and its EXT become 2-3 packed records; returns the
 * packed count), and raftgpu_step_begin_packed ships such a buffer with no staging copy:
 * H2D straight from the caller's buffer, ONE apply wave, the recompute pass, D2H of the
 * results.  The one-record-per-(group, peer) precondition cannot be checked on the host
 * without reading the batch, so the GPU checks it: a duplicate is not applied, counted in
 * raftgpu_step_result.n_duplicates, and raftgpu_step_wait returns RAFTGPU_ERR_INVALID.
 * The buffer must stay untouched until that step's raftgpu_step_wait returns. */
int32_t raftgpu_host_alloc(raftgpu_arena *arena, uint64_t bytes, void **out_pinned);
int32_t raftgpu_host_free(raftgpu_arena *arena, void *pinned);
int32_t raftgpu_pack_records(const raftgpu_append_resp *records, uint64_t n, raftgpu_packed_rec *out,
                             uint64_t out_capacity, uint64_t *out_n);
int32_t raftgpu_step_begin_packed(raftgpu_arena *arena, const raftgpu_packed_rec *pinned_records,
                                  uint64_t n_packed, uint32_t flags);

/* ---- compact stream (the narrow wire form) -------------------------------------
 * PCIe is the end-to-end bottleneck of a step (DESIGN.md 5), so the bytes per record are the
 * end-to-end cost.  The compact stream carries a batch as 4-byte units instead of 16-byte
 * packed records: the records of one group (consecutive in the input, as a multi-raft ready
 * loop produces them) form a RUN
 *      [HDR_A][HDR_B] rec rec rec ...          (at most 8 units after the header)
 * whose header names the group and a 48-bit base index, and each record is a slot, a 14-bit
 * index delta above the base and an 8-bit commit delta:
 *      unit & 3 == 0  REC    [2] LOCAL  [3,6) back  [6,9) peer slot  [9] REJECT  [10,24) index - base
 *                            [24,32) message: index - commit; LOCAL: commit - index (255 = none)
 *                            (the run's header sits at unit positions i-back-2 and i-back-1; a
 *                            REJECT is followed by a payload unit with its next_probe_index hint)
 *      unit & 3 == 1  HDR_A  [2,32) base bits [0,30)
 *      unit & 3 == 2  HDR_B  [2,14) group - g_base[block of HDR_A]   [14,32) base bits [30,48)
 *      unit & 3 == 3  ESC    [2,32) < 0x1fffffff: index into the side table; == 0x1fffffff: padding;
 *                            bit 31 set: the payload of the REJECT in front, [2,31) = hint - index (signed)
 * g_base[] holds one group id per block of RAFTGPU_COMPACT_BLOCK units.  Whatever does not fit
 * (a REJECT that asks for a snapshot, an index more than 8192 away from the run's first, a commit
 * delta above 254, a base above 2^48, a group more than 4095 above its block's g_base, flag bits
 * the format does not know) is an ESC unit pointing at the full 24-byte public record (and its
 * EXT) in the side table -- the format is lossless for ANY input, only less compact for hostile
 * ones.  A 5-peer round is ~22 bytes per group instead of ~57.  The blob is position
 * independent: header, g_base[], units[] (padded to 16 bytes), side[].
 * Same contract as raftgpu_step_begin_packed: pinned buffer (raftgpu_host_alloc), ONE wave
 * checked on the GPU, buffer untouched until the step's raftgpu_step_wait returns.  Result
 * bytes (RAFTGPU_STEP_READ_RESULTS) are per UNIT; raftgpu_pack_compact can report the unit
 * of every public record. */
#define RAFTGPU_COMPACT_MAGIC 0x31434752u /* "RGC1" */
#define RAFTGPU_COMPACT_BLOCK 2048u
typedef struct raftgpu_compact_hdr {
    uint32_t magic;
    uint32_t n_units;   /* 4-byte units */
    uint32_t n_blocks;  /* ceil(n_units / RAFTGPU_COMPACT_BLOCK) */
    uint32_t n_side;    /* 24-byte records in the side table */
    uint64_t n_records; /* public records represented (EXT continuations not counted) */
    uint64_t off_blocks, off_units, off_side; /* byte offsets from the start of the blob, 16-byte aligned */
    uint64_t total_bytes;
    uint32_t flags;     /* RAFTGPU_COMPACT_TILEABLE */
    uint32_t reserved;
} raftgpu_compact_hdr;
/* Set by raftgpu_pack_compact when the groups of the runs ascend and every run has a header
 * (records of one group contiguous, groups in increasing order, no group too far from its
 * block's g_base): the fused tile kernel can then take the stream -- and, because one thread
 * walks a group's records in order, such a stream may hold SEVERAL records per (group, peer). */
#define RAFTGPU_COMPACT_TILEABLE 0x1u
/* ... and no (group, peer) cell occurs twice: the fused kernel may then use one thread per unit
 * (faster than the ordered per-group walk); the kernel still verifies it. */
#define RAFTGPU_COMPACT_ONE_WAVE 0x2u
/* Upper bound of the blob size for n public records (EXT records included in n). */
uint64_t raftgpu_compact_bound(uint64_t n);
/* records[0..n) -> blob at out (out_capacity bytes; any host memory, pinned for the zero-copy
 * step).  unit_of_record: optional [n], the unit index holding record i's result byte
 * (UINT32_MAX for EXT records). */
int32_t raftgpu_pack_compact(const raftgpu_append_resp *records, uint64_t n, void *out, uint64_t out_capacity,
                             uint64_t *out_bytes, uint32_t *unit_of_record);
int32_t raftgpu_step_begin_compact(raftgpu_arena *arena, const void *pinned_blob, uint64_t blob_bytes,
                                   uint32_t flags);
/* Records in ordinary (pageable) host memory -> one step: the library's staging threads pack
 * slices of the batch into the compact stream in pinned memory (cut at group boundaries, so the
 * records of a group must be contiguous for the result to be tileable; any other order still
 * works through the scatter kernel, one record per cell), then the step is submitted like
 * raftgpu_step_begin_compact.  Nothing may have been enqueued for this step.  `records` can be
 * reused as soon as the call returns.  A batch too hostile for the compact form (every record
 * escaping to the side table) goes through raftgpu_enqueue_bulk + raftgpu_step_begin instead, and so does
 * a batch with several records per cell on an arena that cannot run the fused kernel (device-side
 * Inflights, wide groups; RAFTGPU_STEP_ASYNC is ignored on such arenas).
 * raft.rs:1663-1743 + 893-904 for a whole tick, as one call. */
int32_t raftgpu_step_begin_records(raftgpu_arena *arena, const raftgpu_append_resp *records, uint64_t n,
                                   uint32_t flags);
/* The same step for a blob that already sits in device memory (hdr = a host copy of its
 * header): raftgpu_compact_tile_index_device builds the tile table in d_tile_off -- room for
 * 3 * (ceil(n_groups / RAFTGPU_TILE_GROUPS) + 2) + 2 u32: the first unit of every tile, then each
 * tile's group-id bases -- and bumps *d_bad if the stream is not tileable after all, then
 * raftgpu_step_compact_device runs ONE fused kernel: the records of every tile applied to
 * its rows in shared memory, Raft::maybe_commit for its groups, rows stored back. */
int32_t raftgpu_compact_tile_index_device(raftgpu_arena *arena, void *stream, const void *d_blob,
                                          const raftgpu_compact_hdr *hdr, uint32_t *d_tile_off, uint32_t *d_bad);
/* flags: RAFTGPU_COMPACT_STEP_ORDERED forces the per-group walk (records of a cell applied in stream
 * order); otherwise a ONE_WAVE stream gets one thread per unit, and d_dup_count (nullable) is bumped
 * for every record that turns out to be the second one on its cell (such a record is not applied). */
#define RAFTGPU_COMPACT_STEP_ORDERED 0x1u
int32_t raftgpu_step_compact_device(raftgpu_arena *arena, void *stream, const void *d_blob,
                                    const raftgpu_compact_hdr *hdr, const uint32_t *d_tile_off, uint8_t *d_results,
                                    uint32_t *d_adv_bitmap, uint64_t *d_commit_out, uint32_t *d_dup_count,
                                    uint32_t flags);
/* Result bytes of the last completed ZERO-COPY step (packed: one per packed record, compact:
 * one per unit; 0 for EXT payloads / headers), valid until the next raftgpu_step_wait.  Needs
 * RAFTGPU_STEP_READ_RESULTS.  raft.rs:1663-1743: what handle_append_response decided per message. */
int32_t raftgpu_step_slot_results(raftgpu_arena *arena, const uint8_t **results, uint64_t *n_slots);

/* One batched step over everything enqueued: H2D of the staged records, the
 * apply kernel per wave, ONE recompute pass over all allocated groups, D2H of
 * the results.  raftgpu_step = raftgpu_step_begin + raftgpu_step_wait.  Between
 * begin and wait the caller may already enqueue the NEXT step's records, and may even
 * begin it: up to TWO steps can be in flight (three staging sets), so the H2D of step
 * j+1 overlaps the kernels and D2H of step j.  raftgpu_step_wait completes the oldest. */
#define RAFTGPU_STEP_READ_COMMITTED 0x1u /* also copy back the new committed index of advanced groups */
#define RAFTGPU_STEP_READ_RESULTS 0x2u   /* also copy back the per-record result bytes */
/* raftgpu_step_begin_records only: return as soon as the staging threads have the batch; packing, the H2D copies
 * and the kernel launches are queued by the arena's submitter thread.  `records` must then stay untouched until
 * this step's raftgpu_step_wait returns, a submission error is reported by that raftgpu_step_wait, and until
 * then the only arena calls allowed are raftgpu_step_wait and the next raftgpu_step_begin_* (which first waits
 * for the pending submission).  This overlaps ALL host work of tick j+1 with the GPU work of tick j. */
#define RAFTGPU_STEP_ASYNC 0x4u
/* raftgpu_step_begin_records only: ship the 24-byte records AS THEY ARE (one H2D straight from the caller's buffer,
 * which should be pinned: raftgpu_host_alloc) and apply them with the scatter kernel -- no host packing at all.
 * 3.7x the PCIe bytes of the compact stream, zero CPU: the better choice when the caller's CPU share is small
 * (several GPUs per socket: packing is CPU-bound, ~7 ns per record per staging thread, DESIGN.md 5/7).  Contract of
 * the zero-copy paths: at most ONE record per (group, peer) cell, verified on the GPU (a duplicate is not applied,
 * counted in n_duplicates, raftgpu_step_wait returns RAFTGPU_ERR_INVALID); `records` stays untouched until the
 * step's raftgpu_step_wait returns. */
#define RAFTGPU_STEP_RAW 0x8u
/* raftgpu_step_begin_records only, `records` in PINNED host memory (ignored otherwise, and with RAFTGPU_STEP_RAW or
 * RAFTGPU_STEP_READ_RESULTS): HYBRID staging.  Packing costs host CPU time, the raw form costs PCIe time; with few
 * staging threads per GPU (eight GPUs share the host's cores) neither alone keeps up.  The library packs the first
 * part of the batch (cut at a group boundary) into the compact stream while the DMA engine ships the rest as 24-byte
 * records straight from the caller's buffer, sized so that both finish together (model: RAFTGPU_HYBRID_PACK_NS per
 * record and thread, and RAFTGPU_HYBRID_PCIE_GBS: both measured on every step unless set; or RAFTGPU_HYBRID_PACK_PCT to fix the
 * split).  The batch must be in group order with at most ONE record per (group, peer) cell in its tail (a tick with
 * several acknowledgements per peer belongs to the plain form, whose fused kernel walks them in order); both are
 * verified on the device and a violation fails the step's raftgpu_step_wait.  The raw part goes through the scatter kernel, then the
 * fused kernel applies the packed part and recomputes every group.  `records` must stay untouched until
 * raftgpu_step_wait returns. */
#define RAFTGPU_STEP_HYBRID 0x10u
int32_t raftgpu_step_begin(raftgpu_arena *arena, uint32_t flags);
int32_t raftgpu_step_wait(raftgpu_arena *arena, raftgpu_step_result *out);
int32_t raftgpu_step(raftgpu_arena *arena, uint32_t flags, raftgpu_step_result *out);

/* Results of the last completed step, in arena-owned pinned memory, valid until
 * the next raftgpu_step_wait: adv_bitmap has bit g set iff group g advanced
 * (LightReady.commit_index, raw_node.rs:643-650); committed[g] is meaningful
 * for advanced groups when RAFTGPU_STEP_READ_COMMITTED was set. */
int32_t raftgpu_step_results(raftgpu_arena *arena, const uint32_t **adv_bitmap,
                             const uint64_t **committed);
/* Per-record result bytes (RAFTGPU_RES_*) of the last completed step for the
 * records enqueued on `ring`, in that ring's enqueue order (EXT records get 0);
 * needs RAFTGPU_STEP_READ_RESULTS.  *out_n = records enqueued on the ring; with
 * out == NULL only the count is returned. */
int32_t raftgpu_step_record_results(raftgpu_arena *arena, uint32_t ring, uint8_t *out,
                                    uint64_t out_capacity, uint64_t *out_n);

/* ---- post-commit send decisions (SURVEY 8(f) rank 2) --------------------- */

/* The step right after the path: when a group's commit index advanced the leader calls
 * bcast_append (raft.rs:1745-1748, 1012-1013 -> raft.rs:857-865), i.e. send_append for every
 * peer but itself, and maybe_send_append drops the paused ones first (raft.rs:780-788;
 * Progress::is_paused, progress.rs:210-216: Probe -> paused, Replicate -> ins.full(),
 * Snapshot -> always).  raftgpu_send_list_device turns the advanced bitmap of a step into that
 * work list -- one entry per (group, peer) the host has to build a MsgAppend for -- with a
 * stream-compaction kernel: groups [first, first+n) whose bit is set in d_adv_bitmap (NULL = every
 * group: a plain bcast_append), peers = voters and learners of the group except its own slot.
 * Entries come out in no particular order (neither does HashMap iteration in the reference).
 * *d_count = number of entries the pass produced (u64, zeroed here first); entries beyond
 * `capacity` are dropped, so count > capacity means "call again with a larger buffer". */
typedef struct raftgpu_send_entry {
    uint32_t group;
    uint8_t peer_slot;
    uint8_t flags;     /* RAFTGPU_SEND_SNAPSHOT */
    uint16_t reserved;
    uint64_t next_idx; /* Progress::next_idx: entries from here (raft.rs:799) */
} raftgpu_send_entry;
/* pending_request_snapshot != INVALID_INDEX: prepare_send_snapshot comes first (raft.rs:792-797) */
#define RAFTGPU_SEND_SNAPSHOT 0x1u
int32_t raftgpu_send_list_device(raftgpu_arena *arena, void *stream, uint32_t first, uint32_t n,
                                 const uint32_t *d_adv_bitmap, raftgpu_send_entry *d_out, uint64_t capacity,
                                 uint64_t *d_count);
/* The same for the last completed step (its advanced bitmap, all allocated groups), entries
 * copied to host memory; synchronous.  The pause flags and next_idx are read when the kernel runs:
 * call it before the NEXT step is submitted if the list has to reflect exactly this step.  RAFTGPU_ERR_FULL (with *out_n = the number needed) when
 * `capacity` is too small. */
int32_t raftgpu_step_send_list(raftgpu_arena *arena, raftgpu_send_entry *out, uint64_t capacity, uint64_t *out_n);

/* ---- heartbeat commits (SURVEY 8(f) rank 3, leader side) ------------------- */

/* bcast_heartbeat (raft.rs:875-889) calls send_heartbeat for every peer but the leader itself, and
 * send_heartbeat attaches commit = min(pr.matched, raft_log.committed) (raft.rs:826-848: the
 * leader must not forward a follower's commit past what that follower has).  One dense pass
 * over groups [first, first+n): d_out[slot * n + (g - first)] = that commit for every present
 * peer (voter or learner) other than the group's own slot, RAFTGPU_NO_HEARTBEAT elsewhere. */
#define RAFTGPU_NO_HEARTBEAT UINT64_MAX
int32_t raftgpu_heartbeat_commits_device(raftgpu_arena *arena, void *stream, uint32_t first, uint32_t n,
                                         uint64_t *d_out);

/* ---- wire decode (SURVEY 8(f) rank 4) ------------------------------------- */

/* The step from what a transport holds: serialized eraftpb.Message frames (proto/proto/eraftpb.proto:71-92;
 * the reference decodes them with rust-protobuf / prost before RawNode::step, raw_node.rs:402-411).  The host
 * appends frames and their end offsets and parses NOTHING; the GPU decodes the varints and runs the same
 * per-message prefix of handle_append_response (raft.rs:1663-1743) + Raft::maybe_commit.
 *      frame i = bytes[offsets[i], offsets[i+1]) = u32 little-endian (group << 4 | peer_slot), then the Message
 * offsets[0..n] ascend.  Per frame one status byte comes back: RAFTGPU_WIRE_* << 4 | RAFTGPU_RES_* (the latter
 * for applied frames).  Frames the device cannot decide are NOT applied and are the host's to handle: */
#define RAFTGPU_WIRE_OK 0u         /* a MsgAppendResponse, applied (low nibble: RAFTGPU_RES_*) */
#define RAFTGPU_WIRE_SKIP_TYPE 1u  /* any other MessageType: Raft::step on the host */
#define RAFTGPU_WIRE_TERM 2u       /* m.term != the group's term (raftgpu_group_set_term; 0 = not checked): Raft::step's term rules */
#define RAFTGPU_WIRE_NEEDS_LOG 3u  /* reject with log_term > 0: next_probe_index = find_conflict_by_term(..) needs the leader's
                                      log (raft.rs:1562-1661); the host computes it and submits the 24-byte REJECT + EXT records */
#define RAFTGPU_WIRE_MALFORMED 4u  /* not a protobuf message, a bad frame, or a group that is not allocated */
#define RAFTGPU_WIRE_DUP 5u        /* a later frame of a (group, peer) cell that already has one in this batch: cells are
                                      applied in arrival order, one message per step -- resubmit it with the next batch */
typedef struct raftgpu_wire_batch {
    const uint8_t *bytes;    /* the frames, back to back */
    uint64_t n_bytes;
    const uint32_t *offsets; /* [n + 1] */
    uint64_t n;              /* frames */
    /* 24-byte records that travel with the batch and are applied BEFORE the frames: the leader's own
     * RAFTGPU_REC_LOCAL events (append_entry / on_persist_entries are calls, not messages) and REJECTs whose
     * next_probe_index the host has resolved (RAFTGPU_WIRE_NEEDS_LOG of an earlier step).  At most one
     * record per (group, peer) cell, verified on the GPU like raftgpu_step_begin_packed.  May be NULL / 0. */
    const raftgpu_append_resp *records;
    uint64_t n_records;
} raftgpu_wire_batch;
/* Raft::term (raft.rs:227) of a group, for the wire path's term test; 0 (the initial value) = the caller filters. */
int32_t raftgpu_group_set_term(raftgpu_arena *arena, uint32_t group, uint64_t term);
/* Decode + apply for a batch that already sits in device memory (d_bytes 16-byte aligned, d_offsets [n + 1]);
 * d_status [n] is required.  Two kernels (scan: classify + first frame of every cell; apply), asynchronous on
 * `stream`; run raftgpu_recompute afterwards for Raft::maybe_commit. */
int32_t raftgpu_wire_apply_device(raftgpu_arena *arena, void *stream, const void *d_bytes, uint64_t n_bytes,
                                  const uint32_t *d_offsets, uint64_t n, uint8_t *d_status);
/* One step from a wire batch in host memory (pinned -- raftgpu_host_alloc -- for an asynchronous copy): H2D of
 * bytes + offsets, decode + apply, the recompute pass, D2H of the results and the status bytes.  Same
 * begin / wait protocol and result accessors as raftgpu_step_begin; the buffers must stay untouched until
 * raftgpu_step_wait returns.  raftgpu_step_wire_status: the status bytes of the last completed wire step. */
int32_t raftgpu_step_begin_wire(raftgpu_arena *arena, const raftgpu_wire_batch *batch, uint32_t flags);
int32_t raftgpu_step_wire_status(raftgpu_arena *arena, const uint8_t **status, uint64_t *n);

/* ---- heartbeat responses (SURVEY 8(f) rank 3, response side) ---------------- */

/* The tracker part of Raft::handle_heartbeat_response (raft.rs:1777-1804) for a batch of RAFTGPU_REC_HEARTBEAT
 * records: pr.update_committed(m.commit), recent_active = true, resume(), a full inflights window of a
 * Replicate peer frees its first entry (INS_FULL clears), and the result byte says whether the reference would
 * call send_append: RAFTGPU_RES_OK | RAFTGPU_RES_SEND when pr.matched < last_index or a snapshot was requested
 * (raft.rs:1800-1803); RAFTGPU_RES_NO_PROGRESS for an unknown peer.  The read-index tail (:1806-1818) is
 * raftgpu_heartbeat_resp_read (section "ReadIndex" below); this call ignores RAFTGPU_REC_READ_CTX.  A heartbeat batch is its own pass, ordered by the caller between steps (it reads last_index,
 * which a step's LOCAL records write): "all heartbeat responses of the tick after its append responses" is
 * one of the delivery orders raft allows.  One record per (group, peer) cell; a second one is not applied,
 * gets result 0 and -- in the host form -- makes the call return RAFTGPU_ERR_INVALID.
 * _device: records and results in device memory, asynchronous on `stream` (d_dup_count nullable, u32, zeroed by
 * the caller); the host form copies, runs and waits. */
int32_t raftgpu_heartbeat_resp_device(raftgpu_arena *arena, void *stream, const raftgpu_append_resp *d_records,
                                      uint64_t n, uint8_t *d_results, uint32_t *d_dup_count);
int32_t raftgpu_heartbeat_resp(raftgpu_arena *arena, const raftgpu_append_resp *records, uint64_t n, uint8_t *results);

/* Progress::update_state(last) (progress.rs:231-243) for a list of MsgAppends the host has just built -- the
 * follow-up of every send-list entry (raft.rs:753-760): a Replicate peer's next_idx jumps to last + 1
 * (optimistic_update; the matching ins.add(last) is the host's Inflights), a Probe peer is paused until its
 * next response.  entries[i].next_idx carries `last`, the index of the last entry sent to that peer.
 * results[i] (nullable): 1 done, 0xff where the reference panics (a Snapshot-state peer), RAFTGPU_RES_NO_PROGRESS. */
int32_t raftgpu_update_state_device(raftgpu_arena *arena, void *stream, const raftgpu_send_entry *d_entries, uint64_t n,
                                    uint8_t *d_results);
int32_t raftgpu_update_state(raftgpu_arena *arena, const raftgpu_send_entry *entries, uint64_t n, uint8_t *results);

/* ---- Inflights on the device (SURVEY 8(f) rank 2) --------------------------- */

/* Keep every peer's Inflights window (src/tracker/inflights.rs:19-110: the last index of each in-flight MsgAppend, a
 * ring of Config::max_inflight_msgs entries, config.rs:112) in HBM, so that nothing about flow control is left to
 * per-message host work: raftgpu_update_state adds (progress.rs:231-236), an accepted append response frees up to
 * its index (raft.rs:1742), a heartbeat response frees the first entry of a full window (raft.rs:1796-1798), every
 * state change resets (progress.rs:75-80), and RAFTGPU_PF_INS_FULL -- what Progress::is_paused reads in Replicate
 * state -- mirrors ins.full() (raftgpu_progress.ins_full is then an output only).  Call before groups are
 * allocated.  Memory: 8 slots x max_groups x max_inflight x 8 bytes (256 entries: 16 KB per group), which is why
 * it is opt-in.  With windows on, steps run through the scatter kernels (the fused tile kernels keep their rows in
 * shared memory and do not carry the rings): raftgpu_step_sorted_device / raftgpu_step_compact_device return
 * RAFTGPU_ERR_INVALID, every raftgpu_step_begin_* form works. */
int32_t raftgpu_arena_enable_inflights(raftgpu_arena *arena, uint32_t max_inflight);
/* One peer's window: *start, *count (inflights.rs:21-23) and, when buffer != NULL, its `capacity` ring entries. */
int32_t raftgpu_inflights_get(raftgpu_arena *arena, uint32_t group, uint32_t peer_slot, uint32_t *start, uint32_t *count,
                              uint64_t *buffer, uint32_t capacity);

/* ---- ReadIndex (ReadOnlyOption::Safe / LeaseBased, src/read_only.rs) -------- */

/* Keep every group's ReadOnly (read_only.rs:63-68: the queue of pending MsgReadIndex contexts, each with the commit
 * index it was taken at and its set of heartbeat acknowledgements) in HBM, so that a linearizable read costs no
 * per-follower host work.  The caller maps each context (m.entries[0].data) to a 64-bit TOKEN -- equal bytes, equal
 * token within one group's pending set -- and the engine only compares tokens (the same division of labour as the
 * slot <-> peer-id mapping).  At most `max_pending` (1..64) requests wait per group; the reference has no bound (a
 * request beyond it is RAFTGPU_READ_FULL and stays with the caller).  Call before groups are allocated.  Memory:
 * (20 * max_pending + 8) bytes per group, the request pass's scratch word included (168 MB per million groups at 8),
 * counted in raftgpu_info.device_bytes.  Enabling it routes no step to another kernel.  Every entry point of this section
 * returns RAFTGPU_ERR_INVALID on an arena without read-index queues.  The passes of one arena run one at a time. */
int32_t raftgpu_arena_enable_read_index(raftgpu_arena *arena, uint32_t max_pending);

/* One MsgReadIndex as step_leader takes it (raft.rs:2056-2091): 16 bytes.  A peer of a wide group is addressed the
 * way records address it: (group g + 1, slot s) for peer 8 + s. */
typedef struct {
    uint32_t group;
    uint8_t from_slot; /* slot of m.from (ignored with RAFTGPU_READ_LOCAL) */
    uint8_t flags;     /* RAFTGPU_READ_LOCAL | RAFTGPU_READ_LEASE */
    uint16_t reserved;
    uint64_t ctx;      /* token of m.entries[0].data */
} raftgpu_read_req;
/* m.from == INVALID_ID || m.from == self (raft.rs:2791): the answer is a local ReadState, not a MsgReadIndexResp */
#define RAFTGPU_READ_LOCAL 0x1u
/* the group runs ReadOnlyOption::LeaseBased (config.rs:117; a per-Raft option the caller knows) */
#define RAFTGPU_READ_LEASE 0x2u

/* per-request status byte of raftgpu_read_index[_device] */
#define RAFTGPU_READ_DROPPED 0u         /* !commit_to_current_term (raft.rs:2057-2061), a non-leader included */
#define RAFTGPU_READ_READY 1u           /* answered now (singleton or LeaseBased, raft.rs:2063-2069 / 2083-2088) */
#define RAFTGPU_READ_QUEUED 2u          /* ReadOnly::add_request (read_only.rs:86-99): heartbeats carry its ctx */
#define RAFTGPU_READ_ALREADY_PENDING 3u /* the token is pending already (read_only.rs:88-90): nothing added, the
                                           caller still broadcasts heartbeats with the ctx (raft.rs:2081) */
#define RAFTGPU_READ_FULL 4u            /* max_pending requests wait: not queued, the caller keeps the request */
#define RAFTGPU_READ_SPLIT 5u           /* the group's requests were not contiguous in the batch: this run is not
                                           applied (resubmit it) */
#define RAFTGPU_READ_INVALID 6u         /* a group that is not allocated, or from_slot >= 8 on a non-LOCAL request */

/* The MsgReadIndex branch of step_leader for a batch: per request, in batch order within a group, the rules above.
 * The requests of one group must be contiguous in the batch (a later run of the same group is RAFTGPU_READ_SPLIT);
 * an INVALID request ends a run.  d_status[i] = RAFTGPU_READ_*; d_index[i] (nullable) = the read index
 * (raft_log.committed) for READY and QUEUED, 0 otherwise.  Two kernels (scan: the first run of every group;
 * apply: one thread walks that run), asynchronous on `stream`.  The host form copies, runs and waits; it returns
 * RAFTGPU_ERR_INVALID when a request came back RAFTGPU_READ_SPLIT (every other request was applied). */
int32_t raftgpu_read_index_device(raftgpu_arena *arena, void *stream, const raftgpu_read_req *d_reqs, uint64_t n,
                                  uint8_t *d_status, uint64_t *d_index);
int32_t raftgpu_read_index(raftgpu_arena *arena, const raftgpu_read_req *reqs, uint64_t n, uint8_t *status,
                           uint64_t *index);

/* A flag on RAFTGPU_REC_HEARTBEAT records: the MsgHeartbeatResponse carries a non-empty context (raft.rs:1805), and
 * `index` carries its token.  Without it the read tail is skipped.  raftgpu_heartbeat_resp[_device] ignores it. */
#define RAFTGPU_REC_READ_CTX 0x08u

/* ReadOnly::recv_ack (read_only.rs:104-109) for a batch of heartbeat responses: every HEARTBEAT | READ_CTX record
 * whose peer has a Progress (raft.rs:1779-1789) adds its peer to the ack set of the pending request with that token
 * (an unknown token is ignored) and marks the request "acknowledged in this batch".  Acks form a set: a duplicate
 * record changes nothing.  One thread per record, asynchronous on `stream`. */
int32_t raftgpu_read_ack_device(raftgpu_arena *arena, void *stream, const raftgpu_append_resp *d_records, uint64_t n);

/* One released request: a ReadState (RAFTGPU_READ_LOCAL) or a MsgReadIndexResp to `to_slot` (raft.rs:2790-2806).
 * 24 bytes; to_slot of a wide group's peer 8 + s is s on group g + 1, like records. */
typedef struct {
    uint32_t group;
    uint8_t to_slot;
    uint8_t flags;     /* RAFTGPU_READ_LOCAL */
    uint16_t reserved;
    uint64_t index;    /* ReadIndexStatus::index: the commit index when the request was queued */
    uint64_t ctx;      /* the request's token */
} raftgpu_read_state;

/* ReadOnly::advance (read_only.rs:114-129) behind ProgressTracker::has_quorum (tracker.rs:367-372) for groups
 * [first, first + n): per group, the requests up to and including the LAST one that was acknowledged since the
 * previous release pass and whose ack set is a quorum of the current (joint) configuration are released -- for a
 * batch of heartbeat responses the same requests the reference releases one response at a time.  A request that
 * was not acknowledged in the batch is not released even if its set is a quorum (the reference checks only the
 * acked context).  The pass clears the "acknowledged" marks.  Released requests go to d_out as a stream compaction:
 * the states of one group are contiguous and in queue order, groups in no particular order.  d_count[0] = states
 * the pass released or wanted to, d_count[1] = states written (a prefix of d_out); d_count[0] > capacity means
 * that the groups that did not fit kept their queues and marks: call again.  Asynchronous on `stream`.
 * The host form runs over all allocated groups: *out_n = states written to `out`; RAFTGPU_ERR_FULL when groups
 * did not fit (they are released by the next call). */
int32_t raftgpu_read_release_device(raftgpu_arena *arena, void *stream, uint32_t first, uint32_t n,
                                    raftgpu_read_state *d_out, uint64_t capacity, uint64_t *d_count);
int32_t raftgpu_read_release(raftgpu_arena *arena, raftgpu_read_state *out, uint64_t capacity, uint64_t *out_n);

/* The whole of Raft::handle_heartbeat_response (raft.rs:1777-1818) for a batch: raftgpu_heartbeat_resp's tracker
 * part (result bytes into `results`, nullable), then recv_ack, then the release pass over all allocated groups
 * (states as raftgpu_read_release).  Returns RAFTGPU_ERR_FULL as raftgpu_read_release, else RAFTGPU_ERR_INVALID
 * when a (group, peer) cell had two records (as raftgpu_heartbeat_resp; the ack of the second is a no-op). */
int32_t raftgpu_heartbeat_resp_read(raftgpu_arena *arena, const raftgpu_append_resp *records, uint64_t n,
                                    uint8_t *results, raftgpu_read_state *states, uint64_t capacity,
                                    uint64_t *out_n);

/* ReadOnly::last_pending_request_ctx (read_only.rs:132-134) for groups [first, first + n): the context
 * bcast_heartbeat attaches (raft.rs:876).  d_out[g - first] = token, RAFTGPU_NO_READ_CTX when the queue is empty
 * (so token 0 can stand for the empty context).  Asynchronous on `stream`. */
#define RAFTGPU_NO_READ_CTX UINT64_MAX
int32_t raftgpu_read_index_last_ctx_device(raftgpu_arena *arena, void *stream, uint32_t first, uint32_t n,
                                           uint64_t *d_out);

/* The read tail of Raft::post_conf_change (raft.rs:2648-2664), where the reference reaches raft.rs:2650 (after
 * raftgpu_group_set_conf): the self peer acks the LAST pending request, and when its ack set is a quorum of the new
 * configuration every pending request is released into `out`.  Synchronous, one group.  RAFTGPU_ERR_FULL (nothing
 * released, *out_n = the number needed) when `capacity` is too small. */
int32_t raftgpu_group_read_index_conf_changed(raftgpu_arena *arena, uint32_t group, raftgpu_read_state *out,
                                              uint64_t capacity, uint64_t *out_n);

/* One group's queue in order, for tests and inspection: *out_n pending requests; when the arrays are non-NULL
 * (room for `capacity`), ctx[k], index[k] and word[k] of the k-th one, word = ack mask over peer slots 0..15 in bits
 * 0..15 | from slot << 16 | RAFTGPU_READ_WORD_* flags. */
#define RAFTGPU_READ_WORD_LOCAL 0x01000000u /* RAFTGPU_READ_LOCAL request */
#define RAFTGPU_READ_WORD_ACKED 0x02000000u /* acknowledged since the last release pass */
int32_t raftgpu_read_index_get(raftgpu_arena *arena, uint32_t group, uint64_t *ctx, uint64_t *index, uint32_t *word,
                               uint32_t capacity, uint32_t *out_n);

/* ---- votes (SURVEY 8(f) rank 1) ----------------------------------------- */

/* ProgressTracker::reset_votes / record_vote (tracker.rs:301-310). */
int32_t raftgpu_reset_votes(raftgpu_arena *arena, uint32_t group);
int32_t raftgpu_record_vote(raftgpu_arena *arena, uint32_t group, uint32_t peer_slot, int32_t vote);
/* Batched ProgressTracker::tally_votes (tracker.rs:313-340) over [first, first+n):
 * d_out[g] = VoteResult | granted << 8 | rejected << 16.  Asynchronous. */
int32_t raftgpu_tally_votes(raftgpu_arena *arena, void *stream, uint32_t first, uint32_t n,
                            uint32_t *d_out);
/* Single-group form (synchronous). */
int32_t raftgpu_vote_result(raftgpu_arena *arena, uint32_t group, int32_t *out_result,
                            uint32_t *out_granted, uint32_t *out_rejected);

/* ---- plumbing ------------------------------------------------------------ */
int32_t raftgpu_counters_read(raftgpu_arena *arena, raftgpu_counters *out);
int32_t raftgpu_synchronize(raftgpu_arena *arena);
/* Diagnostics: 8 u64 slots the fused kernel fills when RAFTGPU_TILE_DEBUG is set (cycle totals
 * of its phases: wait for loads, records, recompute, stores; [4] = tiles). */
int32_t raftgpu_debug_read(raftgpu_arena *arena, uint64_t *out8);
/* Device scratch owned by the arena (for callers that keep record batches in
 * HBM, e.g. the bench's device-resident leg). */
int32_t raftgpu_device_alloc(raftgpu_arena *arena, uint64_t bytes, void **out_device_ptr);
int32_t raftgpu_device_free(raftgpu_arena *arena, void *device_ptr);
int32_t raftgpu_memcpy_h2d(raftgpu_arena *arena, void *device_dst, const void *host_src,
                           uint64_t bytes);
int32_t raftgpu_memcpy_d2h(raftgpu_arena *arena, void *host_dst, const void *device_src,
                           uint64_t bytes);

#ifdef __cplusplus
}
#endif
#endif /* RAFTGPU_H */
