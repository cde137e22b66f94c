// arena.cu -- host side of the engine: the HBM arena, staging rings, streams and
// the extern "C" surface declared in include/raftgpu.h.
//
// The arena owns every byte of device and pinned memory.  There is no CPU
// compute path: without a CUDA device arena creation fails with
// RAFTGPU_ERR_NO_DEVICE and nothing else can be called.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <thread>
#include <cctype>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <new>
#include <string>
#include <unordered_map>
#include <vector>

#include <sched.h>
#if defined(__x86_64__)
#include <immintrin.h>
#endif

#include "kernels.cuh"
#include "pack_compact.h"

using namespace raftgpu;

namespace {

constexpr int kNumSets = 3;        // staging sets: one filling, up to two steps in flight
constexpr uint32_t kChunk = 2048;  // records per staging chunk (48 KiB)

// A record moved to a later wave: its packed form (1..4 PackedRec) plus where its result goes.
struct OverflowRec {
    PackedRec pk[4];
    int n_pk;
    uint32_t ring;
    uint64_t seq;  // position of the (main) record in the ring's enqueue order
};

// One caller thread's staging ring: a list of chunks of the set's shared pinned
// buffer.  Only its owner thread touches it between steps.
struct Ring {
    std::vector<uint32_t> chunks;        // chunk indices, in fill order
    uint32_t fill = kChunk;              // records used in the last chunk (kChunk = need a new one)
    uint64_t seq = 0;                    // records enqueued on this ring (wave 0 + overflow)
    std::vector<uint64_t> overflow_seq;  // seq numbers that went to a later wave (ascending)
};

struct StagingSet {
    // host (pinned)
    PackedRec *h_recs = nullptr;      // [n_chunks][kChunk] packed wave-0 records, shared by all rings
    PackedRec *h_overflow = nullptr;  // later waves, laid out at submit time
    uint32_t *h_adv_bitmap = nullptr;
    uint64_t *h_committed = nullptr;
    uint8_t *h_results = nullptr;
    uint32_t *h_step_adv = nullptr;
    // host (pageable)
    std::vector<Ring> rings;
    std::atomic<uint32_t> next_chunk{0};
    uint8_t *touched = nullptr;  // [cap] one bit per peer slot: cell has a record in wave 0
    std::mutex overflow_mu;
    std::unordered_map<uint64_t, uint32_t> overflow_depth;      // cell -> waves used beyond 0
    std::vector<std::vector<OverflowRec>> overflow_waves;       // wave w+1 records
    std::vector<std::pair<uint32_t, uint64_t>> overflow_order;  // (ring, seq | UINT64_MAX for EXT) per packed rec
    // device
    PackedRec *d_recs = nullptr;
    uint32_t *d_adv_bitmap = nullptr;
    uint64_t *d_commit_out = nullptr;
    uint8_t *d_results = nullptr;
    uint32_t *d_tile_off = nullptr;  // [cap / kFTile + 2]: tile index of a tileable compact stream
    uint32_t *d_step_adv = nullptr;  // [0] advanced groups of the step, [1] duplicate records (zero-copy)
    uint32_t *d_touched = nullptr;   // [cap/4] zero-copy steps: one bit per (group, slot)
    // wire steps (grown on demand): the frames and their offsets on the device
    uint8_t *d_wire = nullptr;   // also the device copy of a RAFTGPU_STEP_RAW batch
    uint64_t d_wire_cap = 0;
    uint64_t wire_n = 0;             // frames of the wire step this set carried (0 = not a wire step)
    uint64_t raw_n = 0;              // RAFTGPU_STEP_HYBRID: 24-byte records of this step that sit in d_wire as they are
    uint32_t raw_min_group = 0;      // ... all of groups >= this one (the packed part ends below it)
    // sync
    cudaEvent_t ev_h2d = nullptr, ev_compute = nullptr, ev_done = nullptr;
    cudaEvent_t ev_raw0 = nullptr, ev_raw1 = nullptr;  // around the hybrid step's raw H2D copy (timing: the effective PCIe rate)
    uint64_t raw_timed_bytes = 0;                      // bytes of that copy, 0 = nothing to read back
    bool in_flight = false;
    std::atomic<bool> dirty{false};  // touched[] has bits set (set by any enqueueing thread)
    uint32_t flags = 0;
    uint64_t wave0_slots = 0;  // staged wave-0 slots (chunks used * kChunk)
    raftgpu_step_result result{};
    // asynchronous steps (RAFTGPU_STEP_ASYNC): 1 = booked, the submitter thread has not queued it yet;
    // 0 = queued (or not an asynchronous step); < 0 = the submission failed with this status
    std::atomic<int32_t> submit_rc{0};
};

// One raftgpu_step_begin_records in progress (shared by the caller, the staging threads and the submitter).
struct RecJob {
    const raftgpu_append_resp *recs = nullptr;
    uint64_t n = 0;
    uint32_t flags = 0;
    bool async = false, trace = false;
    int T = 1, S = 1;
    StagingSet *set = nullptr;
    uint8_t *buf = nullptr;
    uint64_t cap_bytes = 0, meta_bytes = 0, side_bytes = 0, scratch_units = 0, gb_per_slice = 0;
    uint32_t *stream_units = nullptr;  // the unit stream in the set's pinned buffer
    uint64_t stream_cap_units = 0;
    std::chrono::steady_clock::time_point t_begin;
    std::vector<double> tr_a, tr_b;
    std::atomic<uint64_t> busy_ns{0};  // time the staging threads spent packing this job's slices (for the hybrid split)
    double us_since() const { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t_begin).count(); }
};

// The library's own staging workers (raftgpu_enqueue_bulk, raftgpu_step_begin_records): persistent
// threads, pinned to the GPU-local CPUs.  A step arrives every few hundred microseconds, so a worker
// that has just finished a job SPINS on the generation counter for a while (RAFTGPU_SPIN_US, default
// 2000) before it goes to sleep on the condition variable: waking 32 sleepers through a futex costs
// more than the job itself.  The submitter spins on `pending` likewise.
struct HostPool {
    // One sleeper slot per worker: a worker that has spun long enough sleeps on ITS OWN condition variable.
    // (One shared condition variable makes the wake-up a convoy: the woken threads queue on the one mutex and
    // come back one after the other, each paying its core's idle-state exit -- measured 6-8 ms for 32 workers.)
    struct alignas(128) Sleeper {
        std::mutex mu;
        std::condition_variable cv;
        bool sleeping = false;
    };
    std::vector<std::thread> threads;
    std::unique_ptr<Sleeper[]> sleepers;
    std::atomic<uint64_t> generation{0};
    std::atomic<int> pending{0};
    std::atomic<bool> stop{false};
    std::function<void(int)> job;
    int spin_us = 2000;

    static inline void cpu_relax() {
#if defined(__x86_64__)
        _mm_pause();
#endif
    }
    void wake_all() {
        for (size_t t = 0; t < threads.size(); t++) {
            Sleeper &sl = sleepers[t];
            std::lock_guard<std::mutex> lk(sl.mu);
            if (sl.sleeping) sl.cv.notify_one();
        }
    }
    // start `fn` on every worker and return at once; wait() blocks until all are done
    void start(const std::function<void(int)> &fn) {
        job = fn;
        pending.store(static_cast<int>(threads.size()));
        generation.fetch_add(1);
        wake_all();
    }
    void wait() {
        uint32_t spins = 0;
        while (pending.load(std::memory_order_acquire) != 0) {
            cpu_relax();
            if ((++spins & 63u) == 0) std::this_thread::yield();  // this thread may sit on a worker's CPU
        }
    }
    void run(const std::function<void(int)> &fn) {
        start(fn);
        wait();
    }
    cpu_set_t pool_cpus;      // RAFTGPU_PIN=set: every worker may run on any CPU of the pool's share
    bool pin_set = false;
    void worker(int idx, int cpu) {
        if (pin_set) {
            sched_setaffinity(0, sizeof(pool_cpus), &pool_cpus);
        } else if (cpu >= 0) {  // one CPU per worker (ensure_pool picks them: GPU-local physical cores first)
            cpu_set_t one;
            CPU_ZERO(&one);
            CPU_SET(cpu, &one);
            sched_setaffinity(0, sizeof(one), &one);
        }
        uint64_t seen = 0;
        for (;;) {
            const auto t_idle = std::chrono::steady_clock::now();
            uint32_t spins = 0;
            while (generation.load(std::memory_order_acquire) == seen && !stop.load(std::memory_order_relaxed)) {
                cpu_relax();
                // a spinning worker owns its CPU as far as the scheduler can tell: give way to whatever else is
                // runnable there (measured: the caller's thread, time-sliced against a spinning worker, lost ~0.4 ms
                // per call)
                if ((++spins & 127u) == 0) sched_yield();
                if ((spins & 255u) == 0 &&
                    std::chrono::steady_clock::now() - t_idle > std::chrono::microseconds(spin_us)) {
                    Sleeper &sl = sleepers[idx];
                    std::unique_lock<std::mutex> lk(sl.mu);
                    sl.sleeping = true;  // start() changes `generation` BEFORE it looks at this flag under the lock
                    sl.cv.wait(lk, [&] { return stop.load() || generation.load() != seen; });
                    sl.sleeping = false;
                    break;
                }
            }
            if (stop.load()) return;
            seen = generation.load(std::memory_order_acquire);
            job(idx);
            pending.fetch_sub(1, std::memory_order_release);
        }
    }
    ~HostPool() {
        stop.store(true);
        wake_all();
        for (auto &t : threads) t.join();
    }
};

}  // namespace

struct raftgpu_arena {
    int device = 0;
    uint32_t cap = 0;
    uint32_t n_rings = 0;
    uint32_t n_chunks = 0;  // chunks in each set's shared staging buffer
    uint64_t overflow_records = 0;
    uint32_t voter_hint = 0;                 // superset of every group's voter slots (recompute_kernel)
    int grid_recompute = 0, grid_recompute5 = 0, grid_apply = 0;  // persistent grid sizes (blocks)
    uint32_t hyb_samples = 0;
    double hyb_pcie_gbs = 0.0;               // RAFTGPU_STEP_HYBRID: measured rate of the raw H2D copies (GB/s), 0 = not measured yet
    double hyb_pack_ns = 0.0;                // RAFTGPU_STEP_HYBRID: measured packing cost (ns per record and staging thread), 0 = not measured yet
    bool rec_fallback_sorted = false;        // raftgpu_step_begin_records: the batch going to the general staging path is in group order
    uint32_t n_wide = 0;                     // wide groups (two slots each): the fused tile kernels are not used while any exist
    uint32_t n_simple5 = 0;                  // groups whose meta is the plain 5-voter configuration
    uint32_t tile_smem = 0;                  // dynamic shared memory for the fused tile kernels
    Columns cols{};
    uint32_t *d_wire_first = nullptr;  // [kSlots][cap] wire steps: first frame of every cell (allocated on first use)
    unsigned long long *d_counters = nullptr;
    void *d_scratch = nullptr;  // 256 B for single-group queries
    void *h_scratch = nullptr;  // pinned mirror
    cudaStream_t s_compute = nullptr, s_h2d = nullptr, s_d2h = nullptr;
    StagingSet sets[kNumSets];
    int fill = 0;        // set currently being filled by enqueue
    int last_done = -1;  // set whose results raftgpu_step_results exposes
    int inflight[2] = {-1, -1};  // sets submitted by step_begin and not yet waited for, oldest first
    int n_inflight = 0;
    // control plane: single-group calls share the scratch buffers and the meta mirror
    std::mutex ctl_mu;
    // group allocation
    std::mutex alloc_mu;
    std::vector<uint32_t> free_list;
    std::vector<uint8_t> allocated;
    std::vector<uint32_t> h_meta;  // host mirror of the meta column
    uint32_t hi = 0, n_alloc = 0;
    // info
    int sm_count = 0;
    uint64_t l2_bytes = 0, device_bytes = 0, pinned_bytes = 0;
    std::string last_error;
    std::vector<void *> user_allocs;
    std::vector<void *> host_allocs;  // raftgpu_host_alloc
    HostPool *pool = nullptr;  // created on first raftgpu_enqueue_bulk / raftgpu_step_begin_records
    // raftgpu_step_begin_records scratch, kept between steps (no allocation on the step path)
    std::vector<uint64_t> rec_cut;
    std::vector<PackState> rec_pack;
    std::vector<uint32_t> rec_gbase;
    std::vector<std::atomic<int32_t>> rec_done;
    std::vector<std::atomic<uint64_t>> rec_end;  // where every slice ends in the stream (UINT64_MAX = not packed yet)
    std::vector<uint32_t> rec_scratch;           // one private packing buffer per staging thread
    RecJob rec_job;
    std::atomic<int> rec_next{0};  // next slice to pack
    std::chrono::steady_clock::time_point t_created = std::chrono::steady_clock::now();  // RAFTGPU_TRACE timelines
    // the submitter thread of RAFTGPU_STEP_ASYNC steps
    std::thread sub_thread;
    std::mutex sub_mu;
    std::condition_variable sub_cv;
    bool sub_has_job = false, sub_stop = false;
    std::atomic<int> sub_busy{0};
    cpu_set_t local_cpus;      // GPU-local CPUs (empty when unknown)
    bool have_local_cpus = false;
};

namespace {

thread_local std::string g_create_error;

// Pinned staging must live on the NUMA node the GPU's PCIe root hangs off: DMA reads of
// remote-socket memory cross the inter-socket link and lose about half of the H2D bandwidth
// (measured on the 2-socket B200 hosts: 27 GB/s remote vs ~55 GB/s local).  cudaHostAlloc
// places pages by first touch, so the allocating thread is moved onto the GPU-local CPUs
// (sysfs local_cpulist of the device) for the duration of the allocations.
struct LocalCpuGuard {
    cpu_set_t saved;
    cpu_set_t local;  // the GPU-local CPUs we are allowed to run on
    bool active = false;
    explicit LocalCpuGuard(int device) {
        char bus[32] = {0};
        if (cudaDeviceGetPCIBusId(bus, sizeof(bus), device) != cudaSuccess) return;
        for (char *p = bus; *p; p++) *p = static_cast<char>(tolower(*p));
        std::string path = std::string("/sys/bus/pci/devices/") + bus + "/local_cpulist";
        FILE *f = fopen(path.c_str(), "r");
        if (!f) return;
        char line[512] = {0};
        const bool ok = fgets(line, sizeof(line), f) != nullptr;
        fclose(f);
        if (!ok) return;
        cpu_set_t want;
        CPU_ZERO(&want);
        int n_set = 0;
        for (char *tok = strtok(line, ",\n"); tok; tok = strtok(nullptr, ",\n")) {
            int lo = 0, hi = 0;
            const int k = sscanf(tok, "%d-%d", &lo, &hi);
            if (k == 1) hi = lo;
            if (k < 1) continue;
            for (int c = lo; c <= hi && c < CPU_SETSIZE; c++) {
                CPU_SET(c, &want);
                n_set++;
            }
        }
        if (!n_set) return;
        if (sched_getaffinity(0, sizeof(saved), &saved) != 0) return;
        cpu_set_t both;
        CPU_AND(&both, &want, &saved);  // stay inside the cpuset we are allowed to use
        if (CPU_COUNT(&both) == 0) return;
        local = both;
        if (sched_setaffinity(0, sizeof(both), &both) == 0) active = true;
    }
    ~LocalCpuGuard() {
        if (active) sched_setaffinity(0, sizeof(saved), &saved);
    }
};

int32_t fail(raftgpu_arena *a, int32_t code, const std::string &msg) {
    if (a) a->last_error = msg;
    return code;
}

#define CK(a, call)                                                                          \
    do {                                                                                     \
        cudaError_t e_ = (call);                                                             \
        if (e_ != cudaSuccess) {                                                             \
            return fail((a), RAFTGPU_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
        }                                                                                    \
    } while (0)

#define CKL(a)                                                                                    \
    do {                                                                                          \
        cudaError_t e_ = cudaGetLastError();                                                      \
        if (e_ != cudaSuccess)                                                                    \
            return fail((a), RAFTGPU_ERR_CUDA, std::string("launch: ") + cudaGetErrorString(e_)); \
    } while (0)

template <typename T>
int32_t dev_alloc(raftgpu_arena *a, T **p, size_t count, bool zero = true) {
    const size_t bytes = count * sizeof(T);
    cudaError_t e = cudaMalloc(reinterpret_cast<void **>(p), bytes ? bytes : 1);
    if (e != cudaSuccess)
        return fail(a, e == cudaErrorMemoryAllocation ? RAFTGPU_ERR_NOMEM : RAFTGPU_ERR_CUDA,
                    std::string("cudaMalloc: ") + cudaGetErrorString(e));
    a->device_bytes += bytes;
    if (zero) CK(a, cudaMemset(*p, 0, bytes ? bytes : 1));
    return RAFTGPU_OK;
}

template <typename T>
int32_t pin_alloc(raftgpu_arena *a, T **p, size_t count) {
    const size_t bytes = count * sizeof(T);
    cudaError_t e = cudaHostAlloc(reinterpret_cast<void **>(p), bytes ? bytes : 1, cudaHostAllocDefault);
    if (e != cudaSuccess)
        return fail(a, RAFTGPU_ERR_NOMEM, std::string("cudaHostAlloc: ") + cudaGetErrorString(e));
    a->pinned_bytes += bytes;
    memset(*p, 0, bytes);  // first touch decides the NUMA node
    return RAFTGPU_OK;
}

inline double trace_us(const raftgpu_arena *a) {
    return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - a->t_created).count();
}

inline bool group_ok(const raftgpu_arena *a, uint32_t g) { return g < a->cap && a->allocated[g]; }

inline uint32_t present_mask(uint32_t meta) {
    return RAFTGPU_META_IN(meta) | RAFTGPU_META_OUT(meta) | RAFTGPU_META_LEARN(meta);
}
inline uint32_t voter_mask(uint32_t meta) { return RAFTGPU_META_IN(meta) | RAFTGPU_META_OUT(meta); }

inline cudaStream_t pick_stream(raftgpu_arena *a, void *stream) {
    return stream ? static_cast<cudaStream_t>(stream) : a->s_compute;
}

inline uint32_t div_up(uint64_t a, uint32_t b) { return static_cast<uint32_t>((a + b - 1) / b); }

// True when every group of [first, first+n) is the plain 5-voter configuration in slots 0..4
// (no joint half, no group commit): the host's meta mirror is authoritative, so the kernels
// specialised for that case need no per-group check.
inline bool is_simple5(uint32_t meta) {
    return (meta & (0xffffu | RAFTGPU_META_GROUP_COMMIT | RAFTGPU_META_WIDE_LO | RAFTGPU_META_WIDE_HI)) == 0x1fu;
}
inline bool wide_lo(const raftgpu_arena *a, uint32_t g) { return (a->h_meta[g] & RAFTGPU_META_WIDE_LO) != 0; }
inline bool wide_hi(const raftgpu_arena *a, uint32_t g) { return (a->h_meta[g] & RAFTGPU_META_WIDE_HI) != 0; }
// peer slot 0..15 of a wide group -> (half, slot in the half); false = no such slot in this group
inline bool resolve_slot(const raftgpu_arena *a, uint32_t g, uint32_t slot, uint32_t *g2, uint32_t *s2) {
    if (slot < RAFTGPU_SLOTS) {
        *g2 = g;
        *s2 = slot;
        return true;
    }
    if (slot < 2 * RAFTGPU_SLOTS && wide_lo(a, g)) {
        *g2 = g + 1;
        *s2 = slot - RAFTGPU_SLOTS;
        return true;
    }
    return false;
}
inline bool range_simple5(const raftgpu_arena *a, uint32_t first, uint32_t n) {
    return a->n_simple5 == a->hi && static_cast<uint64_t>(first) + n <= a->hi;
}
// Diagnostic knobs of the fused tile kernels, read once per process -- or on every launch when
// RAFTGPU_TILE_TUNE is set (scripts/micro_tile.py switches them inside one process).
//   RAFTGPU_TILE_DEBUG (phase cycle counters), _SKIP (phases left out: results are WRONG)
struct TileKnobs {
    bool debug;
    uint32_t skip;
};
inline TileKnobs read_tile_knobs() {
    const char *skip = getenv("RAFTGPU_TILE_SKIP");
    return TileKnobs{getenv("RAFTGPU_TILE_DEBUG") != nullptr, static_cast<uint32_t>(skip ? atoi(skip) : 0)};
}
inline const TileKnobs &tile_knobs() {
    static const bool tune = getenv("RAFTGPU_TILE_TUNE") != nullptr;
    static TileKnobs k = read_tile_knobs();
    if (tune) k = read_tile_knobs();
    return k;
}

inline void set_meta(raftgpu_arena *a, uint32_t g, uint32_t meta) {
    a->n_simple5 += static_cast<uint32_t>(is_simple5(meta)) - static_cast<uint32_t>(is_simple5(a->h_meta[g]));
    a->n_wide += ((meta & RAFTGPU_META_WIDE_LO) ? 1u : 0u) - ((a->h_meta[g] & RAFTGPU_META_WIDE_LO) ? 1u : 0u);
    a->h_meta[g] = meta;
    a->voter_hint |= voter_mask(meta);
}

int32_t launch_recompute(raftgpu_arena *a, cudaStream_t st, uint32_t first, uint32_t n, uint32_t hint,
                         uint32_t *d_adv, uint64_t *d_commit, uint64_t *d_mci, uint8_t *d_gc,
                         uint32_t *d_step_adv) {
    if (n == 0) return RAFTGPU_OK;
    const bool simple5 = range_simple5(a, first, n);
    if (simple5) hint = 0x1fu;
    const uint32_t base = first & ~31u;
    const uint64_t threads = static_cast<uint64_t>(first - base) + n;
    if (simple5) {
        const uint32_t blocks = std::min<uint32_t>(div_up(threads, 256), static_cast<uint32_t>(a->grid_recompute5));
        recompute_kernel<true><<<blocks, 256, 0, st>>>(a->cols, first, n, hint, d_adv, d_commit, d_mci, d_gc,
                                                      d_step_adv, a->d_counters);
    } else {
        const uint32_t blocks = std::min<uint32_t>(div_up(threads, 256), static_cast<uint32_t>(a->grid_recompute));
        recompute_kernel<false><<<blocks, 256, 0, st>>>(a->cols, first, n, hint, d_adv, d_commit, d_mci, d_gc,
                                                       d_step_adv, a->d_counters);
    }
    CKL(a);
    return RAFTGPU_OK;
}

int32_t launch_apply(raftgpu_arena *a, cudaStream_t st, const void *d_recs, uint64_t n, uint8_t *d_results,
                     bool packed) {
    if (n == 0) return RAFTGPU_OK;
    const uint32_t blocks = std::min<uint32_t>(div_up(n, 256), static_cast<uint32_t>(a->grid_apply));
    if (packed)
        apply_kernel<true><<<blocks, 256, 0, st>>>(a->cols, d_recs, n, d_results, a->d_counters);
    else
        apply_kernel<false><<<blocks, 256, 0, st>>>(a->cols, d_recs, n, d_results, a->d_counters);
    CKL(a);
    return RAFTGPU_OK;
}

void free_set(StagingSet &s) {
    cudaFreeHost(s.h_recs);
    cudaFreeHost(s.h_overflow);
    cudaFreeHost(s.h_adv_bitmap);
    cudaFreeHost(s.h_committed);
    cudaFreeHost(s.h_results);
    cudaFreeHost(s.h_step_adv);
    free(s.touched);
    cudaFree(s.d_recs);
    cudaFree(s.d_adv_bitmap);
    cudaFree(s.d_commit_out);
    cudaFree(s.d_results);
    cudaFree(s.d_tile_off);
    cudaFree(s.d_step_adv);
    cudaFree(s.d_touched);
    cudaFree(s.d_wire);
    if (s.ev_h2d) cudaEventDestroy(s.ev_h2d);
    if (s.ev_raw0) cudaEventDestroy(s.ev_raw0);
    if (s.ev_raw1) cudaEventDestroy(s.ev_raw1);
    if (s.ev_compute) cudaEventDestroy(s.ev_compute);
    if (s.ev_done) cudaEventDestroy(s.ev_done);
}

void destroy(raftgpu_arena *a) {
    if (!a) return;
    if (a->sub_thread.joinable()) {
        {
            std::lock_guard<std::mutex> lk(a->sub_mu);
            a->sub_stop = true;
        }
        a->sub_cv.notify_one();
        a->sub_thread.join();
    }
    cudaSetDevice(a->device);
    cudaDeviceSynchronize();
    Columns &c = a->cols;
    cudaFree(c.matched);
    cudaFree(c.next_idx);
    cudaFree(c.peer_committed);
    cudaFree(c.pending_snapshot);
    cudaFree(c.pending_req_snapshot);
    cudaFree(c.commit_group_id);
    cudaFree(c.pflags);
    cudaFree(c.votes);
    cudaFree(c.meta);
    cudaFree(c.committed);
    cudaFree(c.term_start);
    cudaFree(c.last_index);
    cudaFree(c.term);
    cudaFree(c.ins_meta);
    cudaFree(c.ins_buf);
    cudaFree(c.rd_meta);
    cudaFree(c.rd_ctx);
    cudaFree(c.rd_index);
    cudaFree(c.rd_word);
    cudaFree(c.rd_first);
    cudaFree(a->d_wire_first);
    cudaFree(a->d_counters);
    cudaFree(a->d_scratch);
    cudaFreeHost(a->h_scratch);
    for (void *p : a->user_allocs) cudaFree(p);
    for (void *p : a->host_allocs) cudaFreeHost(p);
    delete a->pool;
    for (auto &s : a->sets) free_set(s);
    if (a->s_compute) cudaStreamDestroy(a->s_compute);
    if (a->s_h2d) cudaStreamDestroy(a->s_h2d);
    if (a->s_d2h) cudaStreamDestroy(a->s_d2h);
    delete a;
}

int32_t create(int32_t device, uint32_t max_groups, uint32_t slots, uint32_t n_rings,
               uint32_t ring_records, raftgpu_arena **out) {
    if (!out || max_groups == 0) return RAFTGPU_ERR_INVALID;
    if (slots != RAFTGPU_SLOTS) return RAFTGPU_ERR_TOO_MANY_PEERS;  // the documented hard limit (raftgpu.h)
    *out = nullptr;
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {
        cudaGetLastError();
        return RAFTGPU_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= n_dev) return RAFTGPU_ERR_INVALID;
    raftgpu_arena *a = new (std::nothrow) raftgpu_arena();
    if (!a) return RAFTGPU_ERR_NOMEM;
    a->device = device;
    // pad the column stride so every column (and every slot row of it) is 128-byte aligned
    a->cap = (max_groups + 127u) & ~127u;
    a->n_rings = n_rings ? n_rings : 16;
    // staging capacity per step, shared by all rings: ring_records * n_rings when given, else
    // ~5 records per group (a full round of a 5-peer deployment is ~3.5); plus one partially
    // filled chunk per ring
    const uint64_t want = ring_records ? static_cast<uint64_t>(ring_records) * a->n_rings
                                       : std::max<uint64_t>(4096, 5ull * a->cap);
    a->n_chunks = div_up(want, kChunk) + a->n_rings;
    a->overflow_records = std::max<uint64_t>(4096, a->cap / 4);
    int32_t rc = RAFTGPU_OK;
    auto bail = [&](int32_t code) {
        g_create_error = a->last_error;
        destroy(a);
        return code;
    };
#define TRY(x)                                 \
    do {                                       \
        rc = (x);                              \
        if (rc != RAFTGPU_OK) return bail(rc); \
    } while (0)
#define TRYC(call)                                                              \
    do {                                                                        \
        cudaError_t e_ = (call);                                                \
        if (e_ != cudaSuccess) {                                                \
            a->last_error = std::string(#call) + ": " + cudaGetErrorString(e_); \
            return bail(RAFTGPU_ERR_CUDA);                                      \
        }                                                                       \
    } while (0)
    TRYC(cudaSetDevice(device));
    cudaDeviceProp prop{};
    TRYC(cudaGetDeviceProperties(&prop, device));
    a->sm_count = prop.multiProcessorCount;
    a->l2_bytes = static_cast<uint64_t>(prop.l2CacheSize);
    int occ = 0;
    TRYC(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, recompute_kernel<false>, 256, 0));
    a->grid_recompute = std::max(1, occ) * a->sm_count;
    TRYC(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, recompute_kernel<true>, 256, 0));
    a->grid_recompute5 = std::max(1, occ) * a->sm_count;
    TRYC(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, apply_kernel<true>, 256, 0));
    a->grid_apply = std::max(1, occ) * a->sm_count;
    a->tile_smem = 227u * 1024u - 5u * 1024u;  // 227 KB per CTA minus the kernels' static shared memory (barriers, deferred lists)
    const void *const tile_kernels[] = {
        reinterpret_cast<const void *>(step_tile_kernel<false>), reinterpret_cast<const void *>(step_tile_kernel<true>),
        reinterpret_cast<const void *>(step_tile_compact_kernel<false, false>),
        reinterpret_cast<const void *>(step_tile_compact_kernel<true, false>),
        reinterpret_cast<const void *>(step_tile_compact_kernel<false, true>),
        reinterpret_cast<const void *>(step_tile_compact_kernel<true, true>)};
    for (const void *k : tile_kernels)
        TRYC(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(a->tile_smem)));
    TRYC(cudaStreamCreateWithFlags(&a->s_compute, cudaStreamNonBlocking));
    TRYC(cudaStreamCreateWithFlags(&a->s_h2d, cudaStreamNonBlocking));
    TRYC(cudaStreamCreateWithFlags(&a->s_d2h, cudaStreamNonBlocking));

    const size_t cells = static_cast<size_t>(kSlots) * a->cap;
    Columns &c = a->cols;
    c.cap = a->cap;
    TRY(dev_alloc(a, &c.matched, cells));
    TRY(dev_alloc(a, &c.next_idx, cells));
    TRY(dev_alloc(a, &c.peer_committed, cells));
    TRY(dev_alloc(a, &c.pending_snapshot, cells));
    TRY(dev_alloc(a, &c.pending_req_snapshot, cells));
    TRY(dev_alloc(a, &c.commit_group_id, cells));
    TRY(dev_alloc(a, &c.pflags, cells));
    TRY(dev_alloc(a, &c.votes, cells));
    TRY(dev_alloc(a, &c.meta, a->cap));
    TRY(dev_alloc(a, &c.committed, a->cap));
    TRY(dev_alloc(a, &c.term_start, a->cap));
    TRY(dev_alloc(a, &c.last_index, a->cap));
    TRY(dev_alloc(a, &c.term, a->cap));
    TRYC(cudaMemset(c.term_start, 0xff, sizeof(uint64_t) * a->cap));  // RAFTGPU_NO_TERM_START
    TRY(dev_alloc(a, &a->d_counters, kCntCount + 8));  // + 8 diagnostic slots (fused kernel phase cycles)
    TRY(dev_alloc(a, reinterpret_cast<uint8_t **>(&a->d_scratch), 256));
    TRY(pin_alloc(a, reinterpret_cast<uint8_t **>(&a->h_scratch), 256));

    const uint64_t wave0_total = static_cast<uint64_t>(a->n_chunks) * kChunk;
    const uint64_t rec_total = wave0_total + a->overflow_records;
    LocalCpuGuard numa_guard(device);  // pinned pages on the GPU-local NUMA node
    CPU_ZERO(&a->local_cpus);
    if (numa_guard.active) {
        a->local_cpus = numa_guard.local;
        a->have_local_cpus = true;
    }
    for (auto &s : a->sets) {
        TRY(pin_alloc(a, &s.h_recs, wave0_total));
        TRY(pin_alloc(a, &s.h_overflow, a->overflow_records));
        TRY(pin_alloc(a, &s.h_adv_bitmap, a->cap / 32));
        TRY(pin_alloc(a, &s.h_committed, a->cap));
        TRY(pin_alloc(a, &s.h_results, 4 * rec_total));  // one byte per slot; a compact stream has 4-byte units
        TRY(pin_alloc(a, &s.h_step_adv, 4));
        s.rings.assign(a->n_rings, Ring());
        s.touched = static_cast<uint8_t *>(calloc(a->cap, 1));
        if (!s.touched) return bail(RAFTGPU_ERR_NOMEM);
        TRY(dev_alloc(a, &s.d_recs, rec_total, false));
        TRY(dev_alloc(a, &s.d_adv_bitmap, a->cap / 32));
        TRY(dev_alloc(a, &s.d_commit_out, a->cap));
        TRY(dev_alloc(a, &s.d_results, 4 * rec_total));
        TRY(dev_alloc(a, &s.d_tile_off, 3 * (a->cap / kFTile + 2) + 2));
        TRY(dev_alloc(a, &s.d_step_adv, 4));
        TRY(dev_alloc(a, &s.d_touched, a->cap / 4));
        TRYC(cudaEventCreateWithFlags(&s.ev_h2d, cudaEventDisableTiming));
        TRYC(cudaEventCreate(&s.ev_raw0));
        TRYC(cudaEventCreate(&s.ev_raw1));
        TRYC(cudaEventCreateWithFlags(&s.ev_compute, cudaEventDisableTiming));
        TRYC(cudaEventCreateWithFlags(&s.ev_done, cudaEventDisableTiming));
    }
    a->allocated.assign(a->cap, 0);
    a->h_meta.assign(a->cap, 0);
    TRYC(cudaDeviceSynchronize());
#undef TRY
#undef TRYC
    *out = a;
    return RAFTGPU_OK;
}

// Control-plane kernel(s) + sync on the compute stream.
template <typename F>
int32_t sync_op(raftgpu_arena *a, F &&launch) {
    CK(a, cudaSetDevice(a->device));
    launch(a->s_compute);
    CKL(a);
    CK(a, cudaStreamSynchronize(a->s_compute));
    return RAFTGPU_OK;
}

// Group alloc / free on an arena with read-index queues: the groups' queues are empty and marked (un)allocated.
int32_t read_mark_alloc(raftgpu_arena *a, uint32_t first, uint32_t n, bool allocated) {
    if (!a->cols.rd_cap || n == 0) return RAFTGPU_OK;
    const uint32_t blocks = std::min<uint32_t>(div_up(n, 256), 8u * static_cast<uint32_t>(a->sm_count));
    return sync_op(a, [&](cudaStream_t st) {
        read_alloc_kernel<<<blocks, 256, 0, st>>>(a->cols, first, n, allocated ? kRdAlloc : 0u);
    });
}

struct ColumnDesc {
    void *base;
    size_t elem;
    bool per_peer;
};

bool column_desc(raftgpu_arena *a, int32_t col, ColumnDesc *d) {
    Columns &c = a->cols;
    switch (col) {
    case RAFTGPU_COL_MATCHED: *d = {c.matched, 8, true}; return true;
    case RAFTGPU_COL_NEXT_IDX: *d = {c.next_idx, 8, true}; return true;
    case RAFTGPU_COL_PEER_COMMITTED: *d = {c.peer_committed, 8, true}; return true;
    case RAFTGPU_COL_PENDING_SNAPSHOT: *d = {c.pending_snapshot, 8, true}; return true;
    case RAFTGPU_COL_PENDING_REQ_SNAPSHOT: *d = {c.pending_req_snapshot, 8, true}; return true;
    case RAFTGPU_COL_COMMIT_GROUP_ID: *d = {c.commit_group_id, 8, true}; return true;
    case RAFTGPU_COL_PFLAGS: *d = {c.pflags, 1, true}; return true;
    case RAFTGPU_COL_VOTES: *d = {c.votes, 1, true}; return true;
    case RAFTGPU_COL_META: *d = {c.meta, 4, false}; return true;
    case RAFTGPU_COL_COMMITTED: *d = {c.committed, 8, false}; return true;
    case RAFTGPU_COL_TERM_START: *d = {c.term_start, 8, false}; return true;
    case RAFTGPU_COL_LAST_INDEX: *d = {c.last_index, 8, false}; return true;
    case RAFTGPU_COL_TERM: *d = {c.term, 8, false}; return true;
    case RAFTGPU_COL_INS_META:
        if (!c.ins_cap) return false;
        *d = {c.ins_meta, 4, true};
        return true;
    default: return false;
    }
}

// Move a duplicate-cell record (already packed) to a later wave.
void push_overflow(StagingSet &s, uint64_t cell, const PackedRec *pk, int n_pk, uint32_t ring, uint64_t seq) {
    std::lock_guard<std::mutex> lk(s.overflow_mu);
    const uint32_t depth = s.overflow_depth[cell]++;  // 0 -> wave 1
    if (s.overflow_waves.size() <= depth) s.overflow_waves.resize(depth + 1);
    OverflowRec o{};
    for (int k = 0; k < n_pk; k++) o.pk[k] = pk[k];
    o.n_pk = n_pk;
    o.ring = ring;
    o.seq = seq;
    s.overflow_waves[depth].push_back(o);
}

// make a finished set reusable for filling
int32_t reclaim_set(raftgpu_arena *a, StagingSet &s) {
    if (s.in_flight) return RAFTGPU_ERR_BUSY;
    if (s.dirty.load(std::memory_order_relaxed)) {
        memset(s.touched, 0, a->cap);
        s.dirty.store(false, std::memory_order_relaxed);
    }
    for (auto &r : s.rings) {
        r.chunks.clear();
        r.fill = kChunk;
        r.seq = 0;
        r.overflow_seq.clear();
    }
    s.next_chunk.store(0);
    s.wire_n = 0;
    s.overflow_depth.clear();
    s.overflow_waves.clear();
    return RAFTGPU_OK;
}

// host batch -> device scratch (the fill set's record staging, idle between steps) -> kernel -> results
// every entry point that queues work or touches the staging sets first lets a pending asynchronous submission finish
void wait_submitter(raftgpu_arena *a) {
    uint32_t spins = 0;
    while (a->sub_busy.load(std::memory_order_acquire) != 0) {
        HostPool::cpu_relax();
        if ((++spins & 63u) == 0) std::this_thread::yield();
    }
}

template <typename T, typename F>
int32_t host_batch_op(raftgpu_arena *a, const T *in, uint64_t n, uint8_t *results, F &&launch, uint32_t *out_dups) {
    wait_submitter(a);
    StagingSet &s = a->sets[a->fill];
    if (s.in_flight || s.next_chunk.load() != 0) return fail(a, RAFTGPU_ERR_BUSY, "records are staged for a step: step first");
    const uint64_t room = (static_cast<uint64_t>(a->n_chunks) * kChunk + a->overflow_records) * sizeof(PackedRec);
    if (n * sizeof(T) > room || n > 4 * (room / sizeof(PackedRec))) return fail(a, RAFTGPU_ERR_FULL, "batch larger than the staging buffer");
    CK(a, cudaSetDevice(a->device));
    CK(a, cudaMemcpyAsync(s.d_recs, in, n * sizeof(T), cudaMemcpyHostToDevice, a->s_compute));
    CK(a, cudaMemsetAsync(s.d_step_adv, 0, 8, a->s_compute));
    const int32_t rc = launch(reinterpret_cast<const T *>(s.d_recs), s.d_results, s.d_step_adv + 1);
    if (rc != RAFTGPU_OK) return rc;
    if (results) CK(a, cudaMemcpyAsync(results, s.d_results, n, cudaMemcpyDeviceToHost, a->s_compute));
    CK(a, cudaMemcpyAsync(s.h_step_adv, s.d_step_adv, 8, cudaMemcpyDeviceToHost, a->s_compute));
    CK(a, cudaStreamSynchronize(a->s_compute));
    if (out_dups) *out_dups = s.h_step_adv[1];
    return RAFTGPU_OK;
}

}  // namespace

// ===========================================================================
extern "C" {

#include "abi_control.inc"
#include "abi_device.inc"
#include "abi_staging.inc"
#include "abi_compact.inc"
#include "abi_wire.inc"
#include "abi_results.inc"
#include "abi_read.inc"

}  // extern "C"
