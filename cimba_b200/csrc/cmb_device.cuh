// cmb_device.cuh - the cimba public surface on the device: the API a MODEL AUTHOR writes against.
//
// The reference's models are C functions running on stackful coroutines that call cmb_process_hold,
// cmb_objectqueue_put/get, cmb_resourcepool_acquire/release, cmb_random_* ... (include/cmb_process.h,
// include/cmb_event.h:75-323, include/cmb_objectqueue.h, include/cmb_resourcepool.h, include/cmb_random.h).
// A device stack cannot be switched, so here a process body is a function that RETURNS at every blocking call
// and is re-entered at that point when its wake-up event is popped (a resume-point index per process, SURVEY.md
// section 7): the CMB_* macros below expand a blocking call into "begin; remember the resume point; return;
// resume point: end", which is all the reference's cmi_coroutine_yield / resume pair does for a model
// (src/cmi_coroutine.c:280-306).  Body locals that must survive a blocking call live in the model struct or in
// the process record (cmb_process::f[], ::u[]) instead of on a coroutine stack.
//
// ONE engine serves every model written this way (cmb::Sim below): the future-event list and every wait list
// are cmb::HashHeap - the reference's cmi_hashheap (src/cmi_hashheap.c) with its physical layout (1-based binary
// heap, slot 0 = last popped, the same sift and remove steps - src/cmi_hashheap.c:277-370, 529-579), its lazily
// activated Fibonacci-hash key map with linear probing and tombstones (:189-272, 587-622) and its growth by
// doubling with rehash (:381-421).  Keys are 64-bit as in the reference (:449-453).  Capacities are not compile-time
// constants: every container starts in a few inline slots and grows from a per-launch HBM arena, so a model with
// 1 000 processes, 2 000 pending events and cancellations by handle runs on the same code as M/M/1.
//
// Mapping: one trial per CUDA thread.  The per-trial control block (cmb::Sim + the model struct) lives in the
// thread's local memory, which the hardware interleaves across the lanes of a warp - lane-private state at the
// same offset is one coalesced access - and grown containers live in the arena.
//
// The same source text compiles for the host (CMB_HOST_BUILD, tests/cmb_engine_host.cpp): the CPU tests run the
// engine and the shipped models on the CPU against the reference build before any GPU sees them.
#pragma once

#include <cstdint>
#include <utility>
#ifndef CMB_HOST_BUILD
#include <cuda_runtime.h>
#endif

#include "engine.cuh"
#include "rng.cuh"
#include "distributions.cuh"
#include "summary.cuh"

#ifdef CMB_HOST_BUILD
#define CMB_FN inline
#define CMB_FN_NOINLINE __attribute__((noinline))
#else
#define CMB_FN __device__ __forceinline__
#define CMB_FN_NOINLINE __device__ __noinline__
#endif

// ---- the reference's constants, same values (include/cmb_process.h:59-99, include/cmb_objectqueue.h)
#define CMB_PROCESS_CREATED     (cimba_b200::cmb::PROC_CREATED)      // what cmb_process_status(pid) returns
#define CMB_PROCESS_RUNNING     (cimba_b200::cmb::PROC_RUNNING)
#define CMB_PROCESS_FINISHED    (cimba_b200::cmb::PROC_FINISHED)
#define CMB_PROCESS_SUCCESS     ((int64_t)0)
#define CMB_PROCESS_PREEMPTED   ((int64_t)-1)
#define CMB_PROCESS_INTERRUPTED ((int64_t)-2)
#define CMB_PROCESS_STOPPED     ((int64_t)-3)
#define CMB_PROCESS_CANCELLED   ((int64_t)-4)
#define CMB_PROCESS_TIMEOUT     ((int64_t)-5)
#define CMB_UNLIMITED           UINT64_MAX

namespace cimba_b200 {
namespace cmb {

constexpr uint32_t NIL = 0xffffffffu;

enum : uint32_t { TRIAL_ERR_ARENA = 64u };             // the HBM arena ran out: a container could not grow

// ------------------------------------------------------------------------------------------------ arena
// Growth memory shared by all trials of a launch: a bump allocator over a slice of the job's workspace.  Blocks a
// container leaves behind when it doubles are not reused (geometric growth: at most as much again as is live).
struct Arena {
    unsigned char *base;
    unsigned long long *cursor;
    unsigned long long bytes;

    CMB_FN void *alloc(uint64_t n)
    {
        n = (n + 15u) & ~(uint64_t)15u;
#ifdef CMB_HOST_BUILD
        const unsigned long long at = *cursor;
        *cursor += n;
#else
        const unsigned long long at = atomicAdd(cursor, (unsigned long long)n);
#endif
        return (at + n <= bytes) ? (void *)(base + at) : nullptr;
    }
};

// ------------------------------------------------------------------------------------------------ hashheap
// struct cmi_heap_tag (src/cmi_hashheap.h:53-59: hash_key, hash_index, rank_d64, rank_i64, item[4] = 64 bytes)
// packed to 40: the four item pointers become a process / object index, an action or demand id, a 32-bit argument
// (signals are small integers) and a link (head of the event's waiter list).
struct Tag {
    double   d;                 // rank_d64: event time / guard entry time / payload of a priority-queue entry
    uint64_t key;               // hash_key
    int32_t  prio;              // rank_i64
    uint32_t hslot;             // hash_index: this entry's slot in the key map (valid while the map is active)
    uint32_t subj;              // item[1]: process index, or NIL
    uint16_t act;               // item[0]: event action / guard demand id
    uint16_t aux;
    int32_t  arg;               // item[2]: signal, amount, user argument
    uint32_t link;              // item[3]: head of the list of processes waiting for this event (NIL = none)
};
static_assert(sizeof(Tag) == 40, "Tag layout");

struct MapSlot {                // struct cmi_hash_tag (src/cmi_hashheap.h:75-78); key 0 = never used,
    uint64_t key;               // heap_index 0 with a key = tombstone
    uint32_t heap_index;
    uint32_t pad;
};

// default_compare, src/cmi_hashheap.c:55-80: time asc, priority desc, key asc
struct EventOrder {
    static CMB_FN bool before(const Tag &a, const Tag &b)
    {
        if (a.d < b.d) return true;
        if (a.d > b.d) return false;
        if (a.prio > b.prio) return true;
        if (a.prio < b.prio) return false;
        return a.key < b.key;
    }
};
// guard_queue_check, src/cmb_resourceguard.c:71-90 - including its fall-through when a has the LOWER priority
struct GuardOrder {
    static CMB_FN bool before(const Tag &a, const Tag &b)
    {
        if (a.prio > b.prio) return true;
        if (a.d < b.d) return true;
        if (a.key < b.key) return true;
        return false;
    }
};
// holder_queue_check, src/cmb_resourcepool.c:75-92: lowest priority first, then the LARGER key (the reference keys
// holders by process address; here by process index + 1 - SURVEY.md quirk 4)
struct HolderOrder {
    static CMB_FN bool before(const Tag &a, const Tag &b)
    {
        if (a.prio < b.prio) return true;
        if (a.prio == b.prio && a.key > b.key) return true;
        return false;
    }
};
// cmb_priorityqueue's order, src/cmb_priorityqueue.c:43-54: priority desc, then FIFO
struct PrioOrder {
    static CMB_FN bool before(const Tag &a, const Tag &b)
    {
        if (a.prio != b.prio) return a.prio > b.prio;
        return a.key < b.key;
    }
};

template <class Order>
struct HashHeap {
    Tag      *tag;              // [cap + 1], 1-based; tag[0] = the entry popped last (src/cmi_hashheap.c:496-498)
    MapSlot  *map;              // [2 * cap] once active
    uint32_t  exp;              // cap = 1 << exp (heap_exp_cur)
    uint32_t  count;
    uint32_t  map_on;           // map_active: the map is built at the first lookup by key (:538-542, 595-599)
    uint32_t  map_used;         // slots that ever held a key (live + tombstones)
    uint64_t  issued;           // item_counter (:449-453)

    CMB_FN uint32_t cap() const { return 1u << exp; }

    CMB_FN void init(Tag *inline_store, uint32_t inline_exp)
    {
        tag = inline_store;
        map = nullptr;
        exp = inline_exp;
        count = 0u;
        map_on = 0u;
        map_used = 0u;
        issued = 0u;
    }

    CMB_FN void place(uint32_t k, const Tag &t)        // write a tag into heap slot k; the map follows it
    {
        tag[k] = t;
        if (map_on) map[t.hslot].heap_index = k;
    }

    CMB_FN_NOINLINE void sift_up(uint32_t k)           // heap_up, :277-316
    {
        const Tag moving = tag[k];
        uint32_t parent;
        while ((parent = (k >> 1)) > 0u) {
            if (!Order::before(moving, tag[parent])) break;
            place(k, tag[parent]);
            k = parent;
        }
        place(k, moving);
    }

    CMB_FN_NOINLINE void sift_down(uint32_t k)         // heap_down, :321-370
    {
        const Tag moving = tag[k];
        const uint32_t last_parent = count >> 1;
        while (k <= last_parent) {
            uint32_t child = k << 1;
            if (child + 1u <= count && Order::before(tag[child + 1u], tag[child])) child++;
            if (Order::before(moving, tag[child])) break;
            place(k, tag[child]);
            k = child;
        }
        place(k, moving);
    }

    // hash_key, :189-198
    CMB_FN uint32_t hash_of(uint64_t key) const
    {
        return (uint32_t)((key * 11400714819323198485ull) >> (64u - (exp + 1u)));
    }

    // hash_find_slot, :204-223: the first slot that holds no live entry (never used, or a tombstone)
    CMB_FN uint32_t free_slot(uint64_t key) const
    {
        const uint32_t mask = (cap() << 1) - 1u;
        uint32_t h = hash_of(key);
        while (map[h].heap_index != 0u) h = (h + 1u) & mask;
        return h;
    }

    CMB_FN void map_insert(uint32_t k)                 // enter heap slot k's key into the map
    {
        const uint32_t h = free_slot(tag[k].key);
        if (map[h].key == 0u) map_used++;
        map[h].key = tag[k].key;
        map[h].heap_index = k;
        tag[k].hslot = h;
    }

    CMB_FN void map_rebuild()                          // hash_init, :228-241, over a cleared map
    {
        const uint32_t slots = cap() << 1;
        for (uint32_t i = 0u; i < slots; i++) {
            map[i].key = 0u;
            map[i].heap_index = 0u;
        }
        map_used = 0u;
        for (uint32_t k = 1u; k <= count; k++) map_insert(k);
    }

    CMB_FN_NOINLINE bool map_activate(Arena &arena)
    {
        if (map_on) return true;
        map = (MapSlot *)arena.alloc((uint64_t)(cap() << 1) * sizeof(MapSlot));
        if (map == nullptr) return false;
        map_on = 1u;
        map_rebuild();
        return true;
    }

    // hashheap_grow, :381-421: twice the heap, twice the map, live keys rehashed (tombstones dropped)
    CMB_FN_NOINLINE bool grow(Arena &arena)
    {
        const uint32_t old_cap = cap();
        Tag *bigger = (Tag *)arena.alloc((uint64_t)(2u * old_cap + 1u) * sizeof(Tag));
        if (bigger == nullptr) return false;
        for (uint32_t k = 0u; k <= count; k++) bigger[k] = tag[k];
        tag = bigger;
        exp++;
        if (map_on) {
            map = (MapSlot *)arena.alloc((uint64_t)(cap() << 1) * sizeof(MapSlot));
            if (map == nullptr) {
                map_on = 0u;
                return false;
            }
            map_rebuild();
        }
        return true;
    }

    // make room for n entries in one step (a model that knows its population says so up front)
    CMB_FN bool reserve(Arena &arena, uint32_t n)
    {
        while (cap() < n) {
            if (!grow(arena)) return false;
        }
        return true;
    }

    // cmi_hashheap_enqueue, :428-478.  key 0 = issue the next one.  Returns the key, or 0 if the arena is exhausted.
    CMB_FN_NOINLINE uint64_t enqueue(Arena &arena, uint64_t key, double d, int32_t prio,
                                     uint32_t subj, uint32_t act, int32_t arg, uint32_t link)
    {
        issued += 1u;
        if (key == 0u) key = issued;
        if (count == cap() && !grow(arena)) return 0u;
        const uint32_t at = ++count;
        Tag t;
        t.d = d;
        t.key = key;
        t.prio = prio;
        t.hslot = 0u;
        t.subj = subj;
        t.act = (uint16_t)act;
        t.aux = 0u;
        t.arg = arg;
        t.link = link;
        tag[at] = t;
        if (map_on) {
            if (map_used + 1u >= (cap() << 1) - (cap() >> 2)) map_rebuild();    // nearly every slot has held a key: drop the tombstones
            else map_insert(at);
        }
        sift_up(at);
        return key;
    }

    // cmi_hashheap_dequeue, :486-524: the first entry moves to slot 0
    CMB_FN_NOINLINE bool dequeue()
    {
        if (count == 0u) return false;
        tag[0] = tag[1];
        if (map_on) map[tag[0].hslot].heap_index = 0u;                   // tombstone
        if (count > 1u) {
            place(1u, tag[count]);
            count--;
            if (count > 1u) sift_down(1u);
        }
        else {
            count = 0u;
        }
        return true;
    }

    // cmi_hash_find_index, :587-622: heap slot of `key`, 0 = absent
    CMB_FN_NOINLINE uint32_t find(Arena &arena, uint64_t key)
    {
        if (count == 0u) return 0u;
        if (!map_activate(arena)) {                    // no room for a map: fall back to scanning
            for (uint32_t k = 1u; k <= count; k++) {
                if (tag[k].key == key) return k;
            }
            return 0u;
        }
        const uint32_t mask = (cap() << 1) - 1u;
        uint32_t h = hash_of(key);
        const uint32_t start = h;
        for (;;) {
            if (map[h].key == key) return map[h].heap_index;
            if (map[h].key == 0u) return 0u;
            h = (h + 1u) & mask;
            if (h == start) return 0u;
        }
    }

    // cmi_hashheap_remove, :529-579
    CMB_FN_NOINLINE bool remove(Arena &arena, uint64_t key)
    {
        const uint32_t at = find(arena, key);
        if (at == 0u) return false;
        if (map_on) map[tag[at].hslot].heap_index = 0u;                  // lazy deletion: tombstone
        if (at == count) {
            count--;
            return true;
        }
        const bool down = Order::before(tag[at], tag[count]);
        place(at, tag[count]);
        count--;
        if (down) sift_down(at);
        else sift_up(at);
        return true;
    }

    // cmi_hashheap_reprioritize, :679-711
    CMB_FN_NOINLINE bool reprioritize(Arena &arena, uint64_t key, double d, int32_t prio)
    {
        const uint32_t at = find(arena, key);
        if (at == 0u) return false;
        const Tag old = tag[at];
        tag[at].d = d;
        tag[at].prio = prio;
        if (Order::before(old, tag[at])) sift_down(at);
        else sift_up(at);
        return true;
    }
};

// ------------------------------------------------------------------------------------------------ lists
// cmi_slist + cmi_mempool (src/cmi_slist.h:65-85, src/cmi_mempool.h:112-153): LIFO lists of 16-byte nodes drawn
// from one growable per-trial pool - awaitables (a = type, b = event handle / guard address), process waiters and
// event waiters (a = process index), resources held (a = kind, b = address).
struct Node {
    uint32_t a;
    uint32_t next;
    uint64_t b;
};

enum : uint32_t { AWAIT_TIME = 0u, AWAIT_RESOURCE = 1u, AWAIT_PROCESS = 2u, AWAIT_EVENT = 3u };
enum : uint32_t { PROC_CREATED = 0u, PROC_RUNNING = 1u, PROC_FINISHED = 2u };
enum : uint32_t { HOLD_POOL = 1u, HOLD_RESOURCE = 2u };

// event actions: the reference's event functions
enum : uint32_t {
    ACT_CMB_START = 1u,         // start_event,             src/cmb_process.c:115-122
    ACT_CMB_WAKE_TIME = 2u,     // wakeup_event_time,       :292-308
    ACT_CMB_WAKE_RESOURCE = 3u, // wakeup_event_resource,   src/cmb_resourceguard.c:168-180
    ACT_CMB_WAKE_INTERRUPT = 4u,// wakeup_event_interrupt,  src/cmb_process.c:628-643
    ACT_CMB_WAKE_PREEMPT = 6u,  // wakeup_event_preempt,    src/cmb_resource.c:256-268
    ACT_CMB_WAKE_CONDITION = 7u,// wakeup_event_condition,  src/cmb_condition.c:85-103
    ACT_CMB_WAKE_PROCESS = 8u,  // wakeup_event_process,    src/cmb_process.c:386-410
    ACT_CMB_WAKE_EVENT = 9u,    // wakeup_event_event,      src/cmb_event.c:176-198
    ACT_CMB_RESUME = 10u,       // resume_event,            src/cmb_process.c:731-745
    ACT_CMB_USER = 32u,         // first action id a model may use for its own events (cmb_event_schedule)
};

// what a process body asks of the dispatcher when it returns (Sim::cmd)
enum : uint32_t { CMD_NONE = 0u, CMD_HOLD = 1u, CMD_HOLD_EXPONENTIAL = 2u, CMD_GUARD_WAIT = 3u, CMD_EXIT = 4u, CMD_HOLD_SAMPLED = 5u };

// demands a guard entry can carry (the reference stores a predicate function + context, src/cmb_resourceguard.c:125-152)
enum : uint32_t {
    DEMAND_QUEUE_CONTENT = 1u,  // has_content,  src/cmb_objectqueue.c:119-133
    DEMAND_QUEUE_SPACE = 2u,    // has_space,    :135-149
    DEMAND_POOL_AVAILABLE = 3u, // is_available, src/cmb_resourcepool.c:198-211
    DEMAND_RESOURCE_FREE = 4u,  // is_available, src/cmb_resource.c:155-167
    DEMAND_BUFFER_CONTENT = 5u, // buffer_has_content, src/cmb_buffer.c:96-108
    DEMAND_BUFFER_SPACE = 6u,   // buffer_has_space,   :110-122
    DEMAND_PQ_CONTENT = 7u,     // has_content, src/cmb_priorityqueue.c:119-133
    DEMAND_PQ_SPACE = 8u,       // has_space,   :135-149
    DEMAND_USER = 16u,          // first id of a model's own predicates (cmb_condition_wait)
};

// struct cmb_process (include/cmb_process.h:116-123), the parts that act
struct Process {
    uint32_t pc;                // resume point (the coroutine's saved stack pointer)
    uint32_t status;
    uint32_t kind;              // which body (the reference's function pointer)
    int32_t  prio;
    uint32_t ctx;               // the reference's void *context: whatever index the model likes
    uint32_t awaits;            // list heads, NIL = empty
    uint32_t waiters;
    uint32_t holds;
    uint64_t hold_handle;
    uint64_t guard_key;
    int64_t  exit_value;
    uint64_t fr[3];             // locals of the blocking library call in progress (cmi_pool_acquire_inner's)
    double   f[2];              // body locals that live across blocking calls
    uint64_t u[2];
};

constexpr uint32_t GUARD_INLINE_EXP = 2u;               // 4 waiters inline, then the arena
constexpr uint32_t FEL_INLINE_EXP = 3u;                 // the reference starts its event list at 2^3 (src/cmb_event.c:47)
constexpr uint32_t HOLDERS_INLINE_EXP = 3u;

// struct cmb_resourceguard (include/cmb_resourceguard.h): the wait list of one resource
struct resourceguard {
    HashHeap<GuardOrder> heap;
    void    *owner;             // the resource the demands are asked of
    uint32_t observers[2];      // guards registered with cmb_resourceguard_register (addresses kept in Sim), 0 = none
    Tag      store[(1u << GUARD_INLINE_EXP) + 1u];
};

// struct cmb_objectqueue (include/cmb_objectqueue.h): FIFO of 64-bit payloads (the reference queues void *)
struct objectqueue {
    resourceguard front, rear;  // getters wait at the front guard, putters at the rear (src/cmb_objectqueue.c:54-113)
    uint64_t *ring;             // power-of-two ring, grown from the arena
    uint64_t  ring_inline[8];
    uint32_t  ring_exp, head;
    uint64_t  length, capacity;
    uint32_t  recording;
    TimeWeighted history;       // cmb_objectqueue_recording_start: length over time, folded on the fly
};

// struct cmb_resourcepool (include/cmb_resourcepool.h)
struct resourcepool {
    resourceguard guard;
    HashHeap<HolderOrder> holders;      // key = process index + 1, arg = amount held
    Tag      holder_store[(1u << HOLDERS_INLINE_EXP) + 1u];
    uint64_t capacity, in_use;
    uint32_t recording;
    TimeWeighted history;
};

// struct cmb_resource (include/cmb_resource.h): the binary semaphore
struct resource {
    resourceguard guard;
    uint32_t holder;            // process index, NIL = free
    uint32_t recording;
    TimeWeighted history;       // 1 while held, 0 while free
};

// struct cmb_buffer (include/cmb_buffer.h): an amount between 0 and capacity, put and got in parts
struct buffer {
    resourceguard front, rear;  // getters wait at the front guard, putters at the rear
    uint64_t level, capacity;
    uint32_t recording;
    TimeWeighted history;
};

// struct cmb_priorityqueue (include/cmb_priorityqueue.h): objects ordered by priority, then FIFO; handles = keys
struct priorityqueue {
    resourceguard front, rear;
    HashHeap<PrioOrder> queue;  // tag.d carries the object (64 bits), tag.prio its priority
    Tag      store[9];
    uint64_t capacity;
    uint32_t recording;
    TimeWeighted history;
};

// struct cmb_condition (include/cmb_condition.h): a guard whose demands are the model's own predicates
struct condition {
    resourceguard guard;
};

// What a model hands the engine: its process bodies, its own events and its own predicates.
//   void process(Sim &, uint32_t me, uint32_t kind, int64_t sig);
//   void event(Sim &, uint32_t action, uint32_t subject, int64_t arg);
//   bool demand(Sim &, uint32_t id, uint32_t pid, int32_t ctx);
// (static dispatch: the kernel is instantiated per model type, nothing is called through a pointer)

struct Sim {
    using queue_type = objectqueue;     // what a model template declares its queues as (cmb_static.cuh has another)
    using recorded_queue_type = objectqueue;    // ... a queue whose length history will be switched on
    using buffer_type = buffer;
    using recorded_buffer_type = buffer;
    Sfc64          rng;
    const ZigHot  *hot;
    double         now;
    uint32_t       status;
    uint32_t       current;             // the process whose body is running (cmb_process_current), NIL outside
    uint64_t       current_event;       // cmb_event_current
    uint64_t       guard_seq;           // enqueue_seq, src/cmb_resourceguard.c:64
    uint64_t       pops;
    Arena          arena;
    HashHeap<EventOrder> fel;
    Tag            fel_store[(1u << FEL_INLINE_EXP) + 1u];
    Process       *proc;
    uint32_t       nproc, proc_cap;
    uint32_t       proc_free;           // LIFO of records given back with process_destroy (linked through Process::pc)
    Process        proc_inline[4];
    Node          *node;
    uint32_t       node_cap, node_top, node_free;
    Node           node_inline[8];
    uint64_t      *scratch;
    uint32_t       scratch_cap;
    // The blocking call a process body ended on.  The body only RECORDS it and returns; the dispatcher carries it out
    // right after, in code that every lane of the warp passes together - the event-list insert, the wait-list insert
    // and the variate draw are the expensive parts of an event, and lanes whose trials are in different process bodies
    // share them this way.  Nothing happens between the body's return and the command, so the order of key issues and
    // random draws is the reference's.
    FlipCache      flips;               // cmb_random_flip's 64 cached coin flips (src/cmb_random.c: one draw serves 64 calls)
    uint32_t       fel_high;            // the deepest the event list was at a pop (what the oracle calls max_fel)
    uint32_t       cmd;
    uint32_t       cmd_sample;          // CMD_HOLD_SAMPLED: which of the model's samplers draws the duration
    uint32_t       cmd_demand;
    int32_t        cmd_ctx;
    double         cmd_value;           // hold: the duration (or the mean of the exponential to draw); exit: unused
    int64_t        cmd_exit;
    resourceguard *cmd_guard;

    // ---------------------------------------------------------------- set-up
    CMB_FN void init(uint64_t seed, const ZigHot *tables, const Arena &a)
    {
        rng.seed(seed);                                 // cmb_random_initialize
        hot = tables;
        now = 0.0;                                      // cmb_event_queue_initialize(0.0)
        status = 0u;
        current = NIL;
        current_event = 0u;
        guard_seq = 0u;
        pops = 0u;
        fel_high = 0u;
        arena = a;
        fel.init(fel_store, FEL_INLINE_EXP);
        proc = proc_inline;
        nproc = 0u;
        proc_cap = 4u;
        proc_free = NIL;
        node = node_inline;
        node_cap = 8u;
        node_top = 0u;
        node_free = NIL;
        scratch = nullptr;
        scratch_cap = 0u;
        cmd = 0u;
        flips.bits = 0u;
        flips.pos = 0u;
    }

    // ---------------------------------------------------------------- node pool
    CMB_FN_NOINLINE uint32_t node_alloc()
    {
        if (node_free != NIL) {
            const uint32_t n = node_free;
            node_free = node[n].next;
            return n;
        }
        if (node_top == node_cap) {
            Node *bigger = (Node *)arena.alloc((uint64_t)(2u * node_cap) * sizeof(Node));
            if (bigger == nullptr) {
                status |= TRIAL_ERR_ARENA;
                return NIL;
            }
            for (uint32_t i = 0u; i < node_top; i++) bigger[i] = node[i];
            node = bigger;
            node_cap *= 2u;
        }
        return node_top++;
    }

    CMB_FN void node_release(uint32_t n)
    {
        node[n].next = node_free;
        node_free = n;
    }

    CMB_FN void list_push(uint32_t &head, uint32_t a, uint64_t b)   // cmi_slist_push: to the front
    {
        const uint32_t n = node_alloc();
        if (n == NIL) return;
        node[n].a = a;
        node[n].b = b;
        node[n].next = head;
        head = n;
    }

    // remove the first node matching (a, b); any_b = match on a alone.  The list order is otherwise kept.
    CMB_FN_NOINLINE bool list_remove(uint32_t &head, uint32_t a, uint64_t b, bool any_b)
    {
        uint32_t prev = NIL;
        for (uint32_t n = head; n != NIL; prev = n, n = node[n].next) {
            if (node[n].a == a && (any_b || node[n].b == b)) {
                if (prev == NIL) head = node[n].next;
                else node[prev].next = node[n].next;
                node_release(n);
                return true;
            }
        }
        return false;
    }

    // ---------------------------------------------------------------- events (src/cmb_event.c)
    CMB_FN uint64_t schedule(uint32_t act, uint32_t subj, int64_t arg, double t, int64_t prio)     // :123-140
    {
        const uint64_t key = fel.enqueue(arena, 0u, t, (int32_t)prio, subj, act, (int32_t)arg, NIL);
        if (key == 0u) status |= TRIAL_ERR_ARENA;
        return key;
    }

    // wake_event_waiters, :200-221: the list is walked from its head (the latest waiter first)
    CMB_FN_NOINLINE void wake_waiter_list(uint32_t head, int64_t sig)
    {
        uint32_t n = head;
        while (n != NIL) {
            const uint32_t pid = node[n].a;
            const uint32_t next = node[n].next;
            node_release(n);
            schedule(ACT_CMB_WAKE_EVENT, pid, sig, now, proc[pid].prio);
            n = next;
        }
    }

    CMB_FN_NOINLINE bool event_cancel(uint64_t handle)              // :285-302
    {
        const uint32_t at = fel.find(arena, handle);
        if (at == 0u) return false;
        const uint32_t waiters = fel.tag[at].link;
        (void)fel.remove(arena, handle);
        if (waiters != NIL) wake_waiter_list(waiters, CMB_PROCESS_CANCELLED);
        return true;
    }

    CMB_FN bool event_is_scheduled(uint64_t handle) { return fel.find(arena, handle) != 0u; }      // :145-150

    CMB_FN bool event_reschedule(uint64_t handle, double t)         // :308-324
    {
        const uint32_t at = fel.find(arena, handle);
        return at != 0u && fel.reprioritize(arena, handle, t, fel.tag[at].prio);
    }

    CMB_FN bool event_reprioritize(uint64_t handle, int64_t prio)   // :330-344
    {
        const uint32_t at = fel.find(arena, handle);
        return at != 0u && fel.reprioritize(arena, handle, fel.tag[at].d, (int32_t)prio);
    }

    // a reusable list of keys for the two-pass operations (pattern cancel, condition signal)
    CMB_FN_NOINLINE uint64_t *scratch_keys(uint32_t n)
    {
        if (n > scratch_cap) {
            uint32_t want = scratch_cap ? scratch_cap : 8u;
            while (want < n) want *= 2u;
            uint64_t *bigger = (uint64_t *)arena.alloc((uint64_t)want * sizeof(uint64_t));
            if (bigger == nullptr) {
                status |= TRIAL_ERR_ARENA;
                return nullptr;
            }
            scratch = bigger;
            scratch_cap = want;
        }
        return scratch;
    }

    // cmb_event_pattern_cancel(ANY, subject, ANY), :385-425: the matches are collected in heap-array order first and
    // cancelled in a second pass (the keys of the CANCELLED notifications depend on that order).  Events a model
    // schedules itself (actions >= ACT_CMB_USER) carry subjects of the model's own choosing and are not touched.
    CMB_FN_NOINLINE void cancel_events_of(uint32_t subj)
    {
        uint32_t n = 0u;
        for (uint32_t k = 1u; k <= fel.count; k++) n += (fel.tag[k].subj == subj && fel.tag[k].act < ACT_CMB_USER) ? 1u : 0u;
        if (n == 0u) return;
        uint64_t *hit = scratch_keys(n);
        if (hit == nullptr) return;
        uint32_t m = 0u;
        for (uint32_t k = 1u; k <= fel.count; k++) {
            if (fel.tag[k].subj == subj && fel.tag[k].act < ACT_CMB_USER) hit[m++] = fel.tag[k].key;
        }
        for (uint32_t k = 0u; k < m; k++) (void)event_cancel(hit[k]);
    }

    // ---------------------------------------------------------------- processes (src/cmb_process.c)
    // cmb_process_create + cmb_process_initialize: returns the process index the other calls take
    CMB_FN_NOINLINE uint32_t process_create(uint32_t kind, int64_t prio, uint32_t ctx)
    {
        uint32_t pid;
        if (proc_free != NIL) {                         // a record a finished process gave back (cmb_process_destroy)
            pid = proc_free;
            proc_free = proc[pid].pc;
        }
        else {
            if (nproc == proc_cap) {
                Process *bigger = (Process *)arena.alloc((uint64_t)(2u * proc_cap) * sizeof(Process));
                if (bigger == nullptr) {
                    // no memory: the trial is void from here (flagged; the dispatcher stops it at its next step).  Hand back
                    // an index that exists, so that model code which goes on to touch "the new process" stays in bounds.
                    status |= TRIAL_ERR_ARENA;
                    return nproc - 1u;
                }
                for (uint32_t i = 0u; i < nproc; i++) bigger[i] = proc[i];
                proc = bigger;
                proc_cap *= 2u;
            }
            pid = nproc++;
        }
        Process &p = proc[pid];
        p.pc = 0u;
        p.status = PROC_CREATED;
        p.kind = kind;
        p.prio = (int32_t)prio;
        p.ctx = ctx;
        p.awaits = p.waiters = p.holds = NIL;
        p.hold_handle = p.guard_key = 0u;
        p.exit_value = 0;
        p.fr[0] = p.fr[1] = p.fr[2] = 0u;
        p.f[0] = p.f[1] = 0.0;
        p.u[0] = p.u[1] = 0u;
        return pid;
    }

    // cmb_process_terminate + cmb_process_destroy of a process that is FINISHED (or was never started): its record may be
    // handed out again by the next cmb_process_create.  Models that create a process per arrival call this when they are
    // done with its exit value, as the reference's frees its struct (test/test_condition.c:441-446).
    CMB_FN void process_destroy(uint32_t pid)
    {
        proc[pid].status = PROC_FINISHED;
        proc[pid].pc = proc_free;
        proc_free = pid;
    }

    CMB_FN bool process_reserve(uint32_t n)             // room for n processes in one step
    {
        while (proc_cap < n) {
            Process *bigger = (Process *)arena.alloc((uint64_t)(2u * proc_cap) * sizeof(Process));
            if (bigger == nullptr) {
                status |= TRIAL_ERR_ARENA;
                return false;
            }
            for (uint32_t i = 0u; i < nproc; i++) bigger[i] = proc[i];
            proc = bigger;
            proc_cap *= 2u;
        }
        return true;
    }

    CMB_FN void process_start(uint32_t pid)             // :127-135: a FINISHED process may be started again
    {
        if (status & TRIAL_ERR_ARENA) return;           // a void trial (a container could not grow) schedules nothing more
        schedule(ACT_CMB_START, pid, 0, now, proc[pid].prio);
    }

    CMB_FN void await_push(uint32_t pid, uint32_t type, uint64_t ref) { list_push(proc[pid].awaits, type, ref); }

    // cmb_process_hold, :262-285 (first half) / cmb_process_timer_add, :316-333
    CMB_FN void hold_begin(uint32_t pid, double dur)
    {
        if (dur < 0.0) status |= TRIAL_ERR_NEGATIVE_HOLD;
        Process &p = proc[pid];
        p.hold_handle = schedule(ACT_CMB_WAKE_TIME, pid, CMB_PROCESS_SUCCESS, __dadd_rn(now, dur), p.prio);
        await_push(pid, AWAIT_TIME, p.hold_handle);
    }

    CMB_FN int64_t hold_end(uint32_t pid, int64_t sig)  // :274-284: interrupted -> drop the wake-up
    {
        if (sig != CMB_PROCESS_SUCCESS) {
            Process &p = proc[pid];
            (void)list_remove(p.awaits, AWAIT_TIME, p.hold_handle, false);
            (void)event_cancel(p.hold_handle);
        }
        return sig;
    }

    CMB_FN uint64_t timer_add(uint32_t pid, double dur, int64_t sig)        // :316-333
    {
        const uint64_t h = schedule(ACT_CMB_WAKE_TIME, pid, sig, __dadd_rn(now, dur), proc[pid].prio);
        await_push(pid, AWAIT_TIME, h);
        return h;
    }

    CMB_FN bool timer_cancel(uint32_t pid, uint64_t handle)                 // :338-349
    {
        (void)list_remove(proc[pid].awaits, AWAIT_TIME, handle, false);
        return event_cancel(handle);
    }

    CMB_FN_NOINLINE void timers_clear(uint32_t pid)                         // :354-381
    {
        uint32_t prev = NIL, n = proc[pid].awaits;
        while (n != NIL) {
            const uint32_t next = node[n].next;
            if (node[n].a == AWAIT_TIME) {
                const uint64_t handle = node[n].b;
                if (prev == NIL) proc[pid].awaits = next;
                else node[prev].next = next;
                node_release(n);
                (void)event_cancel(handle);
            }
            else {
                prev = n;
            }
            n = next;
        }
    }

    CMB_FN void timer_set(uint32_t pid, double dur, int64_t sig)            // include/cmb_process.h: clear, then add
    {
        timers_clear(pid);
        (void)timer_add(pid, dur, sig);
    }

    // cmi_process_cancel_awaiteds, :581-620
    CMB_FN_NOINLINE void cancel_awaiteds(uint32_t pid)
    {
        while (proc[pid].awaits != NIL) {
            const uint32_t n = proc[pid].awaits;
            const uint32_t type = node[n].a;
            const uint64_t ref = node[n].b;
            proc[pid].awaits = node[n].next;
            node_release(n);
            if (type == AWAIT_TIME) {
                (void)event_cancel(ref);
            }
            else if (type == AWAIT_PROCESS) {           // cmi_process_remove_waiter, :529-551
                (void)list_remove(proc[(uint32_t)ref].waiters, pid, 0u, true);
            }
            else if (type == AWAIT_EVENT) {             // cmi_event_remove_waiter, src/cmb_event.c:486-508
                const uint32_t at = fel.find(arena, ref);
                if (at != 0u) (void)list_remove(fel.tag[at].link, pid, 0u, true);
            }
            // AWAIT_RESOURCE: cmb_resourceguard_remove looks the entry up by process ADDRESS while entries are keyed
            // by sequence number, so it never finds one (SURVEY.md quirk 2); the waiter removes its own entry with
            // the right key when it resumes (guard_wait_end).
        }
        cancel_events_of(pid);
    }

    CMB_FN void interrupt(uint32_t pid, int64_t sig, int64_t pri)           // :653-666
    {
        schedule(ACT_CMB_WAKE_INTERRUPT, pid, sig, now, pri);
    }

    CMB_FN void resume(uint32_t pid, int64_t sig)                           // :751-760
    {
        schedule(ACT_CMB_RESUME, pid, sig, now, proc[pid].prio);
    }

    CMB_FN_NOINLINE void wake_process_waiters(uint32_t pid, int64_t sig)    // :485-505
    {
        uint32_t n = proc[pid].waiters;
        proc[pid].waiters = NIL;
        while (n != NIL) {
            const uint32_t w = node[n].a;
            const uint32_t next = node[n].next;
            node_release(n);
            schedule(ACT_CMB_WAKE_PROCESS, w, sig, now, proc[w].prio);
            n = next;
        }
    }

    CMB_FN void wait_process_begin(uint32_t pid, uint32_t awaited)          // :428-452
    {
        await_push(pid, AWAIT_PROCESS, awaited);
        list_push(proc[awaited].waiters, pid, 0u);
    }

    CMB_FN void wait_event_begin(uint32_t pid, uint64_t handle)             // :461-483
    {
        const uint32_t at = fel.find(arena, handle);
        if (at == 0u) return;
        list_push(fel.tag[at].link, pid, 0u);
        await_push(pid, AWAIT_EVENT, handle);
    }

    // ---------------------------------------------------------------- guards (src/cmb_resourceguard.c)
    CMB_FN void guard_init(resourceguard &g, void *owner)
    {
        g.heap.init(g.store, GUARD_INLINE_EXP);
        g.owner = owner;
        g.observers[0] = g.observers[1] = 0u;
    }

    // what CMB_GUARD_WAIT_ records for the dispatcher (the static tier, cmb_static.cuh, registers the waiter at once instead)
    CMB_FN void guard_wait_cmd(resourceguard &g, uint32_t, uint32_t demand, int32_t ctx)
    {
        cmd_guard = &g;
        cmd_demand = demand;
        cmd_ctx = ctx;
        cmd = CMD_GUARD_WAIT;
    }

    CMB_FN void guard_wait_begin(resourceguard &g, uint32_t pid, uint32_t demand, int32_t ctx)     // :125-152
    {
        Process &p = proc[pid];
        p.guard_key = ++guard_seq;
        if (g.heap.enqueue(arena, p.guard_key, now, p.prio, pid, demand, ctx, NIL) == 0u) status |= TRIAL_ERR_ARENA;
        await_push(pid, AWAIT_RESOURCE, (uint64_t)(uintptr_t)&g);
    }

    CMB_FN int64_t guard_wait_end(resourceguard &g, uint32_t pid, int64_t sig)                     // :153-162
    {
        Process &p = proc[pid];
        if (sig != CMB_PROCESS_SUCCESS) (void)g.heap.remove(arena, p.guard_key);
        (void)list_remove(p.awaits, AWAIT_RESOURCE, (uint64_t)(uintptr_t)&g, false);
        return sig;
    }

};

// built-in demands, evaluated against the guard's owner
CMB_FN bool builtin_demand(uint32_t demand, void *owner)
{
    switch (demand) {
    case DEMAND_QUEUE_CONTENT: return ((objectqueue *)owner)->length > 0u;
    case DEMAND_QUEUE_SPACE:   return ((objectqueue *)owner)->length < ((objectqueue *)owner)->capacity;
    case DEMAND_POOL_AVAILABLE: return ((resourcepool *)owner)->capacity - ((resourcepool *)owner)->in_use > 0u;
    case DEMAND_RESOURCE_FREE: return ((resource *)owner)->holder == NIL;
    case DEMAND_BUFFER_CONTENT: return ((buffer *)owner)->level > 0u;
    case DEMAND_BUFFER_SPACE:  return ((buffer *)owner)->level < ((buffer *)owner)->capacity;
    case DEMAND_PQ_CONTENT:    return ((priorityqueue *)owner)->queue.count > 0u;
    case DEMAND_PQ_SPACE:      return ((priorityqueue *)owner)->queue.count < ((priorityqueue *)owner)->capacity;
    }
    return false;
}

// cmb_resourceguard_signal, src/cmb_resourceguard.c:202-242: wake at most the head, then poke the observers
template <class Model>
CMB_FN_NOINLINE bool guard_signal(Sim &sim, Model &m, resourceguard &g)
{
    bool woke = false;
    if (g.heap.count > 0u) {
        const Tag &head = g.heap.tag[1];
        const uint32_t pid = head.subj;
        const bool ok = head.act >= DEMAND_USER ? m.demand(sim, (uint32_t)head.act, pid, head.arg)
                                                : builtin_demand(head.act, g.owner);
        if (ok) {
            (void)g.heap.dequeue();
            sim.schedule(ACT_CMB_WAKE_RESOURCE, pid, CMB_PROCESS_SUCCESS, sim.now, sim.proc[pid].prio);
            woke = true;
        }
    }
    for (int k = 0; k < 2; k++) {
        if (g.observers[k] != 0u) {
            resourceguard *obs = (resourceguard *)((unsigned char *)&m + g.observers[k]);
            (void)guard_signal(sim, m, *obs);
        }
    }
    return woke;
}

// cmb_resourceguard_register: `observer` (a guard inside the model struct) is signalled whenever `g` is
template <class Model>
CMB_FN void guard_register(Model &m, resourceguard &g, resourceguard &observer)
{
    const uint32_t off = (uint32_t)((unsigned char *)&observer - (unsigned char *)&m);
    if (g.observers[0] == 0u) g.observers[0] = off;
    else g.observers[1] = off;
}

// ------------------------------------------------------------------------------------------------ objectqueue
CMB_FN void objectqueue_initialize(Sim &sim, objectqueue &q, uint64_t capacity)    // src/cmb_objectqueue.c:54-113
{
    sim.guard_init(q.front, &q);
    sim.guard_init(q.rear, &q);
    q.ring = q.ring_inline;
    q.ring_exp = 3u;
    q.head = 0u;
    q.length = 0u;
    q.capacity = capacity;
    q.recording = 0u;
}

CMB_FN void objectqueue_recording_start(Sim &sim, objectqueue &q)                  // :161-177
{
    q.recording = 1u;
    q.history.start();
    q.history.sample((double)q.length, sim.now);
}

CMB_FN void objectqueue_recording_stop(Sim &sim, objectqueue &q)
{
    if (q.recording) q.history.sample((double)q.length, sim.now);
    q.recording = 0u;
}

CMB_FN_NOINLINE bool objectqueue_push(Sim &sim, objectqueue &q, uint64_t obj)
{
    if (q.length == ((uint64_t)1u << q.ring_exp)) {     // the linked list of the reference has no such limit: grow
        const uint32_t old_cap = 1u << q.ring_exp;
        uint64_t *bigger = (uint64_t *)sim.arena.alloc((uint64_t)(2u * old_cap) * sizeof(uint64_t));
        if (bigger == nullptr) {
            sim.status |= TRIAL_ERR_ARENA;
            return false;
        }
        for (uint32_t i = 0u; i < old_cap; i++) bigger[i] = q.ring[(q.head + i) & (old_cap - 1u)];
        q.ring = bigger;
        q.head = 0u;
        q.ring_exp++;
    }
    q.ring[(q.head + (uint32_t)q.length) & ((1u << q.ring_exp) - 1u)] = obj;
    q.length++;
    return true;
}

// the non-blocking halves of cmb_objectqueue_put / _get (src/cmb_objectqueue.c:262-314, 203-260); the CMB_* macros
// wrap them in the reference's "loop { try; else wait at the guard }"
template <class Model>
CMB_FN bool objectqueue_try_put(Sim &sim, Model &m, objectqueue &q, uint64_t obj)
{
    if (q.length >= q.capacity) return false;
    if (!objectqueue_push(sim, q, obj)) return true;    // arena exhausted: flagged, do not block forever
    if (q.recording) q.history.sample((double)q.length, sim.now);
    (void)guard_signal(sim, m, q.front);
    return true;
}

template <class Model>
CMB_FN bool objectqueue_try_get(Sim &sim, Model &m, objectqueue &q, uint64_t &obj)
{
    if (q.length == 0u) return false;
    obj = q.ring[q.head];
    q.head = (q.head + 1u) & ((1u << q.ring_exp) - 1u);
    q.length--;
    if (q.recording) q.history.sample((double)q.length, sim.now);
    (void)guard_signal(sim, m, q.rear);
    return true;
}

// ------------------------------------------------------------------------------------------------ resourcepool
CMB_FN void resourcepool_initialize(Sim &sim, resourcepool &rp, uint64_t capacity) // src/cmb_resourcepool.c:139-170
{
    sim.guard_init(rp.guard, &rp);
    rp.holders.init(rp.holder_store, HOLDERS_INLINE_EXP);
    rp.capacity = capacity;
    rp.in_use = 0u;
    rp.recording = 0u;
}

CMB_FN void resourcepool_recording_start(Sim &sim, resourcepool &rp)
{
    rp.recording = 1u;
    rp.history.start();
    rp.history.sample((double)rp.in_use, sim.now);
}

CMB_FN void resourcepool_recording_stop(Sim &sim, resourcepool &rp)
{
    if (rp.recording) rp.history.sample((double)rp.in_use, sim.now);
    rp.recording = 0u;
}

CMB_FN void pool_sample(Sim &sim, resourcepool &rp)
{
    if (rp.recording) rp.history.sample((double)rp.in_use, sim.now);
}

CMB_FN uint64_t resourcepool_held_by_process(Sim &sim, resourcepool &rp, uint32_t pid)     // :296-309
{
    const uint32_t k = rp.holders.find(sim.arena, (uint64_t)pid + 1u);
    return k ? (uint64_t)(uint32_t)rp.holders.tag[k].arg : 0u;
}

CMB_FN_NOINLINE void pool_update_record(Sim &sim, resourcepool &rp, uint32_t pid, uint64_t amount)   // update_record, :324-355
{
    const uint32_t k = rp.holders.find(sim.arena, (uint64_t)pid + 1u);
    if (k != 0u) {
        rp.holders.tag[k].arg += (int32_t)amount;
    }
    else {
        sim.list_push(sim.proc[pid].holds, HOLD_POOL, (uint64_t)(uintptr_t)&rp);
        if (rp.holders.enqueue(sim.arena, (uint64_t)pid + 1u, 0.0, sim.proc[pid].prio, pid, 0u, (int32_t)amount, NIL) == 0u)
            sim.status |= TRIAL_ERR_ARENA;
    }
}

// cmi_pool_acquire_inner up to its wait (:362-497): true = satisfied (SUCCESS), false = the caller must wait at the guard.
// fr[0] = initially held, fr[1] = remaining claim.
template <class Model>
CMB_FN_NOINLINE bool pool_acquire_step(Sim &sim, Model &m, resourcepool &rp, uint32_t pid, bool preempt)
{
    Process &p = sim.proc[pid];
    uint64_t rem = p.fr[1];
    const uint64_t available = rp.capacity - rp.in_use;
    if (available >= rem) {
        rp.in_use += rem;
        pool_sample(sim, rp);
        pool_update_record(sim, rp, pid, rem);
        (void)guard_signal(sim, m, rp.guard);
        return true;
    }
    if (available > 0u) {
        rp.in_use += available;
        pool_sample(sim, rp);
        rem -= available;
        pool_update_record(sim, rp, pid, available);
    }
    if (preempt) {
        while (rp.holders.count > 0u && rp.holders.tag[1].prio < sim.proc[pid].prio) {
            (void)rp.holders.dequeue();
            const uint32_t victim = rp.holders.tag[0].subj;
            const uint64_t loot = (uint64_t)(uint32_t)rp.holders.tag[0].arg;
            (void)sim.list_remove(sim.proc[victim].holds, HOLD_POOL, (uint64_t)(uintptr_t)&rp, false);
            sim.interrupt(victim, CMB_PROCESS_PREEMPTED, sim.proc[victim].prio);
            if (loot < rem) {
                pool_update_record(sim, rp, pid, loot);
                rem -= loot;
            }
            else {
                pool_update_record(sim, rp, pid, rem);
                rp.in_use -= loot - rem;
                pool_sample(sim, rp);
                (void)guard_signal(sim, m, rp.guard);
                sim.proc[pid].fr[1] = 0u;
                return true;
            }
        }
    }
    sim.proc[pid].fr[1] = rem;
    return false;
}

// the tail of cmi_pool_acquire_inner after an unsuccessful wait (:499-531): roll back to the holding at the call
template <class Model>
CMB_FN_NOINLINE void pool_acquire_rollback(Sim &sim, Model &m, resourcepool &rp, uint32_t pid, int64_t sig)
{
    if (sig == CMB_PROCESS_PREEMPTED) return;           // thrown out: returns empty-handed, nothing to unwind
    const uint64_t initially = sim.proc[pid].fr[0];
    const uint64_t key = (uint64_t)pid + 1u;
    if (initially > 0u) {
        const uint32_t k = rp.holders.find(sim.arena, key);            // reset_holder
        uint64_t surplus = 0u;
        if (k != 0u) {
            surplus = (uint64_t)(uint32_t)rp.holders.tag[k].arg - initially;
            rp.holders.tag[k].arg = (int32_t)initially;
        }
        rp.in_use -= surplus;
        pool_sample(sim, rp);
        (void)guard_signal(sim, m, rp.guard);
    }
    else {
        const uint64_t holds_now = resourcepool_held_by_process(sim, rp, pid);
        rp.in_use -= holds_now;
        pool_sample(sim, rp);
        if (rp.holders.remove(sim.arena, key)) {
            (void)sim.list_remove(sim.proc[pid].holds, HOLD_POOL, (uint64_t)(uintptr_t)&rp, false);
        }
    }
}

// cmb_resourcepool_release, :561-605
template <class Model>
CMB_FN_NOINLINE void resourcepool_release(Sim &sim, Model &m, resourcepool &rp, uint32_t pid, uint64_t amount)
{
    const uint64_t key = (uint64_t)pid + 1u;
    const uint32_t k = rp.holders.find(sim.arena, key);
    if (k != 0u && (uint64_t)(uint32_t)rp.holders.tag[k].arg == amount) {
        (void)rp.holders.remove(sim.arena, key);
        (void)sim.list_remove(sim.proc[pid].holds, HOLD_POOL, (uint64_t)(uintptr_t)&rp, false);
    }
    else if (k != 0u) {
        rp.holders.tag[k].arg -= (int32_t)amount;
    }
    rp.in_use -= amount;
    pool_sample(sim, rp);
    (void)guard_signal(sim, m, rp.guard);
}

// pool_drop_holder, :98-121 (a stopped or exiting holder)
template <class Model>
CMB_FN_NOINLINE void pool_drop_holder(Sim &sim, Model &m, resourcepool &rp, uint32_t pid)
{
    const uint64_t key = (uint64_t)pid + 1u;
    const uint32_t k = rp.holders.find(sim.arena, key);
    if (k != 0u) {
        rp.in_use -= (uint64_t)(uint32_t)rp.holders.tag[k].arg;
        (void)rp.holders.remove(sim.arena, key);        // (no history sample here: resourcepool_drop_holder takes none)
        (void)guard_signal(sim, m, rp.guard);
    }
}

// cmb_process_priority_set, src/cmb_process.c:150-198: the process' events move in the event list, its records in the
// pools it holds from are reshuffled (reprioritize_holder, src/cmb_resourcepool.c:127-137).  An entry in a guard's wait list
// is NOT found - the reference looks it up by process address while entries are keyed by sequence number (SURVEY.md quirk 2).
CMB_FN_NOINLINE void process_priority_set(Sim &sim, uint32_t pid, int64_t pri)
{
    sim.proc[pid].prio = (int32_t)pri;
    for (uint32_t n = sim.proc[pid].awaits; n != NIL; n = sim.node[n].next) {
        if (sim.node[n].a == AWAIT_TIME) (void)sim.event_reprioritize(sim.node[n].b, pri);
    }
    for (uint32_t n = sim.proc[pid].holds; n != NIL; n = sim.node[n].next) {
        if (sim.node[n].a == HOLD_POOL) {
            resourcepool &rp = *(resourcepool *)(uintptr_t)sim.node[n].b;
            (void)rp.holders.reprioritize(sim.arena, (uint64_t)pid + 1u, 0.0, (int32_t)pri);
        }
    }
}

// ------------------------------------------------------------------------------------------------ resource
CMB_FN void resource_initialize(Sim &sim, resource &r)
{
    sim.guard_init(r.guard, &r);
    r.holder = NIL;
    r.recording = 0u;
}

CMB_FN void resource_sample(Sim &sim, resource &r)                                 // record_sample, src/cmb_resource.c
{
    if (r.recording) r.history.sample(r.holder != NIL ? 1.0 : 0.0, sim.now);
}

CMB_FN void resource_recording_start(Sim &sim, resource &r)
{
    r.recording = 1u;
    r.history.start();
    r.history.sample(r.holder != NIL ? 1.0 : 0.0, sim.now);
}

CMB_FN void resource_recording_stop(Sim &sim, resource &r)
{
    resource_sample(sim, r);
    r.recording = 0u;
}

CMB_FN void resource_grab(Sim &sim, resource &r, uint32_t pid)                     // :182-189
{
    r.holder = pid;
    sim.list_push(sim.proc[pid].holds, HOLD_RESOURCE, (uint64_t)(uintptr_t)&r);
}

template <class Model>
CMB_FN void resource_release(Sim &sim, Model &m, resource &r, uint32_t pid)        // :234-250
{
    (void)sim.list_remove(sim.proc[pid].holds, HOLD_RESOURCE, (uint64_t)(uintptr_t)&r, false);
    r.holder = NIL;
    resource_sample(sim, r);
    (void)guard_signal(sim, m, r.guard);
}

// cmb_resource_preempt, :270-320, up to its polite branch: true = the caller holds the resource now
CMB_FN_NOINLINE bool resource_preempt_step(Sim &sim, resource &r, uint32_t pid)
{
    const uint32_t victim = r.holder;
    if (victim == NIL) {
        resource_grab(sim, r, pid);
        resource_sample(sim, r);
        return true;
    }
    if (sim.proc[pid].prio >= sim.proc[victim].prio) {
        (void)sim.list_remove(sim.proc[victim].holds, HOLD_RESOURCE, (uint64_t)(uintptr_t)&r, false);
        sim.cancel_awaiteds(pid);                       // sic: the CALLER's awaiteds (cmi_process_cancel_awaiteds(pp), :296)
        r.holder = NIL;
        sim.schedule(ACT_CMB_WAKE_PREEMPT, victim, CMB_PROCESS_PREEMPTED, sim.now, sim.proc[victim].prio);
        resource_grab(sim, r, pid);                     // no history sample: the resource stays occupied
        return true;
    }
    return false;                                       // wait politely: cmb_resource_acquire
}

// ------------------------------------------------------------------------------------------------ buffer
CMB_FN void buffer_initialize(Sim &sim, buffer &b, uint64_t capacity)              // src/cmb_buffer.c:45-75
{
    sim.guard_init(b.front, &b);
    sim.guard_init(b.rear, &b);
    b.level = 0u;
    b.capacity = capacity;
    b.recording = 0u;
}

CMB_FN void buffer_sample(Sim &sim, buffer &b)
{
    if (b.recording) b.history.sample((double)b.level, sim.now);
}

CMB_FN void buffer_recording_start(Sim &sim, buffer &b)
{
    b.recording = 1u;
    b.history.start();
    b.history.sample((double)b.level, sim.now);
}

CMB_FN void buffer_recording_stop(Sim &sim, buffer &b)
{
    buffer_sample(sim, b);
    b.recording = 0u;
}

// cmb_buffer_get up to its wait (:194-264): fr[1] = remaining claim, fr[2] = obtained so far.  true = satisfied.
template <class Model>
CMB_FN_NOINLINE bool buffer_get_step(Sim &sim, Model &m, buffer &b, uint32_t pid)
{
    uint64_t rem = sim.proc[pid].fr[1];
    if (b.level >= rem) {
        b.level -= rem;
        buffer_sample(sim, b);
        sim.proc[pid].fr[2] += rem;
        (void)guard_signal(sim, m, b.rear);
        if (b.level > 0u) (void)guard_signal(sim, m, b.front);         // leftovers for the next getter
        return true;
    }
    if (b.level > 0u) {
        const uint64_t grab = b.level;
        b.level = 0u;
        buffer_sample(sim, b);
        sim.proc[pid].fr[2] += grab;
        rem -= grab;
        (void)guard_signal(sim, m, b.rear);
    }
    sim.proc[pid].fr[1] = rem;
    (void)guard_signal(sim, m, b.rear);                 // once more before waiting (:241)
    return false;
}

// cmb_buffer_put up to its wait (:279-346): fr[1] = remaining to put.  true = everything is in.
template <class Model>
CMB_FN_NOINLINE bool buffer_put_step(Sim &sim, Model &m, buffer &b, uint32_t pid)
{
    uint64_t rem = sim.proc[pid].fr[1];
    if (b.capacity - b.level >= rem) {
        b.level += rem;
        buffer_sample(sim, b);
        sim.proc[pid].fr[1] = 0u;
        (void)guard_signal(sim, m, b.front);
        if (b.level < b.capacity) (void)guard_signal(sim, m, b.rear);
        return true;
    }
    if (b.level < b.capacity) {
        const uint64_t grab = b.capacity - b.level;
        b.level = b.capacity;
        buffer_sample(sim, b);
        rem -= grab;
        (void)guard_signal(sim, m, b.front);
    }
    sim.proc[pid].fr[1] = rem;
    (void)guard_signal(sim, m, b.front);
    return false;
}

// ------------------------------------------------------------------------------------------------ priorityqueue
CMB_FN void priorityqueue_initialize(Sim &sim, priorityqueue &q, uint64_t capacity)    // src/cmb_priorityqueue.c:56-117
{
    sim.guard_init(q.front, &q);
    sim.guard_init(q.rear, &q);
    q.queue.init(q.store, 3u);
    q.capacity = capacity;
    q.recording = 0u;
}

CMB_FN void priorityqueue_sample(Sim &sim, priorityqueue &q)
{
    if (q.recording) q.history.sample((double)q.queue.count, sim.now);
}

CMB_FN void priorityqueue_recording_start(Sim &sim, priorityqueue &q)
{
    q.recording = 1u;
    q.history.start();
    q.history.sample((double)q.queue.count, sim.now);
}

CMB_FN void priorityqueue_recording_stop(Sim &sim, priorityqueue &q)
{
    priorityqueue_sample(sim, q);
    q.recording = 0u;
}

template <class Model>
CMB_FN bool priorityqueue_try_put(Sim &sim, Model &m, priorityqueue &q, uint64_t obj, int64_t prio, uint64_t *handle)   // :237-284
{
    if (q.queue.count >= q.capacity) return false;
    const uint64_t h = q.queue.enqueue(sim.arena, 0u, __longlong_as_double((long long)obj), (int32_t)prio, NIL, 0u, 0, NIL);
    if (h == 0u) sim.status |= TRIAL_ERR_ARENA;
    if (handle != nullptr) *handle = h;
    priorityqueue_sample(sim, q);
    (void)guard_signal(sim, m, q.front);
    return true;
}

template <class Model>
CMB_FN bool priorityqueue_try_get(Sim &sim, Model &m, priorityqueue &q, uint64_t &obj)       // :189-235
{
    if (q.queue.count == 0u) return false;
    (void)q.queue.dequeue();
    obj = (uint64_t)__double_as_longlong(q.queue.tag[0].d);
    priorityqueue_sample(sim, q);
    (void)guard_signal(sim, m, q.rear);
    return true;
}

// cmb_priorityqueue_reprioritize, include/cmb_priorityqueue.h:170-180 (the tag's double is the object here: it stays)
CMB_FN void priorityqueue_reprioritize(Sim &sim, priorityqueue &q, uint64_t handle, int64_t prio)
{
    const uint32_t at = q.queue.find(sim.arena, handle);
    if (at != 0u) (void)q.queue.reprioritize(sim.arena, handle, q.queue.tag[at].d, (int32_t)prio);
}

// cmb_priorityqueue_position, :286-320: 1 = next to be taken, 0 = not in the queue
CMB_FN_NOINLINE uint64_t priorityqueue_position(Sim &sim, priorityqueue &q, uint64_t handle)
{
    const uint32_t at = q.queue.find(sim.arena, handle);
    if (at == 0u) return 0u;
    uint64_t ahead = 0u;
    for (uint32_t k = 1u; k <= q.queue.count; k++) {
        if (k != at && PrioOrder::before(q.queue.tag[k], q.queue.tag[at])) ahead++;
    }
    return ahead + 1u;
}

// ------------------------------------------------------------------------------------------------ condition
CMB_FN void condition_initialize(Sim &sim, condition &c) { sim.guard_init(c.guard, &c); }

// cmb_condition_signal, src/cmb_condition.c:120-167: every waiter whose predicate holds, in heap-array order; the
// woken entries are removed in a second pass
template <class Model>
CMB_FN_NOINLINE uint32_t condition_signal(Sim &sim, Model &m, condition &c)
{
    HashHeap<GuardOrder> &h = c.guard.heap;
    if (h.count == 0u) return 0u;
    uint64_t *hit = sim.scratch_keys(h.count);
    if (hit == nullptr) return 0u;
    uint32_t n = 0u;
    for (uint32_t k = 1u; k <= h.count; k++) {
        const uint32_t pid = h.tag[k].subj;
        if (m.demand(sim, (uint32_t)h.tag[k].act, pid, h.tag[k].arg)) {
            hit[n++] = h.tag[k].key;
            sim.schedule(ACT_CMB_WAKE_CONDITION, pid, CMB_PROCESS_SUCCESS, sim.now, sim.proc[pid].prio);
        }
    }
    for (uint32_t k = 0u; k < n; k++) (void)h.remove(sim.arena, hit[k]);
    return n;
}

// ------------------------------------------------------------------------------------------------ process end
// cmi_process_drop_resources, src/cmb_process.c:507-527: every held resource through its drop
template <class Model>
CMB_FN_NOINLINE void drop_resources(Sim &sim, Model &m, uint32_t pid)
{
    while (sim.proc[pid].holds != NIL) {
        const uint32_t n = sim.proc[pid].holds;
        const uint32_t kind = sim.node[n].a;
        void *res = (void *)(uintptr_t)sim.node[n].b;
        sim.proc[pid].holds = sim.node[n].next;
        sim.node_release(n);
        if (kind == HOLD_POOL) {
            pool_drop_holder(sim, m, *(resourcepool *)res, pid);
        }
        else if (kind == HOLD_RESOURCE) {               // resource_drop_holder, src/cmb_resource.c:45-56
            ((resource *)res)->holder = NIL;
            resource_sample(sim, *(resource *)res);
            (void)guard_signal(sim, m, ((resource *)res)->guard);
        }
    }
}

// cmb_process_exit / the body returning, :671-684
template <class Model>
CMB_FN_NOINLINE void process_exit(Sim &sim, Model &m, uint32_t pid, int64_t value)
{
    drop_resources(sim, m, pid);
    sim.cancel_awaiteds(pid);
    sim.wake_process_waiters(pid, CMB_PROCESS_SUCCESS);
    sim.proc[pid].status = PROC_FINISHED;
    sim.proc[pid].exit_value = value;
}

// cmb_process_stop, :698-723
template <class Model>
CMB_FN_NOINLINE void process_stop(Sim &sim, Model &m, uint32_t pid, int64_t value)
{
    if (sim.proc[pid].status != PROC_RUNNING) return;
    sim.proc[pid].status = PROC_FINISHED;
    sim.proc[pid].exit_value = value;
    sim.cancel_awaiteds(pid);
    drop_resources(sim, m, pid);
    sim.wake_process_waiters(pid, CMB_PROCESS_STOPPED);
}

// CMB_PROCESS_HOLD_SAMPLED(id): the duration is `m.sample(sim, id)`, drawn by the dispatcher (a model without samplers has none)
template <class Model, class S, class = void>
struct ModelSampler {
    static CMB_FN double draw(Model &, S &, uint32_t) { return 0.0; }
};
template <class Model, class S>
struct ModelSampler<Model, S, decltype((void)std::declval<Model &>().sample(std::declval<S &>(), 0u))> {
    static CMB_FN double draw(Model &m, S &sim, uint32_t id) { return m.sample(sim, id); }
};

// ------------------------------------------------------------------------------------------------ dispatcher
// cmb_event_queue_execute, src/cmb_event.c:259-267 + cmb_event_execute_next, :229-252
template <class Model, bool TRACE>
CMB_FN_NOINLINE void execute(Sim &sim, Model &m, uint64_t trace_cap, uint64_t *trace_key, double *trace_time)
{
    for (;;) {
        // a trial whose containers could not grow (workspace too small) is void: stop it where it stands, flagged
        if (sim.status & TRIAL_ERR_ARENA) return;
        if (sim.fel.count > sim.fel_high) sim.fel_high = sim.fel.count;        // the deepest the event list was when an event was taken
        if (!sim.fel.dequeue()) return;
        const Tag ev = sim.fel.tag[0];
        sim.now = ev.d;
        sim.current_event = ev.key;
        if (TRACE) {
            if (sim.pops < trace_cap) {
                trace_key[sim.pops] = ev.key;
                trace_time[sim.pops] = sim.now;
            }
        }
        sim.pops++;
        if (ev.link != NIL) sim.wake_waiter_list(ev.link, CMB_PROCESS_SUCCESS);     // waiters first, :243-249
        const uint32_t pid = ev.subj;
        bool run = false;
        switch (ev.act) {
        case ACT_CMB_START:
            sim.proc[pid].status = PROC_RUNNING;
            sim.proc[pid].pc = 0u;
            run = true;
            break;
        case ACT_CMB_WAKE_TIME:
            (void)sim.list_remove(sim.proc[pid].awaits, AWAIT_TIME, ev.key, false);
            run = true;
            break;
        case ACT_CMB_WAKE_RESOURCE:
        case ACT_CMB_WAKE_PREEMPT:
            run = sim.proc[pid].status == PROC_RUNNING;
            break;
        case ACT_CMB_WAKE_CONDITION:
            (void)sim.list_remove(sim.proc[pid].awaits, AWAIT_RESOURCE, 0u, true);
            run = sim.proc[pid].status == PROC_RUNNING;
            break;
        case ACT_CMB_WAKE_PROCESS:
            (void)sim.list_remove(sim.proc[pid].awaits, AWAIT_PROCESS, 0u, true);
            run = sim.proc[pid].status == PROC_RUNNING;
            break;
        case ACT_CMB_WAKE_EVENT:
            (void)sim.list_remove(sim.proc[pid].awaits, AWAIT_EVENT, 0u, true);
            run = sim.proc[pid].status == PROC_RUNNING;
            break;
        case ACT_CMB_RESUME:
            run = true;
            break;
        case ACT_CMB_WAKE_INTERRUPT:
            sim.cancel_awaiteds(pid);
            run = true;
            break;
        default:
            m.event(sim, (uint32_t)ev.act, pid, (int64_t)ev.arg);
            break;
        }
        if (run) {
            sim.current = pid;
            m.process(sim, pid, sim.proc[pid].kind, (int64_t)ev.arg);
            sim.current = NIL;
            // the blocking call the body stopped at, carried out where the warp is together again
            const uint32_t cmd = sim.cmd;
            sim.cmd = CMD_NONE;
            if (cmd == CMD_HOLD || cmd == CMD_HOLD_EXPONENTIAL) {
                const double dur = cmd == CMD_HOLD ? sim.cmd_value : gp_exponential(sim.rng, *sim.hot, sim.cmd_value);
                sim.hold_begin(pid, dur);
            }
            else if (cmd == CMD_HOLD_SAMPLED) {
                sim.hold_begin(pid, ModelSampler<Model, Sim>::draw(m, sim, sim.cmd_sample));
            }
            else if (cmd == CMD_GUARD_WAIT) {
                sim.guard_wait_begin(*sim.cmd_guard, pid, sim.cmd_demand, sim.cmd_ctx);
            }
            else if (cmd == CMD_EXIT) {
                process_exit(sim, m, pid, sim.cmd_exit);
            }
        }
    }
}

}  // namespace cmb
}  // namespace cimba_b200

namespace cimba_b200 {
namespace cmb {
// cmb_random_erlang on either engine: k exponentials added up (include/cmb_random.h:366)
template <class S>
CMB_FN double draw_erlang(S &sim, unsigned k, double mean)
{
    double x = 0.0;
    for (unsigned i = 0u; i < k; i++) x = __dadd_rn(x, draw_exponential(sim, mean));
    return x;
}

// the two ziggurat draws behind cmb_random_exponential / cmb_random_normal: out of line on the general engine (one copy of the
// slow paths per kernel); the static tier (cmb_static.cuh) overloads them inline, where a call would force its state into memory
CMB_FN double draw_exponential(Sim &sim, double mean) { return gp_exponential(sim.rng, *sim.hot, mean); }
CMB_FN double draw_std_normal(Sim &sim) { return gp_std_normal(sim.rng, *sim.hot); }
}  // namespace cmb
}  // namespace cimba_b200

// ================================================================================================ the authoring surface
// Inside a process body - a function `void body(cmb::Sim &sim, Model &m, uint32_t me, int64_t sig)` - these read like
// the reference's calls.  `sig` holds the call's return value afterwards (CMB_PROCESS_SUCCESS, a timer's or an
// interrupt's signal).  Arguments are evaluated again after a wait: pass variables, not expressions with side effects
// (cmb_time() after a wait is a different time - stamp first, then put the stamp).
#define CMB_PROCESS_BEGIN        (void)&m; switch (sim.proc[me].pc) { case 0u:
#define CMB_PROCESS_END          } sim.cmd = cimba_b200::cmb::CMD_EXIT; sim.cmd_exit = 0; return;
#define CMB_YIELD_AT_(n)         do { sim.proc[me].pc = (n); return; case (n):; } while (0)
#define CMB_YIELD_()             CMB_YIELD_AT_(__COUNTER__ + 1u)

// cmb_resourceguard_wait up to its yield: the wait-list insert is left to the dispatcher
#define CMB_GUARD_WAIT_(g, demand, ctx) \
    do { sim.guard_wait_cmd((g), me, (demand), (ctx)); CMB_YIELD_(); } while (0)

// cmb_process_hold(dur)
#define CMB_PROCESS_HOLD(dur)    do { sim.cmd_value = (dur); sim.cmd = cimba_b200::cmb::CMD_HOLD; CMB_YIELD_(); sig = sim.hold_end(me, sig); } while (0)
// cmb_process_hold(cmb_random_exponential(mean)) with the draw left to the dispatcher, where the whole warp draws together
// (same stream position: nothing draws between the body's return and the dispatcher)
#define CMB_PROCESS_HOLD_EXPONENTIAL(mean) \
    do { sim.cmd_value = (mean); sim.cmd = cimba_b200::cmb::CMD_HOLD_EXPONENTIAL; CMB_YIELD_(); sig = sim.hold_end(me, sig); } while (0)
// cmb_process_hold(<a variate>) with the draw left to the dispatcher: the model's `double sample(S &sim, uint32_t id)` - a pure
// function of the generator and the model's parameters, e.g. `return cmb_random_erlang(2u, 0.5 * arr_mean);` - is called right
// after the body returns (same stream position as a draw in the hold's argument), where the warp is together; the static tier
// first tries it with the ziggurats' hot paths only and parks the lane if that is not enough (cmb_static.cuh).
// The sampler may be any function that terminates on the reference with the same draws - a rejection loop included (an
// exponential redrawn while above a cap, a normal redrawn while negative, a value only a ziggurat's tail can give): a try that
// leaves the rectangles draws on - from the rectangles, and from a stand-in for the slow paths that reaches the same values -
// until the sampler returns, and only then is thrown away and repeated.  It must not keep state across calls: it runs twice for
// a hold whose first try missed the rectangles.
#define CMB_PROCESS_HOLD_SAMPLED(id) \
    do { sim.cmd_sample = (id); sim.cmd = cimba_b200::cmb::CMD_HOLD_SAMPLED; CMB_YIELD_(); sig = sim.hold_end(me, sig); } while (0)
// cmb_process_yield(): wait for whatever comes (a timer, a resume, an interrupt)
#define CMB_PROCESS_YIELD()      do { CMB_YIELD_(); } while (0)
// cmb_process_exit(value)
#define CMB_PROCESS_EXIT(value)  do { sim.cmd = cimba_b200::cmb::CMD_EXIT; sim.cmd_exit = (value); return; } while (0)
// cmb_process_wait_process(other) / cmb_process_wait_event(handle)
#define CMB_PROCESS_WAIT_PROCESS(other) \
    do { if (sim.proc[(other)].status == cimba_b200::cmb::PROC_FINISHED) { sig = CMB_PROCESS_SUCCESS; } \
         else { sim.wait_process_begin(me, (other)); CMB_YIELD_(); } } while (0)
#define CMB_PROCESS_WAIT_EVENT(handle)  do { sim.wait_event_begin(me, (handle)); CMB_YIELD_(); } while (0)

// sig = cmb_objectqueue_put(&q, obj)   (src/cmb_objectqueue.c:262-314)
#define CMB_OBJECTQUEUE_PUT(q, obj) \
    do { for (;;) { \
        if (cimba_b200::cmb::objectqueue_try_put(sim, m, (q), (uint64_t)(obj))) { sig = CMB_PROCESS_SUCCESS; break; } \
        CMB_GUARD_WAIT_((q).rear, cimba_b200::cmb::DEMAND_QUEUE_SPACE, 0); \
        sig = sim.guard_wait_end((q).rear, me, sig); if (sig != CMB_PROCESS_SUCCESS) break; } } while (0)

// sig = cmb_objectqueue_get(&q, &obj)  (:203-260); obj is a uint64_t lvalue (0 when interrupted)
#define CMB_OBJECTQUEUE_GET(q, obj) \
    do { for (;;) { \
        if (cimba_b200::cmb::objectqueue_try_get(sim, m, (q), (obj))) { sig = CMB_PROCESS_SUCCESS; break; } \
        CMB_GUARD_WAIT_((q).front, cimba_b200::cmb::DEMAND_QUEUE_CONTENT, 0); \
        sig = sim.guard_wait_end((q).front, me, sig); if (sig != CMB_PROCESS_SUCCESS) { (obj) = 0u; break; } } } while (0)

// sig = cmb_resourcepool_acquire(&rp, amount) / cmb_resourcepool_preempt(&rp, amount)   (src/cmb_resourcepool.c:362-554)
#define CMB_RESOURCEPOOL_ACQUIRE_(rp, amount, pre) \
    do { sim.proc[me].fr[0] = cimba_b200::cmb::resourcepool_held_by_process(sim, (rp), me); sim.proc[me].fr[1] = (uint64_t)(amount); \
        for (;;) { \
        if (cimba_b200::cmb::pool_acquire_step(sim, m, (rp), me, (pre))) { sig = CMB_PROCESS_SUCCESS; break; } \
        CMB_GUARD_WAIT_((rp).guard, cimba_b200::cmb::DEMAND_POOL_AVAILABLE, 0); \
        sig = sim.guard_wait_end((rp).guard, me, sig); \
        if (sig != CMB_PROCESS_SUCCESS) { cimba_b200::cmb::pool_acquire_rollback(sim, m, (rp), me, sig); break; } } } while (0)
#define CMB_RESOURCEPOOL_ACQUIRE(rp, amount) CMB_RESOURCEPOOL_ACQUIRE_(rp, amount, false)
#define CMB_RESOURCEPOOL_PREEMPT(rp, amount) CMB_RESOURCEPOOL_ACQUIRE_(rp, amount, true)
#define CMB_RESOURCEPOOL_RELEASE(rp, amount) cimba_b200::cmb::resourcepool_release(sim, m, (rp), me, (uint64_t)(amount))

// sig = cmb_resource_acquire(&r)       (src/cmb_resource.c:191-229): ONE wait, and after a successful one the resource is
// taken without another look - as the reference has it
#define CMB_RESOURCE_ACQUIRE(r) \
    do { if ((r).holder == cimba_b200::cmb::NIL) { \
            cimba_b200::cmb::resource_grab(sim, (r), me); cimba_b200::cmb::resource_sample(sim, (r)); sig = CMB_PROCESS_SUCCESS; } \
        else { CMB_GUARD_WAIT_((r).guard, cimba_b200::cmb::DEMAND_RESOURCE_FREE, 0); \
            sig = sim.guard_wait_end((r).guard, me, sig); \
            if (sig == CMB_PROCESS_SUCCESS) { cimba_b200::cmb::resource_grab(sim, (r), me); cimba_b200::cmb::resource_sample(sim, (r)); } } } while (0)
// sig = cmb_resource_preempt(&r)       (:270-320)
#define CMB_RESOURCE_PREEMPT(r) \
    do { if (cimba_b200::cmb::resource_preempt_step(sim, (r), me)) { sig = CMB_PROCESS_SUCCESS; } else { CMB_RESOURCE_ACQUIRE(r); } } while (0)
#define CMB_RESOURCE_RELEASE(r)  cimba_b200::cmb::resource_release(sim, m, (r), me)

// sig = cmb_buffer_get(&b, &amount) / cmb_buffer_put(&b, &amount)   (src/cmb_buffer.c:194-346); `amount` is a uint64_t lvalue:
// in = the amount wanted / offered, out = the amount obtained (get) / still in hand (put) - partial when interrupted
#define CMB_BUFFER_GET(b, amount) \
    do { sim.proc[me].fr[1] = (uint64_t)(amount); sim.proc[me].fr[2] = 0u; \
        for (;;) { \
        if (cimba_b200::cmb::buffer_get_step(sim, m, (b), me)) { sig = CMB_PROCESS_SUCCESS; break; } \
        CMB_GUARD_WAIT_((b).front, cimba_b200::cmb::DEMAND_BUFFER_CONTENT, 0); \
        sig = sim.guard_wait_end((b).front, me, sig); if (sig != CMB_PROCESS_SUCCESS) break; } \
        (amount) = sim.proc[me].fr[2]; } while (0)
#define CMB_BUFFER_PUT(b, amount) \
    do { sim.proc[me].fr[1] = (uint64_t)(amount); \
        for (;;) { \
        if (cimba_b200::cmb::buffer_put_step(sim, m, (b), me)) { sig = CMB_PROCESS_SUCCESS; break; } \
        CMB_GUARD_WAIT_((b).rear, cimba_b200::cmb::DEMAND_BUFFER_SPACE, 0); \
        sig = sim.guard_wait_end((b).rear, me, sig); if (sig != CMB_PROCESS_SUCCESS) break; } \
        (amount) = sim.proc[me].fr[1]; } while (0)

// sig = cmb_priorityqueue_put(&q, obj, priority, &handle) / cmb_priorityqueue_get(&q, &obj)   (src/cmb_priorityqueue.c:189-284)
#define CMB_PRIORITYQUEUE_PUT(q, obj, prio, handle_ptr) \
    do { for (;;) { \
        if (cimba_b200::cmb::priorityqueue_try_put(sim, m, (q), (uint64_t)(obj), (prio), (handle_ptr))) { sig = CMB_PROCESS_SUCCESS; break; } \
        CMB_GUARD_WAIT_((q).rear, cimba_b200::cmb::DEMAND_PQ_SPACE, 0); \
        sig = sim.guard_wait_end((q).rear, me, sig); if (sig != CMB_PROCESS_SUCCESS) break; } } while (0)
#define CMB_PRIORITYQUEUE_GET(q, obj) \
    do { for (;;) { \
        if (cimba_b200::cmb::priorityqueue_try_get(sim, m, (q), (obj))) { sig = CMB_PROCESS_SUCCESS; break; } \
        CMB_GUARD_WAIT_((q).front, cimba_b200::cmb::DEMAND_PQ_CONTENT, 0); \
        sig = sim.guard_wait_end((q).front, me, sig); if (sig != CMB_PROCESS_SUCCESS) { (obj) = 0u; break; } } } while (0)

// sig = cmb_condition_wait(&c, predicate id, ctx)   (src/cmb_condition.c:63-80); spurious wake-ups are the caller's to re-test
#define CMB_CONDITION_WAIT(c, demand_id, ctx) \
    do { CMB_GUARD_WAIT_((c).guard, (demand_id), (ctx)); sig = sim.guard_wait_end((c).guard, me, sig); } while (0)

// the non-blocking calls, by their reference names
#define cmb_time()                          (sim.now)
#define cmb_process_current()               (sim.current)
#define cmb_event_current()                 (sim.current_event)
#define cmb_random()                        (sim.rng.uniform01())
#define cmb_random_exponential(mean)        (cimba_b200::cmb::draw_exponential(sim, (mean)))
#define cmb_random_std_normal()             (cimba_b200::cmb::draw_std_normal(sim))
#define cmb_random_normal(mu, sigma)        (__dadd_rn((mu), __dmul_rn((sigma), cimba_b200::cmb::draw_std_normal(sim))))
#define cmb_random_uniform(lo, hi)          (sim.rng.uniform((lo), (hi)))
#define cmb_random_erlang(k, mean)          (cimba_b200::cmb::draw_erlang(sim, (k), (mean)))
#define cmb_random_bernoulli(p)             (sim.rng.bernoulli(p))
#define cmb_random_dice(lo, hi)             (sim.rng.dice((lo), (hi)))
#define cmb_random_triangular(a, b, c)      (cimba_b200::rnd_triangular(sim.rng, (a), (b), (c)))
#define cmb_random_rayleigh(s)              (cimba_b200::rnd_rayleigh(sim.rng, *sim.hot, (s)))
#define cmb_random_PERT(lo, mode, hi)       (cimba_b200::rnd_PERT_mod(sim.rng, *sim.hot, (lo), (mode), (hi), 4.0))
#define cmb_random_gamma(shape, scale)      (cimba_b200::rnd_gamma(sim.rng, *sim.hot, (shape), (scale)))
#define cmb_random_beta(a, b, lo, hi)       (cimba_b200::rnd_beta(sim.rng, *sim.hot, (a), (b), (lo), (hi)))
#define cmb_random_weibull(shape, scale)    (cimba_b200::rnd_weibull(sim.rng, *sim.hot, (shape), (scale)))
#define cmb_random_lognormal(m, sd)         (cimba_b200::rnd_lognormal(sim.rng, *sim.hot, (m), (sd)))
#define cmb_random_poisson(rate)            (cimba_b200::rnd_poisson(sim.rng, *sim.hot, (rate)))
#define cmb_resourcepool_available(rp)      ((rp).capacity - (rp).in_use)
#define cmb_process_create(kind, prio, ctx) (sim.process_create((kind), (prio), (ctx)))
#define cmb_process_start(pid)              (sim.process_start(pid))
#define cmb_process_destroy(pid)            (sim.process_destroy(pid))
#define cmb_process_exit_value(pid)         (sim.proc[pid].exit_value)
#define cmb_process_stop(pid, value)        (cimba_b200::cmb::process_stop(sim, m, (pid), (value)))
#define cmb_process_interrupt(pid, s, pri)  (sim.interrupt((pid), (s), (pri)))
#define cmb_process_resume(pid, s)          (sim.resume((pid), (s)))
#define cmb_process_timer_add(dur, s)       (sim.timer_add(me, (dur), (s)))
#define cmb_process_timer_set(dur, s)       (sim.timer_set(me, (dur), (s)))
#define cmb_process_timer_cancel(handle)    (sim.timer_cancel(me, (handle)))
#define cmb_process_timers_clear(pid)       (sim.timers_clear(pid))
#define cmb_process_priority(pid)           ((int64_t)sim.proc[pid].prio)
#define cmb_process_priority_set(pid, pri)  (cimba_b200::cmb::process_priority_set(sim, (pid), (pri)))
#define cmb_random_flip()                   (cimba_b200::rnd_flip(sim.rng, sim.flips))
#define cmb_resourcepool_held_by_process(rp, pid) (cimba_b200::cmb::resourcepool_held_by_process(sim, (rp), (pid)))
#define cmb_resourcepool_start_recording(rp) (cimba_b200::cmb::resourcepool_recording_start(sim, (rp)))
#define cmb_resourcepool_stop_recording(rp)  (cimba_b200::cmb::resourcepool_recording_stop(sim, (rp)))
#define cmb_process_status(pid)             (sim.proc[pid].status)
#define cmb_event_schedule(act, subj, arg, t, prio) (sim.schedule((act), (subj), (arg), (t), (prio)))
#define cmb_event_cancel(handle)            (sim.event_cancel(handle))
#define cmb_event_reschedule(handle, t)     (sim.event_reschedule((handle), (t)))
#define cmb_event_reprioritize(handle, pri) (sim.event_reprioritize((handle), (pri)))
#define cmb_event_is_scheduled(handle)      (sim.event_is_scheduled(handle))
#define cmb_objectqueue_initialize(q, cap)  (cimba_b200::cmb::objectqueue_initialize(sim, (q), (cap)))
#define cmb_objectqueue_length(q)           ((q).length)
#define cmb_resourcepool_initialize(rp, cap) (cimba_b200::cmb::resourcepool_initialize(sim, (rp), (cap)))
#define cmb_resourcepool_in_use(rp)         ((rp).in_use)
#define cmb_resource_initialize(r)          (cimba_b200::cmb::resource_initialize(sim, (r)))
#define cmb_resource_start_recording(r)     (cimba_b200::cmb::resource_recording_start(sim, (r)))
#define cmb_resource_stop_recording(r)      (cimba_b200::cmb::resource_recording_stop(sim, (r)))
#define cmb_buffer_initialize(b, cap)       (cimba_b200::cmb::buffer_initialize(sim, (b), (cap)))
#define cmb_buffer_recording_start(b)       (cimba_b200::cmb::buffer_recording_start(sim, (b)))
#define cmb_buffer_recording_stop(b)        (cimba_b200::cmb::buffer_recording_stop(sim, (b)))
#define cmb_buffer_level(b)                 ((b).level)
#define cmb_priorityqueue_initialize(q, cap) (cimba_b200::cmb::priorityqueue_initialize(sim, (q), (cap)))
#define cmb_priorityqueue_recording_start(q) (cimba_b200::cmb::priorityqueue_recording_start(sim, (q)))
#define cmb_priorityqueue_recording_stop(q)  (cimba_b200::cmb::priorityqueue_recording_stop(sim, (q)))
#define cmb_priorityqueue_length(q)         ((uint64_t)(q).queue.count)
#define cmb_priorityqueue_position(q, h)    (cimba_b200::cmb::priorityqueue_position(sim, (q), (h)))
#define cmb_priorityqueue_cancel(q, h)      ((q).queue.remove(sim.arena, (h)))
#define cmb_priorityqueue_reprioritize(q, h, pri) (cimba_b200::cmb::priorityqueue_reprioritize(sim, (q), (h), (pri)))
#define cmb_objectqueue_recording_start(q)  (cimba_b200::cmb::objectqueue_recording_start(sim, (q)))
#define cmb_objectqueue_recording_stop(q)   (cimba_b200::cmb::objectqueue_recording_stop(sim, (q)))
#define cmb_condition_initialize(c)         (cimba_b200::cmb::condition_initialize(sim, (c)))
#define cmb_condition_signal(c)             (cimba_b200::cmb::condition_signal(sim, m, (c)))
#define cmb_resourceguard_register(g, obs)  (cimba_b200::cmb::guard_register(m, (g), (obs)))
