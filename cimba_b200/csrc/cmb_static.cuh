// cmb_static.cuh - the static tier of the authoring surface.
//
// The general engine (cmb_device.cuh) runs ANY model, and pays for it: every container is in memory and grows.  Many models
// need none of that: a FIXED set of processes that only hold and wait at queues - the benchmark's M/M/1
// (benchmark/MM1_multi.c:52-125), G/G/1, a tandem line.  For those, the same model text - the same CMB_PROCESS_* /
// CMB_OBJECTQUEUE_* macros, the same cmb_* names - compiles against cmb::StaticSim<NPROC, NQUEUE, NEVENT> instead of cmb::Sim:
//   * the event list is one slot per process in registers (SlotFel, engine.cuh): a process that can only hold or wait owns at
//     most one pending event, so an insert is a register write and pop-min an NPROC-way compare;
//   * process records, guards (a bit and a sequence number per process) and the model struct stay in registers: process ids
//     are compile-time constants after inlining, nothing takes an address;
//   * a queue is a ring with its oldest 32 entries in shared memory and the rest in an HBM ring (StampRing, engine.cuh); a
//     cmb_buffer is two counters; either can keep its time-weighted history (S::recorded_queue_type, S::recorded_buffer_type);
//   * blocking calls are commands carried out by the dispatcher where the warp is together, and the ziggurat's slow path
//     is taken by parked lanes in batches - as in the fused kernels (queue_model.cuh, whose shape this generalises); a hold
//     of any distribution can be drawn there too (CMB_PROCESS_HOLD_SAMPLED: rectangles first, rewind + park + batch otherwise).
// What the tier does NOT have - process creation beyond NPROC, priorities other than 0, timers, interrupts, a queue that
// outgrows window + ring - is not an error: the trial is flagged and the launch re-runs it on the general engine from the SAME
// model template (launch_static_model below), so the answer is the reference's either way.
//
// A model is `template <class S> struct M` with S = cmb::Sim or cmb::StaticSim<...>, its queues declared as
// `typename S::queue_type`, exported with CMB_EXPORT_STATIC_MODEL(M, NPROC, NQUEUE, "name") (or ..._EVENTS(M, NPROC, NQUEUE,
// NEVENT, "name")).  In this library: mm1_model.cuh, gg1_model.cuh, mm1_recorded_model.cuh, tutorial1_model.cuh (the reference's
// first tutorial: two processes, a buffer, three events); examples/tandem_model.cuh.
#pragma once

#include <type_traits>

#include "cmb_kernel.cuh"

namespace cimba_b200 {
namespace cmb {

constexpr int STATIC_WINDOW = 32;       // on-chip entries per queue and trial
constexpr int STATIC_BLOCK = 64;

// One event slot per process (the shape of SlotFel, engine.cuh), the action packed into the key's two low bits as mm1_fast.cuh
// does: key = (issue counter << 2) | action, 0 = empty.  Counters are unique, so ordering by this word is ordering by issue
// counter - the reference's tie-break (src/cmi_hashheap.c:55-80).
template <int N, bool PRIO = false>
struct StaticFel {
    double   t[N];
    uint32_t key[N];
    int32_t  prio[N];           // PRIO only (a model with events of its own): higher goes first at equal times
    uint32_t issued;

    CMB_FN void clear()
    {
#pragma unroll
        for (int i = 0; i < N; i++) {
            t[i] = __longlong_as_double(0x7ff0000000000000LL);
            key[i] = 0u;
            prio[i] = 0;
        }
        issued = 0u;
    }

    CMB_FN bool schedule(int p, uint32_t action, double time, int32_t priority = 0)     // false: slot p already had a pending event
    {
        const uint32_t k = (++issued << 2) | action;
        bool ok = true;
#pragma unroll
        for (int i = 0; i < N; i++) {
            if (i == p) {
                ok = key[i] == 0u;
                t[i] = time;
                key[i] = k;
                if (PRIO) prio[i] = priority;
            }
        }
        return ok;
    }

    CMB_FN void drop(int p)
    {
#pragma unroll
        for (int i = 0; i < N; i++) {
            if (i == p) {
                t[i] = __longlong_as_double(0x7ff0000000000000LL);
                key[i] = 0u;
            }
        }
    }

    // cmi_hashheap_dequeue: the first entry under (time asc, priority desc, key asc) - default_compare, src/cmi_hashheap.c:55-80;
    // false when the list is empty
    CMB_FN bool pop(int &p, uint32_t &action, double &time, uint32_t &counter)
    {
        int best = 0;
        double bt = t[0];
        uint32_t bk = key[0];
        int32_t bp = PRIO ? prio[0] : 0;
#pragma unroll
        for (int i = 1; i < N; i++) {
            bool before;
            if (PRIO) {
                before = (t[i] < bt) | ((t[i] == bt) & ((prio[i] > bp) | ((prio[i] == bp) & (key[i] < bk))));
            }
            else {
                before = (t[i] < bt) | ((t[i] == bt) & (key[i] < bk));
            }
            if (before) {
                best = i;
                bt = t[i];
                bk = key[i];
                if (PRIO) bp = prio[i];
            }
        }
        drop(best);
        p = best;
        action = bk & 3u;
        time = bt;
        counter = bk >> 2;
        return bk != 0u;
    }
};

// the wait list of a guard whose only possible waiters are the NPROC processes: who waits, and since when (FIFO)
template <int NPROC>
struct static_guard {
    uint32_t waiting;
    uint32_t seq[NPROC];
};

// RECORD: the queue can keep its length history (cmb_objectqueue_recording_start, src/cmb_objectqueue.c:161-177), folded on the
// fly into the time-weighted summary cmb_timeseries_summarize would make of it (TimeWeighted, summary.cuh).  A queue type of its
// own (S::recorded_queue_type) so that models that never record carry neither the registers nor the sampling code.
template <bool RECORD>
struct static_history {
};
template <>
struct static_history<true> {
    uint32_t recording;
    TimeWeighted history;
};

template <int NPROC, bool RECORD = false>
struct static_objectqueue : static_history<RECORD> {
    static_guard<NPROC> front, rear;
    StampRing<STATIC_WINDOW> ring;
    uint64_t capacity;
    uint32_t longest;
    uint32_t length;            // = ring.len (cmb_objectqueue_length)
};

// struct cmb_buffer for a fixed set of processes (amounts put and got in parts, src/cmb_buffer.c:194-346)
template <int NPROC, bool RECORD = false>
struct static_buffer : static_history<RECORD> {
    static_guard<NPROC> front, rear;
    uint64_t level, capacity;
};

// NEVENT: how many events of its own (cmb_event_schedule) a model may have pending at once; with any, the event list also
// orders by priority
template <int NPROC, int NQUEUE, int NEVENT = 0>
struct StaticSim {
    using queue_type = static_objectqueue<NPROC, false>;
    using recorded_queue_type = static_objectqueue<NPROC, true>;
    using buffer_type = static_buffer<NPROC, false>;
    using recorded_buffer_type = static_buffer<NPROC, true>;
    static constexpr int PROCESSES = NPROC;
    static constexpr int SLOTS = NPROC + NEVENT;
    struct Proc {
        uint32_t pc, status, kind, ctx;
        double   f[2];
        uint64_t u[2];
        uint64_t fr[3];         // scratch of the blocking calls in progress (a buffer call's remaining / obtained amounts)
        int64_t  exit_value;
    };
    struct UserEvent {
        uint32_t act, subj;
        int64_t  arg;
    };
    Sfc64          rng;
    const ZigHot  *hot;
    double         now;
    uint32_t       status;
    uint32_t       current;
    uint32_t       current_event;
    uint32_t       pops;
    uint32_t       nproc, nqueue, guard_seq;
    Proc           proc[NPROC];
    StaticFel<NPROC + NEVENT, (NEVENT > 0)> fel;
    UserEvent      uev[NEVENT > 0 ? NEVENT : 1];
    uint32_t       cmd;
    uint32_t       cmd_sample;
    double         cmd_value;
    int64_t        cmd_exit;
    bool           hot_only;        // a sampler is being tried with the ziggurats' rectangles only ...
    bool           hot_failed;      // ... and that was not enough: the try's result is void, the sampler is run again in a batch
    // where this trial's queues live: column `tid` of the CTA's shared-memory rings, and its HBM rings
    double        *ring_win;
    uint32_t       ring_stride;
    double        *spill;
    uint32_t       spill_cap;

    CMB_FN void init(uint64_t seed, const ZigHot *tables, double *win, uint32_t stride, double *spill_rings, uint32_t cap)
    {
        rng.seed(seed);
        hot = tables;
        now = 0.0;
        status = 0u;
        current = NIL;
        current_event = 0u;
        pops = 0u;
        nproc = nqueue = guard_seq = 0u;
        fel.clear();
        cmd = CMD_NONE;
        cmd_sample = 0u;
        cmd_value = 0.0;
        cmd_exit = 0;
        hot_only = hot_failed = false;
        ring_win = win;
        ring_stride = stride;
        spill = spill_rings;
        spill_cap = cap;
#pragma unroll
        for (int i = 0; i < NPROC; i++) {
            proc[i].pc = 0u;
            proc[i].status = PROC_CREATED;
            proc[i].kind = 0u;
            proc[i].ctx = 0u;
            proc[i].f[0] = proc[i].f[1] = 0.0;
            proc[i].u[0] = proc[i].u[1] = 0u;
            proc[i].fr[0] = proc[i].fr[1] = proc[i].fr[2] = 0u;
            proc[i].exit_value = 0;
        }
    }

    // cmb_event_schedule(action, subject, object, time, priority) for an event of the model's own (src/cmb_event.c:123-140):
    // one of the NEVENT spare slots.  Returns the handle (= key), 0 if there is no slot left (the trial is flagged).
    CMB_FN uint64_t schedule(uint32_t act, uint32_t subj, int64_t arg, double t, int64_t prio)
    {
        int slot = -1;
#pragma unroll
        for (int i = NPROC; i < NPROC + NEVENT; i++) {
            if (slot < 0 && fel.key[i] == 0u) slot = i;
        }
        if (slot < 0) {
            status |= TRIAL_ERR_FEL_OVERFLOW;
            return 0u;
        }
        (void)fel.schedule(slot, 0u, t, (int32_t)prio);
#pragma unroll
        for (int i = 0; i < NEVENT; i++) {
            if (i == slot - NPROC) {
                uev[i].act = act;
                uev[i].subj = subj;
                uev[i].arg = arg;
            }
        }
        return (uint64_t)fel.issued;
    }

    // cmb_process_create + cmb_process_initialize.  One process more than the tier holds, or a priority: the trial goes
    // to the general engine.
    CMB_FN uint32_t process_create(uint32_t kind, int64_t prio, uint32_t ctx)
    {
        const uint32_t id = nproc;
        if (id >= (uint32_t)NPROC || prio != 0) {
            status |= TRIAL_ERR_PROC_OVERFLOW;
            return 0u;
        }
        nproc = id + 1u;
#pragma unroll
        for (int i = 0; i < NPROC; i++) {
            if ((uint32_t)i == id) {
                proc[i].kind = kind;
                proc[i].ctx = ctx;
                proc[i].status = PROC_CREATED;
            }
        }
        return id;
    }

    CMB_FN void process_start(uint32_t pid)             // src/cmb_process.c:127-135
    {
        if (!fel.schedule((int)pid, ACT_START, now)) status |= TRIAL_ERR_FEL_OVERFLOW;
    }

    CMB_FN int64_t hold_end(uint32_t, int64_t sig) { return sig; }          // nobody interrupts here

    // cmb_resourceguard_wait up to its yield (src/cmb_resourceguard.c:125-152)
    CMB_FN void guard_wait_cmd(static_guard<NPROC> &g, uint32_t pid, uint32_t, int32_t)
    {
        const uint32_t s = ++guard_seq;
        g.waiting |= 1u << pid;
#pragma unroll
        for (int i = 0; i < NPROC; i++) {
            if ((uint32_t)i == pid) g.seq[i] = s;
        }
        cmd = CMD_NONE;
    }

    CMB_FN int64_t guard_wait_end(static_guard<NPROC> &, uint32_t, int64_t sig) { return sig; }

    // cmb_resourceguard_signal (:202-226): the HEAD waiter, if its demand holds - `ok`, which the caller knows (every waiter
    // of a queue's front guard wants content, of its rear guard space)
    CMB_FN void guard_signal(static_guard<NPROC> &g, bool ok)
    {
        if (g.waiting == 0u || !ok) return;
        uint32_t head = 0u, best = 0xffffffffu;
#pragma unroll
        for (int i = 0; i < NPROC; i++) {
            const bool here = ((g.waiting >> i) & 1u) != 0u && g.seq[i] < best;
            if (here) {
                head = (uint32_t)i;
                best = g.seq[i];
            }
        }
        g.waiting &= ~(1u << head);
        if (!fel.schedule((int)head, ACT_WAKE_RESOURCE, now)) status |= TRIAL_ERR_FEL_OVERFLOW;
    }
};

// cmb_random_exponential / cmb_random_normal in a process body: inline (a call would take the generator's address and put the
// whole control block in local memory)
// In a sampler the dispatcher is trying out (hot_only), a draw that leaves its ziggurat's rectangles marks the try as failed - the
// dispatcher throws its result away, rewinds the generator and repeats the whole sampler later, slow paths allowed, together with
// other lanes in the same position.  The failed try must still end: a sampler that redraws until it accepts (a truncated
// exponential, a normal redrawn while negative, a value only a ziggurat's tail can give) loops forever on a constant it rejects.
// So the generator keeps advancing, the rectangles still answer where they can, and where the slow path would run the try takes a
// stand-in from the ziggurat's tail (its start plus an exponential): together they reach every value the reference's draw can, so
// any sampler that ends on the reference ends here.  The stand-in is one out-of-line -log(u) of a raw output passed by value -
// the slow paths themselves, inline at this call site as well, cost G/G/1 on the static tier a fifth of its throughput.
CMB_FN_NOINLINE double stand_in_neg_log(uint64_t bits)
{
    return -log(__dmul_rn(__ull2double_rn((bits >> 11) + 1u), TWO_POW_M53));      // u in (0, 1]: finite
}

template <int NPROC, int NQUEUE, int NEVENT>
CMB_FN double draw_exponential(StaticSim<NPROC, NQUEUE, NEVENT> &sim, double mean)        // include/cmb_random.h:319-352
{
    const uint64_t u = sim.rng.next();
    if (Sfc64::exp_is_hot(u)) return __dmul_rn(mean, Sfc64::exp_hot(*sim.hot, u));
    if (sim.hot_only) {
        sim.hot_failed = true;
        return __dmul_rn(mean, __dadd_rn(ZIG_EXP_TAIL, stand_in_neg_log(sim.rng.next())));
    }
    return __dmul_rn(mean, sim.rng.exp_cold(u));
}

template <int NPROC, int NQUEUE, int NEVENT>
CMB_FN double draw_std_normal(StaticSim<NPROC, NQUEUE, NEVENT> &sim)                       // include/cmb_random.h:206-215
{
    const int64_t ix = (int64_t)sim.rng.next();
    const unsigned i = (unsigned)(ix & 0xff);
    if (i <= ZIG_NOR_MAX) return __dmul_rn(sim.hot->nor_x[i], __ll2double_rn(ix));
    if (sim.hot_only) {
        sim.hot_failed = true;
        const double x = __dadd_rn(ZIG_NOR_TAIL, __dmul_rn(ZIG_NOR_INV_TAIL, stand_in_neg_log(sim.rng.next())));
        return ix < 0 ? -x : x;
    }
    return sim.rng.nor_cold(*sim.hot, ix);
}

// ------------------------------------------------------------------------------------------------ objectqueue
template <int NPROC, int NQUEUE, int NEVENT, bool RECORD>
CMB_FN void objectqueue_initialize(StaticSim<NPROC, NQUEUE, NEVENT> &sim, static_objectqueue<NPROC, RECORD> &q, uint64_t capacity)
{
    uint32_t k = sim.nqueue;
    if (k >= (uint32_t)NQUEUE) {
        sim.status |= TRIAL_ERR_PROC_OVERFLOW;
        k = 0u;
    }
    sim.nqueue = k + 1u;
    q.front.waiting = q.rear.waiting = 0u;
#pragma unroll
    for (int i = 0; i < NPROC; i++) q.front.seq[i] = q.rear.seq[i] = 0u;
    q.ring.init(sim.ring_win + (size_t)k * STATIC_WINDOW * sim.ring_stride, sim.ring_stride,
                sim.spill_cap ? sim.spill + (size_t)k * sim.spill_cap : nullptr, sim.spill_cap);
    q.capacity = capacity;
    q.longest = 0u;
    q.length = 0u;
    if constexpr (RECORD) q.recording = 0u;
}

template <int NPROC, int NQUEUE, int NEVENT>
CMB_FN void objectqueue_recording_start(StaticSim<NPROC, NQUEUE, NEVENT> &sim, static_objectqueue<NPROC, true> &q)
{
    q.recording = 1u;
    q.history.start();
    q.history.sample((double)q.ring.len, sim.now);
}

template <int NPROC, int NQUEUE, int NEVENT>
CMB_FN void objectqueue_recording_stop(StaticSim<NPROC, NQUEUE, NEVENT> &sim, static_objectqueue<NPROC, true> &q)
{
    if (q.recording) q.history.sample((double)q.ring.len, sim.now);
    q.recording = 0u;
}

template <class Model, int NPROC, int NQUEUE, int NEVENT, bool RECORD>
CMB_FN bool objectqueue_try_put(StaticSim<NPROC, NQUEUE, NEVENT> &sim, Model &, static_objectqueue<NPROC, RECORD> &q, uint64_t obj)
{
    if ((uint64_t)q.ring.len >= q.capacity) return false;
    if (!q.ring.put(__longlong_as_double((long long)obj))) sim.status |= TRIAL_ERR_QUEUE_OVERFLOW;     // void from here on: re-run
    q.longest = q.ring.len > q.longest ? q.ring.len : q.longest;
    q.length = q.ring.len;
    if constexpr (RECORD) {
        if (q.recording) q.history.sample((double)q.ring.len, sim.now);        // record_sample in put, :289
    }
    sim.guard_signal(q.front, true);
    return true;
}

template <class Model, int NPROC, int NQUEUE, int NEVENT, bool RECORD>
CMB_FN bool objectqueue_try_get(StaticSim<NPROC, NQUEUE, NEVENT> &sim, Model &, static_objectqueue<NPROC, RECORD> &q, uint64_t &obj)
{
    if (q.ring.len == 0u) return false;
    obj = (uint64_t)__double_as_longlong(q.ring.take());
    q.length = q.ring.len;
    if constexpr (RECORD) {
        if (q.recording) q.history.sample((double)q.ring.len, sim.now);        // ... and in get, :226-229
    }
    sim.guard_signal(q.rear, true);
    return true;
}

// ------------------------------------------------------------------------------------------------ buffer
template <int NPROC, int NQUEUE, int NEVENT, bool RECORD>
CMB_FN void buffer_initialize(StaticSim<NPROC, NQUEUE, NEVENT> &, static_buffer<NPROC, RECORD> &b, uint64_t capacity)
{
    b.front.waiting = b.rear.waiting = 0u;
#pragma unroll
    for (int i = 0; i < NPROC; i++) b.front.seq[i] = b.rear.seq[i] = 0u;
    b.level = 0u;
    b.capacity = capacity;
    if constexpr (RECORD) b.recording = 0u;
}

template <int NPROC, int NQUEUE, int NEVENT>
CMB_FN void buffer_recording_start(StaticSim<NPROC, NQUEUE, NEVENT> &sim, static_buffer<NPROC, true> &b)
{
    b.recording = 1u;
    b.history.start();
    b.history.sample((double)b.level, sim.now);
}

template <int NPROC, int NQUEUE, int NEVENT>
CMB_FN void buffer_recording_stop(StaticSim<NPROC, NQUEUE, NEVENT> &sim, static_buffer<NPROC, true> &b)
{
    if (b.recording) b.history.sample((double)b.level, sim.now);
    b.recording = 0u;
}

template <int NPROC, int NQUEUE, int NEVENT, bool RECORD>
CMB_FN void buffer_sample(StaticSim<NPROC, NQUEUE, NEVENT> &sim, static_buffer<NPROC, RECORD> &b)
{
    if constexpr (RECORD) {
        if (b.recording) b.history.sample((double)b.level, sim.now);
    }
}

// cmb_buffer_get / cmb_buffer_put up to their waits, as cmb_device.cuh's buffer_get_step / buffer_put_step (src/cmb_buffer.c:194-346)
template <class Model, int NPROC, int NQUEUE, int NEVENT, bool RECORD>
CMB_FN bool buffer_get_step(StaticSim<NPROC, NQUEUE, NEVENT> &sim, Model &, static_buffer<NPROC, RECORD> &b, uint32_t pid)
{
    uint64_t rem = 0u, got = 0u;
#pragma unroll
    for (int i = 0; i < NPROC; i++) {
        if ((uint32_t)i == pid) {
            rem = sim.proc[i].fr[1];
            got = sim.proc[i].fr[2];
        }
    }
    bool done;
    if (b.level >= rem) {
        b.level -= rem;
        buffer_sample(sim, b);
        got += rem;
        sim.guard_signal(b.rear, b.level < b.capacity);
        if (b.level > 0u) sim.guard_signal(b.front, true);
        done = true;
    }
    else {
        if (b.level > 0u) {
            const uint64_t grab = b.level;
            b.level = 0u;
            buffer_sample(sim, b);
            got += grab;
            rem -= grab;
            sim.guard_signal(b.rear, b.level < b.capacity);
        }
        sim.guard_signal(b.rear, b.level < b.capacity);
        done = false;
    }
#pragma unroll
    for (int i = 0; i < NPROC; i++) {
        if ((uint32_t)i == pid) {
            sim.proc[i].fr[1] = rem;
            sim.proc[i].fr[2] = got;
        }
    }
    return done;
}

template <class Model, int NPROC, int NQUEUE, int NEVENT, bool RECORD>
CMB_FN bool buffer_put_step(StaticSim<NPROC, NQUEUE, NEVENT> &sim, Model &, static_buffer<NPROC, RECORD> &b, uint32_t pid)
{
    uint64_t rem = 0u;
#pragma unroll
    for (int i = 0; i < NPROC; i++) {
        if ((uint32_t)i == pid) rem = sim.proc[i].fr[1];
    }
    bool done;
    if (b.capacity - b.level >= rem) {
        b.level += rem;
        buffer_sample(sim, b);
        rem = 0u;
        sim.guard_signal(b.front, b.level > 0u);
        if (b.level < b.capacity) sim.guard_signal(b.rear, true);
        done = true;
    }
    else {
        if (b.level < b.capacity) {
            const uint64_t grab = b.capacity - b.level;
            b.level = b.capacity;
            buffer_sample(sim, b);
            rem -= grab;
            sim.guard_signal(b.front, b.level > 0u);
        }
        sim.guard_signal(b.front, b.level > 0u);
        done = false;
    }
#pragma unroll
    for (int i = 0; i < NPROC; i++) {
        if ((uint32_t)i == pid) sim.proc[i].fr[1] = rem;
    }
    return done;
}

// cmb_process_stop (src/cmb_process.c:698-723) as far as this tier can need it: the process's pending event goes, it is
// FINISHED; an entry it may have in a guard stays (SURVEY.md quirk 2) and will swallow one signal
template <class Model, int NPROC, int NQUEUE, int NEVENT>
CMB_FN void process_stop(StaticSim<NPROC, NQUEUE, NEVENT> &sim, Model &, uint32_t pid, int64_t value)
{
#pragma unroll
    for (int i = 0; i < NPROC; i++) {
        if ((uint32_t)i == pid && sim.proc[i].status == PROC_RUNNING) {
            sim.proc[i].status = PROC_FINISHED;
            sim.proc[i].exit_value = value;
            sim.fel.drop(i);
        }
    }
}

// ------------------------------------------------------------------------------------------------ dispatcher
// A model may state the kinds of its processes in creation order - `static CMB_FN constexpr uint32_t static_kind(uint32_t i)` -
// and the dispatcher then knows at compile time which body process i runs (one copy of each body instead of NPROC, no run-time
// branch on the kind); a trial whose cmb_process_create calls disagree with the table is flagged and goes to the general engine.
template <class Model, class = void>
struct StaticKinds {
    static constexpr bool known = false;
    template <int I>
    static CMB_FN uint32_t of(uint32_t runtime_kind) { return runtime_kind; }
    template <class S>
    static CMB_FN bool agree(const S &) { return true; }
};
template <class Model>
struct StaticKinds<Model, decltype((void)Model::static_kind(0u))> {
    static constexpr bool known = true;
    template <int I>
    static CMB_FN uint32_t of(uint32_t) { return Model::static_kind((uint32_t)I); }
    template <class S>
    static CMB_FN bool agree(const S &sim)
    {
        return agree_from<S, 0>(sim);
    }
    template <class S, int I>
    static CMB_FN bool agree_from(const S &sim)
    {
        if constexpr (I < S::PROCESSES) {
            return ((uint32_t)I >= sim.nproc || sim.proc[I].kind == Model::static_kind((uint32_t)I)) && agree_from<S, I + 1>(sim);
        }
        else {
            return true;
        }
    }
};

template <class Model, int NPROC, int NQUEUE, int NEVENT, int I>
struct StaticDispatch {
    static CMB_FN void run(StaticSim<NPROC, NQUEUE, NEVENT> &sim, Model &m, int who)
    {
        if (who == I) m.process(sim, (uint32_t)I, StaticKinds<Model>::template of<I>(sim.proc[I].kind), CMB_PROCESS_SUCCESS);
        else StaticDispatch<Model, NPROC, NQUEUE, NEVENT, I + 1>::run(sim, m, who);
    }
};
template <class Model, int NPROC, int NQUEUE, int NEVENT>
struct StaticDispatch<Model, NPROC, NQUEUE, NEVENT, NPROC> {
    static CMB_FN void run(StaticSim<NPROC, NQUEUE, NEVENT> &, Model &, int) {}
};

// one step of cmb_event_queue_execute (src/cmb_event.c:229-252): pop, advance the clock, resume the process.  false = the
// list ran dry.  The body's blocking call is left in sim.cmd for the caller (`who` = the process it belongs to).
template <class Model, int NPROC, int NQUEUE, int NEVENT>
CMB_FN bool static_step(StaticSim<NPROC, NQUEUE, NEVENT> &sim, Model &m, int &who)
{
    uint32_t act, key;
    double when;
    if (!sim.fel.pop(who, act, when, key)) return false;
    sim.now = when;
    sim.current_event = key;
    sim.pops++;
    sim.cmd = CMD_NONE;
    if (NEVENT > 0 && who >= NPROC) {                   // an event of the model's own: its action function, no process resumed
#pragma unroll
        for (int i = 0; i < NEVENT; i++) {
            if (i == who - NPROC) m.event(sim, sim.uev[i].act, sim.uev[i].subj, sim.uev[i].arg);
        }
        return true;
    }
    bool run = true;
#pragma unroll
    for (int i = 0; i < NPROC; i++) {
        if (i == who) {
            if (act == ACT_START) {
                sim.proc[i].status = PROC_RUNNING;
                sim.proc[i].pc = 0u;
            }
            run = sim.proc[i].status == PROC_RUNNING;
        }
    }
    if (run) {
        sim.current = (uint32_t)who;
        StaticDispatch<Model, NPROC, NQUEUE, NEVENT, 0>::run(sim, m, who);
        sim.current = NIL;
    }
    return true;
}

// the blocking call the body ended on, except the holds whose duration the caller draws (exponential, sampled)
template <int NPROC, int NQUEUE, int NEVENT>
CMB_FN void static_finish_command(StaticSim<NPROC, NQUEUE, NEVENT> &sim, int who, uint32_t cmd)
{
    if (cmd == CMD_HOLD) {
        if (sim.cmd_value < 0.0) sim.status |= TRIAL_ERR_NEGATIVE_HOLD;
        if (!sim.fel.schedule(who, ACT_WAKE_TIME, __dadd_rn(sim.now, sim.cmd_value))) sim.status |= TRIAL_ERR_FEL_OVERFLOW;
    }
    else if (cmd == CMD_EXIT) {                         // cmb_process_exit: nothing pending, nobody waiting for it here
#pragma unroll
        for (int i = 0; i < NPROC; i++) {
            if (i == who) {
                sim.proc[i].status = PROC_FINISHED;
                sim.proc[i].exit_value = sim.cmd_exit;
            }
        }
    }
}

#ifdef CMB_HOST_BUILD
// the tier's source text run on the CPU (tests/cmb_engine_host.cpp): one trial, the slow path taken where it occurs
template <class Model, int NPROC, int NQUEUE, int NEVENT>
inline void static_run_trial_host(StaticSim<NPROC, NQUEUE, NEVENT> &sim, Model &m, const TrialIn &in, TrialOut &out,
                                  uint64_t trace_cap, uint64_t *trace_key, double *trace_time)
{
    out.objects = 0u;
    out.sum_wait = 0.0;
    out.max_queue = 0u;
    for (int k = 0; k < 8; k++) out.counters[k] = 0u;
    m.run_trial(sim, in);
    if (!StaticKinds<Model>::agree(sim)) sim.status |= TRIAL_ERR_PROC_OVERFLOW;
    int who = 0;
    while (static_step(sim, m, who)) {
        if (sim.pops <= trace_cap) {
            trace_key[sim.pops - 1u] = sim.current_event;
            trace_time[sim.pops - 1u] = sim.now;
        }
        const uint32_t cmd = sim.cmd;
        sim.cmd = CMD_NONE;
        if (cmd == CMD_HOLD_EXPONENTIAL) {
            const double dur = gp_exponential(sim.rng, *sim.hot, sim.cmd_value);
            if (!sim.fel.schedule(who, ACT_WAKE_TIME, __dadd_rn(sim.now, dur))) sim.status |= TRIAL_ERR_FEL_OVERFLOW;
        }
        else if (cmd == CMD_HOLD_SAMPLED) {
            // as the device does it: the rectangles only first, and if they do not suffice the generator rewound and the whole sampler again
            const Sfc64 saved = sim.rng;
            sim.hot_only = true;
            sim.hot_failed = false;
            double dur = ModelSampler<Model, StaticSim<NPROC, NQUEUE, NEVENT>>::draw(m, sim, sim.cmd_sample);
            sim.hot_only = false;
            if (sim.hot_failed) {
                sim.hot_failed = false;
                sim.rng = saved;
                dur = ModelSampler<Model, StaticSim<NPROC, NQUEUE, NEVENT>>::draw(m, sim, sim.cmd_sample);
            }
            if (dur < 0.0) sim.status |= TRIAL_ERR_NEGATIVE_HOLD;
            if (!sim.fel.schedule(who, ACT_WAKE_TIME, __dadd_rn(sim.now, dur))) sim.status |= TRIAL_ERR_FEL_OVERFLOW;
        }
        else {
            static_finish_command(sim, who, cmd);
        }
    }
    m.finish(sim, out);
}
#else

#ifndef STATIC_COLD_BATCH
#define STATIC_COLD_BATCH 4
#endif
#ifndef STATIC_PARK_MASK
#define STATIC_PARK_MASK 3u     // the parked set is examined every 4th step
#endif

// A model whose process bodies never draw themselves - every variate is the duration of a CMB_PROCESS_HOLD_EXPONENTIAL, drawn
// by the dispatcher - may say `static constexpr bool exponential_holds_only = true;`.  The dispatcher then keeps one raw sfc64
// output of look-ahead with its hot-path variate already formed (as mm1_fast.cuh does): the table look-up and the 64-bit ->
// double conversion leave the pop -> push chain.  The stream order is unchanged BECAUSE nothing else draws in between; a model
// with a cmb_random_* call in a body must not claim it.
template <class Model, class = void>
struct StaticLookahead {
    static constexpr bool value = false;
};
template <class Model>
struct StaticLookahead<Model, typename std::enable_if<Model::exponential_holds_only>::type> {
    static constexpr bool value = true;
};

struct StaticArgs {
    LaunchArgs base;
    double    *spill;           // [num_trials][NQUEUE][spill_cap]
    uint32_t   spill_cap;
};

template <template <class> class ModelT, int NPROC, int NQUEUE, int NEVENT, bool TRACE>
__global__ void __launch_bounds__(STATIC_BLOCK)
static_trial_kernel(const StaticArgs sa)
{
    using S = StaticSim<NPROC, NQUEUE, NEVENT>;
    __shared__ ZigHot hot;
    __shared__ double ring_smem[(NQUEUE > 0 ? NQUEUE : 1) * STATIC_WINDOW * STATIC_BLOCK];
    const LaunchArgs &a = sa.base;
    stage_zig_hot(hot, true);
    __syncthreads();

    constexpr unsigned FULL = 0xffffffffu;
    const uint64_t trial = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool alive = trial < a.num_trials;

    S sim;
    ModelT<S> m;
    TrialOut out;
    out.objects = 0u;
    out.sum_wait = 0.0;
    out.max_queue = 0u;
    for (int k = 0; k < 8; k++) out.counters[k] = 0u;
    sim.init(alive ? fmix64(a.master_seed, a.first_trial + trial) : 0u, &hot, &ring_smem[threadIdx.x], STATIC_BLOCK,
             (sa.spill_cap && alive) ? sa.spill + trial * (uint64_t)NQUEUE * sa.spill_cap : nullptr, sa.spill_cap);
    if (alive) {
        TrialIn in;
        in.arr_mean = a.arr_mean[trial];
        in.srv_mean = a.srv_mean[trial];
        in.num_objects = a.num_objects;
        in.servers = a.servers;
        in.num_params = a.num_params;
        for (int k = 0; k < 16; k++) in.params[k] = a.params[k];
        in.trial = a.first_trial + trial;
        m.run_trial(sim, in);
        if (!StaticKinds<ModelT<S>>::agree(sim)) sim.status |= TRIAL_ERR_PROC_OVERFLOW;
    }

#ifdef STATIC_NO_LOOKAHEAD
    constexpr bool AHEAD = false;
#else
    constexpr bool AHEAD = StaticLookahead<ModelT<S>>::value;
#endif
    bool parked = false;            // the exponential hold of this lane needs the ziggurat's slow path: wait for company
    uint64_t parked_u = 0u;
    int parked_who = 0;
    bool parked_sampled = false;    // ... or the sampler of its CMB_PROCESS_HOLD_SAMPLED does
    uint64_t u_next = 0u;           // AHEAD: the next raw output, drawn as soon as the previous one was consumed ...
    double e_next = 0.0;            // ... and its hot-path standard exponential
    if (AHEAD && alive) {
        u_next = sim.rng.next();
        e_next = Sfc64::exp_hot(hot, u_next);
    }
    uint32_t step = 0u;

    while (__any_sync(FULL, alive)) {
        bool draw = false, sampled = false;
        int who = 0;
        if (alive && !parked) {
            if (!static_step(sim, m, who)) {
                alive = false;                          // cmb_event_queue_execute returns
                m.finish(sim, out);
                if (a.events)    a.events[trial] = sim.pops;
                if (a.objects)   a.objects[trial] = out.objects;
                if (a.t_end)     a.t_end[trial] = sim.now;
                if (a.sum_wait)  a.sum_wait[trial] = out.sum_wait;
                if (a.status)    a.status[trial] = sim.status | (sim.fel.issued > 0x3ffffff0u ? TRIAL_ERR_KEY_OVERFLOW : 0u);
                if (a.max_queue) a.max_queue[trial] = out.max_queue;
                if (a.counters) {
                    for (int k = 0; k < 8; k++) a.counters[trial * 8u + k] = out.counters[k];
                }
            }
            else {
                if (TRACE) {
                    if (sim.pops <= a.trace_cap) {
                        a.trace_key[trial * a.trace_cap + sim.pops - 1u] = sim.current_event;
                        a.trace_time[trial * a.trace_cap + sim.pops - 1u] = sim.now;
                    }
                }
                const uint32_t cmd = sim.cmd;
                draw = cmd == CMD_HOLD_EXPONENTIAL;
                sampled = cmd == CMD_HOLD_SAMPLED;
                if (!draw && !sampled) static_finish_command(sim, who, cmd);
            }
        }
        // ---- converged: a sampled hold (CMB_PROCESS_HOLD_SAMPLED) - the model's sampler with the rectangles only; a lane whose
        // draw needs more rewinds the generator and parks
        if (sampled) {
            const Sfc64 saved = sim.rng;
            sim.hot_only = true;
            sim.hot_failed = false;
            const double dur = ModelSampler<ModelT<S>, S>::draw(m, sim, sim.cmd_sample);
            sim.hot_only = false;
            if (sim.hot_failed) {
                sim.hot_failed = false;
                sim.rng = saved;
                parked = true;
                parked_sampled = true;
                parked_who = who;
            }
            else {
                if (dur < 0.0) sim.status |= TRIAL_ERR_NEGATIVE_HOLD;
                if (!sim.fel.schedule(who, ACT_WAKE_TIME, __dadd_rn(sim.now, dur))) sim.status |= TRIAL_ERR_FEL_OVERFLOW;
            }
        }
        // ---- converged: the hold's variate and its wake-up event (cmb_process_hold, src/cmb_process.c:262-285)
        if (draw) {
            const uint64_t u = AHEAD ? u_next : sim.rng.next();
            if (Sfc64::exp_is_hot(u)) {
                const double dur = __dmul_rn(sim.cmd_value, AHEAD ? e_next : Sfc64::exp_hot(hot, u));
                if (!sim.fel.schedule(who, ACT_WAKE_TIME, __dadd_rn(sim.now, dur))) sim.status |= TRIAL_ERR_FEL_OVERFLOW;
                if (AHEAD) {
                    u_next = sim.rng.next();
                    e_next = Sfc64::exp_hot(hot, u_next);
                }
            }
            else {
                parked = true;
                parked_u = u;
                parked_who = who;
            }
        }
        if ((++step & STATIC_PARK_MASK) != 0u) continue;
        const unsigned pm = __ballot_sync(FULL, parked);
        if (pm != 0u) {
            const unsigned am = __ballot_sync(FULL, alive);
            if (__popc(pm) >= STATIC_COLD_BATCH || pm == am) {
                if (parked) {
                    double dur;
                    if (parked_sampled) {
                        dur = ModelSampler<ModelT<S>, S>::draw(m, sim, sim.cmd_sample);
                        if (dur < 0.0) sim.status |= TRIAL_ERR_NEGATIVE_HOLD;
                    }
                    else {
                        dur = __dmul_rn(sim.cmd_value, sim.rng.exp_cold(parked_u));
                    }
                    if (!sim.fel.schedule(parked_who, ACT_WAKE_TIME, __dadd_rn(sim.now, dur))) sim.status |= TRIAL_ERR_FEL_OVERFLOW;
                    parked = false;
                    parked_sampled = false;
                    if (AHEAD) {
                        u_next = sim.rng.next();
                        e_next = Sfc64::exp_hot(hot, u_next);
                    }
                }
            }
        }
    }
}
#endif  // CMB_HOST_BUILD

}  // namespace cmb
}  // namespace cimba_b200
