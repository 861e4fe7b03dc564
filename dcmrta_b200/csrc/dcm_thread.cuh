// dcm_thread.cuh -- thread-per-env device functions of the TaskEnv step for sm_100a.
//
// One thread simulates one env; the 32 envs of a tile are simulated by the 32 lanes of one warp.  The boolean state of
// an env lives in 64-bit masks held in registers (struct St); loops run over set bits only.  The kernel that runs these
// functions is latency-bound, not bandwidth-bound: a decision is organised as two unconditional rounds of loads (step_env,
// dcm_kernels.cu), per-task data is one 64-byte record (TREC), per-thread arrays that need dynamic indexing live in a
// shared-memory scratch (TC::nds / nws / tmp) filled with cp.async, and data-dependent gathers are staged there and consumed
// by rolled loops.
//
// All event-clock arithmetic is fp64 in the exact operation order of the reference (SURVEY.md App. A, Q1); the file
// is compiled with -fmad=false and the one fused multiply-add the reference performs (inside np.linalg.norm) is
// written as fma().  Each function cites the reference lines (env/task_env.py unless noted) it replaces.
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "dcm_philox.cuh"
#include "dcm_soa.h"

namespace dcm {

typedef unsigned long long u64;

constexpr unsigned ENV_DONE = 1u, ENV_FINISHED = 2u, ENV_STUCK = 4u, ENV_ERR_OVERFLOW = 16u, ENV_ERR_ACTION = 32u,
                   ENV_ERR_FOLLOW = 64u, ENV_ERR_LEADER = 128u, ENV_ACCOUNTED = 256u, ENV_FRESH = 512u;

// thread context: which env, plus the scalar parameters
struct TC {
    const DcmSoa& s;
    unsigned tile, l;          // b = tile*32 + l
    size_t tb;                 // byte offset of the tile's block in the arena
    int A, T, MC;
    double W, vel, max_time;
    // Per-thread scratch in SHARED memory (fused step only, NULL elsewhere).  Element k of this thread lives at [k * SCR_STRIDE]: the
    // bank of an access then depends on the thread alone, so 32 lanes that index 32 DIFFERENT elements never conflict -- a dynamically
    // indexed per-thread array at shared-memory latency instead of a chain of DRAM round trips (next_decision scan) or of register
    // selects (node ids).
    double* nds = nullptr;     // next_decision of the env's agents, write-through copy of a_nd
    unsigned* nws = nullptr;   // route[-1] of the env's agents, four ids per word, write-through copy of a_node
    // Staging area of SCR_TMP doubles (every kernel that runs the update functions provides it): the values a data-dependent SET of
    // tasks / agents needs -- earliest arrivals of the waiting coalitions, the member slots of one task, time_start of the watched
    // agents -- are gathered with cp.async (LDGSTS: no destination registers, any number in flight) and consumed by ROLLED loops.  One
    // round trip per SCR_TMP items, no register arrays, no unrolled copies of the loop bodies.
    double* tmp = nullptr;
};
#define SCR_STRIDE 64          // threads per block of the kernels that carry the scratch (STEP_THREADS)
#define SCR_TMP 16
#define TMPV(c, k) ((c).tmp[(unsigned)(k) * SCR_STRIDE])

// The arena is TILE-MAJOR: all arrays of one tile of 32 envs are contiguous (c.tb = tile * tile_stride bytes), so the
// working set of a warp-step lies in one or two 2 MB pages instead of one page per array (TLB reach is 256 MB, the state
// of 65,536 envs is ~400 MB).  DcmSoa pointers address tile 0.
#define TB(c, arr) ((decltype(+(c).s.arr))((char*)(c).s.arr + (c).tb))
// row-major arrays: element (row k) of this thread's env in an array with K rows per tile
#define EL(c, arr, K, k) (TB(c, arr)[((void)(K), ((unsigned)(k) << 5)) + (c).l])    // K (rows per tile) documents the array's extent
// lane-contiguous arrays
#define LANE_ROW(c, K, k) ((void)(K), (size_t)(((unsigned)(k) << 5) + (c).l))
#define SARR(c, j, sl) (TB(c, t_slot_arr)[LANE_ROW(c, (c).T, j) * (unsigned)(c).MC + (unsigned)(sl)])      // arrival of slot s of task j
// The TASK RECORD: one 64-byte line per (task, lane) = two 32-byte sectors, one DRAM burst.
//   sector 0, everything a decision changes:  [0] amin | time_start   [1] amax | time_finish   [2] member ids (8 bytes)
//                                             [3] count | status << 8 | requirement << 16 | len(abandoned_agent) << 32
//   sector 1, the static instance again:      [4] duration   [5] x   [6] y   [7] -
// A decision's round 2 reads the whole line of the chosen task (round 1 read nine scattered sectors of seven arrays for the same
// fields); a join writes sector 0; the waiting-coalition scan and the evaluation of a task read sector 0.  Row-major copies of what the
// observation kernel streams with TMA (status, requirement, coordinates, fp32 durations) stay beside it.
#define TREC(c, j, k) (TB(c, t_rec)[(LANE_ROW(c, (c).T, j) << 3) + (k)])
#define TINFO(c, j, k) TREC(c, j, k)                                                                    // 0: time_start | amin, 1: time_finish | amax
#define TIDS(c, j) (((unsigned long long*)TB(c, t_rec))[(LANE_ROW(c, (c).T, j) << 3) + 2])
#define SMEM(c, j, sl) (((unsigned char*)&TIDS(c, j))[(unsigned)(sl)])                                   // member id of slot s
#define TPACK(c, j) (((unsigned long long*)TB(c, t_rec))[(LANE_ROW(c, (c).T, j) << 3) + 3])
#define TNMEM(c, j) (((unsigned char*)&TPACK(c, j))[0])                                                  // valid when the non-empty bit is set
#define TSTAT(c, j) (((signed char*)&TPACK(c, j))[1])                                                    // stored status (may be stale, Q3); row-major copy: t_status
#define TREQ(c, j) (((unsigned char*)&TPACK(c, j))[2])
#define TNAB(c, j) (((unsigned short*)&TPACK(c, j))[2])                                                  // len(abandoned_agent)
#define TDUR(c, j) TREC(c, j, 4)
#define TXY2(c, j) (((double2*)TB(c, t_rec))[(LANE_ROW(c, (c).T, j) << 2) + 2])                          // {duration, x}: with TREC(c, j, 6) = y the static sector
// agent record {x, y, arrival_time[-1], travel_dist}: one 32-byte sector.  The location is always the coordinate of the node the agent
// stands at (task_env.py:93, :134, :320) and could be looked up there; it is STORED because the observation kernels then read it with
// the record instead of through a dependent node -> coordinate gather (measured: without it k_obs_tile 51 -> 54 us, the chunked k_obs
// of the large shapes 122 -> 163 us at 30A/100T; profiles/r09_xy_by_node.txt)
#define AREC(c, i, f) (TB(c, a_rec)[(LANE_ROW(c, (c).A, i) << 2) + (f)])
enum { AR_X = 0, AR_Y = 1, AR_LAST = 2, AR_DIST = 3 };
#define AREC2(c, i, h) (((double2*)TB(c, a_rec))[(LANE_ROW(c, (c).A, i) << 1) + (h)])                    // h = 0: {x, y}   h = 1: {last, dist}
#define AOBS2(c, i) (((double2*)TB(c, a_obs))[LANE_ROW(c, (c).A, i)])                                    // observation cache, see dcm_soa.h
#define TINFO2(c, j) (((double2*)TB(c, t_rec))[LANE_ROW(c, (c).T, j) << 2])                              // {time_start | amin, time_finish | amax}
#define TIDPACK2(c, j) (((ulonglong2*)TB(c, t_rec))[(LANE_ROW(c, (c).T, j) << 2) + 1])                  // {ids, count | status | requirement | abandoned}
// route[-1] of the agents of one env, one byte each, four agents per 32-bit word, words row-major [ANB/4][32 lanes]: a warp reads word k of
// its 32 envs with one coalesced access, and the tile's words land in shared memory (cp.async in the step, TMA in k_obs_tile) in a layout
// whose bank depends on the lane alone
#define ANODE_WORD(c, k) (((unsigned*)TB(c, a_node))[((unsigned)(k) << 5) + (c).l])
#define ANODE(c, i) (TB(c, a_node)[((((unsigned)(i) >> 2) << 5) + (c).l) * 4u + ((unsigned)(i) & 3u)])

// register-resident boolean state of one env
template <int TW> struct St {
    u64 feas[TW], fin[TW], ne[TW], open[TW], dirty[TW];
    u64 route, assigned, returned, member, depot, touched, watch;
    // conservative lower bounds (never too high, +inf when the set is empty) that let a step skip whole scans:
    double xfin;    // <= time_finish of every feasible, unfinished task
    double xamin;   // <= earliest member arrival of every non-feasible task that has members
    double xret;    // <= arrival at the depot of every agent that went there and is not `returned` yet
    double xlast;   // running maximum of every arrival since the reset == max over agents of max(arrival_time), what next_decision
                    // returns when everybody is NaN (task_env.py:285-286).  It exceeds the largest LAST arrival only after a preset route
                    // re-visits a feasible task once it has ended: that agent's next_decision lies in the past and the clock goes back.
};

__device__ __forceinline__ int ctz64(u64 m) { return __ffsll((long long)m) - 1; }
__device__ __forceinline__ int kth_bit(u64 m, int k) {            // position of the k-th (0-based) set bit
    for (; k > 0; --k) m &= m - 1;
    return ctz64(m);
}
__device__ __forceinline__ int pick(unsigned word, int n) { return (int)__umulhi(word, (unsigned)n); }
// Visit the set bits of m four at a time: the four loads are issued before any result is consumed (absent bits alias the
// first one), so a set of n items costs ceil(n/4) memory round trips instead of n.  The step kernel is latency-bound.
template <class V, class L, class U> __device__ __forceinline__ void for_bits4(u64 m, int base, L load, U use) {
    while (m) {
        const u64 b0 = m & (0 - m); m ^= b0; const u64 b1 = m & (0 - m); m ^= b1;
        const u64 b2 = m & (0 - m); m ^= b2; const u64 b3 = m & (0 - m); m ^= b3;
        const int j0 = base + ctz64(b0), j1 = b1 ? base + ctz64(b1) : j0, j2 = b2 ? base + ctz64(b2) : j0, j3 = b3 ? base + ctz64(b3) : j0;
        const V v0 = load(j0), v1 = load(j1), v2 = load(j2), v3 = load(j3);
        use(b0, j0, v0); if (b1) use(b1, j1, v1); if (b2) use(b2, j2, v2); if (b3) use(b3, j3, v3);
    }
}
template <int TW> __device__ __forceinline__ u64 all_tasks(int T, int w) {
    const int r = T - 64 * w;
    return r >= 64 ? ~0ull : (r <= 0 ? 0ull : ((1ull << r) - 1));
}
// with TW == 1 the word index is a compile-time 0; for TW > 1 the word is selected without dynamic register indexing
template <int TW> __device__ __forceinline__ bool tbit(const u64 (&a)[TW], int j) {
    if (TW == 1) return (a[0] >> j) & 1ull;
    u64 w = a[0];
#pragma unroll
    for (int k = 1; k < TW; ++k) w = (j >> 6) == k ? a[k] : w;
    return (w >> (j & 63)) & 1ull;
}
template <int TW> __device__ __forceinline__ void tset(u64 (&a)[TW], int j, bool v) {
    const u64 bit = 1ull << (j & 63);
#pragma unroll
    for (int k = 0; k < TW; ++k) if (TW == 1 || (j >> 6) == k) a[k] = v ? (a[k] | bit) : (a[k] & ~bit);
}

template <int TW> __device__ __forceinline__ void ld_state(const TC& c, St<TW>& st) {
#pragma unroll
    for (int w = 0; w < TW; ++w) {
        st.feas[w] = EL(c, m_feas, TW, w); st.fin[w] = EL(c, m_fin, TW, w); st.ne[w] = EL(c, m_ne, TW, w);
        st.open[w] = EL(c, m_open, TW, w); st.dirty[w] = EL(c, m_dirty, TW, w);
    }
    st.route = EL(c, am_route, 1, 0); st.assigned = EL(c, am_assigned, 1, 0); st.returned = EL(c, am_returned, 1, 0);
    st.member = EL(c, am_member, 1, 0); st.depot = EL(c, am_depot, 1, 0); st.touched = EL(c, am_touched, 1, 0);
    st.watch = EL(c, am_watch, 1, 0);
    st.xfin = EL(c, x_fin, 1, 0); st.xamin = EL(c, x_amin, 1, 0);
    st.xret = EL(c, x_ret, 1, 0); st.xlast = EL(c, x_last, 1, 0);
}
template <int TW> __device__ __forceinline__ void st_state(const TC& c, const St<TW>& o, const St<TW>& st) {
#pragma unroll
    for (int w = 0; w < TW; ++w) {
        if (o.feas[w] != st.feas[w]) EL(c, m_feas, TW, w) = st.feas[w];
        if (o.fin[w] != st.fin[w]) EL(c, m_fin, TW, w) = st.fin[w];
        if (o.ne[w] != st.ne[w]) EL(c, m_ne, TW, w) = st.ne[w];
        if (o.open[w] != st.open[w]) EL(c, m_open, TW, w) = st.open[w];
        if (o.dirty[w] != st.dirty[w]) EL(c, m_dirty, TW, w) = st.dirty[w];
    }
    if (o.route != st.route) EL(c, am_route, 1, 0) = st.route;
    if (o.assigned != st.assigned) EL(c, am_assigned, 1, 0) = st.assigned;
    if (o.returned != st.returned) EL(c, am_returned, 1, 0) = st.returned;
    if (o.member != st.member) EL(c, am_member, 1, 0) = st.member;
    if (o.depot != st.depot) EL(c, am_depot, 1, 0) = st.depot;
    if (o.touched != st.touched) EL(c, am_touched, 1, 0) = st.touched;
    if (o.watch != st.watch) EL(c, am_watch, 1, 0) = st.watch;
    if (o.xfin != st.xfin) EL(c, x_fin, 1, 0) = st.xfin;
    if (o.xamin != st.xamin) EL(c, x_amin, 1, 0) = st.xamin;
    if (o.xret != st.xret) EL(c, x_ret, 1, 0) = st.xret;
    if (o.xlast != st.xlast) EL(c, x_last, 1, 0) = st.xlast;
}

// philox(): Philox4x32-10, dcm_philox.cuh
struct Rng { u64 seed; u64 gid; };
// decision stream: ctr = (gid_lo, gid_hi, episode, decision*8 + block), block < 8
// block 0: [0] action  [1] leader of this decision  [2],[3] followers 0,1 ; block 1: followers 2..5 ; ...
__device__ __forceinline__ uint4 draw_block(const Rng& g, unsigned episode, unsigned decision, unsigned block) {
    return philox((unsigned)g.gid, (unsigned)(g.gid >> 32), episode, decision * 8u + block, (unsigned)g.seed, (unsigned)(g.seed >> 32));
}
__device__ __forceinline__ unsigned word_of(const uint4& b, int k) { return k == 0 ? b.x : k == 1 ? b.y : k == 2 ? b.z : b.w; }

__device__ __forceinline__ void node_xy(const TC& c, unsigned node, double& x, double& y) {
    if (node == DCM_NODE_DEPOT) { x = EL(c, s_dep, 2, 0); y = EL(c, s_dep, 2, 1); }
    else { x = EL(c, s_tx, c.T, node); y = EL(c, s_ty, c.T, node); }
}
__device__ __forceinline__ bool lex_less(double ax, double ay, double bx, double by) { return ax < bx || (ax == bx && ay < by); }

// ---- node ids of all agents of one env in the thread's shared-memory scratch (TC::nws) ------------------------------
struct NodeFromScratch {
    const unsigned* w;
    __device__ __forceinline__ unsigned operator()(int i) const { return (w[(unsigned)(i >> 2) * SCR_STRIDE] >> (8 * (i & 3))) & 0xffu; }
};
__device__ __forceinline__ void scratch_set_node(unsigned* w, int i, unsigned v) {
    unsigned& x = w[(unsigned)(i >> 2) * SCR_STRIDE]; const int sh = 8 * (i & 3);
    x = (x & ~(0xffu << sh)) | (v << sh);
}
__device__ __forceinline__ void cp_async8(void* sdst, const void* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" :: "r"((unsigned)__cvta_generic_to_shared(sdst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async4(void* sdst, const void* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"((unsigned)__cvta_generic_to_shared(sdst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
// next_decision of agent i: HBM, plus the scratch copy the slot advance scans
__device__ __forceinline__ void set_nd(const TC& c, int i, double nd) {
    EL(c, a_nd, c.A, i) = nd;
    if (c.nds) c.nds[(unsigned)i * SCR_STRIDE] = nd;
}

// The head of one task's coalition record in registers.  For a task that is NOT feasible TINFO holds {amin, amax} = the earliest and
// the latest arrival over its member slots (exact, maintained by every join / removal); with them the two common outcomes of an
// evaluation -- "enough members and they arrive within max_waiting_time of each other" (:254-258) and "still short and nobody gives
// up" (:266-269) -- need NO member slot at all: mx - mn is amax - amin, and fl(now - a) >= W holds for some member iff it holds for
// the earliest one (fl is monotone).  The fused step fills the record from the loads its join needs anyway, so the task that was
// just joined is evaluated without another round trip to memory.
struct TaskR {
    int j = -1;                // task id, -1 = none
    int n = 0;                 // member count
    int status = 0, req = 0;   // stored status (may be stale, Q3), requirement
    u64 ids = 0;               // member ids of slots 0..7
    double amin = 0, amax = 0; // earliest / latest member arrival (meaningful when n > 0 and the task is not feasible)
    double dur = 0;            // task['time']
    bool feas = false;         // the task is feasible and {ts, tf} = {time_start, time_finish} are known here
    double ts = 0, tf = 0;
};

// ---------------------------------------------------------------------------------------------------------------
// task_update (task_env.py:245-281).  newly: optional per-env [T] u8 (plain row-major global) of ids that became feasible.
//
// The reference recomputes every non-feasible task on every call.  What can actually change for such a task is:
//   - its member count changed since the last call (join or removal)      -> `dirty` bit: recompute status, :252-265;
//   - a waiting member reaches fl(now - arrival) >= max_waiting_time      -> :266-271.  fl() is monotone, so the member
//     with the EARLIEST arrival (amin, kept per task) passes the test first: if it does not, nobody does.
// A non-dirty task with members therefore costs one load and one compare; everything else is evaluated exactly as written
// in the reference, including Q2 (skip after removal) and Q3 (status not refreshed after removals).
// ---------------------------------------------------------------------------------------------------------------
// route[-1] of an agent: read from memory here; the fused step passes a functor that reads its shared-memory copy (NodeFromScratch)
struct NodeFromMemory { const TC& c; __device__ __forceinline__ unsigned operator()(int m) const { return ANODE(c, m); } };

// stored status of a task: in its record (what the step reads) and in the row-major array the observation kernel streams
#define SET_STATUS(c, j, v) do { TSTAT(c, j) = (signed char)(v); EL(c, t_status, (c).T, j) = (signed char)(v); } while (0)

// counters of abandonments (u16 per agent / per task, rows of 32 lanes): bumped with a 32-bit reduction on the word that
// holds the counter of this lane and of its neighbour -- fire-and-forget, where load + add + store would make the warp wait a
// DRAM round trip for a value nothing in the step reads (only the episode accounting does; the counts stay far below 65,536)
__device__ __forceinline__ void bump_u16(unsigned short* p, unsigned by) {
    const size_t a = (size_t)p;
    atomicAdd((unsigned*)(a & ~(size_t)3), by << (8u * (unsigned)(a & 2)));
}

template <int TW, class NF> __device__ __forceinline__ void abandon(const TC& c, St<TW>& st, unsigned m, int j, const NF& node_of) {
    bump_u16(&EL(c, a_nab, c.A, m), 1u);
    if (node_of((int)m) == (unsigned)j) st.member &= ~(1ull << m);           // it no longer belongs to the task it stands at
}

// Evaluation of one non-feasible task that has members (task_env.py:250-271).  `pre` (with use_pre): the head of the task's record when
// the caller holds it in registers (the fused step, for the task that was just joined), else sector 0 of the record is loaded here.  Only the two
// rare outcomes read the member slots (one more batch, then registers only): members leave because the coalition is complete but
// spread over more than max_waiting_time (:260-265, iterates a copy: Q4), or because they have waited long enough (:266-271,
// mutates the list it iterates: Q2).  On return `pre`, when it was used, says whether the task is feasible now and carries {time_start,
// time_finish}; its count / ids / arrivals are stale after a removal (nobody uses them afterwards).
// `expect_removal`: the caller already knows that the earliest member gives up (the waiting-coalition scan), so the member slots are
// loaded together with the head instead of one round trip later.  Returns the earliest member arrival of the task afterwards, +inf when
// it no longer waits (feasible, or empty) -- the caller keeps the per-env bound St::xamin exact with it.
template <int TW, class NF> __device__ __forceinline__ double t_eval_task(const TC& c, St<TW>& st, double now, int j, unsigned char* newly, const NF& node_of, TaskR& pre,
                                                                        bool use_pre, bool expect_removal = false) {
    const int w = j >> 6; const u64 bit = 1ull << (j & 63);
    TaskR r;
    bool have_slots = false;
    auto stage_slots = [&]() { for (int s = 0; s < c.MC; ++s) cp_async8(&TMPV(c, s), &SARR(c, j, s)); have_slots = true; };   // slots past the count hold stale values that are never used
    use_pre = use_pre && pre.j == j;                                          // (`pre` is a reference to a local of the caller, never a selected pointer: it must stay in registers)
    if (use_pre) r = pre;
    else {
        if (expect_removal) stage_slots();
        const double2 mm = TINFO2(c, j); const ulonglong2 ip = TIDPACK2(c, j);                                  // sector 0 of the task's record, :250
        r.amin = mm.x; r.amax = mm.y; r.ids = ip.x;
        r.n = (int)(ip.y & 0xffu); r.status = (int)(signed char)((ip.y >> 8) & 0xffu); r.req = (int)((ip.y >> 16) & 0xffu);
        r.dur = TDUR(c, j);
    }
    double amin_after = r.amin;
    const int n = r.n; const u64 ids = r.ids;
    auto idb = [&](int s) -> unsigned { return (unsigned)(ids >> (8 * s)) & 0xffu; };
    const int stt = r.req - n;                                                // :252 (not refreshed after removals: Q3)
    if (stt != r.status) SET_STATUS(c, j, stt);
    u64 open = stt > 0 ? bit : 0, feas = 0, ne = bit, dirty = 0;
    bool removal = false;
    if (stt <= 0) {                                                           // :254
        if (r.amax - r.amin <= c.W) {                                         // :255 max(arrival) - min(arrival)
            const double mx = r.amax, tf = mx + r.dur;
            TINFO2(c, j) = make_double2(mx, tf);                              // :256-257 time_start, time_finish
            st.xfin = tf < st.xfin ? tf : st.xfin;
            feas = bit; open = 0;                                             // :258
            if (newly) newly[j] = 1;
            for (int i = 0; i < c.A; ++i)                                     // everybody who stands here (member or not, :166-171) now sees a feasible task
                if (node_of(i) == (unsigned)j) AOBS2(c, i) = make_double2(mx, tf);
            for (int s = 0; s < n; ++s) {                                     // members standing here get next_decision = time_finish
                const unsigned m = idb(s);
                if (node_of((int)m) == (unsigned)j) st.touched |= 1ull << m;
            }
            if (use_pre) { pre.feas = true; pre.ts = mx; pre.tf = tf; }
            amin_after = CUDART_INF;
        } else removal = true;
    } else removal = now - r.amin >= c.W;                                     // :269 for the earliest member (Q1: false when fl(arr+W) rounded down)
    if (removal) {
        if (!have_slots) stage_slots();
        cp_async_wait_all();
        const bool q4 = stt <= 0; const double thr = r.amax - c.W;
        int wv = 0, nab = 0; double amin = CUDART_INF, amax = -CUDART_INF; bool skip = false;
        for (int s = 0; s < n; ++s) {
            const double a = TMPV(c, s); const unsigned m = idb(s);
            // Q4 (:260-265) tests every member of a COPY of the list; Q2 (:266-271) removes from the list it iterates, so the member
            // that moves into the vacated slot is skipped by the next index and stays without being tested
            const bool out = q4 ? (a <= thr) : (!skip && now - a >= c.W);
            skip = out;
            if (out) { ++nab; abandon(c, st, m, j, node_of); }
            else {
                if (wv != s) { SARR(c, j, wv) = a; SMEM(c, j, wv) = (unsigned char)m; }
                ++wv; amin = a < amin ? a : amin; amax = a > amax ? a : amax;
            }
        }
        if (nab) {
            TNMEM(c, j) = (unsigned char)wv; bump_u16(&TNAB(c, j), (unsigned)nab);
            TINFO2(c, j) = make_double2(amin, amax);
            if (wv == 0) ne = 0;
            amin_after = amin;                                                // +inf when nobody is left
        }
        if (nab || q4) dirty = bit;                                           // the stored status is not refreshed after a removal (Q3): the next call does it
    } else if (have_slots) cp_async_wait_all();                               // never leave with copies in flight into the staging area
#pragma unroll
    for (int k = 0; k < TW; ++k) if (TW == 1 || k == w) {
        st.open[k] = (st.open[k] & ~bit) | open; st.feas[k] |= feas; st.ne[k] = (st.ne[k] & ~bit) | ne; st.dirty[k] = (st.dirty[k] & ~bit) | dirty;
    }
    return amin_after;
}

// slot_start (worker.py:50, the call right after the clock moved to `now` = min next_decision, deciders `dec`): which feasible
// tasks finish (:272-274) is read off the deciders instead of scanning every running task.  Invariant of the fused protocol: a
// feasible, unfinished task k always has a standing member m (the agent whose arrival made it feasible stays until
// time_finish) and agent_update gave every standing member next_decision = time_finish (:231).  The clock is the minimum
// next_decision, so it cannot pass time_finish_k without stopping AT it with m among the deciders, and a decider that is a
// member of a feasible task has next_decision == time_finish == now.  Hence
//     { k feasible, unfinished, now >= time_finish_k }  ==  { node(m) : m in dec, m member of a feasible unfinished task }.
// st.xfin keeps covering what the rule does not: tasks that became feasible since the last slot start (only the NEXT
// task_update call examines them, :272 is the else-branch) and states that did not come from the fused protocol
// (dcm_import_state, granular calls) until their first slot start; a slot without deciders runs the full scan.
template <int TW, class NF> __device__ __forceinline__ void t_task_update(const TC& c, St<TW>& st, double now, unsigned char* newly, const NF& node_of,
                                                                        bool slot_start, u64 dec, TaskR& pre, bool use_pre) {
    const int T = c.T;
    // ---- load-only pass: which tasks need a full evaluation, which feasible tasks have finished.  Both scans are skipped
    //      while the clock has not reached the per-env lower bounds (fl(now - x) >= W and now >= x are monotone in x).
    const bool scan_wait = now - st.xamin >= c.W, scan_fin = now >= st.xfin || (slot_start && dec == 0);
    double new_amin = CUDART_INF, new_fin = CUDART_INF;                       // new_amin: over the waiting coalitions that are NOT evaluated below
    u64 hot[TW], done[TW], expired[TW];
#pragma unroll
    for (int w = 0; w < TW; ++w) {
        hot[w] = st.dirty[w] & ~st.feas[w] & st.ne[w]; done[w] = 0;
        u64 h = 0, dn = 0;
        if (scan_wait) for (u64 m = ~st.feas[w] & st.ne[w]; m;) {               // waiting coalitions: earliest arrival only, SCR_TMP per round trip
            u64 chunk = 0; int q = 0;
            for (u64 mm = m; mm && q < SCR_TMP; mm &= mm - 1, ++q) { chunk |= mm & (0 - mm); cp_async8(&TMPV(c, q), &TINFO(c, 64 * w + ctz64(mm), 0)); }
            m &= ~chunk; cp_async_wait_all();
            q = 0;
            for (u64 mm = chunk; mm; mm &= mm - 1, ++q) {
                const u64 bit = mm & (0 - mm); const double amin = TMPV(c, q);
                if (now - amin >= c.W) h |= bit; else if (!(hot[w] & bit)) new_amin = amin < new_amin ? amin : new_amin;
            }
        }
        if (scan_fin) for (u64 m = st.feas[w] & ~st.fin[w]; m;) {                 // :272-274
            u64 chunk = 0; int q = 0;
            for (u64 mm = m; mm && q < SCR_TMP; mm &= mm - 1, ++q) { chunk |= mm & (0 - mm); cp_async8(&TMPV(c, q), &TINFO(c, 64 * w + ctz64(mm), 1)); }
            m &= ~chunk; cp_async_wait_all();
            q = 0;
            for (u64 mm = chunk; mm; mm &= mm - 1, ++q) {
                const u64 bit = mm & (0 - mm); const double tf = TMPV(c, q);
                if (now >= tf) dn |= bit; else new_fin = tf < new_fin ? tf : new_fin;
            }
        }
        expired[w] = h; hot[w] |= h; done[w] = dn;
    }
    // ---- tasks that lost their last member in an EARLIER call: status = requirements (:252 with no members); tasks whose
    //      count changed but that are feasible are not recomputed by the reference (:249)
#pragma unroll
    for (int w = 0; w < TW; ++w) {
        for (u64 mm = st.dirty[w] & ~st.feas[w] & ~st.ne[w]; mm; mm &= mm - 1) {
            const int j = 64 * w + ctz64(mm);
            SET_STATUS(c, j, TREQ(c, j));
            st.open[w] |= mm & (0 - mm);                                      // requirements >= 1
        }
        st.dirty[w] &= ~st.feas[w] & st.ne[w];
        st.fin[w] |= done[w];
    }
    if (scan_fin) st.xfin = new_fin;
    if (slot_start) {
        st.xfin = CUDART_INF;                                                 // everything feasible so far is covered by the rule from now on
        for (u64 d = dec & st.member & ~st.depot; d; d &= d - 1) {
            const int k = (int)node_of(ctz64(d));
            if (tbit<TW>(st.feas, k) && !tbit<TW>(st.fin, k)) tset<TW>(st.fin, k, true);
        }
    }
    // ---- full evaluation (rare: the task that was just joined, a coalition whose earliest member gives up)
#pragma unroll
    for (int w = 0; w < TW; ++w)
        for (u64 mm = hot[w]; mm; mm &= mm - 1) {
            const double am = t_eval_task<TW>(c, st, now, 64 * w + ctz64(mm), newly, node_of, pre, use_pre, (expired[w] & mm & (0 - mm)) != 0);
            new_amin = am < new_amin ? am : new_amin;
        }
    // After a scan the bound is EXACT again, evaluated tasks included: the next call at the same clock does not scan unless a member
    // that should have left is still there (Q2).  Without a scan it stays a lower bound (evaluations only raise a task's earliest arrival).
    if (scan_wait) st.xamin = new_amin;
    bool allf = true;
#pragma unroll
    for (int w = 0; w < TW; ++w) allf = allf && st.feas[w] == all_tasks<TW>(T, w);
    if (allf && now >= st.xret) {                                             // :277-280 depot members
        u64 ret = 0; double nx = CUDART_INF;
        for (u64 m = st.depot & st.route & ~st.returned; m;) {
            u64 chunk = 0; int q = 0;
            for (u64 mm = m; mm && q < SCR_TMP; mm &= mm - 1, ++q) { chunk |= mm & (0 - mm); cp_async8(&TMPV(c, q), &AREC(c, ctz64(mm), AR_LAST)); }
            m &= ~chunk; cp_async_wait_all();
            q = 0;
            for (u64 mm = chunk; mm; mm &= mm - 1, ++q) { const double last = TMPV(c, q); if (now >= last) ret |= mm & (0 - mm); else nx = last < nx ? last : nx; }
        }
        st.returned |= ret; st.xret = nx;
    }
}

template <int TW> __device__ __forceinline__ void t_task_update(const TC& c, St<TW>& st, double now, unsigned char* newly) {
    TaskR none;
    t_task_update<TW>(c, st, now, newly, NodeFromMemory{c}, false, 0, none, false);
}

// ---------------------------------------------------------------------------------------------------------------
// agent_update (task_env.py:207-243, reactive_planning False).
//   full:  agents in `which` are recomputed exactly as the reference does (pass st.route for its whole loop);
//   watch: members of a feasible task that are not assigned yet only need `now >= time_start` re-checked (:232-233).
// For every other agent the reference recomputes exactly what is already stored (see DESIGN.md "restricted update").
// ---------------------------------------------------------------------------------------------------------------
// `known` (fused step): a task whose {time_start, time_finish} the caller holds in registers when it is feasible -- the task that was
// just joined -- with `movers` = the agents that moved in this decision, all arriving at `arrival`.  Agents that stand at that task,
// and agents at the depot, are then updated without touching memory; the others take the general path (loads batched by four).
template <int TW, class NF> __device__ __forceinline__ void t_agent_update(const TC& c, St<TW>& st, double now, u64 which, const NF& node_of,
                                                                         const TaskR& known, bool use_known, u64 movers, double arrival) {
    const int A = c.A;
    // `assigned` of a member of a feasible task that has not started yet (:232-233) turns true at the first call with now >= time_start.
    // Nothing in the step reads it before the agent moves again, so that moment is not looked for: the agent keeps its WATCH bit and
    // a_ts = time_start, and every reader -- the observation kernels, k_export, the agent's next move -- takes
    //     assigned || (watch && now >= time_start)
    // (the clock only moves forward, so the first call that would have set it and any later look agree).
    auto member_of_feasible = [&](u64 bit, int i, double ts, double tf) {     // :229-233
        set_nd(c, i, tf);                                                     // :231 time_finish
        if (now >= ts) st.assigned |= bit;                                    // :232-233 (otherwise unchanged: Q5)
        else if (!(st.assigned & bit)) { st.watch |= bit; EL(c, a_ts, A, i) = ts; }
    };
    u64 rest = 0;                                                             // :209
    for (u64 q = which & st.route; q; q &= q - 1) {                           // first the agents that need nothing from memory
        const u64 bit = q & (0 - q); const int i = ctz64(q);
        if (st.depot & bit) { st.watch &= ~bit; set_nd(c, i, CUDART_NAN); continue; }          // :212, :226
        if (!use_known || known.j < 0 || node_of(i) != (unsigned)known.j) { rest |= bit; continue; }
        const bool fj = tbit<TW>(st.feas, known.j);
        const bool fm = fj && (st.member & bit);
        if ((fj && !known.feas) || (!fm && !(movers & bit))) { rest |= bit; continue; }   // {time_start, time_finish} / its last arrival are in memory
        st.watch &= ~bit;
        if (fm) member_of_feasible(bit, i, known.ts, known.tf);
        else { set_nd(c, i, arrival + c.W); st.assigned &= ~bit; }            // :235 / :238
    }
    // general path, five agents per trip: {time_start, time_finish} of the task each stands at and its last arrival, then the stores
    for (u64 m = rest; m;) {
        u64 chunk = 0; int q = 0;
        for (u64 mm = m; mm && q + 3 <= SCR_TMP; mm &= mm - 1, q += 3) {
            const int i = ctz64(mm); const unsigned k = node_of(i);           // not the depot: those are done
            chunk |= mm & (0 - mm);
            cp_async8(&TMPV(c, q), &TINFO(c, k, 0)); cp_async8(&TMPV(c, q + 1), &TINFO(c, k, 1)); cp_async8(&TMPV(c, q + 2), &AREC(c, i, AR_LAST));
        }
        m &= ~chunk; cp_async_wait_all();
        q = 0;
        for (u64 mm = chunk; mm; mm &= mm - 1, q += 3) {
            const u64 bit = mm & (0 - mm); const int i = ctz64(mm);
            st.watch &= ~bit;
            if (tbit<TW>(st.feas, (int)node_of(i)) && (st.member & bit)) member_of_feasible(bit, i, TMPV(c, q), TMPV(c, q + 1));
            else { set_nd(c, i, TMPV(c, q + 2) + c.W); st.assigned &= ~bit; }   // :235 / :238
        }
    }
    st.touched = 0;
}

template <int TW> __device__ __forceinline__ void t_agent_update(const TC& c, St<TW>& st, double now, u64 which) {
    TaskR none;
    t_agent_update<TW>(c, st, now, which, NodeFromMemory{c}, none, false, 0ull, 0.0);
}

// ---------------------------------------------------------------------------------------------------------------
// next_decision (task_env.py:283-289): earliest next_decision over the agents, deciders by exact equality (one pass)
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ u64 t_next_decision(const TC& c, double& t_out, const double* xlast) {
    const int A = c.A;
    double mn = CUDART_INF; u64 mask = 0;
    if (c.nds) {                                                              // fused step: the scratch copy in shared memory, no round trip
#pragma unroll 4
        for (int i = 0; i < A; ++i) {
            const double v = c.nds[(unsigned)i * SCR_STRIDE];
            if (v < mn) { mn = v; mask = 1ull << i; }                         // NaN compares false
            else if (v == mn) mask |= 1ull << i;                              // :288
        }
    } else
    for (int i0 = 0; i0 < A; i0 += 10) {                                      // ten loads in flight per round trip
        double v[10];
#pragma unroll
        for (int q = 0; q < 10; ++q) v[q] = EL(c, a_nd, A, i0 + q < A ? i0 + q : i0);
#pragma unroll
        for (int q = 0; q < 10; ++q) if (i0 + q < A) {
            if (v[q] < mn) { mn = v[q]; mask = 1ull << (i0 + q); }            // NaN compares false
            else if (v[q] == mn) mask |= 1ull << (i0 + q);                    // :288
        }
    }
    if (mask == 0) { t_out = *xlast; return 0; }                              // :285-286 everybody is NaN: the running maximum of all arrivals (St::xlast)
    t_out = mn;
    return mask;
}

// check_finished (task_env.py:366-373) given that nobody can decide
template <int TW> __device__ __forceinline__ bool t_all_returned_and_finished(const TC& c, const St<TW>& st) {
    bool ok = st.returned == (c.A >= 64 ? ~0ull : ((1ull << c.A) - 1));
#pragma unroll
    for (int w = 0; w < TW; ++w) ok = ok && st.fin[w] == all_tasks<TW>(c.T, w);
    return ok;
}

// ---------------------------------------------------------------------------------------------------------------
// get_unique_group (task_env.py:291-298) restricted to the group that acts next: pending agents standing at the
// lexicographically smallest location (np.unique(axis=0) order).  Pending agents never move while they are pending,
// so re-evaluating this after every decision walks the groups in the reference order.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ u64 t_current_group(const TC& c, u64 pending) {
    if ((pending & (pending - 1)) == 0) return pending;                       // zero or one decider
    double bx = CUDART_INF, by = CUDART_INF; u64 g = 0;
    for_bits4<double2>(pending, 0, [&](int i) { return AREC2(c, i, 0); }, [&](u64 bit, int, double2 p) {
        if (lex_less(p.x, p.y, bx, by)) { bx = p.x; by = p.y; g = bit; } else if (p.x == bx && p.y == by) g |= bit;
    });
    return g;
}

// get_unique_group (task_env.py:291-298) for the group that acts next.  Agents that stand at the same node have the same
// location, so when every pending agent stands at one node (always, in every recorded trajectory: SURVEY App. A Q10) the
// group is the pending set and no coordinate is read; otherwise the coordinates decide (t_current_group).
template <class NF> __device__ __forceinline__ u64 f_current_group(const TC& c, const NF& node_of, u64 pending) {
    if ((pending & (pending - 1)) == 0) return pending;
    const unsigned first = node_of(ctz64(pending));
    bool same = true;
    for (u64 m = pending & (pending - 1); m; m &= m - 1) same = same && node_of(ctz64(m)) == first;
    return same ? pending : t_current_group(c, pending);
}


// ---------------------------------------------------------------------------------------------------------------
// agent_step for one member (task_env.py:300-324).  (d, tt) = distance / travel time to the target from the member's
// location, (tx, ty) = target coordinate.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void travel(const TC& c, double ax, double ay, double tx, double ty, double& d, double& tt) {
    const double dx = ax - tx, dy = ay - ty;
    d = sqrt(fma(dy, dy, dx * dx));                                           // :162-163 np.linalg.norm (ddot with FMA)
    tt = d / c.vel;                                                           // :315
}
template <int TW> __device__ __forceinline__ void t_agent_step(const TC& c, St<TW>& st, double now, int i, int action, double tx, double ty,
                                                              double d, double tt, unsigned& flags) {
    const u64 bit = 1ull << i;
    const int j = action - 1;
    const bool to_task = action != 0, feas = to_task && tbit<TW>(st.feas, j), nonempty = to_task && tbit<TW>(st.ne, j);
    // ---- every load first (nothing below can be hoisted above a byte store by the compiler)
    const double2 ld = AREC2(c, i, 1);                                        // {last arrival, travel_dist}
    if (st.watch & bit) {                                                     // leaving a feasible task it was waiting to start: settle `assigned` (lazy, see t_agent_update)
        if (now >= EL(c, a_ts, c.A, i)) st.assigned |= bit;
        st.watch &= ~bit;
    }
    double2 aobs = make_double2(0.0, 0.0);                                    // observation cache (AOBS2)
    if (to_task) { if (feas) aobs = TINFO2(c, j); else aobs.y = 0.0 + TDUR(c, j); }
    int n = 0; u64 ids = 0; double amin = CUDART_INF, amax = -CUDART_INF;
    if (nonempty) {
        n = TNMEM(c, j);
        ids = TIDS(c, j);
        if (!feas) { const double2 mm = TINFO2(c, j); amin = mm.x; amax = mm.y; }   // {earliest, latest} member arrival of a waiting coalition
    }
    const double arrival = now + tt;                                          // :318
    AREC2(c, i, 1) = make_double2(arrival, ld.y + d);                         // :317-318
    AREC2(c, i, 0) = make_double2(tx, ty);                                    // :320
    ANODE(c, i) = (unsigned char)(to_task ? (unsigned)j : DCM_NODE_DEPOT);   // :314
    st.route |= bit; st.touched |= bit;
    st.xlast = arrival > st.xlast ? arrival : st.xlast;
    if (!to_task) { st.depot |= bit; st.member &= ~bit; st.xret = arrival < st.xret ? arrival : st.xret; return; }
    st.depot &= ~bit; AOBS2(c, i) = aobs;
    int pos = -1;                                                             // :321-322
    for (int sl = 0; sl < n; ++sl) { const unsigned id = (unsigned)((ids >> (8 * sl)) & 0xffu); if (id == (unsigned)i) pos = sl; }
    if (pos >= 0) {                                                           // re-visit by a current member (Q8): last arrival wins
        SARR(c, j, pos) = arrival; st.member |= bit;
        if (!feas) {
            double am = CUDART_INF, ax = -CUDART_INF;
            for (int sl = 0; sl < n; ++sl) { const double a = SARR(c, j, sl); am = a < am ? a : am; ax = a > ax ? a : ax; }
            TINFO2(c, j) = make_double2(am, ax); st.xamin = am < st.xamin ? am : st.xamin;
        }
    } else if (n < c.MC) {
        SMEM(c, j, n) = (unsigned char)i; SARR(c, j, n) = arrival;
        TNMEM(c, j) = (unsigned char)(n + 1);
        if (!feas) {
            if (n == 0) { amin = arrival; amax = arrival; } else { amin = arrival < amin ? arrival : amin; amax = arrival > amax ? arrival : amax; }
            TINFO2(c, j) = make_double2(amin, amax); st.xamin = arrival < st.xamin ? arrival : st.xamin;
        }
        tset<TW>(st.ne, j, true); tset<TW>(st.dirty, j, true);
        st.member |= bit;
    } else { flags |= ENV_ERR_OVERFLOW; st.member &= ~bit; }
}

// ---------------------------------------------------------------------------------------------------------------
// built-in policies, evaluated on the state the observation shows
// ---------------------------------------------------------------------------------------------------------------
template <int TW> __device__ __forceinline__ int t_policy_action(const TC& c, const St<TW>& st, int leader, int policy, unsigned word) {
    int n_open = 0;
#pragma unroll
    for (int w = 0; w < TW; ++w) n_open += __popcll(st.open[w]);
    if (n_open == 0) return 0;                                                // only the depot is unmasked
    if (policy == 2) {                                                        // greedy nearest (fp64 squared distance, lowest id on ties)
        const double Lx = AREC(c, leader, AR_X), Ly = AREC(c, leader, AR_Y);
        double bd = CUDART_INF; int bj = -1;
#pragma unroll
        for (int w = 0; w < TW; ++w) for (u64 mm = st.open[w]; mm; mm &= mm - 1) {
            const int j = 64 * w + ctz64(mm);
            const double dx = EL(c, s_tx, c.T, j) - Lx, dy = EL(c, s_ty, c.T, j) - Ly; const double d2 = fma(dy, dy, dx * dx);
            if (bj < 0 || d2 < bd) { bd = d2; bj = j; }
        }
        return bj + 1;
    }
    // uniform over unmasked entries of mask[0..T]; the depot bit is forbidden whenever something is open
    int k = pick(word, n_open);
#pragma unroll
    for (int w = 0; w < TW; ++w) {
        const int cnt = __popcll(st.open[w]);
        if (k < cnt) return 64 * w + kth_bit(st.open[w], k) + 1;
        k -= cnt;
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// episode accounting: calculate_waiting_time (:344-364), get_episode_reward (:420-425), worker.py:103-108.
// ---------------------------------------------------------------------------------------------------------------
template <class F> __device__ __forceinline__ double np_sum_le128(F val, int base, int n) {   // numpy pairwise add.reduce, n <= 128
    if (n < 8) { double r = 0.0; for (int i = 0; i < n; ++i) r += val(base + i); return r; }
    double r0 = val(base), r1 = val(base + 1), r2 = val(base + 2), r3 = val(base + 3), r4 = val(base + 4), r5 = val(base + 5), r6 = val(base + 6), r7 = val(base + 7);
    int i;
    for (i = 8; i < n - (n % 8); i += 8) {
        r0 += val(base + i); r1 += val(base + i + 1); r2 += val(base + i + 2); r3 += val(base + i + 3);
        r4 += val(base + i + 4); r5 += val(base + i + 5); r6 += val(base + i + 6); r7 += val(base + i + 7);
    }
    double res = ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7));
    for (; i < n; ++i) res += val(base + i);
    return res;
}
// n <= 256: numpy splits a block longer than 128 at n/2 - (n/2) % 8 and recurses into each half.  The first half is at most 128
// long; the second is longer than 128 for n = 249..256 and is split once more: blocks [0, n2), [n2, m2), [m2, n) summed as
// b0 + (b1 + b2).  One loop over the blocks keeps one copy of the block sum in the kernel.
__device__ __forceinline__ void np_blocks(int n, int& n2, int& m2) {
    n2 = m2 = n;
    if (n <= 128) return;
    n2 = n / 2; n2 -= n2 % 8;
    const int m = n - n2;
    if (m > 128) { m2 = m / 2; m2 = n2 + m2 - m2 % 8; }
}
template <class F> __device__ __forceinline__ double np_sum(F val, int n) {
    int n2, m2; np_blocks(n, n2, m2);
    double head = 0.0, tail = 0.0;
#pragma unroll 1
    for (int s = 0; s < 3; ++s) {
        const int b = s == 0 ? 0 : (s == 1 ? n2 : m2), e = s == 0 ? n2 : (s == 1 ? m2 : n);
        if (b >= e) continue;
        const double r = np_sum_le128(val, b, e - b);
        if (s == 0) head = r; else if (s == 1) tail = r; else tail += r;
    }
    return n2 < n ? head + tail : head;
}

// Thread-per-env version (granular dcm_compute_metrics).  out[8] (plain global): reward, success_rate, makespan, time_cost,
// waiting_time, travel_dist, efficiency, decisions.  Optional per-element outputs: task_wait [T], agent_wait [A].
// Returns the final clock (the trailing check_finished of :422 may move it).
template <int TW> __device__ __noinline__ double t_episode_metrics(const TC& c, const St<TW>& st, double now, unsigned n_steps, double* out,
                                                                   double* task_wait, double* agent_wait) {
    const int T = c.T, A = c.A;
    for (int i = 0; i < A; ++i) EL(c, w_agent, A, i) = 0.0;                   // :345-346
    auto task_sum = [&](int j) -> double {                                    // task['sum_waiting_time'] :349-357
        const double w_ab = (double)TNAB(c, j) * c.W;
        if (!tbit<TW>(st.ne, j)) return w_ab;
        const int n = TNMEM(c, j);
        double mx = SARR(c, j, 0);
        for (int s = 1; s < n; ++s) { const double a = SARR(c, j, s); mx = a > mx ? a : mx; }
        const bool feas = tbit<TW>(st.feas, j);
        // np.sum: sequential below 8 terms, eight accumulators combined pairwise at 8 (a full coalition of M = 8)
        return np_sum_le128([&](int s) { const double a = SARR(c, j, s); return feas ? (mx - a) : (now - a); }, 0, n) + w_ab;
    };
    // per-agent sums: tasks in id order, members in list order (:358-362); the W * abandon entries are added at the end
    // (the reference interleaves them per task, :363-364 -- differs by summation order only, ~1e-16 relative)
#pragma unroll
    for (int w = 0; w < TW; ++w) for (u64 mm = st.ne[w]; mm; mm &= mm - 1) {
        const int j = 64 * w + ctz64(mm);
        const int n = TNMEM(c, j);
        double mx = SARR(c, j, 0);
        for (int s = 1; s < n; ++s) { const double a = SARR(c, j, s); mx = a > mx ? a : mx; }
        const bool feas = (st.feas[w] >> (j & 63)) & 1ull;
        for (int s = 0; s < n; ++s) {
            const double a = SARR(c, j, s); const unsigned m = SMEM(c, j, s);
            double add;
            if (feas) add = mx - a; else { const double wv = now - a; add = wv > 0.0 ? wv : 0.0; }
            EL(c, w_agent, A, m) = EL(c, w_agent, A, m) + add;
        }
    }
    for (int i = 0; i < A; ++i) {
        double acc = EL(c, w_agent, A, i);
        for (int k = 0; k < (int)EL(c, a_nab, A, i); ++k) acc += c.W;
        EL(c, w_agent, A, i) = acc;
        if (agent_wait) agent_wait[i] = acc;
    }
    if (task_wait) for (int j = 0; j < T; ++j) task_wait[j] = task_sum(j);
    // :422 check_finished side effect on the clock
    double t; const u64 dec = t_next_decision(c, t, &st.xlast);
    if (dec == 0) now = t;
    int nfin = 0;
#pragma unroll
    for (int w = 0; w < TW; ++w) nfin += __popcll(st.fin[w]);
    out[0] = -now;                                                            // :424
    out[1] = (double)nfin / (double)T;                                        // worker.py:103
    out[2] = now;                                                             // :104
    out[3] = np_sum([&](int j) { return tbit<TW>(st.feas, j) ? TINFO(c, j, 0) : 0.0; }, T) / (double)T;   // :105 nanmean(time_start)
    out[4] = np_sum([&](int i) { return EL(c, w_agent, A, i); }, A) / (double)A;     // :106
    out[5] = np_sum([&](int i) { return AREC(c, i, AR_DIST); }, A);                  // :107
    out[6] = np_sum(task_sum, T) / (double)T;                                        // :108
    out[7] = (double)n_steps;
    return now;
}

// The clock goes back when a mover joins (or re-visits) a feasible task whose time_finish has passed: its next_decision = time_finish
// (:231) lies in the past, and the next slot starts there.  The lazy `assigned` of t_agent_update (WATCH, `now >= time_start` read at the
// current clock) would then forget that agent_update (:232-233) had set it at the later clock already.  So the step settles every watch
// against the clock before it goes back.  Returns the agents of `watch` whose time_start (a_ts, rows of 32 lanes from ts0) `now` has
// reached.  Not inlined and given values only: legal play never calls it, and the step's state stays in registers.
__device__ __noinline__ u64 t_watch_reached(const double* ts0, u64 watch, double now) {
    u64 r = 0;
    for (u64 m = watch; m; m &= m - 1) if (now >= ts0[(unsigned)ctz64(m) << 5]) r |= m & (0 - m);
    return r;
}

// ---------------------------------------------------------------------------------------------------------------
// slot boundary (worker.py:45-51, :85): check_finished, loop condition, next_decision, clock, task_update, agent_update
// ---------------------------------------------------------------------------------------------------------------
// The two updates that follow a decision (worker.py:74-76) and the slot boundary are ONE loop with ONE copy of task_update / agent_update
// in the kernel's code: trip 0 is the pair of updates after the members' moves (`pre` = the head of the joined task, `movers` arriving at
// `arrival`), every later trip a slot start.  (Two inlined copies made the step kernel 146 kB of SASS; its warps were stalled on
// instruction fetch 12 % of the time, profiles/r08c.)
template <int TW, class NF> __device__ __forceinline__ void t_update_and_advance(const TC& c, St<TW>& st, double& now, u64& pending, unsigned& flags, const NF& node_of,
                                                                                TaskR& pre, u64 movers, double arrival) {
    int empty_slots = 0; bool slot = false; u64 dec = 0;
    for (;;) {
        t_task_update<TW>(c, st, now, nullptr, node_of, slot, dec, pre, !slot);                                 // worker.py:74 / :50
        t_agent_update<TW>(c, st, now, st.touched, node_of, pre, !slot, slot ? 0ull : movers, arrival);          // worker.py:76 / :51
        if (pending) return;
        // Nobody could decide in this slot.  One such slot is normal (it marks agents as returned); a second in a row means the
        // state can no longer change and the reference `while` (worker.py:45) would spin forever: stop and flag it.
        if (slot && ++empty_slots >= 2) { flags |= ENV_DONE | ENV_STUCK; return; }
        double t; dec = t_next_decision(c, t, &st.xlast);                     // worker.py:85, :45-49
        if (dec == 0) {                                                       // check_finished :368-370
            now = t;
            if (t_all_returned_and_finished(c, st)) flags |= ENV_FINISHED;
        }
        if ((flags & ENV_FINISHED) || !(now < c.max_time)) { flags |= ENV_DONE; return; }     // worker.py:45
        pending = dec; now = t; slot = true;                                  // worker.py:47-49
    }
}

}  // namespace dcm
