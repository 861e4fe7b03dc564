// dcm_kernels.cu -- sm_100a kernels of the TaskEnv step and the C ABI of include/dcmrta.h  (thread-per-env, round 2).
//
// Kernels (state in tiled struct-of-arrays, 32 envs = one tile, see dcm_soa.h):
//   k_step          dcm_step: one leader decision per env per launch, thread / env -- action application, coalition update, agent
//                   update, slot advance, leader choice; two rounds of loads, the rest from registers and a per-thread shared-memory
//                   scratch filled with cp.async (step_env)                                                          (hot path 1/3)
//   k_step_ia       the same step for handles created with DCM_FLAG_INDIVIDUAL: one individual decision per env (worker.py:159-198)
//   k_episode_list  episode accounting + restart of the envs whose episode just ended, warp / env, beside k_obs_tile  (hot path 2/3)
//   k_obs_tile      observation + mask builder, block / tile: TMA bulk loads of the tile's arrays, rows from shared memory, TMA bulk
//                   stores straight into the policy's input tensors; launched programmatically after k_step           (hot path 3/3)
//   k_obs           the same rows by register-staged chunks (granular dcm_build_obs, shapes whose tile does not fit twice per SM)
//   k_episode       dcm_reset
//   k_granular      the individual TaskEnv methods (facade path)
//   k_routes        execute_by_route: a whole preset-route episode per env in one launch
//   k_generate      synthetic instances (generate_env distributions) with Philox
//   k_pack_static / k_unpack_static / k_export / k_import / k_init / k_sum_steps / k_sum_episodes   plumbing
//
// Build: nvcc -std=c++17 -O3 -fmad=false -gencode arch=compute_100a,code=sm_100a -lineinfo -Xcompiler -fPIC -shared
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>

#include "../../include/dcmrta.h"
#include "dcm_thread.cuh"

using namespace dcm;

#define STEP_THREADS 64         // == SCR_STRIDE (dcm_thread.cuh): the stride of the per-thread shared-memory scratch
static_assert(STEP_THREADS == SCR_STRIDE, "scratch stride");
#define OBS_THREADS 64          // 110 registers: capping them at 80 for 12 blocks / SM spills the load batches (92 vs 63 us, profiles/r02b)
#define OBS_PITCH 65            // words per env in the staging tile: 60 floats + 12 mask bytes + pad (odd => conflict-free)
#define OBS_AGENTS_PER_CHUNK 10 // 60 floats
#define OBS_ROWS_PER_CHUNK 12   // 60 floats + 12 mask bytes

// ---------------------------------------------------------------------------------------------------------------
// kernel argument blocks
// ---------------------------------------------------------------------------------------------------------------
struct EnvArgs {
    DcmSoa S;
    double W, vel, max_time;
    u64 seed, first_gid;
    unsigned cflags;
    double gen_max_duration; int gen_random_duration;
};

struct StepArgs {
    const int* action; const int* followers; int fstride; const int* leader_in; int policy;
    int* next_leader; float* reward; unsigned char* done; int* used_action;
    unsigned* elist; unsigned* ecount; unsigned* ecount_next;   // ended-env list of this pass (k_episode_list), its counter, and the next pass's counter to clear
    unsigned long long* trace;                                  // DCM_PASS_TRACE=1: [0] earliest block entry, [1] latest block exit of k_step (globaltimer ns)
    int use_nds;                                                // next_decision scratch in shared memory (handles with A <= STEP_NDS_MAX_AGENTS)
};

struct ObsArgs { const int* leader; /* [B] or NULL = the env's current leader */ float* agent_obs; float* task_obs; unsigned char* mask;
                 int skip_ended; /* envs whose episode ended in this step: 1 = leave them out (the episode kernel, running beside k_obs, writes
                                    theirs); 2 = k_obs_tile writes the observation of the restarted episode itself -- every agent at the depot, no route,
                                    status = requirements, only the depot masked: a function of the static instance alone, which the episode kernel
                                    does not touch unless it regenerates instances */ };

enum GranOp { OP_NEXT_DECISION = 1, OP_UNIQUE_GROUP, OP_SET_CLOCK, OP_GET_CLOCK, OP_TASK_UPDATE, OP_AGENT_UPDATE, OP_APPLY_MEMBERS,
              OP_CHECK_FINISHED, OP_COMPUTE_METRICS, OP_ENV_FLAGS };

struct GranArgs {
    int op;
    u64* deciders; const u64* deciders_in; double* t; const double* t_in; signed char* group_rank; unsigned char* newly;
    const int* action; const int* members; int mstride; const int* n_members; double* reward;
    unsigned char* finished; double* metrics; double* task_wait; double* agent_wait;
    unsigned* flags_out;
};

__device__ __forceinline__ TC make_tc(const EnvArgs& E, int b) {
    return TC{E.S, (unsigned)b >> 5, (unsigned)b & 31u, (size_t)((unsigned)b >> 5) * E.S.tile_stride, E.S.A, E.S.T, E.S.MC, E.W, E.vel, E.max_time};
}

// the static part of a task: row-major arrays (observation kernel, policies) and the static sector of its record (the step)
__device__ __forceinline__ void put_static(const TC& c, int j, double x, double y, unsigned rq, double du) {
    EL(c, s_tx, c.T, j) = x; EL(c, s_ty, c.T, j) = y; EL(c, s_req, c.T, j) = (unsigned char)rq;
    EL(c, s_dur, c.T, j) = du; EL(c, s_dur32, c.T, j) = __double2float_rn(du);
    TXY2(c, j) = make_double2(du, x); TREC(c, j, 6) = y; TREQ(c, j) = (unsigned char)rq;
}

// on-device instance generation for one env; Philox ctr = (gid_lo, gid_hi, instance#, 0x80000000 + 2*j + b)
__device__ __forceinline__ double u01(unsigned hi, unsigned lo) {               // 53-bit uniform in [0,1)
    return (double)(((u64)(hi >> 5) << 26) | (u64)(lo >> 6)) * (1.0 / 9007199254740992.0);
}
__device__ __noinline__ void t_generate(const TC& c, u64 seed, u64 gid, unsigned instance, double max_duration, int random_duration) {
    const unsigned k0 = (unsigned)seed, k1 = (unsigned)(seed >> 32), g0 = (unsigned)gid, g1 = (unsigned)(gid >> 32);
    for (int j = 0; j < c.T; ++j) {
        const uint4 a = philox(g0, g1, instance, 0x80000000u + 2u * j, k0, k1);
        const uint4 b = philox(g0, g1, instance, 0x80000001u + 2u * j, k0, k1);
        const double x = u01(a.x, a.y), y = u01(a.z, a.w);                                 // task_env.py:69
        const unsigned rq = 1u + (unsigned)pick(b.x, c.s.M);                                 // :71
        const double du = random_duration ? u01(b.y, b.z) * max_duration : max_duration;       // :70
        put_static(c, j, x, y, rq, du);
    }
    const uint4 a = philox(g0, g1, instance, 0xFFFFFFFFu, k0, k1);
    EL(c, s_dep, 2, 0) = u01(a.x, a.y); EL(c, s_dep, 2, 1) = u01(a.z, a.w);                // :67
}

// ---------------------------------------------------------------------------------------------------------------
// k_step: one leader decision per env
// ---------------------------------------------------------------------------------------------------------------
// every mask and bound of the env (full-warp 8-byte stores; cheaper than keeping a copy of the loaded state to diff against)
template <int TW> __device__ __forceinline__ void st_state_all(const TC& c, const St<TW>& st) {
#pragma unroll
    for (int w = 0; w < TW; ++w) {
        EL(c, m_feas, TW, w) = st.feas[w]; EL(c, m_fin, TW, w) = st.fin[w]; EL(c, m_ne, TW, w) = st.ne[w];
        EL(c, m_open, TW, w) = st.open[w]; EL(c, m_dirty, TW, w) = st.dirty[w];
    }
    EL(c, am_route, 1, 0) = st.route; EL(c, am_assigned, 1, 0) = st.assigned; EL(c, am_returned, 1, 0) = st.returned;
    EL(c, am_member, 1, 0) = st.member; EL(c, am_depot, 1, 0) = st.depot; EL(c, am_touched, 1, 0) = st.touched; EL(c, am_watch, 1, 0) = st.watch;
    EL(c, x_fin, 1, 0) = st.xfin; EL(c, x_amin, 1, 0) = st.xamin; EL(c, x_ret, 1, 0) = st.xret; EL(c, x_last, 1, 0) = st.xlast;
}

// One leader decision of env b; returns the env's status bits after it.  The duration of k_step is the length of one warp's chain
// of DEPENDENT memory round trips (the grid is less than one wave), so the decision is organised as two rounds of loads:
//   round 1  nothing depends on anything: masks, bounds, scalars; next_decision of every agent and the node ids, copied
//            asynchronously (cp.async, no registers) into the thread's shared-memory scratch (TC::nds / nws);
//   round 2  everything that depends on (action, leader) only: target coordinate, leader position, and the HEAD of the chosen
//            task's record -- count, ids, status, requirement, duration, {amin, amax} or {time_start, time_finish}.
// The members join, the joined task is evaluated (t_eval_task with the head in registers) and the movers' next_decision is set
// (t_agent_update with `known`) from registers; the slot advance scans next_decision in shared memory.  What still goes to memory
// are the rare paths: a re-visit, a removal, the waiting-coalition scan when the earliest waiting member may give up.
// IA: the individual-agent protocol of handles created with DCM_FLAG_INDIVIDUAL (worker.py:159-198), a compile-time switch so that the
// leader-follower kernel is the same code with or without it.
template <int TW, bool IA>
__device__ __forceinline__ unsigned step_env(const EnvArgs& E, const StepArgs& F, int b, double* nds, unsigned* nws, double* tmp) {
    TC c = make_tc(E, b); c.nds = F.use_nds ? nds : nullptr; c.nws = nws; c.tmp = tmp;
    const int A = c.A, T = c.T;
    // ---- round 1
    if (F.use_nds) for (int i = 0; i < A; ++i) cp_async8(&nds[(unsigned)i * SCR_STRIDE], &EL(c, a_nd, A, i));
    for (int k = 0; k < (A + 3) >> 2; ++k) cp_async4(&nws[(unsigned)k * SCR_STRIDE], &ANODE_WORD(c, k));
    unsigned flags = EL(c, flags, 1, 0) & ~ENV_FRESH;
    St<TW> st; ld_state(c, st);
    double now = EL(c, now, 1, 0); u64 pending = EL(c, pending, 1, 0), group = EL(c, group, 1, 0);
    unsigned n_steps = EL(c, n_steps, 1, 0); const unsigned episode = EL(c, episode, 1, 0), total = EL(c, total, 1, 0);
    int leader = EL(c, leader, 1, 0);
    const int ext_action = F.policy == 0 ? F.action[b] : 0;
    const int inj = F.leader_in ? F.leader_in[b] : -1;                        // injected leader of the NEXT decision (trace replay)
    cp_async_wait_all();
    if (flags & ENV_DONE) {                                                   // finished earlier and not restarted: untouched
        if (F.next_leader) F.next_leader[b] = -1;
        if (F.reward) F.reward[b] = 0.f;
        if (F.done) F.done[b] = 1;
        if (F.used_action) F.used_action[b] = -1;
        return flags;
    }
    const NodeFromScratch node_of{nws};              // route[-1] of every agent: who stands where decides the groups without reading coordinates
    const Rng rng{E.seed, E.first_gid + (u64)b};
    float reward_out = 0.f; int action_out = -1;

    bool ok = true;
    uint4 b0 = make_uint4(0, 0, 0, 0);
    bool have_b0 = false;
    int action;
    if (F.policy == 1) { b0 = draw_block(rng, episode, n_steps, 0); have_b0 = true; action = t_policy_action(c, st, leader, 1, b0.x); }
    else if (F.policy == 2) action = t_policy_action(c, st, leader, 2, 0);
    else action = ext_action;
    if (action < 0 || action > T) { flags |= ENV_ERR_ACTION; ok = false; }
    const bool to_task = ok && action != 0; const int j = to_task ? action - 1 : 0;
    const bool feas_j = to_task && tbit<TW>(st.feas, j), ne_j = to_task && tbit<TW>(st.ne, j);
    // ---- round 2
    double tx = 0.0, ty = 0.0; double2 Lp = make_double2(0.0, 0.0), ti = make_double2(0.0, 0.0);
    TaskR tr;
    if (ok) {
        Lp = AREC2(c, leader, 0);
        if (to_task) {
            ti = TINFO2(c, j); const ulonglong2 ip = TIDPACK2(c, j);           // the chosen task's record: one 64-byte line
            const double2 dx = TXY2(c, j); ty = TREC(c, j, 6);
            tr.dur = dx.x; tx = dx.y; tr.ids = ip.x;                            // (count / ids / times are stale when the task has no members: not used then)
            tr.n = (int)(ip.y & 0xffu); tr.status = (int)(signed char)((ip.y >> 8) & 0xffu); tr.req = (int)((ip.y >> 16) & 0xffu);
        } else { tx = EL(c, s_dep, 2, 0); ty = EL(c, s_dep, 2, 1); }
    }
    // task_env.py:328.  Individual agent (DCM_FLAG_INDIVIDUAL, worker.py:170-186): the leader moves alone whatever the stored group
    // holds (dcm_import_state may install a leader-follower record in the middle of a slot): no followers, and the depot takes only it
    int want = 0; u64 g = IA ? 0ull : group & ~(1ull << leader);
    const int* fp = F.followers ? F.followers + (size_t)b * F.fstride : nullptr;
    if (ok) {
        const int vacancy = action == 0 ? __popcll(group) : tr.status;        // :327
        if (vacancy > 1) { const int avail = __popcll(g); want = vacancy - 1 < avail ? vacancy - 1 : avail; }   // :330-331
        if (fp && action != 0) {                                              // validate injected followers before touching state
            u64 gg = g;
            for (int k = 0; k < want && ok; ++k) {
                const int fo = k < F.fstride ? fp[k] : -1;
                if (fo < 0 || fo >= A || !((gg >> fo) & 1ull)) ok = false; else gg &= ~(1ull << fo);
            }
            if (ok && want < F.fstride && fp[want] >= 0) ok = false;
            if (!ok) flags |= ENV_ERR_FOLLOW;
        }
    }
    if (ok) {
        action_out = action;
        // every member stands where the leader stands and goes to the same node: one distance and one arrival for all (:315-318)
        const unsigned target = to_task ? (unsigned)j : DCM_NODE_DEPOT;
        // observation cache of the movers (AOBS2, dcm_thread.cuh): what their agent row shows of the task they now stand at
        double2 aobs = make_double2(0.0, 0.0);
        if (to_task) { if (feas_j) aobs = ti; else aobs.y = 0.0 + tr.dur; }
        // the task's membership was read ONCE (round 2) and stays in registers while the members join (the reference re-reads its
        // lists per agent_step); {amin, amax} = earliest / latest member arrival of a waiting coalition
        int n = ne_j ? tr.n : 0; u64 ids = tr.ids;
        const bool waiting = ne_j && !feas_j;
        double amin = waiting ? ti.x : CUDART_INF, amax = waiting ? ti.y : -CUDART_INF;
        const int n0 = n; bool mm_new = false, revisit = false;
        double d, tt; travel(c, Lp.x, Lp.y, tx, ty, d, tt);
        const double arrival = now + tt;                                      // :318
        double reward = 0.0; int nm = 0; u64 movers = 0;
        auto move = [&](int i) {                                              // agent_step (:300-324)
            const u64 bit = 1ull << i;
            AREC2(c, i, 0) = make_double2(tx, ty);                            // :320
            AREC(c, i, AR_LAST) = arrival;                                    // :318
            atomicAdd(&AREC(c, i, AR_DIST), d);                               // :317 travel_dist += d: a reduction, no load
            ANODE(c, i) = (unsigned char)target; scratch_set_node(nws, i, target);   // :314
            st.route |= bit; st.touched |= bit; pending &= ~bit; movers |= bit;
            // a mover that was waiting for its feasible task to start (WATCH) decides at that task's time_finish >= time_start: `assigned`
            // has turned true meanwhile (lazy, see t_agent_update)
            if (st.watch & bit) { st.assigned |= bit; st.watch &= ~bit; }
            if (!to_task) { st.depot |= bit; st.member &= ~bit; }
            else {
                st.depot &= ~bit; AOBS2(c, i) = aobs;
                int pos = -1;                                                 // :321-322
#pragma unroll
                for (int sl = 0; sl < 8; ++sl) if (sl < n && ((unsigned)(ids >> (8 * sl)) & 0xffu) == (unsigned)i) pos = sl;
                if (pos >= 0) {                                               // re-visit by a current member (Q8): last arrival wins
                    SARR(c, j, pos) = arrival; st.member |= bit; revisit = true;
                } else if (n < c.MC) {
                    SMEM(c, j, n) = (unsigned char)i; SARR(c, j, n) = arrival;
                    ids = (ids & ~(0xffull << (8 * n))) | ((u64)(unsigned)i << (8 * n));                      // (slots past n hold stale ids)
                    if (n == 0) { amin = arrival; amax = arrival; } else { amin = arrival < amin ? arrival : amin; amax = arrival > amax ? arrival : amax; }
                    mm_new = true; ++n; st.member |= bit;
                } else { flags |= ENV_ERR_OVERFLOW; st.member &= ~bit; }
            }
            reward += -tt; ++nm;
        };
        move(leader);
        if (action == 0) {                                                    // Q11: the whole remaining group follows to the depot
            for (; g; g &= g - 1) move(ctz64(g));
        } else {
            uint4 blk = b0;
            for (int k = 0; k < want; ++k) {
                int fo;
                if (fp) fo = fp[k];                                           // injected (trace replay)
                else {                                                        // :331 uniform without replacement
                    const int slot = 2 + k;
                    if ((slot & 3) == 0 || !have_b0) { blk = draw_block(rng, episode, n_steps, (unsigned)(slot >> 2)); have_b0 = true; }
                    fo = kth_bit(g, pick(word_of(blk, slot & 3), __popcll(g)));
                }
                g &= ~(1ull << fo);
                move(fo);
            }
        }
        st.xlast = arrival > st.xlast ? arrival : st.xlast;
        if (!to_task) st.xret = arrival < st.xret ? arrival : st.xret;
        else {
            if (n != n0) { TNMEM(c, j) = (unsigned char)n; tset<TW>(st.ne, j, true); tset<TW>(st.dirty, j, true); }
            if (!feas_j) {
                if (revisit) {                                                // rare: the slots, in one batch (a loop of dependent loads otherwise)
                    for (int sl = 0; sl < n; ++sl) cp_async8(&TMPV(c, sl), &SARR(c, j, sl));
                    cp_async_wait_all();
                    amin = CUDART_INF; amax = -CUDART_INF;
                    for (int sl = 0; sl < n; ++sl) { const double a = TMPV(c, sl); amin = a < amin ? a : amin; amax = a > amax ? a : amax; }
                    mm_new = true;
                }
                if (mm_new) { TINFO2(c, j) = make_double2(amin, amax); st.xamin = amin < st.xamin ? amin : st.xamin; }
            }
            tr.j = j; tr.n = n; tr.ids = ids; tr.amin = amin; tr.amax = amax;  // the head the evaluation below starts from
            tr.feas = feas_j; tr.ts = ti.x; tr.tf = ti.y;
        }
        reward_out = __double2float_rn(reward / (double)nm);                  // :337-341
        ++n_steps; EL(c, total, 1, 0) = total + 1;
        t_update_and_advance<TW>(c, st, now, pending, flags, node_of, tr, movers, arrival);    // worker.py:74-76, then :85 / :45-51 while nobody is pending
        if (flags & ENV_DONE) { leader = -1; group = 0; }                     // episode accounting / restart: k_episode_list
        else {
            group = IA ? pending & (0ull - pending)                           // the lowest pending id acts next (worker.py:170)
                       : f_current_group(c, node_of, pending);                // task_env.py:291-298
            if (inj >= 0) {
                if (inj < A && ((group >> inj) & 1ull)) leader = inj;
                else { flags |= ENV_ERR_LEADER; leader = ctz64(group); }
            } else {
                const int ng = __popcll(group);
                leader = ng == 1 ? ctz64(group) : kth_bit(group, pick(draw_block(rng, episode, n_steps, 0).y, ng));   // worker.py:54
            }
        }
    }
    int leader_out = leader;
    if ((flags & ENV_DONE) && (E.cflags & DCM_FLAG_AUTO_RESET) && 0.0 < E.max_time) {
        // The episode kernel restarts this env; the first leader of the new episode (episode_env, worker.py:54) is a function of the
        // RNG contract alone, so the OUTPUT carries it already: next_leader, reward and done are then final when k_step ends and
        // dcm_step_host sends them to the host while the episode and observation kernels run.  (The stored leader stays -1.)
        if (IA) leader_out = 0;                                               // agent 0 starts (episode_env flags any other injected leader)
        else if (inj >= 0) leader_out = inj < A ? inj : 0;
        else if (A == 1) leader_out = 0;
        else leader_out = kth_bit(A >= 64 ? ~0ull : ((1ull << A) - 1), pick(draw_block(rng, episode + 1, 0, 0).y, A));
    }
    if (F.next_leader) F.next_leader[b] = leader_out;
    if (F.reward) F.reward[b] = reward_out;
    if (F.done) F.done[b] = (flags & ENV_DONE) ? 1 : 0;
    if (F.used_action) F.used_action[b] = action_out;
    EL(c, now, 1, 0) = now; EL(c, pending, 1, 0) = pending; EL(c, group, 1, 0) = group; EL(c, n_steps, 1, 0) = n_steps;
    EL(c, leader, 1, 0) = leader; EL(c, flags, 1, 0) = flags; EL(c, ended, 1, 0) = (flags & ENV_DONE) ? 1 : 0;
    if (ok) st_state_all(c, st);
    return flags;
}

// per-thread scratch of the fused step: [SCR_TMP][64] staging doubles, [A][64] next_decision, [ANB/4][64] node-id words
// (the next_decision rows only for handles with A <= STEP_NDS_MAX_AGENTS: the scratch is carved from the L1 the step's sparse accesses
// live on -- measured at 65,536 envs: 20A/50T 122.2 us with it / 123.0 without, 30A/100T 244.0 with / 230.9 without, profiles/r09_nds_scratch.txt)
#define STEP_NDS_MAX_AGENTS 24
__host__ __device__ inline size_t step_smem_bytes(int A, int ANB, bool nds) { return (size_t)STEP_THREADS * (8 * (size_t)(SCR_TMP + (nds ? A : 0)) + (size_t)ANB); }

template <int TW, bool IA>
__device__ __forceinline__ void step_pass(const EnvArgs& E, const StepArgs& F, unsigned char* step_smem) {
    const int b = blockIdx.x * STEP_THREADS + threadIdx.x;
    unsigned flags = 0;
    // programmatic dependent launch: the observation kernel that follows in the stream may become resident (and run its prologue) as SM
    // resources free up; it waits for this grid to complete (griddepcontrol.wait) before it touches the state
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (F.trace && threadIdx.x == 0) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); atomicMin(F.trace, t); }
    double* const tmp = (double*)step_smem + threadIdx.x; double* const nds = tmp + SCR_TMP * STEP_THREADS;
    if (b < E.S.B) flags = step_env<TW, IA>(E, F, b, nds, (unsigned*)(nds - threadIdx.x + (size_t)STEP_THREADS * (F.use_nds ? E.S.A : 0)) + threadIdx.x, tmp);
    if (F.elist) {                                                            // envs whose episode just ended: one warp-aggregated append per warp that has any
        const bool need = (flags & ENV_DONE) && !(flags & ENV_ACCOUNTED);
        const unsigned m = __ballot_sync(0xffffffffu, need), lane = threadIdx.x & 31u;
        if (m) {
            unsigned base = 0;
            if (lane == (unsigned)(__ffs(m) - 1)) base = atomicAdd(F.ecount, (unsigned)__popc(m));
            base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
            if (need) F.elist[base + __popc(m & ((1u << lane) - 1u))] = (unsigned)b;
        }
        if (b == 0) *F.ecount_next = 0;
    }
    if (F.trace && (threadIdx.x & 31) == 0) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); atomicMax(F.trace + 1, t); }
}

template <int TW>
__global__ void __launch_bounds__(STEP_THREADS, 7) k_step(const __grid_constant__ EnvArgs E, const __grid_constant__ StepArgs F) {
    extern __shared__ __align__(16) unsigned char step_smem[];
    step_pass<TW, false>(E, F, step_smem);
}

// dcm_step of a DCM_FLAG_INDIVIDUAL handle: one individual decision per env
template <int TW>
__global__ void __launch_bounds__(STEP_THREADS, 7) k_step_ia(const __grid_constant__ EnvArgs E, const __grid_constant__ StepArgs F) {
    extern __shared__ __align__(16) unsigned char step_smem[];
    step_pass<TW, true>(E, F, step_smem);
}

// ---------------------------------------------------------------------------------------------------------------
// k_episode: episode accounting (worker.py:87, :103-108) and restart (clear_decisions + first slot + first leader) for
// the envs that need it -- about 1 env in 125 per step -- done WARP-COOPERATIVELY (lanes over tasks / agents) by the
// warp that owns the tile, so that this rare, long path stays off the critical path of k_step.
//   mode 0: envs that k_step just finished (DONE and not yet ACCOUNTED); restart only with DCM_FLAG_AUTO_RESET (k_episode_list)
//   mode 1: dcm_reset (every env, or those selected by `which`) (k_episode)
// ---------------------------------------------------------------------------------------------------------------
#define EPI_WARPS 4
// k_episode_list runs EPI_LIST_WARPS envs (warps) per block and EPI_LIST_WARPS_PER_SM warps per SM.  Its __launch_bounds__ are
// sized for blocks of EPI_LIST_REG_BUDGET_WARPS warps, five per SM: that caps it at 96 registers, which is what lets its warps stay
// co-resident with two k_obs_tile blocks (DESIGN.md section 4, late round-1 findings (1)).
#define EPI_LIST_REG_BUDGET_WARPS 4
#define EPI_LIST_WARPS 2
#define EPI_LIST_WARPS_PER_SM 8
struct EpiArgs { int mode; const unsigned char* which; const int* leader_in; int* next_leader; double* metrics;
                 ObsArgs obs; int write_obs; /* mode 0 + auto-reset: write the restarted env's observation (k_obs runs beside this kernel and skips it) */ };

__device__ __forceinline__ double wmax(double v) { for (int o = 16; o > 0; o >>= 1) { const double w = __shfl_xor_sync(0xffffffffu, v, o); v = w > v ? w : v; } return v; }
__device__ __forceinline__ double wmin(double v) { for (int o = 16; o > 0; o >>= 1) { const double w = __shfl_xor_sync(0xffffffffu, v, o); v = w < v ? w : v; } return v; }

// per-warp scratch of k_episode, carved from dynamic shared memory: the four vectors that are summed (the member data of a task
// stays in the registers of the lane that owns it, w_episode_metrics8)
struct EpiScratch { double *s_task, *s_ts; /* [T] */ double *s_agent, *s_dist; /* [A] */ };
__host__ __device__ inline size_t epi_scratch_bytes(int A, int T, int) { return (size_t)8 * (2 * T + 2 * A); }
__device__ __forceinline__ EpiScratch epi_scratch(unsigned char* base, int A, int T, int) {
    EpiScratch S; double* d = (double*)base;
    S.s_task = d; d += T; S.s_ts = d; d += T; S.s_agent = d; d += A; S.s_dist = d;
    return S;
}

// numpy pairwise add.reduce of n <= 128 values in shared memory by 8 lanes (lane8 = 0..7 of the group); same order of
// additions as np_sum_le128: eight strided accumulators, ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the tail
__device__ __forceinline__ double g_np_sum_le128(const double* v, int base, int n, unsigned lane8, unsigned gmask) {
    if (n < 8) { double r = 0.0; for (int i = 0; i < n; ++i) r += v[base + i]; return r; }
    double r = v[base + lane8];
    int i;
    for (i = 8; i < n - (n % 8); i += 8) r += v[base + i + lane8];
    const double p1 = r + __shfl_xor_sync(gmask, r, 1);                       // lanes 0,2,4,6 hold r0+r1, r2+r3, ...
    const double p2 = p1 + __shfl_xor_sync(gmask, p1, 2);                     // lanes 0,4 hold (r0+r1)+(r2+r3), ...
    double res = p2 + __shfl_xor_sync(gmask, p2, 4);                          // lane 0: the eight-way combination in numpy's order
    for (; i < n; ++i) res += v[base + i];
    return res;                                                               // valid in lane8 == 0
}
// n <= 256: numpy's recursion, blocks of np_blocks (dcm_thread.cuh) summed as b0 + (b1 + b2), one copy of the block sum
__device__ __forceinline__ double g_np_sum(const double* v, int n, unsigned lane8, unsigned gmask) {
    int n2, m2; np_blocks(n, n2, m2);
    double head = 0.0, tail = 0.0;
#pragma unroll 1
    for (int s = 0; s < 3; ++s) {
        const int b = s == 0 ? 0 : (s == 1 ? n2 : m2), e = s == 0 ? n2 : (s == 1 ? m2 : n);
        if (b >= e) continue;
        const double r = g_np_sum_le128(v, b, e - b, lane8, gmask);
        if (s == 0) head = r; else if (s == 1) tail = r; else tail += r;
    }
    return n2 < n ? head + tail : head;
}

// out[8]: reward, success_rate, makespan, time_cost, waiting_time, travel_dist, efficiency, decisions.  Returns the final clock.
// Warp-cooperative, lane <-> task: every load of a 32-task batch is issued in one round (and the next batch's before this one is
// consumed); the four final sums run on four groups of 8 lanes in numpy's pairwise order.
template <int TW>
__device__ __forceinline__ double w_episode_metrics8(const TC& c, const St<TW>& st, unsigned lane, double now, unsigned n_steps, double* out, const EpiScratch& S) {
    const int T = c.T, A = c.A, MC = c.MC;
    struct TL { int n; bool feas; u64 ids; double a[8]; unsigned nab; double ts; };
    auto load_task = [&](int j, TL& L) {
        L.n = 0; L.feas = false; L.ids = 0; L.nab = 0; L.ts = 0.0;
        const bool in = j < T; const int jj = in ? j : 0;
        const bool ne = in && tbit<TW>(st.ne, jj); L.feas = in && tbit<TW>(st.feas, jj);
        if (ne) { L.n = TNMEM(c, jj); L.ids = TIDS(c, jj); }
#pragma unroll
        for (int s2 = 0; s2 < 8; ++s2) L.a[s2] = (ne && s2 < MC) ? SARR(c, jj, s2) : 0.0;
        if (in) L.nab = TNAB(c, jj);
        if (L.feas) L.ts = TINFO(c, jj, 0);
    };
    // agents (lane, lane + 32): issue these loads first as well
    double a_nd_v[2], a_last[2], a_dist[2]; int a_nab_v[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int i = lane + 32 * r; const bool in = i < A; const int ii = in ? i : 0;
        a_nd_v[r] = in ? EL(c, a_nd, A, ii) : CUDART_NAN; const double2 ld = AREC2(c, ii, 1);
        a_last[r] = in ? ld.x : 0.0; a_dist[r] = ld.y; a_nab_v[r] = in ? (int)EL(c, a_nab, A, ii) : 0;
    }
    double acc0 = 0.0, acc1 = 0.0;
    TL cur, nxt;
    load_task((int)lane, cur);
    for (int j0 = 0; j0 < T; j0 += 32) {
        if (j0 + 32 < T) load_task(j0 + 32 + (int)lane, nxt);
        const int j = j0 + (int)lane; const int n = cur.n; const bool feas = cur.feas;
        double mx = 0.0;
#pragma unroll
        for (int s2 = 0; s2 < 8; ++s2) if (s2 < n) mx = (s2 == 0 || cur.a[s2] > mx) ? cur.a[s2] : mx;
        if (j < T) {                                                          // task['sum_waiting_time'] :349-357
            const double w_ab = (double)cur.nab * c.W;
            double v = w_ab;
            if (n) {
                double acc = 0.0;
#pragma unroll
                for (int s2 = 0; s2 < 8; ++s2) if (s2 < n) acc += feas ? (mx - cur.a[s2]) : (now - cur.a[s2]);
                v = acc + w_ab;
            }
            S.s_task[j] = v;
            S.s_ts[j] = feas ? cur.ts : 0.0;
        }
        // agent['sum_waiting_time'] in the reference order: tasks ascending, members in list order (:358-362).  The task's count,
        // latest arrival, ids and arrivals are broadcast from the lane that holds them (no staging in shared memory: the scratch
        // of a block stays small enough for four of these blocks beside two k_obs_tile blocks on an SM)
#pragma unroll
        for (int s2 = 0; s2 < 8; ++s2) {                                      // in place: what each member of this lane's task waited, :360 / :362
            const double wv = now - cur.a[s2]; cur.a[s2] = feas ? mx - cur.a[s2] : (wv > 0.0 ? wv : 0.0);
        }
        for (unsigned tm = __ballot_sync(0xffffffffu, n > 0); tm; tm &= tm - 1) {
            const int t = __ffs(tm) - 1;
            const int cnt = __shfl_sync(0xffffffffu, n, t); const u64 idt = __shfl_sync(0xffffffffu, cur.ids, t);
#pragma unroll
            for (int s2 = 0; s2 < 8; ++s2) if (s2 < cnt) {                    // cnt is warp-uniform
                const double add = __shfl_sync(0xffffffffu, cur.a[s2], t);
                const unsigned m = (unsigned)(idt >> (8 * s2)) & 0xffu;
                if (lane == (m & 31u)) { if (m < 32u) acc0 += add; else acc1 += add; }
            }
        }
        cur = nxt;
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {                                             // + W per abandoned_agent entry (:363-364; added last, ~1e-16 rel.)
        const int i = lane + 32 * r;
        if (i < A) {
            double acc = r ? acc1 : acc0;
            for (int k = 0; k < a_nab_v[r]; ++k) acc += c.W;
            S.s_agent[i] = acc; S.s_dist[i] = a_dist[r];
        }
    }
    // :422 check_finished side effect on the clock
    double mn = CUDART_INF, la = 0.0;
#pragma unroll
    for (int r = 0; r < 2; ++r) { if (a_nd_v[r] < mn) mn = a_nd_v[r]; la = a_last[r] > la ? a_last[r] : la; }
    mn = wmin(mn); la = wmax(la);
    if (mn == CUDART_INF) now = la;
    int nfin = 0;
#pragma unroll
    for (int w = 0; w < TW; ++w) nfin += __popcll(st.fin[w]);
    __syncwarp();
    {                                                                         // four sums on four groups of 8 lanes
        const unsigned grp = lane >> 3, lane8 = lane & 7, gmask = 0xffu << (8 * grp);
        double r;
        if (grp == 0) r = g_np_sum(S.s_ts, T, lane8, gmask);                  // :105 nanmean(time_start)
        else if (grp == 1) r = g_np_sum(S.s_agent, A, lane8, gmask);          // :106
        else if (grp == 2) r = g_np_sum(S.s_dist, A, lane8, gmask);           // :107
        else r = g_np_sum(S.s_task, T, lane8, gmask);                         // :108
        if (lane8 == 0) {
            if (grp == 0) { out[3] = r / (double)T; out[0] = -now; out[1] = (double)nfin / (double)T; out[2] = now; out[7] = (double)n_steps; }   // :424, worker.py:103-104
            else if (grp == 1) out[4] = r / (double)A;
            else if (grp == 2) out[5] = r;
            else out[6] = r / (double)T;
        }
    }
    __syncwarp();
    return now;
}

// episode accounting (mode 0) and restart of ONE env by a whole warp.  With O (fused pass, auto-reset) the observation of
// the restarted env is written from registers: every agent stands at the depot without a route, so the agent rows are zero,
// task row j is [requirement, requirement, duration, task - depot] and only the depot is masked (task_env.py:165-200).
template <int TW>
__device__ __forceinline__ void episode_env(const EnvArgs& E, const EpiArgs& P, int be, unsigned lane, const EpiScratch& scratch, const ObsArgs* O = nullptr) {
    const int A = E.S.A, T = E.S.T;
    const TC c = make_tc(E, be);
    St<TW> st; ld_state(c, st);
    unsigned flags = EL(c, flags, 1, 0), episode = EL(c, episode, 1, 0);
    unsigned inst = EL(c, instance, 1, 0);
    const u64 gid = E.first_gid + (u64)be;
    const bool regen = P.mode == 0 && (E.cflags & DCM_FLAG_REGENERATE);
    if (P.mode == 0) {
        const double now0 = EL(c, now, 1, 0); const unsigned ns = EL(c, n_steps, 1, 0);
        const double now = w_episode_metrics8(c, st, lane, now0, ns, P.metrics + (size_t)be * 8, scratch);
        ++episode; flags |= ENV_ACCOUNTED;
        if (!(E.cflags & DCM_FLAG_AUTO_RESET)) {
            if (lane == 0) { EL(c, now, 1, 0) = now; EL(c, flags, 1, 0) = flags; EL(c, episode, 1, 0) = episode; }
            __syncwarp();
            return;
        }
        if (regen) { ++inst; if (lane == 0) EL(c, instance, 1, 0) = inst; }
    }
    const bool alive = 0.0 < E.max_time;
    const bool obs = O && alive;
    // ---- the instance: generated (same streams as t_generate) or read back; everything below uses registers only
    const unsigned k0 = (unsigned)E.seed, k1 = (unsigned)(E.seed >> 32), g0 = (unsigned)gid, g1 = (unsigned)(gid >> 32);
    double dx, dy;
    if (regen) { const uint4 a = philox(g0, g1, inst, 0xFFFFFFFFu, k0, k1); dx = u01(a.x, a.y); dy = u01(a.z, a.w); if (lane == 0) { EL(c, s_dep, 2, 0) = dx; EL(c, s_dep, 2, 1) = dy; } }
    else { dx = EL(c, s_dep, 2, 0); dy = EL(c, s_dep, 2, 1); }
    // ---- clear_decisions (task_env.py:129-140), lanes over tasks / agents
    for (int j = lane; j < T; j += 32) {
        double tx, ty, du; unsigned rq;
        if (regen) {
            const uint4 a = philox(g0, g1, inst, 0x80000000u + 2u * j, k0, k1);
            const uint4 b2 = philox(g0, g1, inst, 0x80000001u + 2u * j, k0, k1);
            tx = u01(a.x, a.y); ty = u01(a.z, a.w);                            // task_env.py:69
            rq = 1u + (unsigned)pick(b2.x, E.S.M);                            // :71
            du = E.gen_random_duration ? u01(b2.y, b2.z) * E.gen_max_duration : E.gen_max_duration;   // :70
            put_static(c, j, tx, ty, rq, du);
        } else { rq = EL(c, s_req, T, j); if (obs) { tx = EL(c, s_tx, T, j); ty = EL(c, s_ty, T, j); du = EL(c, s_dur, T, j); } }
        TPACK(c, j) = ((u64)rq << 8) | ((u64)rq << 16);                        // no member, status = requirement, nobody abandoned (:129-140)
        EL(c, t_status, T, j) = (signed char)rq;
        if (obs) {
            if (O->task_obs) {
                float* r = O->task_obs + ((size_t)be * (T + 1) + j + 1) * 5;  // :185-186
                r[0] = (float)(int)rq; r[1] = (float)rq; r[2] = __double2float_rn(du); r[3] = __double2float_rn(tx - dx); r[4] = __double2float_rn(ty - dy);
            }
            if (O->mask) O->mask[(size_t)be * (T + 1) + j + 1] = 0;           // :199 every task is open
        }
    }
    if (obs) {
        if (O->task_obs && lane < 5) O->task_obs[(size_t)be * (T + 1) * 5 + lane] = 0.f;       // :188 depot row (depot - depot)
        if (O->mask && lane == 0) O->mask[(size_t)be * (T + 1)] = 1;                            // worker.py:58-61
        if (O->agent_obs) for (int k = lane; k < 6 * A; k += 32) O->agent_obs[(size_t)be * 6 * A + k] = 0.f;   // :165-180 nobody has a route
    }
    for (int i = lane; i < A; i += 32) {
        AREC2(c, i, 0) = make_double2(dx, dy); AREC2(c, i, 1) = make_double2(0.0, 0.0);
        EL(c, a_nd, A, i) = 0.0; ANODE(c, i) = DCM_NODE_DEPOT; EL(c, a_nab, A, i) = 0;
    }
    // ---- first slot (worker.py:45-51): every agent decides at t = 0 from the depot, nothing to update; one group (individual
    // agent: every agent decides, agent 0 first, worker.py:170)
    const u64 all = A >= 64 ? ~0ull : ((1ull << A) - 1);
    unsigned nflags = P.mode == 0 ? ENV_FRESH : 0u; u64 pending = all, group = all; int leader;
    if (!alive) { nflags = ENV_DONE | ENV_ACCOUNTED; pending = 0; group = 0; leader = -1; }
    else {
        const int inj = P.leader_in ? P.leader_in[be] : -1;
        if (E.cflags & DCM_FLAG_INDIVIDUAL) { group = 1; leader = 0; if (inj > 0) nflags |= ENV_ERR_LEADER; }
        else if (inj >= 0) { if (inj < A) leader = inj; else { nflags |= ENV_ERR_LEADER; leader = 0; } }
        else if (A == 1) leader = 0;
        else { const Rng rng{E.seed, gid}; leader = kth_bit(all, pick(draw_block(rng, episode, 0, 0).y, A)); }   // worker.py:54
    }
    if (lane == 0) {
#pragma unroll
        for (int w = 0; w < TW; ++w) {
            EL(c, m_feas, TW, w) = 0; EL(c, m_fin, TW, w) = 0; EL(c, m_ne, TW, w) = 0; EL(c, m_dirty, TW, w) = 0;
            EL(c, m_open, TW, w) = all_tasks<TW>(T, w);
        }
        EL(c, am_route, 1, 0) = 0; EL(c, am_assigned, 1, 0) = 0; EL(c, am_returned, 1, 0) = 0; EL(c, am_member, 1, 0) = 0;
        EL(c, am_depot, 1, 0) = 0; EL(c, am_touched, 1, 0) = 0; EL(c, am_watch, 1, 0) = 0;
        EL(c, x_fin, 1, 0) = CUDART_INF; EL(c, x_amin, 1, 0) = CUDART_INF; EL(c, x_ret, 1, 0) = CUDART_INF; EL(c, x_last, 1, 0) = 0.0;
        EL(c, now, 1, 0) = 0.0; EL(c, pending, 1, 0) = pending; EL(c, group, 1, 0) = group; EL(c, n_steps, 1, 0) = 0;
        EL(c, episode, 1, 0) = episode; EL(c, leader, 1, 0) = leader; EL(c, flags, 1, 0) = nflags;
        if (P.next_leader) P.next_leader[be] = leader;
    }
    __syncwarp();
}

// dcm_reset: EPI_WARPS single-warp blocks per tile; block (tile, r) takes the tile's r-th, (r + EPI_WARPS)-th, ... selected env.
// The mode-0 selection and the observation argument below are unreachable (dcm_reset passes mode 1, write_obs = 0); left in place.
template <int TW>
__global__ void __launch_bounds__(32, 16) k_episode(const __grid_constant__ EnvArgs E, const __grid_constant__ EpiArgs P) {
    extern __shared__ __align__(16) unsigned char epi_smem[];
    const unsigned lane = threadIdx.x;
    const unsigned tile = blockIdx.x / EPI_WARPS, r = blockIdx.x % EPI_WARPS;
    const int B = E.S.B, A = E.S.A, T = E.S.T;
    const int b = (int)(tile * 32 + lane);
    bool need = false;
    if (b < B) {
        if (P.mode == 1) need = !P.which || P.which[b];
        else { const TC cb = make_tc(E, b); const unsigned f = EL(cb, flags, 1, 0); need = (f & ENV_DONE) && !(f & ENV_ACCOUNTED); }
    }
    unsigned todo = __ballot_sync(0xffffffffu, need);
    if (!todo) return;
    const EpiScratch scratch = epi_scratch(epi_smem, A, T, E.S.MC);
    for (unsigned k = 0; todo; todo &= todo - 1, ++k) {
        if ((k % EPI_WARPS) != r) continue;
        episode_env<TW>(E, P, (int)(tile * 32 + (__ffs(todo) - 1)), lane, scratch, P.write_obs ? &P.obs : nullptr);
    }
}

// The step path's episode pass: k_step appended the envs whose episode just ended to a list (about 1 env in 150 per pass), so
// the grid is a few blocks per SM instead of EPI_WARPS blocks per tile -- dispatching 8,192 mostly empty blocks cost ~25 us
// beside k_obs (profiles/r03a_timeline.txt).  Envs are independent: the order of the list does not matter.
// Shared-memory footprint matters more than anything else here.  Two k_obs_tile blocks leave a 13 kB hole at the top of an
// SM's shared memory; episode blocks that fit into it run beside them for free, but a block that does not is placed -- it has
// priority -- at the BOTTOM of the 110 kB an exiting k_obs_tile block frees, after which no second k_obs_tile block fits on that SM
// until it is gone (30-50 us; measured with tools/obs_trace.py: most SMs ran ONE obs block, profiles/r04_pass_trace.txt).  Hence:
// member data in registers (1.1 kB of scratch per env), several envs (warps) per block to share the 1 kB the hardware reserves per
// block, and at most ~100 registers.
template <int TW>
__global__ void __launch_bounds__(32 * EPI_LIST_REG_BUDGET_WARPS, 5) k_episode_list(const __grid_constant__ EnvArgs E, const __grid_constant__ EpiArgs P, const unsigned* elist, const unsigned* ecount,
                                                                         unsigned long long* trace) {
    extern __shared__ __align__(16) unsigned char epi_smem[];
    const unsigned n = *ecount, nw = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const unsigned first = blockIdx.x * nw + warp;
    if (first >= n) return;
    auto stamp = [&](int k) { if (trace && lane == 0) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); trace[(size_t)E.S.NT * 8 + 4 * first + k] = t; } };
    if (trace && lane == 0) { unsigned sm; asm volatile("mov.u32 %0, %%smid;" : "=r"(sm)); trace[(size_t)E.S.NT * 8 + 4 * first + 2] = sm; }
    stamp(0);                                                                 // DCM_PASS_TRACE=1 (tools/obs_trace.py): warp entry / exit / SM, after the obs tiles' stamps
    const size_t per_warp = (epi_scratch_bytes(E.S.A, E.S.T, E.S.MC) + 15) / 16 * 16;
    const EpiScratch scratch = epi_scratch(epi_smem + warp * per_warp, E.S.A, E.S.T, E.S.MC);
    for (unsigned k = first; k < n; k += gridDim.x * nw)
        episode_env<TW>(E, P, (int)elist[k], lane, scratch, P.write_obs ? &P.obs : nullptr);
    stamp(1);
}

// ---------------------------------------------------------------------------------------------------------------
// k_obs: observation + mask for the leader of every env (envs without a leader are skipped).  One warp per
// (tile of 32 envs, chunk of rows): lane <-> env produces the chunk's rows -- loads batched five / six rows at a time --
// into a shared-memory tile with an odd pitch (conflict-free), then the warp walks the 32 envs and streams each env's
// 60 contiguous floats (and its mask bytes) out with unit-stride stores.  blockIdx.y = chunk: [0, NA) agent chunks of 10
// rows, [NA, NA + NR) task chunks of 12 rows.  mask (task_env.py:192-200 + worker.py:58-61), agent rows (:165-180),
// task rows (:182-190), cast to fp32 (worker.py:62,64).
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void flush_rows(const float* tile, float* g0, unsigned row_len, int n, unsigned tile_id, unsigned lane, unsigned valid, int B) {
    // env e of the tile: n floats staged at tile[e*OBS_PITCH ..]  ->  g0[e*row_len ..]; g0 already points at (first env of the tile, first column)
    const int ne = B - (int)(tile_id * 32) < 32 ? B - (int)(tile_id * 32) : 32;
    const float* src = tile + lane; float* dst = g0 + lane;
    for (int e = 0; e < ne; ++e, src += OBS_PITCH, dst += row_len) {
        if (!((valid >> e) & 1u)) continue;
        if ((int)lane < n) dst[0] = src[0];
        if ((int)lane + 32 < n) dst[32] = src[32];
    }
}

// one (tile, chunk) unit by one warp; `tile` is the warp's staging area of 32 * OBS_PITCH floats
template <int TW>
__device__ __forceinline__ void obs_unit(const EnvArgs& E, const ObsArgs& O, unsigned tile_id, int chunk, unsigned lane, float* tile, unsigned skip = 0) {
    const int b = (int)(tile_id * 32 + lane);
    const int B = E.S.B, A = E.S.A, T = E.S.T;
    if (tile_id * 32 >= (unsigned)B) return;
    float* mine = tile + lane * OBS_PITCH;
    const TC c = make_tc(E, b < B ? b : B - 1);
    int leader = -1;
    if (b < B) leader = O.leader ? O.leader[b] : EL(c, leader, 1, 0);
    if (O.skip_ended && b < B && EL(c, ended, 1, 0)) leader = -1;
    const bool ok = leader >= 0 && leader < A && !((skip >> lane) & 1u);      // skip: envs whose observation is built by the warp that restarts them
    const unsigned valid = __ballot_sync(0xffffffffu, ok);
    if (!valid) return;
    double Lx = 0, Ly = 0;
    if (ok) { const double2 p = AREC2(c, leader, 0); Lx = p.x; Ly = p.y; }
    const int NA = (A + OBS_AGENTS_PER_CHUNK - 1) / OBS_AGENTS_PER_CHUNK;
    if (chunk < NA) {                                                         // ---- agent rows (:165-180)
        if (!O.agent_obs) return;
        const int c0 = chunk * OBS_AGENTS_PER_CHUNK;
        const int na = A - c0 < OBS_AGENTS_PER_CHUNK ? A - c0 : OBS_AGENTS_PER_CHUNK;
        if (ok) {
            u64 feas[TW];
#pragma unroll
            for (int w = 0; w < TW; ++w) feas[w] = EL(c, m_feas, TW, w);
            const u64 route = EL(c, am_route, 1, 0), depot = EL(c, am_depot, 1, 0), assigned = EL(c, am_assigned, 1, 0), watch = EL(c, am_watch, 1, 0);
            const double now = EL(c, now, 1, 0);
#pragma unroll
            for (int h = 0; h < OBS_AGENTS_PER_CHUNK; h += 5) {               // five agents per batch: 15 + 10 loads in flight
                double2 xy[5], ld[5], ti[5]; double du[5]; unsigned kk[5];
#pragma unroll
                for (int q = 0; q < 5; ++q) { const int i = c0 + (h + q < na ? h + q : 0); xy[q] = AREC2(c, i, 0); ld[q] = AREC2(c, i, 1); kk[q] = ANODE(c, i); }
#pragma unroll
                for (int q = 0; q < 5; ++q) {                                   // one gather per agent that stands at a task, none otherwise
                    const bool at_task = kk[q] != DCM_NODE_DEPOT; const unsigned k = at_task ? kk[q] : 0u; const bool fe = at_task && tbit<TW>(feas, (int)k);
                    ti[q] = fe ? TINFO2(c, k) : make_double2(0.0, 0.0); du[q] = (at_task && !fe) ? EL(c, s_dur, T, k) : 0.0;
                }
#pragma unroll
                for (int q = 0; q < 5; ++q) if (h + q < na) {
                    const int i = c0 + h + q; const u64 bit = 1ull << i;
                    double travel_t = 0.0, wait = 0.0, remain = 0.0;
                    if ((route & bit) && !(depot & bit)) {                    // :168
                        const bool fe = tbit<TW>(feas, (int)kk[q]);
                        const double arr = ld[q].x;
                        const double ts = fe ? ti[q].x : 0.0;                 // time_start is 0 until the task is feasible (Q6)
                        const double tf = fe ? ti[q].y : 0.0 + du[q];         // fl(time_start + time)
                        const double v = arr - now; travel_t = v < 0.0 ? 0.0 : v;                       // :169
                        if (now <= ts) { const double wv = now - arr; wait = wv < 0.0 ? 0.0 : wv; }     // :170
                        if (now >= ts) { const double qv = tf - now; remain = qv < 0.0 ? 0.0 : qv; }    // :171
                    }
                    float* r = mine + 6 * (h + q);                            // :176-177
                    r[0] = __double2float_rn(travel_t); r[1] = __double2float_rn(remain); r[2] = __double2float_rn(wait);
                    r[3] = __double2float_rn(Lx - xy[q].x); r[4] = __double2float_rn(Ly - xy[q].y);
                    r[5] = ((assigned & bit) || ((watch & bit) && now >= ti[q].x)) ? 1.0f : 0.0f;       // lazy `assigned` (t_agent_update)
                }
            }
        }
        __syncwarp();
        flush_rows(tile, O.agent_obs + (size_t)tile_id * 32 * 6 * A + 6 * c0, 6 * A, 6 * na, tile_id, lane, valid, B);
        return;
    }
    // ---- task rows (:182-190; row 0 = depot) + mask bytes
    const int r0 = (chunk - NA) * OBS_ROWS_PER_CHUNK;
    const int nr = T + 1 - r0 < OBS_ROWS_PER_CHUNK ? T + 1 - r0 : OBS_ROWS_PER_CHUNK;
    if (ok) {
        u64 open[TW]; bool any_open = false;
#pragma unroll
        for (int w = 0; w < TW; ++w) { open[w] = EL(c, m_open, TW, w); any_open = any_open || open[w] != 0; }
        unsigned mlo = 0, mhi = 0, mtop = 0;                                  // mask bytes of the chunk, packed (1 = forbidden)
#pragma unroll
        for (int h = 0; h < OBS_ROWS_PER_CHUNK; h += 6) {                     // six rows per batch: 30 loads in flight
            double tx[6], ty[6], du[6]; int st[6], rq[6];
#pragma unroll
            for (int q = 0; q < 6; ++q) {
                const int jj = r0 + (h + q < nr ? h + q : 0); const int j = jj > 0 ? jj - 1 : 0;
                tx[q] = EL(c, s_tx, T, j); ty[q] = EL(c, s_ty, T, j); du[q] = EL(c, s_dur, T, j); st[q] = EL(c, t_status, T, j); rq[q] = EL(c, s_req, T, j);
            }
            if (r0 == 0 && h == 0) { tx[0] = EL(c, s_dep, 2, 0); ty[0] = EL(c, s_dep, 2, 1); }
#pragma unroll
            for (int q = 0; q < 6; ++q) if (h + q < nr) {
                const int jj = r0 + h + q;
                float* r = mine + 5 * (h + q);
                if (O.task_obs) {
                    if (jj == 0) { r[0] = 0.f; r[1] = 0.f; r[2] = 0.f; }      // :188 depot row
                    else { r[0] = (float)st[q]; r[1] = (float)rq[q]; r[2] = __double2float_rn(du[q]); }   // :185
                    r[3] = __double2float_rn(tx[q] - Lx); r[4] = __double2float_rn(ty[q] - Ly);           // :186
                }
                // :199 task bit: forbidden unless open;  worker.py:58-61 depot bit: allowed only when nothing is open
                const unsigned forbidden = jj == 0 ? (any_open ? 1u : 0u) : (tbit<TW>(open, jj - 1) ? 0u : 1u);
                const int sl = h + q;
                if (sl < 4) mlo |= forbidden << (8 * sl); else if (sl < 8) mhi |= forbidden << (8 * (sl - 4)); else mtop |= forbidden << (8 * (sl - 8));
            }
        }
        unsigned* mw = (unsigned*)(mine + 60);
        mw[0] = mlo; mw[1] = mhi; mw[2] = mtop;
    }
    __syncwarp();
    if (O.task_obs) flush_rows(tile, O.task_obs + (size_t)tile_id * 32 * 5 * (T + 1) + 5 * r0, 5 * (T + 1), 5 * nr, tile_id, lane, valid, B);
    if (O.mask) {
        const int ne = B - (int)(tile_id * 32) < 32 ? B - (int)(tile_id * 32) : 32;
        const unsigned char* src = (const unsigned char*)(tile + 60) + lane; unsigned char* dst = O.mask + (size_t)tile_id * 32 * (T + 1) + r0 + lane;
        for (int e = 0; e < ne; ++e, src += 4 * OBS_PITCH, dst += T + 1) if (((valid >> e) & 1u) && (int)lane < nr) dst[0] = src[0];
    }
}

template <int TW>
__global__ void __launch_bounds__(OBS_THREADS) k_obs(const __grid_constant__ EnvArgs E, const __grid_constant__ ObsArgs O) {
    __shared__ float smem[(OBS_THREADS / 32) * 32 * OBS_PITCH];
    const unsigned warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    obs_unit<TW>(E, O, blockIdx.x * (OBS_THREADS / 32) + warp, (int)blockIdx.y, lane, smem + warp * 32 * OBS_PITCH);
}

// ---------------------------------------------------------------------------------------------------------------
// k_obs_tile: the observation builder of the step path.  ONE BLOCK PER TILE of 32 envs, two blocks per SM, and the TMA
// engine moves the bytes in both directions:
//   in   one thread issues cp.async.bulk global -> shared for the tile's rows of s_tx, s_ty, t_status, s_req, the agent
//        records and the observation cache a_obs (each is one contiguous span of the tile-major arena) against an mbarrier;
//        nothing is held in registers while they fly.  Meanwhile every warp loads the per-env scalars of its role (leader,
//        masks, clock; the fp32 durations of its rows).  No load depends on another: the block waits ONE round trip.
//        (The cache a_obs is what makes that possible: the agent rows need time_start / time_finish of the task an agent
//        stands at, a gather that depends on the node ids; the step keeps its result per agent instead.)
//   rows warp <-> row chunk, lane <-> env, operands from shared memory, rows written in place into the staged output:
//        agent rows [32][6A], task rows [32][5(T+1)] floats and mask [32][T+1] bytes are exactly the three contiguous
//        spans of the policy tensors that belong to the tile.
//   out  one thread hands each span to cp.async.bulk shared -> global: no flush loop and no store instructions.
// A tile with an env that is left out (its episode ended: k_episode_list writes its observation meanwhile; no leader; past
// B) or a destination that is not 16-byte aligned is copied warp by warp, env by env, instead.  Shapes whose tile does not
// fit twice in an SM's shared memory use k_obs.
// ---------------------------------------------------------------------------------------------------------------
#define OBS_TILE_MAX_WARPS 8
struct ObsTileSmem { unsigned oA, oT, oM, iX, iY, iR, iO, iS, iQ, bar, total; };
__host__ __device__ inline ObsTileSmem obs_tile_smem(int A, int T) {
    ObsTileSmem L; unsigned o = 0;
    auto take = [&](unsigned bytes) { const unsigned at = o; o += (bytes + 15u) & ~15u; return at; };
    L.oA = take(32u * 6 * A * 4); L.oT = take(32u * 5 * (T + 1) * 4); L.oM = take(32u * (T + 1));
    L.iX = take(256u * T); L.iY = take(256u * T); L.iR = take(1024u * A); L.iO = take(512u * A); L.iS = take(32u * T); L.iQ = take(32u * T);
    L.bar = take(8); L.total = o;
    return L;
}

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void bulk_store(void* gdst, const void* ssrc, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" :: "l"(gdst), "r"(smem_u32(ssrc)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_load(void* sdst, const void* gsrc, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_u32(sdst)), "l"(gsrc), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
    unsigned done;
    do {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }" : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    } while (!done);
}

template <int TW>
__global__ void __launch_bounds__(32 * OBS_TILE_MAX_WARPS, 3) k_obs_tile(const __grid_constant__ EnvArgs E, const __grid_constant__ ObsArgs O, int use_bulk, unsigned long long* trace) {
    extern __shared__ __align__(128) unsigned char obs_smem[];
    const int B = E.S.B, A = E.S.A, T = E.S.T;
    const unsigned NT = (unsigned)E.S.NT, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    const ObsTileSmem L = obs_tile_smem(A, T);
    float* sA = (float*)(obs_smem + L.oA); float* sT = (float*)(obs_smem + L.oT); unsigned char* sM = obs_smem + L.oM;
    const double* iX = (const double*)(obs_smem + L.iX); const double* iY = (const double*)(obs_smem + L.iY);
    const double2* iR = (const double2*)(obs_smem + L.iR); const double2* iO = (const double2*)(obs_smem + L.iO);
    const signed char* iS = (const signed char*)(obs_smem + L.iS); const unsigned char* iQ = obs_smem + L.iQ;
    const unsigned bar = smem_u32(obs_smem + L.bar);
    const int NA = (A + OBS_AGENTS_PER_CHUNK - 1) / OBS_AGENTS_PER_CHUNK, NR = (T + 1 + OBS_ROWS_PER_CHUNK - 1) / OBS_ROWS_PER_CHUNK;
    const unsigned nA = 6u * A, nT = 5u * (T + 1), nM = (unsigned)(T + 1);
    auto clock_ns = [&]() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; };
    auto issue_loads = [&](unsigned tile) {                                   // thread 0: the tile's rows, one contiguous span per array
        const TC c0 = make_tc(E, (int)(tile * 32));                           // lane 0 of the tile
        const unsigned bytes = 256u * T * 2 + 1024u * A + 512u * A + 32u * T * 2;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
        bulk_load(obs_smem + L.iR, &AREC2(c0, 0, 0), 1024u * A, bar);
        bulk_load(obs_smem + L.iO, &AOBS2(c0, 0), 512u * A, bar);
        bulk_load(obs_smem + L.iX, &EL(c0, s_tx, T, 0), 256u * T, bar);
        bulk_load(obs_smem + L.iY, &EL(c0, s_ty, T, 0), 256u * T, bar);
        bulk_load(obs_smem + L.iS, &EL(c0, t_status, T, 0), 32u * T, bar);
        bulk_load(obs_smem + L.iQ, &EL(c0, s_req, T, 0), 32u * T, bar);
    };
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    asm volatile("griddepcontrol.wait;" ::: "memory");                        // the step kernel's writes are complete and visible (no-op without a programmatic launch)
    if (threadIdx.x == 0 && blockIdx.x < NT) issue_loads(blockIdx.x);
    // The block walks tiles blockIdx.x, + gridDim.x, ...; the grid is one block per tile, so it makes a single trip: the in-loop
    // wait for the previous tile's drain and the next-tile prefetch never run (they served two persistent blocks per SM, measured
    // slower and removed: DESIGN.md section 4).  The loop form stays because this kernel's register allocation is fragile (72-94
    // across builds and variants) and the loop form was adopted in part for its allocation; collapsing it wants a measurement of its own.
    unsigned parity = 0; bool draining = false; unsigned prev_tile = 0;
    for (unsigned tile_id = blockIdx.x; tile_id < NT; tile_id += gridDim.x) {
        const int b = (int)(tile_id * 32 + lane);
        const TC c = make_tc(E, b < B ? b : B - 1);
        auto stamp = [&](int k) { if (trace && threadIdx.x == 0) trace[(size_t)tile_id * 8 + k] = clock_ns(); };
        stamp(0);
        if (trace && threadIdx.x == 0) { unsigned sm; asm volatile("mov.u32 %0, %%smid;" : "=r"(sm)); trace[(size_t)tile_id * 8 + 5] = sm; }
        // per-env scalars of the warp's first chunk, all issued at once and before the leader is known
        int leader = -1; unsigned ended = 0;
        if (b < B) { leader = O.leader ? O.leader[b] : EL(c, leader, 1, 0); if (O.skip_ended) ended = EL(c, ended, 1, 0); }
        u64 open[TW]; u64 route = 0, depot = 0, assigned = 0, watch = 0; double now = 0.0, dpx = 0.0, dpy = 0.0; float dq[OBS_ROWS_PER_CHUNK];
        auto agent_scalars = [&]() { route = EL(c, am_route, 1, 0); depot = EL(c, am_depot, 1, 0); assigned = EL(c, am_assigned, 1, 0); watch = EL(c, am_watch, 1, 0); now = EL(c, now, 1, 0); };
        auto task_scalars = [&](int chunk) {
            const int r0 = (chunk - NA) * OBS_ROWS_PER_CHUNK;
#pragma unroll
            for (int w = 0; w < TW; ++w) open[w] = EL(c, m_open, TW, w);
            if (r0 == 0 || O.skip_ended == 2) { dpx = EL(c, s_dep, 2, 0); dpy = EL(c, s_dep, 2, 1); }
#pragma unroll
            for (int q = 0; q < OBS_ROWS_PER_CHUNK; ++q) { const int jj = r0 + q; dq[q] = EL(c, s_dur32, T, (jj > 0 && jj <= T) ? jj - 1 : 0); }
        };
        if ((int)warp < NA) agent_scalars(); else if ((int)warp < NA + NR) task_scalars((int)warp);
        const bool fresh = ended && O.skip_ended == 2;                        // the restarted episode's first observation (see ObsArgs)
        if (ended) leader = fresh ? 0 : -1;
        const bool ok = leader >= 0 && leader < A;
        const unsigned valid = __ballot_sync(0xffffffffu, ok);                // the same in every warp of the block
        stamp(1);
        mbar_wait(bar, parity); parity ^= 1u;                                 // (also: never leave with copies in flight into this block's shared memory)
        stamp(4);
        if (draining) {                                                       // the previous tile's staged rows must have been read before they are overwritten
            if (threadIdx.x == 0) { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); if (trace) trace[(size_t)prev_tile * 8 + 3] = clock_ns(); }
            __syncthreads();
            draining = false;
        }
        if (valid) for (int chunk = (int)warp; chunk < NA + NR; chunk += (int)nwarps) {
            if (chunk < NA) {                                                 // ---- agent rows (:165-180)
                if (!O.agent_obs) continue;
                if (chunk != (int)warp) agent_scalars();
                if (!ok) continue;
                const int c0 = chunk * OBS_AGENTS_PER_CHUNK;
                const int na = A - c0 < OBS_AGENTS_PER_CHUNK ? A - c0 : OBS_AGENTS_PER_CHUNK;
                const double2 Lp = iR[(((unsigned)leader << 5) + lane) << 1];
                float* mine = sA + lane * 6 * A + 6 * c0;
#pragma unroll 5
                for (int q = 0; q < na; ++q) {
                    const int i = c0 + q; const u64 bit = 1ull << i; const unsigned at = ((unsigned)i << 5) + lane;
                    double travel_t = 0.0, wait = 0.0, remain = 0.0;
                    if (fresh) { float2* r = (float2*)(mine + 6 * q); r[0] = r[1] = r[2] = make_float2(0.f, 0.f); continue; }
                    const double2 xy = iR[at << 1];
                    const double2 tt = iO[at];                                // {time_start or 0 (Q6), fl(time_start + time)}
                    if ((route & bit) && !(depot & bit)) {                    // :168
                        const double arr = iR[(at << 1) + 1].x;
                        const double v = arr - now; travel_t = v < 0.0 ? 0.0 : v;                         // :169
                        if (now <= tt.x) { const double wv = now - arr; wait = wv < 0.0 ? 0.0 : wv; }     // :170
                        if (now >= tt.x) { const double qv = tt.y - now; remain = qv < 0.0 ? 0.0 : qv; }  // :171
                    }
                    float2* r = (float2*)(mine + 6 * q);                      // :176-177 (8-byte aligned: even offsets)
                    r[0] = make_float2(__double2float_rn(travel_t), __double2float_rn(remain));
                    r[1] = make_float2(__double2float_rn(wait), __double2float_rn(Lp.x - xy.x));
                    r[2] = make_float2(__double2float_rn(Lp.y - xy.y), ((assigned & bit) || ((watch & bit) && now >= tt.x)) ? 1.0f : 0.0f);   // lazy `assigned` (t_agent_update)
                }
                continue;
            }
            // ---- task rows (:182-190; row 0 = depot) + mask bytes
            if (chunk != (int)warp) task_scalars(chunk);
            if (!ok) continue;
            const int r0 = (chunk - NA) * OBS_ROWS_PER_CHUNK;
            const int nr = T + 1 - r0 < OBS_ROWS_PER_CHUNK ? T + 1 - r0 : OBS_ROWS_PER_CHUNK;
            bool any_open = false;
#pragma unroll
            for (int w = 0; w < TW; ++w) any_open = any_open || open[w] != 0;
            double2 Lp = iR[(((unsigned)leader << 5) + lane) << 1];
            if (fresh) { Lp = make_double2(dpx, dpy); any_open = true; }       // everybody stands at the depot, every task is open
            float* mine = sT + lane * 5 * (T + 1) + 5 * r0;
            unsigned char* mm = sM + lane * (T + 1) + r0;
#pragma unroll
            for (int q = 0; q < OBS_ROWS_PER_CHUNK; ++q) if (q < nr) {
                const int jj = r0 + q; const unsigned at = ((unsigned)(jj > 0 ? jj - 1 : 0) << 5) + lane;
                float* r = mine + 5 * q;
                if (O.task_obs) {
                    if (jj == 0) { r[0] = 0.f; r[1] = 0.f; r[2] = 0.f; r[3] = __double2float_rn(dpx - Lp.x); r[4] = __double2float_rn(dpy - Lp.y); }   // :188 depot row
                    else {
                        r[0] = (float)(int)(fresh ? (int)iQ[at] : (int)iS[at]); r[1] = (float)(int)iQ[at]; r[2] = dq[q];   // :185 (s_dur32 = fp32(time)); status = requirements after clear_decisions
                        r[3] = __double2float_rn(iX[at] - Lp.x); r[4] = __double2float_rn(iY[at] - Lp.y);             // :186
                    }
                }
                // :199 task bit: forbidden unless open;  worker.py:58-61 depot bit: allowed only when nothing is open
                mm[q] = jj == 0 ? (any_open ? 1 : 0) : ((fresh || tbit<TW>(open, jj - 1)) ? 0 : 1);
            }
        }
        const int ne = B - (int)(tile_id * 32) < 32 ? B - (int)(tile_id * 32) : 32;
        const bool whole = use_bulk && ne == 32 && valid == 0xffffffffu;
        if (whole) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the staged rows must be visible to the TMA engine
        __syncthreads();                                                      // rows staged; nobody reads the staged inputs any more
        stamp(2);
        const unsigned next = tile_id + gridDim.x;
        if (threadIdx.x == 0 && next < NT) issue_loads(next);
        if (!valid) continue;
        if (whole) {
            if (threadIdx.x == 0) {
                if (O.agent_obs) bulk_store(O.agent_obs + (size_t)tile_id * 32 * nA, sA, 32 * nA * 4);
                if (O.task_obs) bulk_store(O.task_obs + (size_t)tile_id * 32 * nT, sT, 32 * nT * 4);
                if (O.mask) bulk_store(O.mask + (size_t)tile_id * 32 * nM, sM, 32 * nM);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
            draining = true; prev_tile = tile_id;
            continue;
        }
        for (int e = (int)warp; e < ne; e += (int)nwarps) {                   // warp <-> env, unit-stride stores; the copies of one env are independent
            if (!((valid >> e) & 1u)) continue;
            const size_t be = (size_t)tile_id * 32 + e;
            if (O.task_obs) {
                const float* src = sT + e * nT; float* dst = O.task_obs + be * nT;
#pragma unroll 8
                for (unsigned k = lane; k < nT; k += 32) dst[k] = src[k];
            }
            if (O.agent_obs) {
                const float* src = sA + e * nA; float* dst = O.agent_obs + be * nA;
#pragma unroll 4
                for (unsigned k = lane; k < nA; k += 32) dst[k] = src[k];
            }
            if (O.mask) for (unsigned k = lane; k < nM; k += 32) O.mask[be * nM + k] = sM[e * nM + k];
        }
        __syncthreads();                                                      // the staged rows are free again
        if (trace && threadIdx.x == 0) trace[(size_t)tile_id * 8 + 3] = clock_ns() | (1ull << 63);
    }
    if (draining && threadIdx.x == 0) {                                       // shared memory is released when the block exits
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        if (trace) trace[(size_t)prev_tile * 8 + 3] = clock_ns();
    }
}

// ---------------------------------------------------------------------------------------------------------------
// k_granular: one TaskEnv method per launch
// ---------------------------------------------------------------------------------------------------------------
template <int TW>
__global__ void __launch_bounds__(STEP_THREADS) k_granular(const __grid_constant__ EnvArgs E, const __grid_constant__ GranArgs G) {
    __shared__ double tmp_smem[SCR_TMP * STEP_THREADS];
    const int b = blockIdx.x * STEP_THREADS + threadIdx.x;
    if (b >= E.S.B) return;
    TC c = make_tc(E, b); c.tmp = tmp_smem + threadIdx.x;
    const double now = EL(c, now, 1, 0);
    St<TW> st, st0; ld_state(c, st); st0 = st;
    switch (G.op) {
    case OP_NEXT_DECISION: { double t; const u64 d = t_next_decision(c, t); G.deciders[b] = d; G.t[b] = t; } break;
    case OP_UNIQUE_GROUP: {
        signed char* out = G.group_rank + (size_t)b * c.A;
        for (int i = 0; i < c.A; ++i) out[i] = -1;
        u64 rest = G.deciders_in[b]; int rank = 0;
        while (rest) {
            const u64 g = t_current_group(c, rest);
            for (u64 m = g; m; m &= m - 1) out[__ffsll((long long)m) - 1] = (signed char)rank;
            rest &= ~g; ++rank;
        }
    } break;
    case OP_SET_CLOCK: EL(c, now, 1, 0) = G.t_in[b]; break;
    case OP_GET_CLOCK: G.t[b] = now; break;
    case OP_TASK_UPDATE: {
        unsigned char* nw = G.newly ? G.newly + (size_t)b * c.T : nullptr;
        if (nw) for (int j = 0; j < c.T; ++j) nw[j] = 0;
        t_task_update(c, st, now, nw);
    } break;
    case OP_AGENT_UPDATE: t_agent_update(c, st, now, st.route); break;   // full reference loop (max_waiting_time may have changed)
    case OP_APPLY_MEMBERS: {
        const int n = G.n_members[b]; const int action = G.action[b];
        if (n <= 0) break;
        unsigned flags = EL(c, flags, 1, 0);
        if (action < 0 || action > c.T || n > c.A) flags |= ENV_ERR_ACTION;
        else {
            double tx, ty; node_xy(c, action == 0 ? DCM_NODE_DEPOT : (unsigned)(action - 1), tx, ty);
            double reward = 0.0;
            for (int k = 0; k < n; ++k) {
                const int i = G.members[(size_t)b * G.mstride + k];
                if (i < 0 || i >= c.A) { flags |= ENV_ERR_ACTION; continue; }
                double d, tt; travel(c, AREC(c, i, AR_X), AREC(c, i, AR_Y), tx, ty, d, tt);
                t_agent_step(c, st, now, i, action, tx, ty, d, tt, flags);
                reward += -tt;                                                // task_env.py:337-339
            }
            if (G.reward) G.reward[b] = reward / (double)n;                   // :341
        }
        EL(c, flags, 1, 0) = flags;
    } break;
    case OP_CHECK_FINISHED: {
        double t; const u64 d = t_next_decision(c, t);
        bool fin = false;
        if (d == 0) { fin = t_all_returned_and_finished(c, st); EL(c, now, 1, 0) = t; }
        G.finished[b] = fin ? 1 : 0;
    } break;
    case OP_COMPUTE_METRICS: {
        const double t = t_episode_metrics(c, st, now, EL(c, n_steps, 1, 0), G.metrics + (size_t)b * 8,
                                           G.task_wait ? G.task_wait + (size_t)b * c.T : nullptr,
                                           G.agent_wait ? G.agent_wait + (size_t)b * c.A : nullptr);
        EL(c, now, 1, 0) = t;
    } break;
    case OP_ENV_FLAGS: G.flags_out[b] = EL(c, flags, 1, 0); break;
    }
    st_state(c, st0, st);
}

// ---------------------------------------------------------------------------------------------------------------
// k_routes: pre_set_route + execute_by_route (task_env.py:562-599), one whole episode per thread
// ---------------------------------------------------------------------------------------------------------------
template <int TW>
__global__ void __launch_bounds__(STEP_THREADS) k_routes(const __grid_constant__ EnvArgs E, const int* routes, int rstride, const int* route_len,
                                                         unsigned char* cursor /*[B,A] scratch*/, double* makespan) {
    __shared__ double tmp_smem[SCR_TMP * STEP_THREADS];
    const int b = blockIdx.x * STEP_THREADS + threadIdx.x;
    if (b >= E.S.B) return;
    TC c{E.S, (unsigned)b >> 5, (unsigned)b & 31u, (size_t)((unsigned)b >> 5) * E.S.tile_stride, E.S.A, E.S.T, E.S.MC, 100.0 /* :564 */, E.vel, E.max_time};
    c.tmp = tmp_smem + threadIdx.x;
    double now = EL(c, now, 1, 0); unsigned flags = EL(c, flags, 1, 0); unsigned n_steps = EL(c, n_steps, 1, 0);
    unsigned char* pos = cursor + (size_t)b * c.A;
    for (int i = 0; i < c.A; ++i) pos[i] = 0;
    St<TW> st, st0; ld_state(c, st); st0 = st;
    bool finished = flags & ENV_FINISHED;
    int guard = 0;
    while (!finished && now < 200.0 && guard < 100000) {                      // :565
        double t; const u64 dec = t_next_decision(c, t);                      // :568
        now = t;                                                              // :569
        t_task_update(c, st, now, nullptr); t_agent_update(c, st, now, st.route);   // :570-571
        for (u64 d = dec; d; d &= d - 1) {                                    // :572 ascending ids
            const int a = __ffsll((long long)d) - 1;
            const int p = pos[a], len = route_len[(size_t)b * c.A + a];
            int act = 0;                                                      // :573-574 empty / exhausted route -> depot
            if (p < len) { act = routes[((size_t)b * c.A + a) * rstride + p]; pos[a] = (unsigned char)(p + 1); }
            if (act < 0 || act > c.T) { flags |= ENV_ERR_ACTION; act = 0; }
            double tx, ty; node_xy(c, act == 0 ? DCM_NODE_DEPOT : (unsigned)(act - 1), tx, ty);
            double dd, tt; travel(c, AREC(c, a, AR_X), AREC(c, a, AR_Y), tx, ty, dd, tt);
            t_agent_step(c, st, now, a, act, tx, ty, dd, tt, flags);          // :585 agent_step
            t_task_update(c, st, now, nullptr); t_agent_update(c, st, now, st.route);   // :586-587
            ++n_steps;
        }
        double t2; const u64 d2 = t_next_decision(c, t2);                     // :588 check_finished
        if (d2 == 0) { now = t2; finished = t_all_returned_and_finished(c, st); }
        ++guard;
    }
    if (finished) flags |= ENV_FINISHED;
    flags |= ENV_DONE | ENV_ACCOUNTED;          // metrics are fetched explicitly with dcm_compute_metrics (baselines/CTAS-D.py:80-94)
    EL(c, now, 1, 0) = now; EL(c, flags, 1, 0) = flags; EL(c, n_steps, 1, 0) = n_steps; EL(c, leader, 1, 0) = -1;
    EL(c, pending, 1, 0) = 0; EL(c, group, 1, 0) = 0;
    st_state(c, st0, st);
    if (makespan) makespan[b] = now;
}

// ---------------------------------------------------------------------------------------------------------------
// instance / plumbing kernels (thread per env)
// ---------------------------------------------------------------------------------------------------------------
__global__ void k_generate(const __grid_constant__ EnvArgs E, int bump_instance) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= E.S.B) return;
    const TC c = make_tc(E, b);
    const unsigned inst = EL(c, instance, 1, 0) + (bump_instance ? 1u : 0u);
    t_generate(c, E.seed, E.first_gid + (u64)b, inst, E.gen_max_duration, E.gen_random_duration);
    EL(c, instance, 1, 0) = inst;
}

__global__ void k_pack_static(const __grid_constant__ EnvArgs E, const double* task_xy, const double* depot_xy, const int* req, const double* dur) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= E.S.B) return;
    const TC c = make_tc(E, b);
    for (int j = 0; j < c.T; ++j) {
        int r = req[(size_t)b * c.T + j]; r = r < 1 ? 1 : (r > c.s.M ? c.s.M : r);
        put_static(c, j, task_xy[((size_t)b * c.T + j) * 2], task_xy[((size_t)b * c.T + j) * 2 + 1], (unsigned)r, dur[(size_t)b * c.T + j]);
    }
    EL(c, s_dep, 2, 0) = depot_xy[2 * (size_t)b]; EL(c, s_dep, 2, 1) = depot_xy[2 * (size_t)b + 1];
}

__global__ void k_unpack_static(const __grid_constant__ EnvArgs E, double* task_xy, double* depot_xy, int* req, double* dur) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= E.S.B) return;
    const TC c = make_tc(E, b);
    for (int j = 0; j < c.T; ++j) {
        if (task_xy) { task_xy[((size_t)b * c.T + j) * 2] = EL(c, s_tx, c.T, j); task_xy[((size_t)b * c.T + j) * 2 + 1] = EL(c, s_ty, c.T, j); }
        if (dur) dur[(size_t)b * c.T + j] = EL(c, s_dur, c.T, j);
        if (req) req[(size_t)b * c.T + j] = EL(c, s_req, c.T, j);
    }
    if (depot_xy) { depot_xy[2 * (size_t)b] = EL(c, s_dep, 2, 0); depot_xy[2 * (size_t)b + 1] = EL(c, s_dep, 2, 1); }
}

__global__ void k_init(const __grid_constant__ EnvArgs E) {                   // every env is "done" until dcm_reset
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= E.S.NT * 32) return;
    const TC c = make_tc(E, b);
    EL(c, flags, 1, 0) = ENV_DONE | ENV_ACCOUNTED; EL(c, leader, 1, 0) = -1;
    EL(c, x_fin, 1, 0) = CUDART_INF; EL(c, x_amin, 1, 0) = CUDART_INF; EL(c, x_ret, 1, 0) = CUDART_INF;
}

// tiled SoA <-> per-env record of dcm_layout.h (export / import / checkpoint format)
template <int TW>
__global__ void k_export(const __grid_constant__ EnvArgs E, const DcmLayout L, unsigned char* dst) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= E.S.B) return;
    const TC c = make_tc(E, b);
    St<TW> st; ld_state(c, st);
    unsigned char* r = dst + (size_t)b * L.dyn_bytes;
    const int T = c.T, A = c.A, Tp = L.Tp;
    const double h_now = EL(c, now, 1, 0);
    for (int j = 0; j < T; ++j) {
        const bool fe = tbit<TW>(st.feas, j); const int n = tbit<TW>(st.ne, j) ? (int)TNMEM(c, j) : 0;
        for (int s = 0; s < n; ++s) { ((double*)(r + L.o_arr))[s * Tp + j] = SARR(c, j, s); (r + L.o_mem)[s * Tp + j] = SMEM(c, j, s); }
        ((double*)(r + L.o_tstart))[j] = fe ? TINFO(c, j, 0) : 0.0; ((unsigned short*)(r + L.o_tnab))[j] = TNAB(c, j);
        (r + L.o_nmem)[j] = (unsigned char)n; ((signed char*)(r + L.o_status))[j] = TSTAT(c, j);
        (r + L.o_tflags)[j] = (unsigned char)((fe ? DCM_TF_FEAS : 0u) | (tbit<TW>(st.fin, j) ? DCM_TF_FIN : 0u) | (tbit<TW>(st.dirty, j) ? DCM_TF_STALE : 0u));
    }
    for (int i = 0; i < A; ++i) {
        ((double*)(r + L.o_alast))[i] = AREC(c, i, AR_LAST); ((double*)(r + L.o_and))[i] = EL(c, a_nd, A, i); ((double*)(r + L.o_adist))[i] = AREC(c, i, AR_DIST);
        ((unsigned short*)(r + L.o_anab))[i] = EL(c, a_nab, A, i); (r + L.o_anode)[i] = ANODE(c, i);
        const u64 bit = 1ull << i;
        const bool started = (st.watch & bit) && h_now >= EL(c, a_ts, A, i);      // lazy `assigned` (t_agent_update): settled here, as every reader does
        (r + L.o_aflags)[i] = (unsigned char)(((st.route & bit) ? DCM_AF_ROUTE : 0u) | (((st.assigned & bit) || started) ? DCM_AF_ASSIGNED : 0u) | ((st.returned & bit) ? DCM_AF_RETURNED : 0u) |
                                              ((st.member & bit) ? DCM_AF_MEMBER : 0u) | ((st.touched & bit) ? DCM_AF_TOUCHED : 0u) | (((st.watch & bit) && !started) ? DCM_AF_WATCH : 0u));
    }
    DcmHdr h;
    h.now = EL(c, now, 1, 0); h.pending = EL(c, pending, 1, 0); h.group = EL(c, group, 1, 0); h.n_steps = EL(c, n_steps, 1, 0);
    h.episode = EL(c, episode, 1, 0); h.leader = EL(c, leader, 1, 0); h.flags = EL(c, flags, 1, 0); h.instance = EL(c, instance, 1, 0);
    h.total_steps = EL(c, total, 1, 0);
    *(DcmHdr*)(r + L.o_hdr) = h;
}

template <int TW>
__global__ void k_import(const __grid_constant__ EnvArgs E, const DcmLayout L, const unsigned char* src) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= E.S.B) return;
    const TC c = make_tc(E, b);
    St<TW> st, st0; ld_state(c, st0);
#pragma unroll
    for (int w = 0; w < TW; ++w) { st.feas[w] = st.fin[w] = st.ne[w] = st.open[w] = st.dirty[w] = 0; }
    st.route = st.assigned = st.returned = st.member = st.depot = st.touched = st.watch = 0;
    st.xfin = st.xamin = st.xret = CUDART_INF; st.xlast = 0.0;
    const unsigned char* r = src + (size_t)b * L.dyn_bytes;
    const int T = c.T, A = c.A, Tp = L.Tp;
    for (int j = 0; j < T; ++j) {
        const int n = (r + L.o_nmem)[j]; const int stt = ((const signed char*)(r + L.o_status))[j]; const unsigned tf = (r + L.o_tflags)[j];
        double amin = CUDART_INF, amax = -CUDART_INF;
        for (int s = 0; s < n && s < c.MC; ++s) {
            const double a = ((const double*)(r + L.o_arr))[s * Tp + j];
            SARR(c, j, s) = a; SMEM(c, j, s) = (r + L.o_mem)[s * Tp + j]; amin = a < amin ? a : amin; amax = a > amax ? a : amax;
        }
        const double ts = ((const double*)(r + L.o_tstart))[j];
        if (tf & DCM_TF_FEAS) {
            const double tfin = ts + TDUR(c, j); TINFO(c, j, 0) = ts; TINFO(c, j, 1) = tfin;
            if (!(tf & DCM_TF_FIN) && tfin < st.xfin) st.xfin = tfin;
        } else { TINFO2(c, j) = make_double2(amin, amax); if (n > 0 && amin < st.xamin) st.xamin = amin; }
        TNAB(c, j) = ((const unsigned short*)(r + L.o_tnab))[j];
        TNMEM(c, j) = (unsigned char)n; SET_STATUS(c, j, stt);
        tset<TW>(st.feas, j, tf & DCM_TF_FEAS); tset<TW>(st.fin, j, tf & DCM_TF_FIN); tset<TW>(st.dirty, j, tf & DCM_TF_STALE);
        tset<TW>(st.ne, j, n > 0); tset<TW>(st.open, j, !(tf & DCM_TF_FEAS) && stt > 0);
    }
    for (int i = 0; i < A; ++i) {
        const unsigned node = (r + L.o_anode)[i]; const unsigned af = (r + L.o_aflags)[i]; const u64 bit = 1ull << i;
        double x, y; node_xy(c, node, x, y);
        AREC2(c, i, 0) = make_double2(x, y); AREC2(c, i, 1) = make_double2(((const double*)(r + L.o_alast))[i], ((const double*)(r + L.o_adist))[i]);
        EL(c, a_nd, A, i) = ((const double*)(r + L.o_and))[i];
        EL(c, a_nab, A, i) = ((const unsigned short*)(r + L.o_anab))[i]; ANODE(c, i) = (unsigned char)node;
        if (node != DCM_NODE_DEPOT) {                                         // observation cache (AOBS2)
            const double du = EL(c, s_dur, T, node), ts = ((const double*)(r + L.o_tstart))[node];
            AOBS2(c, i) = ((r + L.o_tflags)[node] & DCM_TF_FEAS) ? make_double2(ts, ts + du) : make_double2(0.0, 0.0 + du);
        }
        if (af & DCM_AF_ROUTE) st.route |= bit;
        if (af & DCM_AF_ASSIGNED) st.assigned |= bit;
        if (af & DCM_AF_RETURNED) st.returned |= bit;
        if (af & DCM_AF_MEMBER) st.member |= bit;
        if (af & DCM_AF_TOUCHED) st.touched |= bit;
        if ((af & DCM_AF_WATCH) && node != DCM_NODE_DEPOT) { const double ts = ((const double*)(r + L.o_tstart))[node]; st.watch |= bit; EL(c, a_ts, A, i) = ts; }
        if ((af & DCM_AF_ROUTE) && node == DCM_NODE_DEPOT) { st.depot |= bit; if (!(af & DCM_AF_RETURNED)) { const double la = ((const double*)(r + L.o_alast))[i]; if (la < st.xret) st.xret = la; } }
        { const double la = ((const double*)(r + L.o_alast))[i]; if (la > st.xlast) st.xlast = la; }
    }
    st_state(c, st0, st);
    const DcmHdr h = *(const DcmHdr*)(r + L.o_hdr);
    EL(c, now, 1, 0) = h.now; EL(c, pending, 1, 0) = h.pending; EL(c, group, 1, 0) = h.group; EL(c, n_steps, 1, 0) = h.n_steps;
    EL(c, episode, 1, 0) = h.episode; EL(c, leader, 1, 0) = h.leader; EL(c, flags, 1, 0) = h.flags; EL(c, instance, 1, 0) = h.instance;
    EL(c, total, 1, 0) = h.total_steps;
}

__global__ void k_sum_episodes(const __grid_constant__ EnvArgs E, unsigned long long* out) {
    unsigned long long acc = 0;
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < E.S.B; b += gridDim.x * blockDim.x) { const TC c = make_tc(E, b); acc += EL(c, episode, 1, 0); }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, acc);
}

__global__ void k_sum_steps(const __grid_constant__ EnvArgs E, unsigned long long* out) {
    unsigned long long acc = 0;
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < E.S.B; b += gridDim.x * blockDim.x) { const TC c = make_tc(E, b); acc += EL(c, total, 1, 0); }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, acc);
}

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static int fail(int code, const char* msg) { g_err = msg; return code; }
static int fail_cuda(cudaError_t e, const char* where) {
    char buf[256]; snprintf(buf, sizeof buf, "%s: CUDA error %d (%s)", where, (int)e, cudaGetErrorString(e));
    g_err = buf; return DCM_ERR_CUDA;
}
#define CK(call) do { cudaError_t _e = (call); if (_e != cudaSuccess) return fail_cuda(_e, #call); } while (0)
// kernels are instantiated for 1, 2 and 4 mask words (T <= 64 / 128 / 254): TW_KERNEL is the instance for the handle's shape
#define TW_KERNEL(v, kern) ((v)->E.S.TW == 1 ? kern<1> : (v)->E.S.TW == 2 ? kern<2> : kern<4>)
#define LAUNCH_TW(v, kern, grid, block, smem, stream, ...) TW_KERNEL(v, kern)<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__)

struct dcm_env {
    int device; EnvArgs E; DcmLayout L; bool have_instances;
    bool serial_pass;                // DCM_PASS_SERIAL=1 at dcm_create: k_step, k_episode_list, k_obs one after the other on the caller's stream (cross-check)
    unsigned long long* d_trace; size_t trace_units;   // DCM_PASS_TRACE=1: globaltimer stamps of k_obs_tile blocks / k_episode_list warps (tools/obs_trace.py)
    unsigned char* arena; size_t arena_bytes;
    double* metrics;                 // [B,8]
    unsigned long long* d_counter;   // scratch for reductions
    unsigned char* d_cursor;         // [B,A] route cursors
    unsigned char* d_record;         // [B,dyn_bytes] export staging
    // dcm_step_host staging
    int* d_action; float* d_agent; float* d_task; unsigned char* d_mask; int* d_leader; float* d_reward; unsigned char* d_done;
    cudaStream_t hstream, hcopy; bool forked;   // dcm_step_host: its stream; a second one for the results k_step alone produces; the last dcm_step recorded ev_fork
    cudaStream_t side; cudaEvent_t ev_fork, ev_join;   // k_episode_list runs beside k_obs
    int sm_count;
    bool obs_ready, obs_tile, obs_resets;   // k_obs_tile applies to this handle's shape (DCM_OBS_CHUNKED=1: always k_obs); it also writes restarted envs' observations
    unsigned* d_elist; unsigned* d_ecount; unsigned pass_no;   // ended-env list [B] + two alternating counters (k_episode_list)
    // DCM_* cross-checks: second implementations of default paths that the tests compare the defaults against (with serial_pass
    // above; DCM_PASS_TRACE allocates d_trace).  Read once in dcm_create, never on the step path.
    bool sw_obs_reset_by_episode, sw_obs_chunked, sw_step_no_nds;
    // dcm_step_host runs on its own stream: it must start after the asynchronous work earlier calls queued on the CALLER's stream
    cudaStream_t last_stream; bool last_pending; cudaEvent_t ev_order;
    uint64_t launches;
};

// remember the stream an asynchronous entry point queued work on (dcm_step_host orders itself after it)
static inline void note_stream(dcm_env* v, cudaStream_t s) { if (s != v->hstream || !v->hstream) { v->last_stream = s; v->last_pending = true; } }

struct DeviceGuard {
    int prev, target; bool ok;
    explicit DeviceGuard(int dev) : prev(-1), target(dev) { ok = cudaGetDevice(&prev) == cudaSuccess && (prev == dev || cudaSetDevice(dev) == cudaSuccess); }
    ~DeviceGuard() { if (ok && prev != target) cudaSetDevice(prev); }
};

static int grid_env(const dcm_env* v, int threads) { return (v->E.S.B + threads - 1) / threads; }

extern "C" {

const char* dcm_last_error(void) { return g_err.c_str(); }
const char* dcm_version(void) { return "dcmrta_b200 0.4 (sm_100a, thread-per-env, tiled state + bitmask summaries)"; }

int dcm_create(dcm_env** out, int device, int B, int A, int T, int M, uint32_t flags) {
    if (!out) return fail(DCM_ERR_ARG, "dcm_create: out is NULL");
    *out = nullptr;
    if (B < 1 || A < 1 || A > DCM_MAX_AGENTS || T < 1 || T > DCM_MAX_TASKS || M < 1 || M > DCM_MAX_M)
        return fail(DCM_ERR_SHAPE, "dcm_create: need B>=1, 1<=A<=64, 1<=T<=254, 1<=M<=8");
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) { cudaGetLastError(); return fail(DCM_ERR_DEVICE, "dcm_create: no CUDA device (there is no CPU fallback)"); }
    if (device < 0 || device >= n) return fail(DCM_ERR_DEVICE, "dcm_create: bad device index");
    DeviceGuard g(device);
    if (!g.ok) return fail(DCM_ERR_DEVICE, "dcm_create: cudaSetDevice failed");
    dcm_env* v = new (std::nothrow) dcm_env();
    if (!v) return fail(DCM_ERR_NOMEM, "dcm_create: host allocation failed");
    memset(v, 0, sizeof *v);
    v->device = device;
    // the cross-checks and the pass trace (dcm_env), once per handle
    auto on = [](const char* name) { const char* g = getenv(name); return g && g[0] == '1'; };
    v->serial_pass = on("DCM_PASS_SERIAL"); v->sw_obs_chunked = on("DCM_OBS_CHUNKED"); v->sw_obs_reset_by_episode = on("DCM_OBS_RESET_BY_EPISODE");
    v->sw_step_no_nds = on("DCM_STEP_NO_NDS");
    const bool pass_trace = on("DCM_PASS_TRACE");
    v->L = dcm_make_layout(A, T, M);
    DcmSoa& S = v->E.S;
    S.B = B; S.NT = (B + 31) / 32; S.A = A; S.T = T; S.M = M; S.MC = M; S.TW = T <= 64 ? 1 : (T <= 128 ? 2 : 4);
    v->E.W = 10.0; v->E.vel = 0.2; v->E.max_time = 100.0; v->E.seed = 0; v->E.first_gid = 0; v->E.cflags = flags;
    v->E.gen_max_duration = 5.0; v->E.gen_random_duration = 0;
    // carve one tile block; every array is [K][32 lanes] inside it, 256-byte aligned; the arena is NT such blocks
    const int NT = S.NT, TW = S.TW;
    size_t off = 0;
    auto carve = [&](int K, size_t elem) { size_t o = off; off += (dcm_soa_bytes(K, elem) + 255) / 256 * 256; return o; };
    const int MCB = 8; S.MCB = MCB; S.ANB = A <= 32 ? 32 : 64;
    const size_t o_slot_arr = carve(T, 8 * (size_t)M), o_t_rec = carve(T, 64), o_a_rec = carve(A, 32), o_a_obs = carve(A, 16),
                 o_a_nd = carve(A, 8), o_a_ts = carve(A, 8), o_now = carve(1, 8), o_x_fin = carve(1, 8), o_x_amin = carve(1, 8), o_x_ret = carve(1, 8), o_x_last = carve(1, 8), o_pending = carve(1, 8), o_group = carve(1, 8),
                 o_s_tx = carve(T, 8), o_s_ty = carve(T, 8), o_s_dur = carve(T, 8), o_s_dur32 = carve(T, 4), o_s_dep = carve(2, 8), o_w_agent = carve(A, 8),
                 o_m_feas = carve(TW, 8), o_m_fin = carve(TW, 8), o_m_ne = carve(TW, 8), o_m_open = carve(TW, 8), o_m_dirty = carve(TW, 8),
                 o_am_route = carve(1, 8), o_am_assigned = carve(1, 8), o_am_returned = carve(1, 8), o_am_member = carve(1, 8), o_am_depot = carve(1, 8),
                 o_am_touched = carve(1, 8), o_am_watch = carve(1, 8),
                 o_n_steps = carve(1, 4), o_episode = carve(1, 4), o_flags = carve(1, 4), o_instance = carve(1, 4), o_total = carve(1, 4), o_leader = carve(1, 4),
                 o_a_nab = carve(A, 2),
                 o_ended = carve(1, 1), o_t_status = carve(T, 1), o_a_node = carve(1, S.ANB), o_s_req = carve(T, 1);
    S.tile_stride = off;
    v->arena_bytes = off * (size_t)NT;
    cudaError_t e = cudaMalloc((void**)&v->arena, v->arena_bytes);
    if (e == cudaSuccess) e = cudaMemset(v->arena, 0, v->arena_bytes);
    if (e == cudaSuccess) e = cudaMalloc((void**)&v->metrics, (size_t)B * 8 * sizeof(double));
    if (e == cudaSuccess) e = cudaMemset(v->metrics, 0, (size_t)B * 8 * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc((void**)&v->d_counter, sizeof(unsigned long long));
    int prio_lo = 0, prio_hi = 0;
    if (e == cudaSuccess) e = cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    // highest priority: the few long episode chains must get their blocks in before the six waves of k_obs that run beside them
    if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&v->side, cudaStreamNonBlocking, prio_hi);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&v->ev_fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&v->ev_join, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaMalloc((void**)&v->d_elist, (size_t)B * sizeof(unsigned));
    if (e == cudaSuccess) e = cudaMalloc((void**)&v->d_ecount, 2 * sizeof(unsigned));
    if (e == cudaSuccess) e = cudaMemset(v->d_ecount, 0, 2 * sizeof(unsigned));
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&v->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&v->ev_order, cudaEventDisableTiming);
    if (e == cudaSuccess && pass_trace) { v->trace_units = (size_t)NT * 64; e = cudaMalloc((void**)&v->d_trace, v->trace_units * 4 * sizeof(unsigned long long)); if (e == cudaSuccess) e = cudaMemset(v->d_trace, 0, v->trace_units * 4 * sizeof(unsigned long long)); }
    if (e != cudaSuccess) { dcm_destroy(v); return e == cudaErrorMemoryAllocation ? fail(DCM_ERR_NOMEM, "dcm_create: cudaMalloc failed") : fail_cuda(e, "dcm_create"); }
    unsigned char* a = v->arena;
    S.t_slot_arr = (double*)(a + o_slot_arr); S.t_rec = (double*)(a + o_t_rec); S.a_rec = (double*)(a + o_a_rec); S.a_obs = (double*)(a + o_a_obs);
    S.a_nd = (double*)(a + o_a_nd); S.a_ts = (double*)(a + o_a_ts); S.now = (double*)(a + o_now); S.x_fin = (double*)(a + o_x_fin); S.x_amin = (double*)(a + o_x_amin); S.x_ret = (double*)(a + o_x_ret); S.x_last = (double*)(a + o_x_last); S.pending = (u64*)(a + o_pending); S.group = (u64*)(a + o_group);
    S.s_tx = (double*)(a + o_s_tx); S.s_ty = (double*)(a + o_s_ty); S.s_dur = (double*)(a + o_s_dur); S.s_dur32 = (float*)(a + o_s_dur32); S.s_dep = (double*)(a + o_s_dep); S.w_agent = (double*)(a + o_w_agent);
    S.m_feas = (u64*)(a + o_m_feas); S.m_fin = (u64*)(a + o_m_fin); S.m_ne = (u64*)(a + o_m_ne); S.m_open = (u64*)(a + o_m_open); S.m_dirty = (u64*)(a + o_m_dirty);
    S.am_route = (u64*)(a + o_am_route); S.am_assigned = (u64*)(a + o_am_assigned); S.am_returned = (u64*)(a + o_am_returned); S.am_member = (u64*)(a + o_am_member);
    S.am_depot = (u64*)(a + o_am_depot); S.am_touched = (u64*)(a + o_am_touched); S.am_watch = (u64*)(a + o_am_watch);
    S.n_steps = (unsigned*)(a + o_n_steps); S.episode = (unsigned*)(a + o_episode); S.flags = (unsigned*)(a + o_flags);
    S.instance = (unsigned*)(a + o_instance); S.total = (unsigned*)(a + o_total); S.leader = (int*)(a + o_leader);
    S.a_nab = (unsigned short*)(a + o_a_nab);
    S.ended = a + o_ended; S.t_status = (signed char*)(a + o_t_status); S.a_node = a + o_a_node; S.s_req = a + o_s_req;
    k_init<<<(S.NT * 32 + 127) / 128, 128>>>(v->E);
    e = cudaDeviceSynchronize();

    if (e != cudaSuccess) { dcm_destroy(v); return fail_cuda(e, "dcm_create init"); }
    v->launches = 1;
    *out = v;
    return DCM_OK;
}

int dcm_destroy(dcm_env* v) {
    if (!v) return DCM_OK;
    DeviceGuard g(v->device);
    cudaFree(v->arena); cudaFree(v->metrics); cudaFree(v->d_counter); cudaFree(v->d_trace); cudaFree(v->d_cursor); cudaFree(v->d_record); cudaFree(v->d_elist); cudaFree(v->d_ecount);
    cudaFree(v->d_action); cudaFree(v->d_agent); cudaFree(v->d_task); cudaFree(v->d_mask); cudaFree(v->d_leader); cudaFree(v->d_reward); cudaFree(v->d_done);
    if (v->hstream) cudaStreamDestroy(v->hstream);
    if (v->hcopy) cudaStreamDestroy(v->hcopy);
    if (v->side) cudaStreamDestroy(v->side);
    if (v->ev_fork) cudaEventDestroy(v->ev_fork);
    if (v->ev_join) cudaEventDestroy(v->ev_join);
    if (v->ev_order) cudaEventDestroy(v->ev_order);
    delete v;
    return DCM_OK;
}

int dcm_set_params(dcm_env* v, double velocity, double max_wait, double max_time) {
    if (!v) return fail(DCM_ERR_ARG, "dcm_set_params: env is NULL");
    if (!(velocity > 0) || !(max_wait >= 0)) return fail(DCM_ERR_ARG, "dcm_set_params: velocity must be > 0 and max_wait >= 0");
    v->E.vel = velocity; v->E.W = max_wait; v->E.max_time = max_time;
    return DCM_OK;
}

int dcm_seed(dcm_env* v, uint64_t seed, uint64_t first_gid) {
    if (!v) return fail(DCM_ERR_ARG, "dcm_seed: env is NULL");
    v->E.seed = seed; v->E.first_gid = first_gid;
    return DCM_OK;
}

int dcm_load_instances(dcm_env* v, const double* task_xy, const double* depot_xy, const int32_t* req, const double* dur, void* stream) {
    if (!v || !task_xy || !depot_xy || !req || !dur) return fail(DCM_ERR_ARG, "dcm_load_instances: NULL argument");
    DeviceGuard g(v->device);
    k_pack_static<<<grid_env(v, 128), 128, 0, (cudaStream_t)stream>>>(v->E, task_xy, depot_xy, req, dur);
    CK(cudaGetLastError());
    note_stream(v, (cudaStream_t)stream);
    v->launches++; v->have_instances = true;
    return DCM_OK;
}

int dcm_load_instances_host(dcm_env* v, const double* task_xy, const double* depot_xy, const int32_t* req, const double* dur) {
    if (!v || !task_xy || !depot_xy || !req || !dur) return fail(DCM_ERR_ARG, "dcm_load_instances_host: NULL argument");
    DeviceGuard g(v->device);
    const size_t B = v->E.S.B, T = v->E.S.T;
    for (size_t k = 0; k < B * T; ++k) if (req[k] < 1 || req[k] > v->E.S.M) return fail(DCM_ERR_ARG, "dcm_load_instances_host: requirement outside [1, M]");
    double *dxy = nullptr, *ddep = nullptr, *ddur = nullptr; int* dreq = nullptr;
    cudaError_t e = cudaMalloc(&dxy, B * T * 2 * 8);
    if (e == cudaSuccess) e = cudaMalloc(&ddep, B * 2 * 8);
    if (e == cudaSuccess) e = cudaMalloc(&ddur, B * T * 8);
    if (e == cudaSuccess) e = cudaMalloc(&dreq, B * T * 4);
    if (e == cudaSuccess) e = cudaMemcpy(dxy, task_xy, B * T * 2 * 8, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(ddep, depot_xy, B * 2 * 8, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(ddur, dur, B * T * 8, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(dreq, req, B * T * 4, cudaMemcpyHostToDevice);
    int rc = DCM_OK;
    if (e == cudaSuccess) { rc = dcm_load_instances(v, dxy, ddep, dreq, ddur, nullptr); if (rc == DCM_OK) e = cudaDeviceSynchronize(); }
    cudaFree(dxy); cudaFree(ddep); cudaFree(ddur); cudaFree(dreq);
    if (e != cudaSuccess) return fail_cuda(e, "dcm_load_instances_host");
    return rc;
}

int dcm_generate(dcm_env* v, double max_duration, int random_duration, void* stream) {
    if (!v) return fail(DCM_ERR_ARG, "dcm_generate: env is NULL");
    DeviceGuard g(v->device);
    v->E.gen_max_duration = max_duration; v->E.gen_random_duration = random_duration;
    k_generate<<<grid_env(v, 128), 128, 0, (cudaStream_t)stream>>>(v->E, v->have_instances ? 1 : 0);
    CK(cudaGetLastError());
    note_stream(v, (cudaStream_t)stream);
    v->launches++; v->have_instances = true;
    return DCM_OK;
}

int dcm_get_instances(dcm_env* v, double* task_xy, double* depot_xy, int32_t* req, double* dur, void* stream) {
    if (!v) return fail(DCM_ERR_ARG, "dcm_get_instances: env is NULL");
    if (!v->have_instances) return fail(DCM_ERR_STATE, "dcm_get_instances: no instances installed");
    DeviceGuard g(v->device);
    k_unpack_static<<<grid_env(v, 128), 128, 0, (cudaStream_t)stream>>>(v->E, task_xy, depot_xy, req, dur);
    CK(cudaGetLastError());
    v->launches++;
    return DCM_OK;
}

// the step path's observation builder: k_obs_tile when two tiles fit in an SM's shared memory, else (or with DCM_OBS_CHUNKED=1) k_obs
static int launch_obs_tile(dcm_env* v, const ObsArgs& O, cudaStream_t s, bool programmatic = false) {
    const int A = v->E.S.A, T = v->E.S.T;
    const int NA = (A + OBS_AGENTS_PER_CHUNK - 1) / OBS_AGENTS_PER_CHUNK, NR = (T + 1 + OBS_ROWS_PER_CHUNK - 1) / OBS_ROWS_PER_CHUNK;
    const int warps = NA + NR < OBS_TILE_MAX_WARPS ? NA + NR : OBS_TILE_MAX_WARPS;
    const size_t smem = obs_tile_smem(A, T).total;
    const int use_bulk = (((uintptr_t)O.agent_obs | (uintptr_t)O.task_obs | (uintptr_t)O.mask) & 15u) == 0;
    cudaLaunchConfig_t cfg; memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3(v->E.S.NT); cfg.blockDim = dim3(32 * warps); cfg.dynamicSmemBytes = smem; cfg.stream = s;   // one block per tile
    cudaLaunchAttribute attr; memset(&attr, 0, sizeof attr);
    attr.id = cudaLaunchAttributeProgrammaticStreamSerialization; attr.val.programmaticStreamSerializationAllowed = 1;
    if (programmatic) { cfg.attrs = &attr; cfg.numAttrs = 1; }               // after k_step in dcm_step: resident early, waits in griddepcontrol.wait
    CK(cudaLaunchKernelEx(&cfg, TW_KERNEL(v, k_obs_tile), v->E, O, use_bulk, v->d_trace));
    CK(cudaGetLastError());
    v->launches++;
    return DCM_OK;
}

// decide once per handle whether the tile kernel applies, and opt in to the shared memory it needs
static int prepare_obs(dcm_env* v) {
    if (v->obs_ready) return DCM_OK;
    v->obs_ready = true; v->obs_tile = false;
    v->obs_resets = !v->sw_obs_reset_by_episode;
    if (v->sw_obs_chunked) return DCM_OK;
    int optin = 0, per_sm = 0;
    CK(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, v->device));
    CK(cudaDeviceGetAttribute(&per_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, v->device));
    const size_t smem = obs_tile_smem(v->E.S.A, v->E.S.T).total;
    if (smem > (size_t)optin || 2 * (smem + 1024) > (size_t)per_sm) return DCM_OK;
    CK(cudaFuncSetAttribute(TW_KERNEL(v, k_obs_tile), cudaFuncAttributeMaxDynamicSharedMemorySize, optin));   // per function, not per handle: the device maximum
    CK(cudaFuncSetAttribute(TW_KERNEL(v, k_obs_tile), cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    // The episode kernel runs BESIDE this one and has to share SMs with it: blocks of kernels that ask for different L1 /
    // shared-memory splits do not become co-resident on an SM (measured: side by side the two kernels took as long as one
    // after the other, profiles/r03_timeline.txt), so it asks for the same split.
    CK(cudaFuncSetAttribute(TW_KERNEL(v, k_episode_list), cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    v->obs_tile = true;
    return DCM_OK;
}

static int launch_obs(dcm_env* v, const ObsArgs& O, cudaStream_t s, bool programmatic = false) {
    { const int rc = prepare_obs(v); if (rc) return rc; }
    if (v->obs_tile) return launch_obs_tile(v, O, s, programmatic);
    const int tiles_per_block = OBS_THREADS / 32;
    const int NA = (v->E.S.A + OBS_AGENTS_PER_CHUNK - 1) / OBS_AGENTS_PER_CHUNK, NR = (v->E.S.T + 1 + OBS_ROWS_PER_CHUNK - 1) / OBS_ROWS_PER_CHUNK;
    const dim3 grid((v->E.S.NT + tiles_per_block - 1) / tiles_per_block, NA + NR);
    LAUNCH_TW(v, k_obs, grid, OBS_THREADS, 0, s, v->E, O);
    CK(cudaGetLastError());
    v->launches++;
    return DCM_OK;
}

static int launch_episode_list(dcm_env* v, const EpiArgs& P, const unsigned* ecount, cudaStream_t s) {
    const int nw = EPI_LIST_WARPS;
    const size_t smem = nw * ((epi_scratch_bytes(v->E.S.A, v->E.S.T, v->E.S.MC) + 15) / 16 * 16);
    int grid = (v->sm_count * EPI_LIST_WARPS_PER_SM + nw - 1) / nw; if (grid > v->E.S.B) grid = v->E.S.B;
    if (v->d_trace) CK(cudaMemsetAsync(v->d_trace + (size_t)v->E.S.NT * 8, 0, (size_t)grid * nw * 4 * sizeof(unsigned long long), s));
    LAUNCH_TW(v, k_episode_list, grid, 32 * nw, smem, s, v->E, P, v->d_elist, ecount, v->d_trace);
    CK(cudaGetLastError());
    v->launches++;
    return DCM_OK;
}

int dcm_reset(dcm_env* v, const uint8_t* which, const int32_t* leader_in, float* agent_obs, float* task_obs, uint8_t* mask,
              int32_t* next_leader, void* stream) {
    if (!v) return fail(DCM_ERR_ARG, "dcm_reset: env is NULL");
    if (!v->have_instances) return fail(DCM_ERR_STATE, "dcm_reset: load or generate instances first");
    DeviceGuard g(v->device);
    cudaStream_t s = (cudaStream_t)stream;
    note_stream(v, s);
    EpiArgs P{1, which, leader_in, next_leader, v->metrics, ObsArgs{nullptr, nullptr, nullptr, nullptr, 0}, 0};
    LAUNCH_TW(v, k_episode, v->E.S.NT * EPI_WARPS, 32, epi_scratch_bytes(v->E.S.A, v->E.S.T, v->E.S.MC), s, v->E, P);
    CK(cudaGetLastError());
    v->launches++;
    ObsArgs O{nullptr, agent_obs, task_obs, mask, 0};
    if (agent_obs || task_obs || mask) return launch_obs(v, O, s);
    return DCM_OK;
}

int dcm_step(dcm_env* v, const int32_t* action, const int32_t* followers, int fstride, const int32_t* next_leader_in, int policy,
             float* agent_obs, float* task_obs, uint8_t* mask, int32_t* next_leader, float* reward, uint8_t* done, int32_t* used_action, void* stream) {
    if (!v) return fail(DCM_ERR_ARG, "dcm_step: env is NULL");
    if (!v->have_instances) return fail(DCM_ERR_STATE, "dcm_step: load or generate instances first");
    if (policy < 0 || policy > 2) return fail(DCM_ERR_ARG, "dcm_step: unknown policy");
    if (policy == DCM_POLICY_EXTERNAL && !action) return fail(DCM_ERR_ARG, "dcm_step: action is NULL with the external policy");
    if (followers && fstride < 0) return fail(DCM_ERR_ARG, "dcm_step: negative follower stride");
    DeviceGuard g(v->device);
    cudaStream_t s = (cudaStream_t)stream;
    note_stream(v, s);
    StepArgs F; memset(&F, 0, sizeof F);
    F.action = action; F.followers = followers; F.fstride = fstride; F.leader_in = next_leader_in; F.policy = policy;
    F.next_leader = next_leader; F.reward = reward; F.done = done; F.used_action = used_action;
    ObsArgs O{nullptr, agent_obs, task_obs, mask, 0};
    EpiArgs P{0, nullptr, next_leader_in, next_leader, v->metrics, O, 0};
    const bool want_obs = agent_obs || task_obs || mask;
    const unsigned p = v->pass_no++ & 1u;
    unsigned* ecount = v->d_ecount + p; F.elist = v->d_elist; F.ecount = ecount; F.ecount_next = v->d_ecount + (p ^ 1u);
    if (v->d_trace) {                                                         // the last two words of the trace buffer: k_step's first entry / last exit
        F.trace = v->d_trace + v->trace_units * 4 - 2;
        CK(cudaMemsetAsync(F.trace, 0xff, sizeof(unsigned long long), s)); CK(cudaMemsetAsync(F.trace + 1, 0, sizeof(unsigned long long), s));
    }
    {
        F.use_nds = v->E.S.A <= STEP_NDS_MAX_AGENTS && !v->sw_step_no_nds;
        const int grid = grid_env(v, STEP_THREADS); const size_t smem = step_smem_bytes(v->E.S.A, v->E.S.ANB, F.use_nds != 0);
        if (v->E.cflags & DCM_FLAG_INDIVIDUAL) LAUNCH_TW(v, k_step_ia, grid, STEP_THREADS, smem, s, v->E, F);
        else LAUNCH_TW(v, k_step, grid, STEP_THREADS, smem, s, v->E, F);
    }
    CK(cudaGetLastError());
    v->launches++;
    // Episode accounting (+ restart with DCM_FLAG_AUTO_RESET) of the envs that just finished; the injected leader of a
    // restarted env is the same next_leader_in entry.  The episode kernel is a few hundred long, latency-bound warp
    // chains (~30 us) and k_obs is bandwidth-bound (~60 us): they run side by side.  k_obs leaves out the envs k_step marked
    // `ended`; k_episode_list writes the observation of the envs it restarts from registers (episode_env).
    if (v->serial_pass || !want_obs) {
        int rc = launch_episode_list(v, P, ecount, s);
        if (rc) return rc;
        if (want_obs) return launch_obs(v, O, s);
        return DCM_OK;
    }
    { const int rc0 = prepare_obs(v); if (rc0) return rc0; }
    CK(cudaEventRecord(v->ev_fork, s));
    v->forked = true;
    // the restarted envs' observation: by k_obs_tile itself when it only depends on the static instance (auto-reset without
    // regeneration; DCM_OBS_RESET_BY_EPISODE=1 switches back), else by the episode kernel, from the registers that hold the new instance
    const bool auto_reset = (v->E.cflags & DCM_FLAG_AUTO_RESET) != 0;
    const bool obs_resets = auto_reset && v->obs_tile && v->obs_resets && !(v->E.cflags & DCM_FLAG_REGENERATE) && v->E.max_time > 0.0;
    P.obs = O; P.write_obs = (auto_reset && !obs_resets) ? 1 : 0;
    O.skip_ended = obs_resets ? 2 : 1;
    CK(cudaStreamWaitEvent(v->side, v->ev_fork, 0));
    int rc = launch_episode_list(v, P, ecount, v->side);
    if (rc) return rc;
    CK(cudaEventRecord(v->ev_join, v->side));
    rc = launch_obs(v, O, s, true);
    if (rc) return rc;
    CK(cudaStreamWaitEvent(s, v->ev_join, 0));
    return DCM_OK;
}

static int ensure_host_staging(dcm_env* v) {
    if (v->hstream) return DCM_OK;
    const size_t B = v->E.S.B, A = v->E.S.A, T = v->E.S.T;
    CK(cudaMalloc(&v->d_action, B * 4)); CK(cudaMalloc(&v->d_agent, B * A * 6 * 4)); CK(cudaMalloc(&v->d_task, B * (T + 1) * 5 * 4));
    CK(cudaMalloc(&v->d_mask, B * (T + 1))); CK(cudaMalloc(&v->d_leader, B * 4)); CK(cudaMalloc(&v->d_reward, B * 4)); CK(cudaMalloc(&v->d_done, B));
    CK(cudaStreamCreateWithFlags(&v->hstream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&v->hcopy, cudaStreamNonBlocking));
    return DCM_OK;
}

int dcm_step_host(dcm_env* v, const int32_t* action, int policy, float* agent_obs, float* task_obs, uint8_t* mask,
                  int32_t* next_leader, float* reward, uint8_t* done) {
    if (!v) return fail(DCM_ERR_ARG, "dcm_step_host: env is NULL");
    if (policy == DCM_POLICY_EXTERNAL && !action) return fail(DCM_ERR_ARG, "dcm_step_host: action is NULL with the external policy");
    DeviceGuard g(v->device);
    int rc = ensure_host_staging(v);
    if (rc) return rc;
    const size_t B = v->E.S.B, A = v->E.S.A, T = v->E.S.T;
    cudaStream_t s = v->hstream;
    // hstream is a non-blocking stream: order it after whatever earlier calls (dcm_reset, dcm_generate, dcm_load_instances, dcm_step,
    // granular ops, dcm_import_state) queued asynchronously on the caller's stream -- including the legacy NULL stream
    if (v->last_pending) {
        CK(cudaEventRecord(v->ev_order, v->last_stream));
        CK(cudaStreamWaitEvent(s, v->ev_order, 0));
        v->last_pending = false;
    }
    // Actions in PINNED host memory are read in place: under unified addressing the step kernel's first round of loads fetches them over
    // PCIe (one coalesced 128-byte read per warp, beside its reads of the state) instead of waiting for a 256 kB copy to land first.
    // Pageable memory is staged through d_action.  (The attribute query is repeated per call: a cached answer could outlive the buffer.)
    const int32_t* act_d = v->d_action;
    if (action) {
        cudaPointerAttributes pa;
        if (cudaPointerGetAttributes(&pa, action) == cudaSuccess && pa.type == cudaMemoryTypeHost && pa.devicePointer)
            act_d = (const int32_t*)pa.devicePointer;
        else { cudaGetLastError(); CK(cudaMemcpyAsync(v->d_action, action, B * 4, cudaMemcpyHostToDevice, s)); }
    }
    v->forked = false;
    rc = dcm_step(v, act_d, nullptr, 0, nullptr, policy, v->d_agent, v->d_task, v->d_mask, v->d_leader, v->d_reward, v->d_done, nullptr, s);
    if (rc) return rc;
    // next_leader, reward and done are final when k_step ends (ev_fork; k_step also knows the first leader of an episode the
    // episode kernel is about to restart): they travel to the host while the episode and observation kernels run
    if (v->forked && (reward || done || next_leader)) {
        CK(cudaStreamWaitEvent(v->hcopy, v->ev_fork, 0));
        if (next_leader) CK(cudaMemcpyAsync(next_leader, v->d_leader, B * 4, cudaMemcpyDeviceToHost, v->hcopy));
        if (reward) CK(cudaMemcpyAsync(reward, v->d_reward, B * 4, cudaMemcpyDeviceToHost, v->hcopy));
        if (done) CK(cudaMemcpyAsync(done, v->d_done, B, cudaMemcpyDeviceToHost, v->hcopy));
        reward = nullptr; done = nullptr; next_leader = nullptr;
    }
    if (agent_obs) CK(cudaMemcpyAsync(agent_obs, v->d_agent, B * A * 6 * 4, cudaMemcpyDeviceToHost, s));
    if (task_obs) CK(cudaMemcpyAsync(task_obs, v->d_task, B * (T + 1) * 5 * 4, cudaMemcpyDeviceToHost, s));
    if (mask) CK(cudaMemcpyAsync(mask, v->d_mask, B * (T + 1), cudaMemcpyDeviceToHost, s));
    if (next_leader) CK(cudaMemcpyAsync(next_leader, v->d_leader, B * 4, cudaMemcpyDeviceToHost, s));
    if (reward) CK(cudaMemcpyAsync(reward, v->d_reward, B * 4, cudaMemcpyDeviceToHost, s));
    if (done) CK(cudaMemcpyAsync(done, v->d_done, B, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (v->forked) CK(cudaStreamSynchronize(v->hcopy));
    return DCM_OK;
}

int dcm_episode_metrics(dcm_env* v, double* out, void* stream) {
    if (!v || !out) return fail(DCM_ERR_ARG, "dcm_episode_metrics: NULL argument");
    DeviceGuard g(v->device);
    CK(cudaMemcpyAsync(out, v->metrics, (size_t)v->E.S.B * 8 * sizeof(double), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return DCM_OK;
}

static int launch_gran(dcm_env* v, const GranArgs& G, void* stream) {
    if (!v->have_instances) return fail(DCM_ERR_STATE, "granular op: load or generate instances first");
    DeviceGuard g(v->device);
    LAUNCH_TW(v, k_granular, grid_env(v, STEP_THREADS), STEP_THREADS, 0, (cudaStream_t)stream, v->E, G);
    CK(cudaGetLastError());
    note_stream(v, (cudaStream_t)stream);
    v->launches++;
    return DCM_OK;
}
#define GRAN_BEGIN(name, cond) if (!v || !(cond)) return fail(DCM_ERR_ARG, name ": NULL argument"); GranArgs G; memset(&G, 0, sizeof G)

int dcm_next_decision(dcm_env* v, uint64_t* deciders, double* t, void* stream) {
    GRAN_BEGIN("dcm_next_decision", deciders && t); G.op = OP_NEXT_DECISION; G.deciders = (u64*)deciders; G.t = t; return launch_gran(v, G, stream);
}
int dcm_unique_group(dcm_env* v, const uint64_t* deciders, int8_t* group_rank, void* stream) {
    GRAN_BEGIN("dcm_unique_group", deciders && group_rank); G.op = OP_UNIQUE_GROUP; G.deciders_in = (const u64*)deciders; G.group_rank = (signed char*)group_rank; return launch_gran(v, G, stream);
}
int dcm_set_clock(dcm_env* v, const double* t, void* stream) {
    if (!v) return fail(DCM_ERR_ARG, "dcm_set_clock: env is NULL");
    if (!t) return DCM_OK;
    GranArgs G; memset(&G, 0, sizeof G); G.op = OP_SET_CLOCK; G.t_in = t; return launch_gran(v, G, stream);
}
int dcm_get_clock(dcm_env* v, double* t, void* stream) {
    GRAN_BEGIN("dcm_get_clock", t); G.op = OP_GET_CLOCK; G.t = t; return launch_gran(v, G, stream);
}
int dcm_task_update(dcm_env* v, uint8_t* newly, void* stream) {
    GRAN_BEGIN("dcm_task_update", true); G.op = OP_TASK_UPDATE; G.newly = newly; return launch_gran(v, G, stream);
}
int dcm_agent_update(dcm_env* v, void* stream) {
    GRAN_BEGIN("dcm_agent_update", true); G.op = OP_AGENT_UPDATE; return launch_gran(v, G, stream);
}
int dcm_apply_members(dcm_env* v, const int32_t* action, const int32_t* members, int mstride, const int32_t* n_members, double* reward, void* stream) {
    GRAN_BEGIN("dcm_apply_members", action && members && n_members && mstride > 0);
    G.op = OP_APPLY_MEMBERS; G.action = action; G.members = members; G.mstride = mstride; G.n_members = n_members; G.reward = reward;
    return launch_gran(v, G, stream);
}
int dcm_build_obs(dcm_env* v, const int32_t* leader, float* agent_obs, float* task_obs, uint8_t* mask, void* stream) {
    if (!v || !leader) return fail(DCM_ERR_ARG, "dcm_build_obs: NULL argument");
    if (!v->have_instances) return fail(DCM_ERR_STATE, "dcm_build_obs: load or generate instances first");
    DeviceGuard g(v->device);
    ObsArgs O{leader, agent_obs, task_obs, mask, 0};
    note_stream(v, (cudaStream_t)stream);
    return launch_obs(v, O, (cudaStream_t)stream);
}
int dcm_check_finished(dcm_env* v, uint8_t* finished, void* stream) {
    GRAN_BEGIN("dcm_check_finished", finished); G.op = OP_CHECK_FINISHED; G.finished = finished; return launch_gran(v, G, stream);
}
int dcm_compute_metrics(dcm_env* v, double* out, double* task_wait, double* agent_wait, void* stream) {
    GRAN_BEGIN("dcm_compute_metrics", out); G.op = OP_COMPUTE_METRICS; G.metrics = out; G.task_wait = task_wait; G.agent_wait = agent_wait;
    return launch_gran(v, G, stream);
}
int dcm_env_flags(dcm_env* v, uint32_t* flags, void* stream) {
    GRAN_BEGIN("dcm_env_flags", flags); G.op = OP_ENV_FLAGS; G.flags_out = flags; return launch_gran(v, G, stream);
}

int dcm_execute_by_route(dcm_env* v, const int32_t* routes, int rstride, const int32_t* route_len, double* makespan, void* stream) {
    if (!v || !routes || !route_len || rstride < 1) return fail(DCM_ERR_ARG, "dcm_execute_by_route: bad argument");
    if (rstride > 255) return fail(DCM_ERR_SHAPE, "dcm_execute_by_route: routes longer than 255 are not supported");
    if (!v->have_instances) return fail(DCM_ERR_STATE, "dcm_execute_by_route: load instances first");
    DeviceGuard g(v->device);
    if (!v->d_cursor) CK(cudaMalloc(&v->d_cursor, (size_t)v->E.S.B * v->E.S.A));
    LAUNCH_TW(v, k_routes, grid_env(v, STEP_THREADS), STEP_THREADS, 0, (cudaStream_t)stream, v->E, routes, rstride, route_len, v->d_cursor, makespan);
    CK(cudaGetLastError());
    note_stream(v, (cudaStream_t)stream);
    v->launches++;
    return DCM_OK;
}

size_t dcm_record_bytes(const dcm_env* v) { return v ? (size_t)v->L.dyn_bytes : 0; }

int dcm_export_state(dcm_env* v, void* dst, size_t bytes, void* stream) {
    if (!v || !dst) return fail(DCM_ERR_ARG, "dcm_export_state: NULL argument");
    const size_t need = (size_t)v->E.S.B * v->L.dyn_bytes;
    if (bytes < need) return fail(DCM_ERR_ARG, "dcm_export_state: buffer too small");
    DeviceGuard g(v->device);
    if (!v->d_record) { CK(cudaMalloc(&v->d_record, need)); }
    cudaStream_t s = (cudaStream_t)stream;
    CK(cudaMemsetAsync(v->d_record, 0, need, s));
    LAUNCH_TW(v, k_export, grid_env(v, 128), 128, 0, s, v->E, v->L, v->d_record);
    CK(cudaGetLastError());
    v->launches++;
    CK(cudaMemcpyAsync(dst, v->d_record, need, cudaMemcpyDefault, s));
    return DCM_OK;
}
int dcm_import_state(dcm_env* v, const void* src, size_t bytes, void* stream) {
    if (!v || !src) return fail(DCM_ERR_ARG, "dcm_import_state: NULL argument");
    const size_t need = (size_t)v->E.S.B * v->L.dyn_bytes;
    if (bytes != need) return fail(DCM_ERR_ARG, "dcm_import_state: size mismatch");
    DeviceGuard g(v->device);
    if (!v->d_record) { CK(cudaMalloc(&v->d_record, need)); }
    cudaStream_t s = (cudaStream_t)stream;
    CK(cudaMemcpyAsync(v->d_record, src, need, cudaMemcpyDefault, s));
    LAUNCH_TW(v, k_import, grid_env(v, 128), 128, 0, s, v->E, v->L, v->d_record);
    CK(cudaGetLastError());
    note_stream(v, s);
    v->launches++;
    return DCM_OK;
}

int dcm_layout(const dcm_env* v, int32_t* out, int n) {
    if (!v || !out) return 0;
    const DcmLayout& L = v->L;
    const int vals[] = {L.A, L.T, L.M, L.MC, L.Tp, L.Ap, L.o_arr, L.o_tstart, L.o_alast, L.o_and, L.o_adist, L.o_hdr, L.o_tnab, L.o_anab,
                        L.o_mem, L.o_nmem, L.o_status, L.o_tflags, L.o_anode, L.o_aflags, L.dyn_bytes,
                        L.s_tx, L.s_ty, L.s_dur, L.s_depot, L.s_req, L.sta_bytes, L.stage_bytes, 32};
    const int cnt = (int)(sizeof vals / sizeof vals[0]);
    for (int i = 0; i < n && i < cnt; ++i) out[i] = vals[i];
    return cnt < n ? cnt : n;
}

int dcm_total_steps(dcm_env* v, uint64_t* out) {
    if (!v || !out) return fail(DCM_ERR_ARG, "dcm_total_steps: NULL argument");
    DeviceGuard g(v->device);
    CK(cudaMemset(v->d_counter, 0, sizeof(unsigned long long)));
    k_sum_steps<<<v->sm_count, 256>>>(v->E, v->d_counter);
    CK(cudaGetLastError());
    v->launches++;
    unsigned long long h = 0;
    CK(cudaMemcpy(&h, v->d_counter, sizeof h, cudaMemcpyDeviceToHost));
    *out = h;
    return DCM_OK;
}

int dcm_total_episodes(dcm_env* v, uint64_t* out) {
    if (!v || !out) return fail(DCM_ERR_ARG, "dcm_total_episodes: NULL argument");
    DeviceGuard g(v->device);
    CK(cudaMemset(v->d_counter, 0, sizeof(unsigned long long)));
    k_sum_episodes<<<v->sm_count, 256>>>(v->E, v->d_counter);
    CK(cudaGetLastError());
    v->launches++;
    unsigned long long h = 0;
    CK(cudaMemcpy(&h, v->d_counter, sizeof h, cudaMemcpyDeviceToHost));
    *out = h;
    return DCM_OK;
}

size_t dcm_algorithmic_bytes_per_step(const dcm_env* v) {
    if (!v) return 0;
    const size_t A = v->E.S.A, T = v->E.S.T, M = v->E.S.M, w = 8;
    const size_t s_static = 2 * w * T + 2 * w + T + w * T;
    const size_t s_dyn = T * (M * (1 + w) + 2 * w + 5) + A * (3 * w + 4) + 40;
    const size_t s_obs = 4 * 6 * A + 4 * 5 * (T + 1) + (T + 1);
    return s_static + 2 * s_dyn + s_obs + 16;
}

uint64_t dcm_launch_count(const dcm_env* v) { return v ? v->launches : 0; }

int dcm_debug_pass_trace(dcm_env* v, uint64_t* out_h, size_t n_words) {
    if (!v || !out_h) return fail(DCM_ERR_ARG, "dcm_debug_pass_trace: NULL argument");
    if (!v->d_trace) return fail(DCM_ERR_STATE, "dcm_debug_pass_trace: create the handle with DCM_PASS_TRACE=1");
    DeviceGuard g(v->device);
    const size_t have = v->trace_units * 4;
    CK(cudaMemcpy(out_h, v->d_trace, (n_words < have ? n_words : have) * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    return DCM_OK;
}

}  // extern "C"
