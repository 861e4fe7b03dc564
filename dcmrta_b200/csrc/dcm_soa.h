// dcm_soa.h -- device-resident state of a batch of envs: tiled arrays + per-env bitmask summaries (v4).
//
// Execution model (chosen from the r01a..r01d profiles, see DESIGN.md): ONE THREAD OWNS ONE ENV in the step kernel,
// 32 consecutive envs form a TILE owned by one warp.
//
//  * Fields that a warp scans densely (one row for all 32 envs at once: next_decision, byte fields, masks) are stored
//    [tile][row][32 lanes]: lane l reads row k of ITS env at base[((tile*K + k) << 5) + l] -- one coalesced access.
//  * Fields that each env touches sparsely and differently (the few agents that moved, the few tasks that changed) are
//    stored per-lane-contiguous, [tile][row][32 lanes][W words], sized to 16/32-byte sectors, so that a sparse access
//    costs ONE sector: the agent record {last_arrival, x, y, travel_dist}, the task info pair, the member slots.
//  * Boolean state lives in 64-bit masks (one bit per task / agent) that a thread keeps in registers for the whole
//    step; loops run over set bits only, and only what changes is written back.
//
// Live fields are those of SURVEY.md App. A plus derived values that make the step cheap (t_fin, amin, a_ts); the
// per-env RECORD of dcm_layout.h remains the export / import / checkpoint format (k_export / k_import convert).
#pragma once
#include <stdint.h>

#include "dcm_layout.h"

#define DCM_MAX_TW 4     // 64-bit words per task mask (T <= 254)

struct DcmSoa {
    int B;        // envs
    int NT;       // tiles = ceil(B / 32)
    int A, T, M, MC, TW;
    int MCB;      // bytes reserved per (task, lane) for member ids: 8 (MC <= DCM_MAX_M = 8: one 64-bit word)
    int ANB;      // bytes reserved per env for the agents' node ids: 32 (A <= 32) or 64
    size_t tile_stride;   // bytes of one tile's block; every pointer below addresses tile 0, tile t is at + t * tile_stride
    // ---- per task, lane-contiguous ----
    double* t_slot_arr;        // [T][32][MC]   arrival of member slot s (last visit, task_env.py:202-205)
    double* t_rec;             // [T][32][8]    the task record (dcm_thread.cuh TREC): sector 0 {amin | time_start, amax | time_finish, member ids,
                               //               count | status | requirement | len(abandoned_agent)}, sector 1 {duration, x, y, -}
    // ---- per task, row-major (what the observation kernel streams) ----
    signed char* t_status;     // [T]    copy of the record's stored status (may be stale, Q3)
    // ---- task masks (rows: TW) ----
    unsigned long long* m_feas;    // feasible_assignment
    unsigned long long* m_fin;     // finished
    unsigned long long* m_ne;      // len(members) > 0
    unsigned long long* m_open;    // not feasible and status > 0  (== not masked, task_env.py:199)
    unsigned long long* m_dirty;   // len(members) changed since status was computed (join, or removal: Q3)
    // ---- per agent ----
    double* a_rec;             // [A][32][4]   {arrival_time[-1], x, y, travel_dist}   (one 32-byte sector)
    double* a_obs;             // [A][32][2]   observation cache: {time_start, time_finish} of the task the agent stands at if it is feasible,
                               //              else {0, 0 + time} -- the operands of task_env.py:170-171, kept current by agent_step and task_update
    double* a_nd;              // [A]   next_decision
    double* a_ts;              // [A]   time_start of the feasible task the agent is a member of (valid with the watch bit)
    unsigned char* a_node;     // [ANB/4][32 lanes][4]  route[-1] or DCM_NODE_DEPOT: four agents per word, words row-major (ANB = 32 for A <= 32, else 64)
    unsigned short* a_nab;     // [A]   entries in abandoned_agent lists
    // ---- agent masks (rows: 1) ----
    unsigned long long* am_route;     // len(route) > 0
    unsigned long long* am_assigned;
    unsigned long long* am_returned;
    unsigned long long* am_member;    // agent is in the member list of the task it stands at
    unsigned long long* am_depot;     // route[-1] == depot
    unsigned long long* am_touched;   // next_decision / assigned must be recomputed by the next agent_update
    unsigned long long* am_watch;     // member of a feasible task, not assigned yet: re-check `now >= time_start`
    // ---- per env (rows: 1) ----
    double* now;
    double* x_fin; double* x_amin; double* x_asg; double* x_ret;   // conservative lower bounds that let a step skip whole scans (dcm_thread.cuh St)
    double* x_last;            // max over the agents of max(arrival_time) (check_finished clock jump, task_env.py:286/369)
    unsigned long long* pending;
    unsigned long long* group;
    unsigned* n_steps; unsigned* episode; unsigned* flags; unsigned* instance; unsigned* total;
    int* leader;
    unsigned char* ended;     // 1 = the env's episode ended in the last step (its observation comes from the episode kernel, not from k_obs)
    // ---- static instance (rows: T, depot: 2) ----
    double* s_tx; double* s_ty; double* s_dur; double* s_dep;
    unsigned char* s_req;
    float* s_dur32;           // [T] fp32(time): the value the task rows of the observation carry (k_obs_tile copies it with the TMA engine)
    // ---- scratch ----
    double* w_agent;          // [A] per-agent waiting-time accumulator (thread-per-env episode accounting)
};

#ifdef __cplusplus
// bytes of one tile's part of an array with K rows per tile and `per_lane` bytes per (row, lane)
static inline size_t dcm_soa_bytes(int K, size_t per_lane) { return (size_t)K * 32 * per_lane; }
#endif
