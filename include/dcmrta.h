/*
 * include/dcmrta.h -- C ABI of libdcmrta_b200.so: the B200-native replacement of the reference's environment
 * step, marmotlab/DCMRTA  env/task_env.py  class TaskEnv (:8-623), as driven by worker.py:45-87.
 *
 * The reference has no FFI layer: its boundary is the Python class.  This header is what a ctypes / cffi binding
 * of that class binds (dcmrta_b200/_lib.py does, INTEGRATION.md shows the stub); each entry point cites the
 * reference method it replaces.
 *
 * Conventions
 *   - return 0 (DCM_OK) or a negative dcm_status; dcm_last_error() gives a thread-local message.
 *   - no C++ exceptions, no torch types: plain pointers and sizes.
 *   - pointers named *_d are DEVICE pointers on the handle's device; *_h are HOST pointers.
 *   - `stream` is a cudaStream_t passed as void* (torch.cuda.current_stream().cuda_stream); every call that takes
 *     one is asynchronous on it and performs no host synchronisation.  Calls taking host pointers synchronise.
 *   - a handle owns ALL state in HBM (allocated once in dcm_create), is bound to one device, and is not
 *     thread-safe; distinct handles are independent.
 *   - B envs, A agents (<= 64), T tasks (<= 254), M = max coalition size = member slots per task (<= 8).  Requirements
 *     must lie in [1, M].  Legal (unmasked) actions never put more than M agents on a task; preset routes can, so a
 *     handle used for dcm_execute_by_route should be created with M = the largest coalition the routes may form
 *     (DCM_ENV_ERR_OVERFLOW is raised per env otherwise).
 *   - actions use the reference encoding: 0 = depot, j+1 = task j (task_env.py:307).
 *   - there is NO CPU fallback: without a CUDA device every compute entry point returns DCM_ERR_DEVICE.
 */
#ifndef DCMRTA_H
#define DCMRTA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dcm_env dcm_env;

enum dcm_status {
    DCM_OK = 0,
    DCM_ERR_ARG = -1,      /* null pointer / value out of range */
    DCM_ERR_SHAPE = -2,    /* A, T, M, B outside the supported range */
    DCM_ERR_DEVICE = -3,   /* no such CUDA device / no CUDA driver */
    DCM_ERR_CUDA = -4,     /* a CUDA runtime call failed (message has the code) */
    DCM_ERR_STATE = -5,    /* call order violation (e.g. step before instances are loaded) */
    DCM_ERR_NOMEM = -6
};

/* dcm_create flags */
#define DCM_FLAG_AUTO_RESET  1u   /* an env that finishes inside dcm_step starts its next episode in the same call */
#define DCM_FLAG_REGENERATE  2u   /* ... on a freshly generated instance (needs dcm_generate to have set the distribution) */
/* Individual-agent decision protocol (worker.py:159-198 run_test_IS; RL_test.py METHOD = 'IA') instead of leader-follower
 * (worker.py:45-85): every decider of a slot acts alone, in ascending id order -- no location groups, no leader draw, no
 * followers.  One dcm_step call is then one INDIVIDUAL decision per env; the slot boundary (check_finished, next_decision,
 * task_update, agent_update) is unchanged.  The flag belongs to the handle: restarted episodes follow it too.  The contract
 * under this flag is stated at dcm_reset and dcm_step; the granular entry points and dcm_execute_by_route ignore it. */
#define DCM_FLAG_INDIVIDUAL  4u

/* built-in policies for dcm_step(policy=...) */
#define DCM_POLICY_EXTERNAL  0    /* action_d supplies the actions (the attention policy of attention.py) */
#define DCM_POLICY_RANDOM    1    /* uniform over unmasked actions, in-kernel Philox */
#define DCM_POLICY_GREEDY    2    /* nearest unmasked task, depot only when nothing is open */

/* per-env status bits (dcm_env_flags) */
#define DCM_ENV_DONE          1u  /* episode over: finished, or clock >= max_time (worker.py:45) */
#define DCM_ENV_FINISHED      2u  /* check_finished() was true (task_env.py:366-373) */
#define DCM_ENV_STUCK         4u  /* nobody can ever decide again and the episode is not finished: the reference loop would spin */
#define DCM_ENV_FIRST_SLOT    8u
#define DCM_ENV_ERR_OVERFLOW 16u  /* a task received more than M distinct members (only reachable with masked actions / preset routes) */
#define DCM_ENV_ERR_ACTION   32u  /* action outside [0, T] */
#define DCM_ENV_ERR_FOLLOW   64u  /* injected followers are not what step() could have drawn (task_env.py:331) */
#define DCM_ENV_ERR_LEADER  128u  /* injected leader is not in the current group (worker.py:54) */
#define DCM_ENV_ACCOUNTED   256u  /* the finished episode's metrics have been computed (dcm_episode_metrics has them) */
#define DCM_ENV_FRESH       512u  /* restarted by the last dcm_step (auto-reset); cleared by the next one */

/* ---- lifetime ------------------------------------------------------------------------------------------------ */

/* TaskEnv.__init__ (task_env.py:9-34) for B envs at once; allocates every byte of state in HBM. */
int dcm_create(dcm_env** out, int device, int B, int A, int T, int M, uint32_t flags);
int dcm_destroy(dcm_env* env);

/* agent velocity (task_env.py:99), max_waiting_time (:30 / RL_test.py:39), MAX_TIME (parameters.py:19). Defaults 0.2, 10, 100. */
int dcm_set_params(dcm_env* env, double velocity, double max_wait, double max_time);

/* Philox key and the global index of env 0 of this handle (shard-invariant streams: env k of the job always sees the
 * stream of global index first_gid + k, whatever GPU it lives on). */
int dcm_seed(dcm_env* env, uint64_t seed, uint64_t first_gid);

/* ---- instances ------------------------------------------------------------------------------------------------ */

/* TaskEnv.reset(test_env=...) (task_env.py:116-127): install B instances.
 * task_xy [B,T,2] f64, depot_xy [B,2] f64, req [B,T] i32 in [1,M], dur [B,T] f64.  Does not touch dynamic state. */
int dcm_load_instances(dcm_env* env, const double* task_xy_d, const double* depot_xy_d, const int32_t* req_d,
                       const double* dur_d, void* stream);
int dcm_load_instances_host(dcm_env* env, const double* task_xy_h, const double* depot_xy_h, const int32_t* req_h,
                            const double* dur_h);
/* generate_env (task_env.py:57-114) distributions, on device: depot, task xy ~ U[0,1)^2, req ~ U{1..M}, duration =
 * max_duration, or ~ U(0,max_duration) when random_duration != 0 (the bundled pickles).  Philox stream (seed, gid, instance#). */
int dcm_generate(dcm_env* env, double max_duration, int random_duration, void* stream);
/* read the installed instances back (same layouts as dcm_load_instances; any pointer may be NULL) */
int dcm_get_instances(dcm_env* env, double* task_xy_d, double* depot_xy_d, int32_t* req_d, double* dur_d, void* stream);

/* ---- fused path: one call == one leader decision for every env (worker.py:45-85) ------------------------------ */

/* clear_decisions (task_env.py:129-140) + first slot (worker.py:47-51) + first leader (worker.py:54) + observation of
 * that leader (worker.py:57-64).
 *   which_d        [B] u8, 1 = reset this env; NULL = all
 *   leader_in_d    [B] i32 leader to use (trace replay), NULL = Philox
 * outputs as for dcm_step (any may be NULL).
 * DCM_FLAG_INDIVIDUAL: the first agent to act is agent 0 and no random word is drawn; an injected leader other than 0 sets
 * DCM_ENV_ERR_LEADER and agent 0 acts (a negative entry injects nothing, as in leader-follower mode). */
int dcm_reset(dcm_env* env, const uint8_t* which_d, const int32_t* leader_in_d,
              float* agent_obs_d, float* task_obs_d, uint8_t* mask_d, int32_t* next_leader_d, void* stream);

/* TaskEnv.step (task_env.py:326-342) for the current leader, then task_update (:245-281), agent_update (:207-243), and,
 * when the slot's groups are exhausted, check_finished (:366-373), next_decision (:283-289), get_unique_group (:291-298),
 * task_update, agent_update; then leader choice, get_unfinished_task_mask (:192-200) + depot bit (worker.py:58-61),
 * get_current_agent_status (:165-180), get_current_task_status (:182-190) for the next leader, cast to fp32.
 *   action_d         [B] i32 (ignored when policy != DCM_POLICY_EXTERNAL)
 *   followers_d      [B, fstride] i32, -1 padded: the followers random_choice drew (task_env.py:331); NULL = Philox
 *   next_leader_in_d [B] i32 the leader np.random.choice(group) returned for the NEXT decision; NULL = Philox
 *   agent_obs_d [B,A,6] f32   task_obs_d [B,T+1,5] f32   mask_d [B,T+1] u8 (1 = forbidden)
 *   next_leader_d [B] i32 (-1 when done; with DCM_FLAG_AUTO_RESET the first leader of the restarted episode)
 *   reward_d [B] f32 (task_env.py:341)   done_d [B] u8
 *   used_action_d [B] i32 or NULL: the action that was applied (what a built-in policy chose; -1 if the env did not step)
 * Envs already done (and not auto-reset) are left untouched and report done=1.
 * DCM_FLAG_INDIVIDUAL (one call = one individual decision, worker.py:170-186):
 *   - exactly one agent moves, the current leader, whatever the stored group holds (also for the depot action);
 *   - next_leader is the lowest-id pending decider of the slot, or the first decider of the next slot; a restarted episode
 *     (DCM_FLAG_AUTO_RESET) starts with agent 0.  No random word is drawn for leaders or followers; the built-in random policy
 *     draws word 0 of block 0, as in leader-follower mode;
 *   - followers_d must be NULL or all -1 for an env that moves to a task: otherwise DCM_ENV_ERR_FOLLOW is set and the env does
 *     not step (as in leader-follower mode, the depot action ignores followers_d);
 *   - an injected next_leader_in_d entry >= 0 must be that agent: otherwise DCM_ENV_ERR_LEADER is set and that agent acts
 *     anyway (for a restart: agent 0);
 *   - reward is -travel_time of the one mover (task_env.py:315);
 *   - dcm_total_steps and the `decisions` metric count individual decisions. */
int dcm_step(dcm_env* env, const int32_t* action_d, const int32_t* followers_d, int fstride,
             const int32_t* next_leader_in_d, int policy,
             float* agent_obs_d, float* task_obs_d, uint8_t* mask_d,
             int32_t* next_leader_d, float* reward_d, uint8_t* done_d, int32_t* used_action_d, void* stream);

/* Same call with HOST buffers (pageable or pinned), under the same protocol as dcm_step (DCM_FLAG_INDIVIDUAL included: the next
 * leader is then the agent that acts next): actions are copied in -- or, from pinned memory, read in place by the step
 * kernel --, outputs copied out, the call returns when the outputs are valid.  Any output pointer may be NULL (then it is not copied).  next_leader, reward and done are final when the
 * step kernel ends and are copied on a second stream while the episode and observation kernels still run.  The call runs on a
 * stream of the handle; it first waits (on the device, through an event) for the asynchronous work earlier calls on this handle
 * queued on the caller's stream -- dcm_reset / dcm_generate / dcm_load_instances / dcm_step / granular calls -- so no host
 * synchronisation is needed between those and dcm_step_host. */
int dcm_step_host(dcm_env* env, const int32_t* action_h, int policy,
                  float* agent_obs_h, float* task_obs_h, uint8_t* mask_h,
                  int32_t* next_leader_h, float* reward_h, uint8_t* done_h);

/* get_episode_reward (task_env.py:420-425) + calculate_waiting_time (:344-364) + worker.py:103-108 for the episode that
 * last ended in each env: [B,8] f64 = reward(-makespan), success_rate, makespan, time_cost, waiting_time, travel_dist,
 * efficiency, decisions.  Rows of envs that never finished an episode are zero. */
int dcm_episode_metrics(dcm_env* env, double* out_d, void* stream);

/* ---- granular path: the individual TaskEnv methods, batched (used by the TaskEnv-compatible facade) ------------- */

/* next_decision (task_env.py:283-289): deciders_d [B] u64 bitmask (bit i = agent i), t_d [B] f64 */
int dcm_next_decision(dcm_env* env, uint64_t* deciders_d, double* t_d, void* stream);
/* get_unique_group (task_env.py:291-298): group_rank_d [B,A] i8 = index of the agent's location group in np.unique order, -1 if not a decider */
int dcm_unique_group(dcm_env* env, const uint64_t* deciders_d, int8_t* group_rank_d, void* stream);
/* env.current_time = t (worker.py:49); t_d NULL leaves the clock alone */
int dcm_set_clock(dcm_env* env, const double* t_d, void* stream);
int dcm_get_clock(dcm_env* env, double* t_d, void* stream);
/* task_update (task_env.py:245-281): newly_d [B,T] u8 (1 = became feasible in this call) or NULL */
int dcm_task_update(dcm_env* env, uint8_t* newly_d, void* stream);
/* agent_update (task_env.py:207-243) */
int dcm_agent_update(dcm_env* env, void* stream);
/* agent_step for members[b, 0..n_members[b]) in order with action[b] (task_env.py:300-324, 337-341): reward_d [B] f64 */
int dcm_apply_members(dcm_env* env, const int32_t* action_d, const int32_t* members_d, int mstride,
                      const int32_t* n_members_d, double* reward_d, void* stream);
/* mask + agent rows + task rows for leader_d[b] (task_env.py:165-200, worker.py:57-64) */
int dcm_build_obs(dcm_env* env, const int32_t* leader_d, float* agent_obs_d, float* task_obs_d, uint8_t* mask_d, void* stream);
/* check_finished (task_env.py:366-373), including its side effect on the clock: finished_d [B] u8 */
int dcm_check_finished(dcm_env* env, uint8_t* finished_d, void* stream);
/* get_episode_reward + metrics computed NOW for every env (same row layout as dcm_episode_metrics); optionally also the
 * per-element sums calculate_waiting_time leaves in the dicts: task_wait_d [B,T], agent_wait_d [B,A] f64 (or NULL) */
int dcm_compute_metrics(dcm_env* env, double* out_d, double* task_wait_d, double* agent_wait_d, void* stream);
/* pre_set_route + execute_by_route (task_env.py:562-599): routes_d [B,A,rstride] i32 actions (0 = depot), route_len_d [B,A];
 * runs every env to completion in one launch with max_waiting_time = 100 and the 200 clock cap; makespan_d [B] f64.
 *   - agent a plays the first min(route_len, rstride) entries of its row, then goes to the depot; an entry above rstride sets
 *     DCM_ENV_ERR_ACTION on its env (route_len_d is device memory, so only the kernel can check it).  rstride <= 255;
 *   - an entry outside [0, T] sets DCM_ENV_ERR_ACTION and is played as the depot;
 *   - routes can leave a task unfinished once every agent is home (an agent at the depot never decides again): the reference
 *     loop then spins forever.  The env stops after two consecutive passes in which nobody decides, with DCM_ENV_STUCK,
 *     as dcm_step does.  Every env ends with DCM_ENV_DONE, and DCM_ENV_FINISHED if check_finished was true. */
int dcm_execute_by_route(dcm_env* env, const int32_t* routes_d, int rstride, const int32_t* route_len_d,
                         double* makespan_d, void* stream);

/* ---- inspection ------------------------------------------------------------------------------------------------ */

/* raw dynamic records, [B, dcm_record_bytes] (parity / debug / checkpoint).  dst may be host or device memory. */
size_t dcm_record_bytes(const dcm_env* env);
int dcm_export_state(dcm_env* env, void* dst, size_t bytes, void* stream);
int dcm_import_state(dcm_env* env, const void* src, size_t bytes, void* stream);
/* byte offsets of the record fields: out[0..n) as documented in DESIGN.md "record layout"; returns the count written */
int dcm_layout(const dcm_env* env, int32_t* out, int n);
/* per-env status bits, [B] u32.
 * The DCM_ENV_ERR_* bits stay set for the rest of the episode: later legal steps do not clear them.  dcm_reset and an auto-reset
 * restart clear them; a restart whose injected first leader is >= A sets DCM_ENV_ERR_LEADER for the new episode.
 *   - DCM_ENV_ERR_ACTION, DCM_ENV_ERR_FOLLOW: dcm_step refuses the decision.  The env's record is unchanged except this word, the
 *     outputs are reward 0, used_action -1, done 0, the next leader and observation of the unchanged state, and dcm_total_steps does
 *     not count it.  The env may continue with a legal input.
 *   - DCM_ENV_ERR_LEADER: the decision is applied; the lowest id of the group leads next (agent 0 at a restart).
 *   - DCM_ENV_ERR_OVERFLOW: the agent moved to the full task but is not one of its members.
 * An env that is done and not restarted sets no bit, whatever it is given. */
int dcm_env_flags(dcm_env* env, uint32_t* flags_d, void* stream);
/* total leader decisions applied by this handle since creation (device counter read back; synchronises) */
int dcm_total_steps(dcm_env* env, uint64_t* out_h);
/* episodes accounted by this handle since creation, summed over its envs (worker.py:87 runs once per episode; device counters
 * read back; synchronises).  bench.py reports the episode-end rate of the timed passes from it. */
int dcm_total_episodes(dcm_env* env, uint64_t* out_h);
/* algorithmic HBM bytes per env-step for this handle's shape (SURVEY.md 8(d) formula, w = 8) */
size_t dcm_algorithmic_bytes_per_step(const dcm_env* env);
/* number of kernels this handle has launched since creation */
uint64_t dcm_launch_count(const dcm_env* env);

/* developer aid: with DCM_PASS_TRACE=1 in the environment at dcm_create, every k_obs_tile block and every k_episode_list warp of the
 * last dcm_step stamps %globaltimer / %smid: 8 words per observation tile, then 4 per episode warp (tools/obs_trace.py; synchronises) */
int dcm_debug_pass_trace(dcm_env* env, uint64_t* out_h, size_t n_words);

const char* dcm_last_error(void);
const char* dcm_version(void);

#ifdef __cplusplus
}
#endif
#endif /* DCMRTA_H */
