/*
 * oracle/taskenv_oracle.c  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * A scalar, single-env, fp64 CPU restatement of the reference simulator
 * marmotlab/DCMRTA  env/task_env.py  (class TaskEnv) and of the rollout loop
 * in worker.py:45-87 that drives it.  It exists only so that tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
 * can check (and time) the CUDA path against an independent implementation.
 * Nothing under dcmrta_b200/ may import, link or call this file.
 *
 * Parity status: PINNED.  tests/test_oracle_golden.py checks this file against
 *   (i)  the reference's own known-answer file testSet_20A_50T_CONDET/CTAS-D_300s.csv
 *        (CTAS-D routes through execute_by_route, 50 instances), and
 *   (ii) per-step digests + full dumps recorded from the *real* Python reference
 *        in the build container by oracle/make_golden.py (tests/golden/).
 *
 * The restatement deliberately keeps the reference's data model (per-agent
 * route / arrival_time lists that are scanned for the last visit, ordered
 * member lists, abandoned lists) instead of the compact record the GPU uses,
 * so that the two implementations share no design.
 *
 * Every function cites the reference lines it follows (paths relative to the
 * reference root).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <stdio.h>

#define ORC_MAX_AGENTS 64

typedef struct {
    int *v; int n, cap;
} ilist;
typedef struct {
    double *v; int n, cap;
} dlist;

static void il_push(ilist *l, int x) {
    if (l->n == l->cap) { l->cap = l->cap ? 2 * l->cap : 8; l->v = (int *)realloc(l->v, sizeof(int) * l->cap); }
    l->v[l->n++] = x;
}
static void dl_push(dlist *l, double x) {
    if (l->n == l->cap) { l->cap = l->cap ? 2 * l->cap : 8; l->v = (double *)realloc(l->v, sizeof(double) * l->cap); }
    l->v[l->n++] = x;
}
static int il_index(const ilist *l, int x) { for (int i = 0; i < l->n; i++) if (l->v[i] == x) return i; return -1; }
static void il_remove(ilist *l, int x) {          /* python list.remove: first occurrence */
    int i = il_index(l, x);
    if (i < 0) return;
    memmove(l->v + i, l->v + i + 1, sizeof(int) * (l->n - i - 1));
    l->n--;
}
static int il_pop_front(ilist *l) { int x = l->v[0]; memmove(l->v, l->v + 1, sizeof(int) * (l->n - 1)); l->n--; return x; }

typedef struct {
    /* task_dic[j]  (task_env.py:76-89) */
    double x, y;            /* 'location'     */
    int    req;             /* 'requirements' */
    double time;            /* 'time'         */
    ilist  members;         /* 'members' (ordered) */
    ilist  abandoned;       /* 'abandoned_agent'   */
    int    status;          /* 'status' (stored, may be stale) */
    int    feasible;        /* 'feasible_assignment' */
    int    finished;        /* 'finished' */
    double time_start, time_finish;
    double sum_waiting_time;
} orc_task;

typedef struct {
    /* agent_dic[i]  (task_env.py:91-110) */
    double x, y;            /* 'location' */
    ilist  route;           /* 'route'  (task ids, -1 = depot) */
    dlist  arrival;         /* 'arrival_time' */
    double travel_time, travel_dist, velocity;
    double next_decision;   /* 0 initially, NaN after choosing the depot */
    double sum_waiting_time;
    int    assigned, returned;
    int    has_preset; ilist preset;   /* 'pre_set_route' */
} orc_agent;

typedef struct orc_env {
    int A, T;
    double depot_x, depot_y;
    ilist depot_members;
    orc_task  *task;
    orc_agent *agent;
    double now;             /* current_time */
    int    finished;
    double W;               /* max_waiting_time */
    double max_time;        /* MAX_TIME of worker.py (parameters.py:19) */
    /* ---- fused-driver state (worker.py:45-85 folded into one call per decision) ---- */
    uint64_t pending;       /* deciders of the current slot that have not acted yet */
    int    leader;          /* current leader (-1 when done) */
    int    done;            /* episode over (finished or time cap) */
    int    stuck;           /* the reference loop would spin forever here (see orc_advance) */
    int    first_slot;
    long   n_steps;         /* leader decisions applied in this episode */
    /* ---- Philox stream for the synthetic policies ---- */
    uint64_t seed; uint64_t gid; uint32_t episode;
} orc_env;

/* ------------------------------------------------------------------ */
/*  construction / reset                                               */
/* ------------------------------------------------------------------ */

/* task_env.py:129-140 clear_decisions (after reset :116-127 installed the instance) */
void orc_clear_decisions(orc_env *e) {
    for (int j = 0; j < e->T; j++) {
        orc_task *t = &e->task[j];
        t->members.n = 0; t->abandoned.n = 0;
        t->finished = 0; t->status = t->req; t->feasible = 0;
        t->time_start = 0; t->time_finish = 0; t->sum_waiting_time = 0;
    }
    for (int i = 0; i < e->A; i++) {
        orc_agent *a = &e->agent[i];
        a->route.n = 0; a->arrival.n = 0;
        a->x = e->depot_x; a->y = e->depot_y;
        a->next_decision = 0; a->travel_time = 0; a->travel_dist = 0;
        a->assigned = 0; a->sum_waiting_time = 0; a->returned = 0;
        a->has_preset = 0; a->preset.n = 0;
    }
    e->depot_members.n = 0;
    e->now = 0; e->finished = 0;
    e->pending = 0; e->leader = -1; e->done = 0; e->stuck = 0; e->first_slot = 1; e->n_steps = 0;
}

/* task_env.py:9-34 + :57-114: the instance is supplied by the caller (pickle / generator) */
orc_env *orc_create(int A, int T, const double *task_xy, const double *depot_xy, const int *req,
                    const double *dur, double velocity, double max_wait, double max_time) {
    if (A < 1 || A > ORC_MAX_AGENTS || T < 1) return NULL;
    orc_env *e = (orc_env *)calloc(1, sizeof(orc_env));
    e->A = A; e->T = T; e->W = max_wait; e->max_time = max_time;
    e->depot_x = depot_xy[0]; e->depot_y = depot_xy[1];
    e->task = (orc_task *)calloc(T, sizeof(orc_task));
    e->agent = (orc_agent *)calloc(A, sizeof(orc_agent));
    for (int j = 0; j < T; j++) {
        e->task[j].x = task_xy[2 * j]; e->task[j].y = task_xy[2 * j + 1];
        e->task[j].req = req[j]; e->task[j].time = dur[j];
    }
    for (int i = 0; i < A; i++) e->agent[i].velocity = velocity;
    orc_clear_decisions(e);
    return e;
}

void orc_destroy(orc_env *e) {
    if (!e) return;
    for (int j = 0; j < e->T; j++) { free(e->task[j].members.v); free(e->task[j].abandoned.v); }
    for (int i = 0; i < e->A; i++) { free(e->agent[i].route.v); free(e->agent[i].arrival.v); free(e->agent[i].preset.v); }
    free(e->depot_members.v); free(e->task); free(e->agent); free(e);
}

void orc_set_max_wait(orc_env *e, double w) { e->W = w; }
void orc_set_now(orc_env *e, double t) { e->now = t; }      /* worker.py:49 writes env.current_time */
double orc_get_now(const orc_env *e) { return e->now; }
void orc_set_finished(orc_env *e, int f) { e->finished = f; }

/* ------------------------------------------------------------------ */
/*  helpers                                                            */
/* ------------------------------------------------------------------ */

/* task_env.py:202-205 get_arrival_time: arrival of the agent's LAST visit to task_id */
static double get_arrival_time(const orc_env *e, int agent, int task_id) {
    const orc_agent *a = &e->agent[agent];
    for (int k = a->route.n - 1; k >= 0; k--) if (a->route.v[k] == task_id) return a->arrival.v[k];
    return NAN; /* the reference would raise IndexError; never reached on legal paths */
}

/* task_env.py:162-163: np.linalg.norm(a - b) on a 2-vector.  NumPy evaluates it as
 * sqrt(dot(d,d)); on the reference build (OpenBLAS ddot, FMA kernels) that is
 * sqrt(fma(dy,dy, dx*dx)) -- verified by oracle/make_golden.py on every distance it records. */
static double euclid(double ax, double ay, double bx, double by) {
    double dx = ax - bx, dy = ay - by;
    return sqrt(fma(dy, dy, dx * dx));
}

/* numpy add.reduce on a contiguous float64 vector (pairwise summation, blocks of 128, 8 lanes) */
static double np_sum(const double *a, int n) {
    if (n < 8) { double r = 0.; for (int i = 0; i < n; i++) r += a[i]; return r; }
    if (n <= 128) {
        double r[8]; int i;
        for (int k = 0; k < 8; k++) r[k] = a[k];
        for (i = 8; i < n - (n % 8); i += 8) for (int k = 0; k < 8; k++) r[k] += a[i + k];
        double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
        for (; i < n; i++) res += a[i];
        return res;
    }
    int n2 = n / 2; n2 -= n2 % 8;
    return np_sum(a, n2) + np_sum(a + n2, n - n2);
}

static int all_feasible(const orc_env *e) { for (int j = 0; j < e->T; j++) if (!e->task[j].feasible) return 0; return 1; }

/* ------------------------------------------------------------------ */
/*  simulator core                                                     */
/* ------------------------------------------------------------------ */

/* task_env.py:283-289 next_decision.  Returns number of deciders (ascending ids in ids[]). */
int orc_next_decision(const orc_env *e, int *ids, double *t_out) {
    int all_nan = 1; double mn = 0;
    for (int i = 0; i < e->A; i++) {
        double nd = e->agent[i].next_decision;
        if (!isnan(nd)) { if (all_nan || nd < mn) mn = nd; all_nan = 0; }
    }
    if (all_nan) {                       /* :285-286  max over agents of max(arrival_time) (0 if never moved) */
        double mx = 0; int first = 1;
        for (int i = 0; i < e->A; i++) {
            double m = 0;
            const dlist *ar = &e->agent[i].arrival;
            for (int k = 0; k < ar->n; k++) if (k == 0 || ar->v[k] > m) m = ar->v[k];
            if (first || m > mx) mx = m;
            first = 0;
        }
        *t_out = mx; return 0;
    }
    int n = 0;
    for (int i = 0; i < e->A; i++) if (e->agent[i].next_decision == mn) ids[n++] = i;   /* :288 exact equality */
    *t_out = mn; return n;
}

/* task_env.py:291-298 get_unique_group: partition by exact location; np.unique(axis=0) orders the
 * locations lexicographically (x, then y); ids ascending inside a group.
 * out_ids: deciders re-ordered group by group; out_sizes: size of each group.  Returns #groups. */
int orc_get_unique_group(const orc_env *e, const int *ids, int n, int *out_ids, int *out_sizes) {
    int used[ORC_MAX_AGENTS] = {0}; int ng = 0, w = 0;
    for (;;) {
        int best = -1;
        for (int k = 0; k < n; k++) {
            if (used[k]) continue;
            const orc_agent *a = &e->agent[ids[k]];
            if (best < 0) { best = k; continue; }
            const orc_agent *b = &e->agent[ids[best]];
            if (a->x < b->x || (a->x == b->x && a->y < b->y)) best = k;
        }
        if (best < 0) break;
        const orc_agent *b = &e->agent[ids[best]];
        int sz = 0;
        for (int k = 0; k < n; k++) {
            const orc_agent *a = &e->agent[ids[k]];
            if (!used[k] && a->x == b->x && a->y == b->y) { used[k] = 1; out_ids[w++] = ids[k]; sz++; }
        }
        out_sizes[ng++] = sz;
    }
    return ng;
}

/* task_env.py:245-281 task_update.  newly[] receives ids that became feasible (return value f). */
int orc_task_update(orc_env *e, int *newly) {
    int nf = 0;
    double arr[ORC_MAX_AGENTS];
    for (int j = 0; j < e->T; j++) {
        orc_task *t = &e->task[j];
        if (!t->feasible) {                                                   /* :249 */
            int abilities = t->members.n;                                     /* :250 */
            for (int k = 0; k < abilities; k++) arr[k] = get_arrival_time(e, t->members.v[k], j);   /* :251 */
            t->status = t->req - abilities;                                   /* :252 (not refreshed after removals) */
            if (t->status <= 0) {                                             /* :254 */
                double mx = arr[0], mn = arr[0];
                for (int k = 1; k < abilities; k++) { if (arr[k] > mx) mx = arr[k]; if (arr[k] < mn) mn = arr[k]; }
                if (mx - mn <= e->W) {                                        /* :255 */
                    t->time_start = mx;                                       /* :256 */
                    t->time_finish = mx + t->time;                            /* :257 */
                    t->feasible = 1;                                          /* :258 */
                    if (newly) newly[nf] = j;
                    nf++;
                } else {                                                      /* :260-265: iterate a COPY */
                    int snap[ORC_MAX_AGENTS]; int ns = 0;
                    double thr = mx - e->W;
                    for (int k = 0; k < abilities; k++) if (arr[k] <= thr) snap[ns++] = t->members.v[k];
                    for (int k = 0; k < ns; k++) { il_remove(&t->members, snap[k]); il_push(&t->abandoned, snap[k]); }
                }
            } else {                                                          /* :266-271: mutate while iterating */
                int i = 0;
                while (i < t->members.n) {
                    int m = t->members.v[i]; i++;
                    if (e->now - get_arrival_time(e, m, j) >= e->W) {         /* :269 */
                        il_remove(&t->members, m);                            /* next element is skipped */
                        il_push(&t->abandoned, m);
                    }
                }
            }
        } else if (e->now >= t->time_finish) {                                /* :273-274 */
            t->finished = 1;
        }
    }
    /* :277-280 depot */
    int allf = all_feasible(e);
    for (int k = 0; k < e->depot_members.n; k++) {
        int m = e->depot_members.v[k];
        if (e->now >= get_arrival_time(e, m, -1) && allf) e->agent[m].returned = 1;
    }
    return nf;
}

/* task_env.py:207-243 agent_update (reactive_planning == False branch, RL_test.py:40) */
void orc_agent_update(orc_env *e) {
    for (int i = 0; i < e->A; i++) {
        orc_agent *a = &e->agent[i];
        if (a->arrival.n == 0) continue;                                      /* :209 / :242 */
        int last = a->route.v[a->route.n - 1];
        if (last == -1) { a->next_decision = NAN; continue; }                 /* :212, :226 */
        orc_task *t = &e->task[last];
        if (t->feasible) {                                                    /* :229 */
            if (il_index(&t->members, i) >= 0) {                              /* :230 */
                a->next_decision = t->time_finish;                            /* :231 */
                if (e->now >= t->time_start) a->assigned = 1;                 /* :232-233 (sticky otherwise) */
            } else {
                a->next_decision = get_arrival_time(e, i, last) + e->W;       /* :235 */
                a->assigned = 0;
            }
        } else {
            a->next_decision = get_arrival_time(e, i, last) + e->W;           /* :238 */
            a->assigned = 0;
        }
    }
}

/* task_env.py:300-324 agent_step.  action: 0 = depot, j+1 = task j.  Returns -travel_time. */
double orc_agent_step(orc_env *e, int agent, int action) {
    int task_id = action - 1;
    orc_agent *a = &e->agent[agent];
    double tx, ty; ilist *mem;
    if (task_id != -1) { tx = e->task[task_id].x; ty = e->task[task_id].y; mem = &e->task[task_id].members; }
    else               { tx = e->depot_x; ty = e->depot_y; mem = &e->depot_members; }
    il_push(&a->route, task_id);                                              /* :314 */
    double d = euclid(a->x, a->y, tx, ty);
    double travel_time = d / a->velocity;                                     /* :315 */
    a->travel_time = travel_time;
    a->travel_dist += d;                                                      /* :317 */
    dl_push(&a->arrival, e->now + travel_time);                               /* :318 */
    a->x = tx; a->y = ty;                                                     /* :320 */
    if (il_index(mem, agent) < 0) il_push(mem, agent);                        /* :321-322 */
    return -travel_time;
}

/* task_env.py:327: vacancy seen by step() */
int orc_vacancy(const orc_env *e, int action, int group_len) {
    int tid = action - 1;
    return (tid >= 0 && tid < e->T) ? e->task[tid].status : group_len;
}

/* task_env.py:337-342: the deterministic tail of step() once members = [leader] + followers is known */
double orc_step_members(orc_env *e, const int *members, int n, int action) {
    double reward = 0;
    for (int k = 0; k < n; k++) reward += orc_agent_step(e, members[k], action);
    return reward / n;
}

/* task_env.py:192-200 get_unfinished_task_mask + worker.py:58-61 depot bit.  mask[T+1], 1 = forbidden */
void orc_mask(const orc_env *e, uint8_t *mask) {
    int sum = 0;
    for (int j = 0; j < e->T; j++) {
        int unfinished = (!e->task[j].feasible) && (e->task[j].status > 0);
        mask[1 + j] = !unfinished; sum += !unfinished;
    }
    mask[0] = (sum == e->T) ? 0 : 1;
}

static double clip0(double v) { return v < 0 ? 0 : v; }   /* np.clip(v, a_min=0, a_max=None) */

/* task_env.py:165-180 get_current_agent_status(agent=leader) -> [A,6] fp64 */
void orc_agent_status(const orc_env *e, int leader, double *out) {
    const orc_agent *L = &e->agent[leader];
    for (int i = 0; i < e->A; i++) {
        const orc_agent *a = &e->agent[i];
        double travel = 0, wait = 0, remain = 0;
        if (a->route.n > 0 && a->route.v[a->route.n - 1] >= 0) {              /* :168 */
            int k = a->route.v[a->route.n - 1];
            double arr = get_arrival_time(e, i, k);
            const orc_task *t = &e->task[k];
            travel = clip0(arr - e->now);                                     /* :169 */
            wait   = (e->now <= t->time_start) ? clip0(e->now - arr) : 0;     /* :170 */
            remain = (e->now >= t->time_start) ? clip0(t->time_start + t->time - e->now) : 0;   /* :171 */
        }
        double *r = out + 6 * i;
        r[0] = travel; r[1] = remain; r[2] = wait;                            /* :176 order */
        r[3] = L->x - a->x; r[4] = L->y - a->y; r[5] = a->assigned ? 1.0 : 0.0;
    }
}

/* task_env.py:182-190 get_current_task_status(agent=leader) -> [T+1,5] fp64 */
void orc_task_status(const orc_env *e, int leader, double *out) {
    const orc_agent *L = &e->agent[leader];
    out[0] = 0; out[1] = 0; out[2] = 0; out[3] = e->depot_x - L->x; out[4] = e->depot_y - L->y;   /* :188 */
    for (int j = 0; j < e->T; j++) {
        const orc_task *t = &e->task[j];
        double *r = out + 5 * (j + 1);
        r[0] = t->status; r[1] = t->req; r[2] = t->time; r[3] = t->x - L->x; r[4] = t->y - L->y;   /* :185-186 */
    }
}

/* task_env.py:366-373 check_finished (side effect on the clock when nobody can decide) */
int orc_check_finished(orc_env *e) {
    int ids[ORC_MAX_AGENTS]; double t;
    int n = orc_next_decision(e, ids, &t);
    if (n == 0) {
        e->now = t;
        for (int i = 0; i < e->A; i++) if (!e->agent[i].returned) return 0;
        for (int j = 0; j < e->T; j++) if (!e->task[j].finished) return 0;
        return 1;
    }
    return 0;
}

/* task_env.py:344-364 calculate_waiting_time */
void orc_calculate_waiting_time(orc_env *e) {
    double arr[ORC_MAX_AGENTS], tmp[ORC_MAX_AGENTS];
    for (int i = 0; i < e->A; i++) e->agent[i].sum_waiting_time = 0;
    for (int j = 0; j < e->T; j++) {
        orc_task *t = &e->task[j];
        int n = t->members.n;
        double mx = 0;
        for (int k = 0; k < n; k++) { arr[k] = get_arrival_time(e, t->members.v[k], j); if (k == 0 || arr[k] > mx) mx = arr[k]; }
        if (n != 0) {
            if (t->feasible) { for (int k = 0; k < n; k++) tmp[k] = mx - arr[k]; }          /* :351 */
            else             { for (int k = 0; k < n; k++) tmp[k] = e->now - arr[k]; }      /* :354 */
            t->sum_waiting_time = np_sum(tmp, n) + t->abandoned.n * e->W;
        } else {
            t->sum_waiting_time = t->abandoned.n * e->W;                                     /* :357 */
        }
        for (int k = 0; k < n; k++) {
            orc_agent *a = &e->agent[t->members.v[k]];
            if (t->feasible) a->sum_waiting_time += mx - arr[k];                             /* :360 */
            else a->sum_waiting_time += (e->now - arr[k] > 0) ? (e->now - arr[k]) : 0;       /* :362 */
        }
        for (int k = 0; k < t->abandoned.n; k++) e->agent[t->abandoned.v[k]].sum_waiting_time += e->W;   /* :363-364 */
    }
}

/* task_env.py:420-425 get_episode_reward + worker.py:103-108 perf_metrics.
 * out[8] = reward, success_rate, makespan, time_cost(nanmean time_start), waiting_time, travel_dist, efficiency, n_steps */
void orc_episode_metrics(orc_env *e, double *out, uint8_t *finished_tasks) {
    orc_calculate_waiting_time(e);
    (void)orc_check_finished(e);
    double buf[1024]; double *b = buf, *heap = NULL;
    int nmax = e->T > e->A ? e->T : e->A;
    if (nmax > 1024) b = heap = (double *)malloc(sizeof(double) * nmax);
    int nfin = 0;
    for (int j = 0; j < e->T; j++) { nfin += e->task[j].finished; if (finished_tasks) finished_tasks[j] = (uint8_t)e->task[j].finished; }
    out[0] = -e->now;
    out[1] = (double)nfin / (double)e->T;
    out[2] = e->now;
    for (int j = 0; j < e->T; j++) b[j] = e->task[j].time_start;
    out[3] = np_sum(b, e->T) / (double)e->T;
    for (int i = 0; i < e->A; i++) b[i] = e->agent[i].sum_waiting_time;
    out[4] = np_sum(b, e->A) / (double)e->A;
    for (int i = 0; i < e->A; i++) b[i] = e->agent[i].travel_dist;
    out[5] = np_sum(b, e->A);
    for (int j = 0; j < e->T; j++) b[j] = e->task[j].sum_waiting_time;
    out[6] = np_sum(b, e->T) / (double)e->T;
    out[7] = (double)e->n_steps;
    free(heap);
}

/* task_env.py:595-599 pre_set_route */
void orc_pre_set_route(orc_env *e, int agent, const int *route, int n) {
    orc_agent *a = &e->agent[agent];
    a->has_preset = 1;
    for (int k = 0; k < n; k++) il_push(&a->preset, route[k]);
}

/* task_env.py:562-593 execute_by_route (reactive_planning False).  Returns makespan. */
double orc_execute_by_route(orc_env *e) {
    int ids[ORC_MAX_AGENTS]; double t;
    int empty = 0;
    e->W = 100;                                                               /* :564 */
    while (!e->finished && e->now < 200) {                                    /* :565 */
        int n = orc_next_decision(e, ids, &t);                                /* :568 */
        e->now = t;
        orc_task_update(e, NULL); orc_agent_update(e);
        for (int k = 0; k < n; k++) {                                         /* :572 */
            orc_agent *a = &e->agent[ids[k]];
            int act = (!a->has_preset || a->preset.n == 0) ? 0 : il_pop_front(&a->preset);   /* :573-574, :585 */
            orc_agent_step(e, ids[k], act);
            orc_task_update(e, NULL); orc_agent_update(e);
        }
        e->finished = orc_check_finished(e);                                  /* :588 */
        /* Nobody decided in this pass nor in the one before.  An agent at the depot never decides again, so nobody ever will and the
         * reference `while` spins forever (routes that leave a task unfinished).  Stop and flag it, as orc_advance does. */
        empty = n ? 0 : empty + 1;
        if (!e->finished && empty >= 2) { e->stuck = 1; break; }
    }
    return e->now;
}

/* ------------------------------------------------------------------ */
/*  flat state export (same canonical form the GPU export is decoded to) */
/* ------------------------------------------------------------------ */
void orc_export(const orc_env *e, int MC,
                int32_t *n_mem, int32_t *members /*[T,MC] -1 pad*/, double *mem_arr /*[T,MC]*/,
                int32_t *status, uint8_t *feasible, uint8_t *finished, double *time_start, double *time_finish,
                int32_t *n_aband_task,
                int32_t *node, uint8_t *has_route, double *last_arrival, double *next_decision, double *travel_dist,
                uint8_t *assigned, uint8_t *returned, int32_t *n_aband_agent, double *now_finished /*[2]*/) {
    for (int i = 0; i < e->A; i++) n_aband_agent[i] = 0;
    for (int j = 0; j < e->T; j++) {
        const orc_task *t = &e->task[j];
        n_mem[j] = t->members.n;
        for (int k = 0; k < MC; k++) {
            if (k < t->members.n) { members[j * MC + k] = t->members.v[k]; mem_arr[j * MC + k] = get_arrival_time(e, t->members.v[k], j); }
            else { members[j * MC + k] = -1; mem_arr[j * MC + k] = 0; }
        }
        status[j] = t->status; feasible[j] = (uint8_t)t->feasible; finished[j] = (uint8_t)t->finished;
        time_start[j] = t->time_start; time_finish[j] = t->time_finish;
        n_aband_task[j] = t->abandoned.n;
        for (int k = 0; k < t->abandoned.n; k++) n_aband_agent[t->abandoned.v[k]]++;
    }
    for (int i = 0; i < e->A; i++) {
        const orc_agent *a = &e->agent[i];
        has_route[i] = a->route.n > 0;
        node[i] = a->route.n > 0 ? a->route.v[a->route.n - 1] : -1;
        last_arrival[i] = a->arrival.n > 0 ? a->arrival.v[a->arrival.n - 1] : 0;
        next_decision[i] = a->next_decision; travel_dist[i] = a->travel_dist;
        assigned[i] = (uint8_t)a->assigned; returned[i] = (uint8_t)a->returned;
    }
    now_finished[0] = e->now; now_finished[1] = e->finished;
}

int orc_route_len(const orc_env *e, int agent) { return e->agent[agent].route.n; }
void orc_route(const orc_env *e, int agent, int32_t *route, double *arrival) {
    for (int k = 0; k < e->agent[agent].route.n; k++) { route[k] = e->agent[agent].route.v[k]; arrival[k] = e->agent[agent].arrival.v[k]; }
}
void orc_agent_scalars(const orc_env *e, double *sum_wait /*[A]*/, double *task_sum_wait /*[T]*/) {
    for (int i = 0; i < e->A; i++) sum_wait[i] = e->agent[i].sum_waiting_time;
    for (int j = 0; j < e->T; j++) task_sum_wait[j] = e->task[j].sum_waiting_time;
}

/* ------------------------------------------------------------------ */
/*  Philox4x32-10 (Salmon et al., SC'11) -- own implementation, KAT-checked in tests */
/* ------------------------------------------------------------------ */
static void philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
    uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3], k0 = key[0], k1 = key[1];
    for (int r = 0; r < 10; r++) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
void orc_philox(const uint32_t *ctr, const uint32_t *key, uint32_t *out) { philox4x32_10(ctr, key, out); }
double orc_np_sum(const double *a, int n) { return np_sum(a, n); }

/* Random stream contract shared with the CUDA path (DESIGN.md "RNG contract"):
 *   key  = (seed_lo, seed_hi)
 *   ctr  = (global_env_id_lo, global_env_id_hi, episode, decision_index*8 + block), block < 8
 *   block 0 words: [0] action draw  [1] next-leader draw  [2],[3] follower draws 0,1
 *   block 1 words: follower draws 2..5 ; block 2: 6..9 ...
 *   uniform integer in [0,n): (uint64)word * n >> 32
 */
static uint32_t draw(const orc_env *e, uint32_t decision, int slot) {
    uint32_t ctr[4] = {(uint32_t)e->gid, (uint32_t)(e->gid >> 32), e->episode, decision * 8u + (uint32_t)(slot >> 2)};
    uint32_t key[2] = {(uint32_t)e->seed, (uint32_t)(e->seed >> 32)};
    uint32_t out[4]; philox4x32_10(ctr, key, out);
    return out[slot & 3];
}
static int pick(uint32_t word, int n) { return (int)(((uint64_t)word * (uint64_t)n) >> 32); }

void orc_seed(orc_env *e, uint64_t seed, uint64_t gid, uint32_t episode) { e->seed = seed; e->gid = gid; e->episode = episode; }

/* ------------------------------------------------------------------ */
/*  fused driver: one call == one leader decision (worker.py:45-85)    */
/* ------------------------------------------------------------------ */

/* members of `pending` standing at the lexicographically smallest location (np.unique order, :293) */
static uint64_t current_group(const orc_env *e, uint64_t pending) {
    int best = -1;
    for (int i = 0; i < e->A; i++) if (pending >> i & 1) {
        if (best < 0) { best = i; continue; }
        const orc_agent *a = &e->agent[i], *b = &e->agent[best];
        if (a->x < b->x || (a->x == b->x && a->y < b->y)) best = i;
    }
    uint64_t g = 0;
    if (best < 0) return 0;
    for (int i = 0; i < e->A; i++) if ((pending >> i & 1) && e->agent[i].x == e->agent[best].x && e->agent[i].y == e->agent[best].y) g |= 1ull << i;
    return g;
}
static int popcnt(uint64_t m) { return __builtin_popcountll(m); }
static int kth_bit(uint64_t m, int k) { for (int i = 0; i < 64; i++) if (m >> i & 1) { if (k == 0) return i; k--; } return -1; }

/* worker.py:45-51 + :85: run slot boundaries until somebody has to decide or the episode ends. */
static void orc_advance(orc_env *e) {
    int ids[ORC_MAX_AGENTS]; double t;
    int empty_slots = 0;
    for (;;) {
        if (!e->first_slot) e->finished = orc_check_finished(e);              /* worker.py:85 */
        e->first_slot = 0;
        if (e->finished || !(e->now < e->max_time)) { e->done = 1; e->leader = -1; return; }   /* worker.py:45 */
        int n = orc_next_decision(e, ids, &t);                                /* :47 */
        e->pending = 0;
        for (int k = 0; k < n; k++) e->pending |= 1ull << ids[k];
        e->now = t;                                                           /* :49 */
        orc_task_update(e, NULL); orc_agent_update(e);                        /* :50-51 */
        if (e->pending) return;
        /* Nobody can decide.  One such slot is normal (it marks agents as returned).  A second one in a
         * row means nothing can change any more: the reference `while` would spin forever.  Stop and flag. */
        if (++empty_slots >= 2) { e->done = 1; e->stuck = 1; e->leader = -1; return; }
    }
}

/* choose the next leader: injected (>=0) or Philox uniform over the current group (worker.py:54) */
static int choose_leader(orc_env *e, int injected) {
    uint64_t g = current_group(e, e->pending);
    if (!g) return -1;
    if (injected >= 0) return (injected < e->A && (g >> injected & 1)) ? injected : -2;
    return kth_bit(g, pick(draw(e, (uint32_t)e->n_steps, 1), popcnt(g)));
}

/* Begin an episode: clear, first slot, first leader.  Returns the leader id (or <0). */
int orc_fused_reset(orc_env *e, int injected_leader) {
    orc_clear_decisions(e);
    orc_advance(e);
    if (e->done) return -1;
    e->leader = choose_leader(e, injected_leader);
    return e->leader;
}

/* Uniform-random action over unmasked entries, or greedy-nearest (policy 1 / 2); used when action < 0. */
int orc_policy_action(const orc_env *e, int policy) {
    uint8_t mask[1024 + 1]; orc_mask(e, mask);
    if (policy == 2) {               /* greedy nearest: argmin squared distance over unmasked tasks, depot if none */
        const orc_agent *L = &e->agent[e->leader];
        int best = 0; double bd = 0;
        for (int j = 0; j < e->T; j++) if (!mask[1 + j]) {
            double dx = e->task[j].x - L->x, dy = e->task[j].y - L->y;
            double d2 = fma(dy, dy, dx * dx);
            if (best == 0 || d2 < bd) { best = j + 1; bd = d2; }
        }
        return best;
    }
    int n = 0; for (int k = 0; k <= e->T; k++) n += !mask[k];
    int r = pick(draw(e, (uint32_t)e->n_steps, 0), n);
    for (int k = 0; k <= e->T; k++) if (!mask[k]) { if (r == 0) return k; r--; }
    return 0;
}

/* One leader decision.
 *   action      0..T, or <0 : use built-in policy (-1 random, -2 greedy-nearest)
 *   followers   NULL -> Philox; else exactly the follower ids step() would have drawn (task_env.py:331), n_followers of them
 *   next_leader <0 -> Philox; else the id np.random.choice(group) returned in the reference run (worker.py:54)
 * Outputs: *reward (task_env.py:341), *done.  Returns 0, or <0 on a contract violation (state untouched). */
int orc_fused_step(orc_env *e, int action, const int *followers, int n_followers, int next_leader,
                   double *reward, int *done_out, int *used_action, int *members_out, int *n_members_out) {
    if (e->done || e->leader < 0) return -1;
    if (action < 0) action = orc_policy_action(e, -action);
    if (action > e->T) return -2;
    if (used_action) *used_action = action;
    uint64_t g = current_group(e, e->pending);
    int leader = e->leader;
    if (!(g >> leader & 1)) return -3;
    int vacancy = orc_vacancy(e, action, popcnt(g));                          /* :327 (len(group) before removal) */
    g &= ~(1ull << leader);                                                   /* :328 */
    int members[ORC_MAX_AGENTS]; int nm = 0; members[nm++] = leader;
    if (vacancy > 1) {                                                        /* :330 */
        int want = vacancy - 1 < popcnt(g) ? vacancy - 1 : popcnt(g);         /* :331 */
        if (followers) {
            if (n_followers != want) return -4;
            uint64_t gg = g;
            for (int k = 0; k < want; k++) { if (followers[k] < 0 || followers[k] >= e->A || !(gg >> followers[k] & 1)) return -5; gg &= ~(1ull << followers[k]); }
            for (int k = 0; k < want; k++) { members[nm++] = followers[k]; g &= ~(1ull << followers[k]); }
        } else if (action == 0) {
            /* depot: the whole group follows (Q11); order is irrelevant for the depot, take ascending ids */
            while (g) { int f = kth_bit(g, 0); members[nm++] = f; g &= ~(1ull << f); }
        } else {
            for (int k = 0; k < want; k++) {
                int f = kth_bit(g, pick(draw(e, (uint32_t)e->n_steps, 2 + k), popcnt(g)));
                members[nm++] = f; g &= ~(1ull << f);
            }
        }
    } else if (followers && n_followers != 0) return -4;
    for (int k = 0; k < nm; k++) e->pending &= ~(1ull << members[k]);
    if (members_out) { for (int k = 0; k < nm; k++) members_out[k] = members[k]; *n_members_out = nm; }
    *reward = orc_step_members(e, members, nm, action);                       /* :337-341 */
    orc_task_update(e, NULL); orc_agent_update(e);                            /* worker.py:74-76 */
    e->n_steps++;
    if (!e->pending) orc_advance(e);
    if (!e->done) {
        e->leader = choose_leader(e, next_leader);
        if (e->leader < 0) return -6;
    }
    *done_out = e->done;
    return 0;
}

uint64_t orc_current_group(const orc_env *e) { return current_group(e, e->pending); }
int orc_leader(const orc_env *e) { return e->leader; }
int orc_done(const orc_env *e) { return e->done; }
int orc_stuck(const orc_env *e) { return e->stuck; }
uint64_t orc_pending(const orc_env *e) { return e->pending; }
long orc_nsteps(const orc_env *e) { return e->n_steps; }

/* ------------------------------------------------------------------ */
/*  CPU baseline loop for bench.py: episodes of the built-in policy, obs+mask built every step */
/* ------------------------------------------------------------------ */
long orc_rollout_bench(orc_env *e, int policy, long min_steps, uint64_t seed, float *obs_sink) {
    long steps = 0; uint32_t ep = 0;
    double *ag = (double *)malloc(sizeof(double) * 6 * e->A);
    double *tk = (double *)malloc(sizeof(double) * 5 * (e->T + 1));
    uint8_t *mask = (uint8_t *)malloc(e->T + 1);
    float acc = 0;
    while (steps < min_steps) {
        orc_seed(e, seed, e->gid, ep++);
        if (orc_fused_reset(e, -1) < 0) break;
        while (!e->done) {
            /* what worker.py:57-64 builds for the policy: mask, agent rows, task rows, cast to fp32 */
            orc_mask(e, mask); orc_agent_status(e, e->leader, ag); orc_task_status(e, e->leader, tk);
            for (int k = 0; k < 6 * e->A; k++) acc += (float)ag[k];
            for (int k = 0; k < 5 * (e->T + 1); k++) acc += (float)tk[k];
            double r; int d;
            if (orc_fused_step(e, -policy, NULL, 0, -1, &r, &d, NULL, NULL, NULL) < 0) break;
            steps++;
        }
    }
    if (obs_sink) *obs_sink = acc;
    free(ag); free(tk); free(mask);
    return steps;
}
