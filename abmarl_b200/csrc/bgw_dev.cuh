/*
 * bgw_dev.cuh -- device side of the B200 batched GridWorld engine (sm_100a).
 *
 * One CTA advances ONE environment by one manager step (all_step_manager.py:51-95 /
 * turn_based_manager.py:34-94).  The env's agent store (cell / next / flags, structure-of-arrays in HBM,
 * include/bgw.h BgwState) is staged into shared memory, the per-cell occupant lists (the reference's
 * insertion-ordered cell dicts, grid.py:24,79,125) are rebuilt there as singly linked lists, the actor
 * phases run on the shared-memory copy, observations are gathered from it and written with 128-bit
 * stores, and the mutated store goes back to HBM.
 *
 * Sequential semantics (SURVEY.md section 7, hard part 1).  The reference resolves actions one agent at a
 * time in action-dict order.  Here every acting agent owns a RANK (its position in that order) and the
 * attack / move phases run as rounds of deterministic reservations: each pending agent atomicMin()s its
 * rank into a reservation slot for every grid cell its action may read or write (attack: the
 * (2R+1)^2 window; move: source and destination cell); an agent that holds the minimum on ALL of its cells
 * executes this round, the others retry.  Two agents whose cell sets are disjoint commute (they touch
 * disjoint occupant lists, health, flags and reward accumulators), and two agents that share a cell are
 * executed in rank order, so the result equals the sequential loop bit for bit; stochastic outcomes come
 * from the keyed Philox stream (include/bgw_philox.h), which does not depend on execution order.
 *
 * Every function cites the reference lines it reproduces; the CPU oracle (oracle/bgw_oracle.c) restates
 * the same lines sequentially and is what the parity tests compare against.
 */
#pragma once
#include <cuda_runtime.h>
#include "../../include/bgw_stdint.h"

#include "../../include/bgw.h"
#include "../../include/bgw_philox.h"

#define BGW_NONE16 0xFFFFu
#define BGW_SLOT_FREE 0xFFFFFFFFu
#define BGW_CSUM_MIXED (-128)
#define BGW_ATT_MASK_WORDS 8   /* thread-local LOS mask of an attacker: (2R+1)^2 <= 256 bits -> attack_range <= 7 */

enum { CTR_KILLS = 0, CTR_ALLDONE, CTR_REMAINING, CTR_ENC_LO, CTR_ENC_HI, CTR_AND, CTR_NEMIT, CTR_ENVDONE,
       CTR_ERR, CTR_TURN, CTR_MIXED, CTR_PA, CTR_PB, CTR_EPOCH, CTR_COUNT = 16 };

struct DevSpec {
    int H, W, HW, A, L, E, env_offset;
    int program, move_actor, attack_actor, observer, observe_self, done_mask, manager, ravel, no_overlap,
        stacked, horizon, auto_reset;
    int max_enc, n_blk;            /* n_blk: entities of class BLOCKING (static list blk_agents) */
    int obs_h, obs_w, obs_c, obs_stride, nchunks;
    int a_nav, a_target, a_pacman, has_food;
    int a_script[10];              /* PacmanSimSimple: the agent of the k-th script entry (pacman.py:235-246), -1 = absent */
    int hw_words;                  /* ceil(HW / 32) */
    int n_var;                     /* entities with random placement */
    int randomize_placement_order; /* PositionState(randomize_placement_order): keyed placement order per episode */
    int tpl_error;
    int slot_mask;                 /* reservation slots - 1 (power of two) */
    int mask_words, mask_batch;    /* LOS scratch of the observation pass */
    int parallel_actors;           /* 1: reservation rounds (team battle, Box/Cross moves); 0: rank-order loop */
    int act_words;                 /* 32-bit words per learner action row (BgwDims.action_stride / 4) */
    int ammo_offset, n_ammo;       /* AmmoObserver slot in the obs row (-1 none); number of AmmoAgents */
    int position_offset;           /* AbsolutePositionObserver slot in the obs row (-1 none) */
    int obs_cells;                 /* obs_h * obs_w * obs_c: grid bytes of an obs row */
    const int32_t *init_ammo;
    unsigned long long seed;
    double reward[BGW_RW_COUNT];
    /* per-entity tables in global memory (shared by all envs, L1/L2 resident) */
    const int8_t *enc;
    const uint8_t *klass, *role, *init_orient, *simatt;
    const int16_t *view_r, *move_r, *attack_r, *target, *learner_of, *agent_of;
    const double *init_health, *strength, *accuracy;
    const unsigned long long *overlap, *attack_map;
    const uint16_t *blk_agents, *var_agents;   /* blk_agents: the n_dyn_blk dynamic blockers first, then the static ones */
    const uint32_t *static_mask;   /* [HW][mask_words] LOS mask of all STATIC blockers per viewer cell, or NULL */
    int n_dyn_blk;
    /* reset template: the env-independent result of placing the fixed-position entities (state.py:107-109) */
    const uint16_t *tpl_cell, *tpl_next;
    const uint8_t *tpl_flags;
    const uint32_t *tpl_avail;     /* [(max_enc+1)][hw_words] availability bit maps after the fixed placements */
    /* shared memory carve-up (byte offsets) */
    int o_head, o_slot, o_cell, o_next, o_flags, o_enc, o_klass, o_tmp, o_racc, o_act, o_ragent, o_plist,
        o_pstate, o_avail, o_mask, o_ctr, o_csum, smem_bytes;
};

struct Env {
    uint16_t *head, *cell, *next, *ragent, *plist;
    uint32_t *slot, *act, *avail, *mask;
    uint8_t *flags, *klass, *tmp, *pstate;
    int8_t *enc;
    int8_t *csum;     /* [HW] per-cell summary for the observers: 0 empty, e = every occupant has encoding e, CSUM_MIXED */
    double *racc;
    int *ctr;
    double *health;   /* this env's row of BgwState.health (global) */
    int32_t *ammo;    /* this env's row of BgwState.ammo (global), or NULL */
    int e;
    uint32_t genv, episode, step;
};

__device__ __forceinline__ void env_init(Env &ev, const DevSpec &s, unsigned char *sm)
{
    ev.head = (uint16_t *)(sm + s.o_head);
    ev.slot = (uint32_t *)(sm + s.o_slot);
    ev.cell = (uint16_t *)(sm + s.o_cell);
    ev.next = (uint16_t *)(sm + s.o_next);
    ev.flags = sm + s.o_flags;
    ev.enc = (int8_t *)(sm + s.o_enc);
    ev.klass = sm + s.o_klass;
    ev.tmp = sm + s.o_tmp;
    ev.racc = (double *)(sm + s.o_racc);
    ev.act = (uint32_t *)(sm + s.o_act);
    ev.ragent = (uint16_t *)(sm + s.o_ragent);
    ev.plist = (uint16_t *)(sm + s.o_plist);
    ev.pstate = sm + s.o_pstate;
    ev.avail = (uint32_t *)(sm + s.o_avail);
    ev.mask = (uint32_t *)(sm + s.o_mask);
    ev.ctr = (int *)(sm + s.o_ctr);
    ev.csum = (int8_t *)(sm + s.o_csum);
}

__device__ __forceinline__ uint32_t dev_draw(const DevSpec &s, const Env &ev, uint32_t site, uint32_t slot, uint32_t k)
{
    return bgw_draw(s.seed, ev.genv, ev.episode, ev.step, site, slot, k);
}

/* ------------------------------------------------------------------------------------------------- */
/* Grid (grid.py) on the shared-memory occupant lists                                                */
/* ------------------------------------------------------------------------------------------------- */
/* Grid.query grid.py:81-105 */
__device__ __forceinline__ bool grid_query(const DevSpec &s, const Env &ev, int a, int cell)
{
    const unsigned long long row = __ldg(&s.overlap[ev.enc[a]]);
    for (unsigned o = ev.head[cell]; o != BGW_NONE16; o = ev.next[o])
        if (!((row >> ev.enc[o]) & 1ull)) return false;
    return true;
}

/* dict insert of Grid.place grid.py:124-126 (append at the tail = arrival order) */
__device__ __forceinline__ void grid_append(Env &ev, int a, int cell)
{
    ev.next[a] = BGW_NONE16;
    unsigned p = ev.head[cell];
    if (p == BGW_NONE16) ev.head[cell] = (uint16_t)a;
    else {
        for (unsigned q = ev.next[p]; q != BGW_NONE16; q = ev.next[p]) p = q;
        ev.next[p] = (uint16_t)a;
    }
    ev.cell[a] = (uint16_t)cell;
    ev.flags[a] |= BGW_ST_IN_GRID;
}

/* Grid.remove grid.py:131-140; the entity's position stays (actor.py:356-358) */
__device__ __forceinline__ void grid_unlink(Env &ev, int a)
{
    if (!(ev.flags[a] & BGW_ST_IN_GRID)) return;
    const int cell = ev.cell[a];
    unsigned p = ev.head[cell];
    if (p == (unsigned)a) ev.head[cell] = ev.next[a];
    else {
        while (ev.next[p] != (unsigned)a) p = ev.next[p];
        ev.next[p] = ev.next[a];
    }
    ev.next[a] = BGW_NONE16;
    ev.flags[a] &= ~BGW_ST_IN_GRID;
}

/* HealthAgent.health setter agent.py:192-196 (health lives in HBM and is touched on demand) */
__device__ __forceinline__ void set_health(Env &ev, int a, double v)
{
    double h = v < 0.0 ? 0.0 : v;
    h = h > 1.0 ? 1.0 : h;
    __stcg(&ev.health[a], h);
    if (h > 0.0) ev.flags[a] |= BGW_ST_ACTIVE; else ev.flags[a] &= ~BGW_ST_ACTIVE;
}

/* Under AllStepManager every learner's reward accumulator is read (and zeroed) in the call that fills it
 * (smart.py:101-104), so it is zero between calls and need not be staged -- except for entities that can be
 * attacked but never report: non-learners with health (their accumulator keeps the 'die' reward forever). */
__device__ __forceinline__ bool racc_persists(uint8_t klass) { return !(klass & BGW_AG_LEARNER) && (klass & BGW_AG_HEALTH); }

/* rebuild the per-cell list heads from the persisted `next` pointers (all threads; ends synchronised) */
static __device__ void build_heads(const DevSpec &s, Env &ev, int tid, int T)
{
    for (int i = tid; i < (s.HW + 1) / 2; i += T) ((uint32_t *)ev.head)[i] = 0xFFFFFFFFu;
    for (int a = tid; a < s.A; a += T) ev.tmp[a] = 0;
    __syncthreads();
    for (int a = tid; a < s.A; a += T)
        if ((ev.flags[a] & BGW_ST_IN_GRID) && ev.next[a] != BGW_NONE16) ev.tmp[ev.next[a]] = 1;
    __syncthreads();
    for (int a = tid; a < s.A; a += T)
        if ((ev.flags[a] & BGW_ST_IN_GRID) && !ev.tmp[a]) ev.head[ev.cell[a]] = (uint16_t)a;
    __syncthreads();
}

/* ------------------------------------------------------------------------------------------------- */
/* create_grid_and_mask: the mask, utils.py:45-115                                                   */
/* ------------------------------------------------------------------------------------------------- */
template <bool ATOMIC>
__device__ __forceinline__ void mask_clear(uint32_t *m, int idx)
{
    if (ATOMIC) atomicAnd(&m[idx >> 5], ~(1u << (idx & 31)));
    else m[idx >> 5] &= ~(1u << (idx & 31));
}

/* Clear the bits of the cells hidden behind a blocker at offset (rd, cd).  Same two ray families as the
 * oracle's los_apply(); the rays are (a/b)*t in IEEE float64 (explicit _rn intrinsics: never contracted), and
 * the strict comparisons lo < r < up are turned into exact integer bounds floor(lo)+1 .. ceil(up)-1. */
template <bool ATOMIC>
__device__ void los_apply_dev(uint32_t *m, int R, int rd, int cd, int rlo, int rhi, int clo, int chi)
{
    const int n = 2 * R + 1;
    if (rd == 0 && cd == 0) return;
    rlo = max(rlo, -R); rhi = min(rhi, R); clo = max(clo, -R); chi = min(chi, R);
    if (cd != 0) {
        double du, dl;
        if (rd == 0) { du = dl = (cd > 0) ? (double)cd - 0.5 : (double)cd + 0.5; }        /* utils.py:53-54,89-90 */
        else if ((rd > 0) == (cd > 0)) { du = (double)cd - 0.5; dl = (double)cd + 0.5; }  /* :62-63,98-99 */
        else { du = (double)cd + 0.5; dl = (double)cd - 0.5; }                            /* :80-81,107-108 */
        const double ku = __ddiv_rn((double)rd + 0.5, du), kl = __ddiv_rn((double)rd - 0.5, dl);
        const int c0 = cd > 0 ? max(cd, clo) : clo, c1 = cd > 0 ? chi : min(cd, chi);
        int r0 = rd > 0 ? rd : rlo, r1 = rd < 0 ? rd : rhi;
        r0 = max(r0, rlo); r1 = min(r1, rhi);
        for (int c = c0; c <= c1; ++c) {
            const double up = __dmul_rn(ku, (double)c), lo = __dmul_rn(kl, (double)c);
            const int ra = max(r0, __double2int_rd(lo) + 1), rb = min(r1, __double2int_ru(up) - 1);
            for (int r = ra; r <= rb; ++r) {
                if (c == cd && r == rd) continue;
                mask_clear<ATOMIC>(m, (r + R) * n + (c + R));
            }
        }
    } else {
        const double d = rd > 0 ? (double)rd - 0.5 : (double)rd + 0.5;                    /* utils.py:71-72,116-117 */
        const double kl = __ddiv_rn((double)cd - 0.5, d), kr = __ddiv_rn((double)cd + 0.5, d);
        int r0 = rd > 0 ? rd : rlo, r1 = rd > 0 ? rhi : rd;
        r0 = max(r0, rlo); r1 = min(r1, rhi);
        for (int r = r0; r <= r1; ++r) {
            const double le = __dmul_rn(kl, (double)r), ri = __dmul_rn(kr, (double)r);
            const int ca = max(clo, __double2int_rd(le) + 1), cb = min(chi, __double2int_ru(ri) - 1);
            for (int c = ca; c <= cb; ++c) {
                if (c == cd && r == rd) continue;
                mask_clear<ATOMIC>(m, (r + R) * n + (c + R));
            }
        }
    }
}

/* one (viewer, blocker) pair of utils.py:46-51 */
template <bool ATOMIC>
__device__ __forceinline__ void los_pair(const DevSpec &s, const Env &ev, uint32_t *m, int viewer_cell, int R, int b,
                                         bool clip_to_grid)
{
    if (!(ev.flags[b] & BGW_ST_ACTIVE)) return;
    const int bc = ev.cell[b];
    if (bc == BGW_NONE16) return;
    const int r0 = viewer_cell / s.W, c0 = viewer_cell % s.W;
    const int rd = bc / s.W - r0, cd = bc % s.W - c0;
    if (rd < -R || rd > R || cd < -R || cd > R) return;
    int rlo = -R, rhi = R, clo = -R, chi = R;
    if (clip_to_grid) { rlo = -r0; rhi = s.H - 1 - r0; clo = -c0; chi = s.W - 1 - c0; }
    los_apply_dev<ATOMIC>(m, R, rd, cd, rlo, rhi, clo, chi);
}

/* ------------------------------------------------------------------------------------------------- */
/* Actors: actor.py                                                                                  */
/* ------------------------------------------------------------------------------------------------- */
__device__ __forceinline__ void cross_delta(int k, int &dr, int &dc)   /* CrossMoveActor.grid_action actor.py:153-159 */
{
    dr = (k == 2) - (k == 4);
    dc = (k == 3) - (k == 1);
}

/* shared tail of MoveActor / CrossMoveActor.process_action actor.py:99-114,177-194 */
static __device__ bool try_move(const DevSpec &s, Env &ev, int a, int dr, int dc)
{
    const int from = ev.cell[a];
    const int r = from / s.W + dr, c = from % s.W + dc;
    if (r < 0 || r >= s.H || c < 0 || c >= s.W) return false;
    const int to = r * s.W + c;
    if (to == from) return true;
    if (!grid_query(s, ev, a, to)) return false;
    grid_unlink(ev, a);
    grid_append(ev, a, to);
    return true;
}

/* decode the move bytes of a Box / ravelled / cross action (wrapper.py:143-159, ravel_discrete_wrapper.py:90-92) */
__device__ __forceinline__ void decode_move(const DevSpec &s, int a, uint32_t act, int &dr, int &dc)
{
    if (s.move_actor == BGW_MOVE_BOX) {
        if (s.ravel) {
            const int m = __ldg(&s.move_r[a]), w = 2 * m + 1, v = act & 0xFF;
            dr = v / w - m; dc = v % w - m;
        } else {
            dr = (int8_t)(act & 0xFF); dc = (int8_t)((act >> 8) & 0xFF);
        }
    } else {
        cross_delta((int8_t)(act & 0xFF), dr, dc);
    }
}

/* move_result as the user's step() sees it (None counts as failure): actor.py:82-114,161-194,208-234 */
static __device__ bool process_move(const DevSpec &s, Env &ev, int a, uint32_t act)
{
    if (!(ev.klass[a] & BGW_AG_MOVING)) return false;
    if (s.move_actor == BGW_MOVE_BOX || s.move_actor == BGW_MOVE_CROSS) {
        int dr, dc;
        decode_move(s, a, act, dr, dc);
        return try_move(s, ev, a, dr, dc);
    }
    if (s.move_actor == BGW_MOVE_DRIFT) {                          /* DriftMoveActor actor.py:208-234 */
        if (!(ev.klass[a] & BGW_AG_ORIENT)) return false;
        const int k = (int8_t)(act & 0xFF);
        int dr, dc;
        cross_delta(k, dr, dc);
        if (k != 0 && try_move(s, ev, a, dr, dc)) {
            ev.flags[a] = (uint8_t)((ev.flags[a] & 0x8F) | (k << BGW_ST_ORIENT_SHIFT));
            return true;
        }
        const int o = (ev.flags[a] >> BGW_ST_ORIENT_SHIFT) & 7;
        cross_delta(o, dr, dc);
        return try_move(s, ev, a, dr, dc);
    }
    return false;
}

/* AttackActorBaseComponent._basic_criteria actor.py:381-392.  The accuracy draw is keyed by
 * (attacker, candidate); with accuracy >= 1 the comparison u > accuracy can never hold, so the draw is
 * skipped (keyed streams: skipping a draw does not shift any other). */
__device__ __forceinline__ bool basic_criteria(const DevSpec &s, const Env &ev, int attacker, int cand,
                                               unsigned long long map_row, double acc, uint32_t occ = 0)
{
    if (cand == attacker) return false;
    if (!(ev.flags[cand] & BGW_ST_ACTIVE)) return false;
    if (!((map_row >> ev.enc[cand]) & 1ull)) return false;
    if (acc < 1.0) {
        const double u = bgw_u01(dev_draw(s, ev, BGW_SITE_ACC, (uint32_t)attacker, (uint32_t)cand + 4096u * occ));
        if (u > acc) return false;
    }
    return true;
}

/* BinaryAttackActor._determine_attack + AttackActorBaseComponent.process_action (actor.py:455-501,
 * 306-361) followed by the reward lines of TeamBattleSim.step (team_battle_example.py:38-47) for ONE
 * attacker whose `attack` action is 1 (simultaneous_attacks == 1 is enforced at bgw_create). */
static __device__ void exec_attack(const DevSpec &s, Env &ev, int a)
{
    if (!(ev.flags[a] & BGW_ST_ACTIVE)) return;                   /* team_battle_example.py:37 */
    const int R = __ldg(&s.attack_r[a]), n = 2 * R + 1;
    const int from = ev.cell[a], r0 = from / s.W, c0 = from % s.W;
    const unsigned long long row = __ldg(&s.attack_map[ev.enc[a]]);
    const double acc = __ldg(&s.accuracy[a]);
    uint32_t m[BGW_ATT_MASK_WORDS];
    const bool use_mask = s.n_blk > 0;
    if (use_mask) {
#pragma unroll
        for (int i = 0; i < BGW_ATT_MASK_WORDS; ++i) m[i] = 0xFFFFFFFFu;
        for (int i = 0; i < s.n_blk; ++i) los_pair<false>(s, ev, m, from, R, __ldg(&s.blk_agents[i]), false);
    }
    const int ra = max(0, r0 - R), rb = min(s.H - 1, r0 + R), ca = max(0, c0 - R), cb = min(s.W - 1, c0 + R);
    int ncand = 0;
    for (int gr = ra; gr <= rb; ++gr)                              /* actor.py:489-496 */
        for (int gc = ca; gc <= cb; ++gc) {
            if (use_mask) {
                const int idx = (gr - r0 + R) * n + (gc - c0 + R);
                if (!((m[idx >> 5] >> (idx & 31)) & 1u)) continue;
            }
            for (unsigned o = ev.head[gr * s.W + gc]; o != BGW_NONE16; o = ev.next[o])
                ncand += basic_criteria(s, ev, a, (int)o, row, acc) ? 1 : 0;
        }
    if (ncand == 0) { ev.racc[a] += s.reward[BGW_RW_ATTACK_FAIL]; return; }   /* actor.py:500-501, tb:41-42 */
    /* _subset_attackables actor.py:394-414 with n == 1: one keyed draw over the candidate list */
    int j = (int)bgw_index(dev_draw(s, ev, BGW_SITE_SUBSET, (uint32_t)a, 0), (uint32_t)ncand);
    int v = -1;
    for (int gr = ra; gr <= rb && v < 0; ++gr)
        for (int gc = ca; gc <= cb && v < 0; ++gc) {
            if (use_mask) {
                const int idx = (gr - r0 + R) * n + (gc - c0 + R);
                if (!((m[idx >> 5] >> (idx & 31)) & 1u)) continue;
            }
            for (unsigned o = ev.head[gr * s.W + gc]; o != BGW_NONE16; o = ev.next[o])
                if (basic_criteria(s, ev, a, (int)o, row, acc) && j-- == 0) { v = (int)o; break; }
        }
    /* actor.py:353-358 */
    set_health(ev, v, __ldcg(&ev.health[v]) - __ldg(&s.strength[a]));
    if (!(ev.flags[v] & BGW_ST_ACTIVE)) {
        grid_unlink(ev, v);
        atomicAdd(&ev.ctr[CTR_KILLS], 1);
        ev.racc[v] += s.reward[BGW_RW_DIE];                       /* team_battle_example.py:44-47 */
        ev.racc[a] += s.reward[BGW_RW_KILL];
    }
}

/* ---- the other attack actors (and the ammo filter) --------------------------------------------------------- */
/* attack bytes of entity a's action row (layout: bgw.h, bgw_step) and how many of them its action has */
__device__ __forceinline__ const uint8_t *attack_bytes(const DevSpec &s, const Env &ev, int a)
{
    return reinterpret_cast<const uint8_t *>(ev.act + (size_t)__ldg(&s.learner_of[a]) * s.act_words) + 2;
}

__device__ __forceinline__ int attack_width(const DevSpec &s, int a)
{
    if (s.attack_actor == BGW_ATTACK_ENCODING) return s.max_enc;                       /* actor.py:513-519 */
    if (s.attack_actor == BGW_ATTACK_RESTRICTED) return __ldg(&s.simatt[a]);           /* :593-599 */
    if (s.attack_actor == BGW_ATTACK_SELECTIVE) { const int n = 2 * __ldg(&s.attack_r[a]) + 1; return n * n; }   /* :669-679 */
    return 1;                                                                          /* :451-453 */
}

/* `if not attack` / `not any(...)` / `not np.any(attack)` actor.py:478,542,622,703 */
__device__ __forceinline__ bool attack_requested(const DevSpec &s, const Env &ev, int a)
{
    const uint8_t *att = attack_bytes(s, ev, a);
    const int w = attack_width(s, a);
    unsigned any = 0;
    for (int j = 0; j < w; ++j) any |= att[j];
    return any != 0;
}

struct AttackView {                      /* gu.create_grid_and_mask(agent, grid, attack_range, agents) for one attacker */
    int a, R, n, r0, c0;
    unsigned long long row;
    double acc;
    bool use_mask;
    uint32_t m[BGW_ATT_MASK_WORDS];
};

/* grid cell of window cell (wr, wc), or -1 when it is masked or outside the grid (local_grid[r, c] is None) */
__device__ __forceinline__ int attack_window_cell(const DevSpec &s, const AttackView &v, int wr, int wc)
{
    if (v.use_mask) { const int idx = wr * v.n + wc; if (!((v.m[idx >> 5] >> (idx & 31)) & 1u)) return -1; }
    const int gr = v.r0 - v.R + wr, gc = v.c0 - v.R + wc;
    if (gr < 0 || gr >= s.H || gc < 0 || gc >= s.W) return -1;
    return gr * s.W + gc;
}

/* Walk the attackable agents of window cells [wr0..wr1] x [wc0..wc1] in the reference's scan order (cells row-major,
 * occupants in dict order; actor.py:489-496): those that pass _basic_criteria, have encoding enc_only (if > 0) and
 * are not in skip[0..nskip).  f(agent) returns true to stop. */
template <typename F>
__device__ __forceinline__ void for_attackables(const DevSpec &s, const Env &ev, const AttackView &v, int wr0, int wr1, int wc0,
                                                int wc1, int enc_only, uint32_t occ, const uint16_t *skip, int nskip, F f)
{
    for (int wr = wr0; wr <= wr1; ++wr)
        for (int wc = wc0; wc <= wc1; ++wc) {
            const int cell = attack_window_cell(s, v, wr, wc);
            if (cell < 0) continue;
            for (unsigned o = ev.head[cell]; o != BGW_NONE16; o = ev.next[o]) {
                if (enc_only > 0 && ev.enc[o] != enc_only) continue;
                if (!basic_criteria(s, ev, v.a, (int)o, v.row, v.acc, occ)) continue;
                bool skipped = false;
                for (int q = 0; q < nskip; ++q) skipped |= (skip[q] == (uint16_t)o);
                if (skipped) continue;
                if (f((int)o)) return;
            }
        }
}

/* _subset_attackables actor.py:394-414 over the attackables of a window region: appends the chosen agents to
 * victims[nv..] and returns the new count.  Draw keys: BGW_SITE_SUBSET, slot = attacker, k = group << 8 | draw#.  The
 * choice without replacement is a partial Fisher-Yates over the candidate list, kept as a sparse map of the
 * displaced positions (k <= BGW_MAX_SIMATT picks), the positions are resolved by walking the region again. */
static __device__ int subset_attackables_dev(const DevSpec &s, const Env &ev, const AttackView &v, int wr0, int wr1, int wc0, int wc1,
                                      int enc_only, uint32_t group, int k, uint16_t *victims, int nv)
{
    int ncand = 0;
    for_attackables(s, ev, v, wr0, wr1, wc0, wc1, enc_only, 0, nullptr, 0, [&](int) { ++ncand; return false; });
    if (ncand == 0 || k <= 0) return nv;
    if (!s.stacked && k > ncand) {                                  /* the whole list, no draw :410-411 */
        for_attackables(s, ev, v, wr0, wr1, wc0, wc1, enc_only, 0, nullptr, 0,
                        [&](int o) { if (nv < BGW_MAX_VICTIMS) victims[nv++] = (uint16_t)o; return false; });
        return nv;
    }
    k = min(k, BGW_MAX_SIMATT);
    int pos[BGW_MAX_SIMATT];
    if (s.stacked) {
        for (int t = 0; t < k; ++t)
            pos[t] = ncand == 1 ? 0 : (int)bgw_index(dev_draw(s, ev, BGW_SITE_SUBSET, (uint32_t)v.a, (group << 8) | (uint32_t)t), (uint32_t)ncand);
    } else {
        int mk[BGW_MAX_SIMATT], mv[BGW_MAX_SIMATT], nm = 0;
        for (int t = 0; t < k; ++t) {
            const int rem = ncand - t;
            const int j = t + (rem == 1 ? 0 : (int)bgw_index(dev_draw(s, ev, BGW_SITE_SUBSET, (uint32_t)v.a, (group << 8) | (uint32_t)t), (uint32_t)rem));
            int vj = j, vt = t, at = -1;
            for (int q = 0; q < nm; ++q) { if (mk[q] == j) { vj = mv[q]; at = q; } if (mk[q] == t) vt = mv[q]; }
            pos[t] = vj;
            if (at >= 0) mv[at] = vt; else { mk[nm] = j; mv[nm] = vt; ++nm; }
        }
    }
    for (int t = 0; t < k; ++t) {
        int want = pos[t], found = -1;
        for_attackables(s, ev, v, wr0, wr1, wc0, wc1, enc_only, 0, nullptr, 0,
                        [&](int o) { if (want-- == 0) { found = o; return true; } return false; });
        if (found >= 0 && nv < BGW_MAX_VICTIMS) victims[nv++] = (uint16_t)found;
    }
    return nv;
}

/* <attack actor>._determine_attack (actor.py:455-501 Binary, 521-582 EncodingBased, 601-658 RestrictedSelective,
 * 681-728 Selective) + the ammo filter of AttackActorBaseComponent.process_action (:343-351) for ONE attacker that
 * requested an attack: victims[0..n) = attacked_agents.  Returns n. */
static __device__ __forceinline__ int attack_victims(const DevSpec &s, Env &ev, int a, uint16_t *victims)
{
    AttackView v;
    v.a = a; v.R = __ldg(&s.attack_r[a]); v.n = 2 * v.R + 1;
    v.r0 = ev.cell[a] / s.W; v.c0 = ev.cell[a] % s.W;
    v.row = __ldg(&s.attack_map[ev.enc[a]]);
    v.acc = __ldg(&s.accuracy[a]);
    v.use_mask = s.n_blk > 0;
    if (v.use_mask) {
#pragma unroll
        for (int i = 0; i < BGW_ATT_MASK_WORDS; ++i) v.m[i] = 0xFFFFFFFFu;
        for (int i = 0; i < s.n_blk; ++i) los_pair<false>(s, ev, v.m, ev.cell[a], v.R, __ldg(&s.blk_agents[i]), false);
    }
    const uint8_t *att = attack_bytes(s, ev, a);
    const int n = v.n, last = n - 1;
    int nv = 0;
    switch (s.attack_actor) {
    case BGW_ATTACK_BINARY:
        nv = subset_attackables_dev(s, ev, v, 0, last, 0, last, 0, 0u, att[0], victims, nv);
        break;
    case BGW_ATTACK_ENCODING:                                      /* `for encoding, num_attacks in attack.items()`, ascending */
        for (int enc = 1; enc <= s.max_enc; ++enc)
            if (((v.row >> enc) & 1ull) && att[enc - 1])
                nv = subset_attackables_dev(s, ev, v, 0, last, 0, last, enc, (uint32_t)enc, att[enc - 1], victims, nv);
        break;
    case BGW_ATTACK_RESTRICTED: {
        const int width = __ldg(&s.simatt[a]);
        for (int j = 0; j < width; ++j) {
            const int code = att[j];
            if (code == 0) continue;                               /* :635-637 */
            const int rav = code - 1, wr = rav % n, wc = rav / n;  /* :641-643: row = remainder, column = quotient */
            if (wr >= n || wc >= n) continue;
            uint32_t occ = 0;                                      /* earlier attacks of this action on the same cell */
            for (int q = 0; q < j; ++q) occ += (att[q] == code);
            const uint16_t *skip = s.stacked ? nullptr : victims;  /* :652-654 */
            const int nskip = s.stacked ? 0 : nv;
            int ncand = 0;
            for_attackables(s, ev, v, wr, wr, wc, wc, 0, occ, skip, nskip, [&](int) { ++ncand; return false; });
            if (ncand == 0 || nv >= BGW_MAX_VICTIMS) continue;
            int want = ncand == 1 ? 0 : (int)bgw_index(dev_draw(s, ev, BGW_SITE_SUBSET, (uint32_t)a, (uint32_t)nv << 8), (uint32_t)ncand);
            int found = -1;
            for_attackables(s, ev, v, wr, wr, wc, wc, 0, occ, skip, nskip, [&](int o) { if (want-- == 0) { found = o; return true; } return false; });
            if (found >= 0) victims[nv++] = (uint16_t)found;
        }
        break;
    }
    case BGW_ATTACK_SELECTIVE:
        for (int wr = 0; wr < n; ++wr)
            for (int wc = 0; wc < n; ++wc)
                if (att[wr * n + wc])
                    nv = subset_attackables_dev(s, ev, v, wr, wr, wc, wc, 0, (uint32_t)(wr * n + wc), att[wr * n + wc], victims, nv);
        break;
    default: break;
    }
    if ((ev.klass[a] & BGW_AG_AMMO) && ev.ammo) {                  /* actor.py:343-351 */
        int ammo = ev.ammo[a];
        if (nv > ammo) {                                           /* np.random.choice(size=ammo, replace=False) */
            for (int t = 0; t < ammo; ++t) {
                const int j = t + (int)bgw_index(dev_draw(s, ev, BGW_SITE_AMMO, (uint32_t)a, (uint32_t)t), (uint32_t)(nv - t));
                const uint16_t tmp = victims[t]; victims[t] = victims[j]; victims[j] = tmp;
            }
            nv = ammo;
        }
        ev.ammo[a] = max(ammo - nv, 0);
    }
    return nv;
}

/* the damage of process_action (actor.py:353-358): the attacked agents lose the attacker's strength, the dead leave the grid */
static __device__ __forceinline__ void attack_damage(const DevSpec &s, Env &ev, int a, const uint16_t *victims, int nv)
{
    const double strength = __ldg(&s.strength[a]);
    for (int t = 0; t < nv; ++t) {
        const int x = victims[t];
        if (!(ev.flags[x] & BGW_ST_ACTIVE)) continue;
        set_health(ev, x, __ldcg(&ev.health[x]) - strength);
        if (!(ev.flags[x] & BGW_ST_ACTIVE)) { grid_unlink(ev, x); atomicAdd(&ev.ctr[CTR_KILLS], 1); }
    }
}

/* one attacker's process_action + the reward lines of TeamBattleSim.step (team_battle_example.py:37-47) */
static __device__ void exec_attack_ext(const DevSpec &s, Env &ev, int a)
{
    if (!(ev.flags[a] & BGW_ST_ACTIVE)) return;                   /* team_battle_example.py:37 */
    uint16_t victims[BGW_MAX_VICTIMS];
    const int nv = attack_victims(s, ev, a, victims);
    if (nv == 0) { ev.racc[a] += s.reward[BGW_RW_ATTACK_FAIL]; return; }   /* team_battle_example.py:41-42 */
    attack_damage(s, ev, a, victims, nv);
    for (int t = 0; t < nv; ++t)                                    /* team_battle_example.py:44-47 */
        if (!(ev.flags[victims[t]] & BGW_ST_ACTIVE)) { ev.racc[victims[t]] += s.reward[BGW_RW_DIE]; ev.racc[a] += s.reward[BGW_RW_KILL]; }
}

/* one attacker's turn in the attack phase */
__device__ __forceinline__ void run_attack(const DevSpec &s, Env &ev, int a)
{
    if (s.attack_actor == BGW_ATTACK_BINARY && s.n_ammo == 0) exec_attack(s, ev, a); else exec_attack_ext(s, ev, a);
}

/* reservation helpers: slot of a cell */
__device__ __forceinline__ uint32_t *slot_of(const DevSpec &s, const Env &ev, int cell) { return &ev.slot[cell & s.slot_mask]; }

/* PacmanSimSimple.step pacman.py:235-303: the baddies' scripted DriftMoveActor actions of this step.  k indexes the
 * script's entries (baddie_20, 36, 156, 157, 159, 161, 162, 206, 222, 328); sc = step_count, o156 = orientation of
 * baddie_156, x159 = the keyed draw that stands in for np.random.randint(0, 5) */
static __device__ void pacman_script(int sc, int o156, uint32_t x159, int move[10])
{
    const int base[10] = {0, 0, 0, 1, 0, 3, 0, 0, 0, 0};
#pragma unroll
    for (int k = 0; k < 10; ++k) move[k] = base[k];
    move[4] = (int)bgw_index(x159, 5);
    if (sc == 0) { move[2] = 4; move[6] = 4; move[9] = 3; }                              /* :247-250 */
    switch (sc % 10) {                                                                     /* :251-262 */
    case 0: move[0] = 3; move[1] = 1; break;
    case 3: move[0] = 2; move[1] = 2; break;
    case 5: move[0] = 1; move[1] = 3; break;
    case 8: move[0] = 4; move[1] = 4; break;
    default: break;
    }
    if ((((sc - 8) % 16) + 16) % 16 == 0) {                                               /* :263-271 (Python's modulo) */
        if (o156 == 4) { move[2] = 2; move[6] = 2; move[9] = 3; }
        else { move[2] = 4; move[6] = 4; move[9] = 1; }
    }
    switch (sc % 14) {                                                                     /* :272-289 */
    case 0: move[7] = 3; move[8] = 1; break;
    case 3: move[7] = 2; move[8] = 2; break;
    case 7: move[7] = 1; move[8] = 3; break;
    case 9: move[7] = 4; move[8] = 4; break;
    case 11: move[7] = 1; move[8] = 3; break;
    case 12: move[7] = 4; move[8] = 4; break;
    default: break;
    }
}

/* PacmanSimSimple's overlap checks pacman.py:228-239 (with food) and :305-311 (baddies only): true when a baddie ate
 * pacman -- the reference returns from step() at that point */
static __device__ bool pacman_simple_overlaps(const DevSpec &s, Env &ev, int p, bool eat_food)
{
    unsigned nx;
    for (unsigned o = ev.head[ev.cell[p]]; o != BGW_NONE16; o = nx) {
        nx = ev.next[o];
        if ((int)o == p) continue;
        const int role = __ldg(&s.role[o]);
        if (eat_food && role == BGW_ROLE_FOOD) {
            ev.racc[p] += s.reward[BGW_RW_EAT_FOOD];
            grid_unlink(ev, (int)o);
            set_health(ev, (int)o, 0.0);
        } else if (role == BGW_ROLE_BADDIE || role >= BGW_ROLE_SCRIPTED_BADDIE) {
            ev.racc[p] += s.reward[BGW_RW_DIE];
            set_health(ev, p, 0.0);
            grid_unlink(ev, p);
            return true;
        }
    }
    return false;
}

/* ------------------------------------------------------------------------------------------------- */
/* sim programs: the user-written step()                                                             */
/* ------------------------------------------------------------------------------------------------- */
__device__ __forceinline__ bool prog_done(const DevSpec &s, const Env &ev, int a);

/* ReachTheTargetSim.step reach_the_target.py:141-144: a runner standing on the target's cell has reached it.  A runner
 * that is no longer in the grid (killed on that cell) would make the reference's grid.remove raise; it is left alone. */
__device__ __forceinline__ void reach_check(const DevSpec &s, Env &ev, int a)
{
    if (a != s.a_target && (ev.flags[a] & BGW_ST_IN_GRID) && ev.cell[a] == ev.cell[s.a_target]) {
        ev.racc[a] += s.reward[BGW_RW_TARGET];
        grid_unlink(ev, a);
        ev.flags[a] &= ~BGW_ST_ACTIVE;
    }
}

/* TeamBattleSim.step team_battle_example.py:33-59, ReachTheTargetSim.step reach_the_target.py:117-152 (same attack
 * phase; only MovingAgents move, a runner that reaches the target leaves the grid, only runners pay the entropy
 * penalty) and TrafficCorridorSimulation.step traffic_corridor.py:46-53 (moves only; +1 while on the own target, no
 * entropy penalty); ranks 0..nrank-1 hold the acting agents (ragent) */
static __device__ void team_battle_step(const DevSpec &s, Env &ev, int nrank, int tid, int T)
{
    const double *rw = s.reward;
    const bool reach = s.program == BGW_PROG_REACH_TARGET, traffic = s.program == BGW_PROG_TRAFFIC;
    if (!s.parallel_actors) {
        if (tid == 0) {
            for (int i = 0; i < nrank; ++i) {
                const int a = ev.ragent[i];
                if (a == BGW_NONE16) continue;
                if ((ev.klass[a] & BGW_AG_ATTACKING) && attack_requested(s, ev, a)) run_attack(s, ev, a);
            }
            for (int i = 0; i < nrank; ++i) {
                const int a = ev.ragent[i];
                if (a == BGW_NONE16 || (reach && !(ev.klass[a] & BGW_AG_MOVING))) continue;
                if (ev.flags[a] & BGW_ST_ACTIVE)
                    if (!process_move(s, ev, a, ev.act[(size_t)__ldg(&s.learner_of[a]) * s.act_words])) ev.racc[a] += rw[BGW_RW_MOVE_FAIL];
                if (reach) reach_check(s, ev, a);
                if (traffic && prog_done(s, ev, a)) ev.racc[a] += rw[BGW_RW_TARGET];
            }
            for (int i = 0; i < nrank && !traffic; ++i)
                if (ev.ragent[i] != BGW_NONE16 && (!reach || __ldg(&s.role[ev.ragent[i]]) == BGW_ROLE_RUNNER)) ev.racc[ev.ragent[i]] += rw[BGW_RW_ENTROPY];
        }
        __syncthreads();
        return;
    }

    /* ---- attack phase :35-47 ------------------------------------------------------------------ */
    int mine = 0;
    for (int i = tid; i < nrank; i += T) {
        const int a = ev.ragent[i];
        uint8_t p = 0;
        if (a != BGW_NONE16 && (ev.flags[a] & BGW_ST_ACTIVE) && (ev.klass[a] & BGW_AG_ATTACKING) && attack_requested(s, ev, a)) p = 1;
        ev.pstate[i] = p;
        mine |= p;
    }
    int any = __syncthreads_or(mine);
    while (any) {
        for (int i = tid; i < nrank; i += T) {
            if (ev.pstate[i] != 1) continue;
            const int a = ev.ragent[i], R = __ldg(&s.attack_r[a]);
            const int r0 = ev.cell[a] / s.W, c0 = ev.cell[a] % s.W;
            for (int gr = max(0, r0 - R); gr <= min(s.H - 1, r0 + R); ++gr)
                for (int gc = max(0, c0 - R); gc <= min(s.W - 1, c0 + R); ++gc)
                    atomicMin(slot_of(s, ev, gr * s.W + gc), (uint32_t)i);
        }
        __syncthreads();
        for (int i = tid; i < nrank; i += T) {
            if (ev.pstate[i] != 1) continue;
            const int a = ev.ragent[i], R = __ldg(&s.attack_r[a]);
            const int r0 = ev.cell[a] / s.W, c0 = ev.cell[a] % s.W;
            bool win = true;
            for (int gr = max(0, r0 - R); gr <= min(s.H - 1, r0 + R); ++gr)
                for (int gc = max(0, c0 - R); gc <= min(s.W - 1, c0 + R); ++gc)
                    win &= (*slot_of(s, ev, gr * s.W + gc) == (uint32_t)i);
            if (win) ev.pstate[i] = 2;
        }
        __syncthreads();
        mine = 0;
        for (int i = tid; i < nrank; i += T) {
            if (ev.pstate[i] == 2) {
                const int a = ev.ragent[i], R = __ldg(&s.attack_r[a]);
                const int r0 = ev.cell[a] / s.W, c0 = ev.cell[a] % s.W;
                run_attack(s, ev, a);
                for (int gr = max(0, r0 - R); gr <= min(s.H - 1, r0 + R); ++gr)
                    for (int gc = max(0, c0 - R); gc <= min(s.W - 1, c0 + R); ++gc)
                        *slot_of(s, ev, gr * s.W + gc) = BGW_SLOT_FREE;
                ev.pstate[i] = 0;
            }
            mine |= ev.pstate[i];
        }
        any = __syncthreads_or(mine);
    }

    /* ---- move phase :50-55 ---------------------------------------------------------------------- */
    mine = 0;
    for (int i = tid; i < nrank; i += T) {
        const int a = ev.ragent[i];
        uint8_t p = 0;
        if (a != BGW_NONE16 && (ev.flags[a] & BGW_ST_ACTIVE) && (!reach || (ev.klass[a] & BGW_AG_MOVING))) {
            bool ok = false;
            if (ev.klass[a] & BGW_AG_MOVING) {
                int dr, dc;
                decode_move(s, a, ev.act[(size_t)__ldg(&s.learner_of[a]) * s.act_words], dr, dc);
                const int from = ev.cell[a], r = from / s.W + dr, c = from % s.W + dc;
                if (r >= 0 && r < s.H && c >= 0 && c < s.W) {
                    const int to = r * s.W + c;
                    if (to == from) ok = true;
                    else { p = 1; ev.plist[i] = (uint16_t)to; }
                }
            }
            if (!p && !ok) ev.racc[a] += rw[BGW_RW_MOVE_FAIL];
            /* a runner that does not move but stands on the target's cell (placed there) still reaches it: the removal
             * goes through the ordered rounds as a move to its own cell */
            if (reach && !p && (ev.flags[a] & BGW_ST_IN_GRID) && a != s.a_target && ev.cell[a] == ev.cell[s.a_target]) { p = 1; ev.plist[i] = ev.cell[a]; }
            if (traffic && !p && prog_done(s, ev, a)) ev.racc[a] += rw[BGW_RW_TARGET];     /* :52-53, it did not move */
        }
        ev.pstate[i] = p;
        mine |= p;
    }
    any = __syncthreads_or(mine);
    while (any) {
        for (int i = tid; i < nrank; i += T) {
            if (ev.pstate[i] != 1) continue;
            const int a = ev.ragent[i];
            atomicMin(slot_of(s, ev, ev.cell[a]), (uint32_t)i);
            atomicMin(slot_of(s, ev, ev.plist[i]), (uint32_t)i);
        }
        __syncthreads();
        for (int i = tid; i < nrank; i += T) {
            if (ev.pstate[i] != 1) continue;
            const int a = ev.ragent[i];
            if (*slot_of(s, ev, ev.cell[a]) == (uint32_t)i && *slot_of(s, ev, ev.plist[i]) == (uint32_t)i) ev.pstate[i] = 2;
        }
        __syncthreads();
        mine = 0;
        for (int i = tid; i < nrank; i += T) {
            if (ev.pstate[i] == 2) {
                const int a = ev.ragent[i], from = ev.cell[a], to = ev.plist[i];
                if (to != from) {
                    if (grid_query(s, ev, a, to)) { grid_unlink(ev, a); grid_append(ev, a, to); }
                    else ev.racc[a] += rw[BGW_RW_MOVE_FAIL];
                }
                if (reach) reach_check(s, ev, a);
                if (traffic && prog_done(s, ev, a)) ev.racc[a] += rw[BGW_RW_TARGET];
                *slot_of(s, ev, from) = BGW_SLOT_FREE;
                *slot_of(s, ev, to) = BGW_SLOT_FREE;
                ev.pstate[i] = 0;
            }
            mine |= ev.pstate[i];
        }
        any = __syncthreads_or(mine);
    }
    /* ---- entropy :58-59 ------------------------------------------------------------------------ */
    for (int i = tid; i < nrank && !traffic; i += T)
        if (ev.ragent[i] != BGW_NONE16 && (!reach || __ldg(&s.role[ev.ragent[i]]) == BGW_ROLE_RUNNER)) ev.racc[ev.ragent[i]] += rw[BGW_RW_ENTROPY];
    __syncthreads();
}

__device__ __forceinline__ bool same_position(const Env &ev, int a, int b) { return ev.cell[a] == ev.cell[b]; }

/* pacman.py:87-92,116-121: (9,0) <-> (9,20) through raw grid.remove / grid.place */
static __device__ void pacman_teleport(const DevSpec &s, Env &ev, int a)
{
    const int left = 9 * s.W, right = 9 * s.W + 20;
    const int dst = ev.cell[a] == left ? right : ev.cell[a] == right ? left : -1;
    if (dst < 0) return;
    grid_unlink(ev, a);
    if (grid_query(s, ev, a, dst)) grid_append(ev, a, dst);
}

/* pacman.py:94-105,123-131 (iterating a copy of the cell dict == reading `next` before touching the entry) */
static __device__ void pacman_overlaps(const DevSpec &s, Env &ev, int p, bool eat_food)
{
    if (!(ev.flags[p] & BGW_ST_IN_GRID)) return;
    unsigned nx;
    for (unsigned o = ev.head[ev.cell[p]]; o != BGW_NONE16; o = nx) {
        nx = ev.next[o];
        if ((int)o == p) continue;
        const int role = __ldg(&s.role[o]);
        if (eat_food && role == BGW_ROLE_FOOD) {
            ev.racc[p] += s.reward[BGW_RW_EAT_FOOD];
            grid_unlink(ev, (int)o);
            set_health(ev, (int)o, 0.0);
        } else if (role == BGW_ROLE_BADDIE) {
            ev.racc[p] += s.reward[BGW_RW_DIE];
            ev.racc[o] += s.reward[BGW_RW_KILL];
            set_health(ev, p, 0.0);
        }
    }
}

/* the rank-order programs run by one thread: maze_navigation.py:25-36, multi_maze_navigation.py:40-48,
 * pacman.py:80-135 */
static __device__ void serial_program_step(const DevSpec &s, Env &ev, int nrank)
{
    const double *rw = s.reward;
#define ACT(a) ev.act[(size_t)__ldg(&s.learner_of[(a)]) * s.act_words]
    if (s.program == BGW_PROG_MAZE) {
        const int nav = s.a_nav;
        if (!process_move(s, ev, nav, ACT(nav))) ev.racc[nav] += rw[BGW_RW_MOVE_FAIL];
        if (same_position(ev, s.a_nav, s.a_target)) ev.racc[nav] += rw[BGW_RW_TARGET];
        ev.racc[nav] += rw[BGW_RW_ENTROPY];
    } else if (s.program == BGW_PROG_MULTI_MAZE) {
        for (int i = 0; i < nrank; ++i) {
            const int a = ev.ragent[i];
            if (a == BGW_NONE16) continue;
            if (!process_move(s, ev, a, ACT(a))) ev.racc[a] += rw[BGW_RW_MOVE_FAIL];
            ev.racc[a] += rw[BGW_RW_ENTROPY];
        }
    } else if (s.program == BGW_PROG_PACMAN_SIMPLE) {                /* pacman.py:214-310 */
        const int p = s.a_pacman;
        if (!process_move(s, ev, p, ACT(p))) ev.racc[p] += rw[BGW_RW_MOVE_FAIL];
        else ev.racc[p] += rw[BGW_RW_ENTROPY];
        pacman_teleport(s, ev, p);
        if (!pacman_simple_overlaps(s, ev, p, true)) {
            int move[10];
            const int a156 = s.a_script[2], a159 = s.a_script[4];
            const int o156 = a156 >= 0 ? (ev.flags[a156] >> BGW_ST_ORIENT_SHIFT) & 7 : 0;
            const uint32_t x159 = a159 >= 0 ? dev_draw(s, ev, BGW_SITE_SCRIPT, (uint32_t)a159, 0) : 0u;
            pacman_script((int)ev.step - 1, o156, x159, move);
            for (int k = 0; k < 10; ++k) {
                const int a = s.a_script[k];
                if (a < 0) continue;
                process_move(s, ev, a, (uint32_t)move[k]);
                pacman_teleport(s, ev, a);
            }
            pacman_simple_overlaps(s, ev, p, false);
        }
    } else if (s.program == BGW_PROG_PACMAN) {
        const int p = s.a_pacman;
        if (!process_move(s, ev, p, ACT(p))) ev.racc[p] += rw[BGW_RW_MOVE_FAIL];
        else ev.racc[p] += rw[BGW_RW_ENTROPY];
        pacman_teleport(s, ev, p);
        pacman_overlaps(s, ev, p, true);
        for (int i = 0; i < nrank; ++i) {
            const int a = ev.ragent[i];
            if (a == BGW_NONE16 || a == p) continue;
            if (!process_move(s, ev, a, ACT(a))) ev.racc[a] += rw[BGW_RW_MOVE_FAIL];
            else ev.racc[a] += rw[BGW_RW_ENTROPY];
            pacman_teleport(s, ev, a);
        }
        pacman_overlaps(s, ev, p, false);
        if (!(ev.flags[p] & BGW_ST_ACTIVE)) grid_unlink(ev, p);      /* pacman.py:134-135 */
    }
#undef ACT
}

/* ------------------------------------------------------------------------------------------------- */
/* The sim's step / get_all_done / get_done / get_reward: built-in programs, done components         */
/* (done.py), or a user step program                                                                 */
/* ------------------------------------------------------------------------------------------------- */
#ifdef BGW_USER_PROGRAM
/* a user step program (include/bgw_program.h), compiled in at run time by bgw_set_program: defined after the program's
 * source (bgw_program.cuh).  The hooks return -1 when the program does not define them. */
static __device__ void user_step(const DevSpec &s, Env &ev, int nrank);
static __device__ int user_done(const DevSpec &s, const Env &ev, int a);
static __device__ int user_all_done(const DevSpec &s, const Env &ev);
static __device__ double user_reward(const DevSpec &s, const Env &ev, int a, double acc);
#endif

/* sim.step(action_dict); ranks 0..nrank-1 hold the acting agents (ragent).  All threads, ends synchronised */
__device__ __forceinline__ void prog_step(const DevSpec &s, Env &ev, int nrank, int tid, int T)
{
#ifdef BGW_USER_PROGRAM
    if (s.program == BGW_PROG_USER) { if (tid == 0) user_step(s, ev, nrank); __syncthreads(); return; }
#endif
    if (s.program == BGW_PROG_TEAM_BATTLE || s.program == BGW_PROG_REACH_TARGET || s.program == BGW_PROG_TRAFFIC) team_battle_step(s, ev, nrank, tid, T);
    else { if (tid == 0) serial_program_step(s, ev, nrank); __syncthreads(); }
}

/* get_all_done of the sim -> ctr[CTR_ALLDONE]; all threads, ends synchronised */
static __device__ void compute_all_done(const DevSpec &s, Env &ev, int tid, int T)
{
#ifdef BGW_USER_PROGRAM
    if (s.program == BGW_PROG_USER) {                               /* the program's get_all_done, else the rule below */
        if (tid == 0) ev.ctr[CTR_ALLDONE] = user_all_done(s, ev);
        __syncthreads();
        if (ev.ctr[CTR_ALLDONE] >= 0) return;
    }
#endif
    if (s.program == BGW_PROG_MAZE) {                                /* maze_navigation.py:41-42 */
        if (tid == 0) ev.ctr[CTR_ALLDONE] = same_position(ev, s.a_nav, s.a_target);
    } else if (s.program == BGW_PROG_PACMAN || s.program == BGW_PROG_PACMAN_SIMPLE) {   /* pacman.py:140-151 */
        if (tid == 0) ev.ctr[CTR_ALLDONE] = !(ev.flags[s.a_pacman] & BGW_ST_ACTIVE) ? 1 : (s.has_food ? 0 : 1);
    } else if (s.program == BGW_PROG_REACH_TARGET) {                 /* OnlyAgentLeftDone reach_the_target.py:43-57 */
        if (tid == 0) ev.ctr[CTR_AND] = 0;
        __syncthreads();
        int n = 0;
        for (int l = tid; l < s.L; l += T) n += (ev.flags[__ldg(&s.agent_of[l])] & BGW_ST_ACTIVE) ? 1 : 0;
        n = __reduce_add_sync(0xFFFFFFFFu, n);
        if ((tid & 31) == 0 && n) atomicAdd(&ev.ctr[CTR_AND], n);
        __syncthreads();
        if (tid == 0) ev.ctr[CTR_ALLDONE] = ev.ctr[CTR_AND] <= 1;
    } else {
        if (tid == 0) { ev.ctr[CTR_ENC_LO] = 0; ev.ctr[CTR_ENC_HI] = 0; ev.ctr[CTR_AND] = 1; }
        __syncthreads();
        uint32_t lo = 0, hi = 0;
        int ok = 1;
        for (int a = tid; a < s.A; a += T) {
            const bool active = ev.flags[a] & BGW_ST_ACTIVE;
            if (s.program == BGW_PROG_MULTI_MAZE) {                  /* multi_maze_navigation.py:66-71 */
                if (__ldg(&s.role[a]) == BGW_ROLE_NAVIGATOR && !same_position(ev, a, s.a_target)) ok = 0;
                continue;
            }
            if (active) { const int e = ev.enc[a]; if (e < 32) lo |= 1u << e; else hi |= 1u << (e - 32); }
            const int t = __ldg(&s.target[a]);
            if ((s.done_mask & BGW_DONE_TARGET_AGENT) && t >= 0 && !same_position(ev, a, t)) ok = 0;          /* done.py:93-99 */
            if ((s.done_mask & BGW_DONE_TARGET_DESTROYED) && t >= 0 && (ev.flags[t] & BGW_ST_ACTIVE)) ok = 0;  /* :133-137 */
        }
        lo = __reduce_or_sync(0xFFFFFFFFu, lo);
        hi = __reduce_or_sync(0xFFFFFFFFu, hi);
        ok = __all_sync(0xFFFFFFFFu, ok);
        if ((tid & 31) == 0) {
            if (lo) atomicOr((unsigned *)&ev.ctr[CTR_ENC_LO], lo);
            if (hi) atomicOr((unsigned *)&ev.ctr[CTR_ENC_HI], hi);
            if (!ok) atomicAnd((unsigned *)&ev.ctr[CTR_AND], 0u);
        }
        __syncthreads();
        if (tid == 0) {
            const unsigned long long encs = ((unsigned long long)(unsigned)ev.ctr[CTR_ENC_HI] << 32) | (unsigned)ev.ctr[CTR_ENC_LO];
            int d = ev.ctr[CTR_AND];
            if (s.program != BGW_PROG_MULTI_MAZE) {
                if (s.done_mask & BGW_DONE_ACTIVE) d &= (encs == 0);                    /* done.py:49-56   */
                if (s.done_mask & BGW_DONE_ONE_TEAM) d &= ((encs & (encs - 1)) == 0);   /* done.py:147-153 */
            }
            ev.ctr[CTR_ALLDONE] = d;
        }
    }
    __syncthreads();
}

/* get_done(agent): smart.py:106-111 / the programs' overrides */
__device__ __forceinline__ bool prog_done(const DevSpec &s, const Env &ev, int a)
{
#ifdef BGW_USER_PROGRAM
    if (s.program == BGW_PROG_USER) { const int u = user_done(s, ev, a); if (u >= 0) return u != 0; }
#endif
    switch (s.program) {
    case BGW_PROG_MAZE: case BGW_PROG_PACMAN: case BGW_PROG_PACMAN_SIMPLE: return ev.ctr[CTR_ALLDONE] != 0;   /* maze:38-39, pacman:137-138 */
    case BGW_PROG_MULTI_MAZE: return same_position(ev, a, s.a_target);              /* multi_maze:61-64 */
    case BGW_PROG_REACH_TARGET:                                                     /* reach_the_target.py:161-168 */
        if (__ldg(&s.role[a]) == BGW_ROLE_RUNNER) return !(ev.flags[a] & BGW_ST_ACTIVE) || (a != s.a_target && same_position(ev, a, s.a_target));
        return a == s.a_target && ev.ctr[CTR_ALLDONE] != 0;
    default: {
        bool d = true;
        const int t = __ldg(&s.target[a]);
        if (s.done_mask & (BGW_DONE_ACTIVE | BGW_DONE_ONE_TEAM)) d &= !(ev.flags[a] & BGW_ST_ACTIVE);               /* done.py:43-47 */
        if (s.done_mask & BGW_DONE_TARGET_AGENT) d &= (t >= 0 && same_position(ev, a, t));                           /* :87-91 */
        if (s.done_mask & BGW_DONE_TARGET_DESTROYED) d &= (t >= 0 && !(ev.flags[t] & BGW_ST_ACTIVE));                /* :130-131 */
        return d;
    }
    }
}

/* get_reward(agent) of an agent whose get_done is dd: read-and-zero smart.py:101-104, the MultiMaze override
 * multi_maze_navigation.py:56-59, the program's hook */
__device__ __forceinline__ double prog_take_reward(const DevSpec &s, Env &ev, int a, bool dd)
{
    double r = ev.racc[a];
    if (s.program == BGW_PROG_MULTI_MAZE && dd) r = s.reward[BGW_RW_TARGET];
#ifdef BGW_USER_PROGRAM
    if (s.program == BGW_PROG_USER) r = user_reward(s, ev, a, r);
#endif
    ev.racc[a] = 0.0;
    return r;
}

/* ------------------------------------------------------------------------------------------------- */
/* Observers: observer.py                                                                            */
/* ------------------------------------------------------------------------------------------------- */
/* np.random.choice over the encodings of a cell's occupants in arrival order (observer.py:131-134,234-236,
 * 240-248); a one-element list needs no draw (keyed stream) */
static __device__ int choose_encoding(const DevSpec &s, const Env &ev, int observer, int cell, int skip)
{
    int n = 0;
    for (unsigned o = ev.head[cell]; o != BGW_NONE16; o = ev.next[o]) n += ((int)o != skip);
    if (n == 0) return 0;
    int k = (n == 1) ? 0 : (int)bgw_index(dev_draw(s, ev, BGW_SITE_OBS, (uint32_t)observer, (uint32_t)cell), (uint32_t)n);
    for (unsigned o = ev.head[cell]; o != BGW_NONE16; o = ev.next[o]) {
        if ((int)o == skip) continue;
        if (k-- == 0) return ev.enc[o];
    }
    return 0;
}

__device__ __forceinline__ int view_range_eff(const DevSpec &s, int a)
{
    int R = __ldg(&s.view_r[a]);
    if (s.observer == BGW_OBS_ABSOLUTE) R = min(R, max(s.H, s.W) - 1);   /* cells off the grid are never read */
    return R;
}

/* AbsoluteEncodingObserver whose view covers the whole grid (pacman): the 16 cells of a chunk are the 16 summary
 * bytes themselves, with masked cells turned into -2 by a byte mask expanded from the line-of-sight bits and the
 * observer's own cell into -1 (observer.py:125-139); the few cells that hold mixed encodings are resolved one by one. */
__device__ __forceinline__ bool obs_chunk_absolute_whole(const DevSpec &s, const Env &ev, int a, int ch, const uint32_t *maskp, uint32_t out[4])
{
    const int k0 = ch * 16, R = view_range_eff(s, a), n = 2 * R + 1;
    const uint4 v = *reinterpret_cast<const uint4 *>(ev.csum + k0);
    uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t mixed = 0;                                                       /* bit t: cell k0 + t holds mixed encodings */
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint32_t hi = w[j] & 0x80808080u;                               /* BGW_CSUM_MIXED = 0x80 (encodings are < 64) */
        mixed |= (((hi >> 7) * 0x00204081u) >> 21 & 0xFu) << (4 * j);
    }
    if (k0 + 16 > s.HW) mixed &= (1u << (s.HW - k0)) - 1u;
    const int own = ev.cell[a];
    if ((ev.flags[a] & BGW_ST_IN_GRID) && own >= k0 && own < k0 + 16) {      /* "myself" :130-131 (the cell is occupied: by a) */
        const int t = own - k0;
        w[t >> 2] |= 0xFFu << ((t & 3) * 8);
    }
    if (maskp) {
        const int r0 = own / s.W, c0 = own % s.W;
        uint32_t vis = 0;                                                     /* bit t: cell k0 + t is visible */
        int k = k0;
        const int kend = min(k0 + 16, s.HW);
        while (k < kend) {                                                    /* one grid row segment at a time */
            const int gr = k / s.W, gc = k - gr * s.W, len = min(kend - k, s.W - gc);
            const int bit0 = (gr - r0 + R) * n + (gc - c0 + R), wi = bit0 >> 5, sh = bit0 & 31;
            const uint32_t lo = maskp[wi], hi = (sh + len > 32) ? maskp[wi + 1] : 0u;
            const uint32_t bits = __funnelshift_r(lo, hi, sh) & ((1u << len) - 1u);
            vis |= bits << (k - k0);
            k += len;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t m4 = (vis >> (4 * j)) & 0xFu;
            const uint32_t bytes = ((m4 * 0x00204081u) & 0x01010101u) * 0xFFu;      /* bit i -> byte i all ones */
            w[j] = (w[j] & bytes) | (0xFEFEFEFEu & ~bytes);                    /* masked: -2 :135-136 */
        }
    }
    if (k0 + 16 > s.HW) {                                                     /* row padding after the last cell */
#pragma unroll
        for (int t = 0; t < 16; ++t) if (k0 + t >= s.HW) w[t >> 2] &= ~(0xFFu << ((t & 3) * 8));
    }
    for (uint32_t m = mixed; m; m &= m - 1) {                                 /* np.random.choice over the occupants :133-134 */
        const int t = __ffs(m) - 1, sh = (t & 3) * 8;
        if (((w[t >> 2] >> sh) & 0xFFu) != 0x80u) continue;                   /* masked (-2) or myself (-1) */
        const uint32_t e = (uint32_t)(uint8_t)(int8_t)choose_encoding(s, ev, a, k0 + t, -1);
        w[t >> 2] = (w[t >> 2] & ~(0xFFu << sh)) | (e << sh);
    }
    out[0] = w[0]; out[1] = w[1]; out[2] = w[2]; out[3] = w[3];
    return true;
}

/* 16 consecutive bytes [ch*16, ch*16+16) of learner-agent a's observation row */
static __device__ void obs_chunk(const DevSpec &s, const Env &ev, int a, int ch, const uint32_t *maskp, uint32_t out[4])
{
    out[0] = out[1] = out[2] = out[3] = 0;
    if (!(ev.klass[a] & BGW_AG_OBSERVING)) return;                 /* get_obs returns {} observer.py:103,213,301 */
    const int R = view_range_eff(s, a), n = 2 * R + 1;
    const int own = ev.cell[a], r0 = own / s.W, c0 = own % s.W;
    const bool in_own = ev.flags[a] & BGW_ST_IN_GRID;
    const int k0 = ch * 16;
    if (s.observer == BGW_OBS_ABSOLUTE) {                           /* observer.py:95-150 */
        if (R >= max(s.H, s.W) - 1 && k0 < s.HW && obs_chunk_absolute_whole(s, ev, a, ch, maskp, out)) return;
        const int valid = s.HW;
        int gr = k0 / s.W, gc = k0 % s.W;
        for (int t = 0; t < 16 && k0 + t < valid; ++t) {
            const int wr = gr - r0 + R, wc = gc - c0 + R;
            int v;
            if (wr < 0 || wr >= n || wc < 0 || wc >= n) v = -2;                           /* :139 */
            else if (maskp && !((maskp[(wr * n + wc) >> 5] >> ((wr * n + wc) & 31)) & 1u)) v = -2;   /* :135-136 */
            else {
                const int cell = gr * s.W + gc;
                v = ev.csum[cell];                                                        /* 0 = empty :127-128 */
                if (v != 0 && in_own && cell == own) v = -1;                              /* :130-131 */
                else if (v == BGW_CSUM_MIXED) v = choose_encoding(s, ev, a, cell, -1);    /* :133-134 */
            }
            out[t >> 2] |= (uint32_t)(uint8_t)(int8_t)v << ((t & 3) * 8);
            if (++gc == s.W) { gc = 0; ++gr; }
        }
        return;
    }
    const int C = s.obs_c, valid = n * n * C;                       /* observer.py:204-250, 292-334 */
    int cidx = k0 / C, ech = k0 % C, wr = cidx / n, wc = cidx % n;
    for (int t = 0; t < 16 && k0 + t < valid; ++t) {
        const int gr = r0 - R + wr, gc = c0 - R + wc;
        int v;
        if (maskp && !((maskp[(wr * n + wc) >> 5] >> ((wr * n + wc) & 31)) & 1u)) v = -2;   /* mask first :226,248 */
        else if (gr < 0 || gr >= s.H || gc < 0 || gc >= s.W) v = -1;                        /* :228-229 */
        else {
            const int cell = gr * s.W + gc;
            if (s.observer == BGW_OBS_POSITION_CENTERED) {
                v = ev.csum[cell];                                                          /* 0 = empty :230-231 */
                if (v == BGW_CSUM_MIXED || (v != 0 && !s.observe_self && cell == own))
                    v = choose_encoding(s, ev, a, cell, s.observe_self ? -1 : a);           /* :233-246 */
            } else {                                                                        /* :316-326 */
                v = 0;
                if (ev.csum[cell] != 0) {
                    for (unsigned o = ev.head[cell]; o != BGW_NONE16; o = ev.next[o]) v += (ev.enc[o] == ech + 1);
                    v = min(v, 127);
                }
            }
        }
        out[t >> 2] |= (uint32_t)(uint8_t)(int8_t)v << ((t & 3) * 8);
        if (++ech == C) { ech = 0; if (++wc == n) { wc = 0; ++wr; } }
    }
}

/* Observations of the learners listed in plist[0..ne) -> obs rows of this env.  All threads. */
static __device__ void observe_learners(const DevSpec &s, Env &ev, int ne, int8_t *obs_env, int tid, int T)
{
    const int nch = s.nchunks;
    const bool blk = s.n_blk > 0;
    const int batch = blk ? s.mask_batch : ne;
    /* per-cell summary of the occupant lists: the observers read one byte per cell and only walk a list when the
     * cell holds mixed encodings (np.random.choice, observer.py:131-134,233-236) or counts are wanted */
    for (int i = tid; i < s.HW; i += T) ev.csum[i] = 0;
    __syncthreads();
    for (int a = tid; a < s.A; a += T) if (ev.flags[a] & BGW_ST_IN_GRID) ev.csum[ev.cell[a]] = ev.enc[a];
    __syncthreads();
    for (int a = tid; a < s.A; a += T)
        if ((ev.flags[a] & BGW_ST_IN_GRID) && ev.csum[ev.cell[a]] != ev.enc[a]) ev.csum[ev.cell[a]] = (int8_t)BGW_CSUM_MIXED;
    __syncthreads();
    for (int base = 0; base < ne; base += batch) {
        const int nb = min(batch, ne - base);
        if (blk) {
            /* view-blocking entities that never move, die or get re-placed (walls) hide the same cells from a given
             * viewer cell in every env and every step: their combined mask comes from a table built at bgw_create;
             * only the dynamic blockers are traced here */
            const int nblk = s.static_mask ? s.n_dyn_blk : s.n_blk;
            for (int w = tid; w < nb * s.mask_words; w += T) {
                uint32_t v = 0xFFFFFFFFu;
                if (s.static_mask) {
                    const int li = w / s.mask_words, a = __ldg(&s.agent_of[ev.plist[base + li]]), c = ev.cell[a];
                    if (c < s.HW) v = __ldg(&s.static_mask[(size_t)c * s.mask_words + (w - li * s.mask_words)]);
                }
                ev.mask[w] = v;
            }
            __syncthreads();
            for (int it = tid; it < nb * nblk; it += T) {
                const int li = it / nblk, b = __ldg(&s.blk_agents[it % nblk]);
                const int a = __ldg(&s.agent_of[ev.plist[base + li]]);
                if (!(ev.klass[a] & BGW_AG_OBSERVING)) continue;
                los_pair<true>(s, ev, ev.mask + (size_t)li * s.mask_words, ev.cell[a], view_range_eff(s, a), b,
                               s.observer == BGW_OBS_ABSOLUTE);
            }
            __syncthreads();
        }
        for (int it = tid; it < nb * nch; it += T) {
            const int li = it / nch, ch = it % nch;
            const int l = ev.plist[base + li], a = __ldg(&s.agent_of[l]);
            uint32_t w[4];
            obs_chunk(s, ev, a, ch, blk ? ev.mask + (size_t)li * s.mask_words : nullptr, w);
            if (s.ammo_offset >= 0 && ch == (s.ammo_offset >> 4) && (ev.klass[a] & BGW_AG_AMMO) && ev.ammo)   /* AmmoObserver observer.py:406-413 */
                w[(s.ammo_offset & 15) >> 2] = (uint32_t)ev.ammo[a];
            if (s.position_offset >= 0 && ch == (s.position_offset >> 4)) {      /* AbsolutePositionObserver observer.py:366-373 */
                const unsigned cell = ev.cell[a];
                w[(s.position_offset & 15) >> 2] = (cell / (unsigned)s.W) | ((cell % (unsigned)s.W) << 16);
            }
            *reinterpret_cast<uint4 *>(obs_env + (size_t)l * s.obs_stride + ch * 16) = make_uint4(w[0], w[1], w[2], w[3]);
        }
        if (blk) __syncthreads();
    }
}

/* ------------------------------------------------------------------------------------------------- */
/* State components: state.py                                                                        */
/* ------------------------------------------------------------------------------------------------- */
/* AllStepManager.reset / TurnBasedManager.reset -> sim.reset(): PositionState.reset state.py:88-166,
 * HealthState.reset :629-641, OrientationState.reset :666-675, rewards = 0 smart.py:91, done_agents =
 * non-learners all_step_manager.py:41-44.  All threads; ends synchronised with lists built. */
static __device__ void sim_reset(const DevSpec &s, const BgwState &st, Env &ev, int tid, int T)
{
    const int e = ev.e;
    ev.episode = __ldcg(&st.episode[e]) + 1u;
    ev.step = 0;
    __syncthreads();                       /* every thread has read episode[e] */
    if (tid == 0) { st.episode[e] = ev.episode; st.step[e] = 0; ev.ctr[CTR_ERR] = 0; }
    for (int a = tid; a < s.A; a += T) { ev.enc[a] = __ldg(&s.enc[a]); ev.klass[a] = __ldg(&s.klass[a]); ev.racc[a] = 0.0; }

    if (st.layout) {
        /* externally generated placement (MazePlacementState run host-side, state.py:487-527) */
        const uint16_t *lay = st.layout + (size_t)e * s.A;
        for (int a = tid; a < s.A; a += T) { ev.cell[a] = BGW_NONE16; ev.next[a] = BGW_NONE16; ev.flags[a] = 0; }
        for (int i = tid; i < (s.HW + 1) / 2; i += T) ((uint32_t *)ev.head)[i] = 0xFFFFFFFFu;
        __syncthreads();
        if (tid == 0)
            for (int a = 0; a < s.A; ++a) { if (lay[a] != BGW_NONE16) grid_append(ev, a, lay[a]); else ev.ctr[CTR_ERR] = 2; }   /* no cell: state.py:598-603 */
        __syncthreads();
    } else {
        for (int a = tid; a < s.A; a += T) {
            ev.cell[a] = __ldg(&s.tpl_cell[a]); ev.next[a] = __ldg(&s.tpl_next[a]); ev.flags[a] = __ldg(&s.tpl_flags[a]);
        }
        for (int i = tid; i < (s.max_enc + 1) * s.hw_words; i += T) ev.avail[i] = __ldg(&s.tpl_avail[i]);
        if (tid == 0) ev.ctr[CTR_ERR] = s.tpl_error;
        /* scratch in the reward accumulators' storage (8 A bytes, zeroed again below): 4 A bytes of draws, then the
         * placement order as uint16 [A] */
        uint32_t *xs = reinterpret_cast<uint32_t *>(ev.racc);
        uint16_t *ord = reinterpret_cast<uint16_t *>(xs + s.A);
        if (s.randomize_placement_order) {
            /* PositionState(randomize_placement_order) state.py:97-101: random.shuffle of the agents dict = the keyed order
             * of the episode (bgw_philox.h): entity a goes to the rank of (its key, a) among all entities.  The env-independent
             * template stays valid for which cells the fixed-position entities occupy and which remain available (both do
             * not depend on the order), but not for the ARRIVAL order inside a shared cell: their lists are rebuilt. */
            for (int a = tid; a < s.A; a += T) { xs[a] = dev_draw(s, ev, BGW_SITE_PLACE_ORDER, (uint32_t)a, 0); ev.next[a] = BGW_NONE16; }
            for (int i = tid; i < (s.HW + 1) / 2; i += T) ((uint32_t *)ev.head)[i] = 0xFFFFFFFFu;
            __syncthreads();
            for (int a = tid; a < s.A; a += T) {
                const uint32_t k = xs[a];
                int rank = 0;
                for (int b = 0; b < s.A; ++b) { const uint32_t kb = xs[b]; rank += (kb < k) || (kb == k && b < a); }
                ord[rank] = (uint16_t)a;
            }
            __syncthreads();
            if (tid == 0)
                for (int i = 0; i < s.A; ++i) {
                    const int a = ord[i], cell = __ldg(&s.tpl_cell[a]);
                    if (cell != BGW_NONE16) grid_append(ev, a, cell);
                }
            __syncthreads();
        } else {
            __syncthreads();
            build_heads(s, ev, tid, T);
        }
        /* the placement draws are keyed by the entity, not by the state: all threads precompute them so the serial chain
         * holds no Philox rounds */
        for (int vi = tid; vi < s.n_var; vi += T) { const int a = __ldg(&s.var_agents[vi]); xs[a] = dev_draw(s, ev, BGW_SITE_PLACE, (uint32_t)a, 0); }
        __syncthreads();
        if (tid < 32 && s.n_var > 0) {
            /* variable-position entities in dict order (state.py:112-114,152-166), or in the episode's shuffled order:
             * uniform choice over the ascending list of cells still available to the entity's encoding == select the
             * k-th set bit */
            const int lane = tid, per = (s.hw_words + 31) / 32;
            const int w0 = lane * per, w1 = min(s.hw_words, (lane + 1) * per);
            const int n_iter = s.randomize_placement_order ? s.A : s.n_var;
            int err = ev.ctr[CTR_ERR];
            int a_next = s.randomize_placement_order ? (int)ord[0] : (int)__ldg(&s.var_agents[0]);
            for (int vi = 0; vi < n_iter; ++vi) {
                const int a = a_next, en = ev.enc[a];
                if (vi + 1 < n_iter) a_next = s.randomize_placement_order ? (int)ord[vi + 1] : (int)__ldg(&s.var_agents[vi + 1]);
                if (s.randomize_placement_order && __ldg(&s.tpl_cell[a]) != BGW_NONE16) continue;   /* placed with the fixed ones */
                const uint32_t x = xs[a];
                uint32_t *av = ev.avail + (size_t)en * s.hw_words;
                int cnt = 0;
                for (int w = w0; w < w1; ++w) cnt += __popc(av[w]);
                int incl = cnt;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xFFFFFFFFu, incl, d); if (lane >= d) incl += t; }
                const int total = __shfl_sync(0xFFFFFFFFu, incl, 31);
                if (total == 0) { if (!err) err = 2; continue; }          /* RuntimeError state.py:161 */
                const int k = (int)bgw_index(x, (uint32_t)total);
                const int excl = incl - cnt;
                int cell = -1;
                if (k >= excl && k < incl) {
                    int rem = k - excl;
                    for (int w = w0; w < w1; ++w) {
                        uint32_t bits = av[w];
                        const int pc = __popc(bits);
                        if (rem < pc) {                                    /* rem-th set bit of this word */
                            int pos = 0, t;
                            t = __popc(bits & 0xFFFFu); if (rem >= t) { rem -= t; pos += 16; bits >>= 16; }
                            t = __popc(bits & 0xFFu);   if (rem >= t) { rem -= t; pos += 8;  bits >>= 8; }
                            t = __popc(bits & 0xFu);    if (rem >= t) { rem -= t; pos += 4;  bits >>= 4; }
                            t = __popc(bits & 0x3u);    if (rem >= t) { rem -= t; pos += 2;  bits >>= 2; }
                            if (rem >= (int)(bits & 1u)) pos += 1;
                            cell = w * 32 + pos;
                            break;
                        }
                        rem -= pc;
                    }
                }
                const unsigned src = __ballot_sync(0xFFFFFFFFu, cell >= 0);
                cell = __shfl_sync(0xFFFFFFFFu, cell, __ffs(src) - 1);
                if (lane == 0) grid_append(ev, a, cell);
                /* _update_available_positions state.py:126-141 */
                const unsigned long long row = __ldg(&s.overlap[en]);
                for (int e2 = 1 + lane; e2 <= s.max_enc; e2 += 32)
                    if (s.no_overlap || !((row >> e2) & 1ull)) ev.avail[(size_t)e2 * s.hw_words + (cell >> 5)] &= ~(1u << (cell & 31));
                __syncwarp();
            }
            if (lane == 0) ev.ctr[CTR_ERR] = err;
        }
        __syncthreads();
    }
    for (int a = tid; a < s.A; a += T) {
        ev.racc[a] = 0.0;                                             /* rewards = 0 (smart.py:91); also clears the draw scratch */
        uint8_t f = ev.flags[a] | BGW_ST_ACTIVE;                      /* PrincipleAgent.active = True */
        double h = 0.0;
        if (ev.klass[a] & BGW_AG_HEALTH) {                            /* HealthState.reset state.py:635-641 */
            h = __ldg(&s.init_health[a]);
            if (h != h) h = bgw_u01(dev_draw(s, ev, BGW_SITE_HEALTH, (uint32_t)a, 0));
            h = h < 0.0 ? 0.0 : h;
            h = h > 1.0 ? 1.0 : h;
            if (!(h > 0.0)) f &= ~BGW_ST_ACTIVE;
        }
        ev.health[a] = h;
        if (ev.klass[a] & BGW_AG_ORIENT) {                            /* OrientationState.reset state.py:670-675 */
            int o = __ldg(&s.init_orient[a]);
            if (!o) o = 1 + (int)bgw_index(dev_draw(s, ev, BGW_SITE_ORIENT, (uint32_t)a, 0), 4);
            f = (uint8_t)((f & 0x8F) | (o << BGW_ST_ORIENT_SHIFT));
        }
        if (!(ev.klass[a] & BGW_AG_LEARNER)) f |= BGW_ST_DONE_REPORTED;   /* all_step_manager.py:41-44 */
        if (ev.ammo) ev.ammo[a] = ((ev.klass[a] & BGW_AG_AMMO) && s.init_ammo) ? __ldg(&s.init_ammo[a]) : 0;   /* AmmoState.reset state.py:649-656 */
        ev.flags[a] = f;
    }
    __syncthreads();
}

/* store the staged agent arrays back to HBM */
static __device__ void store_env(const DevSpec &s, const BgwState &st, const Env &ev, bool with_racc, int tid, int T)
{
    const size_t off = (size_t)ev.e * s.A;
    for (int a = tid; a < s.A; a += T) {
        st.cell[off + a] = ev.cell[a];
        st.next[off + a] = ev.next[a];
        st.flags[off + a] = ev.flags[a];
        if (with_racc || racc_persists(ev.klass[a])) st.reward_acc[off + a] = ev.racc[a];
    }
}

/* reset one env and emit its first observations (all_step_manager.py:37-49, turn_based_manager.py:22-32) */
static __device__ void env_reset(const DevSpec &s, const BgwState &st, Env &ev, int8_t *obs_env, int tid, int T)
{
    sim_reset(s, st, ev, tid, T);
    int ne;
    if (s.manager == BGW_MANAGER_TURN_BASED) {
        int t = st.turn[ev.e];
        t = (t + 1) % s.L;                                           /* next(self.agent_order), never rewound :17-20 */
        __syncthreads();
        if (tid == 0) { st.turn[ev.e] = (int16_t)t; ev.plist[0] = (uint16_t)t; }
        ne = 1;
    } else if (s.manager == BGW_MANAGER_DYNAMIC_ORDER) {             /* dynamic_order_manager.py:19-28: sim.reset names the first agent */
        __syncthreads();
        if (tid == 0) { st.turn[ev.e] = 0; ev.plist[0] = 0; }
        ne = 1;
    } else {
        for (int l = tid; l < s.L; l += T) ev.plist[l] = (uint16_t)l;
        ne = s.L;
    }
    __syncthreads();
    if (ev.ctr[CTR_ERR]) {
        /* the placement failed (the reference raises, state.py:147-149,161): some entity has no cell, nothing may act on
         * this env.  It is reported BGW_ENV_ERROR | BGW_ENV_ALL_DONE with zero observations and stays inert until it is
         * reset again (auto-reset: by the next step, with the next episode's draws). */
        if (obs_env)
            for (int it = tid; it < ne * s.nchunks; it += T)
                *reinterpret_cast<uint4 *>(obs_env + (size_t)ev.plist[it / s.nchunks] * s.obs_stride + (it % s.nchunks) * 16) = make_uint4(0, 0, 0, 0);
    } else if (obs_env) observe_learners(s, ev, ne, obs_env, tid, T);
    store_env(s, st, ev, true, tid, T);
    if (tid == 0) st.error[ev.e] = (uint32_t)ev.ctr[CTR_ERR];
}

/* ------------------------------------------------------------------------------------------------- */
/* kernels                                                                                           */
/* ------------------------------------------------------------------------------------------------- */
extern __shared__ __align__(16) unsigned char bgw_smem[];

/* The library is built from three translation units so that they compile in parallel and a change to one kernel family
 * does not rebuild the others: bgw.cu (host side, small kernels), bgw_general.cu (bgw_step_kernel instantiations) and
 * bgw_fastk.cu (bgw_step_fast_kernel instantiations).  The kernel TUs hand their entry points to the host side: */
typedef void (*GeneralStepFn)(const DevSpec, const BgwState, const uint32_t *, const int16_t *, int8_t *, float *, uint8_t *, uint8_t *);
#ifndef __CUDACC_RTC__
GeneralStepFn bgw_general_step_fn(int program, int attack_actor);   /* bgw_general.cu; (-1, -1) = every program and actor in one */
const void *bgw_fast_step_fn(int shape, int head_elem);              /* bgw_fastk.cu; shape 0 run-time, 1 FastStaticC5, 2 FastStaticC2 */
#endif

#ifdef BGW_SMALL_KERNELS   /* non-template kernels: defined in exactly one translation unit (bgw.cu) */
__global__ void bgw_reset_kernel(const DevSpec s, const BgwState st, const uint8_t *env_mask, int8_t *obs)
{
    const int e = blockIdx.x, tid = threadIdx.x, T = blockDim.x;
    if (env_mask && !env_mask[e]) return;
    Env ev;
    env_init(ev, s, bgw_smem);
    ev.e = e; ev.genv = (uint32_t)(s.env_offset + e);
    ev.health = st.health + (size_t)e * s.A;
    ev.ammo = st.ammo ? st.ammo + (size_t)e * s.A : nullptr;
    env_reset(s, st, ev, obs ? obs + (size_t)e * s.L * s.obs_stride : nullptr, tid, T);
    if (tid == 0) st.env_flags[e] = (uint8_t)(ev.ctr[CTR_ERR] ? BGW_ENV_ERROR | BGW_ENV_ALL_DONE : 0);
}


/* GridWorldSimulation.get_obs(agent_id) (sim/gridworld/base.py; the observers of sim/gridworld/observer.py) for EVERY learner of
 * the selected envs, on the state as it stands in HBM: nothing is stepped, no state is written.  The random choice among
 * the encodings of a shared cell (observer.py:131-134,233-236) is keyed by the env's current step, so the rows equal the
 * ones the last reset / step wrote for the learners it reported. */
__global__ void bgw_observe_kernel(const DevSpec s, const BgwState st, const uint8_t *env_mask, int8_t *obs)
{
    const int e = blockIdx.x, tid = threadIdx.x, T = blockDim.x;
    if (env_mask && !env_mask[e]) return;
    Env ev;
    env_init(ev, s, bgw_smem);
    ev.e = e; ev.genv = (uint32_t)(s.env_offset + e);
    ev.health = st.health + (size_t)e * s.A;
    ev.ammo = st.ammo ? st.ammo + (size_t)e * s.A : nullptr;
    ev.episode = st.episode[e];
    ev.step = st.step[e];
    const size_t off = (size_t)e * s.A;
    for (int a = tid; a < s.A; a += T) {
        ev.cell[a] = st.cell[off + a]; ev.next[a] = st.next[off + a]; ev.flags[a] = st.flags[off + a];
        ev.enc[a] = __ldg(&s.enc[a]); ev.klass[a] = __ldg(&s.klass[a]);
    }
    for (int l = tid; l < s.L; l += T) ev.plist[l] = (uint16_t)l;
    __syncthreads();
    build_heads(s, ev, tid, T);
    observe_learners(s, ev, s.L, obs + (size_t)e * s.L * s.obs_stride, tid, T);
}

#endif

/* The step kernel is instantiated per sim program (and, for the team battle, per attack actor): PROG / ATT >= 0 overwrite
 * the corresponding spec fields with compile-time constants, so the dispatch on them folds and every instantiation holds
 * only its own program's code.  One CTA of one or two warps per env runs at its own place in the code; the all-in-one
 * instantiation <-1, -1> is 26 k instructions (415 KB) and waits for instruction fetches most of the time. */
template <int PROG, int ATT>
__device__ __forceinline__ void bgw_step_body(const DevSpec &s_in, const BgwState &st, const uint32_t *actions, const int16_t *order,
                                              int8_t *obs, float *reward, uint8_t *done, uint8_t *all_done)
{
    DevSpec s = s_in;
    if (PROG >= 0) s.program = PROG;
    if (ATT >= 0) s.attack_actor = ATT;
#ifdef BGW_JIT_PIN
    BGW_JIT_PIN        /* run-time compilation for one spec (bgw_jit.cpp): the spec's scalars as compile-time constants */
#endif
#ifdef BGW_JIT_T
    const int e = blockIdx.x, tid = threadIdx.x, T = BGW_JIT_T;
#else
    const int e = blockIdx.x, tid = threadIdx.x, T = blockDim.x;
#endif
    Env ev;
    env_init(ev, s, bgw_smem);
    ev.e = e; ev.genv = (uint32_t)(s.env_offset + e);
    ev.health = st.health + (size_t)e * s.A;
    ev.ammo = st.ammo ? st.ammo + (size_t)e * s.A : nullptr;
    int8_t *obs_env = obs ? obs + (size_t)e * s.L * s.obs_stride : nullptr;
    float *rew = reward + (size_t)e * s.L;
    uint8_t *dn = done + (size_t)e * s.L;
    const uint8_t ef0 = st.env_flags[e];

    if (ef0 & BGW_ENV_ALL_DONE) {
        for (int l = tid; l < s.L; l += T) { dn[l] = 0; rew[l] = 0.f; }
        if (s.auto_reset) {
            env_reset(s, st, ev, obs_env, tid, T);
            if (tid == 0) {
                const uint8_t f = (uint8_t)((ev.ctr[CTR_ERR] ? BGW_ENV_ERROR | BGW_ENV_ALL_DONE : 0) | BGW_ENV_RESET);
                st.env_flags[e] = f; all_done[e] = f;
            }
        } else if (tid == 0) all_done[e] = ef0;
        return;
    }

    /* ---- stage the env ---------------------------------------------------------------------- */
    const size_t off = (size_t)e * s.A;
    const bool dynamic = s.manager == BGW_MANAGER_DYNAMIC_ORDER;
    const bool turn_based = s.manager == BGW_MANAGER_TURN_BASED || dynamic;   /* one acting learner per step: BgwState.turn */
    ev.episode = st.episode[e];
    ev.step = st.step[e] + 1u;
    for (int a = tid; a < s.A; a += T) {
        ev.cell[a] = st.cell[off + a]; ev.next[a] = st.next[off + a]; ev.flags[a] = st.flags[off + a];
        ev.enc[a] = __ldg(&s.enc[a]); ev.klass[a] = __ldg(&s.klass[a]);
        ev.racc[a] = (turn_based || racc_persists(ev.klass[a])) ? st.reward_acc[off + a] : 0.0;
    }
    for (int w = tid; w < s.L * s.act_words; w += T) ev.act[w] = actions[(size_t)e * s.L * s.act_words + w];
    for (int i = tid; i <= s.slot_mask; i += T) ev.slot[i] = BGW_SLOT_FREE;
    if (tid < CTR_COUNT) ev.ctr[tid] = 0;
    __syncthreads();
    build_heads(s, ev, tid, T);

    /* ---- acting agents by rank ---------------------------------------------------------------- */
    int nrank, turn = 0;
    if (!turn_based) {                                              /* all_step_manager.py:59-66 */
        nrank = s.L;
        for (int i = tid; i < s.L; i += T) {
            const int l = order ? order[(size_t)e * s.L + i] : i;
            const int a = __ldg(&s.agent_of[l]);
            ev.ragent[i] = (ev.flags[a] & BGW_ST_DONE_REPORTED) ? (uint16_t)BGW_NONE16 : (uint16_t)a;
        }
    } else {                                                        /* turn_based_manager.py:46 */
        nrank = 1;
        turn = st.turn[e];
        if (tid == 0) ev.ragent[0] = (uint16_t)__ldg(&s.agent_of[turn]);
    }
    __syncthreads();

    prog_step(s, ev, nrank, tid, T);                                /* sim.step(action_dict) */
    compute_all_done(s, ev, tid, T);

    /* ---- who receives (obs, reward, done) -------------------------------------------------------- */
    if (!turn_based) {                                              /* all_step_manager.py:68-87 */
        for (int l = tid; l < s.L; l += T) {
            const int a = __ldg(&s.agent_of[l]);
            uint8_t d = 0; float r = 0.f;
            if (!(ev.flags[a] & BGW_ST_DONE_REPORTED)) {
                ev.plist[atomicAdd(&ev.ctr[CTR_NEMIT], 1)] = (uint16_t)l;
                const bool dd = prog_done(s, ev, a);
                r = (float)prog_take_reward(s, ev, a, dd);
                d = (uint8_t)(BGW_OUT_VALID | (dd ? BGW_OUT_DONE : 0));
                if (dd) ev.flags[a] |= BGW_ST_DONE_REPORTED;
                else atomicAdd(&ev.ctr[CTR_REMAINING], 1);
            }
            dn[l] = d; rew[l] = r;
        }
        __syncthreads();
        if (tid == 0) ev.ctr[CTR_ENVDONE] = ev.ctr[CTR_ALLDONE] || ev.ctr[CTR_REMAINING] == 0;   /* :90-93 */
    } else {                                                        /* turn_based_manager.py:48-92 */
        for (int l = tid; l < s.L; l += T) { dn[l] = 0; rew[l] = 0.f; }
        __syncthreads();
        if (tid == 0) {
            int env_done = ev.ctr[CTR_ALLDONE], ne = 0, l = turn;
            if (env_done) {                                         /* :49-57 (dynamic_order_manager.py:43-51 alike) */
                for (int k = 0; k < s.L; ++k)
                    if (!(ev.flags[__ldg(&s.agent_of[k])] & BGW_ST_DONE_REPORTED)) ev.plist[ne++] = (uint16_t)k;
            } else if (dynamic) {
                /* dynamic_order_manager.py:52-85 over next_agent = [the agent that acted, if this step finished it] + [the next
                 * agent in dict order that is not done] (examples: DynamicOrderMultiMazeSim.step) */
                const int a0 = __ldg(&s.agent_of[turn]);
                if (prog_done(s, ev, a0)) { ev.plist[ne++] = (uint16_t)turn; ev.flags[a0] |= BGW_ST_DONE_REPORTED; }   /* :60-69 (someone is not done: no __all__) */
                for (int k = 1; k <= s.L; ++k) {
                    l = (turn + k) % s.L;
                    const int a = __ldg(&s.agent_of[l]);
                    if (prog_done(s, ev, a)) continue;                /* the sim's rule skips the agents that are done */
                    if (!(ev.flags[a] & BGW_ST_DONE_REPORTED)) ev.plist[ne++] = (uint16_t)l;      /* :80-85 */
                    break;
                }
                st.turn[e] = (int16_t)l;
            } else {
                for (;;) {                                          /* :59-92 */
                    l = (l + 1) % s.L;
                    const int a = __ldg(&s.agent_of[l]);
                    if (ev.flags[a] & BGW_ST_DONE_REPORTED) continue;
                    ev.plist[ne++] = (uint16_t)l;
                    if (prog_done(s, ev, a)) {
                        ev.flags[a] |= BGW_ST_DONE_REPORTED;
                        int remaining = 0;
                        for (int k = 0; k < s.L; ++k) remaining += !(ev.flags[__ldg(&s.agent_of[k])] & BGW_ST_DONE_REPORTED);
                        if (remaining) continue;
                        env_done = 1;
                    }
                    break;
                }
                st.turn[e] = (int16_t)l;
            }
            ev.ctr[CTR_NEMIT] = ne;
            ev.ctr[CTR_ENVDONE] = env_done;
        }
        __syncthreads();
        for (int i = tid; i < ev.ctr[CTR_NEMIT]; i += T) {
            const int l = ev.plist[i], a = __ldg(&s.agent_of[l]);
            const bool dd = prog_done(s, ev, a);
            rew[l] = (float)prog_take_reward(s, ev, a, dd);
            dn[l] = (uint8_t)(BGW_OUT_VALID | (dd ? BGW_OUT_DONE : 0));
        }
        __syncthreads();
    }
    const int ne = ev.ctr[CTR_NEMIT];
    if (obs_env) observe_learners(s, ev, ne, obs_env, tid, T);
    store_env(s, st, ev, turn_based, tid, T);

    if (tid == 0) {
        uint8_t ef = 0;
        if (ev.ctr[CTR_ENVDONE]) ef |= BGW_ENV_ALL_DONE;
        if (s.horizon > 0 && (int)ev.step >= s.horizon) ef |= BGW_ENV_ALL_DONE | BGW_ENV_TRUNCATED;
#ifdef BGW_USER_PROGRAM
        if (ev.ctr[CTR_ERR]) { ef |= BGW_ENV_ERROR | BGW_ENV_ALL_DONE; st.error[e] = (uint32_t)ev.ctr[CTR_ERR]; }   /* bad input from the program */
#endif
        st.step[e] = ev.step;
        st.env_flags[e] = ef;
        all_done[e] = ef;
        unsigned long long *sr = (unsigned long long *)st.stats + (size_t)e * BGW_STAT_COUNT;
        sr[BGW_STAT_AGENT_STEPS] += (unsigned long long)ne;
        sr[BGW_STAT_ENV_STEPS] += 1ull;
        if (ev.ctr[CTR_KILLS]) sr[BGW_STAT_KILLS] += (unsigned long long)ev.ctr[CTR_KILLS];
        if (ef & BGW_ENV_ALL_DONE) sr[BGW_STAT_EPISODES] += 1ull;
    }
}

/* the stock instantiations (bgw_general.cu); a run-time compilation for one spec (bgw_specialize, bgw_jit.h) wraps the same
 * body in a kernel of its own */
template <int PROG, int ATT>
__global__ void __launch_bounds__(256, 3) bgw_step_kernel(const DevSpec s_in,   /* <= 80 registers: what the all-in-one kernel needs */ const BgwState st, const uint32_t *actions, const int16_t *order,
                                int8_t *obs, float *reward, uint8_t *done, uint8_t *all_done)
{
    bgw_step_body<PROG, ATT>(s_in, st, actions, order, obs, reward, done, all_done);
}

/* RandomPolicy.compute_action = action_space.sample() (policies/policy.py:81-92) on the keyed stream: one
 * Philox block per (env, step, agent); words 0,1 -> move, word 2 -> attack. */
__device__ __forceinline__ uint32_t sample_action_word(const DevSpec &s, int a, int klass, uint32_t genv, uint32_t episode,
                                                       uint32_t step)
{
    uint32_t x[4];
    bgw_draw4(s.seed, genv, episode, step, BGW_SITE_ACTION, (uint32_t)a, 0, x);
    uint32_t o = 0;
    if (klass & BGW_AG_MOVING) {
        if (s.move_actor == BGW_MOVE_BOX) {                          /* Box(-m, m, (2,), int) actor.py:63-65 */
            const int m = __ldg(&s.move_r[a]), w = 2 * m + 1;
            const int dr = (int)bgw_index(x[0], (uint32_t)w) - m, dc = (int)bgw_index(x[1], (uint32_t)w) - m;
            if (s.ravel) o = (uint32_t)((dr + m) * w + (dc + m)) & 0xFF;
            else o = ((uint32_t)(uint8_t)(int8_t)dr) | ((uint32_t)(uint8_t)(int8_t)dc << 8);
        } else if (s.move_actor != BGW_MOVE_NONE) {                  /* Discrete(5) actor.py:125 */
            o = bgw_index(x[0], 5);
        }
    }
    if ((klass & BGW_AG_ATTACKING) && s.attack_actor == BGW_ATTACK_BINARY)
        o |= (bgw_index(x[2], (uint32_t)__ldg(&s.simatt[a]) + 1) & 0xFF) << 16;   /* Discrete(n+1) actor.py:452 */
    return o;
}

#ifdef BGW_SMALL_KERNELS
/* one thread per (env, learner).  The wider attack actions (EncodingBased / RestrictedSelective / Selective): attack
 * byte j draws word j%4 of the Philox block k = 1 + j/4 of the same (env, step, agent) key. */
__global__ void bgw_sample_actions_kernel(const DevSpec s, const BgwState st, uint32_t *actions)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)s.E * s.L) return;
    const int e = (int)(i / s.L), l = (int)(i % s.L), a = __ldg(&s.agent_of[l]);
    const int klass = __ldg(&s.klass[a]);
    const uint32_t genv = (uint32_t)(s.env_offset + e), episode = st.episode[e], step = st.step[e];
    uint32_t *row = actions + i * s.act_words;
    row[0] = sample_action_word(s, a, klass, genv, episode, step);
    for (int w = 1; w < s.act_words; ++w) row[w] = 0;
    if (!(klass & BGW_AG_ATTACKING) || s.attack_actor <= BGW_ATTACK_BINARY) return;
    const uint32_t sim = __ldg(&s.simatt[a]);
    const int n = 2 * __ldg(&s.attack_r[a]) + 1;
    const int width = s.attack_actor == BGW_ATTACK_ENCODING ? s.max_enc : s.attack_actor == BGW_ATTACK_RESTRICTED ? (int)sim : n * n;
    const unsigned long long map_row = __ldg(&s.attack_map[__ldg(&s.enc[a])]);
    uint32_t x[4];
    for (int j = 0; j < width; ++j) {
        if ((j & 3) == 0) bgw_draw4(s.seed, genv, episode, step, BGW_SITE_ACTION, (uint32_t)a, 1u + ((uint32_t)j >> 2), x);
        uint32_t v;
        if (s.attack_actor == BGW_ATTACK_ENCODING) v = ((map_row >> (j + 1)) & 1ull) ? bgw_index(x[j & 3], sim + 1) : 0;   /* actor.py:513-519 */
        else if (s.attack_actor == BGW_ATTACK_RESTRICTED) v = bgw_index(x[j & 3], (uint32_t)(n * n) + 1);                  /* :593-599 */
        else v = bgw_index(x[j & 3], sim + 1);                                                                            /* :669-679 */
        row[(2 + j) >> 2] |= (v & 0xFFu) << (((2 + j) & 3) * 8);
    }
}

/* AllStepManager(randomize_action_input) all_step_manager.py:62-65 on the device: order[e][0..L) = the learners of env e in
 * the keyed order of the step about to be taken (include/bgw_philox.h, BGW_SITE_ORDER): sorted by (first Philox word of the
 * agent's key, agent index).  The step kernels drop the learners already reported done while they walk the row, and the
 * keyed order of a sub-list is the sub-list of the keyed order, so the row serves whatever subset submits actions.
 * One CTA per env, bitonic sort of (key << 32 | learner) in shared memory (P = L rounded up to a power of two). */
__global__ void bgw_order_kernel(const DevSpec s, const BgwState st, int P, int16_t *order)
{
    extern __shared__ __align__(16) unsigned long long bgw_order_keys[];
    const int e = blockIdx.x, tid = threadIdx.x, T = blockDim.x;
    const uint32_t genv = (uint32_t)(s.env_offset + e), episode = st.episode[e], step = st.step[e] + 1u;
    for (int l = tid; l < P; l += T) {
        unsigned long long v = ~0ull;                               /* padding sorts last */
        if (l < s.L) {
            const int a = __ldg(&s.agent_of[l]);
            v = ((unsigned long long)bgw_draw(s.seed, genv, episode, step, BGW_SITE_ORDER, (uint32_t)a, 0) << 32) | (unsigned)l;
        }
        bgw_order_keys[l] = v;
    }
    __syncthreads();
    for (int k = 2; k <= P; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < P; i += T) {
                const int p = i ^ j;
                if (p > i) {
                    const unsigned long long x = bgw_order_keys[i], y = bgw_order_keys[p];
                    if (((i & k) == 0) ? (x > y) : (x < y)) { bgw_order_keys[i] = y; bgw_order_keys[p] = x; }
                }
            }
            __syncthreads();
        }
    for (int i = tid; i < s.L; i += T) order[(size_t)e * s.L + i] = (int16_t)(bgw_order_keys[i] & 0xFFFFu);
}

/* bgw_gather_valid: one CTA per env; rows are claimed with one global atomicAdd per env and copied as 16-byte chunks */
__global__ void bgw_gather_kernel(int L, int obs_stride, const int8_t *obs, const float *reward, const uint8_t *done,
                                  const uint8_t *all_done, int *count, int *index, int8_t *obs_c, float *reward_c,
                                  uint8_t *done_c)
{
    extern __shared__ __align__(16) unsigned char gsm[];
    int *sc = (int *)gsm;                 /* [0] rows of this env, [1] base in the compacted buffers */
    uint16_t *list = (uint16_t *)(gsm + 16);
    const int e = blockIdx.x, tid = threadIdx.x, T = blockDim.x;
    const bool whole = all_done[e] & BGW_ENV_RESET;
    const uint8_t *dn = done + (size_t)e * L;
    if (tid == 0) sc[0] = 0;
    __syncthreads();
    for (int l = tid; l < L; l += T)
        if (whole || (dn[l] & BGW_OUT_VALID)) list[atomicAdd(&sc[0], 1)] = (uint16_t)l;
    __syncthreads();
    const int n = sc[0];
    if (n == 0) return;
    if (tid == 0) sc[1] = atomicAdd(count, n);
    __syncthreads();
    const int base = sc[1], nch = obs_stride >> 4;
    for (int i = tid; i < n; i += T) {
        const int l = list[i];
        index[base + i] = e * L + l;
        reward_c[base + i] = reward[(size_t)e * L + l];
        done_c[base + i] = dn[l];
    }
    const uint4 *src = (const uint4 *)(obs + (size_t)e * L * obs_stride);
    uint4 *dst = (uint4 *)(obs_c + (size_t)base * obs_stride);
    for (int it = tid; it < n * nch; it += T) {
        const int i = it / nch, ch = it - i * nch;
        dst[(size_t)i * nch + ch] = src[(size_t)list[i] * nch + ch];
    }
}
#endif  /* BGW_SMALL_KERNELS */
