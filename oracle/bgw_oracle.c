/*
 * bgw_oracle.c -- CPU ORACLE (scalar, sequential, plain C).  TEST INFRASTRUCTURE ONLY -- see bgw_oracle.h.
 *
 * Every function restates one piece of the reference (gillette7/Abmarl 0.2.7) and cites it.  The reference
 * keeps each grid cell as an insertion-ordered dict {id: agent} (grid.py:24,79,125); here that dict is a
 * doubly linked list threaded through the entities (head/tail per cell, next/prev per entity), which
 * preserves arrival order -- the only property of the dict the algorithms observe.
 *
 * Build:  gcc -O2 -fPIC -shared -ffp-contract=off -o oracle/libbgw_oracle.so oracle/bgw_oracle.c
 * (-ffp-contract=off: the line-of-sight rays must be evaluated as (a/b)*t in IEEE float64, no FMA.)
 */
#include "bgw_oracle.h"
#include "../include/bgw_philox.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#define NONE 0xFFFFu

typedef struct {
    const BgwSpec *sp;
    BgwState *st;
    int H, W, A, L, HW, max_enc;
    int env;          /* local env index */
    uint32_t genv;    /* global env index (Philox) */
    /* views into the env's state rows */
    uint16_t *cell, *next;
    uint8_t *flags;
    double *health, *racc;
    int32_t *ammo;    /* NULL when the state has no ammo array */
    int astride;      /* bytes per learner action row */
    uint8_t *acc_occ; /* [A] how often the current attacker evaluated each candidate this step (ACC draw key) */
    /* work arrays */
    uint16_t *head, *tail, *prev;
    int *learner_of;  /* [A] learner index or -1 */
    int *agent_of;    /* [L] agent index */
    uint8_t *mask;    /* LOS scratch */
    int mask_cap;
    /* the step in progress (bgwo_step) */
    int *acting;      /* [n_acting] agent per acting slot in processing order, -1 = reported done already */
    int n_acting;
    const int8_t *actions;   /* this env's action rows */
    uint32_t err;     /* bad input from a step program: BgwState.error at the end of the step (the step kernel's CTR_ERR) */
} Ctx;

/* ------------------------------------------------------------------------------------------------- */
/* sizes                                                                                             */
/* ------------------------------------------------------------------------------------------------- */
static int count_learners(const BgwSpec *sp)
{
    int n = 0;
    for (int a = 0; a < sp->n_agents; ++a) n += (sp->klass[a] & BGW_AG_LEARNER) ? 1 : 0;
    return n;
}

static int max_encoding(const BgwSpec *sp)
{
    int m = 0;
    for (int a = 0; a < sp->n_agents; ++a) if (sp->encoding[a] > m) m = sp->encoding[a];
    return m;
}

/* bytes of one learner's action row: 2 move bytes + the widest attack action (layout: bgw.h, bgw_step) */
static int action_stride_of(const BgwSpec *sp)
{
    int payload = 1;                                                        /* Discrete(n+1) actor.py:452 */
    for (int a = 0; a < sp->n_agents; ++a) {
        if (!(sp->klass[a] & BGW_AG_ATTACKING)) continue;
        const int n = 2 * sp->attack_range[a] + 1;
        int w = 1;
        if (sp->attack_actor == BGW_ATTACK_ENCODING) w = max_encoding(sp);             /* Dict per encoding :513-519 */
        else if (sp->attack_actor == BGW_ATTACK_RESTRICTED) w = sp->simultaneous_attacks[a];   /* MultiDiscrete :593-599 */
        else if (sp->attack_actor == BGW_ATTACK_SELECTIVE) w = n * n;                  /* Box (n, n) :669-679 */
        if (w > payload) payload = w;
    }
    return (2 + payload + 3) / 4 * 4;
}

int bgwo_dims(const BgwSpec *sp, BgwDims *d)
{
    memset(d, 0, sizeof(*d));
    d->n_envs = sp->n_envs; d->n_agents = sp->n_agents; d->n_learners = count_learners(sp);
    int rmax = 0;
    for (int a = 0; a < sp->n_agents; ++a)
        if ((sp->klass[a] & BGW_AG_LEARNER) && (sp->klass[a] & BGW_AG_OBSERVING) && sp->view_range[a] > rmax)
            rmax = sp->view_range[a];
    d->obs_c = 1;
    if (sp->observer == BGW_OBS_ABSOLUTE) { d->obs_h = sp->rows; d->obs_w = sp->cols; }   /* observer.py:74 */
    else { d->obs_h = d->obs_w = 2 * rmax + 1; }                                          /* observer.py:170,266 */
    if (sp->observer == BGW_OBS_STACKED) d->obs_c = max_encoding(sp);                     /* observer.py:264 */
    int n = d->obs_h * d->obs_w * d->obs_c;
    d->ammo_offset = -1;
    if (sp->ammo_observer) { d->ammo_offset = (n + 3) / 4 * 4; n = d->ammo_offset + 4; }   /* observer.py:376-413 */
    d->position_offset = -1;
    if (sp->position_observer) { d->position_offset = (n + 3) / 4 * 4; n = d->position_offset + 4; }   /* observer.py:337-373 */
    d->obs_stride = (n + 15) / 16 * 16;
    d->action_stride = action_stride_of(sp);
    return 0;
}

/* ------------------------------------------------------------------------------------------------- */
/* Grid: grid.py                                                                                     */
/* ------------------------------------------------------------------------------------------------- */
/* rebuild head/tail/prev from the persisted per-entity `next` pointers */
static void grid_build(Ctx *c)
{
    for (int i = 0; i < c->HW; ++i) c->head[i] = c->tail[i] = NONE;
    for (int a = 0; a < c->A; ++a) c->prev[a] = NONE;
    for (int a = 0; a < c->A; ++a)
        if ((c->flags[a] & BGW_ST_IN_GRID) && c->next[a] != NONE) c->prev[c->next[a]] = (uint16_t)a;
    for (int a = 0; a < c->A; ++a) {
        if (!(c->flags[a] & BGW_ST_IN_GRID)) continue;
        if (c->next[a] == NONE) c->tail[c->cell[a]] = (uint16_t)a;
        if (c->prev[a] == NONE) c->head[c->cell[a]] = (uint16_t)a;
    }
}

/* Grid.reset grid.py:73-79 */
static void grid_clear(Ctx *c)
{
    for (int i = 0; i < c->HW; ++i) c->head[i] = c->tail[i] = NONE;
    for (int a = 0; a < c->A; ++a) { c->prev[a] = NONE; c->next[a] = NONE; c->flags[a] &= ~BGW_ST_IN_GRID; }
}

/* Grid.query grid.py:81-105: empty, or every occupant's encoding in overlapping[agent.encoding]
 * (a missing key is an all-zero row: KeyError -> False) */
static int grid_query(const Ctx *c, int a, int cell)
{
    uint64_t row = c->sp->overlap[c->sp->encoding[a]];
    for (uint16_t o = c->head[cell]; o != NONE; o = c->next[o])
        if (!((row >> c->sp->encoding[o]) & 1)) return 0;
    return 1;
}

/* the dict insert of Grid.place grid.py:124-126 (no query) */
static void grid_insert(Ctx *c, int a, int cell)
{
    c->next[a] = NONE;
    c->prev[a] = c->tail[cell];
    if (c->tail[cell] != NONE) c->next[c->tail[cell]] = (uint16_t)a; else c->head[cell] = (uint16_t)a;
    c->tail[cell] = (uint16_t)a;
    c->cell[a] = (uint16_t)cell;
    c->flags[a] |= BGW_ST_IN_GRID;
}

/* Grid.place grid.py:107-129 */
static int grid_place(Ctx *c, int a, int cell)
{
    if (!grid_query(c, a, cell)) return 0;
    grid_insert(c, a, cell);
    return 1;
}

/* Grid.remove grid.py:131-140 (the entity's `position` attribute is left as is) */
static void grid_remove(Ctx *c, int a)
{
    if (!(c->flags[a] & BGW_ST_IN_GRID)) return;
    int cell = c->cell[a];
    uint16_t p = c->prev[a], n = c->next[a];
    if (p != NONE) c->next[p] = n; else c->head[cell] = n;
    if (n != NONE) c->prev[n] = p; else c->tail[cell] = p;
    c->next[a] = NONE; c->prev[a] = NONE;
    c->flags[a] &= ~BGW_ST_IN_GRID;
}

/* HealthAgent.health setter agent.py:192-196 */
static void set_health(Ctx *c, int a, double v)
{
    double h = v < 0.0 ? 0.0 : v;
    h = h > 1.0 ? 1.0 : h;
    c->health[a] = h;
    if (h > 0.0) c->flags[a] |= BGW_ST_ACTIVE; else c->flags[a] &= ~BGW_ST_ACTIVE;
}

/* ------------------------------------------------------------------------------------------------- */
/* create_grid_and_mask: the mask part, utils.py:45-115                                              */
/* ------------------------------------------------------------------------------------------------- */
/* Zero the cells of `mask` ((2R+1)^2, row-major, offset (r,c) at [(r+R)*(2R+1) + c+R]) hidden behind a
 * blocker at offset (rd, cd).  The eight branches of the reference collapse to two families:
 *  - cd != 0 : march over columns away from the viewer starting at cd; a cell (r,c) is hidden when
 *              lower(c) < r < upper(c) with  upper(t) = (rd+0.5)/du * t,  lower(t) = (rd-0.5)/dl * t,
 *              where du/dl are the blocker's near/far column edges cd-+0.5 chosen per quadrant;
 *  - cd == 0 : same with rows and columns exchanged.
 * Arithmetic is float64 (a/b)*t with strict comparisons, as the reference evaluates it.
 * [rlo,rhi]x[clo,chi] additionally clips the visited offsets (cells outside are never read by the caller). */
static void los_apply(uint8_t *mask, int R, int rd, int cd, int rlo, int rhi, int clo, int chi)
{
    const int n = 2 * R + 1;
    if (rd == 0 && cd == 0) return;              /* matches no branch of utils.py:52-115 */
    if (rlo < -R) rlo = -R;
    if (rhi > R) rhi = R;
    if (clo < -R) clo = -R;
    if (chi > R) chi = R;
    if (cd != 0) {
        double du, dl;
        if (rd == 0) { du = dl = (cd > 0) ? (double)cd - 0.5 : (double)cd + 0.5; }   /* utils.py:53-54,89-90 */
        else if ((rd > 0) == (cd > 0)) { du = (double)cd - 0.5; dl = (double)cd + 0.5; } /* :62-63,98-99 */
        else { du = (double)cd + 0.5; dl = (double)cd - 0.5; }                          /* :80-81,107-108 */
        const double ku = ((double)rd + 0.5) / du, kl = ((double)rd - 0.5) / dl;
        int c0 = cd > 0 ? cd : clo, c1 = cd > 0 ? chi : cd;
        if (cd > 0 && c0 < clo) c0 = clo;
        if (cd < 0 && c1 > chi) c1 = chi;
        int r0 = rd > 0 ? rd : rlo, r1 = rd < 0 ? rd : rhi;
        if (r0 < rlo) r0 = rlo;
        if (r1 > rhi) r1 = rhi;
        for (int c = c0; c <= c1; ++c) {
            const double up = ku * (double)c, lo = kl * (double)c;
            for (int r = r0; r <= r1; ++r) {
                if (c == cd && r == rd) continue;     /* don't mask the blocker itself */
                if (lo < (double)r && (double)r < up) mask[(r + R) * n + (c + R)] = 0;
            }
        }
    } else {
        const double d = rd > 0 ? (double)rd - 0.5 : (double)rd + 0.5;                  /* utils.py:71-72,116-117 */
        const double kl = ((double)cd - 0.5) / d, kr = ((double)cd + 0.5) / d;
        int r0 = rd > 0 ? rd : rlo, r1 = rd > 0 ? rhi : rd;
        if (r0 < rlo) r0 = rlo;
        if (r1 > rhi) r1 = rhi;
        for (int r = r0; r <= r1; ++r) {
            const double le = kl * (double)r, ri = kr * (double)r;
            for (int c = clo; c <= chi; ++c) {
                if (c == cd && r == rd) continue;
                if (le < (double)c && (double)c < ri) mask[(r + R) * n + (c + R)] = 0;
            }
        }
    }
}

int bgwo_los_mask(int range, int rd, int cd, uint8_t *out)
{
    const int n = 2 * range + 1;
    memset(out, 1, (size_t)n * n);
    if (rd < -range || rd > range || cd < -range || cd > range) return 0;   /* utils.py:49-50 */
    los_apply(out, range, rd, cd, -range, range, -range, range);
    return 0;
}

/* mask for agent `a` at `range`: every active & blocking entity of the sim within +-range  utils.py:45-51 */
static uint8_t *los_mask_for(Ctx *c, int a, int R, int clip_to_grid)
{
    const int n = 2 * R + 1;
    if (n * n > c->mask_cap) { c->mask_cap = n * n; c->mask = (uint8_t *)realloc(c->mask, (size_t)c->mask_cap); }
    memset(c->mask, 1, (size_t)n * n);
    const int r0 = c->cell[a] / c->W, c0 = c->cell[a] % c->W;
    int rlo = -R, rhi = R, clo = -R, chi = R;
    if (clip_to_grid) { rlo = -r0; rhi = c->H - 1 - r0; clo = -c0; chi = c->W - 1 - c0; }
    for (int o = 0; o < c->A; ++o) {
        if (!(c->flags[o] & BGW_ST_ACTIVE) || !(c->sp->klass[o] & BGW_AG_BLOCKING)) continue;
        if (c->cell[o] == NONE) continue;
        const int rd = c->cell[o] / c->W - r0, cd = c->cell[o] % c->W - c0;
        if (rd < -R || rd > R || cd < -R || cd > R) continue;
        los_apply(c->mask, R, rd, cd, rlo, rhi, clo, chi);
    }
    return c->mask;
}

/* ------------------------------------------------------------------------------------------------- */
/* Observers: observer.py                                                                            */
/* ------------------------------------------------------------------------------------------------- */
static uint32_t step_of(const Ctx *c) { return c->st->step[c->env]; }
static uint32_t episode_of(const Ctx *c) { return c->st->episode[c->env]; }
static uint32_t draw(const Ctx *c, uint32_t site, uint32_t slot, uint32_t k)
{
    return bgw_draw(c->sp->seed, c->genv, episode_of(c), step_of(c), site, slot, k);
}

/* np.random.choice([other.encoding for other in cell.values() (if other is not `skip`)])
 * observer.py:131-134,234-236,240-248.  Returns 0 when the list is empty. */
static int choose_encoding(const Ctx *c, int observer, int cell, int skip)
{
    int n = 0;
    for (uint16_t o = c->head[cell]; o != NONE; o = c->next[o]) if ((int)o != skip) ++n;
    if (n == 0) return 0;
    int k = (n == 1) ? 0 : (int)bgw_index(draw(c, BGW_SITE_OBS, (uint32_t)observer, (uint32_t)cell), (uint32_t)n);
    for (uint16_t o = c->head[cell]; o != NONE; o = c->next[o]) {
        if ((int)o == skip) continue;
        if (k-- == 0) return c->sp->encoding[o];
    }
    return 0;
}

static void observe_agent(Ctx *c, int a, int8_t *out, int stride)
{
    const BgwSpec *sp = c->sp;
    memset(out, 0, (size_t)stride);
    if (sp->ammo_observer && (sp->klass[a] & BGW_AG_AMMO) && c->ammo) {      /* AmmoObserver.get_obs observer.py:406-413 */
        BgwDims dd; bgwo_dims(sp, &dd);
        const int32_t v = c->ammo[a];
        memcpy(out + dd.ammo_offset, &v, 4);
    }
    if (sp->position_observer) {                             /* AbsolutePositionObserver.get_obs observer.py:366-373: agent.position */
        BgwDims dd; bgwo_dims(sp, &dd);
        const int16_t rc[2] = {(int16_t)(c->cell[a] / c->W), (int16_t)(c->cell[a] % c->W)};
        memcpy(out + dd.position_offset, rc, 4);
    }
    if (!(sp->klass[a] & BGW_AG_OBSERVING)) return;          /* get_obs returns {} observer.py:103,213,301 */
    const int R = sp->view_range[a], n = 2 * R + 1;
    const int r0 = c->cell[a] / c->W, c0 = c->cell[a] % c->W;
    const int in_own_cell = (c->flags[a] & BGW_ST_IN_GRID) != 0;
    uint8_t *mask = los_mask_for(c, a, R, sp->observer == BGW_OBS_ABSOLUTE);

    if (sp->observer == BGW_OBS_ABSOLUTE) {                  /* observer.py:95-150 */
        memset(out, -2, (size_t)(c->H * c->W));               /* :139 */
        for (int r = 0; r < n; ++r) for (int cc = 0; cc < n; ++cc) {
            const int gr = r0 - R + r, gc = c0 - R + cc;
            if (gr < 0 || gr >= c->H || gc < 0 || gc >= c->W) continue;      /* cropped out :125-126,140-148 */
            const int cell = gr * c->W + gc;
            int v;
            if (!mask[r * n + cc]) v = -2;                                   /* :135-136 */
            else if (c->head[cell] == NONE) v = 0;                            /* :127-128 */
            else if (in_own_cell && cell == c->cell[a]) v = -1;               /* :130-131 */
            else v = choose_encoding(c, a, cell, -1);                         /* :133-134 */
            out[cell] = (int8_t)v;
        }
        return;
    }
    if (sp->observer == BGW_OBS_POSITION_CENTERED) {         /* observer.py:204-250 */
        for (int r = 0; r < n; ++r) for (int cc = 0; cc < n; ++cc) {
            const int gr = r0 - R + r, gc = c0 - R + cc;
            int v;
            if (!mask[r * n + cc]) v = -2;                                   /* mask is tested first :226,248 */
            else if (gr < 0 || gr >= c->H || gc < 0 || gc >= c->W) v = -1;   /* :228-229 */
            else {
                const int cell = gr * c->W + gc;
                if (c->head[cell] == NONE) v = 0;                             /* :230-231 */
                else v = choose_encoding(c, a, cell, sp->observe_self ? -1 : a);   /* :233-246 */
            }
            out[r * n + cc] = (int8_t)v;
        }
        return;
    }
    /* STACKED observer.py:292-334: channel e counts occupants with encoding e+1; layout [r][c][e] */
    const int C = c->max_enc;
    for (int r = 0; r < n; ++r) for (int cc = 0; cc < n; ++cc) {
        const int gr = r0 - R + r, gc = c0 - R + cc;
        for (int e = 0; e < C; ++e) {
            int v;
            if (!mask[r * n + cc]) v = -2;
            else if (gr < 0 || gr >= c->H || gc < 0 || gc >= c->W) v = -1;
            else {
                v = 0;
                for (uint16_t o = c->head[gr * c->W + gc]; o != NONE; o = c->next[o])
                    if (sp->encoding[o] == e + 1) ++v;
                if (v > 127) v = 127;
            }
            out[(r * n + cc) * C + e] = (int8_t)v;
        }
    }
}

/* ------------------------------------------------------------------------------------------------- */
/* Actors: actor.py                                                                                  */
/* ------------------------------------------------------------------------------------------------- */
static const int CROSS_DR[5] = {0, 0, 1, 0, -1};   /* CrossMoveActor.grid_action actor.py:153-159 */
static const int CROSS_DC[5] = {0, -1, 0, 1, 0};

/* the shared tail of MoveActor / CrossMoveActor.process_action  actor.py:99-114,177-194 */
static int try_move(Ctx *c, int a, int dr, int dc)
{
    const int r = c->cell[a] / c->W + dr, cc = c->cell[a] % c->W + dc;
    if (r < 0 || r >= c->H || cc < 0 || cc >= c->W) return 0;
    const int to = r * c->W + cc;
    if (to == c->cell[a]) return 1;
    if (!grid_query(c, a, to)) return 0;
    grid_remove(c, a);
    grid_place(c, a, to);
    return 1;
}

/* returns move_result as the user's step() sees it: 1 True, 0 False/None */
static int process_move(Ctx *c, int a, const int8_t *act)
{
    const BgwSpec *sp = c->sp;
    if (!(sp->klass[a] & BGW_AG_MOVING)) return 0;               /* returns None -> `not None` actor.py:98 */
    if (sp->move_actor == BGW_MOVE_BOX) {                         /* MoveActor actor.py:82-114 */
        int dr = act[0], dc = act[1];
        if (sp->ravel_actions) {      /* ActorWrapper.process_action -> unravel  wrapper.py:143-159,
                                         ravel_discrete_wrapper.py:90-92: unravel_index(a, high+1-low)+low */
            const int m = sp->move_range[a], w = 2 * m + 1, v = (uint8_t)act[0];
            dr = v / w - m; dc = v % w - m;
        }
        return try_move(c, a, dr, dc);
    }
    if (sp->move_actor == BGW_MOVE_CROSS) {                       /* actor.py:161-194 */
        const int k = act[0];
        return try_move(c, a, CROSS_DR[k], CROSS_DC[k]);
    }
    if (sp->move_actor == BGW_MOVE_DRIFT) {                       /* DriftMoveActor actor.py:208-234 */
        if (!(sp->klass[a] & BGW_AG_ORIENT)) return 0;
        const int k = act[0];
        if (k != 0 && try_move(c, a, CROSS_DR[k], CROSS_DC[k])) {
            c->flags[a] = (uint8_t)((c->flags[a] & 0x8F) | (k << BGW_ST_ORIENT_SHIFT));
            return 1;
        }
        const int o = (c->flags[a] >> BGW_ST_ORIENT_SHIFT) & 7;
        return try_move(c, a, CROSS_DR[o], CROSS_DC[o]);
    }
    return 0;
}

/* AttackActorBaseComponent._basic_criteria actor.py:381-392.  The accuracy draw is keyed by (attacker,
 * candidate, how often the pair was evaluated before in this call) -- see BGW_SITE_ACC. */
static int basic_criteria(Ctx *c, int attacker, int cand)
{
    const BgwSpec *sp = c->sp;
    if (cand == attacker) return 0;
    if (!(c->flags[cand] & BGW_ST_ACTIVE)) return 0;
    if (!((sp->attack_map[sp->encoding[attacker]] >> sp->encoding[cand]) & 1)) return 0;
    const uint32_t occ = c->acc_occ[cand]++;
    const double u = bgw_u01(draw(c, BGW_SITE_ACC, (uint32_t)attacker, (uint32_t)cand + 4096u * occ));
    if (u > sp->attack_accuracy[attacker]) return 0;
    return 1;
}

/* AttackActorBaseComponent._subset_attackables actor.py:394-414: appends the chosen agents to out[*nv..] */
static void subset_attackables(Ctx *c, int a, uint32_t group, int *cand, int ncand, int k, int *out, int *nv)
{
    const BgwSpec *sp = c->sp;
    if (!sp->stacked_attacks && k > ncand) {                      /* whole list, no draw :410-411 */
        for (int t = 0; t < ncand && *nv < BGW_MAX_VICTIMS; ++t) out[(*nv)++] = cand[t];
    } else if (sp->stacked_attacks) {                             /* choice with replacement */
        for (int t = 0; t < k && *nv < BGW_MAX_VICTIMS; ++t)
            out[(*nv)++] = cand[bgw_index(draw(c, BGW_SITE_SUBSET, (uint32_t)a, (group << 8) | (uint32_t)t), (uint32_t)ncand)];
    } else {
        /* choice without replacement == partial Fisher-Yates over the candidate list (the replay shim
         * implements np.random.choice(replace=False) the same way) */
        for (int t = 0; t < k; ++t) {
            int j = t + (int)bgw_index(draw(c, BGW_SITE_SUBSET, (uint32_t)a, (group << 8) | (uint32_t)t), (uint32_t)(ncand - t));
            int tmp = cand[t]; cand[t] = cand[j]; cand[j] = tmp;
            if (*nv < BGW_MAX_VICTIMS) out[(*nv)++] = cand[t];
        }
    }
}

/* candidates of one window cell (r, cc) of attacker a: visible, inside the grid, occupants in dict order that pass
 * _basic_criteria; optionally only those with encoding enc_only (> 0) */
static int cell_candidates(Ctx *c, int a, int R, const uint8_t *mask, int r, int cc, int *cand, int ncand)
{
    const int n = 2 * R + 1, r0 = c->cell[a] / c->W, c0 = c->cell[a] % c->W;
    if (!mask[r * n + cc]) return ncand;
    const int gr = r0 - R + r, gc = c0 - R + cc;
    if (gr < 0 || gr >= c->H || gc < 0 || gc >= c->W) return ncand;          /* local_grid[r, c] is None */
    for (uint16_t o = c->head[gr * c->W + gc]; o != NONE; o = c->next[o])
        if (basic_criteria(c, a, o) && ncand < c->A) cand[ncand++] = o;
    return ncand;
}

/* <Attack actor>._determine_attack + AttackActorBaseComponent.process_action (actor.py:306-361) for the four
 * attack actors (:455-501 Binary, :521-582 EncodingBased, :601-658 RestrictedSelective, :681-728 Selective).
 * `att` points at the attack bytes of the agent's action row (layout: bgw.h, bgw_step).  Returns attack_status;
 * victims[0..*nv) receives attacked_agents (at most BGW_MAX_VICTIMS, possibly with repeats). */
static int process_attack(Ctx *c, int a, const uint8_t *att, int *victims, int *nv)
{
    const BgwSpec *sp = c->sp;
    *nv = 0;
    if (!(sp->klass[a] & BGW_AG_ATTACKING)) return 0;             /* actor.py:360-361 */
    const int R = sp->attack_range[a], n = 2 * R + 1;
    int width = 1;
    if (sp->attack_actor == BGW_ATTACK_ENCODING) width = c->max_enc;
    else if (sp->attack_actor == BGW_ATTACK_RESTRICTED) width = sp->simultaneous_attacks[a];
    else if (sp->attack_actor == BGW_ATTACK_SELECTIVE) width = n * n;
    int any = 0;
    for (int j = 0; j < width; ++j) any |= att[j];
    if (!any) return 0;                                           /* actor.py:478-479,542-543,622-623,703-704 */
    memset(c->acc_occ, 0, (size_t)c->A);
    uint8_t *mask = los_mask_for(c, a, R, 0);                     /* gu.create_grid_and_mask */
    int *cand = (int *)malloc(sizeof(int) * (size_t)(c->A + 1));
    int ncand;
    switch (sp->attack_actor) {
    case BGW_ATTACK_BINARY:                                        /* actor.py:489-501 */
        ncand = 0;
        for (int r = 0; r < n; ++r) for (int cc = 0; cc < n; ++cc) ncand = cell_candidates(c, a, R, mask, r, cc, cand, ncand);
        if (ncand) subset_attackables(c, a, 0, cand, ncand, att[0], victims, nv);
        break;
    case BGW_ATTACK_ENCODING: {                                    /* actor.py:554-582: one scan, one list per encoding */
        int *all = (int *)malloc(sizeof(int) * (size_t)(c->A + 1));
        int nall = 0;
        for (int r = 0; r < n; ++r) for (int cc = 0; cc < n; ++cc) nall = cell_candidates(c, a, R, mask, r, cc, all, nall);
        for (int enc = 1; enc <= c->max_enc; ++enc) {             /* `for encoding, num_attacks in attack.items()`, ascending */
            if (!((sp->attack_map[sp->encoding[a]] >> enc) & 1)) continue;   /* not a key of the action space :513-519 */
            ncand = 0;
            for (int t = 0; t < nall; ++t) if (sp->encoding[all[t]] == enc) cand[ncand++] = all[t];
            if (ncand == 0) continue;                              /* :576-577 */
            subset_attackables(c, a, (uint32_t)enc, cand, ncand, att[enc - 1], victims, nv);
        }
        free(all);
        break;
    }
    case BGW_ATTACK_RESTRICTED:                                    /* actor.py:633-657 */
        for (int j = 0; j < width; ++j) {
            if (att[j] == 0) continue;                             /* :635-637 */
            const int rav = att[j] - 1, r = rav % n, cc = rav / n; /* :641-643 (row = remainder, column = quotient) */
            if (r >= n || cc >= n) continue;                       /* outside the action space */
            int *all = (int *)malloc(sizeof(int) * (size_t)(c->A + 1));
            const int nall = cell_candidates(c, a, R, mask, r, cc, all, 0);
            ncand = 0;
            for (int t = 0; t < nall; ++t) {                       /* :649-654 */
                int seen = 0;
                for (int q = 0; q < *nv; ++q) seen |= (victims[q] == all[t]);
                if (seen && !sp->stacked_attacks) continue;
                cand[ncand++] = all[t];
            }
            free(all);
            if (ncand && *nv < BGW_MAX_VICTIMS) {                  /* np.random.choice(attackable_agents) :655-656 */
                const uint32_t x = draw(c, BGW_SITE_SUBSET, (uint32_t)a, (uint32_t)*nv << 8);
                victims[(*nv)++] = cand[bgw_index(x, (uint32_t)ncand)];
            }
        }
        break;
    case BGW_ATTACK_SELECTIVE:                                     /* actor.py:711-727 */
        for (int r = 0; r < n; ++r) for (int cc = 0; cc < n; ++cc) {
            if (!att[r * n + cc]) continue;
            ncand = cell_candidates(c, a, R, mask, r, cc, cand, 0);
            if (ncand) subset_attackables(c, a, (uint32_t)(r * n + cc), cand, ncand, att[r * n + cc], victims, nv);
        }
        break;
    default: break;
    }
    free(cand);
    /* ammo filter actor.py:343-351 */
    if ((sp->klass[a] & BGW_AG_AMMO) && c->ammo) {
        int ammo = c->ammo[a];
        if (*nv > ammo) {                                          /* choice(size=ammo, replace=False): partial Fisher-Yates */
            for (int t = 0; t < ammo; ++t) {
                int j = t + (int)bgw_index(draw(c, BGW_SITE_AMMO, (uint32_t)a, (uint32_t)t), (uint32_t)(*nv - t));
                int tmp = victims[t]; victims[t] = victims[j]; victims[j] = tmp;
            }
            *nv = ammo;
        }
        ammo -= *nv;
        c->ammo[a] = ammo < 0 ? 0 : ammo;                          /* setter agent.py:306-309 */
    }
    /* actor.py:353-358 */
    for (int t = 0; t < *nv; ++t) {
        const int v = victims[t];
        if (!(c->flags[v] & BGW_ST_ACTIVE)) continue;
        set_health(c, v, c->health[v] - sp->attack_strength[a]);
        if (!(c->flags[v] & BGW_ST_ACTIVE)) { grid_remove(c, v); c->st->stats[(size_t)c->env * BGW_STAT_COUNT + BGW_STAT_KILLS]++; }
    }
    return 1;
}

/* ------------------------------------------------------------------------------------------------- */
/* Done components + sim-program overrides                                                           */
/* ------------------------------------------------------------------------------------------------- */
static int find_role(const Ctx *c, int role)
{
    for (int a = 0; a < c->A; ++a) if (c->sp->role[a] == role) return a;
    return -1;
}

static int same_position(const Ctx *c, int a, int b) { return c->cell[a] == c->cell[b]; }

static int prog_all_done(const Ctx *c);

#ifdef BGW_USER_PROGRAM
/* a user step program (include/bgw_program.h), compiled in by build_program (oracle/build.py): defined after the program's
 * source (bgw_oracle_program.c).  The hooks return -1 when the program does not define them. */
static void user_step(Ctx *c);
static int user_done(const Ctx *c, int a);
static int user_all_done(const Ctx *c);
static double user_reward(const Ctx *c, int a, double acc);
#endif

/* PacmanSimSimple.step pacman.py:235-303: the baddies' scripted DriftMoveActor actions for this step.  k indexes the
 * script's entries (baddie_20, 36, 156, 157, 159, 161, 162, 206, 222, 328); sc = step_count; o156 = orientation of
 * baddie_156; x159 = the keyed draw that stands in for np.random.randint(0, 5) */
static void pacman_script(int sc, int o156, uint32_t x159, int move[10])
{
    const int base[10] = {0, 0, 0, 1, 0, 3, 0, 0, 0, 0};
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

static int smart_done(const Ctx *c, int a)   /* SmartGridWorldSimulation.get_done smart.py:106-111 */
{
    const BgwSpec *sp = c->sp;
    int d = 1;
    if (sp->done_mask & (BGW_DONE_ACTIVE | BGW_DONE_ONE_TEAM)) d &= !(c->flags[a] & BGW_ST_ACTIVE);   /* done.py:43-47 */
    if (sp->done_mask & BGW_DONE_TARGET_AGENT) d &= (sp->target[a] >= 0 && same_position(c, a, sp->target[a])); /* :87-91 */
    if (sp->done_mask & BGW_DONE_TARGET_DESTROYED) d &= (sp->target[a] >= 0 && !(c->flags[sp->target[a]] & BGW_ST_ACTIVE)); /* :130-131 */
    return d;
}

static int smart_all_done(const Ctx *c)      /* smart.py:113-117 */
{
    const BgwSpec *sp = c->sp;
    int d = 1;
    if (sp->done_mask & BGW_DONE_ACTIVE) {                        /* done.py:49-56 */
        for (int a = 0; a < c->A; ++a) if (c->flags[a] & BGW_ST_ACTIVE) { d = 0; break; }
    }
    if (sp->done_mask & BGW_DONE_ONE_TEAM) {                      /* done.py:147-153 */
        uint64_t encs = 0;
        for (int a = 0; a < c->A; ++a) if (c->flags[a] & BGW_ST_ACTIVE) encs |= 1ull << sp->encoding[a];
        d &= (encs & (encs - 1)) == 0;
    }
    if (sp->done_mask & BGW_DONE_TARGET_AGENT)                    /* done.py:93-99 */
        for (int a = 0; a < c->A; ++a) if (sp->target[a] >= 0 && !same_position(c, a, sp->target[a])) d = 0;
    if (sp->done_mask & BGW_DONE_TARGET_DESTROYED)                /* done.py:133-137 */
        for (int a = 0; a < c->A; ++a) if (sp->target[a] >= 0 && (c->flags[sp->target[a]] & BGW_ST_ACTIVE)) d = 0;
    return d;
}

/* OnlyAgentLeftDone._agents_remaining reach_the_target.py:47-51: active learning agents */
static int learners_remaining(const Ctx *c)
{
    int n = 0;
    for (int l = 0; l < c->L; ++l) n += (c->flags[c->agent_of[l]] & BGW_ST_ACTIVE) ? 1 : 0;
    return n;
}

static int prog_done(const Ctx *c, int a)
{
#ifdef BGW_USER_PROGRAM
    if (c->sp->program == BGW_PROG_USER) { const int u = user_done(c, a); if (u >= 0) return u; }
#endif
    switch (c->sp->program) {
    case BGW_PROG_REACH_TARGET: {                                                   /* reach_the_target.py:161-168 */
        const int t = find_role(c, BGW_ROLE_TARGET);
        if (c->sp->role[a] == BGW_ROLE_RUNNER)                                      /* ActiveDone or TargetDone :26-40 */
            return !(c->flags[a] & BGW_ST_ACTIVE) || (a != t && same_position(c, a, t));
        if (a == t) return learners_remaining(c) <= 1;                              /* OnlyAgentLeftDone :53-54 */
        return 0;
    }
    case BGW_PROG_MAZE: return prog_all_done(c);                                    /* maze_navigation.py:38-39 */
    case BGW_PROG_MULTI_MAZE: return same_position(c, a, find_role(c, BGW_ROLE_TARGET)); /* multi_maze_navigation.py:61-64 */
    case BGW_PROG_PACMAN: case BGW_PROG_PACMAN_SIMPLE: return prog_all_done(c);     /* pacman.py:137-138 */
    default: return smart_done(c, a);
    }
}

static int prog_all_done(const Ctx *c)
{
#ifdef BGW_USER_PROGRAM
    if (c->sp->program == BGW_PROG_USER) { const int u = user_all_done(c); if (u >= 0) return u; }
#endif
    switch (c->sp->program) {
    case BGW_PROG_REACH_TARGET: return learners_remaining(c) <= 1;                  /* reach_the_target.py:170-171,56-57 */
    case BGW_PROG_MAZE:                                                             /* maze_navigation.py:41-42 */
        return same_position(c, find_role(c, BGW_ROLE_NAVIGATOR), find_role(c, BGW_ROLE_TARGET));
    case BGW_PROG_MULTI_MAZE: {                                                     /* multi_maze_navigation.py:66-71 */
        const int t = find_role(c, BGW_ROLE_TARGET);
        for (int a = 0; a < c->A; ++a)
            if (c->sp->role[a] == BGW_ROLE_NAVIGATOR && !same_position(c, a, t)) return 0;
        return 1;
    }
    case BGW_PROG_PACMAN: case BGW_PROG_PACMAN_SIMPLE: {                            /* pacman.py:140-151 */
        const int p = find_role(c, BGW_ROLE_PACMAN);
        if (!(c->flags[p] & BGW_ST_ACTIVE)) return 1;
        for (int a = 0; a < c->A; ++a) if (c->sp->role[a] == BGW_ROLE_FOOD) return 0;  /* any FoodAgent object */
        return 1;
    }
    default: return smart_all_done(c);
    }
}

/* get_reward: read-and-zero smart.py:101-104; MultiMaze override multi_maze_navigation.py:56-59; a program's hook */
static double prog_take_reward(Ctx *c, int a)
{
    double r = c->racc[a];
    if (c->sp->program == BGW_PROG_MULTI_MAZE && prog_done(c, a)) r = c->sp->reward[BGW_RW_TARGET];
#ifdef BGW_USER_PROGRAM
    if (c->sp->program == BGW_PROG_USER) r = user_reward(c, a, r);
#endif
    c->racc[a] = 0.0;
    return r;
}

/* ------------------------------------------------------------------------------------------------- */
/* sim programs: the user-written step()                                                             */
/* ------------------------------------------------------------------------------------------------- */
static void pacman_teleport(Ctx *c, int a)   /* pacman.py:87-92,116-121: (9,0) <-> (9,20), raw remove/place */
{
    if (c->H <= 9 || c->W <= 20) return;
    const int left = 9 * c->W + 0, right = 9 * c->W + 20;
    if (c->cell[a] == left) { grid_remove(c, a); grid_place(c, a, right); }
    else if (c->cell[a] == right) { grid_remove(c, a); grid_place(c, a, left); }
}

static void pacman_overlaps(Ctx *c, int p, int eat_food)   /* pacman.py:94-105,123-131 */
{
    const double *rw = c->sp->reward;
    if (!(c->flags[p] & BGW_ST_IN_GRID)) return;
    /* iterate over a COPY of the cell dict: collect first */
    uint16_t occ[512]; int n = 0;
    for (uint16_t o = c->head[c->cell[p]]; o != NONE && n < 512; o = c->next[o]) occ[n++] = o;
    for (int i = 0; i < n; ++i) {
        const int o = occ[i];
        if (o == p) continue;
        if (eat_food && c->sp->role[o] == BGW_ROLE_FOOD) {
            c->racc[p] += rw[BGW_RW_EAT_FOOD];
            grid_remove(c, o);
            set_health(c, o, 0.0);
        } else if (c->sp->role[o] == BGW_ROLE_BADDIE) {
            c->racc[p] += rw[BGW_RW_DIE];
            c->racc[o] += rw[BGW_RW_KILL];
            set_health(c, p, 0.0);
        }
    }
}

#define ACT(a) (c->actions + (size_t)c->learner_of[(a)] * c->astride)

/* the attack phase of TeamBattleSim.step team_battle_example.py:35-47 and ReachTheTargetSim.step reach_the_target.py:119-131 */
static void attack_phase(Ctx *c)
{
    const double *rw = c->sp->reward;
    int victims[BGW_MAX_VICTIMS + 1];
    for (int i = 0; i < c->n_acting; ++i) {
        const int a = c->acting[i];
        if (a < 0 || !(c->flags[a] & BGW_ST_ACTIVE)) continue;
        int nv = 0;
        const int status = process_attack(c, a, (const uint8_t *)ACT(a) + 2, victims, &nv);
        if (status) {
            if (nv == 0) c->racc[a] += rw[BGW_RW_ATTACK_FAIL];
            else for (int t = 0; t < nv; ++t)
                if (!(c->flags[victims[t]] & BGW_ST_ACTIVE)) {
                    c->racc[victims[t]] += rw[BGW_RW_DIE];
                    c->racc[a] += rw[BGW_RW_KILL];
                }
        }
    }
}

/* sim.step(action_dict) over the acting set c->acting[0 .. n_acting) (agents in action_dict order; -1: no action, the
 * learner was reported done already) and their action rows */
static void prog_step(Ctx *c)
{
    const BgwSpec *sp = c->sp;
    const double *rw = sp->reward;
    const int n_act = c->n_acting, *acting = c->acting;
    switch (sp->program) {
    case BGW_PROG_TEAM_BATTLE: {                               /* team_battle_example.py:33-59 */
        attack_phase(c);                                       /* :35-47 */
        for (int i = 0; i < n_act; ++i) {                      /* :50-55 */
            const int a = acting[i];
            if (a < 0 || !(c->flags[a] & BGW_ST_ACTIVE)) continue;
            if (!process_move(c, a, ACT(a))) c->racc[a] += rw[BGW_RW_MOVE_FAIL];
        }
        for (int i = 0; i < n_act; ++i) if (acting[i] >= 0) c->racc[acting[i]] += rw[BGW_RW_ENTROPY];   /* :58-59 */
        break;
    }
    case BGW_PROG_REACH_TARGET: {                              /* reach_the_target.py:117-152 */
        const int tgt = find_role(c, BGW_ROLE_TARGET);
        attack_phase(c);                                       /* :119-131 */
        for (int i = 0; i < n_act; ++i) {                      /* :134-145 */
            const int a = acting[i];
            if (a < 0 || !(sp->klass[a] & BGW_AG_MOVING)) continue;
            if (c->flags[a] & BGW_ST_ACTIVE)
                if (!process_move(c, a, ACT(a))) c->racc[a] += rw[BGW_RW_MOVE_FAIL];
            /* TargetDone.get_done :33-40.  A runner that is no longer in the grid (killed while standing on the
             * target's cell) would make the reference's grid.remove raise; it is left alone here */
            if (a != tgt && (c->flags[a] & BGW_ST_IN_GRID) && same_position(c, a, tgt)) {
                c->racc[a] += rw[BGW_RW_TARGET];
                grid_remove(c, a);
                c->flags[a] &= (uint8_t)~BGW_ST_ACTIVE;
            }
        }
        for (int i = 0; i < n_act; ++i)                         /* :148-150 */
            if (acting[i] >= 0 && sp->role[acting[i]] == BGW_ROLE_RUNNER) c->racc[acting[i]] += rw[BGW_RW_ENTROPY];
        break;
    }
    case BGW_PROG_TRAFFIC:                                     /* traffic_corridor.py:46-53 */
        for (int i = 0; i < n_act; ++i) {
            const int a = acting[i];
            if (a < 0) continue;
            if (!process_move(c, a, ACT(a))) c->racc[a] += rw[BGW_RW_MOVE_FAIL];
            if (smart_done(c, a)) c->racc[a] += rw[BGW_RW_TARGET];
        }
        break;
    case BGW_PROG_MAZE: {                                      /* maze_navigation.py:25-36 */
        const int nav = find_role(c, BGW_ROLE_NAVIGATOR);
        if (!process_move(c, nav, ACT(nav))) c->racc[nav] += rw[BGW_RW_MOVE_FAIL];
        if (prog_all_done(c)) c->racc[nav] += rw[BGW_RW_TARGET];
        c->racc[nav] += rw[BGW_RW_ENTROPY];
        break;
    }
    case BGW_PROG_MULTI_MAZE: {                                /* multi_maze_navigation.py:40-48 */
        for (int i = 0; i < n_act; ++i) {
            const int a = acting[i];
            if (a < 0) continue;
            if (!process_move(c, a, ACT(a))) c->racc[a] += rw[BGW_RW_MOVE_FAIL];
            c->racc[a] += rw[BGW_RW_ENTROPY];
        }
        break;
    }
    case BGW_PROG_PACMAN_SIMPLE: {                             /* pacman.py:214-310 */
        const int p = find_role(c, BGW_ROLE_PACMAN);
        if (!process_move(c, p, ACT(p))) c->racc[p] += rw[BGW_RW_MOVE_FAIL];      /* :216-220 */
        else c->racc[p] += rw[BGW_RW_ENTROPY];
        pacman_teleport(c, p);                                                    /* :221-226 */
        int eaten = 0;
        for (int pass = 0; pass < 2 && !eaten; ++pass) {
            /* overlaps with pacman, over a copy of the cell's dict (:228-239 with food, :305-311 baddies only) */
            uint16_t occ[512]; int n = 0;
            for (uint16_t o = c->head[c->cell[p]]; o != NONE && n < 512; o = c->next[o]) occ[n++] = o;
            for (int i = 0; i < n && !eaten; ++i) {
                const int o = occ[i];
                if (o == p) continue;
                if (pass == 0 && sp->role[o] == BGW_ROLE_FOOD) {
                    c->racc[p] += rw[BGW_RW_EAT_FOOD];
                    grid_remove(c, o);
                    set_health(c, o, 0.0);
                } else if (sp->role[o] == BGW_ROLE_BADDIE || sp->role[o] >= BGW_ROLE_SCRIPTED_BADDIE) {
                    c->racc[p] += rw[BGW_RW_DIE];
                    set_health(c, p, 0.0);
                    grid_remove(c, p);
                    eaten = 1;                                                    /* `return`: nothing else happens this step */
                }
            }
            if (pass == 1 || eaten) break;
            /* the scripted baddies move in the script's order (:241-303) */
            int slot_agent[10], move[10], o156 = 0;
            for (int k = 0; k < 10; ++k) slot_agent[k] = -1;
            for (int a = 0; a < c->A; ++a)
                if (sp->role[a] >= BGW_ROLE_SCRIPTED_BADDIE && sp->role[a] < BGW_ROLE_SCRIPTED_BADDIE + 10) slot_agent[sp->role[a] - BGW_ROLE_SCRIPTED_BADDIE] = a;
            if (slot_agent[2] >= 0) o156 = (c->flags[slot_agent[2]] >> BGW_ST_ORIENT_SHIFT) & 7;
            const uint32_t x159 = slot_agent[4] >= 0 ? draw(c, BGW_SITE_SCRIPT, (uint32_t)slot_agent[4], 0) : 0;
            pacman_script((int)step_of(c) - 1, o156, x159, move);
            for (int k = 0; k < 10; ++k) {
                const int a = slot_agent[k];
                if (a < 0) continue;
                const int8_t act4[4] = {(int8_t)move[k], 0, 0, 0};
                process_move(c, a, act4);
                pacman_teleport(c, a);
            }
        }
        break;
    }
    case BGW_PROG_PACMAN: {                                    /* pacman.py:80-135 */
        const int p = find_role(c, BGW_ROLE_PACMAN);
        if (!process_move(c, p, ACT(p))) c->racc[p] += rw[BGW_RW_MOVE_FAIL];
        else c->racc[p] += rw[BGW_RW_ENTROPY];
        pacman_teleport(c, p);
        pacman_overlaps(c, p, 1);
        for (int i = 0; i < n_act; ++i) {
            const int a = acting[i];
            if (a < 0 || a == p) continue;
            if (!process_move(c, a, ACT(a))) c->racc[a] += rw[BGW_RW_MOVE_FAIL];
            else c->racc[a] += rw[BGW_RW_ENTROPY];
            pacman_teleport(c, a);
        }
        pacman_overlaps(c, p, 0);
        if (!(c->flags[p] & BGW_ST_ACTIVE)) grid_remove(c, p);  /* :134-135 */
        break;
    }
#ifdef BGW_USER_PROGRAM
    case BGW_PROG_USER: user_step(c); break;
#endif
    default: break;
    }
}
#undef ACT

/* ------------------------------------------------------------------------------------------------- */
/* State components: state.py                                                                        */
/* ------------------------------------------------------------------------------------------------- */
/* PositionState._update_available_positions state.py:126-141 */
static void update_available(Ctx *c, uint8_t *avail, int placed)
{
    const BgwSpec *sp = c->sp;
    const uint64_t row = sp->overlap[sp->encoding[placed]];
    for (int e = 1; e <= c->max_enc; ++e)
        if (sp->no_overlap_at_reset || !((row >> e) & 1)) avail[(size_t)e * c->HW + c->cell[placed]] = 0;
}

/* The keyed order of a list of entities (include/bgw_philox.h): sorted by (first Philox word of the entity's key, entity
 * index).  Stands for random.shuffle -- state.py:97-101, all_step_manager.py:62-65 -- whose result the replay shim
 * defines the same way.  Insertion sort: the lists are short and this is the checker, not the product. */
static void keyed_order(const Ctx *c, uint32_t site, uint32_t step, int *items, int n)
{
    uint32_t *key = (uint32_t *)malloc(sizeof(uint32_t) * (size_t)(n + 1));
    for (int i = 0; i < n; ++i)
        key[i] = bgw_draw(c->sp->seed, c->genv, c->st->episode[c->env], step, site, (uint32_t)items[i], 0);
    for (int i = 1; i < n; ++i) {
        const uint32_t k = key[i]; const int it = items[i];
        int j = i - 1;
        while (j >= 0 && (key[j] > k || (key[j] == k && items[j] > it))) { key[j + 1] = key[j]; items[j + 1] = items[j]; --j; }
        key[j + 1] = k; items[j + 1] = it;
    }
    free(key);
}

static void sim_reset(Ctx *c)
{
    const BgwSpec *sp = c->sp;
    BgwState *st = c->st;
    st->episode[c->env] += 1;
    st->step[c->env] = 0;
    st->error[c->env] = 0;
    for (int a = 0; a < c->A; ++a) { c->flags[a] = 0; c->cell[a] = NONE; c->racc[a] = 0.0; c->health[a] = 0.0; }
    grid_clear(c);                                              /* state.py:95 */

    if (st->layout) {
        /* externally generated placement (e.g. MazePlacementState state.py:487-527 run host-side) */
        const uint16_t *lay = st->layout + (size_t)c->env * c->A;
        for (int a = 0; a < c->A; ++a) { if (lay[a] != NONE) grid_insert(c, a, lay[a]); else st->error[c->env] = 2; }   /* no cell: state.py:598-603 */
    } else {
        uint8_t *avail = (uint8_t *)malloc((size_t)(c->max_enc + 1) * c->HW);
        memset(avail, 1, (size_t)(c->max_enc + 1) * c->HW);     /* _build_available_positions state.py:116-124 */
        /* placement order: the agents dict, shuffled per episode when asked for (state.py:97-101) */
        int *ord = (int *)malloc(sizeof(int) * (size_t)c->A);
        for (int a = 0; a < c->A; ++a) ord[a] = a;
        if (sp->randomize_placement_order) keyed_order(c, BGW_SITE_PLACE_ORDER, 0, ord, c->A);
        for (int i = 0; i < c->A; ++i) {                        /* state.py:107-109,143-150 */
            const int a = ord[i];
            if (sp->init_row[a] < 0) continue;
            const int cell = sp->init_row[a] * c->W + sp->init_col[a];
            if (!grid_place(c, a, cell)) { st->error[c->env] = 1; grid_insert(c, a, cell); }
            update_available(c, avail, a);
        }
        for (int i = 0; i < c->A; ++i) {                        /* state.py:112-114,152-166 */
            const int a = ord[i];
            if (sp->init_row[a] >= 0) continue;
            const uint8_t *av = avail + (size_t)sp->encoding[a] * c->HW;
            int n = 0;
            for (int j = 0; j < c->HW; ++j) n += av[j];
            if (n == 0) { if (!st->error[c->env]) st->error[c->env] = 2; continue; }   /* RuntimeError :161 */
            int k = (int)bgw_index(draw(c, BGW_SITE_PLACE, (uint32_t)a, 0), (uint32_t)n);
            int cell = 0;
            for (int j = 0; j < c->HW; ++j) if (av[j] && k-- == 0) { cell = j; break; }
            grid_place(c, a, cell);
            update_available(c, avail, a);
        }
        free(ord);
        free(avail);
    }
    for (int a = 0; a < c->A; ++a) {
        c->flags[a] |= BGW_ST_ACTIVE;                           /* PrincipleAgent.active = True */
        if (sp->klass[a] & BGW_AG_HEALTH) {                     /* HealthState.reset state.py:635-641 */
            if (isnan(sp->init_health[a])) set_health(c, a, bgw_u01(draw(c, BGW_SITE_HEALTH, (uint32_t)a, 0)));
            else set_health(c, a, sp->init_health[a]);
        }
        if (sp->klass[a] & BGW_AG_ORIENT) {                     /* OrientationState.reset state.py:670-675 */
            int o = sp->init_orient[a];
            if (!o) o = 1 + (int)bgw_index(draw(c, BGW_SITE_ORIENT, (uint32_t)a, 0), 4);
            c->flags[a] = (uint8_t)((c->flags[a] & 0x8F) | (o << BGW_ST_ORIENT_SHIFT));
        }
        if (!(sp->klass[a] & BGW_AG_LEARNER)) c->flags[a] |= BGW_ST_DONE_REPORTED;  /* all_step_manager.py:41-44 */
        if (c->ammo) c->ammo[a] = (sp->klass[a] & BGW_AG_AMMO) && sp->initial_ammo ? sp->initial_ammo[a] : 0;   /* AmmoState.reset state.py:649-656 */
    }
}

/* ------------------------------------------------------------------------------------------------- */
/* context plumbing                                                                                  */
/* ------------------------------------------------------------------------------------------------- */
static void ctx_init(Ctx *c, const BgwSpec *sp, BgwState *st)
{
    memset(c, 0, sizeof(*c));
    c->sp = sp; c->st = st;
    c->H = sp->rows; c->W = sp->cols; c->A = sp->n_agents; c->HW = c->H * c->W;
    c->max_enc = max_encoding(sp);
    c->L = count_learners(sp);
    c->head = (uint16_t *)malloc(sizeof(uint16_t) * (size_t)c->HW);
    c->tail = (uint16_t *)malloc(sizeof(uint16_t) * (size_t)c->HW);
    c->prev = (uint16_t *)malloc(sizeof(uint16_t) * (size_t)c->A);
    c->learner_of = (int *)malloc(sizeof(int) * (size_t)c->A);
    c->agent_of = (int *)malloc(sizeof(int) * (size_t)(c->L + 1));
    c->acc_occ = (uint8_t *)calloc((size_t)c->A + 1, 1);
    c->astride = action_stride_of(sp);
    int l = 0;
    for (int a = 0; a < c->A; ++a) {
        if (sp->klass[a] & BGW_AG_LEARNER) { c->learner_of[a] = l; c->agent_of[l++] = a; }
        else c->learner_of[a] = -1;
    }
}

static void ctx_free(Ctx *c)
{
    free(c->head); free(c->tail); free(c->prev); free(c->learner_of); free(c->agent_of); free(c->mask); free(c->acc_occ);
}

static void ctx_env(Ctx *c, int e)
{
    c->env = e; c->genv = (uint32_t)(c->sp->env_offset + e);
    const size_t off = (size_t)e * c->A;
    c->cell = c->st->cell + off; c->next = c->st->next + off; c->flags = c->st->flags + off;
    c->health = c->st->health + off; c->racc = c->st->reward_acc + off;
    c->ammo = c->st->ammo ? c->st->ammo + off : NULL;
}

/* reset one env + first observations (AllStepManager.reset all_step_manager.py:37-49,
 * TurnBasedManager.reset turn_based_manager.py:22-32) */
static void env_reset(Ctx *c, int8_t *obs_env, int stride)
{
    sim_reset(c);
    /* a failed placement (the reference raises, state.py:147-149,161): the env is reported ERROR | ALL_DONE with zero
     * observations and stays inert until it is reset again */
    const int bad = c->st->error[c->env] != 0;
    c->st->env_flags[c->env] = (uint8_t)(bad ? BGW_ENV_ERROR | BGW_ENV_ALL_DONE : 0);
    if (c->sp->manager == BGW_MANAGER_DYNAMIC_ORDER) {          /* dynamic_order_manager.py:19-28: the sim names the first agent */
        c->st->turn[c->env] = 0;
        if (obs_env && bad) memset(obs_env, 0, (size_t)stride);
        else if (obs_env) observe_agent(c, c->agent_of[0], obs_env, stride);
    } else if (c->sp->manager == BGW_MANAGER_TURN_BASED) {
        int t = c->st->turn[c->env];
        t = (t + 1) % c->L;                                     /* next(self.agent_order); never rewound :17-20 */
        c->st->turn[c->env] = (int16_t)t;
        if (obs_env && bad) memset(obs_env + (size_t)t * stride, 0, (size_t)stride);
        else if (obs_env) observe_agent(c, c->agent_of[t], obs_env + (size_t)t * stride, stride);
    } else if (obs_env) {
        for (int l = 0; l < c->L; ++l) {
            if (bad) memset(obs_env + (size_t)l * stride, 0, (size_t)stride);
            else observe_agent(c, c->agent_of[l], obs_env + (size_t)l * stride, stride);
        }
    }
}

int bgwo_reset(const BgwSpec *sp, BgwState *st, const uint8_t *env_mask, int8_t *obs)
{
    Ctx c; ctx_init(&c, sp, st);
    BgwDims d; bgwo_dims(sp, &d);
    for (int e = 0; e < sp->n_envs; ++e) {
        if (env_mask && !env_mask[e]) continue;
        ctx_env(&c, e);
        env_reset(&c, obs ? obs + (size_t)e * c.L * d.obs_stride : NULL, d.obs_stride);
    }
    ctx_free(&c);
    return 0;
}

static void emit(Ctx *c, int l, int8_t *obs_env, int stride, float *rew, double *rew64, uint8_t *done)
{
    const int a = c->agent_of[l];
    if (obs_env) observe_agent(c, a, obs_env + (size_t)l * stride, stride);
    const double r = prog_take_reward(c, a);
    const int d = prog_done(c, a);
    if (rew) rew[l] = (float)r;
    if (rew64) rew64[l] = r;
    done[l] = (uint8_t)(BGW_OUT_VALID | (d ? BGW_OUT_DONE : 0));
    c->st->stats[(size_t)c->env * BGW_STAT_COUNT + BGW_STAT_AGENT_STEPS]++;
}

/* One manager step of every env.  A step program (BGW_PROG_USER) needs the library built with it (build_program) and runs
 * under the all-step and turn-based managers; otherwise nothing is touched and the result is non-zero.  Bad input from
 * the program ends the env with BgwState.error = 3 (bgw_program.h). */
int bgwo_step(const BgwSpec *sp, BgwState *st, const int8_t *actions, const int16_t *order, int8_t *obs,
              float *reward, double *reward64, uint8_t *done, uint8_t *all_done)
{
    if (sp->program == BGW_PROG_USER) {
#ifndef BGW_USER_PROGRAM
        return 1;
#endif
        if (sp->manager == BGW_MANAGER_DYNAMIC_ORDER) return 1;
    }
    Ctx c; ctx_init(&c, sp, st);
    BgwDims d; bgwo_dims(sp, &d);
    const int L = c.L, stride = d.obs_stride;
    c.acting = (int *)malloc(sizeof(int) * (size_t)(L + 1));
    for (int e = 0; e < sp->n_envs; ++e) {
        ctx_env(&c, e);
        int8_t *obs_env = obs ? obs + (size_t)e * L * stride : NULL;
        float *rew = reward ? reward + (size_t)e * L : NULL;
        double *rew64 = reward64 ? reward64 + (size_t)e * L : NULL;
        uint8_t *dn = done + (size_t)e * L;
        c.actions = actions + (size_t)e * L * c.astride;
        c.err = 0;
        for (int l = 0; l < L; ++l) { dn[l] = 0; if (rew) rew[l] = 0.f; if (rew64) rew64[l] = 0.0; }

        if (st->env_flags[e] & BGW_ENV_ALL_DONE) {
            if (sp->auto_reset) {
                env_reset(&c, obs_env, stride);
                st->env_flags[e] |= BGW_ENV_RESET;
                all_done[e] = st->env_flags[e];
            } else all_done[e] = st->env_flags[e];
            continue;
        }
        grid_build(&c);
        st->step[e] += 1;
        st->stats[(size_t)e * BGW_STAT_COUNT + BGW_STAT_ENV_STEPS]++;
        int env_done = 0;

        if (sp->manager == BGW_MANAGER_ALL_STEP) {              /* all_step_manager.py:51-95 */
            /* one acting slot per learner in processing order: dict order, the caller's, or (:62-65) the keyed order of
             * this step.  A learner reported done sends no action (:59-61): its slot holds -1.  The keyed order of the
             * others is the restriction of the full one, so it is taken before they are marked. */
            for (int i = 0; i < L; ++i) c.acting[i] = c.agent_of[order ? order[(size_t)e * L + i] : i];
            if (!order && sp->randomize_action_input) keyed_order(&c, BGW_SITE_ORDER, st->step[e], c.acting, L);
            for (int i = 0; i < L; ++i) if (c.flags[c.acting[i]] & BGW_ST_DONE_REPORTED) c.acting[i] = -1;
            c.n_acting = L;
            prog_step(&c);                                      /* :66 */
            for (int l = 0; l < L; ++l) {                       /* :68-87 */
                const int a = c.agent_of[l];
                if (c.flags[a] & BGW_ST_DONE_REPORTED) continue;
                emit(&c, l, obs_env, stride, rew, rew64, dn);
            }
            int remaining = 0;
            for (int l = 0; l < L; ++l) {
                const int a = c.agent_of[l];
                if (dn[l] & BGW_OUT_DONE) c.flags[a] |= BGW_ST_DONE_REPORTED;
                if (!(c.flags[a] & BGW_ST_DONE_REPORTED)) ++remaining;
            }
            env_done = prog_all_done(&c) || remaining == 0;     /* :90-93 */
        } else {                                                /* turn_based_manager.py:34-94 */
            int l = st->turn[e];
            c.acting[0] = c.agent_of[l];
            c.n_acting = 1;
            prog_step(&c);                                      /* :46 */
            env_done = prog_all_done(&c);                       /* :48 */
            if (env_done) {                                     /* :49-57, dynamic_order_manager.py:43-51 */
                for (int k = 0; k < L; ++k)
                    if (!(c.flags[c.agent_of[k]] & BGW_ST_DONE_REPORTED)) emit(&c, k, obs_env, stride, rew, rew64, dn);
            } else if (sp->manager == BGW_MANAGER_DYNAMIC_ORDER) {
                /* dynamic_order_manager.py:52-85 over the sim's next_agent = [the agent that acted, if this step finished
                 * it] + [the next agent in dict order that is not done] (DynamicOrderMultiMazeSim.step) */
                const int turn = l, a0 = c.agent_of[turn];
                if (prog_done(&c, a0)) {                        /* :60-69: just finished; someone else is not done */
                    emit(&c, turn, obs_env, stride, rew, rew64, dn);
                    c.flags[a0] |= BGW_ST_DONE_REPORTED;
                }
                for (int k = 1; k <= L; ++k) {
                    l = (turn + k) % L;
                    const int a = c.agent_of[l];
                    if (prog_done(&c, a)) continue;             /* the sim skips the agents that are done */
                    if (!(c.flags[a] & BGW_ST_DONE_REPORTED)) emit(&c, l, obs_env, stride, rew, rew64, dn);   /* :80-85 */
                    break;
                }
                st->turn[e] = (int16_t)l;
            } else {
                for (;;) {                                      /* :59-92 */
                    l = (l + 1) % L;
                    const int a = c.agent_of[l];
                    if (c.flags[a] & BGW_ST_DONE_REPORTED) continue;
                    if (prog_done(&c, a)) {
                        emit(&c, l, obs_env, stride, rew, rew64, dn);
                        c.flags[a] |= BGW_ST_DONE_REPORTED;
                        int remaining = 0;
                        for (int k = 0; k < L; ++k) if (!(c.flags[c.agent_of[k]] & BGW_ST_DONE_REPORTED)) ++remaining;
                        if (remaining) continue;
                        env_done = 1;
                        break;
                    }
                    emit(&c, l, obs_env, stride, rew, rew64, dn);
                    break;
                }
                st->turn[e] = (int16_t)l;
            }
        }
        uint8_t ef = 0;
        if (env_done) ef |= BGW_ENV_ALL_DONE;
        if (sp->horizon > 0 && (int)st->step[e] >= sp->horizon) ef |= BGW_ENV_ALL_DONE | BGW_ENV_TRUNCATED;
        if (c.err) { ef |= BGW_ENV_ERROR | BGW_ENV_ALL_DONE; st->error[e] = c.err; }
        if (ef & BGW_ENV_ALL_DONE) st->stats[(size_t)e * BGW_STAT_COUNT + BGW_STAT_EPISODES]++;
        st->env_flags[e] = ef;
        all_done[e] = ef;
    }
    free(c.acting);
    ctx_free(&c);
    return 0;
}

int bgwo_observe(const BgwSpec *sp, BgwState *st, int env, int8_t *obs_env)
{
    Ctx c; ctx_init(&c, sp, st);
    BgwDims d; bgwo_dims(sp, &d);
    ctx_env(&c, env);
    grid_build(&c);
    for (int l = 0; l < c.L; ++l) observe_agent(&c, c.agent_of[l], obs_env + (size_t)l * d.obs_stride, d.obs_stride);
    ctx_free(&c);
    return 0;
}

/* RandomPolicy.compute_action = action_space.sample() (policies/policy.py:81-92) restated on the keyed
 * stream: one Philox block per (env, step, agent); words 0,1 -> move, word 2 -> attack. */
int bgwo_sample_actions(const BgwSpec *sp, const BgwState *st, int8_t *actions)
{
    const int A = sp->n_agents, L = count_learners(sp), stride = action_stride_of(sp), menc = max_encoding(sp);
    for (int e = 0; e < sp->n_envs; ++e) {
        int l = 0;
        for (int a = 0; a < A; ++a) {
            if (!(sp->klass[a] & BGW_AG_LEARNER)) continue;
            int8_t *o = actions + ((size_t)e * L + l) * stride;
            ++l;
            uint32_t x[4];
            bgw_draw4(sp->seed, (uint32_t)(sp->env_offset + e), st->episode[e], st->step[e], BGW_SITE_ACTION, (uint32_t)a, 0, x);
            memset(o, 0, (size_t)stride);
            if (sp->klass[a] & BGW_AG_MOVING) {
                if (sp->move_actor == BGW_MOVE_BOX) {            /* Box(-m, m, (2,), int) actor.py:63-65 */
                    const int m = sp->move_range[a], w = 2 * m + 1;
                    const int dr = (int)bgw_index(x[0], (uint32_t)w) - m, dc = (int)bgw_index(x[1], (uint32_t)w) - m;
                    if (sp->ravel_actions) o[0] = (int8_t)(uint8_t)((dr + m) * w + (dc + m));
                    else { o[0] = (int8_t)dr; o[1] = (int8_t)dc; }
                } else if (sp->move_actor != BGW_MOVE_NONE) {    /* Discrete(5) actor.py:125 */
                    o[0] = (int8_t)bgw_index(x[0], 5);
                }
            }
            if (!(sp->klass[a] & BGW_AG_ATTACKING) || sp->attack_actor == BGW_ATTACK_NONE) continue;
            const uint32_t sim = sp->simultaneous_attacks[a];
            if (sp->attack_actor == BGW_ATTACK_BINARY) {
                o[2] = (int8_t)bgw_index(x[2], sim + 1);         /* Discrete(n+1) actor.py:452 */
                continue;
            }
            /* wider attack actions: attack byte j draws word j%4 of the block k = 1 + j/4 */
            const int n = 2 * sp->attack_range[a] + 1;
            const int width = sp->attack_actor == BGW_ATTACK_ENCODING ? menc : sp->attack_actor == BGW_ATTACK_RESTRICTED ? (int)sim : n * n;
            for (int j = 0; j < width; ++j) {
                if ((j & 3) == 0) bgw_draw4(sp->seed, (uint32_t)(sp->env_offset + e), st->episode[e], st->step[e], BGW_SITE_ACTION, (uint32_t)a, 1u + ((uint32_t)j >> 2), x);
                uint32_t v;
                if (sp->attack_actor == BGW_ATTACK_ENCODING)      /* Dict{enc: Discrete(n+1)} actor.py:513-519 */
                    v = ((sp->attack_map[sp->encoding[a]] >> (j + 1)) & 1) ? bgw_index(x[j & 3], sim + 1) : 0;
                else if (sp->attack_actor == BGW_ATTACK_RESTRICTED)   /* MultiDiscrete([cells+1]*n) actor.py:593-599 */
                    v = bgw_index(x[j & 3], (uint32_t)(n * n) + 1);
                else                                              /* Box(0, n, (w, w)) actor.py:669-679 */
                    v = bgw_index(x[j & 3], sim + 1);
                o[2 + j] = (int8_t)(uint8_t)v;
            }
        }
    }
    return 0;
}

/* sizeof the three ABI structs as this C compiler lays them out (tests/test_capi.py checks the ctypes mirrors) */
int bgwo_sizeof(int which) { return which == 0 ? (int)sizeof(BgwSpec) : which == 1 ? (int)sizeof(BgwState) : (int)sizeof(BgwDims); }

/* host-callable draw, same stream as include/bgw_philox.h (used by the replay shim and the Philox KATs) */
int bgwo_rng_draw(uint64_t seed, uint32_t env, uint32_t episode, uint32_t step, uint32_t site, uint32_t slot,
                  uint32_t k, uint32_t out[4])
{
    bgw_draw4(seed, env, episode, step, site, slot, k, out);
    return 0;
}

/* raw Philox4x32-10 block (for the Random123 known-answer test) */
int bgwo_philox_raw(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4])
{
    bgw_philox4x32_10(ctr[0], ctr[1], ctr[2], ctr[3], key[0], key[1], out);
    return 0;
}
