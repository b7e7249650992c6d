/*
 * bgw_program.cuh -- device side of the step-program API (include/bgw_program.h) over DevSpec / Env (bgw_dev.cuh).
 *
 * Only the run-time compilation of bgw_set_program includes this file (bgw_jit.h), twice, around the program's source:
 *
 *     #define BGW_USER_PROGRAM
 *     #include "bgw_dev.cuh"
 *     #include "bgw_program.cuh"        the API, ahead of the program
 *     <program source>
 *     #define BGWP_AFTER_PROGRAM
 *     #include "bgw_program.cuh"        user_step / user_done / ... : the engine's calls into the program
 *     <kernel wrapper>
 *
 * The program runs on thread 0 of the env's CTA between two barriers (bgw_step_body), like the built-in serial programs,
 * so the API functions are the serial primitives of bgw_dev.cuh: process_move, try_move, grid_query, grid_append,
 * grid_unlink, set_health, dev_draw and the attack code.  The oracle (tests/program_oracle.c) implements the same API over
 * its own primitives.
 */
#ifndef BGWP_AFTER_PROGRAM

#include "../../include/bgw_program.h"

struct bgwp_ctx {
    const DevSpec *s;
    Env *ev;         /* the hooks get a const bgwp_ctx: they cannot call a mutating API function, though the pointee is not const */
};

/* bad input from the program (include/bgw_program.h): the env reports BGW_ENV_ERROR at the end of the step */
static __device__ __forceinline__ bool bgwp_fail(const bgwp_ctx *c) { c->ev->ctr[CTR_ERR] = 3; return false; }
static __device__ __forceinline__ bool bgwp_agent_ok(const bgwp_ctx *c, int a) { return ((unsigned)a < (unsigned)c->s->A) || bgwp_fail(c); }
static __device__ __forceinline__ bool bgwp_cell_ok(const bgwp_ctx *c, int r, int col)
{
    return ((unsigned)r < (unsigned)c->s->H && (unsigned)col < (unsigned)c->s->W) || bgwp_fail(c);
}

/* ---- the acting set and the env ------------------------------------------------------------------------------------ */
BGWP_FN int bgwp_n_acting(const bgwp_ctx *c) { return c->s->manager == BGW_MANAGER_ALL_STEP ? c->s->L : 1; }
BGWP_FN int bgwp_acting(const bgwp_ctx *c, int i)
{
    if ((unsigned)i >= (unsigned)bgwp_n_acting(c)) { bgwp_fail(c); return -1; }
    const unsigned a = c->ev->ragent[i];
    return a == BGW_NONE16 ? -1 : (int)a;
}
BGWP_FN int bgwp_step_index(const bgwp_ctx *c) { return (int)c->ev->step; }
BGWP_FN int bgwp_rows(const bgwp_ctx *c) { return c->s->H; }
BGWP_FN int bgwp_cols(const bgwp_ctx *c) { return c->s->W; }
BGWP_FN int bgwp_n_agents(const bgwp_ctx *c) { return c->s->A; }

/* ---- reads ----------------------------------------------------------------------------------------------------------- */
BGWP_FN int bgwp_encoding(const bgwp_ctx *c, int a) { return bgwp_agent_ok(c, a) ? c->ev->enc[a] : 0; }
BGWP_FN int bgwp_klass(const bgwp_ctx *c, int a) { return bgwp_agent_ok(c, a) ? c->ev->klass[a] : 0; }
BGWP_FN int bgwp_role(const bgwp_ctx *c, int a) { return bgwp_agent_ok(c, a) ? __ldg(&c->s->role[a]) : 0; }
BGWP_FN int bgwp_active(const bgwp_ctx *c, int a) { return bgwp_agent_ok(c, a) ? (c->ev->flags[a] & BGW_ST_ACTIVE) != 0 : 0; }
BGWP_FN int bgwp_in_grid(const bgwp_ctx *c, int a) { return bgwp_agent_ok(c, a) ? (c->ev->flags[a] & BGW_ST_IN_GRID) != 0 : 0; }
BGWP_FN int bgwp_row(const bgwp_ctx *c, int a)
{
    if (!bgwp_agent_ok(c, a)) return 0;
    const unsigned cell = c->ev->cell[a];
    return cell == BGW_NONE16 ? -1 : (int)(cell / (unsigned)c->s->W);
}
BGWP_FN int bgwp_col(const bgwp_ctx *c, int a)
{
    if (!bgwp_agent_ok(c, a)) return 0;
    const unsigned cell = c->ev->cell[a];
    return cell == BGW_NONE16 ? -1 : (int)(cell % (unsigned)c->s->W);
}
BGWP_FN double bgwp_health(const bgwp_ctx *c, int a) { return bgwp_agent_ok(c, a) ? __ldcg(&c->ev->health[a]) : 0.0; }
BGWP_FN int bgwp_ammo(const bgwp_ctx *c, int a) { return bgwp_agent_ok(c, a) && c->ev->ammo ? c->ev->ammo[a] : 0; }
BGWP_FN int bgwp_orientation(const bgwp_ctx *c, int a) { return bgwp_agent_ok(c, a) ? (c->ev->flags[a] >> BGW_ST_ORIENT_SHIFT) & 7 : 0; }
BGWP_FN int bgwp_action(const bgwp_ctx *c, int a, int k)
{
    if (!bgwp_agent_ok(c, a)) return 0;
    if ((unsigned)k >= (unsigned)(c->s->act_words * 4)) { bgwp_fail(c); return 0; }
    const int l = __ldg(&c->s->learner_of[a]);
    if (l < 0) return 0;
    return reinterpret_cast<const int8_t *>(c->ev->act + (size_t)l * c->s->act_words)[k];
}
BGWP_FN int bgwp_query(const bgwp_ctx *c, int a, int r, int col)
{
    if (!bgwp_agent_ok(c, a) || !bgwp_cell_ok(c, r, col)) return 0;
    return grid_query(*c->s, *c->ev, a, r * c->s->W + col);
}
BGWP_FN int bgwp_first_occupant(const bgwp_ctx *c, int r, int col)
{
    if (!bgwp_cell_ok(c, r, col)) return -1;
    const unsigned o = c->ev->head[r * c->s->W + col];
    return o == BGW_NONE16 ? -1 : (int)o;
}
BGWP_FN int bgwp_next_occupant(const bgwp_ctx *c, int a)
{
    if (!bgwp_agent_ok(c, a)) return -1;
    if (!(c->ev->flags[a] & BGW_ST_IN_GRID)) return -1;
    const unsigned o = c->ev->next[a];
    return o == BGW_NONE16 ? -1 : (int)o;
}

/* ---- actors ---------------------------------------------------------------------------------------------------------- */
BGWP_FN int bgwp_move(bgwp_ctx *c, int a)
{
    if (!bgwp_agent_ok(c, a)) return 0;
    const int l = __ldg(&c->s->learner_of[a]);
    if (l < 0 || !(c->ev->flags[a] & BGW_ST_IN_GRID)) return 0;
    return process_move(*c->s, *c->ev, a, c->ev->act[(size_t)l * c->s->act_words]);
}
BGWP_FN int bgwp_move_by(bgwp_ctx *c, int a, int dr, int dc)
{
    if (!bgwp_agent_ok(c, a)) return 0;
    if (!(c->ev->klass[a] & BGW_AG_MOVING) || !(c->ev->flags[a] & BGW_ST_IN_GRID)) return 0;
    return try_move(*c->s, *c->ev, a, dr, dc);
}
BGWP_FN int bgwp_attack(bgwp_ctx *c, int a, int *victims)
{
    if (!bgwp_agent_ok(c, a)) return -1;
    const DevSpec &s = *c->s;
    Env &ev = *c->ev;
    if (s.attack_actor == BGW_ATTACK_NONE || !(ev.klass[a] & BGW_AG_ATTACKING) || __ldg(&s.learner_of[a]) < 0) return -1;
    if (!attack_requested(s, ev, a)) return -1;                   /* actor.py:478,542,622,703 */
    uint16_t v[BGW_MAX_VICTIMS];
    const int nv = attack_victims(s, ev, a, v);
    attack_damage(s, ev, a, v, nv);
    for (int t = 0; t < nv; ++t) victims[t] = v[t];
    return nv;
}

/* ---- writes ---------------------------------------------------------------------------------------------------------- */
BGWP_FN void bgwp_set_health(bgwp_ctx *c, int a, double h) { if (bgwp_agent_ok(c, a)) set_health(*c->ev, a, h); }
BGWP_FN void bgwp_set_active(bgwp_ctx *c, int a, int on)
{
    if (!bgwp_agent_ok(c, a)) return;
    if (on) c->ev->flags[a] |= BGW_ST_ACTIVE; else c->ev->flags[a] &= ~BGW_ST_ACTIVE;
}
BGWP_FN int bgwp_place(bgwp_ctx *c, int a, int r, int col)
{
    if (!bgwp_agent_ok(c, a) || !bgwp_cell_ok(c, r, col)) return 0;
    if (c->ev->flags[a] & BGW_ST_IN_GRID) { bgwp_fail(c); return 0; }
    const int cell = r * c->s->W + col;
    if (!grid_query(*c->s, *c->ev, a, cell)) return 0;
    grid_append(*c->ev, a, cell);
    return 1;
}
BGWP_FN void bgwp_remove(bgwp_ctx *c, int a) { if (bgwp_agent_ok(c, a)) grid_unlink(*c->ev, a); }
BGWP_FN void bgwp_add_reward(bgwp_ctx *c, int a, double x)
{
    if (!bgwp_agent_ok(c, a)) return;
    /* the accumulators the step kernel keeps between calls (bgw_step_body: staging and store_env) */
    const uint8_t k = c->ev->klass[a];
    if (c->s->manager != BGW_MANAGER_ALL_STEP || racc_persists(k) || ((k & BGW_AG_LEARNER) && !(c->ev->flags[a] & BGW_ST_DONE_REPORTED)))
        c->ev->racc[a] += x;
}

/* ---- randomness ------------------------------------------------------------------------------------------------------ */
BGWP_FN double bgwp_uniform(const bgwp_ctx *c, int slot, int k)
{
    if ((unsigned)slot >= 4096u || (unsigned)k >= 65536u) { bgwp_fail(c); return 0.0; }
    return bgw_u01(dev_draw(*c->s, *c->ev, BGW_SITE_PROGRAM, (uint32_t)slot, (uint32_t)k));
}

#else  /* BGWP_AFTER_PROGRAM: the engine's calls into the program (bgw_dev.cuh declares them) */

static __device__ void user_step(const DevSpec &s, Env &ev, int nrank)
{
    (void)nrank;                                                    /* = bgwp_n_acting */
    bgwp_ctx c = {&s, &ev};
    bgwp_step(&c);
}

static __device__ int user_done(const DevSpec &s, const Env &ev, int a)
{
#ifdef BGWP_HAS_GET_DONE
    const bgwp_ctx c = {&s, const_cast<Env *>(&ev)};
    return bgwp_get_done(&c, a) != 0;
#else
    (void)s; (void)ev; (void)a;
    return -1;
#endif
}

static __device__ int user_all_done(const DevSpec &s, const Env &ev)
{
#ifdef BGWP_HAS_GET_ALL_DONE
    const bgwp_ctx c = {&s, const_cast<Env *>(&ev)};
    return bgwp_get_all_done(&c) != 0;
#else
    (void)s; (void)ev;
    return -1;
#endif
}

static __device__ double user_reward(const DevSpec &s, const Env &ev, int a, double acc)
{
#ifdef BGWP_HAS_GET_REWARD
    const bgwp_ctx c = {&s, const_cast<Env *>(&ev)};
    return bgwp_get_reward(&c, a, acc);
#else
    (void)s; (void)ev; (void)a;
    return acc;
#endif
}

#endif /* BGWP_AFTER_PROGRAM */
