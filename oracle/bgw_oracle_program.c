/*
 * bgw_oracle_program.c -- the CPU oracle with a user step program (include/bgw_program.h) compiled in.  TEST INFRASTRUCTURE
 * ONLY.
 *
 * It includes bgw_oracle.c with BGW_USER_PROGRAM defined, so the oracle's one manager step (bgwo_step) calls the program
 * through prog_step / prog_done / prog_all_done / prog_take_reward.  This half implements the step-program API over the
 * oracle's primitives, includes the program, and defines the four calls into it (user_step, user_done, user_all_done,
 * user_reward).  The device twin is abmarl_b200/csrc/bgw_program.cuh.
 *
 * Build (oracle/build.py, build_program):
 *     gcc -O2 -fPIC -shared -ffp-contract=off -fno-fast-math -Werror=discarded-qualifiers
 *         -DBGW_PROGRAM_FILE='"<program.c>"' -o <lib.so> oracle/bgw_oracle_program.c -lm
 * (-Werror=discarded-qualifiers: a get_done / get_all_done / get_reward hook that calls a mutating API function fails.)
 */
#define BGW_USER_PROGRAM
#include "bgw_oracle.c"
#include "../include/bgw_program.h"

struct bgwp_ctx {
    Ctx *c;                   /* the hooks get a const bgwp_ctx: a mutating API call from one discards the qualifier */
};

static int bgwp_fail(const bgwp_ctx *x) { x->c->err = 3; return 0; }
static int bgwp_agent_ok(const bgwp_ctx *x, int a) { return ((unsigned)a < (unsigned)x->c->A) || bgwp_fail(x); }
static int bgwp_cell_ok(const bgwp_ctx *x, int r, int col) { return ((unsigned)r < (unsigned)x->c->H && (unsigned)col < (unsigned)x->c->W) || bgwp_fail(x); }

/* ---- the acting set and the env ------------------------------------------------------------------------------------ */
BGWP_FN int bgwp_n_acting(const bgwp_ctx *x) { return x->c->n_acting; }
BGWP_FN int bgwp_acting(const bgwp_ctx *x, int i)
{
    if ((unsigned)i >= (unsigned)x->c->n_acting) { bgwp_fail(x); return -1; }
    return x->c->acting[i];
}
BGWP_FN int bgwp_step_index(const bgwp_ctx *x) { return (int)step_of(x->c); }
BGWP_FN int bgwp_rows(const bgwp_ctx *x) { return x->c->H; }
BGWP_FN int bgwp_cols(const bgwp_ctx *x) { return x->c->W; }
BGWP_FN int bgwp_n_agents(const bgwp_ctx *x) { return x->c->A; }

/* ---- reads ----------------------------------------------------------------------------------------------------------- */
BGWP_FN int bgwp_encoding(const bgwp_ctx *x, int a) { return bgwp_agent_ok(x, a) ? x->c->sp->encoding[a] : 0; }
BGWP_FN int bgwp_klass(const bgwp_ctx *x, int a) { return bgwp_agent_ok(x, a) ? x->c->sp->klass[a] : 0; }
BGWP_FN int bgwp_role(const bgwp_ctx *x, int a) { return bgwp_agent_ok(x, a) ? x->c->sp->role[a] : 0; }
BGWP_FN int bgwp_active(const bgwp_ctx *x, int a) { return bgwp_agent_ok(x, a) ? (x->c->flags[a] & BGW_ST_ACTIVE) != 0 : 0; }
BGWP_FN int bgwp_in_grid(const bgwp_ctx *x, int a) { return bgwp_agent_ok(x, a) ? (x->c->flags[a] & BGW_ST_IN_GRID) != 0 : 0; }
BGWP_FN int bgwp_row(const bgwp_ctx *x, int a)
{
    if (!bgwp_agent_ok(x, a)) return 0;
    return x->c->cell[a] == NONE ? -1 : x->c->cell[a] / x->c->W;
}
BGWP_FN int bgwp_col(const bgwp_ctx *x, int a)
{
    if (!bgwp_agent_ok(x, a)) return 0;
    return x->c->cell[a] == NONE ? -1 : x->c->cell[a] % x->c->W;
}
BGWP_FN double bgwp_health(const bgwp_ctx *x, int a) { return bgwp_agent_ok(x, a) ? x->c->health[a] : 0.0; }
BGWP_FN int bgwp_ammo(const bgwp_ctx *x, int a) { return bgwp_agent_ok(x, a) && x->c->ammo ? x->c->ammo[a] : 0; }
BGWP_FN int bgwp_orientation(const bgwp_ctx *x, int a) { return bgwp_agent_ok(x, a) ? (x->c->flags[a] >> BGW_ST_ORIENT_SHIFT) & 7 : 0; }
BGWP_FN int bgwp_action(const bgwp_ctx *x, int a, int k)
{
    if (!bgwp_agent_ok(x, a)) return 0;
    if ((unsigned)k >= (unsigned)x->c->astride) { bgwp_fail(x); return 0; }
    if (x->c->learner_of[a] < 0) return 0;
    return x->c->actions[(size_t)x->c->learner_of[a] * x->c->astride + k];
}
BGWP_FN int bgwp_query(const bgwp_ctx *x, int a, int r, int col)
{
    if (!bgwp_agent_ok(x, a) || !bgwp_cell_ok(x, r, col)) return 0;
    return grid_query(x->c, a, r * x->c->W + col);
}
BGWP_FN int bgwp_first_occupant(const bgwp_ctx *x, int r, int col)
{
    if (!bgwp_cell_ok(x, r, col)) return -1;
    const uint16_t o = x->c->head[r * x->c->W + col];
    return o == NONE ? -1 : (int)o;
}
BGWP_FN int bgwp_next_occupant(const bgwp_ctx *x, int a)
{
    if (!bgwp_agent_ok(x, a) || !(x->c->flags[a] & BGW_ST_IN_GRID)) return -1;
    return x->c->next[a] == NONE ? -1 : (int)x->c->next[a];
}

/* ---- actors ---------------------------------------------------------------------------------------------------------- */
BGWP_FN int bgwp_move(bgwp_ctx *x, int a)
{
    Ctx *c = x->c;
    if (!bgwp_agent_ok(x, a)) return 0;
    if (c->learner_of[a] < 0 || !(c->flags[a] & BGW_ST_IN_GRID)) return 0;
    return process_move(c, a, c->actions + (size_t)c->learner_of[a] * c->astride);
}
BGWP_FN int bgwp_move_by(bgwp_ctx *x, int a, int dr, int dc)
{
    if (!bgwp_agent_ok(x, a)) return 0;
    if (!(x->c->sp->klass[a] & BGW_AG_MOVING) || !(x->c->flags[a] & BGW_ST_IN_GRID)) return 0;
    return try_move(x->c, a, dr, dc);
}
BGWP_FN int bgwp_attack(bgwp_ctx *x, int a, int *victims)
{
    Ctx *c = x->c;
    if (!bgwp_agent_ok(x, a)) return -1;
    if (c->sp->attack_actor == BGW_ATTACK_NONE || c->learner_of[a] < 0) return -1;
    int nv = 0;
    const int status = process_attack(c, a, (const uint8_t *)(c->actions + (size_t)c->learner_of[a] * c->astride) + 2, victims, &nv);
    return status ? nv : -1;
}

/* ---- writes ---------------------------------------------------------------------------------------------------------- */
BGWP_FN void bgwp_set_health(bgwp_ctx *x, int a, double h) { if (bgwp_agent_ok(x, a)) set_health(x->c, a, h); }
BGWP_FN void bgwp_set_active(bgwp_ctx *x, int a, int on)
{
    if (!bgwp_agent_ok(x, a)) return;
    if (on) x->c->flags[a] |= BGW_ST_ACTIVE; else x->c->flags[a] &= (uint8_t)~BGW_ST_ACTIVE;
}
BGWP_FN int bgwp_place(bgwp_ctx *x, int a, int r, int col)
{
    if (!bgwp_agent_ok(x, a) || !bgwp_cell_ok(x, r, col)) return 0;
    if (x->c->flags[a] & BGW_ST_IN_GRID) { bgwp_fail(x); return 0; }
    return grid_place(x->c, a, r * x->c->W + col);
}
BGWP_FN void bgwp_remove(bgwp_ctx *x, int a) { if (bgwp_agent_ok(x, a)) grid_remove(x->c, a); }
BGWP_FN void bgwp_add_reward(bgwp_ctx *x, int a, double v)
{
    Ctx *c = x->c;
    if (!bgwp_agent_ok(x, a)) return;
    /* under AllStepManager a reward nobody will report is dropped, as in the step kernel (bgw_program.h) */
    const uint8_t k = c->sp->klass[a];
    if (c->sp->manager != BGW_MANAGER_ALL_STEP || (!(k & BGW_AG_LEARNER) && (k & BGW_AG_HEALTH)) ||
        ((k & BGW_AG_LEARNER) && !(c->flags[a] & BGW_ST_DONE_REPORTED)))
        c->racc[a] += v;
}

/* ---- randomness ------------------------------------------------------------------------------------------------------ */
BGWP_FN double bgwp_uniform(const bgwp_ctx *x, int slot, int k)
{
    if ((unsigned)slot >= 4096u || (unsigned)k >= 65536u) { bgwp_fail(x); return 0.0; }
    return bgw_u01(draw(x->c, BGW_SITE_PROGRAM, (uint32_t)slot, (uint32_t)k));
}

#include BGW_PROGRAM_FILE

/* ---- the oracle's calls into the program (bgw_oracle.c declares them): -1 from a hook the program does not define ------- */
static void user_step(Ctx *c)
{
    bgwp_ctx x = {c};
    bgwp_step(&x);
}

static int user_done(const Ctx *c, int a)
{
#ifdef BGWP_HAS_GET_DONE
    const bgwp_ctx x = {(Ctx *)c};
    return bgwp_get_done(&x, a) != 0;
#else
    (void)c; (void)a;
    return -1;
#endif
}

static int user_all_done(const Ctx *c)
{
#ifdef BGWP_HAS_GET_ALL_DONE
    const bgwp_ctx x = {(Ctx *)c};
    return bgwp_get_all_done(&x) != 0;
#else
    (void)c;
    return -1;
#endif
}

static double user_reward(const Ctx *c, int a, double acc)
{
#ifdef BGWP_HAS_GET_REWARD
    const bgwp_ctx x = {(Ctx *)c};
    return bgwp_get_reward(&x, a, acc);
#else
    (void)c; (void)a;
    return acc;
#endif
}
