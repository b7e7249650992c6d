/*
 * program_oracle.c -- the CPU oracle with a user step program (include/bgw_program.h) compiled in.  TEST INFRASTRUCTURE ONLY.
 *
 * It includes oracle/bgw_oracle.c for everything that does not depend on the program -- grid, actors, observers, placement,
 * reset, sampling -- implements the step-program API over those primitives, includes the program, and restates the manager
 * step (bgwo_step: AllStepManager, TurnBasedManager) around the program's step() and hooks.  The device twin is
 * abmarl_b200/csrc/bgw_program.cuh + bgw_step_body; tests/program_oracle.py builds and loads this file.
 *
 * Build: gcc -O2 -fPIC -shared -ffp-contract=off -fno-fast-math -Werror=discarded-qualifiers
 *            -DBGW_PROGRAM_FILE='"<program.c>"' -o <lib.so> tests/program_oracle.c -lm
 * (-Werror=discarded-qualifiers: a get_done / get_all_done / get_reward hook that calls a mutating API function fails.)
 */
#define bgwo_step bgwo_step_builtin      /* the built-in programs' step; this file defines the program's bgwo_step */
#include "../oracle/bgw_oracle.c"
#undef bgwo_step
#include "../include/bgw_program.h"

struct bgwp_ctx {
    Ctx *c;
    const int *acting;        /* [n_acting] agent per acting slot, -1 = reported done already */
    int n_acting;
    const int8_t *actions;    /* this env's action rows */
    uint32_t *err;            /* bad input from the program: BgwState.error at the end of the step */
};                            /* the hooks get a const bgwp_ctx: a mutating API call from one discards the qualifier */

static int bgwp_fail(const bgwp_ctx *x) { *x->err = 3; return 0; }
static int bgwp_agent_ok(const bgwp_ctx *x, int a) { return ((unsigned)a < (unsigned)x->c->A) || bgwp_fail(x); }
static int bgwp_cell_ok(const bgwp_ctx *x, int r, int col) { return ((unsigned)r < (unsigned)x->c->H && (unsigned)col < (unsigned)x->c->W) || bgwp_fail(x); }

/* ---- the acting set and the env ------------------------------------------------------------------------------------ */
BGWP_FN int bgwp_n_acting(const bgwp_ctx *x) { return x->n_acting; }
BGWP_FN int bgwp_acting(const bgwp_ctx *x, int i)
{
    if ((unsigned)i >= (unsigned)x->n_acting) { bgwp_fail(x); return -1; }
    return x->acting[i];
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
    return x->actions[(size_t)x->c->learner_of[a] * x->c->astride + k];
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
    return process_move(c, a, x->actions + (size_t)c->learner_of[a] * c->astride);
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
    const int status = process_attack(c, a, (const uint8_t *)(x->actions + (size_t)c->learner_of[a] * c->astride) + 2, victims, &nv);
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

/* ---- the program's get_done / get_all_done / get_reward, else the SmartGridWorldSimulation rule (smart.py:101-120) ------ */
static int user_done(const bgwp_ctx *x, int a)
{
#ifdef BGWP_HAS_GET_DONE
    return bgwp_get_done(x, a) != 0;
#else
    return smart_done(x->c, a);
#endif
}

static int user_all_done(const bgwp_ctx *x)
{
#ifdef BGWP_HAS_GET_ALL_DONE
    return bgwp_get_all_done(x) != 0;
#else
    return smart_all_done(x->c);
#endif
}

static double user_take_reward(const bgwp_ctx *x, int a)
{
    double r = x->c->racc[a];
#ifdef BGWP_HAS_GET_REWARD
    r = bgwp_get_reward(x, a, r);
#endif
    x->c->racc[a] = 0.0;
    return r;
}

static void user_emit(const bgwp_ctx *x, int l, int8_t *obs_env, int stride, float *rew, double *rew64, uint8_t *done)
{
    Ctx *c = x->c;
    const int a = c->agent_of[l];
    if (obs_env) observe_agent(c, a, obs_env + (size_t)l * stride, stride);
    const double r = user_take_reward(x, a);
    const int d = user_done(x, a);
    if (rew) rew[l] = (float)r;
    if (rew64) rew64[l] = r;
    done[l] = (uint8_t)(BGW_OUT_VALID | (d ? BGW_OUT_DONE : 0));
    c->st->stats[(size_t)c->env * BGW_STAT_COUNT + BGW_STAT_AGENT_STEPS]++;
}

/* One manager step (all_step_manager.py:51-95 / turn_based_manager.py:34-94) of every env with the program as sim.step.
 * Under AllStepManager the program sees one acting slot per learner in processing order, -1 for those reported done
 * (bgwp_acting); bad input from the program ends the env with BgwState.error = 3 (bgw_program.h). */
int bgwo_step(const BgwSpec *sp, BgwState *st, const int8_t *actions, const int16_t *order, int8_t *obs,
              float *reward, double *reward64, uint8_t *done, uint8_t *all_done)
{
    if (sp->program != BGW_PROG_USER || sp->manager == BGW_MANAGER_DYNAMIC_ORDER) return 1;
    Ctx c; ctx_init(&c, sp, st);
    BgwDims d; bgwo_dims(sp, &d);
    const int L = c.L, stride = d.obs_stride;
    int *acting = (int *)malloc(sizeof(int) * (size_t)(L + 1));
    for (int e = 0; e < sp->n_envs; ++e) {
        ctx_env(&c, e);
        int8_t *obs_env = obs ? obs + (size_t)e * L * stride : NULL;
        float *rew = reward ? reward + (size_t)e * L : NULL;
        double *rew64 = reward64 ? reward64 + (size_t)e * L : NULL;
        uint8_t *dn = done + (size_t)e * L;
        uint32_t err = 0;
        bgwp_ctx x = {&c, acting, 0, actions + (size_t)e * L * c.astride, &err};
        for (int l = 0; l < L; ++l) { dn[l] = 0; if (rew) rew[l] = 0.f; if (rew64) rew64[l] = 0.0; }

        if (st->env_flags[e] & BGW_ENV_ALL_DONE) {
            if (sp->auto_reset) {
                env_reset(&c, obs_env, stride);
                st->env_flags[e] |= BGW_ENV_RESET;
            }
            all_done[e] = st->env_flags[e];
            continue;
        }
        grid_build(&c);
        st->step[e] += 1;
        st->stats[(size_t)e * BGW_STAT_COUNT + BGW_STAT_ENV_STEPS]++;
        int env_done = 0;

        if (sp->manager == BGW_MANAGER_ALL_STEP) {
            for (int i = 0; i < L; ++i) acting[i] = c.agent_of[order ? order[(size_t)e * L + i] : i];
            /* all_step_manager.py:62-65: the keyed order of this step */
            if (!order && sp->randomize_action_input) keyed_order(&c, BGW_SITE_ORDER, st->step[e], acting, L);
            for (int i = 0; i < L; ++i) if (c.flags[acting[i]] & BGW_ST_DONE_REPORTED) acting[i] = -1;   /* :59-61 */
            x.n_acting = L;
            bgwp_step(&x);                                       /* :66 */
            for (int l = 0; l < L; ++l)                           /* :68-87 */
                if (!(c.flags[c.agent_of[l]] & BGW_ST_DONE_REPORTED)) user_emit(&x, l, obs_env, stride, rew, rew64, dn);
            int remaining = 0;
            for (int l = 0; l < L; ++l) {
                const int a = c.agent_of[l];
                if (dn[l] & BGW_OUT_DONE) c.flags[a] |= BGW_ST_DONE_REPORTED;
                if (!(c.flags[a] & BGW_ST_DONE_REPORTED)) ++remaining;
            }
            env_done = user_all_done(&x) || remaining == 0;       /* :90-93 */
        } else {
            int l = st->turn[e];
            acting[0] = c.agent_of[l];
            x.n_acting = 1;
            bgwp_step(&x);                                        /* :46 */
            env_done = user_all_done(&x);                         /* :48 */
            if (env_done) {                                       /* :49-57 */
                for (int k = 0; k < L; ++k)
                    if (!(c.flags[c.agent_of[k]] & BGW_ST_DONE_REPORTED)) user_emit(&x, k, obs_env, stride, rew, rew64, dn);
            } else {
                for (;;) {                                        /* :59-92 */
                    l = (l + 1) % L;
                    const int a = c.agent_of[l];
                    if (c.flags[a] & BGW_ST_DONE_REPORTED) continue;
                    if (user_done(&x, a)) {
                        user_emit(&x, l, obs_env, stride, rew, rew64, dn);
                        c.flags[a] |= BGW_ST_DONE_REPORTED;
                        int remaining = 0;
                        for (int k = 0; k < L; ++k) if (!(c.flags[c.agent_of[k]] & BGW_ST_DONE_REPORTED)) ++remaining;
                        if (remaining) continue;
                        env_done = 1;
                        break;
                    }
                    user_emit(&x, l, obs_env, stride, rew, rew64, dn);
                    break;
                }
                st->turn[e] = (int16_t)l;
            }
        }
        uint8_t ef = 0;
        if (env_done) ef |= BGW_ENV_ALL_DONE;
        if (sp->horizon > 0 && (int)st->step[e] >= sp->horizon) ef |= BGW_ENV_ALL_DONE | BGW_ENV_TRUNCATED;
        if (err) { ef |= BGW_ENV_ERROR | BGW_ENV_ALL_DONE; st->error[e] = err; }
        if (ef & BGW_ENV_ALL_DONE) st->stats[(size_t)e * BGW_STAT_COUNT + BGW_STAT_EPISODES]++;
        st->env_flags[e] = ef;
        all_done[e] = ef;
    }
    free(acting);
    ctx_free(&c);
    return 0;
}
