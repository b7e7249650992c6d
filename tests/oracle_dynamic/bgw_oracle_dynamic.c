/*
 * bgw_oracle_dynamic.c -- the CPU reference of a step program under the dynamic-order manager (include/bgw_program.h,
 * bgwp_next_agent).  TEST INFRASTRUCTURE ONLY.
 *
 * It includes the oracle built with a program (oracle/bgw_oracle_program.c, which includes oracle/bgw_oracle.c) and adds one
 * entry point, bgwo_step_dynamic: the oracle's manager step for a BGW_PROG_USER spec under BGW_MANAGER_DYNAMIC_ORDER, over
 * the oracle's own primitives (grid_build, prog_step, prog_all_done, emit, env_reset).  It is the twin of the
 * BGW_USER_PROGRAM branches of bgw_step_body (abmarl_b200/csrc/bgw_dev.cuh):
 *   1. the acting set: on the first step of an episode BgwState.turn (the reset names learner 0), otherwise the learners
 *      carrying BGW_ST_NEXT; learners already reported done are left out; dict order, whatever the caller's order;
 *   2. the program's step, then get_all_done;
 *   3. done: every learner not yet reported receives (obs, reward, done) (dynamic_order_manager.py:43-51);
 *   4. otherwise the hook is evaluated for every learner, and each named learner not yet reported receives (obs, reward,
 *      done) and is marked reported if done; the named ones that are not done carry BGW_ST_NEXT, BgwState.turn is the
 *      lowest of them or -1.
 * Every other call (bgwo_reset, bgwo_sample_actions, bgwo_observe, bgwo_step for the other managers) is the oracle's own.
 *
 * Build (tests/dynamic_cases.py, build_dynamic): oracle/build.py's gcc flags and
 *     -DBGW_PROGRAM_FILE='"<program.c>"' -o <lib.so> tests/oracle_dynamic/bgw_oracle_dynamic.c -lm
 * (-Werror=discarded-qualifiers: a next_agent hook that calls a mutating API function fails, as the other hooks do.)
 */
#include "../../oracle/bgw_oracle_program.c"

#ifdef BGWP_HAS_NEXT_AGENT
#define BGWO_HAS_NEXT_AGENT 1
#else
#define BGWO_HAS_NEXT_AGENT 0
#endif

static int user_next_agent(const Ctx *c, int a)
{
#ifdef BGWP_HAS_NEXT_AGENT
    const bgwp_ctx x = {(Ctx *)c};
    return bgwp_next_agent(&x, a) != 0;
#else
    (void)c; (void)a;
    return 0;
#endif
}

/* 1. */
static void named_acting(Ctx *c, int first_step)
{
    c->n_acting = 0;
    for (int l = 0; l < c->L; ++l) {
        const int a = c->agent_of[l];
        const int named = first_step ? l == c->st->turn[c->env] : (c->flags[a] & BGW_ST_NEXT) != 0;
        if (named && !(c->flags[a] & BGW_ST_DONE_REPORTED)) c->acting[c->n_acting++] = a;
    }
}

/* 4. (dynamic_order_manager.py:52-85 over sim.next_agent = the learners the hook names) */
static void named_emit(Ctx *c, int8_t *obs_env, int stride, float *rew, double *rew64, uint8_t *dn)
{
    uint8_t *named = (uint8_t *)malloc((size_t)c->L + 1);
    for (int l = 0; l < c->L; ++l) named[l] = (uint8_t)user_next_agent(c, c->agent_of[l]);
    int next = -1;
    for (int l = 0; l < c->L; ++l) {
        const int a = c->agent_of[l];
        c->flags[a] &= (uint8_t)~BGW_ST_NEXT;
        if (!named[l] || (c->flags[a] & BGW_ST_DONE_REPORTED)) continue;
        emit(c, l, obs_env, stride, rew, rew64, dn);
        if (dn[l] & BGW_OUT_DONE) c->flags[a] |= BGW_ST_DONE_REPORTED;
        else {
            c->flags[a] |= BGW_ST_NEXT;
            if (next < 0) next = l;
        }
    }
    c->st->turn[c->env] = (int16_t)next;
    free(named);
}

/* bgwo_step's arguments; non-zero (nothing touched) for any other spec, or when the program has no next_agent hook */
int bgwo_step_dynamic(const BgwSpec *sp, BgwState *st, const int8_t *actions, const int16_t *order, int8_t *obs,
                      float *reward, double *reward64, uint8_t *done, uint8_t *all_done)
{
    (void)order;
    if (!BGWO_HAS_NEXT_AGENT || sp->program != BGW_PROG_USER || sp->manager != BGW_MANAGER_DYNAMIC_ORDER) return 1;
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
            }
            all_done[e] = st->env_flags[e];
            continue;
        }
        grid_build(&c);
        st->step[e] += 1;
        st->stats[(size_t)e * BGW_STAT_COUNT + BGW_STAT_ENV_STEPS]++;

        named_acting(&c, st->step[e] == 1);                     /* 1. */
        prog_step(&c);                                          /* 2. */
        const int env_done = prog_all_done(&c);
        if (env_done) {                                         /* 3. */
            for (int k = 0; k < L; ++k)
                if (!(c.flags[c.agent_of[k]] & BGW_ST_DONE_REPORTED)) emit(&c, k, obs_env, stride, rew, rew64, dn);
        } else named_emit(&c, obs_env, stride, rew, rew64, dn);  /* 4. */

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
