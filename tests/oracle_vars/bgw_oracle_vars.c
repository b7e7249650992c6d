/*
 * bgw_oracle_vars.c -- the CPU reference of a step program's variables (include/bgw_program.h: bgwp_env_var, bgwp_set_env_var,
 * bgwp_agent_var, bgwp_set_agent_var, bgwp_n_env_vars, bgwp_n_agent_vars).  TEST INFRASTRUCTURE ONLY.
 *
 * It includes the oracle built with a program and its dynamic-order manager step (tests/oracle_dynamic/bgw_oracle_dynamic.c,
 * which includes oracle/bgw_oracle_program.c and oracle/bgw_oracle.c), defines the six API functions the program calls, and
 * wraps the entry points that reset an env so that every reset writes the initial row:
 *   bgwo_bind_program_vars   the counts, the initial row [n_env + A * n_agent] and the rows [E][n_env + A * n_agent] of the
 *                            next calls (BgwState does not carry them; the library is shared by every env of one program)
 *   bgwo_reset_vars          bgwo_reset, then the initial row for the envs env_mask selects (a failed placement included)
 *   bgwo_step_vars           bgwo_step / bgwo_step_dynamic, then the initial row for the envs the step auto-reset
 *                            (BGW_ENV_RESET): a reset runs no program code, so writing the row after it is the same as during
 * The device twin is the ProgVars row of abmarl_b200/csrc/bgw_program.cuh and bgw_dev.cuh.
 *
 * Build (tests/vars_oracle.py): oracle/build.py's gcc flags and
 *     -DBGW_PROGRAM_FILE='"<program.c>"' -o <lib.so> tests/oracle_vars/bgw_oracle_vars.c -lm
 * (-Werror=discarded-qualifiers: a hook that writes a variable fails, as for the other mutating calls.)
 */
#include "../oracle_dynamic/bgw_oracle_dynamic.c"

static struct { int n_env, n_agent; const double *init; double *vars; } prog_vars;

static int vars_stride(int A) { return prog_vars.n_env + A * prog_vars.n_agent; }

int bgwo_bind_program_vars(int n_env, int n_agent, const double *init, double *vars)
{
    prog_vars.n_env = n_env; prog_vars.n_agent = n_agent; prog_vars.init = init; prog_vars.vars = vars;
    return 0;
}

/* ---- the API (declared in include/bgw_program.h, called by the program included above) ------------------------------ */
BGWP_FN int bgwp_n_env_vars(const bgwp_ctx *x) { (void)x; return prog_vars.n_env; }
BGWP_FN int bgwp_n_agent_vars(const bgwp_ctx *x) { (void)x; return prog_vars.n_agent; }
static double *env_row(const bgwp_ctx *x) { return prog_vars.vars + (size_t)x->c->env * vars_stride(x->c->A); }
static double *bgwp_env_slot(const bgwp_ctx *x, int k)
{
    if ((unsigned)k >= (unsigned)prog_vars.n_env) { bgwp_fail(x); return NULL; }
    return env_row(x) + k;
}
static double *bgwp_agent_slot(const bgwp_ctx *x, int a, int k)
{
    if (!bgwp_agent_ok(x, a)) return NULL;
    if ((unsigned)k >= (unsigned)prog_vars.n_agent) { bgwp_fail(x); return NULL; }
    return env_row(x) + prog_vars.n_env + (size_t)a * prog_vars.n_agent + k;
}
BGWP_FN double bgwp_env_var(const bgwp_ctx *x, int k) { const double *p = bgwp_env_slot(x, k); return p ? *p : 0.0; }
BGWP_FN void bgwp_set_env_var(bgwp_ctx *x, int k, double v) { double *p = bgwp_env_slot(x, k); if (p) *p = v; }
BGWP_FN double bgwp_agent_var(const bgwp_ctx *x, int a, int k) { const double *p = bgwp_agent_slot(x, a, k); return p ? *p : 0.0; }
BGWP_FN void bgwp_set_agent_var(bgwp_ctx *x, int a, int k, double v) { double *p = bgwp_agent_slot(x, a, k); if (p) *p = v; }

/* ---- resets ------------------------------------------------------------------------------------------------------------ */
static void init_row(const BgwSpec *sp, int e)
{
    const int n = vars_stride(sp->n_agents);
    if (n) memcpy(prog_vars.vars + (size_t)e * n, prog_vars.init, sizeof(double) * (size_t)n);
}

int bgwo_reset_vars(const BgwSpec *sp, BgwState *st, const uint8_t *env_mask, int8_t *obs)
{
    const int rc = bgwo_reset(sp, st, env_mask, obs);
    for (int e = 0; e < sp->n_envs; ++e)
        if (!env_mask || env_mask[e]) init_row(sp, e);
    return rc;
}

int bgwo_step_vars(const BgwSpec *sp, BgwState *st, const int8_t *actions, const int16_t *order, int8_t *obs,
                   float *reward, double *reward64, uint8_t *done, uint8_t *all_done)
{
    const int rc = sp->manager == BGW_MANAGER_DYNAMIC_ORDER
        ? bgwo_step_dynamic(sp, st, actions, order, obs, reward, reward64, done, all_done)
        : bgwo_step(sp, st, actions, order, obs, reward, reward64, done, all_done);
    if (rc) return rc;
    for (int e = 0; e < sp->n_envs; ++e)
        if (all_done[e] & BGW_ENV_RESET) init_row(sp, e);
    return 0;
}
