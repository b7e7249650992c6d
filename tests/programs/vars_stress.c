/* Variables of a step program under stress (tests/test_program_vars_oracle.py, tests/test_gpu_program_vars.py): an env
 * scalar and an env array, two agent variables with per-agent initial values, and every hook reading them.
 * Constants: DONE_MOVES, ALL_DONE_STEPS.  Variables: STEPS, HIST[8] (env), ENERGY, MOVES (agent). */
BGWP_FN void bgwp_step(bgwp_ctx *c)
{
    int victims[BGW_MAX_VICTIMS];
    bgwp_set_env_var(c, STEPS, bgwp_env_var(c, STEPS) + 1.0);
    for (int i = 0; i < bgwp_n_acting(c); ++i) {
        const int a = bgwp_acting(c, i);
        if (a < 0 || !bgwp_active(c, a)) continue;
        const double e = bgwp_agent_var(c, a, ENERGY);
        if (e >= 1.0) {                                        /* moving costs energy, resting restores it */
            if (bgwp_move(c, a)) {
                bgwp_set_agent_var(c, a, ENERGY, e - 0.75);
                bgwp_set_agent_var(c, a, MOVES, bgwp_agent_var(c, a, MOVES) + 1.0);
            }
        } else bgwp_set_agent_var(c, a, ENERGY, e + 0.25);
        const int k = bgwp_action(c, a, 0) & 7;
        bgwp_set_env_var(c, HIST + k, bgwp_env_var(c, HIST + k) + 1.0);
        const int nv = bgwp_attack(c, a, victims);
        for (int t = 0; t < nv; ++t)
            if (!bgwp_active(c, victims[t])) bgwp_add_reward(c, a, bgwp_agent_var(c, victims[t], ENERGY));
        bgwp_add_reward(c, a, bgwp_agent_var(c, a, ENERGY) / 64.0);
    }
}

#define BGWP_HAS_GET_DONE
BGWP_FN int bgwp_get_done(const bgwp_ctx *c, int a)
{
    return !bgwp_active(c, a) || bgwp_agent_var(c, a, MOVES) >= DONE_MOVES;
}

#define BGWP_HAS_GET_ALL_DONE
BGWP_FN int bgwp_get_all_done(const bgwp_ctx *c)
{
    double hist = 0.0;
    for (int k = 0; k < 8; ++k) hist += bgwp_env_var(c, HIST + k);
    return bgwp_env_var(c, STEPS) >= ALL_DONE_STEPS || hist >= 4.0 * ALL_DONE_STEPS;
}

#define BGWP_HAS_GET_REWARD
BGWP_FN double bgwp_get_reward(const bgwp_ctx *c, int a, double acc)
{
    return acc + bgwp_agent_var(c, a, MOVES) / 128.0 + bgwp_env_var(c, HIST + (a & 7)) / 1024.0;
}

#define BGWP_HAS_NEXT_AGENT
BGWP_FN int bgwp_next_agent(const bgwp_ctx *c, int a)           /* the DynamicOrderManager's rule; the others ignore it */
{
    return !bgwp_active(c, a) || ((int)bgwp_env_var(c, STEPS) + a) % 3 == 0 || bgwp_agent_var(c, a, ENERGY) >= 1.5;
}
