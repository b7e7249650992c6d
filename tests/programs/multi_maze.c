/* MultiMazeNavigationSim (multi_maze_navigation.py:17-74) as a step program: step, get_done, get_all_done and the
 * get_reward override.  Constants: TARGET (agent), MOVE_FAIL, ENTROPY, REACHED.  Role 1 = navigator. */
BGWP_FN int at_target(const bgwp_ctx *c, int a)
{
    return bgwp_row(c, a) == bgwp_row(c, TARGET) && bgwp_col(c, a) == bgwp_col(c, TARGET);
}

BGWP_FN void bgwp_step(bgwp_ctx *c)                        /* :40-48 */
{
    const int n = bgwp_n_acting(c);
    for (int i = 0; i < n; ++i) {
        const int a = bgwp_acting(c, i);
        if (a < 0) continue;
        if (!bgwp_move(c, a)) bgwp_add_reward(c, a, MOVE_FAIL);
        bgwp_add_reward(c, a, ENTROPY);
    }
}

#define BGWP_HAS_GET_DONE
BGWP_FN int bgwp_get_done(const bgwp_ctx *c, int a) { return at_target(c, a); }   /* :61-64 */

#define BGWP_HAS_GET_ALL_DONE
BGWP_FN int bgwp_get_all_done(const bgwp_ctx *c)          /* :66-71 */
{
    for (int a = 0; a < bgwp_n_agents(c); ++a)
        if (bgwp_role(c, a) == 1 && !at_target(c, a)) return 0;
    return 1;
}

#define BGWP_HAS_GET_REWARD
BGWP_FN double bgwp_get_reward(const bgwp_ctx *c, int a, double acc)   /* :56-59 */
{
    return at_target(c, a) ? REACHED : acc;
}
