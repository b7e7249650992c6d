/* TeamBattleSim.step (team_battle_example.py:33-59) as a step program: the built-in BGW_PROG_TEAM_BATTLE, re-expressed over
 * the program API.  Constants: ATTACK_FAIL, KILL, DIE, MOVE_FAIL, ENTROPY.  No hooks: the Smart-sim done rule applies. */
BGWP_FN void bgwp_step(bgwp_ctx *c)
{
    int victims[BGW_MAX_VICTIMS];
    const int n = bgwp_n_acting(c);
    for (int i = 0; i < n; ++i) {                          /* :35-47 */
        const int a = bgwp_acting(c, i);
        if (a < 0 || !bgwp_active(c, a)) continue;
        const int nv = bgwp_attack(c, a, victims);
        if (nv == 0) bgwp_add_reward(c, a, ATTACK_FAIL);
        for (int t = 0; t < nv; ++t)
            if (!bgwp_active(c, victims[t])) {
                bgwp_add_reward(c, victims[t], DIE);
                bgwp_add_reward(c, a, KILL);
            }
    }
    for (int i = 0; i < n; ++i) {                          /* :50-55 */
        const int a = bgwp_acting(c, i);
        if (a < 0 || !bgwp_active(c, a)) continue;
        if (!bgwp_move(c, a)) bgwp_add_reward(c, a, MOVE_FAIL);
    }
    for (int i = 0; i < n; ++i) {                          /* :58-59 */
        const int a = bgwp_acting(c, i);
        if (a >= 0) bgwp_add_reward(c, a, ENTROPY);
    }
}
