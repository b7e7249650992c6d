/* DynamicOrderMultiMazeSim's next_agent rule (abmarl_b200/examples/sims.py) as a next_agent hook, appended to
 * multi_maze.c: the agent that just acted if this step took it to the target (its last report), then the next navigator
 * after it in dict order that is not at the target (itself, if it is the only one left). */
#define BGWP_HAS_NEXT_AGENT
BGWP_FN int bgwp_next_agent(const bgwp_ctx *c, int a)
{
    const int last = bgwp_acting(c, 0);
    if (a == last && at_target(c, a)) return 1;
    const int n = bgwp_n_agents(c);
    for (int k = 1; k <= n; ++k) {
        const int b = (last + k) % n;
        if (bgwp_role(c, b) == 1 && !at_target(c, b)) return b == a;
    }
    return 0;
}
