/*
 * bgw_general.cu -- the instantiations of the general step kernel (bgw_dev.cuh, bgw_step_kernel): one translation unit of
 * its own (they take two minutes to compile; the host side and the specialised kernel build in parallel).
 */
#include "bgw_dev.cuh"

/* the general step kernel specialised for a sim program / attack actor (bgw_dev.cuh, bgw_step_kernel) */
const void *bgw_general_step_fn(int program, int attack_actor)
{
    switch (program) {
    case BGW_PROG_TEAM_BATTLE:
        switch (attack_actor) {
        case BGW_ATTACK_BINARY: return (const void *)bgw_step_kernel<BGW_PROG_TEAM_BATTLE, BGW_ATTACK_BINARY>;
        case BGW_ATTACK_ENCODING: return (const void *)bgw_step_kernel<BGW_PROG_TEAM_BATTLE, BGW_ATTACK_ENCODING>;
        case BGW_ATTACK_RESTRICTED: return (const void *)bgw_step_kernel<BGW_PROG_TEAM_BATTLE, BGW_ATTACK_RESTRICTED>;
        case BGW_ATTACK_SELECTIVE: return (const void *)bgw_step_kernel<BGW_PROG_TEAM_BATTLE, BGW_ATTACK_SELECTIVE>;
        default: break;
        }
        break;
    case BGW_PROG_REACH_TARGET:                      /* examples/rllib_reach_the_target.py: SelectiveAttackActor */
        if (attack_actor == BGW_ATTACK_SELECTIVE) return (const void *)bgw_step_kernel<BGW_PROG_REACH_TARGET, BGW_ATTACK_SELECTIVE>;
        break;
    case BGW_PROG_TRAFFIC:                           /* traffic_corridor.py: movers only */
        if (attack_actor == BGW_ATTACK_NONE) return (const void *)bgw_step_kernel<BGW_PROG_TRAFFIC, BGW_ATTACK_NONE>;
        break;
    case BGW_PROG_MAZE: return (const void *)bgw_step_kernel<BGW_PROG_MAZE, -1>;
    case BGW_PROG_MULTI_MAZE: return (const void *)bgw_step_kernel<BGW_PROG_MULTI_MAZE, -1>;
    case BGW_PROG_PACMAN: return (const void *)bgw_step_kernel<BGW_PROG_PACMAN, -1>;
    /* BGW_PROG_PACMAN_SIMPLE: measured slower in its own instantiation (4.0e8 against 4.9e8 agent-steps/s): all-in-one */
    default: break;
    }
    return (const void *)bgw_step_kernel<-1, -1>;    /* every program and actor in one */
}
