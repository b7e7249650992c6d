/*
 * bgw_program.h -- the step-program API: a user-written simulation step() that runs inside the engine.
 *
 * In the reference a simulation is a subclass of GridWorldSimulation / SmartGridWorldSimulation whose author writes
 * step(action_dict) and, sometimes, get_done / get_all_done / get_reward (abmarl/sim/agent_based_simulation.py:238-294).
 * Here that code is ONE C source text, a "step program".  It is compiled twice from the same text:
 *   - by NVRTC as CUDA C++ into the general step kernel (bgw_set_program, include/bgw.h; abmarl_b200/csrc/bgw_program.cuh),
 *   - by gcc as C into the CPU oracle (oracle/bgw_oracle_program.c over oracle/bgw_oracle.c), which checks it bit for bit.
 * So a program is written in the common subset of C99 and C++17: no references, templates, classes, `bool` or library calls.
 * Its own functions are declared with BGWP_FN.
 *
 * What a program defines
 *   required  BGWP_FN void bgwp_step(bgwp_ctx *c)
 *               = sim.step(action_dict).  Runs on one thread per env, once per manager step, after the manager has
 *               collected the actions (all_step_manager.py:66, turn_based_manager.py:46).
 *   optional, each announced by a #define before its definition:
 *     #define BGWP_HAS_GET_DONE       BGWP_FN int bgwp_get_done(const bgwp_ctx *c, int a)
 *     #define BGWP_HAS_GET_ALL_DONE   BGWP_FN int bgwp_get_all_done(const bgwp_ctx *c)
 *     #define BGWP_HAS_GET_REWARD     BGWP_FN double bgwp_get_reward(const bgwp_ctx *c, int a, double acc)
 *               acc is the reward accumulated for `a` since its last report (self.rewards[id], smart.py:101-104); the
 *               value returned is what the manager reports (e.g. multi_maze_navigation.py:56-59).  The accumulator is
 *               cleared after the report either way.
 *   A hook that is not defined follows the SmartGridWorldSimulation rule over the spec's done components (smart.py:106-120:
 *   all() over them, so with none at all every agent is done) and reports the accumulator as it is.  The hooks take a const context: they may be
 *   evaluated on any thread, any number of times, so they must only read.  Every function that changes the simulation
 *   takes a non-const bgwp_ctx *: calling one from a hook does not compile (C++: type error; the oracle's gcc build
 *   runs with -Werror=discarded-qualifiers).
 *
 * Indices: agents are numbered in `sim.agents` dict order, 0 .. bgwp_n_agents(c) - 1; cells are (row, col).
 *
 * Bad input: a call that names an agent outside [0, A), a cell off the grid, an acting slot, action byte or random slot
 * out of range does nothing and returns 0 (-1 where the function returns an agent index).  The env then records
 * BgwState.error = 3 and reports BGW_ENV_ERROR | BGW_ENV_ALL_DONE at the end of that step, as a failed placement does
 * (include/bgw.h): the env is inert until it is reset.
 *
 * Arithmetic: both compilations evaluate double arithmetic in IEEE float64 without contraction (NVRTC --fmad=false, gcc
 * -ffp-contract=off).  That is the ONLY guarantee: sqrt, exp, pow and every other library function may differ between the
 * two and must not be used.  Keep to + - * / and comparisons, and to integer arithmetic.
 */
#ifndef BGW_PROGRAM_H_
#define BGW_PROGRAM_H_

#include "bgw.h"

#if defined(__CUDACC__)
#define BGWP_FN static __device__
#else
#define BGWP_FN static inline
#endif

typedef struct bgwp_ctx bgwp_ctx;

BGWP_FN void bgwp_step(bgwp_ctx *c);

/* ---- the acting set and the env ------------------------------------------------------------------------------------ */
/* number of acting slots: the learners under AllStepManager, 1 under TurnBasedManager */
BGWP_FN int bgwp_n_acting(const bgwp_ctx *c);
/* agent of acting slot i in the order the manager hands the actions over (dict order, the caller's `order`, the keyed order
 * of randomize_action_input, all_step_manager.py:59-66; the learner whose turn it is, turn_based_manager.py:46), or -1 when
 * that learner was already reported done and sent no action (all_step_manager.py:59-61) */
BGWP_FN int bgwp_acting(const bgwp_ctx *c, int i);
BGWP_FN int bgwp_step_index(const bgwp_ctx *c);   /* number of this step in the episode: 1 on the first step after a reset */
BGWP_FN int bgwp_rows(const bgwp_ctx *c);         /* Grid.rows grid.py:20 */
BGWP_FN int bgwp_cols(const bgwp_ctx *c);         /* Grid.cols */
BGWP_FN int bgwp_n_agents(const bgwp_ctx *c);     /* len(sim.agents) */

/* ---- reads ----------------------------------------------------------------------------------------------------------- */
BGWP_FN int bgwp_encoding(const bgwp_ctx *c, int a);     /* GridWorldAgent.encoding agent.py:31-37 */
BGWP_FN int bgwp_klass(const bgwp_ctx *c, int a);        /* BGW_AG_* bits: which agent classes it derives from */
BGWP_FN int bgwp_role(const bgwp_ctx *c, int a);         /* the spec's role byte (DeviceProgram(roles=...)) */
BGWP_FN int bgwp_active(const bgwp_ctx *c, int a);       /* PrincipleAgent.active agent.py:192-196 */
BGWP_FN int bgwp_in_grid(const bgwp_ctx *c, int a);      /* the agent is in its cell's dict grid.py:107-140 */
BGWP_FN int bgwp_row(const bgwp_ctx *c, int a);          /* agent.position[0]; stays where the agent left the grid
                                                            (actor.py:356-358); -1 if it was never placed */
BGWP_FN int bgwp_col(const bgwp_ctx *c, int a);          /* agent.position[1] */
BGWP_FN double bgwp_health(const bgwp_ctx *c, int a);    /* HealthAgent.health agent.py:185-196 (0 for other agents) */
BGWP_FN int bgwp_ammo(const bgwp_ctx *c, int a);         /* AmmoAgent.ammo agent.py:299-309 (0 for other agents) */
BGWP_FN int bgwp_orientation(const bgwp_ctx *c, int a);  /* OrientationAgent.orientation 1..4 agent.py:344 (0: none) */
/* byte k of a's action row (layout: bgw.h, bgw_step); 0 for an agent that is not a learner (it has no action) */
BGWP_FN int bgwp_action(const bgwp_ctx *c, int a, int k);
BGWP_FN int bgwp_query(const bgwp_ctx *c, int a, int r, int col);   /* Grid.query grid.py:81-105 */
/* the occupants of cell (r, col) in dict order (grid.py:24,125): the first one, then the one after a; -1 at the end.
 * Read the next occupant before you move or remove the current one. */
BGWP_FN int bgwp_first_occupant(const bgwp_ctx *c, int r, int col);
BGWP_FN int bgwp_next_occupant(const bgwp_ctx *c, int a);

/* ---- actors ---------------------------------------------------------------------------------------------------------- */
/* move_actor.process_action(agent, action) with a's own action (actor.py:82-114 MoveActor, :161-194 CrossMoveActor,
 * :208-234 DriftMoveActor): 1 on success, 0 on failure or None (not a MovingAgent, not a learner, not in the grid) */
BGWP_FN int bgwp_move(bgwp_ctx *c, int a);
/* the same move by (dr, dc) instead of a's action, for scripted agents (actor.py:99-114; no orientation update) */
BGWP_FN int bgwp_move_by(bgwp_ctx *c, int a, int dr, int dc);
/* attack_actor.process_action(agent, action) with a's own action (actor.py:306-361 over _determine_attack :455-501 Binary,
 * :521-582 EncodingBased, :601-658 RestrictedSelective, :681-728 Selective): -1 when no attack was attempted (not an
 * AttackingAgent, not a learner, or the action asks for none); otherwise the number n <= BGW_MAX_VICTIMS of attacked agents
 * after the ammo filter, written to victims[0..n) (repeats possible with stacked attacks).  Damage is applied and the agents
 * it kills are removed from the grid.  No reward is given and the attacker's own activity is not checked: both are the
 * step's business (team_battle_example.py:37-47). */
BGWP_FN int bgwp_attack(bgwp_ctx *c, int a, int *victims);

/* ---- writes ---------------------------------------------------------------------------------------------------------- */
BGWP_FN void bgwp_set_health(bgwp_ctx *c, int a, double h);   /* HealthAgent.health setter: clamped to [0, 1], active = h > 0
                                                                 agent.py:192-196 */
BGWP_FN void bgwp_set_active(bgwp_ctx *c, int a, int on);     /* agent.active = on (reach_the_target.py:144) */
/* Grid.place grid.py:107-129: 0 (nothing placed) when Grid.query refuses; an agent that is in the grid already must be
 * removed first (else: bad input) */
BGWP_FN int bgwp_place(bgwp_ctx *c, int a, int r, int col);
BGWP_FN void bgwp_remove(bgwp_ctx *c, int a);                 /* Grid.remove grid.py:131-140 (nothing if not in the grid) */
/* self.rewards[id] += x.  Under AllStepManager a reward that will never be reported is dropped: one for a learner that was
 * reported done already, or for an entity that is neither a learner nor a HealthAgent. */
BGWP_FN void bgwp_add_reward(bgwp_ctx *c, int a, double x);

/* ---- randomness ------------------------------------------------------------------------------------------------------ */
/* u in [0, 1), float64: a pure function of (seed, global env, episode, step, slot, k) -- keyed Philox site
 * BGW_SITE_PROGRAM (bgw_philox.h), slot in [0, 4096), k in [0, 65536).  The same (slot, k) gives the same number within a
 * step; vary them to get independent draws.  Allowed in the hooks. */
BGWP_FN double bgwp_uniform(const bgwp_ctx *c, int slot, int k);

#endif /* BGW_PROGRAM_H_ */
