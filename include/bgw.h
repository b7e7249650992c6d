/*
 * bgw.h -- C-ABI of the B200 batched GridWorld engine (libbgw.so).
 *
 * The reference (gillette7/Abmarl 0.2.7, pure Python) has no FFI: its boundary for the hot path is the
 * Python object protocol
 *     SimulationManager.reset() / .step(action_dict)          abmarl/managers/simulation_manager.py:27-53
 *     AllStepManager.reset / .step                            abmarl/managers/all_step_manager.py:37-95
 *     TurnBasedManager.reset / .step                          abmarl/managers/turn_based_manager.py:22-94
 *     AgentBasedSimulation.{reset,step,get_obs,get_reward,get_done,get_all_done}
 *                                                             abmarl/sim/agent_based_simulation.py:238-294
 * over ONE simulation.  This library is what a maintainer would bind (ctypes / cffi; see INTEGRATION.md)
 * to advance E independent copies of one compiled simulation in lockstep on one B200.
 *
 * Conventions
 *   - plain C: pointers + sizes, no torch types.  Every call returns 0 on success, non-zero on error;
 *     bgw_last_error() returns a thread-local message.
 *   - ALL large buffers are CALLER-OWNED DEVICE memory (e.g. torch CUDA tensors -> data_ptr()).
 *     The library owns only the opaque handle and a few KB of constant tables.
 *   - kernels are enqueued on the cudaStream_t passed as `stream` (void*, 0 = legacy default stream); no
 *     internal threads, no host synchronisation inside bgw_reset / bgw_step.
 *   - there is NO CPU fallback: without a CUDA device bgw_create fails.
 *
 * Index spaces
 *   agent index a in [0, A)   : position in the reference's `sim.agents` dict (insertion order);
 *   learner index l in [0, L) : rank of a among entities that are `abmarl.sim.Agent` instances
 *                               (observing AND acting, agent_based_simulation.py:174-186);
 *   cell index                : r * cols + c   (np.ravel_multi_index, state.py:135).
 */
#ifndef BGW_H_
#define BGW_H_

#include "bgw_stdint.h"

#ifdef __cplusplus
extern "C" {
#endif

#define BGW_ABI_VERSION 5
#define BGW_MAX_ENCODING 63   /* encodings are bit positions in 64-bit overlap / attack rows */
#define BGW_MAX_AGENTS 4096   /* Philox slot field (bgw_philox.h)                           */
#define BGW_MAX_CELLS 65535   /* cell index is u16, 0xFFFF = none                           */
#define BGW_NONE 0xFFFFu
#define BGW_MAX_VICTIMS 256   /* attacked agents one attacker can name in one step (simultaneous_attacks x groups) */
#define BGW_MAX_SIMATT 16     /* AttackingAgent.simultaneous_attacks                                             */

/* ---- per-agent class flags (which reference mixins the entity derives from) ------------------- */
enum {
    BGW_AG_OBSERVING = 1 << 0,  /* GridObservingAgent   agent.py:115-132 */
    BGW_AG_MOVING = 1 << 1,     /* MovingAgent          agent.py:135-157 */
    BGW_AG_ATTACKING = 1 << 2,  /* AttackingAgent       agent.py:199-288 */
    BGW_AG_HEALTH = 1 << 3,     /* HealthAgent          agent.py:160-196 */
    BGW_AG_ORIENT = 1 << 4,     /* OrientationAgent     agent.py:342-373 */
    BGW_AG_LEARNER = 1 << 5,    /* isinstance(x, Agent) agent_based_simulation.py:174-186 */
    BGW_AG_BLOCKING = 1 << 6,   /* GridWorldAgent.blocking  agent.py:60-68 */
    BGW_AG_AMMO = 1 << 7        /* AmmoAgent            agent.py:291-321 */
};

/* ---- per-agent role inside a sim program ----------------------------------------------------- */
enum {
    BGW_ROLE_NONE = 0,
    BGW_ROLE_NAVIGATOR = 1, /* MazeNavigationSim.navigator / MultiMazeNavigationAgent */
    BGW_ROLE_TARGET = 2,    /* maze target                                           */
    BGW_ROLE_PACMAN = 3,    /* pacman.py:11                                          */
    BGW_ROLE_FOOD = 4,      /* pacman.py:19                                          */
    BGW_ROLE_BADDIE = 5,    /* pacman.py:24                                          */
    BGW_ROLE_WALL = 6,
    BGW_ROLE_RUNNER = 7,    /* reach_the_target.py:80-87 RunningAgent                */
    BGW_ROLE_SCRIPTED_BADDIE = 16 /* + k: the baddie of the k-th entry of PacmanSimSimple's script (pacman.py:235-246),
                                     k = 0..9 for baddie_20, 36, 156, 157, 159, 161, 162, 206, 222, 328 */
};

/* ---- sim program: the user-written step()/get_* the engine reproduces ------------------------ */
enum {
    BGW_PROG_TEAM_BATTLE = 0, /* abmarl/examples/sim/team_battle_example.py:23-59 */
    BGW_PROG_MAZE = 1,        /* abmarl/examples/sim/maze_navigation.py:14-42     */
    BGW_PROG_MULTI_MAZE = 2,  /* abmarl/examples/sim/multi_maze_navigation.py:17-74 */
    BGW_PROG_PACMAN = 3,      /* abmarl/examples/sim/pacman.py:29-151             */
    BGW_PROG_REACH_TARGET = 4,/* abmarl/examples/sim/reach_the_target.py:90-176   */
    BGW_PROG_TRAFFIC = 5,     /* abmarl/examples/sim/traffic_corridor.py:24-53    */
    BGW_PROG_PACMAN_SIMPLE = 6, /* abmarl/examples/sim/pacman.py:172-326 (scripted baddies, examples/rllib_pacman.py) */
    BGW_PROG_USER = 7          /* a user-written step program (include/bgw_program.h), installed with bgw_set_program */
};

enum { BGW_MOVE_NONE = 0, BGW_MOVE_BOX = 1 /* MoveActor actor.py:55 */, BGW_MOVE_CROSS = 2 /* :117 */,
       BGW_MOVE_DRIFT = 3 /* :197 */ };
enum { BGW_ATTACK_NONE = 0, BGW_ATTACK_BINARY = 1 /* BinaryAttackActor actor.py:441 */,
       BGW_ATTACK_ENCODING = 2 /* EncodingBasedAttackActor actor.py:504 */,
       BGW_ATTACK_RESTRICTED = 3 /* RestrictedSelectiveAttackActor actor.py:585 */,
       BGW_ATTACK_SELECTIVE = 4 /* SelectiveAttackActor actor.py:661 */ };
enum {
    BGW_OBS_POSITION_CENTERED = 0, /* PositionCenteredEncodingObserver (SingleGridObserver) observer.py:153 */
    BGW_OBS_ABSOLUTE = 1,          /* AbsoluteEncodingObserver                              observer.py:55  */
    BGW_OBS_STACKED = 2            /* StackedPositionCenteredEncodingObserver (MultiGridObserver) :253     */
};
enum {
    BGW_DONE_ACTIVE = 1 << 0,           /* ActiveDone            done.py:39-56   */
    BGW_DONE_ONE_TEAM = 1 << 1,         /* OneTeamRemainingDone  done.py:140-153 */
    BGW_DONE_TARGET_AGENT = 1 << 2,     /* TargetAgentDone       done.py:59-99   */
    BGW_DONE_TARGET_DESTROYED = 1 << 3  /* TargetDestroyedDone   done.py:102-137 */
};
enum { BGW_LAYOUT_POSITION_STATE = 0 /* PositionState state.py:18-166 */, BGW_LAYOUT_MAZE = 1 /* MazePlacementState :385-619 */,
       BGW_LAYOUT_TARGET_BARRIERS_FREE = 2 /* TargetBarriersFreePlacementState :169-383 */ };
enum { BGW_MANAGER_ALL_STEP = 0 /* all_step_manager.py */, BGW_MANAGER_TURN_BASED = 1 /* turn_based_manager.py */,
       /* managers/dynamic_order_manager.py:7-87 over a DynamicOrderSimulation (sim/agent_based_simulation.py:297-317) whose
        * next_agent rule is: the agent that just acted if that step finished it (it expects its last observation), then
        * the next agent in dict order that is not done -- abmarl_b200.examples.DynamicOrderMultiMazeSim.  BgwState.turn
        * holds the learner whose action the next step consumes. */
       BGW_MANAGER_DYNAMIC_ORDER = 2 };

/* reward constant slots (float64; values live in the user's sim, e.g. team_battle_example.py:42-59) */
enum {
    BGW_RW_ATTACK_FAIL = 0, /* -0.1  team_battle_example.py:42 */
    BGW_RW_KILL = 1,        /* +1    :47 / pacman 'kill'       */
    BGW_RW_DIE = 2,         /* -1    :46 / pacman 'die'        */
    BGW_RW_MOVE_FAIL = 3,   /* -0.1  :55 / pacman 'bad_move'   */
    BGW_RW_ENTROPY = 4,     /* -0.01 :59 / pacman 'entropy'    */
    BGW_RW_TARGET = 5,      /* +1    maze_navigation.py:33 / multi_maze_navigation.py:57 / reach_the_target.py:142 / traffic_corridor.py:53 */
    BGW_RW_EAT_FOOD = 6,    /* pacman 'eat_food' pacman.py:97  */
    BGW_RW_COUNT = 8
};

/* ---- flags stored per agent in BgwState.flags -------------------------------------------------- */
enum {
    BGW_ST_ACTIVE = 1 << 0,        /* PrincipleAgent.active / HealthAgent: health > 0   agent.py:192-196 */
    BGW_ST_IN_GRID = 1 << 1,       /* entity is present in its cell's dict              grid.py:107-140  */
    BGW_ST_DONE_REPORTED = 1 << 2, /* member of SimulationManager.done_agents           all_step_manager.py:85-87 */
    BGW_ST_ORIENT_SHIFT = 4        /* bits 4..6: orientation 1..4 (0 = none)            agent.py:344     */
};

/* per-learner output byte `done` */
enum { BGW_OUT_DONE = 1 << 0, BGW_OUT_VALID = 1 << 1 /* this learner got (obs,reward,done) this call */ };
/* per-env output byte `all_done` */
enum {
    BGW_ENV_ALL_DONE = 1 << 0,  /* dones['__all__']                                     all_step_manager.py:90-93 */
    BGW_ENV_RESET = 1 << 1,     /* this call reset the env instead of stepping it (auto-reset): obs rows hold
                                   the reset observations of every learner, reward/done rows are zero   */
    BGW_ENV_TRUNCATED = 1 << 2, /* horizon reached (RLlib `horizon`, rllib_team_battle.py:89)           */
    BGW_ENV_ERROR = 1 << 3      /* placement failed (state.py:147-149,161; the reference raises) -- see BgwState.error.
                                   Reported together with BGW_ENV_ALL_DONE and zero observations: the env is inert
                                   until it is reset again (auto-reset: by the next step, with the next episode's draws) */
};

/*
 * Flat description of ONE simulation, compiled from a reference-style sim object (agents dict,
 * grid.overlapping, actor.attack_mapping, chosen state / observer / done components, reward constants).
 * All pointers are HOST pointers, read during bgw_create only.
 */
typedef struct BgwSpec {
    int32_t abi_version;   /* BGW_ABI_VERSION */
    int32_t rows, cols;    /* Grid(rows, cols)  grid.py:20 */
    int32_t n_agents;      /* A */
    int32_t n_envs;        /* E: envs on THIS device */
    int32_t env_offset;    /* global index of env 0 on this device (Philox is keyed by the GLOBAL env
                              index, so results do not depend on how envs are sharded over GPUs) */
    int32_t program;       /* BGW_PROG_* */
    int32_t move_actor;    /* BGW_MOVE_* */
    int32_t attack_actor;  /* BGW_ATTACK_* */
    int32_t observer;      /* BGW_OBS_* */
    int32_t observe_self;  /* PositionCenteredEncodingObserver(observe_self=...) observer.py:164 */
    int32_t done_mask;     /* BGW_DONE_* (Smart sims: all() over the set, smart.py:106-120) */
    int32_t manager;       /* BGW_MANAGER_* */
    int32_t ravel_actions; /* 1: RavelActionWrapper(MoveActor) wrapper.py:180 -- action byte 0 is the
                              ravelled move  a = (dr+m)(2m+1) + (dc+m) */
    int32_t no_overlap_at_reset; /* PositionState(no_overlap_at_reset=) state.py:29 */
    int32_t stacked_attacks;     /* AttackActorBaseComponent(stacked_attacks=) actor.py:245 */
    int32_t horizon;       /* 0 = none; else all_done|TRUNCATED once the episode has this many steps */
    int32_t auto_reset;    /* 1: an env that reported __all__ is reset by the NEXT bgw_step call */
    int32_t ammo_observer; /* 1: the sim has an AmmoObserver (observer.py:376-413): learners with BGW_AG_AMMO
                              also observe their ammo (BgwDims.ammo_offset) */
    int32_t layout_kind;   /* BGW_LAYOUT_*: which placement state builds the start layout of an episode */
    int32_t layout_target; /* target_agent of the placement state (agent index) state.py:200-222, 417-439 */
    int32_t cluster_barriers, scatter_free_agents;   /* state.py:462-485 */
    int32_t randomize_placement_order;  /* PositionState(randomize_placement_order=) state.py:97-101: the entities are
                                           placed in the keyed order BGW_SITE_PLACE_ORDER of the episode (bgw_philox.h) */
    int32_t randomize_action_input;     /* AllStepManager(randomize_action_input=) all_step_manager.py:62-65: without a
                                           caller-given `order`, bgw_step processes the actions in the keyed order
                                           BGW_SITE_ORDER of the step */
    int32_t position_observer;          /* 1: the sim has an AbsolutePositionObserver (observer.py:337-373): learners also
                                           observe their own (row, col) (BgwDims.position_offset) */
    uint64_t seed;         /* Philox key */
    uint64_t barrier_encodings, free_encodings;       /* bit e set <=> encoding e in the set, state.py:430-460 */
    double reward[BGW_RW_COUNT];

    /* per-agent tables, length n_agents */
    const int8_t *encoding;       /* GridWorldAgent.encoding (1..BGW_MAX_ENCODING)  agent.py:31-37 */
    const uint8_t *klass;         /* BGW_AG_* */
    const uint8_t *role;          /* BGW_ROLE_* */
    const int16_t *init_row;      /* initial_position[0], -1 = random placement  state.py:107-114 */
    const int16_t *init_col;
    const double *init_health;    /* NaN = np.random.uniform(0,1)                state.py:637-641 */
    const uint8_t *init_orient;   /* 0 = np.random.randint(1,5)                  state.py:672-675 */
    const int16_t *view_range;    /* GridObservingAgent.view_range               agent.py:122 */
    const int16_t *move_range;    /* MovingAgent.move_range                      agent.py:147 */
    const int16_t *attack_range;  /* AttackingAgent.attack_range                 agent.py:213 */
    const double *attack_strength;
    const double *attack_accuracy;
    const uint8_t *simultaneous_attacks;
    const int16_t *target;        /* TargetAgentDone / TargetDestroyedDone mapping: agent -> target agent, -1 none */
    const int32_t *initial_ammo;  /* AmmoAgent.initial_ammo (agent.py:311-321) of entities with BGW_AG_AMMO; may be
                                     NULL when no entity has the flag */

    /* per-encoding bit rows, length BGW_MAX_ENCODING+1; row e bit f set <=> f in map[e] */
    const uint64_t *overlap;      /* Grid.overlapping, already symmetrised        grid.py:53-71 */
    const uint64_t *attack_map;   /* AttackActorBaseComponent.attack_mapping      actor.py:272-288 */
} BgwSpec;

/*
 * Mutable simulation state: structure-of-arrays in HBM, caller-owned (device pointers).
 * [E][A] arrays are env-major so one CTA loads one env with coalesced accesses.
 */
typedef struct BgwState {
    uint16_t *cell;      /* [E][A] r*cols+c; stays stale after death (actor.py:356-358)                */
    uint16_t *next;      /* [E][A] next entity in the same cell's dict (arrival order, grid.py:125);
                            BGW_NONE = tail.  Meaningful only while BGW_ST_IN_GRID.                     */
    uint8_t *flags;      /* [E][A] BGW_ST_*                                                              */
    double *health;      /* [E][A] float64 like the reference (agent.py:192-196)                        */
    double *reward_acc;  /* [E][A] SmartGridWorldSimulation.rewards between reads (smart.py:91,101-104) */
    uint32_t *episode;   /* [E]  number of resets - 1 (Philox key); initialise to 0xFFFFFFFF             */
    uint32_t *step;      /* [E]  steps since the last reset (Philox key)                                */
    uint8_t *env_flags;  /* [E]  BGW_ENV_* of the last call                                             */
    int16_t *turn;       /* [E]  TurnBasedManager cursor: learner whose action is expected next         */
    uint32_t *error;     /* [E]  0 ok; 1 fixed-position placement failed; 2 no cell available            */
    uint16_t *layout;    /* [E][A] optional (NULL = unused): externally generated start cells that replace
                            PositionState's placement at reset (BGW_NONE = leave the entity unplaced); used
                            for MazePlacementState layouts generated host-side (state.py:385-619)          */
    uint64_t *stats;     /* [E][BGW_STAT_COUNT] per-env running counters, see below (sum over E on demand;
                            per-env rows avoid same-address atomics in the step kernel)                 */
    int32_t *ammo;       /* [E][A] AmmoAgent.ammo (agent.py:299-309; AmmoState.reset state.py:644-656);
                            required only when some entity has BGW_AG_AMMO, else may be NULL             */
} BgwState;

enum {
    BGW_STAT_AGENT_STEPS = 0, /* learners that received (obs,reward,done) */
    BGW_STAT_EPISODES = 1,    /* envs that reported __all__               */
    BGW_STAT_KILLS = 2,       /* entities whose health reached 0 by attack */
    BGW_STAT_ENV_STEPS = 3,
    BGW_STAT_COUNT = 4
};

/* Derived sizes the caller needs to allocate buffers. */
typedef struct BgwDims {
    int32_t n_envs, n_agents, n_learners;
    int32_t obs_h, obs_w, obs_c; /* logical observation shape per learner (obs_c = 1 unless STACKED) */
    int32_t obs_stride;          /* bytes per learner in the int8 obs buffer = roundup(h*w*c (+4), 16) */
    int32_t action_stride;       /* bytes per learner in the action buffer, a multiple of 4 (see bgw_step) */
    int32_t threads_per_env, envs_per_cta, smem_bytes; /* launch geometry (informational)             */
    int32_t ammo_offset;         /* AmmoObserver (observer.py:376-413): byte offset inside a learner's obs row of
                                    its int32 'ammo' observation (little endian, 4-byte aligned), or -1       */
    int32_t device_layouts;      /* 1: bgw_generate_layouts can build this spec's start layouts on the device    */
    int32_t position_offset;     /* AbsolutePositionObserver (observer.py:337-373): byte offset inside a learner's obs row of
                                    its 'position' observation, int16 row then int16 col (4-byte aligned), or -1; the
                                    position stays where the agent died (actor.py:356-358)                       */
} BgwDims;

typedef struct BgwEngine *bgw_handle;

#ifndef __CUDACC_RTC__   /* (the device code includes this header for the structs and constants when it is compiled at run time) */
/* Compile the spec onto `device`; builds the line-of-sight LUT (utils.py:45-115 in IEEE float64). */
int bgw_create(const BgwSpec *spec, int device, bgw_handle *out);
int bgw_destroy(bgw_handle h);
int bgw_dims(bgw_handle h, BgwDims *out);
/* Attach the caller-owned state arrays (must stay alive while the handle is used). */
int bgw_bind_state(bgw_handle h, const BgwState *state);

/*
 * AllStepManager.reset / TurnBasedManager.reset for the envs selected by env_mask ([E] u8 on device,
 * NULL = all): PositionState.reset, HealthState.reset, OrientationState.reset (state.py:88-166,629-641,
 * 666-675), rewards = 0 (smart.py:91), done_agents = non-learners (all_step_manager.py:41-44), then the
 * first observations into obs[E][L][obs_stride] (rows of unselected envs are untouched).
 */
int bgw_reset(bgw_handle h, const uint8_t *env_mask, int8_t *obs, void *stream);

/*
 * sim.get_obs(agent_id) for EVERY learner of the envs selected by env_mask (NULL = all), on the state as it stands:
 * SmartGridWorldSimulation.get_obs (sim/gridworld/smart.py:93-99) = the sim's observers (observer.py:95-150 absolute,
 * :195-248 position centred, :287-335 stacked, :366-373 position, :406-413 ammo) -> obs[E][L][obs_stride] (rows of
 * unselected envs are untouched).  Nothing is stepped and no state is written; learners that are inactive or already
 * reported done get the row the reference computes from their last position.  The random choice among the encodings
 * sharing a cell (observer.py:131-134,233-236) is keyed by the env's current (episode, step): the rows equal the ones
 * the last bgw_reset / bgw_step wrote for the learners it reported.  What a manager calls between steps
 * (all_step_manager.py:47,69), and the bandwidth-bound piece of the path on its own (128 bytes written per 3 read).
 */
int bgw_observe(bgw_handle h, const uint8_t *env_mask, int8_t *obs, void *stream);

/*
 * One manager step for every env (all_step_manager.py:51-95 / turn_based_manager.py:34-94):
 *   actions  [E][L][action_stride] i8
 *                           byte0,1 = move (dr,dc | cross 0..4 | ravelled); from byte 2 the attack action:
 *                             BinaryAttackActor               byte2 = number of attacks (actor.py:451-453)
 *                             EncodingBasedAttackActor        byte 2+(e-1) = attacks on encoding e (:513-519)
 *                             RestrictedSelectiveAttackActor  byte 2+j = ravelled cell + 1 of attack j, 0 = unused
 *                                                             (:593-599; j < simultaneous_attacks)
 *                             SelectiveAttackActor            byte 2+(r*n+c) = attacks on window cell (r,c),
 *                                                             n = 2*attack_range+1 of that agent (:669-679)
 *                           action_stride = roundup(2 + widest attack action, 4): 4 for the Binary actor;
 *                           rows of learners already reported done are ignored (the reference asserts
 *                           they are absent, all_step_manager.py:59-61)
 *   order    [E][L] i16     optional processing order of learners (randomize_action_input,
 *                           all_step_manager.py:62-65); NULL = dict order
 *   obs      [E][L][obs_stride] i8, reward [E][L] f32, done [E][L] u8 (BGW_OUT_*), all_done [E] u8 (BGW_ENV_*)
 * Rows whose BGW_OUT_VALID bit is clear (and BGW_ENV_RESET is clear) are not written.
 * The launch may be captured into a CUDA graph and replayed (the library detects the capture with cudaStreamIsCapturing).
 */
int bgw_step(bgw_handle h, const int8_t *actions, const int16_t *order, int8_t *obs, float *reward,
             uint8_t *done, uint8_t *all_done, void *stream);

/* bgw_sample_actions + bgw_step in one call: every acting learner draws its action from the keyed random policy
 * and the batch is stepped with them.  actions_out[E][L][action_stride] receives the sampled actions of the learners that acted
 * (rows of learners already reported done are not written).  Same results as the two calls made separately. */
int bgw_step_sampled(bgw_handle h, int8_t *actions_out, const int16_t *order, int8_t *obs, float *reward,
                     uint8_t *done, uint8_t *all_done, void *stream);

/* n_steps consecutive bgw_step_sampled calls on the same buffers (a random-policy rollout that stays on the device, as
 * the reference's RandomPolicy episodes do, policies/policy.py:81-92 + trainers/base.py:123-142): afterwards the
 * outputs hold the last step's rows and BgwState / the statistics are those after n_steps steps -- bit for bit what
 * n_steps separate calls leave behind.  Sims with a device-side layout generator get their next-episode layouts after
 * every step, as after bgw_step.  Because the library enqueues the launches itself, with nothing between them, launch
 * k+1 starts each env as soon as launch k has finished THAT env instead of waiting for the whole batch (one launch
 * per step either way; abmarl_b200/csrc/bgw_fast.cuh, "env tickets and chained launches"). */
int bgw_rollout_sampled(bgw_handle h, int n_steps, int8_t *actions_out, const int16_t *order, int8_t *obs, float *reward,
                        uint8_t *done, uint8_t *all_done, void *stream);

/*
 * Compact the outputs of the last bgw_step for a host consumer.  The reference's managers return dicts that hold
 * only the agents that received something (all_step_manager.py:68-83, turn_based_manager.py:49-92); the dense
 * [E][L] outputs of bgw_step keep a row for every learner.  bgw_gather_valid copies the rows whose BGW_OUT_VALID
 * bit is set -- and every row of an env that was reset by this call (BGW_ENV_RESET: first observations) -- into
 * contiguous buffers, so that only those bytes have to cross PCIe:
 *   count    [1] i32 device      number of compacted rows n
 *   index    [E*L] i32           index[i] = e * L + l of compacted row i (grouped by env, env order unspecified)
 *   obs_c    [E*L][obs_stride] i8, reward_c [E*L] f32, done_c [E*L] u8    rows 0..n-1 are written
 */
int bgw_gather_valid(bgw_handle h, const int8_t *obs, const float *reward, const uint8_t *done, const uint8_t *all_done,
                     int32_t *count, int32_t *index, int8_t *obs_c, float *reward_c, uint8_t *done_c, void *stream);

/*
 * MazePlacementState.reset (state.py:487-619, generate_maze utils.py:120-212) / TargetBarriersFreePlacementState.reset
 * (state.py:281-383) on the device: writes the start layout
 * of the NEXT episode (episode[e] + 1) of the selected envs into BgwState.layout ([E][A], must be bound), where the
 * next bgw_reset / auto-reset consumes it.  only_done != 0: the envs whose last step reported BGW_ENV_ALL_DONE;
 * otherwise the envs selected by env_mask ([E] u8 on the device, NULL = all).  Placement failures set BgwState.error.
 * Fails when BgwDims.device_layouts is 0 (grid above 18x18 or more than 8 placed encodings: generate the layouts
 * host-side then, abmarl_b200/layouts.py).
 */
int bgw_generate_layouts(bgw_handle h, const uint8_t *env_mask, int only_done, void *stream);

/* on == 0: the caller supplies BgwState.layout itself (host-generated layouts, state.py:487-527 run elsewhere): the library
 * never regenerates it, in particular bgw_rollout_sampled does not write the finished envs' next layouts between its steps.
 * on != 0 (the default when BgwDims.device_layouts is 1): bgw_rollout_sampled does, as a caller of bgw_step would through
 * bgw_generate_layouts(only_done = 1). */
int bgw_use_device_layouts(bgw_handle h, int on);

/* The same generator on the host for one (global env, episode): layout[A].  Test / replay hook, like bgw_rng_draw. */
int bgw_maze_layout_host(const BgwSpec *spec, uint32_t global_env, uint32_t episode, uint16_t *layout);

/* Synthetic random policy (policies/policy.py:81-92 `action_space.sample()`), keyed Philox site ACTION:
 * fills actions[E][L][action_stride] for the CURRENT step of every env.  Used by bench.py and the parity tests. */
int bgw_sample_actions(bgw_handle h, int8_t *actions, void *stream);

/* Host-callable Philox draw, identical to the device stream (used by the replay shim). */
int bgw_rng_draw(uint64_t seed, uint32_t env, uint32_t episode, uint32_t step, uint32_t site,
                 uint32_t slot, uint32_t k, uint32_t out[4]);

/* Line-of-sight mask of utils.py:45-115 for one blocker offset: writes (2*range+1)^2 bytes (1 = visible). */
int bgw_los_mask(int range, int r_diff, int c_diff, uint8_t *out);

/* Number of kernels this handle has launched since creation (bench.py `gpu_launches`). */
uint64_t bgw_launch_count(bgw_handle h);

/*
 * Compile the general step kernel for THIS handle's spec at run time (NVRTC, sm_100a) and use it for every later step:
 * the spec's scalars (grid and entity counts, program, actors, observer, manager, flags) become compile-time constants,
 * so the kernel holds only the code this sim runs (a third to a half of the instructions of the per-program build; the
 * general kernel spends most of its stall cycles waiting for instructions).  Sims that run the specialised team-battle
 * kernel are left alone (returns 0).  Needs libnvrtc.so.12 and the library's own sources (abmarl_b200/csrc, include/)
 * next to libbgw.so; takes 5-15 s per spec, cached in `cache_dir` (NULL: $BGW_JIT_CACHE, else no cache) by spec hash.
 * Results are bit-identical to the stock kernel's: it is the same source.
 */
int bgw_specialize(bgw_handle h, const char *cache_dir);

/*
 * Install the step program of a BGW_PROG_USER handle: `source` is the program's C text (include/bgw_program.h), compiled at
 * run time (NVRTC, sm_100a) into the general step kernel, which then runs it for every step.  Needs what bgw_specialize
 * needs; the cubin is cached in `cache_dir` (NULL: $BGW_JIT_CACHE, else no cache) by the hash of the spec, the program and
 * the kernel sources.  On a compile error the NVRTC diagnostic is in bgw_last_error().  Fails on a handle of any other
 * program and when the handle has a program already.  Until a program is set, bgw_reset, bgw_observe, bgw_sample_actions
 * and bgw_gather_valid work (they do not depend on the program) and bgw_step / bgw_step_sampled / bgw_rollout_sampled fail
 * without touching any buffer.  A program handle never runs the specialised team-battle kernel, and bgw_specialize on it
 * does nothing (the program's kernel is compiled for the spec already).  BGW_MANAGER_DYNAMIC_ORDER is not available to
 * programs (its next_agent rule is not programmable).
 */
int bgw_set_program(bgw_handle h, const char *source, const char *cache_dir);

const char *bgw_last_error(void);
int bgw_abi_version(void);
#endif /* __CUDACC_RTC__ */

#ifdef __cplusplus
}
#endif
#endif /* BGW_H_ */
