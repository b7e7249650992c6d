"""ForagingSim: a simulation of the user's own, run on the device through a step program (abmarl_b200.program).

None of the built-in programs can express it, which makes it the template to copy for a new simulation:

  - foragers (observe, move, have health; learners) walk the grid and harvest the resources in their cell;
  - predators (observe, move, attack foragers with the BinaryAttackActor; learners) hunt the foragers;
  - resources (HealthAgents, not learners) lose `bite` health per harvest, leave the grid when depleted and come back
    with probability `respawn_probability` per step, at a random cell that Grid.query allows, with full health.

step() in the reference's terms (what FORAGING_PROGRAM below does on the device, in this order):
  1. each acting predator that is active attacks; no victim: `attack_fail`; each victim killed: `die` to it, `kill` to
     the predator (team_battle_example.py:37-47);
  2. each acting agent that is active moves; a failed move: `move_fail`;
  3. each acting forager that is active harvests every resource of its cell in dict order: the resource loses `bite`
     health, the forager gets `harvest`, a resource at 0 is removed from the grid;
  4. each depleted resource (dict order) respawns with probability `respawn_probability`.
get_done is ActiveDone's (a forager is done when it has been killed); get_all_done: no forager or no resource is active.
"""
from abmarl_b200.program import DeviceProgram
from abmarl_b200.sim.gridworld.actor import BinaryAttackActor, MoveActor
from abmarl_b200.sim.gridworld.agent import AttackingAgent, GridObservingAgent, HealthAgent, MovingAgent
from abmarl_b200.sim.gridworld.smart import SmartGridWorldSimulation

FORAGER, PREDATOR, RESOURCE = 1, 2, 3      # role bytes (bgwp_role) and encodings

FORAGING_PROGRAM = r'''
/* ForagingSim.step (abmarl_b200/examples/foraging.py).  Constants: KILL, DIE, ATTACK_FAIL, MOVE_FAIL, HARVEST, BITE,
 * RESPAWN_P.  Roles: 1 forager, 2 predator, 3 resource. */
#define FORAGER 1
#define PREDATOR 2
#define RESOURCE 3

BGWP_FN void bgwp_step(bgwp_ctx *c)
{
    int victims[BGW_MAX_VICTIMS];
    const int n = bgwp_n_acting(c);
    for (int i = 0; i < n; ++i) {                              /* 1. predators attack, in action order */
        const int a = bgwp_acting(c, i);
        if (a < 0 || bgwp_role(c, a) != PREDATOR || !bgwp_active(c, a)) continue;
        const int nv = bgwp_attack(c, a, victims);
        if (nv == 0) bgwp_add_reward(c, a, ATTACK_FAIL);
        for (int t = 0; t < nv; ++t)
            if (!bgwp_active(c, victims[t])) {
                bgwp_add_reward(c, victims[t], DIE);
                bgwp_add_reward(c, a, KILL);
            }
    }
    for (int i = 0; i < n; ++i) {                              /* 2. every mover moves */
        const int a = bgwp_acting(c, i);
        if (a < 0 || !bgwp_active(c, a)) continue;
        if (!bgwp_move(c, a)) bgwp_add_reward(c, a, MOVE_FAIL);
    }
    for (int i = 0; i < n; ++i) {                              /* 3. foragers harvest their cell, in dict order */
        const int a = bgwp_acting(c, i);
        if (a < 0 || bgwp_role(c, a) != FORAGER || !bgwp_active(c, a)) continue;
        int o = bgwp_first_occupant(c, bgwp_row(c, a), bgwp_col(c, a));
        while (o >= 0) {
            const int next = bgwp_next_occupant(c, o);         /* before o may leave the cell */
            if (bgwp_role(c, o) == RESOURCE && bgwp_active(c, o)) {
                bgwp_set_health(c, o, bgwp_health(c, o) - BITE);
                bgwp_add_reward(c, a, HARVEST);
                if (!bgwp_active(c, o)) bgwp_remove(c, o);
            }
            o = next;
        }
    }
    const int cells = bgwp_rows(c) * bgwp_cols(c);
    for (int r = 0; r < bgwp_n_agents(c); ++r) {               /* 4. depleted resources respawn */
        if (bgwp_role(c, r) != RESOURCE || bgwp_active(c, r) || bgwp_uniform(c, r, 0) >= RESPAWN_P) continue;
        const int cell = (int)(bgwp_uniform(c, r, 1) * cells);
        const int row = cell / bgwp_cols(c), col = cell % bgwp_cols(c);
        if (!bgwp_query(c, r, row, col)) continue;
        bgwp_set_health(c, r, 1.0);
        bgwp_place(c, r, row, col);
    }
}

#define BGWP_HAS_GET_ALL_DONE
BGWP_FN int bgwp_get_all_done(const bgwp_ctx *c)              /* no forager or no resource is active */
{
    int foragers = 0, resources = 0;
    for (int a = 0; a < bgwp_n_agents(c); ++a) {
        if (!bgwp_active(c, a)) continue;
        foragers += bgwp_role(c, a) == FORAGER;
        resources += bgwp_role(c, a) == RESOURCE;
    }
    return foragers == 0 || resources == 0;
}
'''


class Forager(GridObservingAgent, MovingAgent, HealthAgent):
    def __init__(self, view_range=2, **kwargs):
        kwargs.setdefault('initial_health', 1)
        super().__init__(encoding=FORAGER, move_range=1, view_range=view_range, **kwargs)


class Predator(GridObservingAgent, MovingAgent, AttackingAgent):
    def __init__(self, view_range=2, **kwargs):
        super().__init__(encoding=PREDATOR, move_range=1, view_range=view_range, attack_range=1, attack_strength=1,
                         attack_accuracy=1, **kwargs)


class Resource(HealthAgent):
    def __init__(self, **kwargs):
        kwargs.setdefault('initial_health', 1)
        super().__init__(encoding=RESOURCE, **kwargs)


class ForagingSim(SmartGridWorldSimulation):
    """Build with ForagingSim.build_sim(rows, cols, agents=...) (or build_sim_from_file, ...) or ForagingSim.build(...).
    The components default to PositionState + HealthState, a PositionCenteredEncodingObserver, ActiveDone, MoveActor and a
    BinaryAttackActor {predator: {forager}}; foragers share cells with resources and predators, two resources never do."""
    reward_constants = dict(kill=1.0, die=-1.0, attack_fail=-0.1, move_fail=-0.1, harvest=0.5)
    components = dict(overlapping={FORAGER: {PREDATOR, RESOURCE}, PREDATOR: {FORAGER, RESOURCE}, RESOURCE: {FORAGER, PREDATOR}},
                      attack_mapping={PREDATOR: {FORAGER}}, states={'PositionState', 'HealthState'},
                      observers={'PositionCenteredEncodingObserver'}, dones={'ActiveDone'})

    def __init__(self, bite=0.25, respawn_probability=0.05, reward_constants=None, **kwargs):
        super().__init__(**kwargs)
        self.move_actor = MoveActor(**kwargs)
        self.attack_actor = BinaryAttackActor(**kwargs)
        self.bite, self.respawn_probability = float(bite), float(respawn_probability)
        self.reward_constants = dict(self.reward_constants, **(reward_constants or {}))
        self.finalize()

    @classmethod
    def _build_sim(cls, rows, cols, **kwargs):
        for name, value in cls.components.items():
            kwargs.setdefault(name, value)
        return super()._build_sim(rows, cols, **kwargs)

    @classmethod
    def build(cls, rows=12, cols=12, n_foragers=6, n_predators=2, n_resources=10, view_range=2, **kwargs):
        """A random-start instance: every agent is placed at random each episode."""
        agents = {f'forager{i}': Forager(id=f'forager{i}', view_range=view_range) for i in range(n_foragers)}
        agents.update({f'predator{i}': Predator(id=f'predator{i}', view_range=view_range) for i in range(n_predators)})
        agents.update({f'resource{i}': Resource(id=f'resource{i}') for i in range(n_resources)})
        return cls.build_sim(rows, cols, agents=agents, **kwargs)

    def program(self):
        return 'user'                                   # BGW_PROG_USER: device_program() below

    def device_program(self):
        """The step program of this sim: FORAGING_PROGRAM with the sim's constants and the agents' roles."""
        rc = self.reward_constants
        return DeviceProgram(
            FORAGING_PROGRAM,
            constants=dict(KILL=float(rc['kill']), DIE=float(rc['die']), ATTACK_FAIL=float(rc['attack_fail']),
                           MOVE_FAIL=float(rc['move_fail']), HARVEST=float(rc['harvest']), BITE=self.bite,
                           RESPAWN_P=self.respawn_probability),
            roles={agent: role for agent in self.agents.values()
                   for cls, role in ((Forager, FORAGER), (Predator, PREDATOR), (Resource, RESOURCE)) if isinstance(agent, cls)})
