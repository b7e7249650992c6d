"""AlternatingBattleSim: teams of BattleAgents that take turns, run on the device under the DynamicOrderManager through a
step program with a next_agent hook (abmarl_b200.program, include/bgw_program.h).

No built-in rule expresses it: the built-in dynamic-order rule (DynamicOrderMultiMazeSim) hands the turn to one agent at
a time, here a whole team acts at once.

  - Each agent's team is its encoding 1..n_teams; a team attacks every other team (BinaryAttackActor) and no two agents
    share a cell.
  - step() runs the acting team's turn as TeamBattleSim does (team_battle_example.py:33-59): every active member attacks,
    then every active member moves, then every acting member pays the entropy penalty.
  - next_agent names every agent that is done (killed), so that a kill is reported to its victim even off its team's
    turn, and every active member of the next team in cyclic order that still has an active member: teams wiped out
    are skipped.
  - get_done is ActiveDone's; get_all_done: at most one team has an active member.

The DynamicOrderManager's reset names the first learner, so the first step of an episode is that agent's alone; from
then on whole teams alternate.
"""
from abmarl_b200.program import DeviceProgram
from abmarl_b200.sim.agent_based_simulation import DynamicOrderSimulation
from abmarl_b200.sim.gridworld.actor import BinaryAttackActor, MoveActor
from abmarl_b200.sim.gridworld.smart import SmartGridWorldSimulation

from .sims import BattleAgent

ALTERNATING_BATTLE_PROGRAM = r'''
/* AlternatingBattleSim (abmarl_b200/examples/alternating_battle.py).  Constants: N_TEAMS, ATTACK_FAIL, KILL, DIE,
 * MOVE_FAIL, ENTROPY.  Role = team, 1 .. N_TEAMS. */
BGWP_FN void bgwp_step(bgwp_ctx *c)
{
    int victims[BGW_MAX_VICTIMS];
    const int n = bgwp_n_acting(c);
    for (int i = 0; i < n; ++i) {                              /* the acting team attacks */
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
    for (int i = 0; i < n; ++i) {                              /* then moves */
        const int a = bgwp_acting(c, i);
        if (a < 0 || !bgwp_active(c, a)) continue;
        if (!bgwp_move(c, a)) bgwp_add_reward(c, a, MOVE_FAIL);
    }
    for (int i = 0; i < n; ++i) {
        const int a = bgwp_acting(c, i);
        if (a >= 0) bgwp_add_reward(c, a, ENTROPY);
    }
}

BGWP_FN int team_alive(const bgwp_ctx *c, int team)
{
    for (int a = 0; a < bgwp_n_agents(c); ++a)
        if (bgwp_role(c, a) == team && bgwp_active(c, a)) return 1;
    return 0;
}

#define BGWP_HAS_GET_ALL_DONE
BGWP_FN int bgwp_get_all_done(const bgwp_ctx *c)             /* one team remaining (or none) */
{
    int alive = 0;
    for (int t = 1; t <= N_TEAMS; ++t) alive += team_alive(c, t);
    return alive <= 1;
}

/* the team after the one that just acted, in cyclic order, that still has an active member (0: none) */
BGWP_FN int next_team(const bgwp_ctx *c)
{
    const int last = bgwp_n_acting(c) > 0 ? bgwp_role(c, bgwp_acting(c, 0)) : 0;
    for (int k = 1; k <= N_TEAMS; ++k) {
        const int t = (last + k - 1) % N_TEAMS + 1;
        if (team_alive(c, t)) return t;
    }
    return 0;
}

#define BGWP_HAS_NEXT_AGENT
BGWP_FN int bgwp_next_agent(const bgwp_ctx *c, int a)
{
    if (!bgwp_active(c, a)) return 1;                          /* done: its death is reported, whoever's turn it is */
    return bgwp_role(c, a) == next_team(c);
}
'''


class AlternatingBattleSim(SmartGridWorldSimulation, DynamicOrderSimulation):
    """Build with AlternatingBattleSim.build_sim(rows, cols, agents=...) (BattleAgents, team = encoding) or
    AlternatingBattleSim.build(...).  The components default to PositionState + HealthState, a
    PositionCenteredEncodingObserver, ActiveDone, MoveActor and a BinaryAttackActor in which every team attacks every
    other team.  Run it with abmarl_b200.managers.DynamicOrderManager."""
    reward_constants = dict(attack_fail=-0.1, kill=1.0, die=-1.0, move_fail=-0.1, entropy=-0.01)

    def __init__(self, reward_constants=None, **kwargs):
        super().__init__(**kwargs)
        self.move_actor = MoveActor(**kwargs)
        self.attack_actor = BinaryAttackActor(**kwargs)
        self.reward_constants = dict(self.reward_constants, **(reward_constants or {}))
        self.finalize()

    @classmethod
    def _build_sim(cls, rows, cols, **kwargs):
        teams = sorted({agent.encoding for agent in kwargs['agents'].values()})
        kwargs.setdefault('attack_mapping', {t: set(teams) - {t} for t in teams})
        kwargs.setdefault('states', {'PositionState', 'HealthState'})
        kwargs.setdefault('observers', {'PositionCenteredEncodingObserver'})
        kwargs.setdefault('dones', {'ActiveDone'})
        return super()._build_sim(rows, cols, **kwargs)

    @classmethod
    def build(cls, rows=10, cols=10, n_teams=2, team_size=4, **kwargs):
        """A random-start instance: team t (1 .. n_teams) has team_size members, agents in team order."""
        agents = {f'team{t}_{i}': BattleAgent(id=f'team{t}_{i}', encoding=t)
                  for t in range(1, n_teams + 1) for i in range(team_size)}
        return cls.build_sim(rows, cols, agents=agents, **kwargs)

    def program(self):
        return 'user'                                   # BGW_PROG_USER: device_program() below

    def device_program(self):
        """The step program of this sim: ALTERNATING_BATTLE_PROGRAM with the sim's constants; role = team."""
        rc = self.reward_constants
        return DeviceProgram(
            ALTERNATING_BATTLE_PROGRAM,
            constants=dict(N_TEAMS=max(agent.encoding for agent in self.agents.values()),
                           ATTACK_FAIL=float(rc['attack_fail']), KILL=float(rc['kill']), DIE=float(rc['die']),
                           MOVE_FAIL=float(rc['move_fail']), ENTROPY=float(rc['entropy'])),
            roles={agent: agent.encoding for agent in self.agents.values()})
