"""KingOfTheHillSim: teams of fighters contest a hill, run on the device through a step program that keeps variables of its
own (abmarl_b200.program, include/bgw_program.h): each team's score, the winner, and every fighter's attack cooldown.

No program could express it without them: the score grows over the episode, and an attack leaves its attacker unable to
attack again for a while.

  - Each fighter's team is its encoding 1..n_teams; a team attacks every other team (BinaryAttackActor) and no two fighters
    share a cell.  The hill is the rectangle rows hill[0]..hill[2], columns hill[1]..hill[3] (inclusive).
  - step(): every active acting fighter attacks, then every active acting fighter moves (MoveActor), then the hill is
    scored.
  - Attacks: an attack puts the attacker on cooldown for `cooldown` of its next steps (agent variable COOLDOWN: how many
    remain).  An attack asked for while on cooldown is ignored: no draw, no reward; the step still counts one down.  A
    kill gives the attacker `kill` and the victim `die`.
  - The hill: a team that alone has active fighters on it scores 1 (env variable SCORE[team]), and each of its fighters on
    the hill gets `hold`.  The first team whose score reaches `target_score` is the WINNER (env variable, 0 while there is
    none), and each of its active fighters gets `win`.
  - get_done is ActiveDone's; get_all_done: there is a winner, or fewer than two teams have an active fighter.

The variables are not part of the observation; a trainer reads them from SimulationManager.program_vars().
"""
from abmarl_b200.program import DeviceProgram
from abmarl_b200.sim.gridworld.actor import BinaryAttackActor, MoveActor
from abmarl_b200.sim.gridworld.smart import SmartGridWorldSimulation

from .sims import BattleAgent

KING_OF_THE_HILL_PROGRAM = r'''
/* KingOfTheHillSim (abmarl_b200/examples/king_of_the_hill.py).  Constants: N_TEAMS, HILL_TOP, HILL_LEFT, HILL_BOTTOM,
 * HILL_RIGHT, TARGET_SCORE, COOLDOWN_STEPS, KILL, DIE, HOLD, WIN.  Variables: SCORE[N_TEAMS + 1], WINNER, COOLDOWN (agent).
 * Role = team, 1 .. N_TEAMS. */
BGWP_FN int on_hill(const bgwp_ctx *c, int a)
{
    const int r = bgwp_row(c, a), col = bgwp_col(c, a);
    return bgwp_active(c, a) && bgwp_in_grid(c, a) && r >= HILL_TOP && r <= HILL_BOTTOM && col >= HILL_LEFT && col <= HILL_RIGHT;
}

BGWP_FN void bgwp_step(bgwp_ctx *c)
{
    int victims[BGW_MAX_VICTIMS];
    const int n = bgwp_n_acting(c);
    for (int i = 0; i < n; ++i) {                              /* attacks, each on its own cooldown */
        const int a = bgwp_acting(c, i);
        if (a < 0 || !bgwp_active(c, a)) continue;
        const double cd = bgwp_agent_var(c, a, COOLDOWN);
        if (cd > 0.0) { bgwp_set_agent_var(c, a, COOLDOWN, cd - 1.0); continue; }
        const int nv = bgwp_attack(c, a, victims);
        if (nv < 0) continue;                                  /* no attack asked for */
        bgwp_set_agent_var(c, a, COOLDOWN, COOLDOWN_STEPS);
        for (int t = 0; t < nv; ++t)
            if (!bgwp_active(c, victims[t])) {
                bgwp_add_reward(c, victims[t], DIE);
                bgwp_add_reward(c, a, KILL);
            }
    }
    for (int i = 0; i < n; ++i) {                              /* then moves */
        const int a = bgwp_acting(c, i);
        if (a >= 0 && bgwp_active(c, a)) bgwp_move(c, a);
    }
    int holder = 0;                                            /* the hill: the one team on it, 0 none, -1 contested */
    for (int a = 0; a < bgwp_n_agents(c); ++a)
        if (on_hill(c, a)) holder = (holder == 0 || holder == bgwp_role(c, a)) ? bgwp_role(c, a) : -1;
    if (holder <= 0) return;
    const double score = bgwp_env_var(c, SCORE + holder) + 1.0;
    bgwp_set_env_var(c, SCORE + holder, score);
    for (int a = 0; a < bgwp_n_agents(c); ++a)
        if (on_hill(c, a)) bgwp_add_reward(c, a, HOLD);
    if (bgwp_env_var(c, WINNER) == 0.0 && score >= TARGET_SCORE) {
        bgwp_set_env_var(c, WINNER, holder);
        for (int a = 0; a < bgwp_n_agents(c); ++a)
            if (bgwp_role(c, a) == holder && bgwp_active(c, a)) bgwp_add_reward(c, a, WIN);
    }
}

#define BGWP_HAS_GET_ALL_DONE
BGWP_FN int bgwp_get_all_done(const bgwp_ctx *c)             /* a winner, or fewer than two teams with an active fighter */
{
    if (bgwp_env_var(c, WINNER) != 0.0) return 1;
    int teams = 0;
    for (int t = 1; t <= N_TEAMS; ++t)
        for (int a = 0; a < bgwp_n_agents(c); ++a)
            if (bgwp_role(c, a) == t && bgwp_active(c, a)) { ++teams; break; }
    return teams < 2;
}
'''


class KingOfTheHillSim(SmartGridWorldSimulation):
    """Build with KingOfTheHillSim.build_sim(rows, cols, agents=..., hill=...) (BattleAgents, team = encoding) or
    KingOfTheHillSim.build(...).  The components default to PositionState + HealthState, a PositionCenteredEncodingObserver,
    ActiveDone, MoveActor and a BinaryAttackActor in which every team attacks every other team.  Runs under
    AllStepManager and TurnBasedManager; SimulationManager.program_vars() holds SCORE [E, n_teams + 1], WINNER [E] and
    COOLDOWN [E, A]."""
    reward_constants = dict(kill=1.0, die=-1.0, hold=0.1, win=1.0)

    def __init__(self, hill=(4, 4, 5, 5), target_score=10, cooldown=2, reward_constants=None, **kwargs):
        super().__init__(**kwargs)
        self.move_actor = MoveActor(**kwargs)
        self.attack_actor = BinaryAttackActor(**kwargs)
        top, left, bottom, right = (int(x) for x in hill)
        assert 0 <= top <= bottom < self.grid.rows and 0 <= left <= right < self.grid.cols, "the hill must lie on the grid"
        assert int(target_score) >= 1 and int(cooldown) >= 0
        self.hill, self.target_score, self.cooldown = (top, left, bottom, right), int(target_score), int(cooldown)
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
        """A random-start instance: team t (1 .. n_teams) has team_size fighters of full health, agents in team order."""
        agents = {f'team{t}_{i}': BattleAgent(id=f'team{t}_{i}', encoding=t, initial_health=1.0)
                  for t in range(1, n_teams + 1) for i in range(team_size)}
        return cls.build_sim(rows, cols, agents=agents, **kwargs)

    def program(self):
        return 'user'                                   # BGW_PROG_USER: device_program() below

    def device_program(self):
        """The step program of this sim: KING_OF_THE_HILL_PROGRAM with the sim's constants and variables; role = team."""
        rc = self.reward_constants
        n_teams = max(agent.encoding for agent in self.agents.values())
        top, left, bottom, right = self.hill
        return DeviceProgram(
            KING_OF_THE_HILL_PROGRAM,
            constants=dict(N_TEAMS=n_teams, HILL_TOP=top, HILL_LEFT=left, HILL_BOTTOM=bottom, HILL_RIGHT=right,
                           TARGET_SCORE=float(self.target_score), COOLDOWN_STEPS=float(self.cooldown),
                           KILL=float(rc['kill']), DIE=float(rc['die']), HOLD=float(rc['hold']), WIN=float(rc['win'])),
            roles={agent: agent.encoding for agent in self.agents.values()},
            env_vars=dict(SCORE=[0.0] * (n_teams + 1), WINNER=0.0),
            agent_vars=dict(COOLDOWN=0.0))
