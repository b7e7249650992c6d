"""Step programs with variables of their own, shared by the CPU and GPU tests: tests/programs/vars_stress.c on a small team
battle under each manager, and the hand-checked known-answer case of KingOfTheHillSim."""
import numpy as np

from abmarl_b200 import _capi as K
from abmarl_b200.examples import AlternatingBattleSim, BattleAgent, KingOfTheHillSim
from abmarl_b200.program import DeviceProgram
from abmarl_b200.spec import compile_sim
from tests import program_cases as P

MANAGERS = ('all_step', 'turn_based', 'dynamic_order')


def stress_program(sim, done_moves=6, all_done_steps=25):
    """vars_stress.c over `sim`: an env scalar, an env array with initial values 0, 0.5, ..., and agent variables whose
    initial values differ per agent (ENERGY) or are one value for all (MOVES)."""
    agents = list(sim.agents)
    return DeviceProgram(P.program_text('vars_stress'), constants=dict(DONE_MOVES=float(done_moves), ALL_DONE_STEPS=float(all_done_steps)),
                         env_vars=dict(STEPS=0.0, HIST=[0.5 * k for k in range(8)]),
                         agent_vars=dict(ENERGY={agent: 1.0 + 0.25 * (i % 4) for i, agent in enumerate(agents) if i % 3},
                                         MOVES=0.0))


def stress_spec(manager='all_step', **kw):
    """A 2-team battle of 3 a side (AlternatingBattleSim's components) running vars_stress.c under `manager`."""
    sim = AlternatingBattleSim.build(rows=8, cols=8, n_teams=2, team_size=3)
    program = stress_program(sim, **{k: kw.pop(k) for k in ('done_moves', 'all_done_steps') if k in kw})
    sim.device_program = lambda: program
    return compile_sim(sim, manager=manager, **kw)


def assert_vars_equal(got, want, where):
    got, want = np.asarray(got), np.asarray(want)
    if not np.array_equal(got, want):
        bad = np.argwhere(got != want)[:5]
        raise AssertionError(f"{where}: program_vars differ at {bad.tolist()}: {got[tuple(bad[0])]} vs {want[tuple(bad[0])]}")


# ---- KingOfTheHillSim, worked out by hand ----------------------------------------------------------------------------------
# 5x5 grid, the hill is the centre cell (2, 2), cooldown 1, every fighter dies to one hit (health 1, strength 1).
#   red0 (team 1) at (2, 1), blue0 (team 2) at (2, 3), blue1 (team 2) at (4, 0); AllStepManager, dict order.
# step 1: blue0 attacks; red0 is two cells away, nobody is in range: an attack all the same, so blue0's COOLDOWN = 1.
#         red0 moves onto the hill, alone there: SCORE[1] = 1, red0 gets HOLD 0.1.
# step 2: blue0 attacks red0 (now adjacent) while on cooldown: ignored, COOLDOWN 1 -> 0; red0 survives and stays:
#         SCORE[1] = 2, red0 0.1.  With target_score 2 red team wins: WINNER = 1, red0 gets WIN too (1.1), episode over.
# step 3 (target_score 3): blue0 attacks again, off cooldown: red0 dies (red0 DIE -1, blue0 KILL 1), COOLDOWN = 1; blue0
#         moves into the freed hill cell: SCORE[2] = 1, blue0 1 + 0.1.  No red fighter is left: the episode is over.
KAT_ACTIONS = [  # (dr, dc, attack) of red0, blue0, blue1
    [(0, 1, 0), (0, 0, 1), (0, 0, 0)],
    [(0, 0, 0), (0, 0, 1), (0, 0, 0)],
    [(0, 0, 0), (0, -1, 1), (0, 0, 0)],
]
# per target_score: per step (rewards, done bits, all_done, SCORE, WINNER, COOLDOWN)
KAT_EXPECTED = {
    2: [([0.1, 0.0, 0.0], [0, 0, 0], 0, [0, 1, 0], 0, [0, 1, 0]),
        ([1.0 + 0.1, 0.0, 0.0], [0, 0, 0], 1, [0, 2, 0], 1, [0, 0, 0])],
    3: [([0.1, 0.0, 0.0], [0, 0, 0], 0, [0, 1, 0], 0, [0, 1, 0]),
        ([0.1, 0.0, 0.0], [0, 0, 0], 0, [0, 2, 0], 0, [0, 0, 0]),
        ([-1.0, 1.0 + 0.1, 0.0], [1, 0, 0], 1, [0, 2, 1], 0, [0, 1, 0])],
}


def kat_sim(target_score):
    agents = {'red0': BattleAgent(id='red0', encoding=1, initial_health=1.0, initial_position=np.array([2, 1])),
              'blue0': BattleAgent(id='blue0', encoding=2, initial_health=1.0, initial_position=np.array([2, 3])),
              'blue1': BattleAgent(id='blue1', encoding=2, initial_health=1.0, initial_position=np.array([4, 0]))}
    return KingOfTheHillSim.build_sim(5, 5, agents=agents, hill=(2, 2, 2, 2), target_score=target_score, cooldown=1)


def kat_actions(env, step):
    """int8 [E, L, action_stride] of the scripted step for every env"""
    act = np.zeros((env.E, env.L, env.dims.action_stride), dtype=np.int8)
    for l, (dr, dc, att) in enumerate(KAT_ACTIONS[step]):
        act[:, l, :3] = (dr, dc, att)
    return act


def check_kat_step(env, step, target_score, host):
    """Compare env's outputs and variables after scripted step `step` with KAT_EXPECTED; `host` gives numpy arrays."""
    rewards, dones, all_done, score, winner, cooldown = KAT_EXPECTED[target_score][step]
    where = f'king of the hill, target {target_score}, step {step + 1}'
    np.testing.assert_array_equal(host(env.reward), np.tile(np.float32(rewards), (env.E, 1)), err_msg=where)
    np.testing.assert_array_equal(host(env.done), np.tile(np.uint8([K.OUT_VALID | d for d in dones]), (env.E, 1)), err_msg=where)
    assert (host(env.all_done) & K.ENV_ALL_DONE == all_done).all(), where
    v = {k: host(x) for k, x in env.program_vars().items()}
    np.testing.assert_array_equal(v['SCORE'], np.tile(np.float64(score), (env.E, 1)), err_msg=where)
    np.testing.assert_array_equal(v['WINNER'], np.full(env.E, float(winner)), err_msg=where)
    np.testing.assert_array_equal(v['COOLDOWN'], np.tile(np.float64(cooldown), (env.E, 1)), err_msg=where)
