"""Variables of a step program's own (include/bgw_program.h, DeviceProgram(env_vars=, agent_vars=)) on the CPU oracle: the
declarations, persistence across steps, initial values at every kind of reset, caller writes, bad indices, hooks that may
only read, and the hand-checked KingOfTheHillSim case."""
import subprocess

import numpy as np
import pytest

from abmarl_b200 import _capi as K
from abmarl_b200.examples import AlternatingBattleSim, KingOfTheHillSim
from abmarl_b200.program import DeviceProgram
from abmarl_b200.spec import compile_sim
from tests import program_cases as P
from tests import vars_cases as V
from tests.vars_oracle import VarsOracleEnv, build_vars


# ---- declarations ----------------------------------------------------------------------------------------------------------
def test_declarations_are_checked():
    src = 'BGWP_FN void bgwp_step(bgwp_ctx *c) { (void)c; }'
    for kw in (dict(env_vars={'2X': 0.0}), dict(agent_vars={'bgwp_x': 0.0}), dict(env_vars={'int': 1.0}),
               dict(env_vars={'X': float('nan')}), dict(env_vars={'X': []}), dict(env_vars={'X': 'abc'}),
               dict(env_vars={'X': [1.0, float('inf')]}), dict(agent_vars={'X': True}), dict(agent_vars={'X': {'a': 'b'}}),
               dict(constants={'X': 1}, env_vars={'X': 0.0}), dict(env_vars={'X': 0.0}, agent_vars={'X': 0.0})):
        with pytest.raises(ValueError):
            DeviceProgram(src, **kw)


def test_defines_and_initial_row():
    sim = AlternatingBattleSim.build(rows=6, cols=6, n_teams=2, team_size=2)
    ids = list(sim.agents)
    prog = DeviceProgram('BGWP_FN void bgwp_step(bgwp_ctx *c) { (void)c; }', constants={'N': 3},
                         env_vars=dict(A=1.5, B=[1, 2, 3], C=-2), agent_vars=dict(X=0.25, Y={ids[1]: 4.0, sim.agents[ids[3]]: -1}))
    text = prog.assemble(sim.agents)
    for line in ('#define N (3)', '#define A (0)', '#define B (1)', '#define C (4)', '#define X (0)', '#define Y (1)'):
        assert line in text.splitlines(), line
    assert prog.env_var_slots() == {'A': (0, None), 'B': (1, 3), 'C': (4, None)}
    assert (prog.n_env_vars, prog.n_agent_vars) == (5, 2)
    assert prog.var_init(sim.agents) == [1.5, 1.0, 2.0, 3.0, -2.0] + [0.25, 0.0, 0.25, 4.0, 0.25, 0.0, 0.25, -1.0]
    with pytest.raises(ValueError):
        DeviceProgram(prog.source, agent_vars=dict(Y={'nobody': 1.0})).var_init(sim.agents)
    sim.device_program = lambda: prog
    spec = compile_sim(sim, n_envs=3)
    assert spec.env_var_slots == prog.env_var_slots() and spec.agent_var_names == ['X', 'Y'] and spec.n_env_vars == 5
    np.testing.assert_array_equal(spec.program_var_init, prog.var_init(sim.agents))
    views = spec.program_var_views(np.arange(3 * 13, dtype=np.float64).reshape(3, 13))
    assert {k: v.shape for k, v in views.items()} == {'A': (3,), 'B': (3, 3), 'C': (3,), 'X': (3, 4), 'Y': (3, 4)}
    np.testing.assert_array_equal(views['Y'][1], [13 + 6, 13 + 8, 13 + 10, 13 + 12])
    # a program without variables carries none
    plain = compile_sim(AlternatingBattleSim.build(rows=6, cols=6, n_teams=2, team_size=2), n_envs=3)
    assert plain.program_var_init is None and plain.env_var_slots == {} and plain.agent_var_names == []


# ---- the oracle ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('manager', V.MANAGERS)
def test_variables_persist_and_reset(manager):
    """Variables change only through the program between resets and come back at auto-resets; every env holds its own."""
    spec = V.stress_spec(manager, n_envs=8, seed=11, horizon=30, auto_reset=True)
    ora = VarsOracleEnv(spec)
    ora.reset()
    init = spec.program_var_init
    assert (ora.state['program_vars'] == init).all()
    resets = 0
    for t in range(120):
        before = ora.state['program_vars'].copy()
        was_done = (ora.state['env_flags'] & K.ENV_ALL_DONE) != 0
        ora.step(ora.sample_actions())
        rows = ora.state['program_vars']
        v = ora.program_vars()
        for e in range(spec.n_envs):
            if was_done[e]:                                   # auto-reset: the initial row
                resets += 1
                V.assert_vars_equal(rows[e], init, f'{manager} step {t} env {e} auto-reset')
            else:                                             # the program counted this step
                assert v['STEPS'][e] == before[e, 0] + 1.0
                assert v['HIST'][e].sum() >= before[e, 1:9].sum()
    assert resets > 0
    assert not ora.state['error'].any()
    assert len({tuple(r) for r in ora.state['program_vars']}) > 1          # the envs went their own ways


def test_masked_reset_and_caller_writes():
    spec = V.stress_spec('all_step', n_envs=6, seed=5, horizon=40, auto_reset=True)
    ora = VarsOracleEnv(spec)
    ora.reset()
    for _ in range(5):
        ora.step(ora.sample_actions())
    v = ora.program_vars()
    v['ENERGY'][:] = 0.0                                  # the caller owns the buffer: the next step sees what it writes
    v['STEPS'][:] = 100.0
    ora.step(ora.sample_actions())
    assert (v['STEPS'] == 101.0).all() and (ora.all_done & K.ENV_ALL_DONE).all()   # >= ALL_DONE_STEPS: every env ends
    live = (ora.state['flags'][:, :] & K.ST_ACTIVE) != 0
    assert (v['ENERGY'][live] == 0.25).all()               # nobody had the energy to move: everyone rested
    mask = np.array([1, 0, 1, 0, 0, 1], dtype=np.uint8)
    before = ora.state['program_vars'].copy()
    ora.reset(mask)
    rows = ora.state['program_vars']
    for e in range(spec.n_envs):
        V.assert_vars_equal(rows[e], spec.program_var_init if mask[e] else before[e], f'masked reset env {e}')


def test_failed_placement_resets_the_variables():
    """A reset whose placement fails (BGW_ENV_ERROR) still writes the initial values."""
    spec = V.stress_spec('all_step', n_envs=2, seed=1)
    spec.init_row[:] = 0                                   # every agent on cell (0, 0): a fixed-position conflict
    spec.init_col[:] = 0
    ora = VarsOracleEnv(spec)
    ora.state['program_vars'][:] = 7.0
    ora.reset()
    assert (ora.state['error'] == 1).all() and (ora.state['env_flags'] & K.ENV_ERROR).all()
    assert (ora.state['program_vars'] == spec.program_var_init).all()


BAD_INDEX = {
    'env var': 'bgwp_set_env_var(c, bgwp_n_env_vars(c), 1.0);',
    'negative env var': 'x = bgwp_env_var(c, -1);',
    'agent var': 'x = bgwp_agent_var(c, 0, bgwp_n_agent_vars(c));',
    'agent': 'bgwp_set_agent_var(c, bgwp_n_agents(c), 0, 1.0);',
}


def bad_index_spec(statement):
    src = ('BGWP_FN void bgwp_step(bgwp_ctx *c)\n{\n    double x = 0.0;\n    if (bgwp_step_index(c) == 2) { ' + statement +
           ' }\n    bgwp_set_env_var(c, S, bgwp_env_var(c, S) + 1.0 + x);\n}\n')
    sim = AlternatingBattleSim.build(rows=6, cols=6, n_teams=2, team_size=2)
    prog = DeviceProgram(src, env_vars=dict(S=0.0, T=[1.0, 2.0]), agent_vars=dict(U=3.0))
    sim.device_program = lambda: prog
    return compile_sim(sim, n_envs=2, seed=3)


@pytest.mark.parametrize('case', list(BAD_INDEX))
def test_index_out_of_range_is_error_3(case):
    ora = VarsOracleEnv(bad_index_spec(BAD_INDEX[case]))
    ora.reset()
    ora.step(ora.sample_actions())
    assert not ora.state['error'].any() and not (ora.all_done & K.ENV_ALL_DONE).any()
    ora.step(ora.sample_actions())
    assert (ora.state['error'] == 3).all()
    assert (ora.all_done == (K.ENV_ERROR | K.ENV_ALL_DONE)).all()
    v = ora.program_vars()
    assert (v['S'] == 2.0).all() and (v['T'] == [1.0, 2.0]).all() and (v['U'] == 3.0).all()   # nothing written, 0.0 read


WRITING_HOOKS = {
    'get_done': '#define BGWP_HAS_GET_DONE\nBGWP_FN int bgwp_get_done(const bgwp_ctx *c, int a) { bgwp_set_env_var(c, S, 1.0); return a < 0; }',
    'get_all_done': '#define BGWP_HAS_GET_ALL_DONE\nBGWP_FN int bgwp_get_all_done(const bgwp_ctx *c) { bgwp_set_agent_var(c, 0, U, 1.0); return 0; }',
    'get_reward': '#define BGWP_HAS_GET_REWARD\nBGWP_FN double bgwp_get_reward(const bgwp_ctx *c, int a, double acc) '
                  '{ bgwp_set_agent_var(c, a, U, acc); return acc; }',
}


@pytest.mark.parametrize('hook', list(WRITING_HOOKS))
def test_a_hook_that_writes_a_variable_does_not_compile(hook):
    body = 'BGWP_FN void bgwp_step(bgwp_ctx *c) { bgwp_set_env_var(c, S, bgwp_agent_var(c, 0, U)); }\n'
    ok_src = DeviceProgram(body, env_vars=dict(S=0.0), agent_vars=dict(U=0.0)).assemble({'a': None})
    bad_src = DeviceProgram(body + WRITING_HOOKS[hook], env_vars=dict(S=0.0), agent_vars=dict(U=0.0)).assemble({'a': None})
    build_vars(ok_src)
    with pytest.raises(subprocess.CalledProcessError) as err:
        build_vars(bad_src)
    assert 'discards' in err.value.stderr and 'qualifier' in err.value.stderr
    assert P.nvrtc_compile(P.jit_source(ok_src))[0]
    ok, log, _ = P.nvrtc_compile(P.jit_source(bad_src))
    assert not ok and 'error' in log and 'const' in log, log


# ---- KingOfTheHillSim --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('target_score', sorted(V.KAT_EXPECTED))
def test_king_of_the_hill_known_answer(target_score):
    ora = VarsOracleEnv(compile_sim(V.kat_sim(target_score), n_envs=2, seed=1))
    ora.reset()
    assert (ora.program_vars()['COOLDOWN'] == 0.0).all()
    for t in range(len(V.KAT_EXPECTED[target_score])):
        ora.step(V.kat_actions(ora, t))
        V.check_kat_step(ora, t, target_score, np.asarray)


@pytest.mark.parametrize('manager', ['all_step', 'turn_based'])
def test_king_of_the_hill_plays_out(manager):
    ora = VarsOracleEnv(compile_sim(KingOfTheHillSim.build(target_score=5), manager=manager, n_envs=16, seed=9, horizon=100,
                                auto_reset=True))
    ora.reset()
    winners = 0
    for _ in range(300):
        ora.step(ora.sample_actions())
        winners += int(((ora.program_vars()['WINNER'] > 0) & ((ora.all_done & K.ENV_ALL_DONE) != 0)).sum())
    v = ora.program_vars()
    assert not ora.state['error'].any() and winners > 0
    assert (v['SCORE'][:, 0] == 0).all() and (v['SCORE'] <= 5).all() and (v['COOLDOWN'] <= 2).all()
