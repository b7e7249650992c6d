"""Step programs (include/bgw_program.h) on the CPU: the oracle built with a program reproduces the recorded transcripts of
the unmodified reference when the program re-expresses the reference's step(), runs in lockstep with the built-in program,
runs ForagingSim (a sim no built-in program expresses) to a hand-computed answer, and guards against bad input; every
program compiles under NVRTC for sm_100a as the engine assembles it; compile_sim / DeviceProgram checks."""
import copy
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from abmarl_b200 import _capi as K
from abmarl_b200.examples.foraging import Forager, ForagingSim, Predator, Resource
from abmarl_b200.program import DeviceProgram
from abmarl_b200.spec import compile_sim
from oracle.build import build_program
from oracle.oracle import OracleEnv, _ptr, lib as oracle_lib
from tests import program_cases as P
from tests import scenarios
from tests.helpers import assert_state_equal

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


@pytest.mark.parametrize('name', list(P.PROGRAM_OF))
def test_program_reproduces_reference_transcript(name):
    """The checks of test_engine_reproduces_reference_transcript, on the oracle built with the re-expressed program."""
    g = np.load(os.path.join(GOLDEN, name + '.npz'))
    _, spec = P.specs(name, n_envs=1, seed=int(g['seed']), auto_reset=False)
    ora = OracleEnv(spec)
    n_valid, episode = 0, -1
    for t in range(len(g['kind'])):
        present = g['obs_present'][t]
        if g['kind'][t] == 0:
            episode += 1
            if spec.layout_generator is not None:
                from abmarl_b200.layouts import layouts_for
                ora.set_layout(layouts_for(spec, [0], [episode]))
            ora.reset()
        else:
            ora.step(g['actions'][t][None])
            np.testing.assert_array_equal(ora.done[0], g['done'][t], err_msg=f'call {t} done')
            np.testing.assert_array_equal(ora.reward64[0], g['reward'][t], err_msg=f'call {t} reward (float64, exact)')
            assert int(ora.all_done[0] & K.ENV_ALL_DONE) == int(g['all_done'][t])
            assert not ora.all_done[0] & K.ENV_ERROR
            n_valid += int(present.sum())
        np.testing.assert_array_equal(ora.obs[0][present], g['obs'][t][present], err_msg=f'call {t} obs')
        st = ora.state
        np.testing.assert_array_equal(st['flags'][0], g['flags'][t], err_msg=f'call {t} flags')
        np.testing.assert_array_equal(st['cell'][0], g['cell'][t], err_msg=f'call {t} cell')
        np.testing.assert_array_equal(st['health'][0], g['health'][t], err_msg=f'call {t} health')
        np.testing.assert_array_equal(st['ammo'][0], g['ammo'][t], err_msg=f'call {t} ammo')
        in_grid = (g['flags'][t] & K.ST_IN_GRID) != 0
        np.testing.assert_array_equal(st['next'][0][in_grid], g['next'][t][in_grid], err_msg=f'call {t} next')
    assert n_valid > 0


def _lockstep(a, b, steps, label, order_fn=None):
    """Drive two oracles with the keyed random policy through auto-resets; outputs (float64 rewards), state equal."""
    feeder = None
    if a.spec.layout_generator is not None:
        from abmarl_b200.layouts import LayoutFeeder
        feeder = LayoutFeeder(a.spec)
        rows = feeder.prime(a.state['episode'])
        a.set_layout(rows)
        b.set_layout(rows)
    a.reset()
    b.reset()
    np.testing.assert_array_equal(a.obs, b.obs)
    episodes = 0
    for t in range(steps):
        act = a.sample_actions()
        np.testing.assert_array_equal(act, b.sample_actions())
        order = None if order_fn is None else order_fn(t)
        a.step(act, order)
        b.step(act, order)
        if feeder is not None and feeder.after_step(a.all_done, a.state['episode']):
            a.set_layout(feeder.rows)
            b.set_layout(feeder.rows)
        for k in ('obs', 'reward64', 'done', 'all_done'):
            np.testing.assert_array_equal(getattr(a, k), getattr(b, k), err_msg=f'{label} step {t} {k}')
        assert_state_equal(a.state, b.state, f'{label} step {t}')
        episodes += int((a.all_done & K.ENV_ALL_DONE).sum())
    assert not (a.state['error'] == 3).any()
    return episodes


@pytest.mark.parametrize('name', ['tb_c2', 'tb_shuffled', 'tb_ammo_selective', 'tb_restricted_stacked', 'mm_c4', 'mm_tiny_allstep',
                                  'pacman_c3'])
def test_program_runs_in_lockstep_with_builtin_program(name):
    """16 envs, 120 steps, auto-reset: the program and the built-in program give identical state, obs, float64 rewards, dones."""
    base, prog = P.specs(name, n_envs=16, env_offset=5, seed=0xBEEF, horizon=30, auto_reset=True)
    episodes = _lockstep(OracleEnv(base), OracleEnv(prog), 120, name)
    assert episodes > 0


def test_program_lockstep_with_caller_order():
    """A caller-given processing order (all_step_manager.py:62-65) reaches the program as its acting order."""
    base, prog = P.specs('tb_c2', n_envs=16, seed=11, horizon=40, auto_reset=True)
    rng = np.random.default_rng(0)
    orders = [np.stack([rng.permutation(base.n_learners) for _ in range(16)]).astype(np.int16) for _ in range(100)]
    _lockstep(OracleEnv(base), OracleEnv(prog), 100, 'tb_c2/order', order_fn=lambda t: orders[t])


# ---- ForagingSim ---------------------------------------------------------------------------------------------------------
def _foraging_kat_sim():
    """3x3: forager f0 at (0,0), forager f1 at (2,2), predator p0 at (2,1), resource r0 at (0,1) with 0.25 health."""
    agents = {'f0': Forager(id='f0', initial_position=np.array([0, 0])),
              'f1': Forager(id='f1', initial_position=np.array([2, 2])),
              'p0': Predator(id='p0', initial_position=np.array([2, 1])),
              'r0': Resource(id='r0', initial_position=np.array([0, 1]), initial_health=0.25)}
    return ForagingSim.build_sim(3, 3, agents=agents, respawn_probability=1.0)


def test_foraging_known_answer():
    """One step: p0 kills f1 (its only candidate), p0's move off the grid fails, f0 steps onto r0 and harvests it to depletion,
    r0 respawns (probability 1) at the cell its keyed draw names."""
    sim = _foraging_kat_sim()
    spec = compile_sim(sim, n_envs=1, seed=1234)
    assert spec.program == K.PROG_USER and list(spec.role) == [1, 1, 2, 3]
    ora = OracleEnv(spec)
    ora.reset()
    np.testing.assert_array_equal(ora.state['health'][0], [1.0, 1.0, 0.0, 0.25])
    act = np.zeros((1, 3, 4), dtype=np.int8)          # learners f0, f1, p0: [dr, dc, attack, 0]
    act[0, 0] = [0, 1, 0, 0]                          # f0 -> (0,1)
    act[0, 1] = [0, 0, 0, 0]                          # f1 stays (it dies first)
    act[0, 2] = [1, 0, 1, 0]                          # p0 attacks, then tries (3,1): off the grid
    ora.step(act)
    st = ora.state
    # where r0 comes back: u = x * 2^-32 of BGW_SITE_PROGRAM slot 3 k 1 at (env 0, episode 0, step 1); cell = floor(u * 9)
    out = (C.c_uint32 * 4)()
    oracle_lib().bgwo_rng_draw(C.c_uint64(1234), 0, 0, 1, K.SITE_PROGRAM, 3, 1, out)
    cell = int(out[0] * 9 // 2**32)
    # rewards (float64, in the order the program adds them): f0 +harvest; f1 die; p0 kill, move_fail
    np.testing.assert_array_equal(ora.reward64[0], [0.0 + 0.5, 0.0 + -1.0, (0.0 + 1.0) + -0.1])
    np.testing.assert_array_equal(ora.done[0], [K.OUT_VALID, K.OUT_VALID | K.OUT_DONE, K.OUT_VALID])
    assert ora.all_done[0] == 0 and st['error'][0] == 0
    np.testing.assert_array_equal(st['health'][0], [1.0, 0.0, 0.0, 1.0])
    np.testing.assert_array_equal(st['flags'][0][:4] & (K.ST_ACTIVE | K.ST_IN_GRID),
                                  [3, 0, 3, 3])                  # f1 dead and out of the grid, r0 back in it
    np.testing.assert_array_equal(st['cell'][0], [1, 8, 7, cell])   # f1 keeps its last cell (actor.py:356-358)
    # cell order: r0 was appended at the tail of its new cell's dict
    occupants = [a for a in (0, 2) if st['cell'][0][a] == cell]
    if occupants:
        assert st['next'][0][occupants[-1]] == 3 and st['next'][0][3] == K.BGW_NONE
    # the episode goes on: f0 and r0 are active (get_all_done is false)
    act[0, 0] = [0, 0, 0, 0]
    act[0, 2] = [0, 0, 1, 0]                          # p0: no forager in range now -> attack_fail
    ora.step(act)
    assert ora.reward64[0][2] == -0.1 and ora.done[0][1] == 0       # f1 was reported done: no row


def test_foraging_runs_200_steps_without_error():
    spec = compile_sim(ForagingSim.build(), n_envs=16, env_offset=3, seed=9, horizon=60, auto_reset=True)
    ora = OracleEnv(spec)
    ora.reset()
    episodes = 0
    for t in range(200):
        ora.step(ora.sample_actions())
        assert not ora.state['error'].any(), f'step {t}'
        assert not (ora.all_done & K.ENV_ERROR).any()
        episodes += int((ora.all_done & K.ENV_ALL_DONE).sum())
    assert episodes > 0
    assert ora.state['stats'][:, K.STAT_KILLS].sum() > 0


def test_oracle_without_the_program_refuses_to_step_it():
    """The plain oracle refuses to step a spec with a step program and writes nothing; OracleEnv(spec) runs the program."""
    spec = compile_sim(ForagingSim.build(), n_envs=2, seed=1)
    ora = OracleEnv(spec)
    ora.reset()
    act = ora.sample_actions()
    state = copy.deepcopy(ora.state)
    outputs = [x.copy() for x in (ora.obs, ora.reward64, ora.done, ora.all_done)]
    rc = oracle_lib().bgwo_step(C.byref(ora._c), C.byref(ora._state_struct()), _ptr(act), None, _ptr(ora.obs), _ptr(ora.reward),
                                _ptr(ora.reward64), _ptr(ora.done), _ptr(ora.all_done))
    assert rc != 0
    assert_state_equal(ora.state, state, 'refused step')
    for x, y in zip((ora.obs, ora.reward64, ora.done, ora.all_done), outputs):
        np.testing.assert_array_equal(x, y)
    ora.step(act)
    assert (ora.state['step'] == 1).all() and not ora.state['error'].any()
    assert (ora.state['cell'] != state['cell']).any() and (ora.done & K.OUT_VALID).all()


def test_program_guard_reports_bad_agent_index():
    """An agent index outside [0, A) does nothing; the env records error 3 and reports ERROR | ALL_DONE, then auto-resets."""
    bad = DeviceProgram('BGWP_FN void bgwp_step(bgwp_ctx *c) { if (bgwp_step_index(c) == 2) bgwp_set_health(c, bgwp_n_agents(c), 0.5); }')
    sim = ForagingSim.build()
    sim.device_program = lambda: bad
    spec = compile_sim(sim, n_envs=4, seed=1, auto_reset=True)
    ora = OracleEnv(spec)
    ora.reset()
    ora.step(ora.sample_actions())
    assert not (ora.all_done & K.ENV_ERROR).any() and not ora.state['error'].any()
    health = ora.state['health'].copy()
    ora.step(ora.sample_actions())
    assert (ora.state['error'] == 3).all()
    assert (ora.all_done == K.ENV_ERROR | K.ENV_ALL_DONE).all()
    np.testing.assert_array_equal(ora.state['health'], health)
    ora.step(ora.sample_actions())                   # auto-reset clears it
    assert (ora.all_done & K.ENV_RESET).all() and not ora.state['error'].any()


# ---- NVRTC: each program compiles into the step kernel; hooks cannot mutate -------------------------------------------------
_HOOK_MUTATES = '''
BGWP_FN void bgwp_step(bgwp_ctx *c) { (void)c; }
#define BGWP_HAS_GET_DONE
BGWP_FN int bgwp_get_done(const bgwp_ctx *c, int a) { bgwp_add_reward(c, a, 1.0); return 0; }
'''


def _program_sources():
    sim = ForagingSim.build()
    yield 'foraging', sim.device_program().assemble(sim.agents)
    for name in ('tb_c2', 'mm_c4', 'pacman_c3'):
        builder = scenarios.SCENARIOS[name][0]
        s = builder(scenarios.mirror_api())
        yield P.PROGRAM_OF[name], P.reexpression(s).assemble(s.agents)


@pytest.mark.parametrize('which', ['foraging', 'team_battle', 'multi_maze', 'pacman'])
def test_program_compiles_under_nvrtc(which):
    pytest.importorskip('cuda.bindings.nvrtc')
    src = dict(_program_sources())[which]
    ok, log, cubin = P.nvrtc_compile(P.jit_source(src))
    assert ok, log[:3000]
    assert b'bgw_step_jit' in cubin


def test_mutating_hook_fails_to_compile():
    with pytest.raises(subprocess.CalledProcessError) as e:
        build_program(_HOOK_MUTATES)
    assert 'discarded-qualifiers' in e.value.stderr, e.value.stderr
    pytest.importorskip('cuda.bindings.nvrtc')
    ok, log, _ = P.nvrtc_compile(P.jit_source(_HOOK_MUTATES))
    assert not ok and 'program' in log, log[:2000]


# ---- compile_sim / DeviceProgram ---------------------------------------------------------------------------------------------
def test_float_constant_round_trips_exactly():
    x = 0.1 + 0.2                                      # not a short decimal
    program = DeviceProgram('BGWP_FN void bgwp_step(bgwp_ctx *c) { bgwp_add_reward(c, 0, X); }', constants={'X': x})
    sim = ForagingSim.build(n_foragers=1, n_predators=1, n_resources=1)
    sim.device_program = lambda: program
    spec = compile_sim(sim, n_envs=1, seed=5)
    assert f'#define X ({x.hex()})' in spec.program_source
    ora = OracleEnv(spec)
    ora.reset()
    act = ora.sample_actions()
    ora.step(act)
    assert ora.reward64[0][0] == x


def test_teambattle_subclass_with_device_program_runs_it(mirror):
    program = DeviceProgram(P.program_text('team_battle'), constants=dict(ATTACK_FAIL=-0.5, KILL=2.0, DIE=-2.0, MOVE_FAIL=0.0,
                                                                          ENTROPY=0.0))

    class MyBattle(mirror.ex.TeamBattleSim):
        def device_program(self):
            return program

    agents = {f'agent{i}': mirror.ex.BattleAgent(id=f'agent{i}', encoding=i % 2 + 1) for i in range(6)}
    sim = MyBattle.build_sim(5, 5, agents=agents, overlapping={1: {1}, 2: {2}}, attack_mapping={1: {2}, 2: {1}},
                             states={'PositionState', 'HealthState'}, observers={'PositionCenteredEncodingObserver'},
                             dones={'OneTeamRemainingDone'})
    spec = compile_sim(sim, n_envs=2, seed=3)
    assert spec.program == K.PROG_USER and '#define KILL (0x1.0000000000000p+1)' in spec.program_source
    assert compile_sim(mirror.ex.TeamBattleSim.build_sim(5, 5, agents=agents, overlapping={1: {1}, 2: {2}},
                                                         attack_mapping={1: {2}, 2: {1}}, states={'PositionState'},
                                                         observers={'PositionCenteredEncodingObserver'})).program == K.PROG_TEAM_BATTLE


def test_program_inputs_are_checked():
    src = 'BGWP_FN void bgwp_step(bgwp_ctx *c) { (void)c; }'
    for bad in ('1X', 'int', 'bgwp_thing', 'BGW_X', 'a-b', ''):
        with pytest.raises(ValueError):
            DeviceProgram(src, constants={bad: 1})
    with pytest.raises(ValueError):
        DeviceProgram(src, constants={'X': float('nan')})
    with pytest.raises(ValueError):
        DeviceProgram(src, roles={'f0': 256})
    sim = ForagingSim.build(n_foragers=2, n_predators=1, n_resources=1)
    for program in (DeviceProgram(src, constants={'T': 'nobody'}), DeviceProgram(src, roles={'nobody': 1}),
                    DeviceProgram(src, constants={'T': Forager(id='stranger')})):
        sim.device_program = lambda program=program: program
        with pytest.raises(ValueError):
            compile_sim(sim)
    sim.device_program = lambda: DeviceProgram(src, constants={'T': sim.agents['forager1'], 'P': 'predator0'})
    assert '#define T (1)\n#define P (2)\n' in compile_sim(sim).program_source
    with pytest.raises(ValueError):
        compile_sim(sim, manager='dynamic_order')
