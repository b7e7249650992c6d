"""Step programs under the DynamicOrderManager on the CPU: the next_agent hook (include/bgw_program.h) of multi_maze.c
reproduces the mm_dynamic transcript of the reference and runs in lockstep with the built-in rule; AlternatingBattleSim
to a hand-computed answer; a program without the hook is refused, a hook that names nobody steps with no actors, a
mutating hook does not compile; the new programs compile under NVRTC as the engine assembles them."""
import copy
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from abmarl_b200 import _capi as K
from abmarl_b200.examples import AlternatingBattleSim, BattleAgent
from abmarl_b200.layouts import LayoutFeeder, layouts_for
from abmarl_b200.program import DeviceProgram
from abmarl_b200.spec import compile_sim
from oracle.oracle import _ptr
from tests import dynamic_cases as D
from tests import program_cases as P
from tests import scenarios

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def test_mm_dynamic_program_reproduces_reference_transcript():
    """multi_maze.c + the next_agent hook on the oracle replays the 500 calls of mm_dynamic (flags without BGW_ST_NEXT)."""
    g = np.load(os.path.join(GOLDEN, 'mm_dynamic.npz'))
    _, spec = D.mm_dynamic_specs(n_envs=1, seed=int(g['seed']), auto_reset=False)
    ora = D.oracle_env(spec)
    n_valid, episodes = 0, 0
    for t in range(len(g['kind'])):
        present = g['obs_present'][t]
        if g['kind'][t] == 0:
            ora.set_layout(layouts_for(spec, [0], [episodes]))
            episodes += 1
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
        np.testing.assert_array_equal(st['flags'][0] & ~np.uint8(K.ST_NEXT), g['flags'][t], err_msg=f'call {t} flags')
        for k in ('cell', 'health', 'ammo'):
            np.testing.assert_array_equal(st[k][0], g[k][t], err_msg=f'call {t} {k}')
        in_grid = (g['flags'][t] & K.ST_IN_GRID) != 0
        np.testing.assert_array_equal(st['next'][0][in_grid], g['next'][t][in_grid], err_msg=f'call {t} next')
    assert n_valid > 0 and episodes > 1


def _lockstep(a, b, steps, label):
    """Drive two oracles with the keyed random policy through auto-resets: outputs and state equal but for BGW_ST_NEXT."""
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
        a.step(act)
        b.step(act)
        if feeder.after_step(a.all_done, a.state['episode']):
            a.set_layout(feeder.rows)
            b.set_layout(feeder.rows)
        for k in ('obs', 'reward64', 'done', 'all_done'):
            np.testing.assert_array_equal(getattr(a, k), getattr(b, k), err_msg=f'{label} step {t} {k}')
        D.assert_state_equal_but_next(a.state, b.state, f'{label} step {t}')
        episodes += int((a.all_done & K.ENV_ALL_DONE).sum())
    return episodes


def test_mm_dynamic_program_lockstep_with_builtin_rule():
    """32 envs, 400 steps, auto-reset and a horizon: the built-in rule and the hook give identical outputs and state."""
    base, prog = D.mm_dynamic_specs(n_envs=32, env_offset=3, seed=0xD1CE, horizon=40, auto_reset=True)
    episodes = _lockstep(D.oracle_env(base), D.oracle_env(prog), 400, 'mm_dynamic')
    assert episodes > 32


# ---- AlternatingBattleSim ------------------------------------------------------------------------------------------------
def _battle_kat_sim():
    """3x3, health 1 (one hit kills): team 1 = a0 (0,0), a1 (2,2); team 2 = b0 (0,1), b1 (2,0)."""
    pos = {'a0': (0, 0), 'a1': (2, 2), 'b0': (0, 1), 'b1': (2, 0)}
    agents = {k: BattleAgent(id=k, encoding=1 if k[0] == 'a' else 2, initial_position=np.array(p), initial_health=1.0)
              for k, p in pos.items()}
    return AlternatingBattleSim.build_sim(3, 3, agents=agents)


def test_alternating_battle_known_answer():
    spec = compile_sim(_battle_kat_sim(), manager='dynamic_order', n_envs=1, seed=77)
    assert spec.program == K.PROG_USER and list(spec.role) == [1, 1, 2, 2]
    ora = D.oracle_env(spec)
    ora.reset()
    assert ora.state['turn'][0] == 0
    act = np.zeros((1, 4, 4), dtype=np.int8)          # learners a0, a1, b0, b1: [dr, dc, attack, 0]
    act[0, :, 2] = 1                                   # everyone asks for an attack; only the acting rows are read
    act[0, 3, :2] = [0, 1]                             # b1 steps right when it acts
    VD = K.OUT_VALID | K.OUT_DONE

    # step 1: reset named a0 alone.  a0 kills b0 (its only candidate), stays, pays the entropy.  next_agent: b0 (dead) and
    # team 2's active member b1; a0 is not named, its reward waits
    ora.step(act)
    np.testing.assert_array_equal(ora.done[0], [0, 0, VD, K.OUT_VALID])
    np.testing.assert_array_equal(ora.reward64[0], [0.0, 0.0, 0.0 + -1.0, 0.0])
    assert ora.all_done[0] == 0 and ora.state['turn'][0] == 3
    np.testing.assert_array_equal(ora.state['flags'][0] & (K.ST_NEXT | K.ST_DONE_REPORTED), [0, 0, K.ST_DONE_REPORTED, K.ST_NEXT])
    np.testing.assert_array_equal(D.acting(spec, ora.state)[0], [False, False, False, True])

    # step 2: b1 alone: no team-1 agent within range (attack_fail), moves to (2,1), entropy.  next_agent: team 1 (a0, a1)
    ora.step(act)
    np.testing.assert_array_equal(ora.done[0], [K.OUT_VALID, K.OUT_VALID, 0, 0])
    np.testing.assert_array_equal(ora.reward64[0], [(0.0 + 1.0) + -0.01, 0.0, 0.0, 0.0])
    assert ora.all_done[0] == 0 and ora.state['turn'][0] == 0
    assert ora.state['cell'][0][3] == 2 * 3 + 1
    np.testing.assert_array_equal(D.acting(spec, ora.state)[0], [True, True, False, False])

    # step 3: a0 and a1 together: a0 finds nobody (attack_fail), a1 kills b1 next to it; one team remains: every learner not
    # yet reported receives its accumulated reward
    ora.step(act)
    np.testing.assert_array_equal(ora.done[0], [K.OUT_VALID, K.OUT_VALID, 0, VD])
    np.testing.assert_array_equal(ora.reward64[0], [(0.0 + -0.1) + -0.01, (0.0 + 1.0) + -0.01, 0.0, ((0.0 + -0.1) + -0.01) + -1.0])
    assert ora.all_done[0] == K.ENV_ALL_DONE and ora.state['turn'][0] == 0
    assert ora.state['stats'][0][K.STAT_AGENT_STEPS] == 2 + 2 + 3


def test_alternating_battle_runs_with_auto_reset():
    """3 and 4 teams, 300 steps: episodes end by one team remaining and by the horizon, never by an error; acting sets of
    more than one learner and deaths reported off-turn occur."""
    for n_teams in (3, 4):
        spec = D.battle_spec(n_teams, n_envs=32, seed=n_teams, horizon=50, auto_reset=True)
        ora = D.oracle_env(spec)
        ora.reset()
        wide = off_turn = 0
        for _ in range(300):
            before = D.acting(spec, ora.state)
            wide += int((before.sum(1) > 1).sum())
            ora.step(ora.sample_actions())
            off_turn += int(((ora.done & K.OUT_DONE) != 0)[~before & ((ora.all_done & K.ENV_ALL_DONE) == 0)[:, None]].sum())
            assert not ora.state['error'].any() and not (ora.all_done & K.ENV_ERROR).any()
        st = ora.state['stats']
        assert st[:, K.STAT_EPISODES].sum() > 0 and st[:, K.STAT_KILLS].sum() > 0
        assert wide > 0 and off_turn > 0


# ---- edges and errors ----------------------------------------------------------------------------------------------------
_NAMES_NOBODY = P.program_text('team_battle') + '''
#define BGWP_HAS_GET_ALL_DONE
BGWP_FN int bgwp_get_all_done(const bgwp_ctx *c) { (void)c; return 0; }
#define BGWP_HAS_NEXT_AGENT
BGWP_FN int bgwp_next_agent(const bgwp_ctx *c, int a) { (void)c; (void)a; return 0; }
'''
_BATTLE_CONSTANTS = dict(ATTACK_FAIL=-0.1, KILL=1.0, DIE=-1.0, MOVE_FAIL=-0.1, ENTROPY=-0.01)


def names_nobody_spec(**kw):
    sim = AlternatingBattleSim.build(rows=6, cols=6, n_teams=2, team_size=2)
    program = DeviceProgram(_NAMES_NOBODY, constants=_BATTLE_CONSTANTS)
    sim.device_program = lambda: program
    return compile_sim(sim, manager='dynamic_order', **kw)


def test_hook_naming_nobody_steps_without_actors_until_the_horizon():
    spec = names_nobody_spec(n_envs=4, seed=3, horizon=6)
    ora = D.oracle_env(spec)
    ora.reset()
    ora.step(ora.sample_actions())                     # learner 0 acts, nobody is named
    assert (ora.done == 0).all() and (ora.state['turn'] == -1).all() and not D.acting(spec, ora.state).any()
    cell = ora.state['cell'].copy()
    for t in range(2, 7):
        ora.step(ora.sample_actions())
        assert (ora.done == 0).all() and not ora.state['error'].any()
        np.testing.assert_array_equal(ora.state['cell'], cell)
        want = K.ENV_ALL_DONE | K.ENV_TRUNCATED if t == 6 else 0
        assert (ora.all_done == want).all(), t
    assert (ora.state['stats'][:, K.STAT_AGENT_STEPS] == 0).all()


_NO_HOOK = 'BGWP_FN void bgwp_step(bgwp_ctx *c) { (void)c; }\n'


def test_dynamic_program_without_next_agent_is_refused():
    sim = AlternatingBattleSim.build(n_teams=2, team_size=2)
    sim.device_program = lambda: DeviceProgram(_NO_HOOK)
    with pytest.raises(ValueError, match='BGWP_HAS_NEXT_AGENT'):
        compile_sim(sim, manager='dynamic_order')
    spec = compile_sim(sim, manager='all_step', n_envs=2, seed=1)   # the other managers do not need it
    D.oracle_env(spec).step(np.zeros((2, spec.n_learners, 4), dtype=np.int8))
    # the CPU reference built with such a program refuses a dynamic-order spec and writes nothing; so does the oracle's
    # own manager step, which runs programs under the other managers only
    spec.manager = K.MANAGER_DYNAMIC_ORDER
    ora = D.oracle_env(spec)
    ora.reset()
    state = copy.deepcopy(ora.state)
    act = ora.sample_actions()
    assert ora.step_rc(act) != 0
    rc = ora._lib.bgwo_step(C.byref(ora._c), C.byref(ora._state_struct()), _ptr(act), None, _ptr(ora.obs), _ptr(ora.reward),
                            _ptr(ora.reward64), _ptr(ora.done), _ptr(ora.all_done))
    assert rc != 0
    D.assert_state_equal_but_next(ora.state, state, 'refused step')


def test_a_dynamic_program_needs_a_dynamic_order_simulation():
    sim = D.mm_dynamic_program(scenarios.SCENARIOS['mm_tiny'][0](scenarios.mirror_api()))
    with pytest.raises(ValueError, match='DynamicOrderSimulation'):
        compile_sim(sim, manager='dynamic_order')


def test_one_program_serves_every_manager():
    """The hook is ignored under the all-step and turn-based managers."""
    for manager in ('all_step', 'turn_based'):
        spec = compile_sim(AlternatingBattleSim.build(rows=8, cols=8), manager=manager, n_envs=4, seed=2, horizon=20,
                           auto_reset=True)
        ora = D.oracle_env(spec)
        ora.reset()
        for _ in range(40):
            ora.step(ora.sample_actions())
            assert not (ora.state['flags'] & K.ST_NEXT).any()


# ---- NVRTC and gcc: the programs compile into the step kernel; the hook cannot mutate --------------------------------------
def dynamic_jit_source(program_source):
    """The kernel source bgwjit::build assembles for a handle under the dynamic-order manager."""
    return (P.jit_source(program_source).replace('s.manager=0;', 's.manager=2;')
            .replace('#include "bgw_dev.cuh"\n', '#include "bgw_dev.cuh"\n#define BGWP_DYNAMIC_ORDER\n', 1))


def _dynamic_sources():
    _, spec = D.mm_dynamic_specs()
    yield 'multi_maze_next_agent', spec.program_source
    yield 'alternating_battle', D.battle_spec(2).program_source


@pytest.mark.parametrize('which', ['multi_maze_next_agent', 'alternating_battle'])
def test_dynamic_program_compiles_under_nvrtc(which):
    pytest.importorskip('cuda.bindings.nvrtc')
    ok, log, cubin = P.nvrtc_compile(dynamic_jit_source(dict(_dynamic_sources())[which]))
    assert ok, log[:3000]
    assert b'bgw_step_jit' in cubin


def test_missing_next_agent_fails_under_nvrtc():
    pytest.importorskip('cuda.bindings.nvrtc')
    ok, log, _ = P.nvrtc_compile(dynamic_jit_source(_NO_HOOK))
    assert not ok and 'bgwp_next_agent' in log, log[:2000]
    ok, log, _ = P.nvrtc_compile(P.jit_source(_NO_HOOK))          # the other managers: no hook needed
    assert ok, log[:2000]


_HOOK_MUTATES = '''
BGWP_FN void bgwp_step(bgwp_ctx *c) { (void)c; }
#define BGWP_HAS_NEXT_AGENT
BGWP_FN int bgwp_next_agent(const bgwp_ctx *c, int a) { bgwp_set_active(c, a, 0); return 1; }
'''


def test_mutating_next_agent_fails_to_compile():
    with pytest.raises(subprocess.CalledProcessError) as e:
        D.build_dynamic(_HOOK_MUTATES)
    assert 'discarded-qualifiers' in e.value.stderr, e.value.stderr
    pytest.importorskip('cuda.bindings.nvrtc')
    ok, log, _ = P.nvrtc_compile(dynamic_jit_source(_HOOK_MUTATES))
    assert not ok and 'program' in log, log[:2000]
