"""Step programs under the DynamicOrderManager on the B200: the next_agent hook compiled into the step kernel
(bgw_set_program) replays the mm_dynamic transcript, matches the built-in rule and the oracle; AlternatingBattleSim
against the oracle, through rollouts and through the DynamicOrderManager; the refusal of a program without the hook."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from abmarl_b200 import _capi as K
from abmarl_b200.examples import AlternatingBattleSim
from abmarl_b200.layouts import LayoutFeeder, layouts_for
from abmarl_b200.program import DeviceProgram
from abmarl_b200.spec import compile_sim
from tests import dynamic_cases as D
from tests.helpers import assert_outputs_equal, assert_state_equal, run_lockstep
from tests.test_program_dynamic_oracle import names_nobody_spec

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


@pytest.fixture(scope='module', autouse=True)
def _jit_cache(tmp_path_factory):
    """One compilation per (spec, program) for the whole module."""
    with pytest.MonkeyPatch.context() as mp:
        mp.setenv('BGW_JIT_CACHE', str(tmp_path_factory.mktemp('jit')))
        yield


def _engine(spec):
    from abmarl_b200.engine import BatchedGridWorld
    return BatchedGridWorld(spec, device='cuda:0')


def test_mm_dynamic_program_on_the_engine():
    """(1) multi_maze.c + the hook replays mm_dynamic on the device (flags without BGW_ST_NEXT); (2) it matches the oracle
    built with it, 64 envs through auto-resets; (3) it matches the built-in rule on the engine, step by step."""
    g = np.load(os.path.join(GOLDEN, 'mm_dynamic.npz'))
    _, spec = D.mm_dynamic_specs(n_envs=1, seed=int(g['seed']), auto_reset=True)
    eng = _engine(spec)
    episode = 0
    for t in range(len(g['kind'])):
        present = g['obs_present'][t]
        if g['kind'][t] == 0:
            eng.set_layout(layouts_for(spec, [0], [episode]))
            episode += 1
            eng.reset()
        else:
            eng.step(torch.from_numpy(g['actions'][t][None].copy()).cuda())
            np.testing.assert_array_equal(eng.done.cpu().numpy()[0], g['done'][t], err_msg=f'call {t} done')
            np.testing.assert_allclose(eng.reward.cpu().numpy()[0], g['reward'][t], rtol=0, atol=1e-6)
            assert int(eng.all_done.cpu().numpy()[0] & K.ENV_ALL_DONE) == int(g['all_done'][t])
        np.testing.assert_array_equal(eng.obs.cpu().numpy()[0][present], g['obs'][t][present], err_msg=f'call {t} obs')
        st = D.without_next(eng.state_numpy())
        for k in ('flags', 'cell', 'health', 'ammo'):
            np.testing.assert_array_equal(st[k][0], g[k][t], err_msg=f'call {t} {k}')
        in_grid = (g['flags'][t] & K.ST_IN_GRID) != 0
        np.testing.assert_array_equal(st['next'][0][in_grid], g['next'][t][in_grid], err_msg=f'call {t} next')
    assert episode > 1
    # (2) against the oracle with the program
    base, spec = D.mm_dynamic_specs(n_envs=64, env_offset=7, seed=0xC0FFEE, horizon=40, auto_reset=True)
    n = run_lockstep(_engine(spec), D.oracle_env(spec), 300, label='program/mm_dynamic')
    assert n > 0
    # (3) against the built-in rule on the engine
    a, b = _engine(base), _engine(spec)
    for e in (a, b):
        if not e.device_layouts:
            e.feeder = LayoutFeeder(spec)
            e.set_layout(e.feeder.prime(e.state_numpy()['episode']))
        e.reset()
    for t in range(300):
        for e in (a, b):
            e.step_sampled()
            if getattr(e, 'feeder', None) is not None and e.feeder.after_step(e.all_done.cpu().numpy(), e.state_numpy()['episode']):
                e.set_layout(e.feeder.rows)
        for k in ('obs', 'reward', 'done', 'all_done'):
            assert torch.equal(getattr(a, k), getattr(b, k)), f'step {t}: {k} differs from the built-in rule'
        D.assert_state_equal_but_next(a.state_numpy(), b.state_numpy(), f'step {t} (built-in vs program)')


@pytest.mark.parametrize('n_teams', [2, 4])
def test_alternating_battle_engine_matches_oracle(n_teams):
    spec = D.battle_spec(n_teams, n_envs=128, env_offset=5, seed=2026 + n_teams, horizon=40, auto_reset=True)
    eng, ora = _engine(spec), D.oracle_env(spec)
    n = run_lockstep(eng, ora, 300, label=f'alternating_battle/{n_teams}')
    assert n > 0 and int(eng.stats()[K.STAT_AGENT_STEPS].item()) == n
    st = ora.state
    assert not st['error'].any() and st['stats'][:, K.STAT_EPISODES].sum() > 0 and st['stats'][:, K.STAT_KILLS].sum() > 0


def test_alternating_battle_rollout_equals_separate_steps():
    spec = D.battle_spec(3, n_envs=128, seed=5, horizon=30, auto_reset=True)
    a, b = _engine(spec), _engine(spec)
    a.reset()
    b.reset()
    for n in (1, 17, 40):
        a.rollout_sampled(n)
        for _ in range(n):
            b.step_sampled()
        for k in ('obs', 'reward', 'done', 'all_done', 'actions'):
            assert torch.equal(getattr(a, k), getattr(b, k)), f'rollout {n}: {k}'
        assert_state_equal(a.state_numpy(), b.state_numpy(), f'rollout {n}')


def test_alternating_battle_through_the_dynamic_order_manager():
    """`acting` and as_dicts of DynamicOrderManager against the oracle's state and outputs, step by step."""
    from abmarl_b200.managers import DynamicOrderManager
    sim = AlternatingBattleSim.build(rows=8, cols=8, n_teams=3, team_size=3)
    mgr = DynamicOrderManager(sim, n_envs=16, seed=4, horizon=25, auto_reset=True, device='cuda:0')
    ora = D.oracle_env(mgr.spec)
    mgr.reset()
    ora.reset()
    first = mgr.as_dicts(3, after_reset=True)
    assert list(first) == [mgr.learner_ids[int(ora.state['turn'][3])]]
    for t in range(60):
        acting = mgr.acting
        assert acting.dtype == torch.bool and acting.shape == (16, mgr.n_learners) and acting.is_cuda
        np.testing.assert_array_equal(acting.cpu().numpy(), D.acting(mgr.spec, ora.state), err_msg=f'step {t} acting')
        act = mgr.sample_actions()
        mgr.step(act)
        ora.step(act.cpu().numpy())
        assert_outputs_equal(mgr.engine, ora, f'manager step {t}')
        for env in (0, 7):
            if ora.all_done[env] & K.ENV_RESET:
                continue
            obs, rew, done, _ = mgr.as_dicts(env)
            valid = [mgr.learner_ids[l] for l in range(mgr.n_learners) if ora.done[env, l] & K.OUT_VALID]
            assert list(obs) == valid and list(rew) == valid
            assert [done[k] for k in valid] == [bool(ora.done[env, mgr.learner_ids.index(k)] & K.OUT_DONE) for k in valid]
            assert done['__all__'] == bool(ora.all_done[env] & K.ENV_ALL_DONE)


def test_hook_naming_nobody_on_the_engine():
    spec = names_nobody_spec(n_envs=8, seed=3, horizon=6, auto_reset=True)
    eng, ora = _engine(spec), D.oracle_env(spec)
    run_lockstep(eng, ora, 20, label='names nobody')
    assert (ora.state['stats'][:, K.STAT_AGENT_STEPS] == 0).all()
    assert (ora.state['stats'][:, K.STAT_EPISODES] == 3).all()


def test_set_program_without_next_agent_fails_on_a_dynamic_handle():
    spec = D.battle_spec(2, n_envs=4, seed=1)
    lib = K.load()
    c = spec.c_struct()
    h = C.c_void_p()
    K.check(lib.bgw_create(C.byref(c), 0, C.byref(h)), lib)
    try:
        rc = lib.bgw_set_program(h, b'BGWP_FN void bgwp_step(bgwp_ctx *c) { (void)c; }', None)
        msg = lib.bgw_last_error().decode()
        assert rc != 0 and 'nvrtcCompileProgram' in msg and 'bgwp_next_agent' in msg, msg
        K.check(lib.bgw_set_program(h, spec.program_source.encode(), None), lib)
    finally:
        lib.bgw_destroy(h)
    # the same program without the hook runs under the other managers
    program = DeviceProgram('BGWP_FN void bgwp_step(bgwp_ctx *c) { (void)c; }')
    sim = AlternatingBattleSim.build(n_teams=2, team_size=2)
    sim.device_program = lambda: program
    eng = _engine(compile_sim(sim, manager='turn_based', n_envs=4, seed=1))
    eng.reset()
    eng.step_sampled()
