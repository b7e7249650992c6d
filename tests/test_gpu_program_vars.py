"""Variables of a step program's own on the B200: the engine against the CPU oracle bit for bit on outputs, state and
program_vars under every manager, rollouts, masked resets, caller writes, the bgw_set_program_vars rules, and
KingOfTheHillSim."""
import ctypes as C

import numpy as np
import pytest
import torch

from abmarl_b200 import _capi as K
from abmarl_b200.examples import KingOfTheHillSim
from abmarl_b200.spec import compile_sim
from tests import vars_cases as V
from tests.vars_oracle import VarsOracleEnv
from tests.helpers import assert_outputs_equal, assert_state_equal

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module', autouse=True)
def _jit_cache(tmp_path_factory):
    with pytest.MonkeyPatch.context() as mp:
        mp.setenv('BGW_JIT_CACHE', str(tmp_path_factory.mktemp('jit')))
        yield


def _engine(spec):
    from abmarl_b200.engine import BatchedGridWorld
    return BatchedGridWorld(spec, device='cuda:0')


def _compare(eng, ora, where):
    assert_outputs_equal(eng, ora, where)
    assert_state_equal(eng.state_numpy(), ora.state, where)
    V.assert_vars_equal(eng.state['program_vars'].cpu().numpy(), ora.state['program_vars'], where)


@pytest.mark.parametrize('manager', V.MANAGERS)
def test_engine_matches_oracle(manager):
    """Through auto-resets, with env_offset != 0; under the DynamicOrderManager the next_agent hook reads variables."""
    spec = V.stress_spec(manager, n_envs=64, env_offset=13, seed=0xBEEF, horizon=30, auto_reset=True)
    eng, ora = _engine(spec), VarsOracleEnv(spec)
    eng.reset()
    ora.reset()
    _compare(eng, ora, f'{manager} reset')
    for t in range(150):
        act = ora.sample_actions()
        assert np.array_equal(eng.sample_actions().cpu().numpy(), act)
        eng.step(eng.actions)
        ora.step(act)
        _compare(eng, ora, f'{manager} step {t}')
    st = ora.state
    assert not st['error'].any() and st['stats'][:, K.STAT_EPISODES].sum() > 0


def test_rollout_equals_separate_steps():
    spec = V.stress_spec('all_step', n_envs=128, seed=5, horizon=20, auto_reset=True)
    a, b = _engine(spec), _engine(spec)
    a.reset()
    b.reset()
    for n in (1, 13, 40):
        a.rollout_sampled(n)
        for _ in range(n):
            b.step_sampled()
        for k in ('obs', 'reward', 'done', 'all_done', 'actions', 'program_vars'):
            x, y = (getattr(a, k), getattr(b, k)) if k != 'program_vars' else (a.state[k], b.state[k])
            assert torch.equal(x, y), f'rollout {n}: {k}'


def test_masked_reset_and_caller_writes():
    spec = V.stress_spec('turn_based', n_envs=6, seed=8, horizon=40, auto_reset=True)
    eng, ora = _engine(spec), VarsOracleEnv(spec)
    eng.reset()
    ora.reset()
    for t in range(7):
        act = ora.sample_actions()
        eng.step(torch.from_numpy(act).cuda())
        ora.step(act)
    live = (ora.state['env_flags'] & K.ENV_ALL_DONE) == 0      # the others are reset by the next step
    for views in (eng.program_vars(), ora.program_vars()):     # written by the caller, read by the next step
        views['ENERGY'][:] = 0.0
        views['HIST'][:, 3] = 1000.0
    act = ora.sample_actions()
    eng.step(torch.from_numpy(act).cuda())
    ora.step(act)
    _compare(eng, ora, 'after caller writes')
    assert live.any() and (ora.all_done[live] & K.ENV_ALL_DONE).all()   # HIST sums past 4 * ALL_DONE_STEPS
    mask = np.array([0, 1, 1, 0, 0, 1], dtype=np.uint8)
    before = eng.state['program_vars'].clone()
    eng.reset(mask)
    ora.reset(mask)
    _compare(eng, ora, 'masked reset')
    for e in range(spec.n_envs):
        want = torch.from_numpy(spec.program_var_init).cuda() if mask[e] else before[e]
        assert torch.equal(eng.state['program_vars'][e], want), e


@pytest.mark.parametrize('case', ['env var', 'agent'])
def test_index_out_of_range_on_the_device(case):
    from tests.test_program_vars_oracle import BAD_INDEX, bad_index_spec
    spec = bad_index_spec(BAD_INDEX[case])
    eng, ora = _engine(spec), VarsOracleEnv(spec)
    eng.reset()
    ora.reset()
    for t in range(3):
        act = ora.sample_actions()
        eng.step(torch.from_numpy(act).cuda())
        ora.step(act)
        _compare(eng, ora, f'{case} step {t}')
    assert (eng.state['error'] == 3).all()


K_MAX_ENV, K_MAX_AGENT = 65536, 64      # BGW_MAX_ENV_VARS, BGW_MAX_AGENT_VARS (include/bgw.h)


def test_set_program_vars_rules():
    spec = V.stress_spec('all_step', n_envs=4, seed=1)
    lib = K.load()
    init = np.ascontiguousarray(spec.program_var_init)
    vars_ = torch.zeros((4, init.size), dtype=torch.float64, device='cuda:0')
    ip, vp = init.ctypes.data_as(C.c_void_p), vars_.data_ptr()
    n_env, n_agent = spec.n_env_vars, len(spec.agent_var_names)

    def handle(s):
        c = s.c_struct()
        h = C.c_void_p()
        K.check(lib.bgw_create(C.byref(c), 0, C.byref(h)), lib)
        return h

    h = handle(spec)
    try:
        for args in ((-1, 0, ip, vp), (0, -1, ip, vp), (K_MAX_ENV + 1, 0, ip, vp), (0, K_MAX_AGENT + 1, ip, vp),
                     (n_env, n_agent, None, vp), (n_env, n_agent, ip, None)):
            assert lib.bgw_set_program_vars(h, *args) != 0, args
        assert lib.bgw_set_program_vars(h, 0, 0, None, None) == 0             # an empty row needs no buffers
        K.check(lib.bgw_set_program_vars(h, n_env, n_agent, ip, vp), lib)
        K.check(lib.bgw_set_program(h, spec.program_source.encode(), None), lib)
        assert lib.bgw_set_program_vars(h, n_env, n_agent, ip, vp) != 0      # after the program: its counts are compiled in
        assert b'bgw_set_program' in lib.bgw_last_error()
    finally:
        lib.bgw_destroy(h)
    builtin = compile_sim(KingOfTheHillSim.build(), n_envs=4)
    builtin.program, builtin.program_source = K.PROG_TEAM_BATTLE, None
    h = handle(builtin)
    try:
        assert lib.bgw_set_program_vars(h, 1, 0, ip, vp) != 0 and b'BGW_PROG_USER' in lib.bgw_last_error()
    finally:
        lib.bgw_destroy(h)


def test_reset_launches_the_init_kernel_only_with_variables():
    from abmarl_b200.examples import ForagingSim
    with_vars = _engine(V.stress_spec('all_step', n_envs=4, seed=1))
    without = _engine(compile_sim(ForagingSim.build(), n_envs=4, seed=1))
    for eng, extra in ((with_vars, 1), (without, 0)):
        n0 = eng.launches
        eng.reset()
        assert eng.launches - n0 == 1 + extra


def test_a_smaller_handle_leaves_a_larger_one_working():
    """The stock reset and observe kernels are shared by every handle: creating one with less shared memory per env must not
    lower what another one launches with (KingOfTheHillSim needs less than ForagingSim)."""
    from abmarl_b200.examples import ForagingSim
    large = _engine(compile_sim(ForagingSim.build(), n_envs=8, seed=1))
    small = _engine(compile_sim(KingOfTheHillSim.build(), n_envs=8, seed=1))
    assert small.dims.smem_bytes < large.dims.smem_bytes
    for eng in (large, small, large):
        eng.reset()
        eng.observe()
        eng.rollout_sampled(3)
    torch.cuda.synchronize()


# ---- KingOfTheHillSim ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('target_score', sorted(V.KAT_EXPECTED))
def test_king_of_the_hill_known_answer_on_the_device(target_score):
    eng = _engine(compile_sim(V.kat_sim(target_score), n_envs=3, seed=1))
    eng.reset()
    for t in range(len(V.KAT_EXPECTED[target_score])):
        eng.step(torch.from_numpy(V.kat_actions(eng, t)).cuda())
        V.check_kat_step(eng, t, target_score, lambda x: x.cpu().numpy())


@pytest.mark.parametrize('manager', ['all_step', 'turn_based'])
def test_king_of_the_hill_through_the_managers(manager):
    from abmarl_b200.managers import AllStepManager, TurnBasedManager
    cls = AllStepManager if manager == 'all_step' else TurnBasedManager
    mgr = cls(KingOfTheHillSim.build(target_score=4), n_envs=64, env_offset=5, seed=21, horizon=80, auto_reset=True, device='cuda:0')
    ora = VarsOracleEnv(mgr.spec)
    mgr.reset()
    ora.reset()
    for t in range(200):
        act = ora.sample_actions()
        mgr.step(torch.from_numpy(act).cuda())
        ora.step(act)
        _compare(mgr.engine, ora, f'king of the hill {manager} step {t}')
    views = mgr.program_vars()
    assert set(views) == {'SCORE', 'WINNER', 'COOLDOWN'} and views['SCORE'].shape == (64, 3) and views['COOLDOWN'].shape == (64, 8)
    assert ora.state['stats'][:, K.STAT_EPISODES].sum() > 0
