"""Step programs on the B200: the engine with a program compiled into its step kernel (bgw_set_program) against the reference
transcripts, the oracle built with the same program, and the built-in programs; ForagingSim through the managers; the
C-ABI rules of bgw_set_program."""
import copy
import ctypes as C
import os

import numpy as np
import pytest
import torch

from abmarl_b200 import _capi as K
from abmarl_b200.examples.foraging import ForagingSim
from abmarl_b200.program import DeviceProgram
from abmarl_b200.spec import compile_sim
from tests import program_cases as P
from tests.helpers import assert_outputs_equal, assert_state_equal, run_lockstep

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


@pytest.fixture(scope='module', autouse=True)
def _jit_cache(tmp_path_factory):
    """One compilation per (spec, program) for the whole module: the handles of one scenario share their cubin."""
    with pytest.MonkeyPatch.context() as mp:
        mp.setenv('BGW_JIT_CACHE', str(tmp_path_factory.mktemp('jit')))
        yield


def _engine(spec):
    from abmarl_b200.engine import BatchedGridWorld
    return BatchedGridWorld(spec, device='cuda:0')


def _oracle(spec):
    from tests.program_oracle import ProgramOracleEnv
    return ProgramOracleEnv(spec)


# the scenario sizes of test_gpu_parity.CASES (tb_c5, the 64x64 headline shape, which that list leaves to other tests: 16 envs)
CASES = {'tb_c2': (64, 120, 50), 'tb_c5': (16, 40, 20), 'tb_c5_small': (24, 90, 40), 'tb_dense': (64, 120, 30), 'tb_blocking': (48, 100, 40),
         'tb_stacked': (48, 80, 30), 'tb_noself': (48, 80, 30), 'tb_shuffled': (48, 120, 25), 'tb_c5_shuffled': (24, 90, 30),
         'tb_position': (48, 90, 30), 'tb_encoding': (48, 100, 30), 'tb_encoding_stacked': (48, 100, 30),
         'tb_restricted': (48, 100, 30), 'tb_restricted_stacked': (48, 100, 30), 'tb_selective': (48, 100, 30),
         'tb_selective_stacked': (48, 100, 30), 'tb_ammo': (48, 100, 30), 'tb_ammo_selective': (48, 100, 30),
         'pacman_c3': (6, 40, 25), 'mm_c4': (12, 150, 60), 'mm_random': (12, 120, 50), 'mm_allstep': (12, 100, 40),
         'mm_tbf': (16, 200, 30), 'mm_tbf_scatter': (16, 200, 30), 'mm_tiny': (16, 300, 0), 'mm_tiny_allstep': (16, 200, 0)}


@pytest.mark.parametrize('name', list(P.PROGRAM_OF))
def test_program_on_the_engine(name):
    """The re-expressed program on the device: (1) it replays the reference's transcript; (2) it matches the oracle built
    with the program at the parity-test size, through auto-resets, env_offset != 0; (3) its outputs and state are
    bit-identical to the built-in program's on the engine, step by step."""
    assert name in CASES
    # (1) the transcript (auto_reset on: every episode of a transcript starts with an explicit reset, and the handle then
    # shares its compiled kernel with the runs below)
    g = np.load(os.path.join(GOLDEN, name + '.npz'))
    _, spec = P.specs(name, n_envs=1, seed=int(g['seed']), auto_reset=True)
    eng = _engine(spec)
    episode = -1
    for t in range(len(g['kind'])):
        present = g['obs_present'][t]
        if g['kind'][t] == 0:
            episode += 1
            if spec.layout_generator is not None:
                from abmarl_b200.layouts import layouts_for
                eng.set_layout(layouts_for(spec, [0], [episode]))
            eng.reset()
        else:
            eng.step(torch.from_numpy(g['actions'][t][None].copy()).cuda())
            np.testing.assert_array_equal(eng.done.cpu().numpy()[0], g['done'][t], err_msg=f'{name} call {t} done')
            np.testing.assert_allclose(eng.reward.cpu().numpy()[0], g['reward'][t], rtol=0, atol=1e-6)
            assert int(eng.all_done.cpu().numpy()[0] & K.ENV_ALL_DONE) == int(g['all_done'][t])
        np.testing.assert_array_equal(eng.obs.cpu().numpy()[0][present], g['obs'][t][present], err_msg=f'{name} call {t} obs')
        st = eng.state_numpy()
        for k in ('flags', 'cell', 'health', 'ammo'):
            np.testing.assert_array_equal(st[k][0], g[k][t], err_msg=f'{name} call {t} {k}')
        in_grid = (g['flags'][t] & K.ST_IN_GRID) != 0
        np.testing.assert_array_equal(st['next'][0][in_grid], g['next'][t][in_grid], err_msg=f'{name} call {t} next')
    # (2) against the oracle with the program
    E, steps, horizon = CASES[name]
    base, spec = P.specs(name, n_envs=E, env_offset=7, seed=0xC0FFEE, horizon=horizon, auto_reset=True)
    eng = _engine(spec)
    n = run_lockstep(eng, _oracle(spec), steps, label=f'program/{name}')
    assert n > 0 and int(eng.stats()[K.STAT_AGENT_STEPS].item()) == n
    # (3) against the built-in program on the engine (its own kernel: the specialised team-battle one where it qualifies)
    a, b = _engine(base), _engine(spec)
    for e in (a, b):
        if spec.layout_generator is not None and not e.device_layouts:
            from abmarl_b200.layouts import LayoutFeeder
            e.feeder = LayoutFeeder(spec)
            e.set_layout(e.feeder.prime(e.state_numpy()['episode']))
        e.reset()
    for t in range(steps):
        for e in (a, b):
            e.step_sampled()
            if getattr(e, 'feeder', None) is not None and e.feeder.after_step(e.all_done.cpu().numpy(), e.state_numpy()['episode']):
                e.set_layout(e.feeder.rows)
        for k in ('obs', 'reward', 'done', 'all_done'):     # (the specialised kernel leaves the action rows of done learners alone)
            assert torch.equal(getattr(a, k), getattr(b, k)), f'{name} step {t}: {k} differs from the built-in program'
        sa, sb = a.state_numpy(), b.state_numpy()
        assert_state_equal(sa, sb, f'{name} step {t} (built-in vs program)')


# ---- ForagingSim -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('manager,shuffled', [('all_step', False), ('turn_based', False), ('all_step', True)])
def test_foraging_engine_matches_oracle(manager, shuffled):
    spec = compile_sim(ForagingSim.build(), manager=manager, n_envs=128, env_offset=11, seed=2024, horizon=40, auto_reset=True,
                       randomize_action_input=shuffled)
    eng, ora = _engine(spec), _oracle(spec)
    n = run_lockstep(eng, ora, 300, label=f'foraging/{manager}/{shuffled}')
    assert n > 0
    st = ora.state
    assert not st['error'].any() and st['stats'][:, K.STAT_EPISODES].sum() > 0
    # bgw_observe = the oracle's observer on the state the run ended in
    got = eng.observe(out=torch.full_like(eng.obs, 99)).cpu().numpy()
    np.testing.assert_array_equal(got, np.stack([ora.observe(e) for e in range(eng.E)]))


def test_foraging_rollout_equals_separate_steps():
    spec = compile_sim(ForagingSim.build(), n_envs=128, seed=5, horizon=30, auto_reset=True)
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


def test_foraging_two_halves_equal_one_handle():
    spec = compile_sim(ForagingSim.build(), n_envs=128, env_offset=64, seed=8, horizon=25, auto_reset=True)
    whole = _engine(spec)
    halves = [_engine(spec.with_envs(64, 64 + 64 * k)) for k in range(2)]
    for e in [whole] + halves:
        e.reset()
    for t in range(80):
        for e in [whole] + halves:
            e.step_sampled()
        for k in ('obs', 'reward', 'done', 'all_done'):
            assert torch.equal(getattr(whole, k), torch.cat([getattr(h, k) for h in halves])), f'step {t}: {k}'
    st = whole.state_numpy()
    for k in ('cell', 'flags', 'health', 'reward_acc', 'step', 'episode'):
        np.testing.assert_array_equal(st[k], np.concatenate([h.state_numpy()[k] for h in halves]), err_msg=k)


def test_foraging_through_the_all_step_manager():
    from abmarl_b200.managers import AllStepManager
    sim = ForagingSim.build(rows=8, cols=8, n_foragers=3, n_predators=1, n_resources=4)
    mgr = AllStepManager(sim, n_envs=32, seed=3, horizon=20, auto_reset=True, device='cuda:0')
    mgr.reset()
    for _ in range(30):
        mgr.step(mgr.engine.sample_actions())
    obs, reward, done = mgr.as_dicts(0)[:3]
    assert set(obs) <= {'forager0', 'forager1', 'forager2', 'predator0'}
    assert all(isinstance(r, float) for r in reward.values())
    assert '__all__' in done


# ---- the C-ABI -------------------------------------------------------------------------------------------------------------
def _raw_handle(spec):
    lib = K.load()
    c = spec.c_struct()
    h = C.c_void_p()
    K.check(lib.bgw_create(C.byref(c), 0, C.byref(h)), lib)
    return lib, h, c


def test_step_before_set_program_fails_and_writes_nothing():
    spec = compile_sim(ForagingSim.build(), n_envs=8, seed=1, auto_reset=True)
    bare = copy.copy(spec)
    bare.program_source = None                        # the engine then leaves the BGW_PROG_USER handle without a program
    eng = _engine(bare)
    eng.obs.fill_(7)
    eng.reward.fill_(3.0)
    eng.done.fill_(5)
    eng.all_done.fill_(9)
    before = {k: v.clone() for k, v in eng.state.items() if v is not None}
    n0 = eng.launches
    for call in (lambda: eng.step(eng.actions), eng.step_sampled, lambda: eng.rollout_sampled(3)):
        with pytest.raises(RuntimeError, match='bgw_set_program'):
            call()
    torch.cuda.synchronize()
    assert eng.launches == n0
    assert (eng.obs == 7).all() and (eng.reward == 3.0).all() and (eng.done == 5).all() and (eng.all_done == 9).all()
    assert (eng.actions == 0).all()
    for k, v in before.items():
        assert torch.equal(eng.state[k], v), k
    # the program-independent entry points work before it, and bgw_specialize has nothing to do on a program handle
    eng.reset()
    eng.observe()
    eng.sample_actions()
    eng.specialize()
    K.check(eng.lib.bgw_set_program(eng._h, spec.program_source.encode(), None), eng.lib)
    ora = _oracle(spec)
    ora.reset()
    for t in range(20):
        eng.step(eng.sample_actions())
        ora.step(ora.sample_actions())
        assert_outputs_equal(eng, ora, f'late program, step {t}')


def test_set_program_errors():
    spec = compile_sim(ForagingSim.build(), n_envs=4, seed=1)
    lib, h, _ = _raw_handle(spec)
    try:
        rc = lib.bgw_set_program(h, b'BGWP_FN void bgwp_step(bgwp_ctx *c) { bgwp_move(c, 0) }', None)   # missing ';'
        msg = lib.bgw_last_error().decode()
        assert rc != 0 and 'nvrtcCompileProgram' in msg and 'program(1)' in msg and 'error' in msg, msg
        K.check(lib.bgw_set_program(h, spec.program_source.encode(), None), lib)
        assert lib.bgw_set_program(h, spec.program_source.encode(), None) != 0
        assert b'already' in lib.bgw_last_error()
    finally:
        lib.bgw_destroy(h)
    builtin = compile_sim(ForagingSim.build(), n_envs=4, seed=1)
    builtin.program, builtin.program_source = K.PROG_TEAM_BATTLE, None
    lib, h, _ = _raw_handle(builtin)
    try:
        assert lib.bgw_set_program(h, spec.program_source.encode(), None) != 0
        assert b'BGW_PROG_USER' in lib.bgw_last_error()
    finally:
        lib.bgw_destroy(h)


def test_set_program_uses_the_cache(tmp_path, monkeypatch):
    """A second handle of the same spec and program loads the cached cubin (no new file) and gives identical results."""
    monkeypatch.setenv('BGW_JIT_CACHE', str(tmp_path))
    spec = compile_sim(ForagingSim.build(), n_envs=64, seed=4, horizon=20, auto_reset=True)
    a = _engine(spec)
    files = sorted(os.listdir(tmp_path))
    assert len(files) == 1 and files[0].endswith('.cubin')
    mtime = os.path.getmtime(tmp_path / files[0])
    b = _engine(spec)
    assert sorted(os.listdir(tmp_path)) == files and os.path.getmtime(tmp_path / files[0]) == mtime
    for e in (a, b):
        e.reset()
        e.rollout_sampled(50)
    for k in ('obs', 'reward', 'done', 'all_done', 'actions'):
        assert torch.equal(getattr(a, k), getattr(b, k)), k
    other = DeviceProgram(spec.program_source + '\n/* another program */')
    sim = ForagingSim.build()
    sim.device_program = lambda: other
    _engine(compile_sim(sim, n_envs=64, seed=4, horizon=20, auto_reset=True))
    assert len(os.listdir(tmp_path)) == 2                        # the program is part of the key
