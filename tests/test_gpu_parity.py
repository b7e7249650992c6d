"""GPU parity: the CUDA engine, called through the C-ABI (libbgw.so), against the CPU oracle on the same
seeded inputs -- bit-exact observations, dones, __all__, positions, cell-list order, flags, float64 health,
float32 rewards (both sides round the same float64 sum), episode statistics."""
import os

import numpy as np
import pytest
import torch

from abmarl_b200 import _capi as K
from abmarl_b200.spec import compile_sim
from tests import scenarios
from tests.helpers import run_lockstep, assert_outputs_equal, assert_state_equal

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def _pair(spec):
    from abmarl_b200.engine import BatchedGridWorld
    from oracle.oracle import OracleEnv
    return BatchedGridWorld(spec, device='cuda:0'), OracleEnv(spec)


CASES = [
    # scenario, envs, steps, horizon
    ('tb_c2', 64, 120, 50),
    ('tb_c5_small', 24, 90, 40),
    ('tb_dense', 64, 120, 30),
    ('tb_blocking', 48, 100, 40),
    ('tb_stacked', 48, 80, 30),
    ('tb_noself', 48, 80, 30),
    ('tb_shuffled', 48, 120, 25),            # keyed random.shuffle: placement order + action input order
    ('tb_c5_shuffled', 24, 90, 30),          # the same on the specialised kernel's shape
    ('tb_position', 48, 90, 30),             # AbsolutePositionObserver slot of the obs row
    ('tb_encoding', 48, 100, 30),
    ('tb_encoding_stacked', 48, 100, 30),
    ('tb_restricted', 48, 100, 30),
    ('tb_restricted_stacked', 48, 100, 30),
    ('tb_selective', 48, 100, 30),
    ('tb_selective_stacked', 48, 100, 30),
    ('tb_ammo', 48, 100, 30),
    ('tb_ammo_selective', 48, 100, 30),
    ('reach_target', 64, 150, 40),
    ('reach_target_crowd', 64, 150, 40),
    ('traffic', 64, 200, 50),
    ('maze_c1', 32, 150, 60),
    ('pacman_c3', 6, 40, 25),
    ('pacman_simple', 8, 120, 60),
    ('mm_c4', 12, 150, 60),
    ('mm_random', 12, 120, 50),
    ('mm_allstep', 12, 100, 40),
    ('mm_tbf', 16, 200, 30),
    ('mm_tbf_scatter', 16, 200, 30),
    ('mm_tiny', 16, 300, 0),
    ('mm_tiny_allstep', 16, 200, 0),
    ('mm_dynamic', 16, 300, 0),              # DynamicOrderManager: the sim names the next agent(s)
]


@pytest.mark.parametrize('name,n_envs,steps,horizon', CASES)
def test_engine_matches_oracle(mirror, name, n_envs, steps, horizon):
    builder, manager, _ = scenarios.SCENARIOS[name]
    spec = compile_sim(builder(mirror), manager=manager, n_envs=n_envs, env_offset=7, seed=0xC0FFEE,
                       horizon=horizon, auto_reset=True)
    eng, ora = _pair(spec)
    n = run_lockstep(eng, ora, steps, label=name)
    assert n > 0
    assert int(eng.stats()[K.STAT_AGENT_STEPS].item()) == n


OBSERVE_CASES = ['tb_c2', 'tb_c5', 'tb_c5_small', 'tb_dense', 'tb_blocking', 'tb_stacked', 'tb_noself', 'tb_position', 'tb_ammo',
                 'tb_encoding_stacked', 'reach_target_crowd', 'traffic', 'maze_c1', 'pacman_c3', 'mm_c4', 'mm_dynamic']


@pytest.mark.parametrize('generic', ['0', '1'])
@pytest.mark.parametrize('name', OBSERVE_CASES)
def test_observe_equals_get_obs_of_every_learner(mirror, name, generic, monkeypatch):
    """bgw_observe = sim.get_obs(agent_id) for every learner on the state as it stands (smart.py:93-99), against the oracle's
    observer on the same state: after a reset, mid-episode (dead and already-reported learners included) and after
    auto-resets; it writes no state, repeats the rows the last step reported, and honours the env mask.  generic=1 forces
    the general kernel's observer where the gather-only kernel would run."""
    if generic == '1':
        if name not in ('tb_c2', 'tb_c5', 'tb_c5_small', 'tb_dense'):
            pytest.skip('the general observer runs anyway')
        monkeypatch.setenv('BGW_GENERIC_OBSERVE', '1')
    builder, manager, _ = scenarios.SCENARIOS[name] if name != 'tb_c5' else (scenarios.build_tb_c5, 'all_step', None)
    E = 6 if name in ('tb_c5', 'pacman_c3') else 20
    spec = compile_sim(builder(mirror), manager=manager, n_envs=E, env_offset=3, seed=0x0B5, horizon=25, auto_reset=True)
    eng, ora = _pair(spec)
    for steps in (0, 9, 40):
        run_lockstep(eng, ora, steps, label=f'{name}/observe')
        before = eng.state_numpy()
        reported = eng.obs.cpu().numpy().copy()
        out = torch.full_like(eng.obs, 99)
        assert eng.observe(out=out) is out
        got = out.cpu().numpy()
        want = np.stack([ora.observe(e) for e in range(E)])
        bad = np.argwhere(got != want)
        assert bad.size == 0, f'{name} after {steps} steps: observe differs at {bad[:5].tolist()}'
        assert_state_equal(eng.state_numpy(), before, f'{name}: observe wrote state')
        fresh = np.ones(E, dtype=bool) if steps == 0 else (ora.all_done & K.ENV_RESET) != 0
        rows = np.zeros((E, eng.L), dtype=bool) if steps == 0 else (ora.done & K.OUT_VALID) != 0
        if spec.manager == K.MANAGER_ALL_STEP:
            rows |= fresh[:, None]                                          # a reset reports every learner
        else:
            rows[fresh, before['turn'][fresh]] = True                       # a turn-based reset reports the learner whose turn it is
        assert np.array_equal(got[rows], reported[rows]), f'{name}: observe does not repeat the reported rows'
        mask = (np.arange(E) % 3 == 0).astype(np.uint8)
        out2 = torch.full_like(eng.obs, 99)
        eng.observe(env_mask=mask, out=out2)
        got2 = out2.cpu().numpy()
        assert np.array_equal(got2[mask != 0], want[mask != 0]) and (got2[mask == 0] == 99).all()


@pytest.mark.parametrize('name', ['tb_blocking', 'tb_encoding_stacked', 'tb_ammo_selective', 'reach_target_crowd', 'traffic',
                                  'maze_c1', 'pacman_c3', 'mm_c4', 'mm_dynamic'])
def test_specialized_kernel_matches_oracle(mirror, name, tmp_path):
    """bgw_specialize: the general step kernel compiled at run time for the spec alone (NVRTC; the spec's scalars as
    compile-time constants) gives the oracle's results like the stock instantiation; a second handle takes the cubin
    from the cache directory."""
    builder, manager, _ = scenarios.SCENARIOS[name]
    E = 6 if name == 'pacman_c3' else 24
    spec = compile_sim(builder(mirror), manager=manager, n_envs=E, env_offset=2, seed=0x51EC, horizon=30, auto_reset=True)
    eng, ora = _pair(spec)
    launches = eng.launches
    eng.specialize(cache_dir=str(tmp_path))
    cached = sorted(os.listdir(tmp_path))
    assert len(cached) == 1 and cached[0].startswith('bgw_jit_') and cached[0].endswith('.cubin')
    n = run_lockstep(eng, ora, 70, label=name + '/specialized')
    assert n > 0 and eng.launches > launches
    if name in ('tb_blocking', 'mm_c4'):
        eng2, ora2 = _pair(spec)
        stamp = os.path.getmtime(os.path.join(tmp_path, cached[0]))
        eng2.specialize(cache_dir=str(tmp_path))
        assert sorted(os.listdir(tmp_path)) == cached and os.path.getmtime(os.path.join(tmp_path, cached[0])) == stamp
        run_lockstep(eng2, ora2, 30, label=name + '/specialized from the cache')


@pytest.mark.parametrize('name', ['tb_c5_small', 'tb_dense', 'tb_noself', 'tb_shuffled', 'tb_c5_shuffled'])
def test_specialized_team_battle_shape_matches_oracle(mirror, name, tmp_path):
    """bgw_specialize on a sim of the specialised team-battle kernel whose shape is not one of the two the library ships: the
    kernel body compiled at run time with THIS spec's shape as its compile-time shape (mixed cells, accuracy < 1,
    non-uniform ranges, keyed placement order included), against the oracle through resets, rollouts and chained launches."""
    builder, manager, _ = scenarios.SCENARIOS[name]
    spec = compile_sim(builder(mirror), manager=manager, n_envs=40, env_offset=5, seed=0x51ED, horizon=25, auto_reset=True)
    eng, ora = _pair(spec)
    eng.specialize(cache_dir=str(tmp_path))
    assert len(os.listdir(tmp_path)) == 1
    run_lockstep(eng, ora, 80, label=name + '/specialized shape')
    eng.rollout_sampled(37)
    for _ in range(37):
        ora.step(ora.sample_actions())
    assert_outputs_equal(eng, ora, name + '/specialized shape, rollout')
    assert_state_equal(eng.state_numpy(), ora.state, name + '/specialized shape, rollout')


@pytest.mark.parametrize('name,n_envs,kernel', [('tb_c5_shuffled', 1000, 'stock'), ('tb_c5_shuffled', 1000, 'specialized'),
                                                ('tb_c5_256_shuffled', 300, 'stock'), ('tb_c5_shuffled', 1000, 'general')])
def test_shuffled_placement_over_thousands_of_resets(mirror, name, n_envs, kernel, tmp_path, monkeypatch):
    """PositionState(randomize_placement_order): sim_reset draws the keyed placement order into the storage of the reward
    accumulators, and a thread that zeroed its accumulator after another thread had drawn there (no barrier between the
    two) reordered the placement, so the first observations and cells of an occasional episode differed from the
    reference's.  Horizon 1: every second call resets every env -- bgw_reset, auto-resets in the step kernel (one CTA of
    three warps per env), in chained rollouts and in the general kernel -- and each is compared with the oracle."""
    if kernel == 'general':
        monkeypatch.setenv('BGW_GENERIC_KERNEL', '1')
    if name == 'tb_c5_256_shuffled':          # the headline shape, two warps in bgw_reset's kernel
        spec = compile_sim(scenarios.build_tb_c5(mirror), n_envs=n_envs, env_offset=5, seed=0x5EED, horizon=1, auto_reset=True)
        spec.randomize_placement_order = 1
    else:
        builder, manager, _ = scenarios.SCENARIOS[name]
        spec = compile_sim(builder(mirror), manager=manager, n_envs=n_envs, env_offset=5, seed=0x5EED, horizon=1, auto_reset=True)
    eng, ora = _pair(spec)
    if kernel == 'specialized':
        eng.specialize(cache_dir=str(tmp_path))
    run_lockstep(eng, ora, 8, label=f'{name}/{kernel} shuffled resets')
    eng.rollout_sampled(11)
    for _ in range(11):
        ora.step(ora.sample_actions())
    assert_outputs_equal(eng, ora, f'{name}/{kernel} shuffled resets, rollout')
    assert_state_equal(eng.state_numpy(), ora.state, f'{name}/{kernel} shuffled resets, rollout')
    assert (ora.state['episode'] >= 9).all()


def test_specialize_recompiles_over_a_damaged_cache_entry(mirror, tmp_path):
    """A cache file that does not load (truncated, or from another build) is replaced by a fresh compilation."""
    builder, manager, _ = scenarios.SCENARIOS['traffic']
    spec = compile_sim(builder(mirror), manager=manager, n_envs=8, seed=5, horizon=20, auto_reset=True)
    eng, ora = _pair(spec)
    eng.specialize(cache_dir=str(tmp_path))
    (name,) = os.listdir(tmp_path)
    good = os.path.getsize(os.path.join(tmp_path, name))
    with open(os.path.join(tmp_path, name), 'wb') as fh:
        fh.write(b'not a cubin')
    eng2, ora2 = _pair(spec)
    eng2.specialize(cache_dir=str(tmp_path))
    assert os.path.getsize(os.path.join(tmp_path, name)) == good
    run_lockstep(eng2, ora2, 30, label='traffic/specialized after a damaged cache entry')


def test_specialize_leaves_the_shipped_shapes_alone(mirror, tmp_path):
    spec = compile_sim(scenarios.SCENARIOS['tb_c2'][0](mirror), n_envs=16, seed=3, horizon=30, auto_reset=True)
    eng, ora = _pair(spec)
    eng.specialize(cache_dir=str(tmp_path))
    assert os.listdir(tmp_path) == []
    run_lockstep(eng, ora, 40, label='tb_c2 after specialize')


@pytest.mark.parametrize('name', ['tb_c2', 'tb_c5_small', 'tb_dense', 'tb_noself'])
def test_general_kernel_on_fast_path_scenarios(mirror, name, monkeypatch):
    """Scenarios that qualify for the specialised team-battle kernel must give the same results through the
    general kernel (BGW_GENERIC_KERNEL=1), i.e. both equal the oracle."""
    builder, manager, _ = scenarios.SCENARIOS[name]
    spec = compile_sim(builder(mirror), manager=manager, n_envs=32, seed=21, horizon=40, auto_reset=True)
    monkeypatch.setenv('BGW_GENERIC_KERNEL', '1')
    eng, ora = _pair(spec)
    run_lockstep(eng, ora, 60, label=name + '/general')


@pytest.mark.parametrize('threads', ['32', '64', '96', '256'])
def test_thread_count_does_not_change_results(mirror, threads, monkeypatch):
    spec = compile_sim(scenarios.build_tb_c5_small(mirror), n_envs=16, seed=9, horizon=30, auto_reset=True)
    monkeypatch.setenv('BGW_THREADS', threads)
    eng, ora = _pair(spec)
    run_lockstep(eng, ora, 45, label='tb_c5_small/T' + threads)


@pytest.mark.parametrize('name', ['tb_c2', 'tb_dense', 'tb_blocking', 'tb_restricted_stacked', 'tb_ammo_selective', 'reach_target_crowd', 'traffic'])
def test_serial_and_reservation_actor_paths_agree(mirror, name, monkeypatch):
    """The rank-order loop (one thread) and the reservation rounds must both equal the oracle."""
    builder, manager, _ = scenarios.SCENARIOS[name]
    spec = compile_sim(builder(mirror), manager=manager, n_envs=32, seed=11, horizon=40, auto_reset=True)
    monkeypatch.setenv('BGW_SERIAL_ACTORS', '1')
    monkeypatch.setenv('BGW_GENERIC_KERNEL', '1')
    eng, ora = _pair(spec)
    run_lockstep(eng, ora, 60, label=name + '/serial')


def test_aliased_reservation_slots(mirror, monkeypatch):
    """Few reservation slots (many cells share one) only add rounds; results stay identical."""
    spec = compile_sim(scenarios.build_tb_c5_small(mirror), n_envs=16, seed=5, horizon=30, auto_reset=True)
    monkeypatch.setenv('BGW_SLOTS', '32')
    eng, ora = _pair(spec)
    run_lockstep(eng, ora, 45, label='tb_c5_small/slots32')


def test_reservation_epochs_run_out(mirror, monkeypatch):
    """The ordered rounds tag reservations with a decreasing epoch; a launch that starts with almost none left refills
    the slot tables and starts over (never reached in practice: a launch has about a million epochs)."""
    spec = compile_sim(scenarios.build_tb_c5_small(mirror), n_envs=400, seed=5, horizon=30, auto_reset=True)
    monkeypatch.setenv('BGW_EPOCH0', '4100')
    monkeypatch.setenv('BGW_GRID', '3')                     # three persistent CTAs: many envs, hence many rounds, per CTA
    eng, ora = _pair(spec)
    run_lockstep(eng, ora, 12, label='tb_c5_small/epochs')


def test_randomized_action_order(mirror):
    """AllStepManager(randomize_action_input=True): a per-env processing order (all_step_manager.py:62-65)."""
    spec = compile_sim(scenarios.build_tb_dense(mirror), n_envs=32, seed=3, horizon=30, auto_reset=True)
    eng, ora = _pair(spec)
    rng = np.random.default_rng(0)

    def order(t):
        return np.stack([rng.permutation(eng.L) for _ in range(eng.E)]).astype(np.int16)
    run_lockstep(eng, ora, 60, order_fn=order, label='tb_dense/order')


@pytest.mark.parametrize('name', list(scenarios.SCENARIOS))
def test_engine_reproduces_reference_transcript(mirror, name):
    """Replay the actions recorded from the UNMODIFIED reference (tests/golden/*.npz) through the engine."""
    g = np.load(os.path.join(GOLDEN, name + '.npz'))
    builder, manager, _ = scenarios.SCENARIOS[name]
    spec = compile_sim(builder(mirror), manager=manager, n_envs=1, seed=int(g['seed']), auto_reset=False)
    from abmarl_b200.engine import BatchedGridWorld
    eng = BatchedGridWorld(spec, device='cuda:0')
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
            act = torch.from_numpy(g['actions'][t][None].copy()).cuda()
            eng.step(act)
            np.testing.assert_array_equal(eng.done.cpu().numpy()[0], g['done'][t], err_msg=f'{name} call {t} done')
            np.testing.assert_allclose(eng.reward.cpu().numpy()[0], g['reward'][t], rtol=0, atol=1e-6)
            assert int(eng.all_done.cpu().numpy()[0] & K.ENV_ALL_DONE) == int(g['all_done'][t])
        np.testing.assert_array_equal(eng.obs.cpu().numpy()[0][present], g['obs'][t][present], err_msg=f'{name} call {t} obs')
        st = eng.state_numpy()
        np.testing.assert_array_equal(st['flags'][0], g['flags'][t], err_msg=f'{name} call {t} flags')
        np.testing.assert_array_equal(st['cell'][0], g['cell'][t], err_msg=f'{name} call {t} cell')
        np.testing.assert_array_equal(st['health'][0], g['health'][t], err_msg=f'{name} call {t} health')
        np.testing.assert_array_equal(st['ammo'][0], g['ammo'][t], err_msg=f'{name} call {t} ammo')
        in_grid = (g['flags'][t] & K.ST_IN_GRID) != 0
        np.testing.assert_array_equal(st['next'][0][in_grid], g['next'][t][in_grid], err_msg=f'{name} call {t} next')


@pytest.mark.parametrize('name', ['mm_c4', 'mm_random', 'mm_tbf', 'mm_tbf_scatter'])
def test_device_maze_layouts(mirror, name):
    """bgw_generate_layouts (MazePlacementState on the device, one thread per env) against the Python restatement that
    the golden transcripts pin to the reference; then whole episodes with auto-reset run without any host layout."""
    from abmarl_b200.engine import BatchedGridWorld
    from abmarl_b200.layouts import layouts_for
    builder, manager, _ = scenarios.SCENARIOS[name]
    E = 96
    spec = compile_sim(builder(mirror), manager=manager, n_envs=E, env_offset=1000, seed=77, horizon=15, auto_reset=True)
    eng = BatchedGridWorld(spec, device='cuda:0')
    assert eng.device_layouts and eng.dims.device_layouts == 1
    eng.reset()
    np.testing.assert_array_equal(eng.state_numpy()['layout'].view(np.uint16), layouts_for(spec, range(E), [0] * E))
    seen = 0
    for t in range(40):
        eng.step_sampled()
        flags = eng.all_done.cpu().numpy()
        done = np.flatnonzero(flags & K.ENV_ALL_DONE)
        if len(done):                                          # their next layouts are already on the device
            ep = eng.state_numpy()['episode']
            want = layouts_for(spec, done, [int(ep[e]) + 1 for e in done])
            np.testing.assert_array_equal(eng.state_numpy()['layout'].view(np.uint16)[done], want)
            seen += len(done)
    assert seen > E and (eng.state_numpy()['error'] == 0).all()


def test_rng_draw_and_los_mask_exports():
    import ctypes as C
    from abmarl_b200 import philox
    from oracle.oracle import los_mask
    lib = K.load()
    out = (C.c_uint32 * 4)()
    for key in [(0xB200, 0, 0, 0, 0, 0, 0), (2**63 + 5, 4095, 17, 199, 5, 255, 4000), (1, 2, 3, 4, 6, 7, 8)]:
        assert lib.bgw_rng_draw(*key, C.byref(out)) == 0
        assert tuple(out) == philox.draw4(*key)
    for R in (1, 2, 5, 16):
        n = 2 * R + 1
        buf = np.empty((n, n), dtype=np.uint8)
        for rd in range(-R, R + 1):
            for cd in range(-R, R + 1):
                assert lib.bgw_los_mask(R, rd, cd, buf.ctypes.data_as(C.c_void_p)) == 0
                assert np.array_equal(buf, los_mask(R, rd, cd)), (R, rd, cd)


def test_full_size_c5_properties(mirror):
    """BASELINE config 5 at full size (64x64, 256 agents, view 5, 4096 envs): oracle parity on a slice of envs
    plus size-independent invariants over the whole batch."""
    E = 4096
    spec = compile_sim(scenarios.build_tb_c5(mirror), n_envs=E, seed=0xB200, horizon=200, auto_reset=True)
    from abmarl_b200.engine import BatchedGridWorld
    from oracle.oracle import OracleEnv
    eng = BatchedGridWorld(spec, device='cuda:0')
    ora = OracleEnv(spec.with_envs(8, 0))                 # Philox is keyed by the global env index
    eng.reset()
    ora.reset()
    total = 0
    for t in range(30):
        act = eng.sample_actions()
        ora_act = ora.sample_actions()
        assert np.array_equal(act[:8].cpu().numpy(), ora_act)
        eng.step(act)
        ora.step(ora_act)
        assert np.array_equal(eng.obs[:8].cpu().numpy(), ora.obs), f'step {t}'
        assert np.array_equal(eng.done[:8].cpu().numpy(), ora.done)
        assert np.array_equal(eng.reward[:8].cpu().numpy(), ora.reward)
        done = eng.done.cpu().numpy()
        total += int(((done & K.OUT_VALID) != 0).sum())
    st = eng.state_numpy()
    flags, cell, health = st['flags'], st['cell'], st['health']
    active, in_grid = (flags & K.ST_ACTIVE) != 0, (flags & K.ST_IN_GRID) != 0
    assert np.array_equal(active, health > 0)                          # agent.py:192-196
    assert np.array_equal(active, in_grid)                             # dead entities leave the grid (actor.py:357-358)
    assert (cell < 64 * 64).all()
    # cells hold one team only (overlapping = {k: {k}}): no two active agents of different encodings share a cell
    enc = np.asarray(spec.encoding)
    for e in range(0, E, 257):
        cells = {}
        for a in np.nonzero(in_grid[e])[0]:
            assert cells.setdefault(int(cell[e, a]), int(enc[a])) == int(enc[a])
    assert int(eng.stats()[K.STAT_AGENT_STEPS].item()) == total
    obs = eng.obs_view().cpu().numpy()
    valid = (eng.done.cpu().numpy() & K.OUT_VALID) != 0
    assert obs.min() >= -1 and obs.max() <= 4                          # no blockers => never -2
    own = obs[..., 5, 5][valid & (eng.done.cpu().numpy() & K.OUT_DONE == 0)]
    assert (own >= 1).all()                                            # a live agent sees its own team on its cell


@pytest.mark.parametrize('name,steps', [('tb_c2', 60), ('pacman_c3', 12)])
def test_full_size_16k_envs(mirror, name, steps):
    """BASELINE configs 2 and 3 at their full batch (16384 envs per GPU): oracle parity on the first and the last envs
    of the batch (the Philox key is the global env index) plus invariants over all envs."""
    E, S = 16384, 6
    builder, manager, _ = scenarios.SCENARIOS[name]
    spec = compile_sim(builder(mirror), manager=manager, n_envs=E, seed=0xB200, horizon=40, auto_reset=True)
    from abmarl_b200.engine import BatchedGridWorld
    from oracle.oracle import OracleEnv
    eng = BatchedGridWorld(spec, device='cuda:0')
    head, tail = OracleEnv(spec.with_envs(S, 0)), OracleEnv(spec.with_envs(S, E - S))
    eng.reset()
    for o in (head, tail):
        o.reset()
    assert np.array_equal(eng.obs[:S].cpu().numpy(), head.obs) and np.array_equal(eng.obs[E - S:].cpu().numpy(), tail.obs)
    total = 0
    for t in range(steps):
        act = eng.sample_actions()
        eng.step(act)
        for o, sl in ((head, slice(0, S)), (tail, slice(E - S, E))):
            a = o.sample_actions()
            assert np.array_equal(act[sl].cpu().numpy(), a)
            o.step(a)
            assert np.array_equal(eng.obs[sl].cpu().numpy(), o.obs), f'{name} step {t}'
            assert np.array_equal(eng.done[sl].cpu().numpy(), o.done)
            assert np.array_equal(eng.reward[sl].cpu().numpy(), o.reward)
            assert np.array_equal(eng.all_done[sl].cpu().numpy(), o.all_done)
        total += int(((eng.done.cpu().numpy() & K.OUT_VALID) != 0).sum())
    st = eng.state_numpy()
    assert_state_equal({k: (None if v is None else v[:S]) for k, v in st.items()}, head.state, f'{name} head')
    assert_state_equal({k: (None if v is None else v[E - S:]) for k, v in st.items()}, tail.state, f'{name} tail')
    assert int(eng.stats()[K.STAT_AGENT_STEPS].item()) == total
    assert (st['error'] == 0).all() and (st['cell'][(st['flags'] & K.ST_IN_GRID) != 0] < spec.rows * spec.cols).all()
    health_agents = (np.asarray(spec.klass) & K.AG_HEALTH) != 0
    active = (st['flags'] & K.ST_ACTIVE) != 0
    assert np.array_equal(active[:, health_agents], st['health'][:, health_agents] > 0)      # agent.py:192-196


@pytest.mark.parametrize('zero_copy', [True, False])
def test_step_host_returns_exactly_the_valid_rows(mirror, zero_copy):
    """bgw_gather_valid / BatchedGridWorld.step_host: the compacted host buffers hold the rows with BGW_OUT_VALID
    (and every row of an env that was auto-reset), identical to the dense device outputs."""
    spec = compile_sim(scenarios.build_tb_dense(mirror), n_envs=48, seed=13, horizon=12, auto_reset=True)
    from abmarl_b200.engine import BatchedGridWorld
    eng = BatchedGridWorld(spec, device='cuda:0')
    eng.reset()
    seen_reset = False
    for t in range(40):
        act = eng.sample_actions().cpu().pin_memory()
        n, index, obs_c, rew_c, done_c, all_done = eng.step_host(act, zero_copy=zero_copy)
        dense_obs, dense_rew = eng.obs.cpu().numpy().reshape(-1, eng.dims.obs_stride), eng.reward.cpu().numpy().ravel()
        dense_done, flags = eng.done.cpu().numpy().ravel(), eng.all_done.cpu().numpy()
        want = ((dense_done & K.OUT_VALID) != 0).reshape(eng.E, eng.L) | ((flags & K.ENV_RESET) != 0)[:, None]
        idx = index.numpy()
        assert n == int(want.sum()) and sorted(idx.tolist()) == np.flatnonzero(want.ravel()).tolist()
        np.testing.assert_array_equal(obs_c.numpy(), dense_obs[idx])
        np.testing.assert_array_equal(rew_c.numpy(), dense_rew[idx])
        np.testing.assert_array_equal(done_c.numpy(), dense_done[idx])
        np.testing.assert_array_equal(all_done.numpy(), flags)
        seen_reset |= bool((flags & K.ENV_RESET).any())
    assert seen_reset


def test_host_pipeline_equals_one_batch(mirror):
    """HostPipeline (K sub-batches on their own streams, send / recv) returns, sub-batch by sub-batch, the rows one
    BatchedGridWorld over all the envs returns for the same actions: the Philox key is the global env index."""
    from abmarl_b200.engine import BatchedGridWorld, HostPipeline
    spec = compile_sim(scenarios.build_tb_dense(mirror), n_envs=48, env_offset=5, seed=13, horizon=12, auto_reset=True)
    eng = BatchedGridWorld(spec, device='cuda:0')
    pipe = HostPipeline(spec, shards=3, device='cuda:0')
    eng.reset()
    pipe.reset()
    Ek, L = pipe.Ek, pipe.L
    act = eng.sample_actions().cpu().pin_memory()
    for k in range(pipe.K):
        pipe.send(k, act[k * Ek:(k + 1) * Ek])
    for t in range(30):
        n, index, obs_c, rew_c, done_c, all_done = eng.step_host(act)
        order = np.argsort(index.numpy(), kind='stable')
        idx, obs_c, rew_c, done_c = index.numpy()[order], obs_c.numpy()[order], rew_c.numpy()[order], done_c.numpy()[order]
        nxt = eng.sample_actions().cpu().pin_memory()
        got = 0
        for k in range(pipe.K):
            nk, ik, ok, rk, dk, ak = pipe.recv(k)
            o = np.argsort(ik.numpy(), kind='stable')
            sel = (idx >= k * Ek * L) & (idx < (k + 1) * Ek * L)
            np.testing.assert_array_equal(ik.numpy()[o] + k * Ek * L, idx[sel])
            np.testing.assert_array_equal(ok.numpy()[o], obs_c[sel])
            np.testing.assert_array_equal(rk.numpy()[o], rew_c[sel])
            np.testing.assert_array_equal(dk.numpy()[o], done_c[sel])
            np.testing.assert_array_equal(ak.numpy(), all_done.numpy()[k * Ek:(k + 1) * Ek])
            got += nk
            pipe.send(k, nxt[k * Ek:(k + 1) * Ek])
        assert got == n
        act = nxt
    eng.step_host(act)                                                  # the step the pipeline still has in flight
    for k in range(pipe.K):
        pipe.recv(k)
    assert int(pipe.stats()[K.STAT_AGENT_STEPS]) == int(eng.stats()[K.STAT_AGENT_STEPS])


@pytest.mark.parametrize('name', ['tb_c2', 'tb_c5_small', 'tb_blocking', 'maze_c1'])
def test_step_sampled_equals_sample_then_step(mirror, name):
    """bgw_step_sampled (fused on the specialised kernel, two launches on the general one) against the oracle's
    sample_actions + step."""
    builder, manager, _ = scenarios.SCENARIOS[name]
    spec = compile_sim(builder(mirror), manager=manager, n_envs=24, env_offset=3, seed=31, horizon=25, auto_reset=True)
    eng, ora = _pair(spec)
    eng.reset()
    ora.reset()
    for t in range(60):
        act = ora.sample_actions()
        before = ora.state['flags'].copy()
        was_done = (ora.state['env_flags'] & K.ENV_ALL_DONE) != 0
        ora.step(act)
        eng.step_sampled()
        assert_outputs_equal(eng, ora, f'{name} step {t}')
        assert_state_equal(eng.state_numpy(), ora.state, f'{name} step {t}')
        acting = np.stack([(before[:, a] & K.ST_DONE_REPORTED) == 0 for a in spec.learner_agents], axis=1) & ~was_done[:, None]
        np.testing.assert_array_equal(eng.actions.cpu().numpy()[acting], act[acting])


@pytest.mark.parametrize('name,n_envs', [('tb_c2', 700), ('tb_c5_small', 24), ('tb_blocking', 24), ('mm_tbf', 16)])
def test_rollout_sampled_equals_separate_steps(mirror, name, n_envs):
    """bgw_rollout_sampled(n) (launches chained per env on the specialised kernel) leaves the state, the statistics, the
    sampled actions and the last step's outputs of n separate bgw_step_sampled calls, which the oracle pins."""
    from abmarl_b200.engine import BatchedGridWorld
    builder, manager, _ = scenarios.SCENARIOS[name]
    spec = compile_sim(builder(mirror), manager=manager, n_envs=n_envs, env_offset=5, seed=77, horizon=25, auto_reset=True)
    a, b = BatchedGridWorld(spec, device='cuda:0'), BatchedGridWorld(spec, device='cuda:0')
    a.reset()
    b.reset()
    for n in (1, 7, 40, 2, 33):
        a.rollout_sampled(n)
        for _ in range(n):
            b.step_sampled()
        for k in ('obs', 'reward', 'done', 'all_done', 'actions'):
            assert torch.equal(getattr(a, k), getattr(b, k)), (name, n, k)
        assert_state_equal(a.state_numpy(), b.state_numpy(), f'{name} rollout {n}')
        assert torch.equal(a.stats(), b.stats())


def test_rollout_keeps_caller_supplied_layouts(mirror):
    """set_layout() switches the device-side layout generator off in the HANDLE too (bgw_use_device_layouts): a rollout
    must not overwrite the caller's layout rows between its steps, i.e. rollout_sampled(n) == n x step_sampled()."""
    from abmarl_b200.engine import BatchedGridWorld
    from abmarl_b200.layouts import layouts_for
    builder, manager, _ = scenarios.SCENARIOS['mm_tbf']
    spec = compile_sim(builder(mirror), manager=manager, n_envs=16, env_offset=3, seed=21, horizon=6, auto_reset=True)
    a, b = BatchedGridWorld(spec, device='cuda:0'), BatchedGridWorld(spec, device='cuda:0')
    assert a.device_layouts, "the scenario must be one the device generator supports"
    rows = layouts_for(spec, list(range(16)), [5] * 16)              # some fixed layout for every episode (episode 5's)
    for eng in (a, b):
        eng.set_layout(rows)
        eng.reset()
    for n in (3, 9, 14):                                             # horizon 6: every env resets inside the rollouts
        a.rollout_sampled(n)
        for _ in range(n):
            b.step_sampled()
        for k in ('obs', 'reward', 'done', 'all_done', 'actions'):
            assert torch.equal(getattr(a, k), getattr(b, k)), (n, k)
        assert_state_equal(a.state_numpy(), b.state_numpy(), f'rollout {n}')
        np.testing.assert_array_equal(a.state['layout'].cpu().numpy().view(np.uint16), np.asarray(rows, dtype=np.uint16))


@pytest.mark.parametrize('name,n_envs', [('tb_c2', 48), ('tb_c5', 6), ('tb_c5_small', 24)])
def test_compile_time_shapes_with_caller_supplied_layouts(mirror, name, n_envs):
    """The compile-time-shape instantiations of the specialised kernel have no layout path in their inlined reset;
    bgw_bind_state moves a handle that is given layouts to the run-time-shape instantiation.  Layout = the cells of a normal
    reset (so every placement is legal), bound before the first reset and used by every auto-reset after it."""
    builder = scenarios.build_tb_c5 if name == 'tb_c5' else scenarios.SCENARIOS[name][0]
    spec = compile_sim(builder(mirror), n_envs=n_envs, env_offset=1, seed=31, horizon=7, auto_reset=True)
    eng, ora = _pair(spec)
    if name == 'tb_c5_small':                 # a shape compiled at run time (bgw_specialize) behaves like the shipped ones
        eng.specialize()
    from oracle.oracle import OracleEnv
    scout = OracleEnv(spec)
    scout.reset()
    layout = scout.state['cell'].copy()
    for x in (eng, ora):
        x.set_layout(layout)
    eng.reset()
    ora.reset()
    assert np.array_equal(eng.obs.cpu().numpy(), ora.obs)
    np.testing.assert_array_equal(eng.state_numpy()['cell'], layout)
    for t in range(20):
        act = ora.sample_actions()
        eng.step(torch.from_numpy(act).cuda())
        ora.step(act)
        assert_outputs_equal(eng, ora, f'{name} layouts step {t}')
        assert_state_equal(eng.state_numpy(), ora.state, f'{name} layouts step {t}')


def test_step_launch_replayed_from_a_cuda_graph(mirror):
    """A step launch captured into a CUDA graph runs with the parameters of capture time at every replay: the library
    must not bake a ticket base or a chain dependency into it.  Replays, eager steps and chained rollouts mixed on one
    engine against separate eager steps on another (2500 envs: more than one env per resident CTA)."""
    from abmarl_b200.engine import BatchedGridWorld
    spec = compile_sim(scenarios.build_tb_c5(mirror), n_envs=2500, seed=5, horizon=15, auto_reset=True)
    a, b = BatchedGridWorld(spec, device='cuda:0'), BatchedGridWorld(spec, device='cuda:0')
    a.reset()
    b.reset()
    a.step_sampled()
    b.step_sampled()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        a.step_sampled()                                   # capture only: nothing runs
    done = 1
    for kind, n in (('graph', 4), ('rollout', 6), ('graph', 3), ('eager', 2), ('rollout', 20), ('graph', 5)):
        for _ in range(n):
            b.step_sampled()
        if kind == 'graph':
            for _ in range(n):
                g.replay()
        elif kind == 'rollout':
            a.rollout_sampled(n)
        else:
            for _ in range(n):
                a.step_sampled()
        done += n
        torch.cuda.synchronize()
        for k in ('obs', 'reward', 'done', 'all_done', 'actions'):
            assert torch.equal(getattr(a, k), getattr(b, k)), (kind, done, k)
        assert_state_equal(a.state_numpy(), b.state_numpy(), f'{kind} after {done} steps')
        assert torch.equal(a.stats(), b.stats())


def test_chained_rollout_full_size_against_oracle(mirror):
    """The headline workload at full size (4096 envs: three envs per resident CTA, tickets, per-env stamps) through
    chained rollouts of several lengths, against the oracle on env slices at both ends of the batch, and against
    serialised launches (one unchained step_sampled per step) over the whole batch."""
    from abmarl_b200.engine import BatchedGridWorld
    from oracle.oracle import OracleEnv
    E, S = 4096, 6
    spec = compile_sim(scenarios.build_tb_c5(mirror), n_envs=E, seed=0xB200, horizon=40, auto_reset=True)
    eng, ser = BatchedGridWorld(spec, device='cuda:0'), BatchedGridWorld(spec, device='cuda:0')
    head, tail = OracleEnv(spec.with_envs(S, 0)), OracleEnv(spec.with_envs(S, E - S))
    for x in (eng, ser, head, tail):
        x.reset()
    done_steps = 0
    for n in (3, 50, 1, 29, 45):                              # crosses the horizon: every env auto-resets inside a chain
        eng.rollout_sampled(n)
        for _ in range(n):
            ser.step_sampled()
            for o in (head, tail):
                o.step(o.sample_actions())
        done_steps += n
        for o, sl in ((head, slice(0, S)), (tail, slice(E - S, E))):
            for k in ('obs', 'done', 'reward', 'all_done'):
                assert np.array_equal(getattr(eng, k)[sl].cpu().numpy(), getattr(o, k)), (done_steps, k)
        st = eng.state_numpy()
        assert_state_equal({k: (None if v is None else v[:S]) for k, v in st.items()}, head.state, f'head {done_steps}')
        assert_state_equal({k: (None if v is None else v[E - S:]) for k, v in st.items()}, tail.state, f'tail {done_steps}')
        for k in ('obs', 'reward', 'done', 'all_done', 'actions'):
            assert torch.equal(getattr(eng, k), getattr(ser, k)), (done_steps, k)
        assert_state_equal(st, ser.state_numpy(), f'all envs {done_steps}')
        assert torch.equal(eng.stats(), ser.stats())


@pytest.mark.parametrize('dynamic', ['0', '1'])
@pytest.mark.parametrize('name', ['tb_c5', 'tb_c2'])
def test_static_and_dynamic_shape_instantiations(mirror, name, dynamic, monkeypatch):
    """The exact shapes of BASELINE configs 5 and 2 select compile-time-shape instantiations of the specialised kernel;
    BGW_DYNAMIC_SHAPES=1 forces the run-time-shape one.  Both against the oracle over a full episode + reset."""
    monkeypatch.setenv('BGW_DYNAMIC_SHAPES', dynamic)
    builder = scenarios.build_tb_c5 if name == 'tb_c5' else scenarios.SCENARIOS[name][0]
    spec = compile_sim(builder(mirror), n_envs=6 if name == 'tb_c5' else 300, env_offset=11, seed=0xB200, horizon=40, auto_reset=True)
    eng, ora = _pair(spec)
    run_lockstep(eng, ora, 90, label=f'{name}/dynamic={dynamic}')


@pytest.mark.parametrize('name', ['maze_c1', 'pacman_c3', 'tb_blocking'])
def test_static_wall_table_and_traced_blockers_agree(mirror, name, monkeypatch):
    """Walls use a per-viewer-cell LOS table built at bgw_create; BGW_NO_STATIC_MASK=1 traces every blocker
    instead.  Both must equal the oracle (the default path is covered by test_engine_matches_oracle)."""
    builder, manager, _ = scenarios.SCENARIOS[name]
    spec = compile_sim(builder(mirror), manager=manager, n_envs=4, seed=17, horizon=20, auto_reset=True)
    monkeypatch.setenv('BGW_NO_STATIC_MASK', '1')
    eng, ora = _pair(spec)
    run_lockstep(eng, ora, 30, label=name + '/traced')


def test_more_than_256_entities_use_16_bit_list_heads(mirror):
    """The specialised kernel keeps 8-bit list heads up to 256 entities and 16-bit ones beyond."""
    sim = scenarios.build_tb_c5(mirror, rows=40, cols=36, n_agents=300, view_range=4)
    spec = compile_sim(sim, n_envs=5, env_offset=2, seed=99, horizon=30, auto_reset=True)
    eng, ora = _pair(spec)
    run_lockstep(eng, ora, 70, label='tb_300_agents')


@pytest.mark.parametrize('name', ['tb_c2', 'maze_c1'])
def test_masked_reset_touches_only_the_selected_envs(mirror, name):
    """bgw_reset(env_mask): AllStepManager.reset for a subset of the batch, the rest keeps running."""
    builder, manager, _ = scenarios.SCENARIOS[name]
    spec = compile_sim(builder(mirror), manager=manager, n_envs=10, seed=8, horizon=0, auto_reset=False)
    eng, ora = _pair(spec)
    eng.reset()
    ora.reset()
    rng = np.random.default_rng(3)
    for t in range(30):
        act = ora.sample_actions()
        ora.step(act)
        eng.step(torch.from_numpy(act).cuda())
        if t % 7 == 6:
            mask = (rng.random(10) < 0.4).astype(np.uint8)
            ora.reset(mask)
            eng.reset(mask)
        assert np.array_equal(eng.obs.cpu().numpy(), ora.obs), f'{name} step {t}'
        assert_state_equal(eng.state_numpy(), ora.state, f'{name} step {t}')


def _tiny_battle(api, rows, cols, n_agents, teams=2, view=1, blocking=False, overlap_all=True):
    agents = {}
    for i in range(n_agents):
        ag = api.ex.BattleAgent(id=f'a{i}', encoding=i % teams + 1, initial_health=1.0, blocking=blocking and i == 0)
        ag.view_range = view
        agents[ag.id] = ag
    everyone = set(range(1, teams + 1))
    overlap = {k: set(everyone) for k in everyone} if overlap_all else {k: {k} for k in everyone}
    attack = {k: everyone - {k} for k in everyone}
    return api.ex.TeamBattleSim.build_sim(rows, cols, agents=agents, overlapping=overlap, attack_mapping=attack,
                                          states={'PositionState', 'HealthState'}, observers={'PositionCenteredEncodingObserver'},
                                          dones={'OneTeamRemainingDone'})


@pytest.mark.parametrize('rows,cols,n_agents,blocking', [(1, 1, 3, False), (1, 1, 1, False), (1, 7, 4, False), (5, 1, 4, True),
                                                         (2, 2, 9, False), (3, 3, 2, True), (1, 700, 12, False)])
def test_degenerate_grids(mirror, rows, cols, n_agents, blocking):
    """One-cell and one-line grids (one with more words per row than a CTA has threads), a single agent, more agents than
    cells (everything overlaps): both kernels against the oracle -- every window cell out of bounds, every move into a
    border, every agent on one cell; and bgw_observe on the state they end in."""
    E = 40 if cols < 100 else 8
    spec = compile_sim(_tiny_battle(mirror, rows, cols, n_agents, blocking=blocking, overlap_all=cols < 100), n_envs=E,
                       seed=rows * 100 + cols, horizon=12, auto_reset=True)     # the wide grid: no mixed cells, the gather-only observe kernel
    eng, ora = _pair(spec)
    run_lockstep(eng, ora, 40, label=f'{rows}x{cols}/{n_agents}')
    got = eng.observe(out=torch.full_like(eng.obs, 99)).cpu().numpy()
    assert np.array_equal(got, np.stack([ora.observe(e) for e in range(E)]))


def test_placement_failure_is_reported_not_raised(mirror):
    """More agents than cells without overlapping: the reference raises RuntimeError at state.py:161; the batch reports
    BGW_ENV_ERROR / BgwState.error == 2 for the env and carries on, engine and oracle alike."""
    spec = compile_sim(_tiny_battle(mirror, 2, 2, 6, teams=6, overlap_all=False), n_envs=16, seed=4, horizon=10, auto_reset=True)
    eng, ora = _pair(spec)
    eng.reset()
    ora.reset()
    assert (ora.state['error'] == 2).all() and (ora.state['env_flags'] & K.ENV_ERROR).all()
    assert_state_equal(eng.state_numpy(), ora.state, 'placement failure')
    for t in range(5):
        act = ora.sample_actions()
        eng.step(torch.from_numpy(act).cuda())
        ora.step(act)
        assert_outputs_equal(eng, ora, f'placement failure step {t}')
        assert_state_equal(eng.state_numpy(), ora.state, f'placement failure step {t}')


def test_create_rejects_what_it_cannot_run(mirror):
    """bgw_create fails loudly (non-zero code + message) instead of running something else."""
    import ctypes as C
    lib = K.load()

    def create(spec):
        h = C.c_void_p()
        rc = lib.bgw_create(C.byref(spec.c_struct()), 0, C.byref(h))
        if rc == 0:
            lib.bgw_destroy(h)
        return rc, lib.bgw_last_error().decode()

    spec = compile_sim(scenarios.build_tb_c2(mirror), n_envs=4)
    spec.simultaneous_attacks = spec.simultaneous_attacks.copy()
    spec.simultaneous_attacks[0] = 2                                    # Binary actor: TeamBattleSim.step raises in the reference
    rc, msg = create(spec)
    assert rc != 0 and 'simultaneous_attacks' in msg
    spec = compile_sim(scenarios.build_tb_selective(mirror), n_envs=4)
    spec.simultaneous_attacks = np.full_like(spec.simultaneous_attacks, 16)
    spec.attack_range = np.full_like(spec.attack_range, 2)             # 25 cells x 16 attacks > BGW_MAX_VICTIMS
    rc, msg = create(spec)
    assert rc != 0 and 'could attack' in msg
    spec = compile_sim(scenarios.build_tb_c2(mirror), n_envs=4)
    spec.encoding = spec.encoding.copy()
    spec.encoding[3] = 0
    rc, msg = create(spec)
    assert rc != 0 and 'encoding' in msg
    spec = compile_sim(scenarios.build_tb_ammo(mirror), n_envs=4)
    from abmarl_b200.engine import BatchedGridWorld
    eng = BatchedGridWorld(spec, device='cuda:0')
    st = K.BgwState()
    for name in ('cell', 'next', 'flags', 'health', 'reward_acc', 'episode', 'step', 'env_flags', 'turn', 'error', 'stats'):
        setattr(st, name, eng.state[name].data_ptr())
    assert lib.bgw_bind_state(eng._h, C.byref(st)) != 0 and b'ammo' in lib.bgw_last_error()      # AmmoAgents need `ammo`
    spec = compile_sim(scenarios.build_tb_c2(mirror), n_envs=4)
    eng = BatchedGridWorld(spec, device='cuda:0')
    assert lib.bgw_generate_layouts(eng._h, None, 0, None) != 0 and b'layout' in lib.bgw_last_error()


@pytest.mark.parametrize('name', ['tb_encoding', 'tb_restricted', 'tb_selective', 'tb_ammo'])
def test_manager_encodes_reference_style_action_dicts(mirror, name):
    """AllStepManager.encode_actions packs the reference's action dicts ({'move': ..., 'attack': dict | vector | matrix |
    count}) into the action rows the kernels read: driving the manager with dicts equals driving the oracle with bytes;
    as_dicts() hands back reference-shaped observations (with 'ammo' where the sim has an AmmoObserver)."""
    from abmarl_b200.managers import AllStepManager
    from oracle.oracle import OracleEnv
    builder, _, _ = scenarios.SCENARIOS[name]
    sim = builder(mirror)
    mgr = AllStepManager(sim, n_envs=3, seed=19, horizon=30, auto_reset=True, device='cuda:0')
    spec = mgr.spec
    ora = OracleEnv(spec)
    mgr.reset()
    ora.reset()
    for t in range(25):
        act = ora.sample_actions()
        dicts = []
        for e in range(3):
            d = {}
            for l, a in enumerate(spec.learner_agents):
                agent = sim.agents[spec.agent_ids[a]]
                att = act[e, l, 2:].view(np.uint8).astype(int)
                n = 2 * agent.attack_range + 1
                if spec.attack_actor == K.ATTACK_ENCODING:
                    attack = {enc: int(att[enc - 1]) for enc in sorted(agent.action_space['attack'].spaces)}
                elif spec.attack_actor == K.ATTACK_RESTRICTED:
                    attack = att[:agent.simultaneous_attacks]
                elif spec.attack_actor == K.ATTACK_SELECTIVE:
                    attack = att[:n * n].reshape(n, n)
                else:
                    attack = int(att[0])
                d[agent.id] = {'move': np.array([int(act[e, l, 0]), int(act[e, l, 1])]), 'attack': attack}
            dicts.append(d)
        packed = mgr.encode_actions(dicts)
        np.testing.assert_array_equal(packed.cpu().numpy(), act)
        mgr.step(packed)
        ora.step(act)
        assert_outputs_equal(mgr.engine, ora, f'{name} step {t}')
        obs, rew, dn, _ = mgr.as_dicts(env=1)
        for agent_id, o in obs.items():
            if spec.ammo_observer:
                assert o['ammo'] == int(ora.state['ammo'][1, spec.agent_ids.index(agent_id)])
            assert 'position_centered_encoding' in o
