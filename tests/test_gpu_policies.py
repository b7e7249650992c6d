"""The step kernels driven by the structured policies of tests/policies.py, against the CPU oracle after every step.

Random actions almost never reach what the kernels' hardest machinery exists for: the ordered reservation rounds and
touch bit maps under long chains of contested moves (a convoy runs 48 move rounds in one env-step), the hashed slot
tables under load (the C5 instantiation's 128 slots per table alias rows r and r + 2), occupant lists of 64 entities
unlinked and appended by movers that all name the same cell, melees in which many attackers share windows, and the
summary grid and occupant lists a block of steps keeps in shared memory.  Each case proves through BGW_VERBOSE which
kernel ran and compares every output and the full state, `next` order included, with the oracle."""
import numpy as np
import pytest
import torch

from abmarl_b200 import _capi as K
from abmarl_b200.spec import compile_sim
from tests import policies as P
from tests import scenarios
from tests.helpers import assert_outputs_equal, assert_state_equal
from tests.test_gpu_edges import _created, battle

pytestmark = pytest.mark.gpu

C5 = ('C5 (compile-time)', 64)
C2 = ('C2 (compile-time)', 32)


def _snap(ora):
    return {k: (None if v is None else v.copy()) for k, v in ora.state.items()}


def lockstep(eng, ora, policy, steps, order=None, seed=0, label=''):
    """Reset both, then step both with `policy` (computed from the oracle's state) for `steps` steps, comparing
    everything after each; returns the longest move chain and the largest pile seen."""
    spec = ora.spec
    eng.reset()
    ora.reset()
    assert_state_equal(eng.state_numpy(), ora.state, f'{label} reset')
    rng = np.random.default_rng(seed)
    o = None if order is None else np.ascontiguousarray(np.broadcast_to(order, (ora.E, ora.L)), dtype=np.int16)
    chain = pile = 0
    for t in range(steps):
        before = _snap(ora)
        act = policy(spec, before, t, rng)
        P.assert_in_action_space(spec, act)
        eng.step(torch.from_numpy(act).cuda(), None if o is None else torch.from_numpy(o).cuda())
        ora.step(act, o)
        assert_outputs_equal(eng, ora, f'{label} step {t}')
        assert_state_equal(eng.state_numpy(), ora.state, f'{label} step {t}')
        chain = max(chain, int(P.move_chains(spec, before, ora.state).max()))
        pile = max(pile, int(P.largest_pile(spec, ora.state).max()))
    return chain, pile


def _sim(name, mirror, n_envs, horizon=200, seed=0x501):
    builder, manager, _ = scenarios.SCENARIOS[name]
    return compile_sim(builder(mirror), manager=manager, n_envs=n_envs, env_offset=3, seed=seed, horizon=horizon,
                       auto_reset=True)


def gather_melee(gather):
    """rendezvous for `gather` steps, a dispersal step, then a melee"""
    return P.schedule((gather, P.Rendezvous()), (1, P.disperse), (1, P.melee()))


# name: (spec builder(mirror), policy factory, steps, kernel reported by bgw_create, least chain, least pile)
FAST = {
    'c5_rendezvous_melee': (lambda m: compile_sim(scenarios.build_tb_c5(m), n_envs=2, seed=0x501, horizon=300, auto_reset=True),
                            lambda: gather_melee(100), 130, C5, 2, 64),
    'c5_convoy': (lambda m: P.convoy_spec(n_envs=4), P.convoy, 16, C5, 48, 1),
    'c5_wall_herding': (lambda m: compile_sim(scenarios.build_tb_c5(m), n_envs=2, seed=0x502, horizon=300, auto_reset=True),
                        lambda: P.wall_herding, 50, C5, 2, 3),
    'c2_disperse_melee': (lambda m: _sim('tb_c2', m, 48), lambda: P.schedule((1, P.disperse), (20, P.melee()), (1, P.wall_herding)),
                          40, C2, 1, 6),
    'c5_small_rendezvous_melee': (lambda m: _sim('tb_c5_small', m, 16), lambda: gather_melee(40), 70, ('run-time', 96), 2, 20),
    'dense_rendezvous_melee': (lambda m: _sim('tb_dense', m, 32), lambda: gather_melee(12), 40, ('run-time', 32), 2, 5),
    'swap_box': (lambda m: P.swap_spec(n_envs=16)[0], lambda: P.swap(P.swap_spec()[1]), 40, ('run-time', 64), 1, 2),
    'swap_cross': (lambda m: P.swap_spec(n_envs=16, cross=True)[0], lambda: P.swap(P.swap_spec(cross=True)[1]), 40,
                   ('run-time', 64), 1, 1),
    'heads16_A257_rendezvous_melee': (lambda m: battle(20, 20, 257, [1, 2, 3, 4], view=5, att=1, n_envs=4, horizon=200),
                                      lambda: gather_melee(50), 75, ('run-time', 96), 2, 60),
}


@pytest.mark.parametrize('name', list(FAST))
def test_fast_kernel_under_structured_policies(mirror, name, capfd, monkeypatch):
    build, policy, steps, kernel, least_chain, least_pile = FAST[name]
    spec = build(mirror)
    eng, ora, fast, _ = _created(spec, capfd, monkeypatch)
    assert fast == kernel, f'{name}: bgw_create reported {fast}'
    chain, pile = lockstep(eng, ora, policy(), steps, label=name)
    assert chain >= least_chain and pile >= least_pile, (name, chain, pile)


def test_specialized_fast_kernel_under_structured_policies(mirror, capfd, monkeypatch, tmp_path):
    spec = _sim('tb_c5_small', mirror, 16)
    eng, ora, fast, _ = _created(spec, capfd, monkeypatch)
    assert fast == ('run-time', 96)
    monkeypatch.setenv('BGW_VERBOSE', '1')
    capfd.readouterr()
    eng.specialize(cache_dir=str(tmp_path))
    assert "fast kernel compiled for this spec's shape" in capfd.readouterr().err
    monkeypatch.delenv('BGW_VERBOSE')
    chain, pile = lockstep(eng, ora, gather_melee(40), 70, label='tb_c5_small/specialized')
    assert pile >= 20


GENERAL = ['tb_stacked', 'tb_blocking', 'tb_selective_stacked', 'tb_encoding_stacked', 'tb_restricted_stacked',
           'tb_ammo_selective', 'reach_target_crowd']


@pytest.mark.parametrize('serial', ['0', '1'])
@pytest.mark.parametrize('name', GENERAL)
def test_general_kernel_under_structured_policies(mirror, name, serial, capfd, monkeypatch):
    """Rendezvous, dispersal, melee at each attack actor's maximum and wall herding, through the reservation rounds of
    the general kernel and (BGW_SERIAL_ACTORS=1) its rank-order loop."""
    monkeypatch.setenv('BGW_SERIAL_ACTORS', serial)
    spec = _sim(name, mirror, 16, horizon=60)
    eng, ora, fast, _ = _created(spec, capfd, monkeypatch)
    assert fast is None, f'{name}: expected the general kernel, bgw_create reported {fast}'
    policy = P.schedule((15, P.Rendezvous()), (2, P.disperse), (20, P.melee()), (1, P.wall_herding))
    chain, pile = lockstep(eng, ora, policy, 50, label=f'{name}/serial={serial}')
    assert pile >= 4


@pytest.mark.parametrize('reverse', [False, True])
@pytest.mark.parametrize('kernel', ['fast', 'general'])
def test_convoy_under_caller_order(mirror, kernel, reverse, capfd, monkeypatch):
    """order= in dict order (front to back: 48-long chains) and reversed (back to front: single moves)."""
    if kernel == 'general':
        monkeypatch.setenv('BGW_GENERIC_KERNEL', '1')
    spec = P.convoy_spec(n_envs=4)
    eng, ora, fast, _ = _created(spec, capfd, monkeypatch)
    assert fast == (C5 if kernel == 'fast' else None)
    order = np.arange(spec.n_learners, dtype=np.int16)
    chain, _ = lockstep(eng, ora, P.convoy(), 14, order=order[::-1] if reverse else order, label=f'convoy/{kernel}/{reverse}')
    assert chain == (1 if reverse else 48)


@pytest.mark.parametrize('name,kernel', [('tb_c5_small', ('run-time', 96)), ('tb_selective_stacked', None)])
def test_rows_of_done_learners_are_ignored(mirror, name, kernel, capfd, monkeypatch):
    """bgw_step ignores the action rows of learners already reported done: 0x7F junk there gives what zero rows give,
    and both what the oracle gives."""
    from abmarl_b200.engine import BatchedGridWorld
    spec = _sim(name, mirror, 16, horizon=40)
    a, ora, fast, _ = _created(spec, capfd, monkeypatch)
    assert fast == kernel
    b = BatchedGridWorld(spec, device='cuda:0')
    for x in (a, b, ora):
        x.reset()
    rng = np.random.default_rng(1)
    policy = P.melee()
    junk_rows = 0
    for t in range(40):
        st = _snap(ora)
        act = policy(spec, st, t, rng)
        done = (st['flags'][:, P.learners(spec)] & K.ST_DONE_REPORTED) != 0
        bad = act.copy()
        bad[done] = 0x7F
        junk_rows += int(done.sum())
        a.step(torch.from_numpy(bad).cuda())
        b.step(torch.from_numpy(act).cuda())
        ora.step(act)
        for k in ('obs', 'reward', 'done', 'all_done'):
            assert torch.equal(getattr(a, k), getattr(b, k)), (t, k)
        assert_state_equal(a.state_numpy(), b.state_numpy(), f'{name} junk vs zero, step {t}')
        assert_outputs_equal(a, ora, f'{name} step {t}')
        assert_state_equal(a.state_numpy(), ora.state, f'{name} step {t}')
    assert junk_rows > 50


@pytest.mark.parametrize('grid', [None, '5'])
def test_rollout_blocks_from_rendezvous_piles(mirror, grid, capfd, monkeypatch):
    """Engines a and b and the oracle walk to four 64-entity piles in lockstep; then the keyed random policy disperses
    them: a.rollout_sampled(n) against n x b.step_sampled() against the oracle, n crossing block ends.  With BGW_GRID=5
    the 8 envs outnumber the CTAs."""
    from abmarl_b200.engine import BatchedGridWorld
    if grid:
        monkeypatch.setenv('BGW_GRID', grid)
    spec = compile_sim(scenarios.build_tb_c5(mirror), n_envs=8, env_offset=5, seed=0xB10C, horizon=400, auto_reset=True)
    a, ora, fast, _ = _created(spec, capfd, monkeypatch)
    assert fast == C5
    b = BatchedGridWorld(spec, device='cuda:0')
    for x in (a, b, ora):
        x.reset()
    rng = np.random.default_rng(2)
    policy = P.Rendezvous()
    for t in range(120):
        act = policy(spec, _snap(ora), t, rng)
        for x in (a, b):
            x.step(torch.from_numpy(act).cuda())
        ora.step(act)
    assert_outputs_equal(a, ora, 'rendezvous')
    assert_state_equal(a.state_numpy(), ora.state, 'rendezvous')
    assert_state_equal(b.state_numpy(), ora.state, 'rendezvous b')
    assert (P.largest_pile(spec, ora.state) == 64).all()
    done_steps = 0
    for n in (1, 5, 16, 17, 33):
        a.rollout_sampled(n)
        for _ in range(n):
            b.step_sampled()
            ora.step(ora.sample_actions())
        done_steps += n
        for k in ('obs', 'reward', 'done', 'all_done', 'actions'):
            assert torch.equal(getattr(a, k), getattr(b, k)), (done_steps, k)
        assert_state_equal(a.state_numpy(), b.state_numpy(), f'a vs b after {done_steps} random steps')
        assert torch.equal(a.stats(), b.stats())
        assert_outputs_equal(a, ora, f'oracle after {done_steps} random steps')
        assert_state_equal(a.state_numpy(), ora.state, f'oracle after {done_steps} random steps')


def test_large_batch_policy_from_the_engines_state(mirror, capfd, monkeypatch):
    """tb_c5 with 2500 envs (several per resident CTA, so tickets and epochs carry across envs): the policy is computed
    from the engine's own state every step; the oracle follows env slices at both ends of the batch."""
    from oracle.oracle import OracleEnv
    E, S = 2500, 3
    spec = compile_sim(scenarios.build_tb_c5(mirror), n_envs=E, seed=0x2500, horizon=45, auto_reset=True)
    eng, _, fast, _ = _created(spec, capfd, monkeypatch)
    assert fast == C5
    head, tail = OracleEnv(spec.with_envs(S, 0)), OracleEnv(spec.with_envs(S, E - S))
    for x in (eng, head, tail):
        x.reset()
    rng = np.random.default_rng(3)
    policy = P.schedule((50, P.Rendezvous(attack=True)), (1, P.disperse), (1, P.melee()))
    for t in range(80):
        st = eng.state_numpy()
        for o, sl in ((head, slice(0, S)), (tail, slice(E - S, E))):
            assert_state_equal({k: (None if v is None else v[sl]) for k, v in st.items()}, o.state, f'step {t} env slice {sl}')
        act = policy(spec, st, t, rng)
        eng.step(torch.from_numpy(act).cuda())
        for o, sl in ((head, slice(0, S)), (tail, slice(E - S, E))):
            o.step(act[sl])
            for k in ('obs', 'done', 'reward', 'all_done'):
                assert np.array_equal(getattr(eng, k)[sl].cpu().numpy(), getattr(o, k)), (t, k)
