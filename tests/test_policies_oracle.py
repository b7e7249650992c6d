"""The structured policies of tests/policies.py reach the inputs they exist for, on the CPU oracle: long chains of
cross-team moves, piles of 64 entities, mass dispersal from one cell, melees with many kills and overlapping attack
windows, moves against the walls, exchanges of cells between teams -- and every action they emit stays inside the
reference's action spaces.  The GPU parity tests (test_gpu_policies.py) drive the kernels with these policies; a later
edit that leaves a policy vacuous fails here, on any machine."""
import numpy as np
import pytest

from abmarl_b200 import _capi as K
from abmarl_b200.spec import compile_sim
from tests import policies as P
from tests import scenarios


def _snap(ora):
    return {k: (None if v is None else v.copy()) for k, v in ora.state.items()}


def drive(spec, policy, steps, order=None, seed=7):
    """Run `policy` on the oracle; per step (before, actions, after)."""
    from oracle.oracle import OracleEnv
    ora = OracleEnv(spec)
    ora.reset()
    rng = np.random.default_rng(seed)
    out = []
    for t in range(steps):
        before = _snap(ora)
        act = policy(spec, before, t, rng)
        P.assert_in_action_space(spec, act)
        ora.step(act, None if order is None else np.broadcast_to(order, (ora.E, ora.L)))
        out.append((before, act, _snap(ora)))
    return out


def test_convoy_chains_front_to_back_and_single_moves_back_to_front():
    """The headline shape in bands of 48: processed front to back (dict order) every learner moves and the chain is the
    band; processed back to front (a reversed order=) a learner moves only into a gap opened in an earlier step."""
    spec = P.convoy_spec(n_envs=2)
    assert (spec.n_agents, spec.rows, spec.cols) == (256, 64, 64)
    fwd = drive(spec, P.convoy(), 10)
    for before, act, after in fwd:
        assert (P.move_chains(spec, before, after) >= 40).all()
        assert (P.move_chains(spec, before, after) == 48).all()
    L = spec.n_learners
    back = drive(spec, P.convoy(), 10, order=np.arange(L)[::-1].astype(np.int16))
    for t, (before, act, after) in enumerate(back):
        assert (P.move_chains(spec, before, after) == 1).all()
        moved = (before['cell'] != after['cell']).sum(axis=1)
        assert (moved == 6 * (t + 1)).all(), moved             # the six band fronts, then one more per band and step


def test_rendezvous_piles_every_team_on_its_corner_then_disperse_empties_it(mirror):
    spec = compile_sim(scenarios.build_tb_c5(mirror), n_envs=2, seed=1, horizon=300, auto_reset=True)
    steps = drive(spec, P.schedule((100, P.Rendezvous()), (1, P.disperse)), 101)
    before, act, after = steps[-1]
    assert (P.largest_pile(spec, before) >= 60).all()
    assert (P.largest_pile(spec, before) == 64).all()          # 4 teams of 64, each on its own corner cell
    for e in range(spec.n_envs):                                # the dispersal: every learner names its pile's cell
        assert (act[e, :, :2] != 0).any(axis=1).all()
        leavers = np.bincount(before['cell'][e][before['cell'][e] != after['cell'][e]].astype(np.int64))
        assert leavers.max() >= 3                               # a corner leaves three ways out


def test_melee_kills_many_in_one_env_step(mirror):
    spec = compile_sim(scenarios.build_tb_c5(mirror), n_envs=2, seed=1, horizon=300, auto_reset=True)
    steps = drive(spec, P.melee(), 80)
    assert max(P.kills(spec, b, a).max() for b, _, a in steps) >= 20
    assert max(P.overlapping_attackers(spec, b, act).max() for b, act, _ in steps) >= 100
    assert max(P.largest_pile(spec, a).max() for _, _, a in steps) >= 8


@pytest.mark.parametrize('name', ['tb_c2', 'tb_c5_small', 'tb_dense', 'tb_stacked', 'tb_blocking', 'tb_selective_stacked',
                                  'tb_encoding_stacked', 'tb_restricted_stacked', 'tb_ammo_selective', 'reach_target_crowd'])
def test_melee_at_maximal_attack_per_actor(mirror, name):
    """Every attack actor's maximal action (Binary, EncodingBased, Selective, RestrictedSelective) kills and its
    attack windows overlap; the actions stay inside the actor's bounds (drive checks every step)."""
    builder, manager, _ = scenarios.SCENARIOS[name]
    spec = compile_sim(builder(mirror), manager=manager, n_envs=8, seed=3, horizon=60, auto_reset=True)
    steps = drive(spec, P.melee(), 40)
    assert max(P.kills(spec, b, a).max() for b, _, a in steps) >= 3
    if name != 'reach_target_crowd':                            # one attacker there: the target
        assert max(P.overlapping_attackers(spec, b, act).max() for b, act, _ in steps) >= 10
    sim = spec.simultaneous_attacks[P.learners(spec)]
    att = (spec.klass[P.learners(spec)] & K.AG_ATTACKING) != 0
    _, act, _ = steps[0]
    if spec.attack_actor == K.ATTACK_BINARY:
        assert (act[:, att, 2] == sim[att]).all()
    elif spec.attack_actor == K.ATTACK_RESTRICTED:
        for l in np.nonzero(att)[0]:
            assert (act[:, l, 2:2 + sim[l]] > 0).all() and (act[:, l, 2:2 + sim[l]] == act[:, l, 2:3]).all()
    elif spec.attack_actor == K.ATTACK_SELECTIVE:
        assert ((act[:, att, 2:] > 0).sum(axis=-1) == 1).all()
        assert (act[:, att, 2:].max(axis=-1) == sim[att]).all()
    elif spec.attack_actor == K.ATTACK_ENCODING:
        assert (act[:, att, 2:].max(axis=-1) == sim[att]).all()


def test_wall_herding_pushes_moves_off_the_grid(mirror):
    spec = compile_sim(scenarios.build_tb_c5(mirror), n_envs=2, seed=1, horizon=300, auto_reset=True)
    steps = drive(spec, P.wall_herding, 60)
    assert max(P.off_grid_moves(spec, b, act).max() for b, act, _ in steps) >= 150


@pytest.mark.parametrize('cross', [False, True])
def test_swap_exchanges_cells_between_teams(cross):
    """Pairs and triples named each other's cells; where teams may share a cell (1 and 2) some exchanges succeed."""
    spec, partner = P.swap_spec(cross=cross)
    assert (spec.encoding[partner] != spec.encoding).all()
    steps = drive(spec, P.swap(partner), 20)
    assert max(P.exchanges(spec, b, a).max() for b, _, a in steps) >= 4
    before, act, after = steps[0]
    assert (act[:, :, :2] != 0).any(axis=-1).all()             # every learner names its partner's cell


def test_policies_on_the_other_move_actions(mirror):
    """The cross actor and ravelled box moves (range 2) stay in their action spaces too."""
    from tests.test_gpu_edges import battle
    for spec in (battle(8, 9, 24, [1, 2, 3], cross=True, n_envs=3), battle(8, 9, 24, [1, 2, 3], move=2, n_envs=3)):
        for pol in (P.Rendezvous(attack=True), P.disperse, P.melee(), P.wall_herding, P.convoy(1, -1)):
            drive(spec, pol, 8)
    spec = compile_sim(scenarios.build_mm_random(mirror), manager='all_step', n_envs=3, seed=1, horizon=20, auto_reset=True)
    assert spec.ravel_actions
    for pol in (P.Rendezvous(), P.disperse, P.wall_herding):
        acts = [act for _, act, _ in drive(spec, pol, 6)]
        assert max(int(a[..., 0].view(np.uint8).max()) for a in acts) > 12      # moves other than the centre of the 5x5 box
