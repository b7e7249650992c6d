"""The kernels at their structural edges, against the CPU oracle (and, for the line of sight, the reference's fixture).

The kernels branch on properties of the spec, not on scenarios: the team-battle kernel on the view and attack ranges,
the move actor, whether cells can hold mixed encodings, accuracy draws, observe_self, the entity count (thread count,
cp.async chunking, 8- or 16-bit list heads), the padded grid width, and whether every entity is a learner; the general
kernel on the entity count (threads), the grid size (16-bit cells next to the 0xFFFF sentinel), the number of LOS masks
that fit in shared memory; both on encodings above 31 (64-bit team sets, overlap and attack rows, stacked channels).
Each test builds specs that sit on such an edge, proves which kernel and which observe path ran (BGW_VERBOSE), and
compares everything with the oracle.
"""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from abmarl_b200 import _capi as K
from abmarl_b200.spec import compile_sim
from tests import scenarios
from tests.helpers import run_lockstep, assert_outputs_equal, assert_state_equal
from tests.kat_cases import make_spec, OBS, MOV, ATT, HEA, LRN, BLK
from tests.test_oracle_relabel import RELABEL_SCENARIOS, relabel_map, relabel_spec, relabel_obs

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
FAST_LINE = re.compile(r'\[bgw\] fast kernel: shape ([^,]+), T=(\d+)')
OBSERVE_LINE = re.compile(r'\[bgw\] observe kernel: (gather-only, view (\d)|general)')


def _pair(spec):
    from abmarl_b200.engine import BatchedGridWorld
    from oracle.oracle import OracleEnv
    return BatchedGridWorld(spec, device='cuda:0'), OracleEnv(spec)


def _created(spec, capfd, monkeypatch):
    """Engine + oracle, and what bgw_create reported: (fast kernel shape and threads or None, observe view or 0)."""
    monkeypatch.setenv('BGW_VERBOSE', '1')
    capfd.readouterr()
    eng, ora = _pair(spec)
    err = capfd.readouterr().err
    monkeypatch.delenv('BGW_VERBOSE')
    fast = FAST_LINE.search(err)
    obs = OBSERVE_LINE.search(err)
    assert obs, err
    return eng, ora, (fast.group(1), int(fast.group(2))) if fast else None, int(obs.group(2) or 0)


def _observe_matches(eng, ora, where):
    got = eng.observe(out=torch.full_like(eng.obs, 99)).cpu().numpy()
    want = np.stack([ora.observe(e) for e in range(eng.E)])
    bad = np.argwhere(got != want)
    assert bad.size == 0, f'{where}: bgw_observe differs at {bad[:5].tolist()}'


def _fast_threads(A):
    """threads per env of the team-battle kernel (bgw.cu): one warp up to 32 entities, two up to 64, else three"""
    return 32 if A <= 32 else 64 if A <= 64 else 96


def _general_threads(A):
    return 32 if A <= 128 else 64 if A <= 1024 else 128


# ---------------------------------------------------------------------------------------------------
# A. the team-battle kernel's branch matrix
# ---------------------------------------------------------------------------------------------------
def battle(rows, cols, n_learners, encs, view=1, att=1, move=1, cross=False, mix=False, acc=1.0, observe_self=True,
           rpo=False, health_npc=0, plain_npc=0, n_envs=16, horizon=8, seed=1):
    """A team battle the specialised kernel runs (BinaryAttackActor, position-centred observer, no blockers).  `view` and
    `att` may be lists (cycled over the learners); `mix`: every team may share a cell with every other; non-learners:
    `health_npc` entities with health that every team may attack (encoding max(encs) + 1), `plain_npc` entities without
    anything (encoding max(encs) + 2)."""
    views, atts = np.atleast_1d(view), np.atleast_1d(att)
    agents = [dict(enc=encs[i % len(encs)], klass=LRN | OBS | MOV | ATT | HEA, view=int(views[i % len(views)]),
                   att_range=int(atts[i % len(atts)]), move=move, strength=0.6 if i % 3 == 0 else 1.0,
                   accuracy=acc if i % 2 else 1.0) for i in range(n_learners)]
    teams = set(encs)
    npc_enc, plain_enc = max(encs) + 1, max(encs) + 2
    assert max(encs) + (2 if plain_npc else 1 if health_npc else 0) <= 63
    # the non-learners come first: entity index != learner index for every learner (the learner_of indirection)
    agents = [dict(enc=npc_enc, klass=HEA) for _ in range(health_npc)] + [dict(enc=plain_enc, klass=0) for _ in range(plain_npc)] + agents
    overlap = {t: set(teams) if mix else {t} for t in teams}
    attack = {t: (teams - {t}) | ({npc_enc} if health_npc else set()) for t in teams}
    sp = make_spec(rows, cols, agents, overlapping=overlap, attack_mapping=attack, attack_actor=K.ATTACK_BINARY,
                   move_actor=K.MOVE_CROSS if cross else K.MOVE_BOX, observe_self=observe_self, done_mask=K.DONE_ONE_TEAM,
                   n_envs=n_envs, seed=seed)
    sp.horizon, sp.auto_reset, sp.randomize_placement_order, sp.env_offset = horizon, 1, int(rpo), 5
    return sp


def branch_props(sp):
    """The spec properties the team-battle kernel specialises on, by the rules of bgw_create (bgw.cu)."""
    A, W = sp.n_agents, sp.cols
    lrn = [a for a in range(A) if sp.klass[a] & LRN]
    views = {int(sp.view_range[a]) for a in lrn if sp.klass[a] & OBS}
    atts = {int(sp.attack_range[a]) for a in range(A) if sp.klass[a] & ATT}
    P = max(max(views), max(atts))
    present = {int(e) for e in sp.encoding}
    can_mix = any(int(sp.overlap[e]) & sum(1 << f for f in present - {e}) for e in present)
    return dict(A=A, view=views.pop() if len(views) == 1 else -1, att=atts.pop() if len(atts) == 1 else -1,
                move=(int(sp.move_actor), int(sp.move_range[lrn[0]])), can_mix=int(bool(can_mix)),
                acc_lt1=int(any(sp.attack_accuracy[a] < 1 for a in range(A) if sp.klass[a] & ATT)),
                observe_self=int(sp.observe_self), rpo=int(sp.randomize_placement_order), identity=int(len(lrn) == A),
                async_ok=1 if A % 16 == 0 else 2 if A % 8 == 0 else 0, head_elem=1 if A <= 256 else 2,
                wmod=(W + 2 * P) % 4, narrow=int(W < 2 * max(sp.view_range[a] for a in lrn) + 1), max_enc=max(present),
                health_npc=int(any(sp.klass[a] == HEA for a in range(A))), plain_npc=int(any(sp.klass[a] == 0 for a in range(A))))


# name: (spec builder, lockstep steps, checks rollout_sampled, checks bgw_specialize)
ROWS = {
    'A1_view1':            (lambda: battle(3, 3, 1, [1], view=1, att=1), 20, False, False),
    'A31_view2_cross':     (lambda: battle(6, 6, 31, [1, 2, 3], view=2, att=2, cross=True, acc=0.75, observe_self=False), 24, False, True),
    'A32_view3_enc63':     (lambda: battle(8, 9, 32, [5, 31, 32, 63], view=3, att=1, move=2), 24, True, True),
    'A33_view4_npc':       (lambda: battle(7, 8, 30, [1, 40], view=4, att=1, cross=True, rpo=True, health_npc=3), 24, True, True),
    'A63_view5_mix':       (lambda: battle(10, 10, 63, [1, 2, 3], view=5, att=2, mix=True, acc=0.75), 24, False, False),
    'A64_view0_npc':       (lambda: battle(9, 11, 56, [2, 33], view=0, att=0, health_npc=4, plain_npc=4), 24, True, True),
    'A65_view6_cross':     (lambda: battle(12, 9, 65, [1, 2, 3, 4], view=6, att=1, cross=True, move=2), 24, False, False),
    'A72_view7_plain':     (lambda: battle(10, 13, 64, [32, 33], view=7, att=2, move=2, plain_npc=8), 24, False, True),
    'A97_mixed_ranges':    (lambda: battle(12, 12, 90, [1, 2, 3], view=[1, 2, 3, 4, 5], att=[0, 1, 2], health_npc=7), 24, True, True),
    'A120_view3_mix_noself': (lambda: battle(14, 14, 120, [3, 4], view=3, att=1, cross=True, mix=True, observe_self=False), 24, False, False),
    'A255_view2_npc':      (lambda: battle(20, 20, 240, [1, 2, 60, 61], view=2, att=1, health_npc=10, plain_npc=5, n_envs=8), 20, False, True),
    'A257_view5':          (lambda: battle(20, 20, 257, [1, 2, 3, 4], view=5, att=1, n_envs=8), 20, True, False),
    'A6_narrow_view4':     (lambda: battle(5, 3, 6, [1, 2], view=4, att=1, cross=True, acc=0.75, rpo=True), 24, False, True),
}


def test_branch_matrix_covers_every_value():
    """The rows of ROWS together take every value the team-battle kernel specialises on."""
    props = [branch_props(ROWS[name][0]()) for name in ROWS]
    seen = lambda k: {p[k] for p in props}
    assert set(range(8)) | {-1} <= seen('view')
    assert {0, 1, 2, -1} <= seen('att')
    assert {(K.MOVE_BOX, 1), (K.MOVE_BOX, 2), (K.MOVE_CROSS, 1), (K.MOVE_CROSS, 2)} <= seen('move')
    for k in ('can_mix', 'acc_lt1', 'observe_self', 'rpo', 'identity', 'narrow', 'health_npc', 'plain_npc'):
        assert seen(k) == {0, 1}, k
    assert {1, 31, 32, 33, 63, 64, 65, 97, 255, 257} <= seen('A')
    assert any(p['A'] > 32 and p['A'] % 8 for p in props) and any(p['A'] > 32 and p['A'] % 16 == 8 for p in props)
    assert seen('async_ok') == {0, 1, 2} and seen('head_elem') == {1, 2} and seen('wmod') == {0, 1, 2, 3}
    assert max(seen('max_enc')) == 63 and any(p['max_enc'] >= 32 and p['att'] == 1 for p in props)
    assert sum(ROWS[n][2] for n in ROWS) >= 4 and sum(ROWS[n][3] for n in ROWS) >= 8


@pytest.mark.parametrize('name', list(ROWS))
def test_team_battle_kernel_branch(name, capfd, monkeypatch, tmp_path):
    build, steps, rollout, specialize = ROWS[name]
    spec = build()
    p = branch_props(spec)
    eng, ora, fast, observe_view = _created(spec, capfd, monkeypatch)
    assert fast == ('run-time', _fast_threads(p['A'])), f'{name}: expected the team-battle kernel, bgw_create reported {fast}'
    assert eng.dims.threads_per_env == _fast_threads(p['A'])
    gather = p['can_mix'] == 0 and p['observe_self'] == 1 and 1 <= p['view'] <= 5
    assert observe_view == (p['view'] if gather else 0), f'{name}: observe kernel'
    run_lockstep(eng, ora, steps, label=name)
    assert (ora.state['episode'] >= 1).all(), f'{name}: every env should have been auto-reset'
    _observe_matches(eng, ora, name)
    if rollout:
        from abmarl_b200.engine import BatchedGridWorld
        from oracle.oracle import OracleEnv
        a, b, o = BatchedGridWorld(spec, device='cuda:0'), BatchedGridWorld(spec, device='cuda:0'), OracleEnv(spec)
        for x in (a, b, o):
            x.reset()
        for n in (1, 11, 6):
            a.rollout_sampled(n)
            for _ in range(n):
                b.step_sampled()
                o.step(o.sample_actions())
            for k in ('obs', 'reward', 'done', 'all_done', 'actions'):
                assert torch.equal(getattr(a, k), getattr(b, k)), (name, n, k)
            assert_state_equal(a.state_numpy(), b.state_numpy(), f'{name} rollout {n}')
            assert torch.equal(a.stats(), b.stats())
            assert_outputs_equal(a, o, f'{name} rollout {n} vs oracle')
            assert_state_equal(a.state_numpy(), o.state, f'{name} rollout {n} vs oracle')
    if specialize:
        eng2, ora2 = _pair(spec)
        monkeypatch.setenv('BGW_VERBOSE', '1')
        capfd.readouterr()
        eng2.specialize(cache_dir=str(tmp_path))
        assert "fast kernel compiled for this spec's shape" in capfd.readouterr().err
        monkeypatch.delenv('BGW_VERBOSE')
        assert len([f for f in os.listdir(tmp_path) if f.endswith('.cubin')]) == 1
        run_lockstep(eng2, ora2, steps, label=name + '/specialized')
        _observe_matches(eng2, ora2, name + '/specialized')


# ---------------------------------------------------------------------------------------------------
# A. the general kernel's edges
# ---------------------------------------------------------------------------------------------------
def general(rows, cols, n_learners, view=2, wall=True, stacked=False, blocking_learner=False, walls=(), n_envs=4,
            horizon=5, encs=(1, 2)):
    """A team battle the general kernel runs: a view-blocking wall (or the stacked observer) rules the other one out."""
    agents = [dict(enc=encs[i % len(encs)], klass=LRN | OBS | MOV | ATT | HEA | (BLK if blocking_learner and i == 0 else 0),
                   view=view, att_range=1, move=1, strength=1.0) for i in range(n_learners)]
    wall_enc = max(encs) + 1
    if wall:
        agents.append(dict(enc=wall_enc, pos=(rows - 1, 0), klass=BLK))
    agents += [dict(enc=wall_enc, pos=rc, klass=BLK) for rc in walls]
    teams = set(encs)
    sp = make_spec(rows, cols, agents, overlapping={t: {t} for t in teams}, attack_mapping={t: teams - {t} for t in teams},
                   attack_actor=K.ATTACK_BINARY, observer=K.OBS_STACKED if stacked else K.OBS_POSITION_CENTERED,
                   done_mask=K.DONE_ONE_TEAM, n_envs=n_envs, seed=7)
    sp.horizon, sp.auto_reset, sp.env_offset = horizon, 1, 2
    return sp


@pytest.mark.parametrize('A', [128, 129, 1024, 1025, 4096])
def test_general_kernel_entity_counts(A, capfd, monkeypatch):
    """Thread count 32 / 64 / 128 at 128 | 129 and 1024 | 1025 entities, and the largest entity count (Philox slot 4095)."""
    side = 40 if A <= 1025 else 80
    spec = general(side, side, A - 1, view=1 if A == 4096 else 2, n_envs=2 if A == 4096 else 4)
    assert spec.n_agents == A
    eng, ora, fast, observe_view = _created(spec, capfd, monkeypatch)
    assert fast is None and observe_view == 0
    assert eng.dims.threads_per_env == _general_threads(A)
    run_lockstep(eng, ora, 12 if A < 4096 else 6, label=f'general/{A}')
    _observe_matches(eng, ora, f'general/{A}')


@pytest.mark.parametrize('kernel', ['fast', 'general'])
def test_largest_grid_with_an_entity_next_to_the_sentinel(kernel, capfd, monkeypatch):
    """255 x 257 = 65535 cells: the last cell, 65534, sits next to the 0xFFFF 'no cell' sentinel.  An observing learner is
    fixed there; its window reaches past both borders.  The team-battle kernel takes this grid too (no blocker)."""
    agents = [dict(enc=1 + i % 2, klass=LRN | OBS | MOV | ATT | HEA, view=2, att_range=1, move=1, strength=1.0) for i in range(6)]
    agents[0]['pos'] = (254, 256)
    agents[1]['pos'] = (254, 255)
    spec = make_spec(255, 257, agents, overlapping={1: {1}, 2: {2}}, attack_mapping={1: {2}, 2: {1}},
                     attack_actor=K.ATTACK_BINARY, observer=K.OBS_STACKED if kernel == 'general' else K.OBS_POSITION_CENTERED,
                     done_mask=K.DONE_ONE_TEAM, n_envs=6, seed=11)
    spec.horizon, spec.auto_reset = 6, 1
    eng, ora, fast, _ = _created(spec, capfd, monkeypatch)
    assert (fast is not None) == (kernel == 'fast')
    run_lockstep(eng, ora, 14, label=f'65535 cells/{kernel}')
    eng.reset()
    ora.reset()
    assert (eng.state_numpy()['cell'][:, 0] == 65534).all()
    _observe_matches(eng, ora, f'65535 cells/{kernel}')


def test_stacked_observer_counts_127_entities_in_one_cell(capfd, monkeypatch):
    agents = [dict(enc=1, klass=LRN | OBS | MOV | ATT | HEA, view=1, att_range=1, move=1) for _ in range(127)]
    spec = make_spec(1, 1, agents, overlapping={1: {1}}, attack_actor=K.ATTACK_BINARY, observer=K.OBS_STACKED, n_envs=3, seed=5)
    spec.horizon, spec.auto_reset = 4, 1
    eng, ora, fast, _ = _created(spec, capfd, monkeypatch)
    assert fast is None
    run_lockstep(eng, ora, 10, label='127 in one cell')
    v = eng.obs_view().cpu().numpy()                           # [E, L, 3, 3]: one channel
    assert (v[:, :, 1, 1] == 127).all() and (v[:, :, 0, :] == -1).all()
    _observe_matches(eng, ora, '127 in one cell')


def test_more_observing_learners_than_one_los_batch(capfd, monkeypatch):
    """View 16 with walls: a LOS mask is 35 words, 234 of them fit the shared-memory batch; 240 learners take two batches
    per env.  Fixed walls come from the static table, a blocking learner is traced."""
    walls = [(3, 3), (3, 20), (20, 3), (20, 20), (11, 11), (12, 12), (6, 15), (17, 8)]
    spec = general(24, 24, 240, view=16, wall=False, walls=walls, blocking_learner=True, n_envs=3)
    n_words = ((2 * 16 + 1) ** 2 + 31) // 32
    assert spec.n_learners > (32 * 1024) // (4 * n_words)
    eng, ora, fast, _ = _created(spec, capfd, monkeypatch)
    assert fast is None
    run_lockstep(eng, ora, 8, label='two LOS batches')
    assert (eng.obs_view().cpu().numpy() == -2).any()
    _observe_matches(eng, ora, 'two LOS batches')


def test_create_rejects_specs_over_the_documented_limits():
    """4097 entities, 65536 cells, 128 entities under the stacked observer: bgw_create refuses with a message (never launched)."""
    lib = K.load()

    def create(spec):
        h = C.c_void_p()
        rc = lib.bgw_create(C.byref(spec.c_struct()), 0, C.byref(h))
        if rc == 0:
            lib.bgw_destroy(h)
        return rc, lib.bgw_last_error().decode()

    learner = dict(enc=1, klass=LRN | OBS | MOV, view=1, move=1)
    rc, msg = create(make_spec(70, 70, [learner] * 4097))
    assert rc != 0 and 'n_agents 4097' in msg
    rc, msg = create(make_spec(256, 256, [learner] * 2))
    assert rc != 0 and 'grid 256x256' in msg
    rc, msg = create(make_spec(12, 12, [learner] * 128, observer=K.OBS_STACKED))
    assert rc != 0 and 'stacked' in msg
    for spec in (make_spec(70, 70, [learner] * 4096), make_spec(255, 257, [learner] * 2),
                 make_spec(12, 12, [learner] * 127, observer=K.OBS_STACKED)):
        assert create(spec)[0] == 0                            # the limits themselves are accepted


# ---------------------------------------------------------------------------------------------------
# B. encodings up to 63: relabelling on the engine
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('name', RELABEL_SCENARIOS)
def test_engine_is_invariant_under_relabelled_encodings(mirror, name, capfd, monkeypatch):
    """engine(relabelled) == relabel(engine(original)) == oracle(relabelled), through steps, bgw_observe and rollouts;
    tb_c2 and tb_dense run the team-battle kernel, tb_blocking and tb_stacked the general one."""
    builder, manager, _ = scenarios.SCENARIOS[name]
    spec = compile_sim(builder(mirror), manager=manager, n_envs=24, env_offset=9, seed=0xE63, horizon=12, auto_reset=True)
    m = relabel_map(spec.encoding)
    spec2 = relabel_spec(spec, m)
    from abmarl_b200.engine import BatchedGridWorld
    eo = BatchedGridWorld(spec, device='cuda:0')
    er, ora, fast, _ = _created(spec2, capfd, monkeypatch)
    assert (fast is not None) == (name in ('tb_c2', 'tb_dense'))
    if fast:
        assert fast[0] == 'run-time'
    mo = lambda eng: relabel_obs(eng.obs_view().cpu().numpy(), m, spec.observer, 63)

    def compare(where):
        assert_outputs_equal(er, ora, where)
        assert_state_equal(er.state_numpy(), ora.state, where)
        for k in ('reward', 'done', 'all_done'):
            assert torch.equal(getattr(er, k), getattr(eo, k)), (where, k)
        assert_state_equal(er.state_numpy(), eo.state_numpy(), where + ' vs original')
        np.testing.assert_array_equal(er.obs_view().cpu().numpy(), mo(eo), err_msg=where + ': relabelled observations')

    for x in (eo, er, ora):
        x.reset()
    compare('reset')
    for t in range(30):
        act = eo.sample_actions()
        assert torch.equal(er.sample_actions(), act)
        ora_act = ora.sample_actions()
        np.testing.assert_array_equal(ora_act, act.cpu().numpy())
        eo.step(act)
        er.step(er.actions)
        ora.step(ora_act)
        compare(f'{name} step {t}')
    for x in (eo, er):
        x.observe()
    for e in range(ora.E):
        ora.obs[e] = ora.observe(e)
    compare(f'{name} observe')
    for n in (7, 13):
        eo.rollout_sampled(n)
        er.rollout_sampled(n)
        for _ in range(n):
            ora.step(ora.sample_actions())
        compare(f'{name} rollout {n}')


def test_encoding_based_attack_with_encoding_63(capfd, monkeypatch):
    """EncodingBasedAttackActor: one attack byte per encoding up to the largest, 63 -> action rows of 68 bytes."""
    encs = [1, 32, 63]
    agents = [dict(enc=encs[i % 3], klass=LRN | OBS | MOV | ATT | HEA, view=2, att_range=1, move=1, strength=0.6, simatt=2)
              for i in range(15)]
    spec = make_spec(6, 6, agents, overlapping={e: {e} for e in encs}, attack_mapping={e: set(encs) - {e} for e in encs},
                     attack_actor=K.ATTACK_ENCODING, done_mask=K.DONE_ONE_TEAM, n_envs=24, seed=63)
    spec.horizon, spec.auto_reset = 10, 1
    eng, ora, fast, _ = _created(spec, capfd, monkeypatch)
    assert fast is None and eng.dims.action_stride == 68
    run_lockstep(eng, ora, 40, label='encoding-based attack, encoding 63')
    _observe_matches(eng, ora, 'encoding-based attack, encoding 63')


# ---------------------------------------------------------------------------------------------------
# C. the device line of sight against the reference fixture
# ---------------------------------------------------------------------------------------------------
def _fixture():
    g = np.load(os.path.join(GOLDEN, 'los_r16.npz'))
    R = int(g['range'])
    n = 2 * R + 1
    return R, np.unpackbits(g['packed'], axis=-1)[..., :n * n].reshape(n, n, n, n)


def _los_world(rows, cols, viewer, view, walls_per_env, observer=K.OBS_POSITION_CENTERED):
    """One observing learner at `viewer`; env k has view-blocking walls at viewer + each offset of walls_per_env[k].  The
    walls have no start position, so they are dynamic blockers: the device traces them (no host table)."""
    n_walls = len(walls_per_env[0])
    agents = [dict(enc=1, pos=viewer, klass=LRN | OBS | MOV, view=view, move=1)] + [dict(enc=2, klass=BLK)] * n_walls
    spec = make_spec(rows, cols, agents, observer=observer, n_envs=len(walls_per_env), seed=16)
    layout = np.empty((len(walls_per_env), 1 + n_walls), dtype=np.uint16)
    layout[:, 0] = viewer[0] * cols + viewer[1]
    for k, offs in enumerate(walls_per_env):
        layout[k, 1:] = [(viewer[0] + rd) * cols + viewer[1] + cd for rd, cd in offs]
    eng, ora = _pair(spec)
    for x in (eng, ora):
        x.set_layout(layout)
    return eng, ora


def _check_los(eng, ora, hidden, where):
    """hidden [E, h, w]: the cells the learner's row must show as -2; after reset, after bgw_observe and after a step in
    which it stays put; the engine equals the oracle throughout."""
    eng.reset()
    ora.reset()
    for when in ('reset', 'observe', 'step'):
        if when == 'observe':
            eng.observe()
            for e in range(ora.E):
                ora.obs[e] = ora.observe(e)
        elif when == 'step':
            act = np.zeros((eng.E, eng.L, eng.dims.action_stride), dtype=np.int8)
            eng.step(torch.from_numpy(act).cuda())
            ora.step(act)
            assert_state_equal(eng.state_numpy(), ora.state, f'{where} {when}')
        got = eng.obs_view().cpu().numpy()[:, 0]
        assert np.array_equal(got, ora.obs_view()[:, 0]), f'{where}: engine and oracle differ after {when}'
        bad = np.argwhere((got == -2) != hidden)
        assert bad.size == 0, f'{where} after {when}: hidden cells differ at (env, r, c) {bad[:5].tolist()}'


def test_device_los_every_blocker_offset_at_range_16():
    R, masks = _fixture()
    offs = [(rd, cd) for rd in range(-R, R + 1) for cd in range(-R, R + 1) if (rd, cd) != (0, 0)]
    assert len(offs) == 1088
    eng, ora = _los_world(2 * R + 1, 2 * R + 1, (R, R), R, [[o] for o in offs])
    _check_los(eng, ora, np.stack([masks[rd + R, cd + R] == 0 for rd, cd in offs]), 'range 16')


def test_device_los_several_walls_per_env():
    """Three walls per env: the hidden cells are the union of each wall's (atomic mask updates of one viewer)."""
    R, masks = _fixture()
    rng = np.random.default_rng(16)
    offs = [(rd, cd) for rd in range(-R, R + 1) for cd in range(-R, R + 1) if (rd, cd) != (0, 0)]
    envs = [[offs[i] for i in rng.choice(len(offs), 3, replace=False)] for _ in range(512)]
    eng, ora = _los_world(2 * R + 1, 2 * R + 1, (R, R), R, envs)
    hidden = np.stack([np.logical_or.reduce([masks[rd + R, cd + R] == 0 for rd, cd in ws]) for ws in envs])
    _check_los(eng, ora, hidden, 'three walls')


@pytest.mark.parametrize('rows,cols,viewer', [(17, 17, (0, 0)), (17, 33, (0, 16))])
def test_device_los_absolute_observer_clipped_to_the_grid(rows, cols, viewer):
    """AbsoluteEncodingObserver: the rays are clipped to the grid.  In the corner of a 17 x 17 grid the view (16) covers the
    whole grid; on the edge of a 17 x 33 grid it does not span the grid's width.  Expected: the fixture cropped to the grid."""
    R, masks = _fixture()
    r0, c0 = viewer
    offs = [(r - r0, c - c0) for r in range(rows) for c in range(cols) if (r, c) != viewer]
    eng, ora = _los_world(rows, cols, viewer, R, [[o] for o in offs], observer=K.OBS_ABSOLUTE)
    hidden = np.stack([masks[rd + R, cd + R][R - r0:R - r0 + rows, R - c0:R - c0 + cols] == 0 for rd, cd in offs])
    _check_los(eng, ora, hidden, f'absolute {rows}x{cols} at {viewer}')


@pytest.mark.parametrize('R', [1, 2, 7, 8])
def test_device_los_smaller_ranges(R):
    from oracle.oracle import los_mask
    offs = [(rd, cd) for rd in range(-R, R + 1) for cd in range(-R, R + 1) if (rd, cd) != (0, 0)]
    eng, ora = _los_world(2 * R + 1, 2 * R + 1, (R, R), R, [[o] for o in offs])
    _check_los(eng, ora, np.stack([los_mask(R, rd, cd) == 0 for rd, cd in offs]), f'range {R}')
