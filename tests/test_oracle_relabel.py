"""The CPU oracle is invariant under an order-preserving relabelling of the encodings.

Encodings are labels: the reference compares them for equality, looks them up in the overlap and attack maps and
writes them into observations, and nothing else.  The keyed draws are per entity, not per encoding.  So a spec whose
encodings go through an increasing map m -- with the overlap and attack maps relabelled row and bit alike -- must
play the same game: the same actions, rewards, dones and state, and observations that are m of the original ones.
The golden transcripts only use encodings 1-6; this pins the oracle up to the largest encoding, 63, across the
32-bit boundary of the team sets, without a new reference transcript.
"""
import copy

import numpy as np
import pytest

from abmarl_b200 import _capi as K
from abmarl_b200.spec import compile_sim
from oracle.oracle import OracleEnv
from tests import scenarios


def relabel_map(encodings):
    """Increasing map of the encodings in use onto values on both sides of 32, the largest onto 63."""
    encs = sorted({int(e) for e in encodings})
    assert 2 <= len(encs) <= 5
    return dict(zip(encs, [31, 32, 33, 62][:len(encs) - 1] + [63]))


def relabel_spec(spec, m):
    """`spec` with encoding e replaced by m[e] everywhere: the entities' encodings and the overlap / attack rows and bits."""
    s = copy.copy(spec)
    s.encoding = np.array([m[int(e)] for e in spec.encoding], dtype=spec.encoding.dtype)
    for name in ('overlap', 'attack_map'):
        src, dst = getattr(spec, name), np.zeros_like(getattr(spec, name))
        for e in range(len(src)):
            row = int(src[e])
            if row == 0:
                continue
            assert e in m and all(o in m for o in range(64) if (row >> o) & 1), f'{name}[{e}] names an encoding not in use'
            dst[m[e]] = np.uint64(sum(1 << m[o] for o in range(64) if (row >> o) & 1))
        setattr(s, name, dst)
    return s


def relabel_obs(obs_view, m, observer, max_enc):
    """Observations of the relabelled spec, from those of the original one ([..., h, w] or, stacked, [..., h, w, c])."""
    if observer != K.OBS_STACKED:
        lut = np.arange(-128, 128, dtype=np.int16)
        for e, v in m.items():
            lut[e + 128] = v
        return lut[obs_view.astype(np.int16) + 128].astype(np.int8)
    out = np.zeros(obs_view.shape[:-1] + (max_enc,), dtype=np.int8)
    for e, v in m.items():
        out[..., v - 1] = obs_view[..., e - 1]
    neg = obs_view[..., 0] < 0                      # off the grid (-1) or hidden (-2): the value in every channel
    out[neg] = obs_view[..., :1][neg]
    return out


RELABEL_SCENARIOS = ['tb_c2', 'tb_dense', 'tb_blocking', 'tb_stacked']


@pytest.mark.parametrize('name', RELABEL_SCENARIOS)
def test_oracle_is_invariant_under_relabelled_encodings(mirror, name):
    builder, manager, _ = scenarios.SCENARIOS[name]
    spec = compile_sim(builder(mirror), manager=manager, n_envs=8, env_offset=3, seed=0x5EED, horizon=20, auto_reset=True)
    m = relabel_map(spec.encoding)
    spec2 = relabel_spec(spec, m)
    assert spec2.max_encoding == 63 and min(m.values()) < 32 < max(m.values())
    a, b = OracleEnv(spec), OracleEnv(spec2)
    if spec.observer == K.OBS_STACKED:
        assert b.dims.obs_c == 63
    a.reset()
    b.reset()
    resets = 0
    for t in range(61):
        if t:
            act = a.sample_actions()
            np.testing.assert_array_equal(b.sample_actions(), act, err_msg=f'{name} step {t}: actions')
            a.step(act)
            b.step(act)
            resets += int(((a.all_done & K.ENV_RESET) != 0).sum())
        for k in ('reward', 'done', 'all_done'):
            np.testing.assert_array_equal(getattr(b, k), getattr(a, k), err_msg=f'{name} step {t}: {k}')
        for k in ('cell', 'flags', 'health', 'reward_acc', 'episode', 'step', 'env_flags', 'error'):
            np.testing.assert_array_equal(b.state[k], a.state[k], err_msg=f'{name} step {t}: state[{k}]')
        in_grid = (a.state['flags'] & K.ST_IN_GRID) != 0
        np.testing.assert_array_equal(b.state['next'][in_grid], a.state['next'][in_grid], err_msg=f'{name} step {t}: next')
        want = relabel_obs(a.obs_view(), m, spec.observer, 63)
        np.testing.assert_array_equal(b.obs_view(), want, err_msg=f'{name} step {t}: observations')
    for e in range(spec.n_envs):                    # the observer on its own (bgw_observe's checker), on the final state
        np.testing.assert_array_equal(b.obs_view(b.observe(e)), relabel_obs(a.obs_view(a.observe(e)), m, spec.observer, 63))
    assert resets > 0, 'the run should cross at least one auto-reset'


def test_relabel_helpers_map_rows_and_channels():
    """The helpers themselves: rows and bits move together, stacked channels move and the border stays -1 in all of them."""
    from tests.kat_cases import make_spec, LRN, OBS
    sp = make_spec(3, 3, [dict(enc=1, pos=(0, 0), klass=LRN | OBS, view=1), dict(enc=3, pos=(1, 1), klass=LRN | OBS, view=1)],
                   overlapping={1: {3}}, attack_mapping={3: {1}})
    m = {1: 31, 3: 63}
    s2 = relabel_spec(sp, m)
    assert list(s2.encoding) == [31, 63]
    assert int(s2.overlap[31]) == 1 << 63 and int(s2.overlap[63]) == 1 << 31 and int(s2.attack_map[63]) == 1 << 31
    assert int(s2.overlap[1]) == int(s2.overlap[3]) == int(s2.attack_map[3]) == 0
    v = np.array([[[-1, -1, -1], [0, 2, 0]]], dtype=np.int8)           # one border cell, one cell with two of encoding 2
    got = relabel_obs(v, {1: 5, 2: 9, 3: 40}, K.OBS_STACKED, 40)
    assert got.shape == (1, 2, 40) and (got[0, 0] == -1).all()
    assert got[0, 1, 8] == 2 and np.count_nonzero(got[0, 1]) == 1
    np.testing.assert_array_equal(relabel_obs(np.array([-2, -1, 0, 1, 2], dtype=np.int8), {1: 33, 2: 63}, K.OBS_POSITION_CENTERED, 63),
                                  [-2, -1, 0, 33, 63])
