"""Fused rollouts whose tickets are blocks of consecutive steps of one env (bgw_fast.cuh, "env tickets and chained
launches"): inside a block the env stays on its CTA with its rows, summary grid and occupant lists in shared memory.  Block
boundaries against episode ends at every offset -- horizons and rollout lengths around the block length, episodes that end
before the horizon (OneTeamRemainingDone), sims with mixed cells, batches below and above the resident CTA count, no
auto-reset -- against separate step_sampled calls over the whole batch and against the oracle on env slices."""
import numpy as np
import pytest
import torch

from abmarl_b200 import _capi as K
from abmarl_b200.spec import compile_sim
from tests import scenarios
from tests.helpers import assert_state_equal

pytestmark = pytest.mark.gpu

# rollout lengths: 1 and the neighbours of the block lengths 2, 4, 8 and 16 and of three blocks and a bit
LENGTHS = (1, 3, 4, 5, 7, 8, 9, 2, 15, 16, 17, 26, 50)


# (BGW_GRID: a grid of 5 CTAs puts 24 envs above the resident CTA count, where the block length follows the rollout length)
@pytest.mark.parametrize('name,n_envs,horizon,auto_reset,grid', [
    ('tb_c5_small', 24, 1, True, None), ('tb_c5_small', 24, 2, True, None), ('tb_c5_small', 24, 15, True, None),
    ('tb_c5_small', 24, 16, True, None), ('tb_c5_small', 24, 17, True, None),
    ('tb_c5_small', 24, 3, True, '5'), ('tb_c5_small', 24, 5, True, '5'),
    ('tb_c5_small', 2500, 7, True, None), ('tb_c5_small', 2500, 16, True, None),
    ('tb_c2', 24, 8, True, None), ('tb_c2', 2500, 30, True, None),
    ('tb_dense', 24, 40, True, None), ('tb_dense', 2500, 40, True, None),
    ('tb_stacked', 24, 9, True, None), ('tb_stacked', 2500, 25, True, None),
    ('tb_c5_small', 24, 6, False, None), ('tb_dense', 24, 40, False, None),
])
def test_rollout_blocks_against_separate_steps_and_oracle(mirror, monkeypatch, name, n_envs, horizon, auto_reset, grid):
    if grid:
        monkeypatch.setenv('BGW_GRID', grid)
    from abmarl_b200.engine import BatchedGridWorld
    from oracle.oracle import OracleEnv
    builder, manager, _ = scenarios.SCENARIOS[name]
    spec = compile_sim(builder(mirror), manager=manager, n_envs=n_envs, env_offset=3, seed=0xB10C, horizon=horizon,
                       auto_reset=auto_reset)
    E, S = n_envs, 3
    a, b = BatchedGridWorld(spec, device='cuda:0'), BatchedGridWorld(spec, device='cuda:0')
    head, tail = OracleEnv(spec.with_envs(S, spec.env_offset)), OracleEnv(spec.with_envs(S, spec.env_offset + E - S))
    for x in (a, b, head, tail):
        x.reset()
    early_end = False                                     # some episode ended before the horizon (OneTeamRemainingDone)
    done_steps = 0
    for n in LENGTHS:
        a.rollout_sampled(n)
        for _ in range(n):
            b.step_sampled()
            fl = b.all_done.cpu().numpy()
            early_end |= bool(np.any((fl & K.ENV_ALL_DONE) & ~(fl & (K.ENV_TRUNCATED | K.ENV_RESET))))
            for o in (head, tail):
                o.step(o.sample_actions())
        done_steps += n
        for k in ('obs', 'reward', 'done', 'all_done', 'actions'):
            assert torch.equal(getattr(a, k), getattr(b, k)), (done_steps, k)
        st = a.state_numpy()
        assert_state_equal(st, b.state_numpy(), f'{name} after {done_steps} steps')
        assert torch.equal(a.stats(), b.stats())
        for o, sl in ((head, slice(0, S)), (tail, slice(E - S, E))):
            for k in ('obs', 'done', 'reward', 'all_done'):
                assert np.array_equal(getattr(a, k)[sl].cpu().numpy(), getattr(o, k)), (done_steps, k)
            assert_state_equal({k: (None if v is None else v[sl]) for k, v in st.items()}, o.state, f'oracle {done_steps}')
    if name == 'tb_dense':
        assert early_end, 'tb_dense is the case whose episodes end inside a block, before the horizon'
