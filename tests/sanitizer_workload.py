import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from tests import scenarios
from abmarl_b200.spec import compile_sim
from abmarl_b200.engine import BatchedGridWorld
from oracle.oracle import OracleEnv
from tests.helpers import run_lockstep
api = scenarios.mirror_api()
for name, E, steps in (('tb_c5_small', 4, 12), ('tb_dense', 4, 30), ('tb_blocking', 3, 8), ('maze_c1', 2, 6), ('mm_tiny', 3, 20)):
    b, m, _ = scenarios.SCENARIOS[name]
    spec = compile_sim(b(api), manager=m, n_envs=E, seed=5, horizon=10, auto_reset=True)
    run_lockstep(BatchedGridWorld(spec, device='cuda:0'), OracleEnv(spec), steps, label=name)
spec = compile_sim(scenarios.build_tb_c5(api), n_envs=3, seed=5, horizon=6, auto_reset=True)
run_lockstep(BatchedGridWorld(spec, device='cuda:0'), OracleEnv(spec), 9, label='tb_c5')
torch.cuda.synchronize()
print('sanitizer workload ok')
