"""The specialised kernel's ordering machinery (reservation rounds, touch bit maps, tickets, per-env stamps) under perturbed
interleavings: the -DBGW_JITTER build (abmarl_b200/csrc/bgw_fast.cuh; built by __graft_entry__.build() as libbgw_jitter.so)
sleeps a pseudo-random 0..2 us before every reservation, table look-up, ticket draw and stamp access.  The parity tests that
exercise that machinery must pass unchanged under it.  (compute-sanitizer racecheck is closed on this pool.)"""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, 'abmarl_b200', 'csrc', 'libbgw_jitter.so')


@pytest.mark.skipif(not os.path.exists(LIB), reason='libbgw_jitter.so not built (python __graft_entry__.py)')
def test_parity_under_the_jitter_build():
    env = dict(os.environ, BGW_LIB=LIB)
    sel = 'rollout or chained or full_size or step_sampled or cuda_graph or tb_c5 or tb_c2 or tb_dense or aliased or epochs'
    # the structured policies: long reservation rounds and long occupant lists (the general kernel has no jitter points)
    for path, k in (('test_gpu_parity.py', sel), ('test_gpu_policies.py', 'not general')):
        r = subprocess.run([sys.executable, '-m', 'pytest', os.path.join(ROOT, 'tests', path), '-x', '-q', '-k', k],
                           env=env, cwd=ROOT, capture_output=True, text=True, timeout=1200)
        assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
        assert ' passed' in r.stdout
