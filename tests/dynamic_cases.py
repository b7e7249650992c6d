"""Step programs under the DynamicOrderManager, shared by the CPU and GPU tests: the CPU reference of the rule
(tests/oracle_dynamic/bgw_oracle_dynamic.c over the oracle built with the program), mm_dynamic with multi_maze.c plus its
next_agent hook, the AlternatingBattleSim example, and state comparisons that leave out BGW_ST_NEXT (the goldens and the
built-in rule predate it)."""
import ctypes as C
import hashlib
import os

import numpy as np

from abmarl_b200 import _capi as K
from abmarl_b200.examples import AlternatingBattleSim
from abmarl_b200.program import DeviceProgram
from abmarl_b200.spec import compile_sim
from oracle import build as oracle_build
from oracle.oracle import OracleEnv, _load, _ptr
from tests import program_cases as P
from tests import scenarios
from tests.helpers import assert_state_equal

DYNAMIC_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'oracle_dynamic', 'bgw_oracle_dynamic.c')
_LIBS = {}


def build_dynamic(source):
    """Path of bgw_oracle_dynamic.c built with the step program `source` (a cache entry outside the tree, like
    oracle.build.build_program).  Raises CalledProcessError with gcc's diagnostic when the program does not compile."""
    h = hashlib.sha1(source.encode())
    for f in oracle_build.DEPS + [DYNAMIC_SRC]:
        with open(f, 'rb') as fp:
            h.update(fp.read())
    key = h.hexdigest()[:16]
    d = oracle_build.cache_dir()
    out = os.path.join(d, f'libbgw_dynamic_oracle_{key}.so')
    if os.path.exists(out):
        return out
    prog = os.path.join(d, f'dynamic_program_{key}.c')
    tmp = f'{prog}.{os.getpid()}.tmp'
    with open(tmp, 'w') as fp:
        fp.write(source)
    os.replace(tmp, prog)
    tmp = f'{out}.{os.getpid()}.tmp'
    oracle_build._gcc(DYNAMIC_SRC, tmp, [f'-DBGW_PROGRAM_FILE="{prog}"'])
    os.replace(tmp, out)
    return out


def dynamic_lib(source):
    if source not in _LIBS:
        lib = _load(build_dynamic(source))
        p = C.c_void_p
        lib.bgwo_step_dynamic.argtypes = [C.POINTER(K.BgwSpec), C.POINTER(K.BgwState), p, p, p, p, p, p, p]
        _LIBS[source] = lib
    return _LIBS[source]


class DynamicOracleEnv(OracleEnv):
    """OracleEnv of a step program under the dynamic-order manager: the oracle built with the program plus
    bgwo_step_dynamic, which step() calls."""

    def __init__(self, spec):
        assert spec.program == K.PROG_USER and spec.manager == K.MANAGER_DYNAMIC_ORDER
        super().__init__(spec)
        self._lib = dynamic_lib(spec.program_source)

    def step_rc(self, actions, order=None):
        """bgwo_step_dynamic's return code (non-zero: refused, nothing written)."""
        actions = np.ascontiguousarray(actions, dtype=np.int8)
        assert actions.shape == (self.E, self.L, self.dims.action_stride)
        o = None if order is None else np.ascontiguousarray(order, dtype=np.int16)
        s = self._state_struct()
        return self._lib.bgwo_step_dynamic(C.byref(self._c), C.byref(s), _ptr(actions), _ptr(o), _ptr(self.obs),
                                           _ptr(self.reward), _ptr(self.reward64), _ptr(self.done), _ptr(self.all_done))

    def step(self, actions, order=None):
        assert self.step_rc(actions, order) == 0, "bgwo_step_dynamic refused the step (no next_agent hook?)"
        return self.obs, self.reward, self.done, self.all_done


def oracle_env(spec):
    """The CPU reference of `spec`: DynamicOracleEnv for a step program under the dynamic-order manager, else OracleEnv."""
    if spec.program == K.PROG_USER and spec.manager == K.MANAGER_DYNAMIC_ORDER:
        return DynamicOracleEnv(spec)
    return OracleEnv(spec)


def mm_dynamic_program(sim):
    """The re-expression of DynamicOrderMultiMazeSim: multi_maze.c with the next_agent hook appended."""
    base = P.reexpression(sim)
    program = DeviceProgram(base.source + '\n' + P.program_text('multi_maze_next_agent'), constants=base.constants,
                            roles=base.roles)
    sim.device_program = lambda: program
    return sim


def mm_dynamic_specs(**kw):
    """(built-in spec, program spec) of mm_dynamic with the same compile arguments."""
    builder, manager, _ = scenarios.SCENARIOS['mm_dynamic']
    api = scenarios.mirror_api()
    base = compile_sim(builder(api), manager=manager, **kw)
    prog = compile_sim(mm_dynamic_program(builder(api)), manager=manager, **kw)
    assert prog.program == K.PROG_USER and base.program == K.PROG_MULTI_MAZE
    return base, prog


def battle_spec(n_teams, **kw):
    return compile_sim(AlternatingBattleSim.build(rows=8, cols=8, n_teams=n_teams, team_size=3), manager='dynamic_order', **kw)


def without_next(state):
    """A copy of `state` with BGW_ST_NEXT cleared in flags."""
    out = dict(state)
    out['flags'] = np.asarray(state['flags']) & np.uint8(~K.ST_NEXT & 0xFF)
    return out


def assert_state_equal_but_next(a, b, where):
    assert_state_equal(without_next(a), without_next(b), where)


def acting(spec, state):
    """bool [E, L]: who acts in the next step (DynamicOrderManager.acting), from a host state."""
    flags = np.asarray(state['flags'])[:, spec.learner_agents]
    by_turn = np.arange(spec.n_learners)[None, :] == np.asarray(state['turn']).astype(np.int64)[:, None]
    named = np.where((np.asarray(state['step']) == 0)[:, None], by_turn, (flags & K.ST_NEXT) != 0)
    live = (np.asarray(state['env_flags']) & K.ENV_ALL_DONE) == 0
    return named & ((flags & K.ST_DONE_REPORTED) == 0) & live[:, None]
