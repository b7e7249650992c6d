"""The CPU reference of a step program with variables (tests/oracle_vars/bgw_oracle_vars.c over the oracle built with the
program and its dynamic-order manager step), wrapped as VarsOracleEnv: OracleEnv plus state['program_vars'] and
program_vars(), as BatchedGridWorld keeps them."""
import ctypes as C
import hashlib
import os

import numpy as np

from abmarl_b200 import _capi as K
from oracle import build as oracle_build
from oracle.oracle import OracleEnv, _load, _ptr, alloc_state
from tests.dynamic_cases import DYNAMIC_SRC

VARS_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'oracle_vars', 'bgw_oracle_vars.c')
_LIBS = {}


def build_vars(source):
    """Path of bgw_oracle_vars.c built with the step program `source` (a cache entry outside the tree).  Raises
    CalledProcessError with gcc's diagnostic when the program does not compile."""
    h = hashlib.sha1(source.encode())
    for f in oracle_build.DEPS + [DYNAMIC_SRC, VARS_SRC]:
        with open(f, 'rb') as fp:
            h.update(fp.read())
    key = h.hexdigest()[:16]
    d = oracle_build.cache_dir()
    out = os.path.join(d, f'libbgw_vars_oracle_{key}.so')
    if os.path.exists(out):
        return out
    prog = os.path.join(d, f'vars_program_{key}.c')
    tmp = f'{prog}.{os.getpid()}.tmp'
    with open(tmp, 'w') as fp:
        fp.write(source)
    os.replace(tmp, prog)
    tmp = f'{out}.{os.getpid()}.tmp'
    oracle_build._gcc(VARS_SRC, tmp, [f'-DBGW_PROGRAM_FILE="{prog}"'])
    os.replace(tmp, out)
    return out


def vars_lib(source):
    if source not in _LIBS:
        lib = _load(build_vars(source))
        p = C.c_void_p
        lib.bgwo_bind_program_vars.argtypes = [C.c_int, C.c_int, p, p]
        lib.bgwo_reset_vars.argtypes = lib.bgwo_reset.argtypes
        lib.bgwo_step_vars.argtypes = lib.bgwo_step.argtypes
        _LIBS[source] = lib
    return _LIBS[source]


class VarsOracleEnv(OracleEnv):
    """OracleEnv of a step program (any manager) whose variables live in state['program_vars'], float64
    [E, n_env_vars + A * n_agent_vars]; every reset and step binds them first."""

    def __init__(self, spec):
        # OracleEnv.__init__ with this library instead of the plain program build, which lacks the variables' API
        assert spec.program_source is not None
        self.spec = spec
        self._c = spec.c_struct()
        self._lib = vars_lib(spec.program_source)
        d = K.BgwDims()
        self._lib.bgwo_dims(C.byref(self._c), C.byref(d))
        self.dims = d
        self.E, self.A, self.L = spec.n_envs, spec.n_agents, d.n_learners
        self.state = alloc_state(self.E, self.A)
        self.obs = np.zeros((self.E, self.L, d.obs_stride), dtype=np.int8)
        self.reward = np.zeros((self.E, self.L), dtype=np.float32)
        self.reward64 = np.zeros((self.E, self.L), dtype=np.float64)
        self.done = np.zeros((self.E, self.L), dtype=np.uint8)
        self.all_done = np.zeros(self.E, dtype=np.uint8)
        init = spec.program_var_init
        self._init = None if init is None else np.ascontiguousarray(init, dtype=np.float64)
        self.state['program_vars'] = None if init is None else np.zeros((self.E, init.size), dtype=np.float64)

    def _bind_vars(self):
        self._lib.bgwo_bind_program_vars(self.spec.n_env_vars, len(self.spec.agent_var_names), _ptr(self._init),
                                         _ptr(self.state['program_vars']))

    def reset(self, env_mask=None):
        self._bind_vars()
        m = None if env_mask is None else np.ascontiguousarray(env_mask, dtype=np.uint8)
        s = self._state_struct()
        self._lib.bgwo_reset_vars(C.byref(self._c), C.byref(s), _ptr(m), _ptr(self.obs))
        return self.obs

    def step(self, actions, order=None):
        actions = np.ascontiguousarray(actions, dtype=np.int8)
        assert actions.shape == (self.E, self.L, self.dims.action_stride)
        o = None if order is None else np.ascontiguousarray(order, dtype=np.int16)
        self._bind_vars()
        s = self._state_struct()
        rc = self._lib.bgwo_step_vars(C.byref(self._c), C.byref(s), _ptr(actions), _ptr(o), _ptr(self.obs),
                                      _ptr(self.reward), _ptr(self.reward64), _ptr(self.done), _ptr(self.all_done))
        assert rc == 0, "the oracle refused the step (a dynamic-order program without a next_agent hook?)"
        return self.obs, self.reward, self.done, self.all_done

    def observe(self, env=0):
        self._bind_vars()
        return super().observe(env)

    def program_vars(self):
        """{name: view} of the program's variables, as BatchedGridWorld.program_vars ({} without)."""
        rows = self.state['program_vars']
        return {} if rows is None else self.spec.program_var_views(rows)
