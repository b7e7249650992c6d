"""ctypes front-end of the C oracle (oracle/bgw_oracle.c).  TEST INFRASTRUCTURE ONLY.

OracleEnv mirrors abmarl_b200.engine.BatchedGridWorld on numpy arrays so the parity tests can drive both
with the same code and compare array for array.  A spec with a step program (CompiledSpec.program_source) runs on the
oracle built with that program (build_program).
"""
import ctypes as C

import numpy as np

from abmarl_b200 import _capi as K
from oracle.build import build, build_program

_LIBS = {}          # program source (None: the plain oracle) -> loaded library


def _load(path):
    lib = C.CDLL(path)
    p = C.c_void_p
    lib.bgwo_dims.argtypes = [C.POINTER(K.BgwSpec), C.POINTER(K.BgwDims)]
    lib.bgwo_reset.argtypes = [C.POINTER(K.BgwSpec), C.POINTER(K.BgwState), p, p]
    lib.bgwo_step.argtypes = [C.POINTER(K.BgwSpec), C.POINTER(K.BgwState), p, p, p, p, p, p, p]
    lib.bgwo_sample_actions.argtypes = [C.POINTER(K.BgwSpec), C.POINTER(K.BgwState), p]
    lib.bgwo_los_mask.argtypes = [C.c_int, C.c_int, C.c_int, p]
    lib.bgwo_observe.argtypes = [C.POINTER(K.BgwSpec), C.POINTER(K.BgwState), C.c_int, p]
    return lib


def lib(program_source=None):
    """The plain oracle, or the oracle built with a step program."""
    if program_source not in _LIBS:
        _LIBS[program_source] = _load(build() if program_source is None else build_program(program_source))
    return _LIBS[program_source]


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


STATE_FIELDS = (('cell', np.uint16, 'EA'), ('next', np.uint16, 'EA'), ('flags', np.uint8, 'EA'),
                ('health', np.float64, 'EA'), ('reward_acc', np.float64, 'EA'), ('episode', np.uint32, 'E'),
                ('step', np.uint32, 'E'), ('env_flags', np.uint8, 'E'), ('turn', np.int16, 'E'),
                ('error', np.uint32, 'E'))


def alloc_state(E, A):
    """Fresh numpy state in the layout of BgwState (include/bgw.h)."""
    st = {}
    for name, dt, shape in STATE_FIELDS:
        st[name] = np.zeros((E, A) if shape == 'EA' else (E,), dtype=dt)
    st['cell'][:] = K.BGW_NONE
    st['next'][:] = K.BGW_NONE
    st['episode'][:] = 0xFFFFFFFF
    st['turn'][:] = -1
    st['stats'] = np.zeros((E, K.BGW_STAT_COUNT), dtype=np.uint64)
    st['layout'] = None
    st['ammo'] = np.zeros((E, A), dtype=np.int32)
    return st


def los_mask(rng, rd, cd):
    n = 2 * rng + 1
    out = np.empty((n, n), dtype=np.uint8)
    lib().bgwo_los_mask(rng, rd, cd, _ptr(out))
    return out


class OracleEnv:
    def __init__(self, spec):
        self.spec = spec
        self._c = spec.c_struct()
        self._lib = lib(spec.program_source)
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

    def _state_struct(self):
        s = K.BgwState()
        for name in ('cell', 'next', 'flags', 'health', 'reward_acc', 'episode', 'step', 'env_flags', 'turn',
                     'error', 'layout', 'stats', 'ammo'):
            setattr(s, name, _ptr(self.state[name]))
        return s

    def set_layout(self, layout):
        self.state['layout'] = None if layout is None else np.ascontiguousarray(layout, dtype=np.uint16)

    def reset(self, env_mask=None):
        m = None if env_mask is None else np.ascontiguousarray(env_mask, dtype=np.uint8)
        s = self._state_struct()
        self._lib.bgwo_reset(C.byref(self._c), C.byref(s), _ptr(m), _ptr(self.obs))
        return self.obs

    def sample_actions(self):
        act = np.zeros((self.E, self.L, self.dims.action_stride), dtype=np.int8)
        s = self._state_struct()
        self._lib.bgwo_sample_actions(C.byref(self._c), C.byref(s), _ptr(act))
        return act

    def step(self, actions, order=None):
        actions = np.ascontiguousarray(actions, dtype=np.int8)
        assert actions.shape == (self.E, self.L, self.dims.action_stride)
        o = None if order is None else np.ascontiguousarray(order, dtype=np.int16)
        s = self._state_struct()
        rc = self._lib.bgwo_step(C.byref(self._c), C.byref(s), _ptr(actions), _ptr(o), _ptr(self.obs), _ptr(self.reward),
                                 _ptr(self.reward64), _ptr(self.done), _ptr(self.all_done))
        assert rc == 0, "the oracle runs a step program under the all-step and turn-based managers only"
        return self.obs, self.reward, self.done, self.all_done

    def observe(self, env=0):
        out = np.zeros((self.L, self.dims.obs_stride), dtype=np.int8)
        s = self._state_struct()
        self._lib.bgwo_observe(C.byref(self._c), C.byref(s), env, _ptr(out))
        return out

    # ---- helpers shared with the tests ---------------------------------------------------------
    def obs_view(self, obs=None):
        """[E, L, h, w(, c)] logical view of the padded int8 rows."""
        obs = self.obs if obs is None else obs
        d = self.dims
        v = obs[..., :d.obs_h * d.obs_w * d.obs_c]
        shape = obs.shape[:-1] + ((d.obs_h, d.obs_w) if d.obs_c == 1 else (d.obs_h, d.obs_w, d.obs_c))
        return v.reshape(shape)
