"""The CPU oracle with a user step program compiled in (tests/program_oracle.c).  TEST INFRASTRUCTURE ONLY.

build_program(source) compiles the oracle with the program into a shared object named by the hash of the program and the
sources, in a cache directory outside the tree; ProgramOracleEnv(spec) is oracle.oracle.OracleEnv over that library for a
spec compiled from a sim with a device_program() (CompiledSpec.program_source).
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from abmarl_b200 import _capi as K
from oracle.oracle import OracleEnv, _ptr

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SRC = os.path.join(HERE, 'program_oracle.c')
# the flags of oracle/build.py (-ffp-contract=off: float64 arithmetic is never fused), plus the const check of the hooks
FLAGS = ['-O2', '-fPIC', '-shared', '-ffp-contract=off', '-fno-fast-math', '-Werror=discarded-qualifiers']
DEPS = [SRC, os.path.join(ROOT, 'oracle', 'bgw_oracle.c'), os.path.join(ROOT, 'oracle', 'bgw_oracle.h')] + \
    [os.path.join(ROOT, 'include', h) for h in ('bgw.h', 'bgw_philox.h', 'bgw_program.h', 'bgw_stdint.h')]

_LIBS = {}


def cache_dir():
    """$BGW_ORACLE_CACHE, else a per-user directory under the system temp directory (never the source tree)."""
    d = os.environ.get('BGW_ORACLE_CACHE') or os.path.join(tempfile.gettempdir(), f'bgw_oracle_{os.getuid()}')
    os.makedirs(d, exist_ok=True)
    return d


def build_program(source):
    """Path of the oracle built with `source`.  Raises CalledProcessError (gcc's diagnostic in .stderr) when it does not compile."""
    h = hashlib.sha1(source.encode())
    for f in DEPS:
        with open(f, 'rb') as fp:
            h.update(fp.read())
    key = h.hexdigest()[:16]
    d = cache_dir()
    out = os.path.join(d, f'libbgw_program_oracle_{key}.so')
    if os.path.exists(out):
        return out
    prog = os.path.join(d, f'program_{key}.c')
    tmp = f'{prog}.{os.getpid()}.tmp'            # concurrent builders: each writes its own files, the renames are atomic
    with open(tmp, 'w') as fp:
        fp.write(source)
    os.replace(tmp, prog)
    tmp = f'{out}.{os.getpid()}.tmp'
    subprocess.run(['gcc'] + FLAGS + [f'-DBGW_PROGRAM_FILE="{prog}"', '-o', tmp, SRC, '-lm'],
                   check=True, capture_output=True, text=True)
    os.replace(tmp, out)
    return out


def program_lib(source):
    if source not in _LIBS:
        lib = C.CDLL(build_program(source))
        p = C.c_void_p
        lib.bgwo_reset.argtypes = [C.POINTER(K.BgwSpec), C.POINTER(K.BgwState), p, p]
        lib.bgwo_step.argtypes = [C.POINTER(K.BgwSpec), C.POINTER(K.BgwState), p, p, p, p, p, p, p]
        lib.bgwo_sample_actions.argtypes = [C.POINTER(K.BgwSpec), C.POINTER(K.BgwState), p]
        lib.bgwo_observe.argtypes = [C.POINTER(K.BgwSpec), C.POINTER(K.BgwState), C.c_int, p]
        _LIBS[source] = lib
    return _LIBS[source]


class ProgramOracleEnv(OracleEnv):
    """OracleEnv whose step runs the spec's step program (the same text the engine compiles with bgw_set_program)."""

    def __init__(self, spec):
        assert spec.program_source is not None, "ProgramOracleEnv needs a spec with a step program"
        super().__init__(spec)
        self._lib = program_lib(spec.program_source)

    def reset(self, env_mask=None):
        m = None if env_mask is None else np.ascontiguousarray(env_mask, dtype=np.uint8)
        self._lib.bgwo_reset(C.byref(self._c), C.byref(self._state_struct()), _ptr(m), _ptr(self.obs))
        return self.obs

    def sample_actions(self):
        act = np.zeros((self.E, self.L, self.dims.action_stride), dtype=np.int8)
        self._lib.bgwo_sample_actions(C.byref(self._c), C.byref(self._state_struct()), _ptr(act))
        return act

    def step(self, actions, order=None):
        actions = np.ascontiguousarray(actions, dtype=np.int8)
        assert actions.shape == (self.E, self.L, self.dims.action_stride)
        o = None if order is None else np.ascontiguousarray(order, dtype=np.int16)
        rc = self._lib.bgwo_step(C.byref(self._c), C.byref(self._state_struct()), _ptr(actions), _ptr(o), _ptr(self.obs),
                                 _ptr(self.reward), _ptr(self.reward64), _ptr(self.done), _ptr(self.all_done))
        assert rc == 0, "the program oracle runs BGW_PROG_USER specs under the all-step and turn-based managers"
        return self.obs, self.reward, self.done, self.all_done

    def observe(self, env=0):
        out = np.zeros((self.L, self.dims.obs_stride), dtype=np.int8)
        self._lib.bgwo_observe(C.byref(self._c), C.byref(self._state_struct()), env, _ptr(out))
        return out
