"""Step programs used by the program tests: the re-expressions of built-in sims in tests/programs/ and how to attach them
to a scenario's sim, plus the assembly of a program's run-time kernel source (what bgwjit::build compiles)."""
import os

from abmarl_b200 import _capi as K
from abmarl_b200.program import DeviceProgram
from abmarl_b200.spec import compile_sim
from tests import scenarios

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def program_text(name):
    with open(os.path.join(HERE, 'programs', name + '.c')) as f:
        return f.read()


def reexpression(sim):
    """The DeviceProgram that re-expresses sim's built-in program (team battle, multi maze or pacman), with the constants
    and roles the built-in compilation gives it."""
    builtin = compile_sim(sim)
    rw = [float(x) for x in builtin.reward]
    roles = {agent_id: int(r) for agent_id, r in zip(builtin.agent_ids, builtin.role) if r}
    if builtin.program == K.PROG_TEAM_BATTLE:
        return DeviceProgram(program_text('team_battle'), constants=dict(
            ATTACK_FAIL=rw[K.RW_ATTACK_FAIL], KILL=rw[K.RW_KILL], DIE=rw[K.RW_DIE], MOVE_FAIL=rw[K.RW_MOVE_FAIL],
            ENTROPY=rw[K.RW_ENTROPY]))
    if builtin.program == K.PROG_MULTI_MAZE:
        target = [a for a, r in roles.items() if r == K.ROLE_TARGET][0]
        return DeviceProgram(program_text('multi_maze'), constants=dict(
            TARGET=target, MOVE_FAIL=rw[K.RW_MOVE_FAIL], ENTROPY=rw[K.RW_ENTROPY], REACHED=rw[K.RW_TARGET]),
            roles={a: 1 for a, r in roles.items() if r == K.ROLE_NAVIGATOR})
    if builtin.program == K.PROG_PACMAN:
        return DeviceProgram(program_text('pacman'), constants=dict(
            PACMAN='pacman', BAD_MOVE=rw[K.RW_MOVE_FAIL], ENTROPY=rw[K.RW_ENTROPY], EAT_FOOD=rw[K.RW_EAT_FOOD],
            KILL=rw[K.RW_KILL], DIE=rw[K.RW_DIE]), roles=roles)
    raise ValueError(f"no re-expression of program {builtin.program}")


def with_program(sim):
    """sim with the re-expression of its built-in program as its device_program (an instance attribute)."""
    program = reexpression(sim)
    sim.device_program = lambda: program
    return sim


# the scenarios each re-expression reproduces (their golden transcripts)
TB = [n for n in scenarios.SCENARIOS if n.startswith('tb_')]
MM = [n for n in scenarios.SCENARIOS if n.startswith('mm_') and n != 'mm_dynamic']
PACMAN = ['pacman_c3']
PROGRAM_OF = dict([(n, 'team_battle') for n in TB] + [(n, 'multi_maze') for n in MM] + [(n, 'pacman') for n in PACMAN])


def specs(name, **kw):
    """(built-in spec, program spec) of scenario `name` with the same compile arguments."""
    builder, manager, _ = scenarios.SCENARIOS[name]
    api = scenarios.mirror_api()
    base = compile_sim(builder(api), manager=manager, **kw)
    prog = compile_sim(with_program(builder(api)), manager=manager, **kw)
    assert prog.program == K.PROG_USER and base.program != K.PROG_USER
    return base, prog


# ---- the run-time kernel source of a program, as bgwjit::build (abmarl_b200/csrc/bgw_jit.h) assembles it ------------------
PINS = ('s.H=8;s.W=8;s.HW=64;s.A=24;s.L=24;s.program=7;s.move_actor=1;s.observer=0;s.observe_self=1;s.manager=0;s.ravel=0;'
        's.stacked=0;s.n_blk=0;s.static_mask=nullptr;')


def jit_source(program_source, attack_actor=K.ATTACK_BINARY):
    return ('#define BGW_USER_PROGRAM\n#define BGW_JIT_T 32\n#define BGW_JIT_PIN ' + PINS + '\n#include "bgw_dev.cuh"\n'
            '#include "bgw_program.cuh"\n#line 1 "program"\n' + program_source +
            '\n#define BGWP_AFTER_PROGRAM\n#include "bgw_program.cuh"\n'
            'extern "C" __global__ void __launch_bounds__(32) bgw_step_jit(const DevSpec s_in, const BgwState st, '
            'const uint32_t *actions, const int16_t *order, int8_t *obs, float *reward, uint8_t *done, uint8_t *all_done)\n'
            f'{{ bgw_step_body<7, {attack_actor}>(s_in, st, actions, order, obs, reward, done, all_done); }}\n')


def nvrtc_compile(src):
    """(ok, log, cubin) of compiling `src` for sm_100a with the options of bgwjit::compile_and_load."""
    from cuda.bindings import nvrtc
    err, prog = nvrtc.nvrtcCreateProgram(src.encode(), b'bgw_jit.cu', 0, [], [])
    assert int(err) == 0
    opts = [b'--gpu-architecture=sm_100a', b'-std=c++17', b'--fmad=false', b'-I' + os.path.join(ROOT, 'abmarl_b200', 'csrc').encode(),
            b'-I' + os.path.join(ROOT, 'include').encode(), b'-I/usr/local/cuda/include']
    err, = nvrtc.nvrtcCompileProgram(prog, len(opts), opts)
    _, n = nvrtc.nvrtcGetProgramLogSize(prog)
    log = b' ' * n
    nvrtc.nvrtcGetProgramLog(prog, log)
    cubin = b''
    if int(err) == 0:
        _, size = nvrtc.nvrtcGetCUBINSize(prog)
        cubin = b' ' * size
        nvrtc.nvrtcGetCUBIN(prog, cubin)
    nvrtc.nvrtcDestroyProgram(prog)
    return int(err) == 0, log.decode(errors='replace'), cubin
