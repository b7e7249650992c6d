"""Build the CPU oracle with gcc.  Test infrastructure only.

build() compiles oracle/bgw_oracle.c into oracle/libbgw_oracle.so.  build_program(source) compiles the oracle with a step
program (oracle/bgw_oracle_program.c) into a shared object named by the hash of the program and the sources, in a cache
directory outside the tree.
"""
import hashlib
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SRC = os.path.join(HERE, 'bgw_oracle.c')
PROGRAM_SRC = os.path.join(HERE, 'bgw_oracle_program.c')
OUT = os.path.join(HERE, 'libbgw_oracle.so')
DEPS = [SRC, PROGRAM_SRC, os.path.join(HERE, 'bgw_oracle.h')] + \
    [os.path.join(ROOT, 'include', h) for h in ('bgw.h', 'bgw_philox.h', 'bgw_program.h', 'bgw_stdint.h')]
# -ffp-contract=off: float64 arithmetic is never fused (the line-of-sight rays are (a/b)*t, utils.py:45-115);
# -Werror=discarded-qualifiers: a program's get_done / get_all_done / get_reward hook that calls a mutating API function fails
FLAGS = ['-O2', '-fPIC', '-shared', '-ffp-contract=off', '-fno-fast-math', '-Werror=discarded-qualifiers']


def _gcc(src, out, defines=()):
    """Raises CalledProcessError, gcc's diagnostic in .stderr and on stderr, when `src` does not compile."""
    r = subprocess.run(['gcc'] + FLAGS + list(defines) + ['-o', out, src, '-lm'], capture_output=True, text=True)
    if r.returncode:
        sys.stderr.write(r.stderr)
        raise subprocess.CalledProcessError(r.returncode, r.args, r.stdout, r.stderr)


def build(force=False):
    if not force and os.path.exists(OUT) and all(os.path.getmtime(OUT) >= os.path.getmtime(d) for d in DEPS):
        return OUT
    _gcc(SRC, OUT)
    return OUT


def cache_dir():
    """$BGW_ORACLE_CACHE, else a per-user directory under the system temp directory (never the source tree)."""
    d = os.environ.get('BGW_ORACLE_CACHE') or os.path.join(tempfile.gettempdir(), f'bgw_oracle_{os.getuid()}')
    os.makedirs(d, exist_ok=True)
    return d


def build_program(source):
    """Path of the oracle built with the step program `source`."""
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
    _gcc(PROGRAM_SRC, tmp, [f'-DBGW_PROGRAM_FILE="{prog}"'])
    os.replace(tmp, out)
    return out


if __name__ == '__main__':
    print(build(force=True))
