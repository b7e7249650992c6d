#!/usr/bin/env python
"""What a step program costs: agent-steps/s of one sim through a user step program against the built-in kernels.

    python profiles/program_bench.py [--envs 16384] [--steps 200] [--warmup 20] [--out FILE.jsonl] [--repeat N]

Rows (16384 envs, keyed random policy, device-resident rollout through bgw_rollout_sampled, CUDA-event timing after a
warm-up rollout; auto-reset, horizon 200):
  tb_c2/program            tb_c2's sim (BASELINE configs[1]) through tests/programs/team_battle.c (bgw_set_program)
  tb_c2/general            the same sim on the built-in general kernel (BGW_GENERIC_KERNEL=1)
  tb_c2/general_specialized  ... after bgw_specialize
  tb_c2/default            the kernel bgw_create picks by default (the specialised team-battle kernel)
  foraging/program         abmarl_b200.examples.ForagingSim (ForagingSim.build(): 12x12, 6 foragers, 2 predators, 10 resources)
Every row carries the card's name and power limit; the program rows carry the NVRTC compile time.  --repeat N runs the
list N times (alternating the kernels) to show the spread.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from abmarl_b200 import _capi as K                      # noqa: E402
from abmarl_b200.engine import BatchedGridWorld         # noqa: E402
from abmarl_b200.examples.foraging import ForagingSim   # noqa: E402
from abmarl_b200.spec import compile_sim                # noqa: E402
from tests import program_cases                         # noqa: E402


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
    name, power, clock = [x.strip() for x in q.stdout.strip().split(',')] if q.returncode == 0 else (torch.cuda.get_device_name(0), '?', '?')
    return {'gpu': name, 'power_limit': power, 'max_sm_clock': clock}


def timed(eng, steps, warmup):
    eng.reset()
    eng.rollout_sampled(warmup)
    torch.cuda.synchronize()
    n0 = int(eng.stats()[K.STAT_AGENT_STEPS])
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    eng.rollout_sampled(steps)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b)
    n = int(eng.stats()[K.STAT_AGENT_STEPS]) - n0
    return ms, n


def engines(n_envs):
    """(label, thunk returning (engine, compile seconds or None))"""
    kw = dict(n_envs=n_envs, seed=7, horizon=200, auto_reset=True)
    base, prog = program_cases.specs('tb_c2', **kw)

    def program(spec):
        t0 = time.time()
        eng = BatchedGridWorld(spec, device='cuda:0')                  # bgw_set_program inside
        return eng, time.time() - t0

    def general(specialized):
        os.environ['BGW_GENERIC_KERNEL'] = '1'
        try:
            eng = BatchedGridWorld(base, device='cuda:0')
        finally:
            del os.environ['BGW_GENERIC_KERNEL']
        t0 = time.time()
        if specialized:
            eng.specialize()
        return eng, (time.time() - t0) if specialized else None

    return [('tb_c2/program', lambda: program(prog)),
            ('tb_c2/general', lambda: general(False)),
            ('tb_c2/general_specialized', lambda: general(True)),
            ('tb_c2/default', lambda: (BatchedGridWorld(base, device='cuda:0'), None)),
            ('foraging/program', lambda: program(compile_sim(ForagingSim.build(), **kw)))]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--envs', type=int, default=16384)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=20)
    ap.add_argument('--repeat', type=int, default=1)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("program_bench.py measures on a CUDA device; there is none")
    info = card()
    out = open(args.out, 'a') if args.out else None
    rows = engines(args.envs)
    built = {}
    for rep in range(args.repeat):
        for label, make in rows:
            if label not in built:
                built[label] = make()
            eng, compile_s = built[label]
            ms, n = timed(eng, args.steps, args.warmup)
            rec = dict(info, row=label, repeat=rep, envs=args.envs, learners_per_env=eng.L, entities_per_env=eng.A,
                       steps=args.steps, warmup=args.warmup, ms_per_step=ms / args.steps, agent_steps_per_s=n / (ms * 1e-3),
                       calls='bgw_rollout_sampled', threads_per_env=eng.dims.threads_per_env, compile_seconds=compile_s)
            line = json.dumps(rec)
            print(line, flush=True)
            if out:
                out.write(line + '\n')
    if out:
        out.close()


if __name__ == '__main__':
    main()
