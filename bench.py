#!/usr/bin/env python
"""bench.py -- agent-steps/sec of the batched GridWorld step path (BASELINE.json metric).

Workload (BASELINE.json configs[4], SURVEY.md section 8(d) "C5"): synthetic team battle, 64x64 grid, 256
agents/env (4 teams), view range 5, move/attack range 1, random placement and random initial health,
OneTeamRemainingDone, AllStepManager semantics, horizon 200 with auto-reset, random actions from the keyed
Philox stream; 4096 envs per GPU (env batches shard across GPUs with no data-path collective -> weak scaling;
NCCL only sums the episode statistics).

One "step" = one manager step of every env on this GPU, in which the keyed random policy draws every acting learner's
action (actor resolution -> observation -> reward/done); the K timed steps are enqueued by ONE bgw_rollout_sampled call
(= K x bgw_step_sampled; on the specialised kernel one launch whose CTAs draw (step, env) tickets).  An agent-step = one
learning agent receiving (obs, reward, done).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Prints ONE JSON line on rank 0.  With --dump-outputs, rank 0 also writes what the last timed step returned (see
dump_outputs): the inputs depend on the arguments alone, so two builds run with the same arguments can be compared output
for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "agent-steps/sec (obs+reward+done) over batched envs"
BYTES_PER_AGENT_STEP = 165     # SURVEY.md 8(d): action 4 + int8 obs 128 + reward 4 + done 1 + agent state r/w 28
ENVS_PER_GPU = 4096
WORKLOAD = "synthetic team battle 64x64, 256 agents/env, view 5, horizon 200 (BASELINE configs[4])"


def build_spec(n_envs, env_offset, seed=0xB200):
    from abmarl_b200.examples.workloads import headline_spec
    return headline_spec(n_envs, env_offset, seed=seed)


def workload_config(world, envs_per_gpu=ENVS_PER_GPU):
    """The workload both arms run, as ONE dict (the driver compares the two arms' `config`)."""
    return {"workload": WORKLOAD, "envs_per_gpu": envs_per_gpu, "agents_per_env": 256, "global_envs": envs_per_gpu * world,
            "parallelism": f"env-sharded x{world}, no data-path collective",
            "l2": "working set per step (obs 134 MB + actions/state 10 MB per GPU) exceeds the 126 MB L2"}


# the reference itself (pure Python) cannot travel to the GPU box; its single-core figure for this workload was measured in
# the survey container (BASELINE.md section 2) and is quoted next to the C port's, which is what runs here
PYTHON_REFERENCE_PER_CORE = {"value": 3.8e3, "unit": "agent-steps/s", "where": "survey container, one core, unmodified reference AllStepManager loop (BASELINE.md section 2); not measured in this run"}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '50'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(',')] + [time.perf_counter()])
        except Exception:
            pass

    def stop(self, t0=None, t1=None):
        """Summary of the samples read between host times t0 and t1 (the measured period); all samples if too few."""
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=2)
        rows = [r for r in self.rows if len(r) >= 10]
        inside = [r for r in rows if t0 is not None and t0 - 0.06 <= r[-1] <= t1 + 0.06]
        if len(inside) >= 2:
            rows = inside
        sm = [float(r[1]) for r in rows if r[1].replace('.', '').isdigit()]
        mx = [float(r[2]) for r in rows if r[2].replace('.', '').isdigit()]
        names = ('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap')
        reasons = sorted({n for r in rows for n, v in zip(names, r[5:9]) if v.lower().startswith('active')})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "period_ms": 50}


DUMP_ENVS = 256                 # envs of the --dump-outputs sample: obs of 256 envs x 256 learners x 11x11 in float32 = 32 MB


def dump_outputs(eng, out_dir, n_envs=DUMP_ENVS):
    """Write to `out_dir`/<name>.npy what the caller of the timed path receives after its last step -- obs (the logical
    [h, w] view of the padded rows), reward, done, all_done and the sampled actions -- for a fixed, seeded sample of
    `n_envs` envs (all envs if there are fewer; their indices in env_index.npy), and the episode statistics summed over all
    envs (stats.npy: agent_steps, episodes, kills, env_steps).  float32, or float64 where float32 would round."""
    import torch
    envs = np.sort(np.random.default_rng(0xB200).choice(eng.E, size=min(eng.E, n_envs), replace=False))
    idx = torch.from_numpy(envs).to(eng.device)
    pick = lambda t: t.index_select(0, idx).cpu().numpy().astype(np.float32)
    arrays = {'env_index': envs.astype(np.float64), 'obs': pick(eng.obs_view()), 'reward': pick(eng.reward),
              'done': pick(eng.done), 'all_done': pick(eng.all_done), 'actions': pick(eng.actions),
              'stats': eng.stats().cpu().numpy().astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def measured_peak():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


# ---------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's AllStepManager loop on the host cores
# ---------------------------------------------------------------------------------------------------
def cpu_rollout(n_envs, steps, threads, warmup=0):
    """The C oracle (oracle/bgw_oracle.c: scalar restatement of the reference's per-agent loops) on `threads`
    host threads, each advancing its own shard of envs.  Returns (agent_steps, seconds)."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle.oracle import OracleEnv
    from abmarl_b200 import _capi as K
    threads = max(1, min(threads, n_envs))
    sizes = [n_envs // threads + (1 if i < n_envs % threads else 0) for i in range(threads)]
    offs = [sum(sizes[:i]) for i in range(threads)]
    envs = [OracleEnv(build_spec(sz, off)) for sz, off in zip(sizes, offs)]

    def work(o, n):
        before = int(o.state['stats'][:, K.STAT_AGENT_STEPS].sum())
        for _ in range(n):
            o.step(o.sample_actions())
        return int(o.state['stats'][:, K.STAT_AGENT_STEPS].sum()) - before

    with ThreadPoolExecutor(threads) as pool:        # ctypes releases the GIL inside the C calls
        list(pool.map(lambda o: o.reset(), envs))
        if warmup:
            list(pool.map(lambda o: work(o, warmup), envs))
        t0 = time.perf_counter()
        n = sum(pool.map(lambda o: work(o, steps), envs))
        dt = time.perf_counter() - t0
    return n, dt, n_envs


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    world = int(os.environ.get('WORLD_SIZE', '1'))
    cores = len(os.sched_getaffinity(0))
    # the same workload as the GPU arm: every step advances all 4096 envs (sharded over the host threads), starting from the
    # same reset state; a step is ~0.55 M agent-steps, a few tens of milliseconds on 16 threads
    n, dt, envs = cpu_rollout(args.envs_per_gpu, args.steps, cores, warmup=args.warmup)
    value = n / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "agent-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "i8/f64", "data": "synthetic",
        "config": workload_config(world, args.envs_per_gpu),
        "agent_steps_per_step": n / max(args.steps, 1),
        "cpu_baseline": {"value": value, "unit": "agent-steps/s", "cores": cores, "kind": "port",
                         "sample": f"oracle C port of the reference loop, {envs} envs x {args.steps} steps on {cores} host threads",
                         "python_reference_per_core": PYTHON_REFERENCE_PER_CORE},
        "e2e": {"value": value, "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from abmarl_b200 import _capi as K
    from abmarl_b200.engine import BatchedGridWorld

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)

    E = args.envs_per_gpu
    eng = BatchedGridWorld(build_spec(E, rank * E), device=dev)
    L = eng.L
    stream = torch.cuda.current_stream(dev)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def agent_steps():
        return int(eng.stats()[K.STAT_AGENT_STEPS].item())

    # ---------------- device-resident rollout: `value` + roofline of the step kernel -----------------
    # clocks / throttle reasons are sampled from before the warm-up until after the end-to-end loop (50 ms period):
    # the timed regions are tens of milliseconds long, so the samples taken while the GPU is busy bracket them
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.5)
    # bring the GPU out of its idle power state before anything is measured: about 50 ms of the same kernel on the same engine,
    # then a fresh reset -- the W warm-up steps and the K timed steps below are steps 0..W+K of the episode that starts there
    # (a 20-step timed region is one millisecond: without this it runs while the clocks are still ramping, measured 5 % jitter)
    eng.reset()
    eng.rollout_sampled(args.spinup_steps)
    torch.cuda.synchronize(dev)
    eng.reset()
    def rollout(n):
        # bgw_rollout_sampled: n step launches enqueued by the library back to back (chained per env); --per-step-calls
        # makes one bgw_step_sampled call per step instead (launches serialised by griddepcontrol.wait)
        if args.per_step_calls:
            for _ in range(n):
                eng.step_sampled()
        else:
            eng.rollout_sampled(n)

    rollout(args.warmup)
    barrier()
    n0, launches0 = agent_steps(), eng.launches
    host_t0 = time.perf_counter()
    # The timed region holds nothing but the K step launches between two events: consecutive launches are programmatic
    # dependent launches chained per env (launch k+1 starts an env once launch k has finished that env; its
    # env-independent set-up overlaps launch k's tail), which an event record between them would serialise.  The step kernel's average launch duration over the timed region is
    # therefore region / launches (one launch per step); `kernel_ms_isolated` is the same kernel bracketed by its own
    # events on every launch in a second pass of the same workload (serialised launches, --kernel-steps of them).
    t_beg, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_beg.record(stream)
    rollout(args.steps)                               # keyed random policy + manager step, one launch per step
    t_end.record(stream)
    barrier()
    ms = t_beg.elapsed_time(t_end)
    n_dev = agent_steps() - n0
    launches = eng.launches - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(eng, args.dump_outputs)
    kernel_ms = ms
    ks = max(1, min(args.kernel_steps, args.steps))
    k_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(ks)]
    n_iso0 = agent_steps()
    for i in range(ks):
        k_ev[i][0].record(stream)
        eng.step_sampled()
        k_ev[i][1].record(stream)
    barrier()
    per_step_ms = [a.elapsed_time(b) for a, b in k_ev]
    iso_ms_per_launch = sum(per_step_ms) / ks
    iso_units_per_launch = (agent_steps() - n_iso0) / ks
    # the call an RL trainer makes: bgw_step with a caller-supplied, device-resident action tensor (one launch per step,
    # programmatic dependent launches, no fused policy); actions from a pool of pre-drawn random tensors of the same ranges
    gs = max(1, min(args.given_steps, args.steps))
    gpool = []
    for i in range(8):
        a = torch.zeros((E, L, eng.action_stride), dtype=torch.int8, device=dev)
        a[..., 0:2] = torch.randint(-1, 2, (E, L, 2), device=dev, dtype=torch.int8)
        a[..., 2] = torch.randint(0, 2, (E, L), device=dev, dtype=torch.int8)
        gpool.append(a)
    for i in range(3):
        eng.step(gpool[i])
    barrier()
    n_g0 = agent_steps()
    g_beg, g_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g_beg.record(stream)
    for i in range(gs):
        eng.step(gpool[i % 8])
    g_end.record(stream)
    barrier()
    given_ms_per_step = g_beg.elapsed_time(g_end) / gs
    given_units_per_step = (agent_steps() - n_g0) / gs
    # the observer on its own (bgw_observe = sim.get_obs of every learner on the state as it stands): the bandwidth-bound piece
    # of the path (SURVEY 8(d) "K3"); every launch writes E*L rows of obs_stride bytes (more than the L2) and reads 3 bytes of
    # state per entity
    obs_launches = max(1, args.observe_launches)
    obs_out = torch.empty_like(eng.obs)
    for i in range(3):
        eng.observe(out=obs_out)
    barrier()
    o_beg, o_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    o_beg.record(stream)
    for i in range(obs_launches):
        eng.observe(out=obs_out)
    o_end.record(stream)
    barrier()
    observe_ms = o_beg.elapsed_time(o_end) / obs_launches
    observe_bytes = E * L * eng.dims.obs_stride + E * eng.A * 3
    del obs_out
    if args.dump_steps and rank == 0:
        with open(args.dump_steps, 'w') as fh:
            json.dump(per_step_ms, fh)

    # ---------------- end to end through the public API with HOST buffers -----------------------------
    e2e_steps = max(4, args.e2e_steps)
    rng = np.random.default_rng(1234 + rank)
    pool = []
    for _ in range(8):                                # pinned host action buffers (random policy, same ranges)
        a = np.zeros((E, L, 4), dtype=np.int8)
        a[..., 0:2] = rng.integers(-1, 2, size=(E, L, 2), dtype=np.int8)
        a[..., 2] = rng.integers(0, 2, size=(E, L), dtype=np.int8)
        pool.append(torch.from_numpy(a).pin_memory())
    d2h_total = [0]
    KS = args.e2e_shards
    if KS > 1:
        # public host-facing API for callers that keep several sub-batches in flight (send / recv, as asynchronous
        # vector envs do): HostPipeline = KS sub-batches of E/KS envs, each on its own stream.  Every step of every
        # sub-batch uploads its pinned host actions (H2D) and lands its compacted rows in pinned host memory (D2H)
        # inside the timed region; the timed region also contains the pipeline's fill and drain.
        from abmarl_b200.engine import HostPipeline
        pipe = HostPipeline(build_spec(E, rank * E), shards=KS, device=dev, zero_copy=not args.e2e_staged)
        Ek = E // KS
        pipe.reset()

        def pipe_steps(i0, n):
            for k in range(KS):
                pipe.send(k, pool[i0 % len(pool)][k * Ek:(k + 1) * Ek])
            for i in range(i0 + 1, i0 + n):
                for k in range(KS):
                    pipe.recv(k)
                    d2h_total[0] += pipe.engines[k].last_d2h_bytes
                    pipe.send(k, pool[i % len(pool)][k * Ek:(k + 1) * Ek])
            for k in range(KS):
                pipe.recv(k)
                d2h_total[0] += pipe.engines[k].last_d2h_bytes

        e2e_stats = lambda: int(pipe.stats()[K.STAT_AGENT_STEPS].item())
        e2e_api = (f"HostPipeline.send/recv: {KS} sub-batches of {Ek} envs in flight on their own streams; per step pinned "
                   "host actions in (H2D), valid rows compacted by the gather kernel straight into pinned host memory (D2H)")
    else:
        def pipe_steps(i0, n):
            # pinned host actions -> H2D, step, on-device compaction of the rows the reference's manager would
            # return, D2H of exactly those rows (+ all_done); each call returns when they are on the host
            for i in range(i0, i0 + n):
                eng.step_host(pool[i % len(pool)], zero_copy=args.e2e_zero_copy)
                d2h_total[0] += eng.last_d2h_bytes

        e2e_stats = agent_steps
        e2e_api = "BatchedGridWorld.step_host: pinned host actions in, valid rows compacted on the device and copied out"

    pipe_steps(0, 3)
    barrier()
    n1 = e2e_stats()
    d2h_total[0] = 0
    e_beg, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e_beg.record(stream)
    pipe_steps(3, e2e_steps)
    e_end.record(stream)
    barrier()
    e2e_ms = e_beg.elapsed_time(e_end)
    n_e2e = e2e_stats() - n1
    clocks = sampler.stop(host_t0, time.perf_counter()) if sampler else None
    h2d = E * L * 4
    d2h = d2h_total[0] / e2e_steps

    # ---------------- strong scaling: BASELINE's "4096 envs sharded across 1/2/4/8" -------------------
    strong = None
    if world > 1 and E % world == 0:
        Es = E // world
        seng = BatchedGridWorld(build_spec(Es, rank * Es), device=dev)
        seng.reset()
        seng.rollout_sampled(args.warmup)
        barrier()
        s0 = int(seng.stats()[K.STAT_AGENT_STEPS].item())
        s_beg, s_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        s_beg.record(stream)
        seng.rollout_sampled(args.steps)
        s_end.record(stream)
        barrier()
        strong = [s_beg.elapsed_time(s_end), int(seng.stats()[K.STAT_AGENT_STEPS].item()) - s0]

    # ---------------- reduce over ranks: times = max, counts = sum (NCCL: episode statistics only) ----
    t = torch.tensor([ms, e2e_ms, kernel_ms, strong[0] if strong else 0.0], dtype=torch.float64, device=dev)
    c = torch.tensor([n_dev, n_e2e, launches, strong[1] if strong else 0.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
    ms, e2e_ms, kernel_ms_max, strong_ms = (float(x) for x in t.tolist())
    n_dev_all, n_e2e_all, launches_all, strong_n = (float(x) for x in c.tolist())

    if rank == 0:
        peak, peak_src = measured_peak()
        launches_rank = max(1, launches)
        per_step_ms_rank = kernel_ms / args.steps                           # this rank
        per_launch_ms = kernel_ms / launches_rank                           # this rank's step kernel, average launch duration
        algo_bytes = BYTES_PER_AGENT_STEP * n_dev / launches_rank          # algorithmic bytes one launch processes, this rank
        achieved = algo_bytes / (per_launch_ms * 1e-3) / 1e9
        traffic, traffic_src = None, None
        try:
            with open(os.path.join(ROOT, 'profiles', 'step_kernel_traffic.json')) as f:
                tj = json.load(f)
                key = 'dram_bytes_per_step_early' if args.steps + args.warmup <= 60 else 'dram_bytes_per_step'
                traffic, traffic_src = tj.get(key) * args.steps / launches_rank, tj.get('source')   # per launch, like `achieved`
        except Exception:
            pass
        line = {
            "metric": METRIC, "value": n_dev_all / (ms * 1e-3), "unit": "agent-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "i8/f64", "data": "synthetic",
            "config": workload_config(world, E),
            "agent_steps_per_step": n_dev_all / args.steps,
            "e2e": {"value": n_e2e_all / (e2e_ms * 1e-3), "unit": "agent-steps/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                    "api": e2e_api},
            "gpu_launches": int(launches_all),
            "clocks": clocks,
            "roofline": {"bound": "hbm",
                         "kernel": "bgw_step_fast_kernel (bgw_rollout_sampled: the K timed manager steps of all envs in "
                                   f"{launches_rank} launch(es); its CTAs draw (step, env) tickets)" if not args.per_step_calls else
                                   "bgw_step_fast_kernel (one bgw_step_sampled launch per step)",
                         "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic,
                         "traffic_source": traffic_src, "peak_source": peak_src,
                         "algorithmic_bytes_per_agent_step": BYTES_PER_AGENT_STEP,
                         "algorithmic_bytes_per_launch": algo_bytes,
                         "kernel_ms_per_launch": per_launch_ms, "kernel_ms_per_step": per_step_ms_rank, "kernel_share_of_step": 1.0,
                         "launch_duration": "timed region (CUDA events on the launching stream) / launches; nothing else is in the region",
                         "kernel_ms_isolated": iso_ms_per_launch,
                         "isolated_achieved": BYTES_PER_AGENT_STEP * iso_units_per_launch / (iso_ms_per_launch * 1e-3) / 1e9,
                         "isolated_note": f"{ks} further steps, one bgw_step_sampled launch each, every launch bracketed by its own CUDA events (launches serialised, per-CTA set-up and tail exposed)",
                         "kernel_ms_given_actions": given_ms_per_step,
                         "given_actions_achieved": BYTES_PER_AGENT_STEP * given_units_per_step / (given_ms_per_step * 1e-3) / 1e9,
                         "given_actions_note": f"{gs} bgw_step calls with caller-supplied device-resident action tensors (what a trainer calls): one launch per step, no fused policy",
                         "observe_kernel": {"kernel": "bgw_observe_fast_kernel (bgw_observe: get_obs of every learner, no step)",
                                            "ms_per_launch": observe_ms, "bytes_per_launch": observe_bytes,
                                            "achieved": observe_bytes / (observe_ms * 1e-3) / 1e9, "unit": "GB/s",
                                            "frac": observe_bytes / (observe_ms * 1e-3) / 1e9 / peak,
                                            "rows_per_s": E * L / (observe_ms * 1e-3),
                                            "note": f"{obs_launches} launches back to back; bytes = E*L obs rows of obs_stride written + 3 B of state per entity read"}},
        }
        if strong is not None:
            line["strong"] = {"global_envs": E, "envs_per_gpu": E // world, "ms_per_step": strong_ms / args.steps,
                              "value": strong_n / (strong_ms * 1e-3), "unit": "agent-steps/s",
                              "note": "BASELINE configs[4] as written: 4096 envs in total sharded over the GPUs (the weak line above keeps 4096 per GPU); with E/N envs a GPU's resident CTA slots are no longer all filled, the step time is bounded below by one env's latency"}
        if world == 1 and not args.no_cpu:
            cores = len(os.sched_getaffinity(0))
            n, dt, envs = cpu_rollout(E, args.cpu_steps, cores, warmup=2)
            line["cpu_baseline"] = {"value": n / dt, "unit": "agent-steps/s", "cores": cores, "kind": "port",
                                    "sample": f"oracle C port of the reference loop (scalar C per thread) on {cores} host threads, {envs} envs x {args.cpu_steps} steps of the same workload from reset, {dt:.1f} s",
                                    "python_reference_per_core": PYTHON_REFERENCE_PER_CORE}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=1000, help='timed steps (default: five 200-step episodes, SURVEY 8(d))')
    ap.add_argument('--warmup', type=int, default=50)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--envs-per-gpu', type=int, default=ENVS_PER_GPU)
    ap.add_argument('--e2e-steps', type=int, default=200, help='steps of the host-buffer loop (one full episode)')
    ap.add_argument('--e2e-shards', type=int, default=2, help='sub-batches the e2e loop keeps in flight (1 = one blocking step_host call per step)')
    ap.add_argument('--e2e-staged', action='store_true', help='e2e pipeline: compact on the device and copy with the copy engine instead of writing pinned host memory from the gather kernel')
    ap.add_argument('--kernel-steps', type=int, default=1000, help='steps of the second pass that brackets every launch with its own events')
    ap.add_argument('--per-step-calls', action='store_true', help='one bgw_step_sampled call per step instead of bgw_rollout_sampled (A/B)')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--spinup-steps', type=int, default=1500, help='untimed steps before the reset that starts the measured episode (GPU clock ramp)')
    ap.add_argument('--cpu-steps', type=int, default=200, help='steps of the cpu_baseline sample (all host cores, all envs)')
    ap.add_argument('--given-steps', type=int, default=200, help='bgw_step calls with caller-supplied device actions timed next to the fused rollout')
    ap.add_argument('--e2e-zero-copy', action='store_true', help='e2e: the gather kernel writes the pinned host buffers directly instead of compacting on the device and copying')
    ap.add_argument('--observe-launches', type=int, default=50, help='bgw_observe launches timed next to the step kernel')
    ap.add_argument('--dump-steps', default=None, help='write the per-step kernel times (ms) to this JSON file')
    ap.add_argument('--dump-outputs', default=None, metavar='DIR',
                    help="write the outputs of the last timed step (rank 0's envs) to DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
