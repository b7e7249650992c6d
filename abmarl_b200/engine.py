"""BatchedGridWorld: E independent copies of one compiled simulation advanced in lockstep on one B200.

Thin host object over the C-ABI of include/bgw.h (libbgw.so, abmarl_b200/csrc): PyTorch provides the device
memory and the CUDA stream, every buffer is handed to the library as a raw device pointer, and the kernels
are enqueued on torch's current stream.  There is no CPU fallback: constructing the engine without the built
extension or without a CUDA device raises.
"""
import ctypes as C

import os

import numpy as np
import torch

from abmarl_b200 import _capi as K

_STATE_FIELDS = (('cell', torch.int16, 'EA'), ('next', torch.int16, 'EA'), ('flags', torch.uint8, 'EA'),
                 ('health', torch.float64, 'EA'), ('reward_acc', torch.float64, 'EA'),
                 ('episode', torch.int32, 'E'), ('step', torch.int32, 'E'), ('env_flags', torch.uint8, 'E'),
                 ('turn', torch.int16, 'E'), ('error', torch.int32, 'E'), ('ammo', torch.int32, 'EA'))
_NP_VIEW = {'cell': np.uint16, 'next': np.uint16, 'episode': np.uint32, 'step': np.uint32, 'error': np.uint32}


class BatchedGridWorld:
    """reset() / step(actions) over device tensors.

    actions  int8  [E, L, action_stride]   byte 0,1 = move (dr, dc | cross 0..4 | ravelled), from byte 2 the attack
                   action (layout: include/bgw.h, bgw_step; action_stride = 4 for the BinaryAttackActor)
    obs      int8  [E, L, obs_stride]   (see obs_view)
    reward   f32   [E, L];  done uint8 [E, L] (OUT_VALID | OUT_DONE);  all_done uint8 [E] (ENV_* bits)
    """

    def __init__(self, spec, device=None):
        if not torch.cuda.is_available():
            raise RuntimeError("abmarl_b200 needs a CUDA device: the engine has no CPU fallback")
        self.lib = K.load()
        self.spec = spec
        self.check_order = True        # validate caller-given `order` rows on every step (a device reduction; switch off in tight loops)
        self.device = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.index is None:              # 'cuda' without an index: the handle and the tensors must name the same device
            self.device = torch.device('cuda', torch.cuda.current_device())
        self._c = spec.c_struct()
        h = C.c_void_p()
        K.check(self.lib.bgw_create(C.byref(self._c), self.device.index, C.byref(h)), self.lib)
        self._h = h
        source = getattr(spec, 'program_source', None)
        init = getattr(spec, 'program_var_init', None)
        program_vars = None
        if source is not None and init is not None:   # the program's variables: their counts are compiled into its kernel
            program_vars = torch.zeros((spec.n_envs, init.size), dtype=torch.float64, device=self.device)
            init = np.ascontiguousarray(init, dtype=np.float64)
            K.check(self.lib.bgw_set_program_vars(h, spec.n_env_vars, len(spec.agent_var_names),
                                                  init.ctypes.data_as(C.c_void_p), program_vars.data_ptr()), self.lib)
        if source is not None:                     # the sim's own step program, compiled into the step kernel (cached in $BGW_JIT_CACHE)
            K.check(self.lib.bgw_set_program(h, source.encode(), None), self.lib)
        d = K.BgwDims()
        K.check(self.lib.bgw_dims(h, C.byref(d)), self.lib)
        self.dims = d
        self.E, self.A, self.L = d.n_envs, d.n_agents, d.n_learners
        dev = self.device
        self.state = {}
        for name, dt, shape in _STATE_FIELDS:
            self.state[name] = torch.zeros((self.E, self.A) if shape == 'EA' else (self.E,), dtype=dt, device=dev)
        self.state['cell'].fill_(-1)         # 0xFFFF
        self.state['next'].fill_(-1)
        self.state['episode'].fill_(-1)      # 0xFFFFFFFF: first reset makes it 0
        self.state['turn'].fill_(-1)
        self.state['stats'] = torch.zeros((self.E, K.BGW_STAT_COUNT), dtype=torch.int64, device=dev)
        self.state['program_vars'] = program_vars    # float64 [E, n_env_vars + A * n_agent_vars] (program_vars()), or None
        # MazePlacementState: start layouts are generated on the device when the library can (bgw_generate_layouts),
        # else host-side (abmarl_b200/layouts.py) and handed over with set_layout()
        self.device_layouts = bool(d.device_layouts)
        self.state['layout'] = torch.full((self.E, self.A), -1, dtype=torch.int16, device=dev) if self.device_layouts else None
        self.obs = torch.zeros((self.E, self.L, d.obs_stride), dtype=torch.int8, device=dev)
        self.reward = torch.zeros((self.E, self.L), dtype=torch.float32, device=dev)
        self.done = torch.zeros((self.E, self.L), dtype=torch.uint8, device=dev)
        self.all_done = torch.zeros((self.E,), dtype=torch.uint8, device=dev)
        self.action_stride = d.action_stride
        self.actions = torch.zeros((self.E, self.L, d.action_stride), dtype=torch.int8, device=dev)
        self._bind()

    # ---- plumbing -------------------------------------------------------------------------------
    def _bind(self):
        s = K.BgwState()
        for name in ('cell', 'next', 'flags', 'health', 'reward_acc', 'episode', 'step', 'env_flags', 'turn',
                     'error', 'layout', 'stats', 'ammo'):
            t = self.state[name]
            setattr(s, name, None if t is None else t.data_ptr())
        K.check(self.lib.bgw_bind_state(self._h, C.byref(s)), self.lib)

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def close(self):
        if getattr(self, '_h', None):
            self.lib.bgw_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- the managers' interface ---------------------------------------------------------------
    def set_layout(self, layout):
        """[E, A] start cells generated host-side (0xFFFF = leave unplaced); None = PositionState placement.  Explicit
        layouts switch the device-side generator off."""
        if self.device_layouts:                    # the handle must know too: bgw_rollout_sampled regenerates layouts between its steps otherwise
            K.check(self.lib.bgw_use_device_layouts(self._h, 0), self.lib)
        self.device_layouts = False
        if layout is None:
            self.state['layout'] = None
        else:
            lay = np.ascontiguousarray(layout, dtype=np.uint16).view(np.int16)
            assert lay.shape == (self.E, self.A)
            self.state['layout'] = torch.from_numpy(lay).to(self.device)
        self._bind()

    def reset(self, env_mask=None):
        m = None
        if env_mask is not None:
            m = torch.as_tensor(env_mask, dtype=torch.uint8, device=self.device).contiguous()
        if self.device_layouts:                       # MazePlacementState.reset: the layouts of the episodes about to start
            K.check(self.lib.bgw_generate_layouts(self._h, None if m is None else m.data_ptr(), 0, self._stream()), self.lib)
        K.check(self.lib.bgw_reset(self._h, None if m is None else m.data_ptr(), self.obs.data_ptr(), self._stream()),
                self.lib)
        return self.obs

    def specialize(self, cache_dir=None):
        """Compile the general step kernel for this spec alone (bgw_specialize: NVRTC at run time, cached by spec hash in
        `cache_dir` or $BGW_JIT_CACHE).  Same source, same results; a third of the instructions.  A no-op for the sims
        that run the specialised team-battle kernel."""
        K.check(self.lib.bgw_specialize(self._h, None if cache_dir is None else os.fsencode(cache_dir)), self.lib)
        return self

    def observe(self, env_mask=None, out=None):
        """`sim.get_obs(agent_id)` of every learner for the state as it stands (bgw_observe; smart.py:93-99): nothing is
        stepped.  Into `out` ([E, L, obs_stride] int8 CUDA; default: the engine's obs tensor), rows of unselected envs untouched."""
        out = self.obs if out is None else out
        assert out.dtype == torch.int8 and tuple(out.shape) == tuple(self.obs.shape) and out.is_cuda and out.is_contiguous()
        m = None
        if env_mask is not None:
            m = torch.as_tensor(env_mask, dtype=torch.uint8, device=self.device).contiguous()
            assert tuple(m.shape) == (self.E,)
        K.check(self.lib.bgw_observe(self._h, None if m is None else m.data_ptr(), out.data_ptr(), self._stream()), self.lib)
        return out

    def sample_actions(self, out=None):
        out = self.actions if out is None else out
        K.check(self.lib.bgw_sample_actions(self._h, out.data_ptr(), self._stream()), self.lib)
        return out

    def step(self, actions, order=None):
        assert actions.dtype == torch.int8 and tuple(actions.shape) == (self.E, self.L, self.action_stride) and actions.is_cuda \
            and actions.is_contiguous(), "actions must be a contiguous int8 CUDA tensor [E, L, action_stride]"
        o = None
        if order is not None:
            o = torch.as_tensor(order, dtype=torch.int16, device=self.device).contiguous()
            assert tuple(o.shape) == (self.E, self.L)
            if __debug__ and self.check_order:       # the kernels index the learner table with these values
                assert int(o.min()) >= 0 and int(o.max()) < self.L, "order must hold learner indices 0..L-1"
        K.check(self.lib.bgw_step(self._h, actions.data_ptr(), None if o is None else o.data_ptr(),
                                  self.obs.data_ptr(), self.reward.data_ptr(), self.done.data_ptr(),
                                  self.all_done.data_ptr(), self._stream()), self.lib)
        self._layouts_for_finished_envs()
        return self.obs, self.reward, self.done, self.all_done

    def _layouts_for_finished_envs(self):
        """auto-reset: the envs that just reported __all__ are reset by the next step and need their next layout"""
        if self.device_layouts and self.spec.auto_reset:
            K.check(self.lib.bgw_generate_layouts(self._h, None, 1, self._stream()), self.lib)

    def step_sampled(self, order=None):
        """sample_actions() + step() in one call (one launch on the specialised kernel): the keyed random policy
        acts for every learner that may act; the sampled actions land in self.actions."""
        o = None
        if order is not None:
            o = torch.as_tensor(order, dtype=torch.int16, device=self.device).contiguous()
        K.check(self.lib.bgw_step_sampled(self._h, self.actions.data_ptr(), None if o is None else o.data_ptr(),
                                          self.obs.data_ptr(), self.reward.data_ptr(), self.done.data_ptr(),
                                          self.all_done.data_ptr(), self._stream()), self.lib)
        self._layouts_for_finished_envs()
        return self.obs, self.reward, self.done, self.all_done

    def rollout_sampled(self, n_steps, order=None):
        """n_steps x step_sampled() in one call (bgw_rollout_sampled): a random-policy rollout that stays on the device.
        Same state, statistics and final outputs as n_steps separate calls; on the specialised kernel the launches are
        chained per env (launch k+1 starts an env as soon as launch k has finished it)."""
        o = None
        if order is not None:
            o = torch.as_tensor(order, dtype=torch.int16, device=self.device).contiguous()
        K.check(self.lib.bgw_rollout_sampled(self._h, int(n_steps), self.actions.data_ptr(), None if o is None else o.data_ptr(),
                                             self.obs.data_ptr(), self.reward.data_ptr(), self.done.data_ptr(),
                                             self.all_done.data_ptr(), self._stream()), self.lib)
        return self.obs, self.reward, self.done, self.all_done

    # ---- host-facing step: HOST buffers in, only the rows the reference's manager would return out ---------
    def _host_buffers(self):
        if getattr(self, '_hb', None) is None:
            E, L, dev = self.E, self.L, self.device
            n = E * L
            self._hb = dict(
                count=torch.zeros(1, dtype=torch.int32, device=dev), index=torch.empty(n, dtype=torch.int32, device=dev),
                obs=torch.empty((n, self.dims.obs_stride), dtype=torch.int8, device=dev),
                reward=torch.empty(n, dtype=torch.float32, device=dev), done=torch.empty(n, dtype=torch.uint8, device=dev),
                h_count=torch.zeros(1, dtype=torch.int32).pin_memory(), h_index=torch.empty(n, dtype=torch.int32).pin_memory(),
                h_obs=torch.empty((n, self.dims.obs_stride), dtype=torch.int8).pin_memory(),
                h_reward=torch.empty(n, dtype=torch.float32).pin_memory(), h_done=torch.empty(n, dtype=torch.uint8).pin_memory(),
                h_all=torch.empty(E, dtype=torch.uint8).pin_memory(), d_act=torch.empty((E, L, self.action_stride), dtype=torch.int8, device=dev))
        return self._hb

    def enqueue_host(self, actions_host, order=None, zero_copy=False):
        """The device side of step_host, enqueued on the current stream without waiting: H2D of the pinned action
        buffer, the step, the compaction of the valid rows (with zero_copy straight into the pinned host buffers)
        and the D2H of the row count and all_done."""
        hb = self._host_buffers()
        hb['d_act'].copy_(actions_host, non_blocking=True)
        self.step(hb['d_act'], order)
        p = lambda t: t.data_ptr()
        dst = {k: hb[('h_' if zero_copy else '') + k] for k in ('index', 'obs', 'reward', 'done')}
        K.check(self.lib.bgw_gather_valid(self._h, p(self.obs), p(self.reward), p(self.done), p(self.all_done),
                                          p(hb['count']), p(dst['index']), p(dst['obs']), p(dst['reward']), p(dst['done']),
                                          self._stream()), self.lib)
        hb['h_count'].copy_(hb['count'], non_blocking=True)
        hb['h_all'].copy_(self.all_done, non_blocking=True)

    def collect_host(self, zero_copy=False):
        """Wait for the work enqueue_host put on the current stream; returns what step_host returns."""
        hb = self._hb
        stream = torch.cuda.current_stream(self.device)
        stream.synchronize()
        n = int(hb['h_count'][0])
        if not zero_copy:
            for k in ('index', 'obs', 'reward', 'done'):
                hb['h_' + k][:n].copy_(hb[k][:n], non_blocking=True)
            stream.synchronize()
        self.last_d2h_bytes = n * (self.dims.obs_stride + 9) + self.E + 4
        return n, hb['h_index'][:n], hb['h_obs'][:n], hb['h_reward'][:n], hb['h_done'][:n], hb['h_all']

    def step_host(self, actions_host, order=None, zero_copy=False):
        """One manager step for a HOST caller: `actions_host` int8 [E, L, 4] (pinned for speed) is copied to the
        device, the batch is stepped, and the rows of the learners that received (obs, reward, done) -- plus all
        rows of envs that were auto-reset -- are compacted and land in pinned host buffers.  Returns
        (n, index[:n], obs[:n], reward[:n], done[:n], all_done[E]) as pinned host tensors; index = env * L + learner.
        With zero_copy the gather kernel writes the compacted rows straight into the pinned buffers (they are
        device-addressable under UVA): one stream synchronisation per call and no separate copies; measured equal to
        the staged copies on this pool (both PCIe-bound), so staged is the default.
        Bytes over PCIe per call: 4*E*L in, n*(obs_stride + 9) + E + 4 out."""
        self.enqueue_host(actions_host, order, zero_copy)
        return self.collect_host(zero_copy)

    # ---- views / introspection -------------------------------------------------------------------
    def obs_view(self, obs=None):
        """[E, L, h, w(, c)] logical view of the 16-byte padded int8 rows."""
        obs = self.obs if obs is None else obs
        d = self.dims
        v = obs[..., :d.obs_h * d.obs_w * d.obs_c]
        shape = tuple(obs.shape[:-1]) + ((d.obs_h, d.obs_w) if d.obs_c == 1 else (d.obs_h, d.obs_w, d.obs_c))
        return v.reshape(shape)

    def ammo_view(self, obs=None):
        """[E, L] int32: the AmmoObserver's 'ammo' observation stored in the obs rows (None without an AmmoObserver)."""
        obs = self.obs if obs is None else obs
        off = self.dims.ammo_offset
        if off < 0:
            return None
        return obs[..., off:off + 4].contiguous().view(torch.int32).squeeze(-1)

    def position_view(self, obs=None):
        """[E, L, 2] int16 (row, col): the AbsolutePositionObserver's 'position' observation stored in the obs rows (None
        without one)."""
        obs = self.obs if obs is None else obs
        off = self.dims.position_offset
        if off < 0:
            return None
        return obs[..., off:off + 4].contiguous().view(torch.int16)

    def state_numpy(self):
        """Host copy of the state in the oracle's numpy layout (tests)."""
        out = {}
        for name, t in self.state.items():
            if t is None:
                out[name] = None
                continue
            a = t.cpu().numpy()
            if name in _NP_VIEW:
                a = a.view(_NP_VIEW[name])
            elif name == 'stats':
                a = a.view(np.uint64)
            out[name] = a
        return out

    def load_state(self, st):
        """Overwrite the device state from numpy arrays in the oracle's layout (parity tests)."""
        for name, t in self.state.items():
            if t is None or name not in st or st[name] is None:
                continue
            a = np.ascontiguousarray(st[name])
            if name in _NP_VIEW or name == 'stats':
                a = a.view({2: np.int16, 4: np.int32, 8: np.int64}[a.dtype.itemsize])
            t.copy_(torch.from_numpy(a).reshape(t.shape))

    def program_vars(self):
        """{name: view} of the step program's variables in state['program_vars'] (DeviceProgram(env_vars=, agent_vars=)):
        float64 [E] for an env scalar, [E, n] for an env array, [E, A] for an agent variable ({} without variables).
        The obs rows do not carry them; these views are what a trainer reads, and what it writes is what the next
        step reads."""
        rows = self.state['program_vars']
        return {} if rows is None else self.spec.program_var_views(rows)

    def stats(self):
        """Summed episode statistics (agent_steps, episodes, kills, env_steps) of this device's envs."""
        return self.state['stats'].sum(dim=0)

    @property
    def launches(self):
        return int(self.lib.bgw_launch_count(self._h))


class HostPipeline:
    """K sub-batches of one compiled simulation, each a BatchedGridWorld on its own CUDA stream, for HOST callers
    that keep several sub-batches in flight (the send / recv pattern of asynchronous vector envs): while the
    host consumes sub-batch k, the other sub-batches' action upload (H2D), step kernel and compacted result rows
    (the gather kernel writes them straight into pinned host memory) overlap on the device and on both PCIe
    directions.  Sub-batch k owns the global envs [env_offset + k*E/K, env_offset + (k+1)*E/K): the Philox key is
    global, so the results are those of one BatchedGridWorld over all E envs (tests/test_gpu_parity.py).

        pipe.reset()
        for k in range(pipe.K): pipe.send(k, actions[k])          # prime
        loop: for k in range(pipe.K): out = pipe.recv(k); ...; pipe.send(k, next_actions[k])
    """

    def __init__(self, spec, shards=4, device=None, zero_copy=True):
        self.zero_copy = bool(zero_copy)     # True: the gather kernel writes pinned host memory; False: compact on the device, then copy
        assert spec.n_envs % shards == 0, "n_envs must divide evenly over the sub-batches"
        self.K, self.Ek = shards, spec.n_envs // shards
        self.device = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.index is None:
            self.device = torch.device('cuda', torch.cuda.current_device())
        self.engines = [BatchedGridWorld(spec.with_envs(self.Ek, spec.env_offset + k * self.Ek), device=self.device)
                        for k in range(shards)]
        self.streams = [torch.cuda.Stream(self.device) for _ in range(shards)]
        self.E, self.L, self.A = spec.n_envs, self.engines[0].L, self.engines[0].A
        self.in_flight = [False] * shards

    def reset(self):
        for eng, s in zip(self.engines, self.streams):
            with torch.cuda.stream(s):
                eng.reset()
        for s in self.streams:
            s.synchronize()

    def send(self, k, actions_host, order=None):
        """Enqueue one manager step of sub-batch k: actions_host int8 [E/K, L, 4] in pinned host memory."""
        assert not self.in_flight[k], "recv(k) the previous step of this sub-batch first"
        with torch.cuda.stream(self.streams[k]):
            self.engines[k].enqueue_host(actions_host, order, zero_copy=self.zero_copy)
        self.in_flight[k] = True

    def recv(self, k):
        """Wait for sub-batch k's step; (n, index, obs, reward, done, all_done) as step_host, index = local env * L +
        learner (global env = env_offset + k * E/K + local env)."""
        assert self.in_flight[k]
        with torch.cuda.stream(self.streams[k]):
            out = self.engines[k].collect_host(zero_copy=self.zero_copy)
        self.in_flight[k] = False
        return out

    def step_host(self, actions_host):
        """All sub-batches one step: actions_host int8 [E, L, 4] pinned; returns the K recv() tuples."""
        for k in range(self.K):
            self.send(k, actions_host[k * self.Ek:(k + 1) * self.Ek])
        return [self.recv(k) for k in range(self.K)]

    @property
    def last_d2h_bytes(self):
        return sum(e.last_d2h_bytes for e in self.engines)

    @property
    def launches(self):
        return sum(e.launches for e in self.engines)

    def stats(self):
        for s in self.streams:
            s.synchronize()
        return sum(e.stats() for e in self.engines)
