"""AllStepManager / TurnBasedManager over E lockstep environments.

The reference managers wrap ONE simulation and trade dicts keyed by agent id
(abmarl/managers/simulation_manager.py:27-53, all_step_manager.py:37-95, turn_based_manager.py:22-94).  These
wrap a simulation *definition* and drive E copies of it on the device: `reset()` and `step(actions)` trade
dense tensors indexed [env, learner] (learner order = the order of `sim.agents`), and the manager rules --
done agents stop acting and are never reported again, `__all__`, the turn cursor that is never rewound --
are applied per env inside the step kernel (abmarl_b200/csrc/bgw_dev.cuh).  `as_dicts(env)` converts one
env's last outputs into the reference's dict-of-dicts form.
"""
from abc import ABC

import os

import numpy as np
import torch

from abmarl_b200 import _capi as K
from abmarl_b200.spec import compile_sim
from abmarl_b200.engine import BatchedGridWorld


class SimulationManager(ABC):
    """simulation_manager.py:7-53 (batched)."""
    _manager = None

    def __init__(self, sim, n_envs=1, env_offset=0, seed=0, horizon=0, auto_reset=False, device=None,
                 randomize_action_input=False, layouts=None, specialize=False):
        assert type(randomize_action_input) is bool, "Randomize action input must be a boolean."   # all_step_manager.py:32-35
        assert not randomize_action_input or self._manager == 'all_step', \
            "randomize_action_input is an AllStepManager option (all_step_manager.py:24-35)"
        self.sim = sim
        self.randomize_action_input = bool(randomize_action_input)
        inner = sim.unwrapped if hasattr(sim, 'super_agent_mapping') else sim      # SuperAgentWrapper(sim, mapping)
        self.spec = compile_sim(inner, manager=self._manager, n_envs=n_envs, env_offset=env_offset, seed=seed,
                                horizon=horizon, auto_reset=auto_reset, randomize_action_input=randomize_action_input)
        self.engine = BatchedGridWorld(self.spec, device=device)
        if specialize:                 # compile the step kernel for this sim alone (bgw_specialize; `specialize` may name a cache directory)
            self.engine.specialize(specialize if isinstance(specialize, (str, bytes, os.PathLike)) else None)
        self.super_view = None
        if hasattr(sim, 'super_agent_mapping'):
            from abmarl_b200.sim.wrappers import SuperAgentView
            self.super_view = SuperAgentView(self.spec, sim.super_agent_mapping, n_envs, device=self.engine.device)
        self._feeder = None
        if layouts is not None:
            self.engine.set_layout(layouts)
        elif self.spec.layout_generator is not None and not self.engine.device_layouts:   # MazePlacementState above the device generator's limits: host-side layouts
            from abmarl_b200.layouts import LayoutFeeder
            self._feeder = LayoutFeeder(self.spec)
        self.learner_ids = self.spec.learner_ids

    # -- tensors ---------------------------------------------------------------------------------
    @property
    def n_envs(self):
        return self.engine.E

    @property
    def n_learners(self):
        return self.engine.L

    def reset(self, env_mask=None):
        """-> obs int8 [E, L, h, w(, c)] (first observations; turn-based: only the row of the env's turn is fresh)."""
        if self._feeder is not None:
            episode = self.engine.state['episode'].cpu().numpy().view(np.uint32)
            mask = None if env_mask is None else np.asarray(torch.as_tensor(env_mask).cpu())
            self.engine.set_layout(self._feeder.prime(episode, mask))
        self.engine.reset(env_mask)
        if self.super_view is not None:
            self.super_view.reset(env_mask)
        return self.engine.obs_view()

    def step(self, actions, order=None):
        """actions int8 [E, L, action_stride] on the device -> (obs, reward f32 [E, L], done uint8 [E, L], all_done uint8 [E]).

        `done` carries OUT_VALID for the learners that received (obs, reward, done) this call and OUT_DONE for
        those that are done; rows of learners already reported done are ignored on input (the reference
        asserts they are absent, all_step_manager.py:59-61)."""
        # (randomize_action_input, all_step_manager.py:62-65: the library shuffles on the device -- the keyed order of the
        # step, BgwSpec.randomize_action_input -- whenever no explicit order is given)
        if order is None and self.super_view is not None:       # SuperAgentWrapper.step: super agents' members first
            order = self.super_view.order
        _, reward, done, all_done = self.engine.step(actions, order)
        if self._feeder is not None and self.spec.auto_reset:
            if self._feeder.after_step(all_done.cpu().numpy(), self.engine.state['episode'].cpu().numpy().view(np.uint32)):
                self.engine.set_layout(self._feeder.rows)
        return self.engine.obs_view(), reward, done, all_done

    def observe(self, env_mask=None):
        """sim.get_obs(agent_id) of EVERY learner on the state as it stands (bgw_observe; smart.py:93-99) -> obs int8
        [E, L, h, w(, c)] in the engine's obs tensor: nothing is stepped, learners already reported done included."""
        self.engine.observe(env_mask)
        return self.engine.obs_view()

    def get_obs(self, agent_id, env=0):
        """The reference's `sim.get_obs(agent_id)` for one env: the observers' dict of that learner (smart.py:93-99)."""
        self.engine.observe()
        snap = self.host_snapshot()
        l = list(self.learner_ids).index(agent_id)
        snap['done'] = np.zeros_like(snap['done'])
        snap['done'][env, l] = K.OUT_VALID
        return self.dicts_from(snap, env)[0][agent_id]

    def program_vars(self):
        """{name: view} of the device program's variables (BatchedGridWorld.program_vars): float64 [E] / [E, n] per env
        variable, [E, A] per agent variable, on the device; {} for a sim without them."""
        return self.engine.program_vars()

    def super_outputs(self):
        """SuperAgentWrapper view of the last step (super_agent_wrapper.py:112-216): (obs rows with null observations for
        covered agents done earlier, mask [E, L], reward [E, G] f64, done [E, G], valid [E, G]); groups = `super_view.groups`.
        Call once per step."""
        assert self.super_view is not None, "the simulation is not wrapped in a SuperAgentWrapper"
        e = self.engine
        return self.super_view.update(e.obs, e.reward, e.done, e.all_done)

    def sample_actions(self):
        """A random action per learner from the keyed Philox stream (== action_space.sample() ranges)."""
        return self.engine.sample_actions()

    def encode_actions(self, action_dicts):
        """[{agent_id: {'move': ..., 'attack': ...}}, ...] (one dict per env, reference format) -> int8
        [E, L, action_stride] (layout: include/bgw.h, bgw_step)."""
        sp = self.spec
        act = np.zeros((self.engine.E, self.engine.L, self.engine.action_stride), dtype=np.uint8)
        index = {aid: l for l, aid in enumerate(self.learner_ids)}
        for e, d in enumerate(action_dicts):
            for agent_id, a in d.items():
                l = index[agent_id]
                if 'move' in a:
                    mv = a['move']
                    if sp.move_actor == K.MOVE_BOX and not sp.ravel_actions:
                        act[e, l, 0], act[e, l, 1] = np.int8(int(mv[0])).view(np.uint8), np.int8(int(mv[1])).view(np.uint8)
                    else:
                        act[e, l, 0] = int(mv)
                if 'attack' in a:
                    att = a['attack']
                    if sp.attack_actor == K.ATTACK_ENCODING:          # {encoding: count} actor.py:513-519
                        for enc, count in att.items():
                            act[e, l, 2 + int(enc) - 1] = int(count)
                    elif sp.attack_actor == K.ATTACK_RESTRICTED:       # [cell + 1 | 0] * simultaneous_attacks :593-599
                        att = np.asarray(att, dtype=int).ravel()
                        act[e, l, 2:2 + att.size] = att
                    elif sp.attack_actor == K.ATTACK_SELECTIVE:        # (n, n) counts :669-679
                        att = np.asarray(att, dtype=int).ravel()
                        act[e, l, 2:2 + att.size] = att
                    else:
                        act[e, l, 2] = int(att)
        return torch.from_numpy(act.view(np.int8)).to(self.engine.device)

    # -- reference-shaped view of one env --------------------------------------------------------
    def host_snapshot(self):
        """One device->host copy of the last outputs of ALL envs (numpy): what as_dicts / the external adapters slice."""
        eng = self.engine
        ammo, position = eng.ammo_view(), eng.position_view()
        return dict(obs=eng.obs_view().cpu().numpy(), reward=eng.reward.cpu().numpy(), done=eng.done.cpu().numpy(),
                    all_done=eng.all_done.cpu().numpy(), turn=eng.state['turn'].cpu().numpy(),
                    ammo=None if ammo is None else ammo.cpu().numpy(),
                    position=None if position is None else position.cpu().numpy())

    def dicts_from(self, snap, env=0, after_reset=False):
        """(obs, rewards, dones, infos) of env `env` as the reference's dicts (simulation_manager.py:38-53), built from a
        host_snapshot()."""
        key = {K.OBS_POSITION_CENTERED: 'position_centered_encoding', K.OBS_ABSOLUTE: 'absolute_encoding',
               K.OBS_STACKED: 'stacked_position_centered_encoding'}[self.spec.observer]
        obs_all = snap['obs'][env].astype(np.int64)
        ammo = None if snap['ammo'] is None else snap['ammo'][env]
        position = None if snap['position'] is None else snap['position'][env].astype(np.int64)
        done, reward, flags = snap['done'][env], snap['reward'][env], int(snap['all_done'][env])
        obs, rew, dn, info = {}, {}, {}, {}
        # TurnBasedManager / DynamicOrderManager.reset return the first agent's observation only (turn_based_manager.py:22-32)
        first = int(snap['turn'][env]) if after_reset and self._manager in ('turn_based', 'dynamic_order') else None
        for l, agent_id in enumerate(self.learner_ids):
            if (after_reset and (first is None or l == first)) or (not after_reset and (done[l] & K.OUT_VALID)):
                a = self.spec.learner_agents[l]
                n = 2 * int(self.spec.view_range[a]) + 1
                o = obs_all[l]
                if self.spec.observer != K.OBS_ABSOLUTE and o.shape[0] != n:     # agent with a smaller view
                    flat = o.reshape(-1)[:n * n * (o.shape[2] if o.ndim == 3 else 1)]
                    o = flat.reshape((n, n) + o.shape[2:])
                obs[agent_id] = {key: o} if self.spec.klass[a] & K.AG_OBSERVING else {}
                if ammo is not None and self.spec.klass[a] & K.AG_AMMO:      # AmmoObserver observer.py:406-413
                    obs[agent_id]['ammo'] = int(ammo[l])
                if position is not None:                                  # AbsolutePositionObserver observer.py:366-373
                    obs[agent_id]['position'] = position[l]
                if not after_reset:
                    rew[agent_id] = float(reward[l])
                    dn[agent_id] = bool(done[l] & K.OUT_DONE)
                    info[agent_id] = {}
        if after_reset:
            return obs
        dn['__all__'] = bool(flags & K.ENV_ALL_DONE)
        return obs, rew, dn, info

    def as_dicts(self, env=0, after_reset=False):
        """(obs, rewards, dones, infos) of env `env` as the reference's dicts (simulation_manager.py:38-53)."""
        return self.dicts_from(self.host_snapshot(), env, after_reset)


class AllStepManager(SimulationManager):
    """all_step_manager.py:7-95: every not-done learner acts each step."""
    _manager = 'all_step'


class TurnBasedManager(SimulationManager):
    """turn_based_manager.py:7-94: one learner per step, in `sim.agents` order; `actions[e, turn[e]]` is read."""
    _manager = 'turn_based'

    @property
    def turn(self):
        """int16 [E]: the learner whose action the next step() consumes."""
        return self.engine.state['turn']


class DynamicOrderManager(SimulationManager):
    """dynamic_order_manager.py:7-87: the simulation decides whose turn it is.  `actions[e, l]` is read for every acting
    learner (`acting`); the step reports the agents the simulation names next (sim.next_agent) that were not reported
    done before, or every agent not yet reported once the simulation is done.  The built-in DynamicOrderMultiMazeSim names
    the one that just finished, if any, and the next one that is not done: one learner acts, `turn[e]`.  A sim with a
    device program names its agents with the program's next_agent hook (include/bgw_program.h): any number of learners
    act at once, in dict order."""
    _manager = 'dynamic_order'

    def __init__(self, sim, **kwargs):
        from abmarl_b200.sim import DynamicOrderSimulation
        assert isinstance(sim, DynamicOrderSimulation), \
            "To use the DynamicOrderManager, the simulation must be a DynamicOrderSimulation."
        super().__init__(sim, **kwargs)

    @property
    def turn(self):
        """int16 [E]: the learner whose action the next step() consumes (the not-done agent the simulation named); with a
        device program the lowest such learner, -1 if it named none."""
        return self.engine.state['turn']

    @property
    def acting(self):
        """bool [E, L] on the device: the learners whose action rows the next step() reads.  After a reset that is
        learner `turn[e]`; after a step, the learners the simulation named that are not done.  Learners already reported
        done never act, and nobody acts in an env whose episode is over (the next step resets it)."""
        st = self.engine.state
        flags = st['flags'][:, self.spec.learner_agents]
        by_turn = torch.arange(self.engine.L, device=flags.device)[None, :] == st['turn'].long()[:, None]
        if self.spec.program == K.PROG_USER:
            named = torch.where((st['step'] == 0)[:, None], by_turn, (flags & K.ST_NEXT) != 0)
        else:
            named = by_turn
        live = (st['env_flags'] & K.ENV_ALL_DONE) == 0
        return named & ((flags & K.ST_DONE_REPORTED) == 0) & live[:, None]

