"""compile_sim: walk an already-built, reference-style simulation object into the flat BgwSpec.

Works by duck typing, so it accepts both this package's definitions (abmarl_b200.sim / .examples) and
objects built by the unmodified reference (used when generating the golden vectors): it reads
`sim.agents` (dict order = agent index), `sim.grid.{rows,cols,overlapping}`, the actors' class and
`attack_mapping`, the chosen state / observer / done components and the sim's reward constants
(SURVEY.md section 3.4: "the point where the new repo hooks in").
"""
import ctypes as C
import math

import numpy as np

from abmarl_b200 import _capi as K
from abmarl_b200.program import DeviceProgram


def _mro_names(obj):
    return {c.__name__ for c in type(obj).__mro__}


def _rows(mapping):
    """{enc: {enc,...}} -> uint64[BGW_MAX_ENCODING+1] bit rows."""
    out = np.zeros(K.BGW_MAX_ENCODING + 1, dtype=np.uint64)
    for e, others in (mapping or {}).items():
        assert 0 < e <= K.BGW_MAX_ENCODING, f"encoding {e} out of range for the device engine"
        for f in others:
            assert 0 < f <= K.BGW_MAX_ENCODING, f"encoding {f} out of range for the device engine"
            out[e] |= np.uint64(1) << np.uint64(f)
    return out


class CompiledSpec:
    """Numpy tables + scalars of one simulation; `.c_struct()` gives the BgwSpec the C-ABI takes."""

    SCALARS = ('rows', 'cols', 'n_agents', 'n_envs', 'env_offset', 'program', 'move_actor', 'attack_actor',
               'observer', 'observe_self', 'done_mask', 'manager', 'ravel_actions', 'no_overlap_at_reset',
               'stacked_attacks', 'horizon', 'auto_reset', 'ammo_observer', 'randomize_placement_order',
               'randomize_action_input', 'position_observer', 'seed')
    TABLES = (('encoding', np.int8), ('klass', np.uint8), ('role', np.uint8), ('init_row', np.int16),
              ('init_col', np.int16), ('init_health', np.float64), ('init_orient', np.uint8),
              ('view_range', np.int16), ('move_range', np.int16), ('attack_range', np.int16),
              ('attack_strength', np.float64), ('attack_accuracy', np.float64),
              ('simultaneous_attacks', np.uint8), ('target', np.int16), ('initial_ammo', np.int32))

    def __init__(self):
        for s in self.SCALARS:
            setattr(self, s, 0)
        self.reward = np.zeros(K.BGW_RW_COUNT, dtype=np.float64)
        self.agent_ids = []
        self.layout_generator = None     # e.g. ('maze', params) -> host-side layouts (abmarl_b200.layouts)
        self.program_source = None       # PROG_USER: the step program's C source (abmarl_b200.program, bgw_set_program)

    # ---- derived -----------------------------------------------------------------------------
    @property
    def learner_agents(self):
        return [a for a in range(self.n_agents) if self.klass[a] & K.AG_LEARNER]

    @property
    def learner_ids(self):
        return [self.agent_ids[a] for a in self.learner_agents]

    @property
    def n_learners(self):
        return len(self.learner_agents)

    @property
    def max_encoding(self):
        return int(self.encoding.max())

    def obs_shape(self):
        """(h, w, c, stride) -- same rule as bgw_dims."""
        la = [a for a in self.learner_agents if self.klass[a] & K.AG_OBSERVING]
        rmax = max([int(self.view_range[a]) for a in la], default=0)
        if self.observer == K.OBS_ABSOLUTE:
            h, w = self.rows, self.cols
        else:
            h = w = 2 * rmax + 1
        c = self.max_encoding if self.observer == K.OBS_STACKED else 1
        return h, w, c, (h * w * c + 15) // 16 * 16

    def with_envs(self, n_envs, env_offset=0):
        import copy
        s = copy.copy(self)
        s.n_envs, s.env_offset = int(n_envs), int(env_offset)
        return s

    def c_struct(self):
        s = K.BgwSpec()
        s.abi_version = K.BGW_ABI_VERSION
        for name in self.SCALARS:
            setattr(s, name, int(getattr(self, name)))
        for i in range(K.BGW_RW_COUNT):
            s.reward[i] = float(self.reward[i])
        if self.layout_generator is not None:            # MazePlacementState state.py:385-485 / TargetBarriersFreePlacementState :169-279
            p = self.layout_generator[1]
            s.layout_kind = K.LAYOUT_MAZE if self.layout_generator[0] == 'maze' else K.LAYOUT_TARGET_BARRIERS_FREE
            s.layout_target = int(p['target'])
            s.cluster_barriers, s.scatter_free_agents = int(p['cluster_barriers']), int(p['scatter_free_agents'])
            s.barrier_encodings = sum(1 << int(e) for e in p['barrier_encodings'])
            s.free_encodings = sum(1 << int(e) for e in p['free_encodings'])
        keep = []
        for name, dt in self.TABLES + (('overlap', np.uint64), ('attack_map', np.uint64)):
            arr = np.ascontiguousarray(getattr(self, name), dtype=dt)
            keep.append(arr)
            setattr(s, name, arr.ctypes.data_as(C.c_void_p))
        s._keep = keep          # keep the tables alive as long as the struct
        return s


_PROGRAMS = (('PacmanSimSimple', K.PROG_PACMAN_SIMPLE), ('ReachTheTargetSim', K.PROG_REACH_TARGET), ('TrafficCorridorSimulation', K.PROG_TRAFFIC), ('TeamBattleSim', K.PROG_TEAM_BATTLE), ('MultiMazeNavigationSim', K.PROG_MULTI_MAZE),
             ('MazeNavigationSim', K.PROG_MAZE), ('PacmanSim', K.PROG_PACMAN))
_OBSERVERS = (('StackedPositionCenteredEncodingObserver', K.OBS_STACKED),
              ('PositionCenteredEncodingObserver', K.OBS_POSITION_CENTERED),
              ('AbsoluteEncodingObserver', K.OBS_ABSOLUTE))
_DONES = (('OneTeamRemainingDone', K.DONE_ONE_TEAM), ('TargetAgentDone', K.DONE_TARGET_AGENT),
          ('TargetDestroyedDone', K.DONE_TARGET_DESTROYED), ('ActiveDone', K.DONE_ACTIVE))


_SCRIPTED_BADDIES = ('baddie_20', 'baddie_36', 'baddie_156', 'baddie_157', 'baddie_159', 'baddie_161', 'baddie_162',
                     'baddie_206', 'baddie_222', 'baddie_328')


def _first(names, table, what):
    for name, value in table:
        if name in names:
            return value
    raise NotImplementedError(f"no device implementation for this {what}: {sorted(names)}")


def compile_sim(sim, manager='all_step', n_envs=1, env_offset=0, seed=0, horizon=0, auto_reset=False,
                randomize_action_input=False):
    """Flatten `sim` (reference-style object) into a CompiledSpec."""
    sp = CompiledSpec()
    if manager == 'all_step_shuffled':                  # scenario shorthand: AllStepManager(randomize_action_input=True)
        manager, randomize_action_input = 'all_step', True
    names = _mro_names(sim)
    # a sim that declares its own step program runs it, whatever class it derives from (abmarl_b200.program)
    device_program = getattr(sim, 'device_program', None)
    program = device_program() if callable(device_program) else None
    if program is not None:
        if not isinstance(program, DeviceProgram):
            raise TypeError(f"{type(sim).__name__}.device_program() must return an abmarl_b200.program.DeviceProgram")
        if manager == 'dynamic_order':
            raise ValueError("a device program cannot run under the DynamicOrderManager: its next_agent rule is not programmable")
        sp.program = K.PROG_USER
    else:
        sp.program = _first(names, _PROGRAMS, 'simulation class')
    sp.manager = {'all_step': K.MANAGER_ALL_STEP, 'turn_based': K.MANAGER_TURN_BASED,
                  'dynamic_order': K.MANAGER_DYNAMIC_ORDER}[manager]
    if sp.manager == K.MANAGER_DYNAMIC_ORDER:
        # the sim's next_agent rule runs on the device; the one rule built is DynamicOrderMultiMazeSim's (include/bgw.h)
        assert 'DynamicOrderSimulation' in names and 'MultiMazeNavigationSim' in names, \
            "To use the DynamicOrderManager, the simulation must be a DynamicOrderSimulation (built: DynamicOrderMultiMazeSim)."
    sp.rows, sp.cols = int(sim.grid.rows), int(sim.grid.cols)
    assert sp.rows * sp.cols <= 65535, "grid too large for 16-bit cell indices"
    sp.n_envs, sp.env_offset, sp.seed = int(n_envs), int(env_offset), int(seed) & (2**64 - 1)
    sp.horizon, sp.auto_reset = int(horizon), int(bool(auto_reset))
    assert not randomize_action_input or manager == 'all_step', "randomize_action_input is an AllStepManager option"
    sp.randomize_action_input = int(bool(randomize_action_input))    # all_step_manager.py:24-35,62-65

    agents = list(sim.agents.values())
    A = len(agents)
    assert A <= K.BGW_MAX_AGENTS, "too many entities per env"
    sp.n_agents = A
    sp.agent_ids = [a.id for a in agents]
    index = {a.id: i for i, a in enumerate(agents)}
    for name, dt in CompiledSpec.TABLES:
        setattr(sp, name, np.zeros(A, dtype=dt))
    sp.init_row[:] = -1
    sp.init_col[:] = -1
    sp.init_health[:] = math.nan
    sp.target[:] = -1

    for i, ag in enumerate(agents):
        assert 0 < ag.encoding <= K.BGW_MAX_ENCODING, f"{ag.id}: encoding must be in 1..{K.BGW_MAX_ENCODING}"
        sp.encoding[i] = ag.encoding
        k = 0
        acting, observing = hasattr(ag, 'action_space'), hasattr(ag, 'observation_space')
        if hasattr(ag, 'view_range'):
            k |= K.AG_OBSERVING
            sp.view_range[i] = min(int(ag.view_range), 32767)
        if hasattr(ag, 'move_range'):
            k |= K.AG_MOVING
            sp.move_range[i] = ag.move_range
        if hasattr(ag, 'attack_range'):
            k |= K.AG_ATTACKING
            sp.attack_range[i] = ag.attack_range
            sp.attack_strength[i] = ag.attack_strength
            sp.attack_accuracy[i] = ag.attack_accuracy
            sp.simultaneous_attacks[i] = ag.simultaneous_attacks
        if hasattr(ag, 'initial_health'):
            k |= K.AG_HEALTH
            if ag.initial_health is not None:
                sp.init_health[i] = float(ag.initial_health)
        if hasattr(ag, 'initial_orientation'):
            k |= K.AG_ORIENT
            sp.init_orient[i] = ag.initial_orientation or 0
        if hasattr(ag, 'initial_ammo'):
            k |= K.AG_AMMO
            sp.initial_ammo[i] = int(ag.initial_ammo)
        if acting and observing:
            k |= K.AG_LEARNER
        if ag.blocking:
            k |= K.AG_BLOCKING
        sp.klass[i] = k
        if ag.initial_position is not None:
            sp.init_row[i], sp.init_col[i] = int(ag.initial_position[0]), int(ag.initial_position[1])
            assert 0 <= sp.init_row[i] < sp.rows and 0 <= sp.init_col[i] < sp.cols, f"{ag.id}: initial position off grid"

    sp.overlap = _rows(sim.grid.overlapping)

    # ---- actors --------------------------------------------------------------------------------
    sp.attack_map = _rows(None)
    move = getattr(sim, 'move_actor', None)
    if move is not None:
        inner = move
        while hasattr(inner, 'wrapped_component'):
            assert 'RavelActionWrapper' in _mro_names(inner), "only RavelActionWrapper is supported on actors"
            sp.ravel_actions = 1
            inner = inner.wrapped_component
        mn = _mro_names(inner)
        sp.move_actor = K.MOVE_DRIFT if 'DriftMoveActor' in mn else K.MOVE_CROSS if 'CrossMoveActor' in mn \
            else _first(mn, (('MoveActor', K.MOVE_BOX),), 'move actor')
        if sp.ravel_actions:
            assert sp.move_actor == K.MOVE_BOX and int(sp.move_range.max()) <= 7, \
                "ravelled move must fit one byte: move_range <= 7"
    attack = getattr(sim, 'attack_actor', None)
    if attack is not None:
        sp.attack_actor = _first(_mro_names(attack), (
            ('BinaryAttackActor', K.ATTACK_BINARY), ('EncodingBasedAttackActor', K.ATTACK_ENCODING),
            ('RestrictedSelectiveAttackActor', K.ATTACK_RESTRICTED), ('SelectiveAttackActor', K.ATTACK_SELECTIVE)), 'attack actor')
        sp.attack_map = _rows(attack.attack_mapping)
        sp.stacked_attacks = int(bool(attack.stacked_attacks))

    # ---- observers / dones / states ------------------------------------------------------------
    observers = list(getattr(sim, '_observers', None) or [])
    if hasattr(sim, 'grid_observer'):
        observers.append(sim.grid_observer)
    if any('AmmoObserver' in _mro_names(o) for o in observers):            # observer.py:376-413
        sp.ammo_observer = 1
        observers = [o for o in observers if 'AmmoObserver' not in _mro_names(o)]
    if any('AbsolutePositionObserver' in _mro_names(o) for o in observers):    # observer.py:337-373
        sp.position_observer = 1
        observers = [o for o in observers if 'AbsolutePositionObserver' not in _mro_names(o)]
    assert len(observers) == 1, "exactly one grid observer per compiled sim is supported"
    sp.observer = _first(_mro_names(observers[0]), _OBSERVERS, 'observer')
    sp.observe_self = int(getattr(observers[0], 'observe_self', True))
    if sp.observer == K.OBS_STACKED:
        assert A <= 127, "stacked counts are int8"

    for done in list(getattr(sim, '_dones', None) or []):
        sp.done_mask |= _first(_mro_names(done), _DONES, 'done component')
        for agent_id, target_id in getattr(done, 'target_mapping', {}).items():
            sp.target[index[agent_id]] = index[target_id]

    states = list(getattr(sim, '_states', None) or [])
    if hasattr(sim, 'position_state'):
        states.append(sim.position_state)
    for state in states:
        sn = _mro_names(state)
        if 'PositionState' in sn:
            sp.no_overlap_at_reset = int(bool(state.no_overlap_at_reset))
            sp.randomize_placement_order = int(bool(state.randomize_placement_order))    # state.py:97-101
            if 'MazePlacementState' in sn or 'TargetBarriersFreePlacementState' in sn:
                sp.layout_generator = ('maze' if 'MazePlacementState' in sn else 'target_barriers_free', dict(
                    target=index[state.target_agent.id],
                    barrier_encodings=set(state.barrier_encodings), free_encodings=set(state.free_encodings),
                    cluster_barriers=bool(state.cluster_barriers), scatter_free_agents=bool(state.scatter_free_agents)))

    assert not (sp.randomize_placement_order and sp.layout_generator is not None), \
        "randomize_placement_order with a layout-generating placement state is not supported (the generator places in agent order)"

    # ---- program-specific roles and reward constants ----------------------------------------------
    rc = getattr(sim, 'reward_constants', {})
    if sp.program == K.PROG_USER:               # the program carries its own constants and roles
        sp.program_source = program.assemble(sim.agents)
        sp.role[:] = program.role_table(sim.agents)
    elif sp.program == K.PROG_TEAM_BATTLE:      # team_battle_example.py:42-59
        sp.reward[K.RW_ATTACK_FAIL] = rc.get('attack_fail', -0.1)
        sp.reward[K.RW_KILL] = rc.get('kill', 1.0)
        sp.reward[K.RW_DIE] = rc.get('die', -1.0)
        sp.reward[K.RW_MOVE_FAIL] = rc.get('move_fail', -0.1)
        sp.reward[K.RW_ENTROPY] = rc.get('entropy', -0.01)
        # Binary hands TeamBattleSim.step an ndarray: `not attacked_agents` raises for more than one element
        assert sp.attack_actor != K.ATTACK_BINARY or int(sp.simultaneous_attacks.max(initial=0)) <= 1, \
            "TeamBattleSim.step with the BinaryAttackActor is only defined for simultaneous_attacks == 1 (team_battle_example.py:41)"
    elif sp.program == K.PROG_TRAFFIC:          # traffic_corridor.py:46-53
        sp.reward[K.RW_MOVE_FAIL] = rc.get('move_fail', -0.1)
        sp.reward[K.RW_TARGET] = rc.get('target', 1.0)
        assert sp.done_mask == K.DONE_TARGET_AGENT, "TrafficCorridorSimulation.step rewards TargetAgentDone.get_done"
    elif sp.program == K.PROG_REACH_TARGET:     # reach_the_target.py:117-152
        sp.reward[K.RW_ATTACK_FAIL] = rc.get('attack_fail', -0.1)
        sp.reward[K.RW_KILL] = rc.get('kill', 1.0)
        sp.reward[K.RW_DIE] = rc.get('die', -1.0)
        sp.reward[K.RW_MOVE_FAIL] = rc.get('move_fail', -0.1)
        sp.reward[K.RW_TARGET] = rc.get('target', 1.0)
        sp.reward[K.RW_ENTROPY] = rc.get('entropy', -0.01)
        sp.role[index[sim.target.id]] = K.ROLE_TARGET
        for i, ag in enumerate(agents):
            if 'RunningAgent' in _mro_names(ag):
                sp.role[i] = K.ROLE_RUNNER
        assert sp.attack_actor != K.ATTACK_BINARY or int(sp.simultaneous_attacks.max(initial=0)) <= 1
    elif sp.program in (K.PROG_MAZE, K.PROG_MULTI_MAZE):   # maze_navigation.py:29-36, multi_maze_navigation.py:45-59
        sp.reward[K.RW_MOVE_FAIL] = rc.get('move_fail', -0.1)
        sp.reward[K.RW_TARGET] = rc.get('target', 1.0)
        sp.reward[K.RW_ENTROPY] = rc.get('entropy', -0.01)
        if sp.program == K.PROG_MAZE:
            sp.role[index['navigator']] = K.ROLE_NAVIGATOR
            sp.role[index['target']] = K.ROLE_TARGET
        else:
            sp.role[index[sim.position_state.target_agent.id]] = K.ROLE_TARGET
            for i, ag in enumerate(agents):
                if 'MultiMazeNavigationAgent' in _mro_names(ag):
                    sp.role[i] = K.ROLE_NAVIGATOR
    elif sp.program in (K.PROG_PACMAN, K.PROG_PACMAN_SIMPLE):   # pacman.py:72-78, 196-212
        scheme = {'bad_move': -0.1, 'entropy': 0.01, 'eat_food': 0.1, 'kill': 1, 'die': -1}
        scheme.update(sim.reward_scheme)
        sp.reward[K.RW_MOVE_FAIL] = scheme['bad_move']
        sp.reward[K.RW_ENTROPY] = scheme['entropy']
        sp.reward[K.RW_EAT_FOOD] = scheme['eat_food']
        sp.reward[K.RW_KILL] = scheme['kill']
        sp.reward[K.RW_DIE] = scheme['die']
        for i, ag in enumerate(agents):
            n = _mro_names(ag)
            sp.role[i] = K.ROLE_PACMAN if ag.id == 'pacman' else K.ROLE_FOOD if 'FoodAgent' in n else \
                K.ROLE_BADDIE if 'BaddieAgent' in n else K.ROLE_WALL if 'WallAgent' in n else K.ROLE_NONE
            if sp.program == K.PROG_PACMAN_SIMPLE and ag.id in _SCRIPTED_BADDIES:     # pacman.py:235-246
                sp.role[i] = K.ROLE_SCRIPTED_BADDIE + _SCRIPTED_BADDIES.index(ag.id)
        assert sp.rows > 9 and sp.cols > 20, "PacmanSim hardcodes the (9,0)<->(9,20) tunnel (pacman.py:87-92)"
    return sp
