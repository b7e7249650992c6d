"""Host-side mirror of abmarl/sim/agent_based_simulation.py.

Same class names, constructor arguments and validation as the reference so an existing sim definition
builds unchanged; the objects are *declarations* that abmarl_b200.spec.compile_sim() flattens into the
device spec -- they hold no per-step state (that lives in HBM, one copy per env).
"""
from abc import ABC, abstractmethod

from abmarl_b200 import spaces as gu


class PrincipleAgent:
    """agent_based_simulation.py:7-57"""

    def __init__(self, id=None, seed=None, **kwargs):
        self.id = id
        self.seed = seed
        self.active = True

    @property
    def id(self):
        return self._id

    @id.setter
    def id(self, value):
        assert type(value) is str, "id must be a string."
        self._id = value

    @property
    def seed(self):
        return self._seed

    @seed.setter
    def seed(self, value):
        assert value is None or type(value) is int, "Seed must be an integer."
        self._seed = value

    @property
    def active(self):
        return self._active

    @active.setter
    def active(self, value):
        assert type(value) is bool, "Active must be either True or False."
        self._active = value

    @property
    def configured(self):
        return self.id is not None

    def finalize(self, **kwargs):
        pass

    def __eq__(self, other):
        return self.__dict__ == other.__dict__ if isinstance(other, self.__class__) else False

    __hash__ = object.__hash__


class ActingAgent(PrincipleAgent):
    """agent_based_simulation.py:60-117"""

    def __init__(self, action_space=None, null_action=None, **kwargs):
        super().__init__(**kwargs)
        self.action_space = action_space
        self.null_action = null_action

    @property
    def action_space(self):
        return self._action_space

    @action_space.setter
    def action_space(self, value):
        assert value is None or gu.check_space(value), \
            "The action space must be None, a Space, or a dict of Spaces."
        self._action_space = {} if value is None else value

    @property
    def null_action(self):
        return self._null_action

    @null_action.setter
    def null_action(self, value):
        self._null_action = {} if value is None else value

    @property
    def configured(self):
        return super().configured and gu.check_space(self.action_space, strict=True)

    def finalize(self, **kwargs):
        super().finalize(**kwargs)
        if type(self.action_space) is dict:
            self.action_space = gu.make_dict(self.action_space)
        self.action_space.seed(self.seed)
        if self.null_action:
            assert self.null_action in self.action_space, \
                "The null action must be in the action space."


class ObservingAgent(PrincipleAgent):
    """agent_based_simulation.py:120-171"""

    def __init__(self, observation_space=None, null_observation=None, **kwargs):
        super().__init__(**kwargs)
        self.observation_space = observation_space
        self.null_observation = null_observation

    @property
    def observation_space(self):
        return self._observation_space

    @observation_space.setter
    def observation_space(self, value):
        assert value is None or gu.check_space(value), \
            "The observation space must be None, a Space, or a dict of Spaces."
        self._observation_space = {} if value is None else value

    @property
    def null_observation(self):
        return self._null_observation

    @null_observation.setter
    def null_observation(self, value):
        self._null_observation = {} if value is None else value

    @property
    def configured(self):
        return super().configured and gu.check_space(self.observation_space, strict=True)

    def finalize(self, **kwargs):
        super().finalize(**kwargs)
        if type(self.observation_space) is dict:
            self.observation_space = gu.make_dict(self.observation_space)
        self.observation_space.seed(self.seed)
        if self.null_observation:
            assert self.null_observation in self.observation_space, \
                "The null observation must be in the observation space."


class AgentMeta(type):
    """An Agent is anything that both observes and acts (agent_based_simulation.py:174-181)."""

    def __instancecheck__(self, instance):
        return isinstance(instance, ObservingAgent) and isinstance(instance, ActingAgent)


class Agent(ObservingAgent, ActingAgent, metaclass=AgentMeta):
    pass


class AgentBasedSimulation(ABC):
    """agent_based_simulation.py:189-294 (the pull interface).

    In this package a simulation object is a *definition*: `reset/step/get_*` are executed on the GPU for
    every env of the batch by the engine the manager owns, so the per-agent getters are not host methods.
    """

    def __init__(self, agents=None, **kwargs):
        self.agents = agents

    @property
    def agents(self):
        return self._agents

    @agents.setter
    def agents(self, value_agents):
        assert type(value_agents) is dict, "Agents must be a dict"
        for agent_id, agent in value_agents.items():
            assert isinstance(agent, PrincipleAgent), "Values of agents dict must be instance of PrincipleAgent."
            assert agent_id == agent.id, "Keys of agents dict must be the same as the Agent's id."
        self._agents = value_agents

    def finalize(self):
        for agent in self.agents.values():
            agent.finalize()
            assert agent.configured, f"Agent {agent.id} is not configured."

    @abstractmethod
    def program(self):
        """Which built-in device program reproduces this sim's step()/get_* (BGW_PROG_*)."""


class DynamicOrderSimulation(AgentBasedSimulation):
    """agent_based_simulation.py:297-317: an AgentBasedSimulation where the simulation chooses the agents' turns
    dynamically.  On the device the choice is part of the step kernel (BGW_MANAGER_DYNAMIC_ORDER, include/bgw.h): built in for
    DynamicOrderMultiMazeSim, a step program's next_agent hook otherwise (include/bgw_program.h); this
    declaration keeps the reference's property for host-side code that inspects it."""

    @property
    def next_agent(self):
        """The next agent(s) in the game."""
        return self._next_agent

    @next_agent.setter
    def next_agent(self, value):
        assert isinstance(value, (list, tuple, set, frozenset, dict, str)), \
            "The next agent must be a single string or a Container of strings."
        if type(value) is str:
            value = [value]
        for agent_id in value:
            assert agent_id in self.agents, "Every next agent must be an agent in the simulation."
        self._next_agent = value

