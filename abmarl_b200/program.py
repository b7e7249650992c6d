"""DeviceProgram: a user-written step() for the device, as a C step program (include/bgw_program.h).

A simulation class that the engine has no built-in program for declares its step() -- and, if it overrides them, get_done,
get_all_done and get_reward -- as C source with a `device_program()` method:

    class ForagingSim(SmartGridWorldSimulation):
        def device_program(self):
            return DeviceProgram(SOURCE, constants={'KILL': 1.0, 'TARGET': self.agents['target']},
                                 roles={agent: 1 for agent in self.agents.values() if isinstance(agent, Forager)})

compile_sim() then compiles the sim to BGW_PROG_USER with the assembled source, the engine compiles it into its step kernel
at run time (bgw_set_program) and the CPU oracle compiles the same text with gcc.  abmarl_b200/examples/foraging.py is a
complete example; abmarl_b200/examples/king_of_the_hill.py keeps variables of its own (env_vars, agent_vars).
"""
import math
import numbers
import re

_NAME = re.compile(r'[A-Za-z_][A-Za-z0-9_]*\Z')
_RESERVED_PREFIXES = ('bgw', 'BGW', '__')
_C_KEYWORDS = frozenset('''auto break case char const continue default do double else enum extern float for goto if inline int long
register restrict return short signed sizeof static struct switch typedef union unsigned void volatile while bool true false
class delete new namespace template this typename using virtual operator private public protected friend nullptr'''.split())


def _check_name(name, what):
    if not isinstance(name, str) or not _NAME.match(name) or name in _C_KEYWORDS or name.startswith(_RESERVED_PREFIXES):
        raise ValueError(f"{what} name {name!r} is not a C identifier of the program's own "
                         f"(names starting with {', '.join(_RESERVED_PREFIXES)} are the API's)")


def _number(value, what):
    """A finite int or float (not a bool) as a float; raises otherwise."""
    if isinstance(value, bool) or not isinstance(value, numbers.Real) or not math.isfinite(float(value)):
        raise ValueError(f"{what} = {value!r}: must be a finite number")
    return float(value)


def _agent_index(value, index):
    """An agent id or an agent object -> its index in sim.agents; raises for anything else."""
    agent_id = value if isinstance(value, str) else getattr(value, 'id', None)
    if not isinstance(agent_id, str) or agent_id not in index:
        raise ValueError(f"{value!r} is not an agent of this simulation")
    return index[agent_id]


class DeviceProgram:
    """A step program: `source` (C, include/bgw_program.h), `constants` {C identifier: int | float | agent} emitted as
    #defines ahead of it (agents become their index in sim.agents; floats are written as C99 hex literals, so the device
    and the oracle read the very same double), and `roles` {agent: 0..255} written into the spec's role table
    (bgwp_role).

    The program's own variables, float64 values that persist between steps and are set to their initial values by every
    reset (bgwp_env_var / bgwp_agent_var):
      env_vars    {C identifier: float | sequence of floats}: a scalar, or an array of that many slots initialised to the
                  sequence's values
      agent_vars  {C identifier: float | {agent or agent id: float}}: one value per entity of sim.agents, initialised to
                  the float, or to the dict's value (0.0 for the entities it does not name)
    Each name is #defined as its index: the env slot (an array's first slot) or the agent variable's k."""

    def __init__(self, source, constants=None, roles=None, env_vars=None, agent_vars=None):
        if not isinstance(source, str) or not source.strip():
            raise ValueError("the program source must be a non-empty string")
        self.source = source
        self.constants = dict(constants or {})
        self.roles = dict(roles or {})
        self.env_vars = dict(env_vars or {})
        self.agent_vars = dict(agent_vars or {})
        for name, value in self.constants.items():
            _check_name(name, 'constant')
            if isinstance(value, float) and not math.isfinite(value):
                raise ValueError(f"constant {name} = {value}: only finite numbers have a C literal")
        for agent, role in self.roles.items():
            if not isinstance(role, int) or isinstance(role, bool) or not 0 <= role <= 255:
                raise ValueError(f"role {role!r} of {agent!r} must be an int in 0..255")
        seen = set(self.constants)
        for name in list(self.env_vars) + list(self.agent_vars):
            _check_name(name, 'variable')
            if name in seen:
                raise ValueError(f"variable name {name!r} is used twice (constants and variables share the #define names)")
            seen.add(name)
        for name, value in self.env_vars.items():
            if isinstance(value, (str, bytes)) or not hasattr(value, '__len__'):
                _number(value, f"env variable {name}")
            elif len(value) == 0:
                raise ValueError(f"env variable {name}: an array needs at least one slot")
            else:
                for i, x in enumerate(value):
                    _number(x, f"env variable {name}[{i}]")
        for name, value in self.agent_vars.items():
            for agent, x in (value.items() if isinstance(value, dict) else [(None, value)]):
                _number(x, f"agent variable {name}" + ('' if agent is None else f" of {agent!r}"))

    def env_var_slots(self):
        """{name: (first slot, None for a scalar | number of slots of an array)} in declaration order."""
        out, k = {}, 0
        for name, value in self.env_vars.items():
            n = None if not hasattr(value, '__len__') else len(value)
            out[name] = (k, n)
            k += 1 if n is None else n
        return out

    @property
    def n_env_vars(self):
        return sum(1 if n is None else n for _, n in self.env_var_slots().values())

    @property
    def n_agent_vars(self):
        return len(self.agent_vars)

    def var_init(self, agents):
        """float64 initial row of the variables: the env slots, then [A][n_agent_vars] (the layout of bgw_set_program_vars).
        `agents` is the sim's agents dict (indices = dict order)."""
        index = {agent_id: i for i, agent_id in enumerate(agents)}
        row = []
        for value in self.env_vars.values():
            row += [float(x) for x in value] if hasattr(value, '__len__') else [float(value)]
        per_agent = [[0.0] * self.n_agent_vars for _ in index]
        for k, value in enumerate(self.agent_vars.values()):
            if isinstance(value, dict):
                for agent, x in value.items():
                    per_agent[_agent_index(agent, index)][k] = float(x)
            else:
                for a in range(len(index)):
                    per_agent[a][k] = float(value)
        return row + [x for values in per_agent for x in values]

    def assemble(self, agents):
        """The source the engine and the oracle compile: the constants as #defines, then the program.  `agents` is the
        sim's agents dict (indices = dict order)."""
        index = {agent_id: i for i, agent_id in enumerate(agents)}
        lines = []
        for name, value in self.constants.items():
            if isinstance(value, bool):
                text = str(int(value))
            elif isinstance(value, int):
                text = str(value)
            elif isinstance(value, float):
                text = value.hex()
            else:
                text = str(_agent_index(value, index))
            lines.append(f"#define {name} ({text})")
        for name, (k, _) in self.env_var_slots().items():
            lines.append(f"#define {name} ({k})")
        for k, name in enumerate(self.agent_vars):
            lines.append(f"#define {name} ({k})")
        return '\n'.join(lines + [self.source])

    def role_table(self, agents):
        """uint8 role per agent (0 for the agents `roles` does not name)."""
        index = {agent_id: i for i, agent_id in enumerate(agents)}
        table = [0] * len(index)
        for agent, role in self.roles.items():
            table[_agent_index(agent, index)] = role
        return table
