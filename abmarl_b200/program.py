"""DeviceProgram: a user-written step() for the device, as a C step program (include/bgw_program.h).

A simulation class that the engine has no built-in program for declares its step() -- and, if it overrides them, get_done,
get_all_done and get_reward -- as C source with a `device_program()` method:

    class ForagingSim(SmartGridWorldSimulation):
        def device_program(self):
            return DeviceProgram(SOURCE, constants={'KILL': 1.0, 'TARGET': self.agents['target']},
                                 roles={agent: 1 for agent in self.agents.values() if isinstance(agent, Forager)})

compile_sim() then compiles the sim to BGW_PROG_USER with the assembled source, the engine compiles it into its step kernel
at run time (bgw_set_program) and the CPU oracle compiles the same text with gcc.  abmarl_b200/examples/foraging.py is a
complete example.
"""
import math
import re

_NAME = re.compile(r'[A-Za-z_][A-Za-z0-9_]*\Z')
_RESERVED_PREFIXES = ('bgw', 'BGW', '__')
_C_KEYWORDS = frozenset('''auto break case char const continue default do double else enum extern float for goto if inline int long
register restrict return short signed sizeof static struct switch typedef union unsigned void volatile while bool true false
class delete new namespace template this typename using virtual operator private public protected friend nullptr'''.split())


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
    (bgwp_role)."""

    def __init__(self, source, constants=None, roles=None):
        if not isinstance(source, str) or not source.strip():
            raise ValueError("the program source must be a non-empty string")
        self.source = source
        self.constants = dict(constants or {})
        self.roles = dict(roles or {})
        for name, value in self.constants.items():
            if not isinstance(name, str) or not _NAME.match(name) or name in _C_KEYWORDS or name.startswith(_RESERVED_PREFIXES):
                raise ValueError(f"constant name {name!r} is not a C identifier of the program's own "
                                 f"(names starting with {', '.join(_RESERVED_PREFIXES)} are the API's)")
            if isinstance(value, float) and not math.isfinite(value):
                raise ValueError(f"constant {name} = {value}: only finite numbers have a C literal")
        for agent, role in self.roles.items():
            if not isinstance(role, int) or isinstance(role, bool) or not 0 <= role <= 255:
                raise ValueError(f"role {role!r} of {agent!r} must be an int in 0..255")

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
        return '\n'.join(lines + [self.source])

    def role_table(self, agents):
        """uint8 role per agent (0 for the agents `roles` does not name)."""
        index = {agent_id: i for i, agent_id in enumerate(agents)}
        table = [0] * len(index)
        for agent, role in self.roles.items():
            table[_agent_index(agent, index)] = role
        return table
