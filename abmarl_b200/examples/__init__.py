"""Example simulations (definitions): the four sims named by the BASELINE configs, ReachTheTargetSim, ForagingSim (a sim
of its own that runs through a step program, abmarl_b200.program), AlternatingBattleSim (teams that take turns under the
DynamicOrderManager, through a step program's next_agent hook) and KingOfTheHillSim (teams that contest a hill, through a
step program with variables of its own)."""
from .sims import (  # noqa: F401
    BattleAgent, TeamBattleSim,
    MazeNavigationAgent, MazeNavigationSim,
    MultiMazeNavigationAgent, MultiMazeNavigationSim, DynamicOrderMultiMazeSim,
    PacmanAgent, WallAgent, FoodAgent, BaddieAgent, PacmanSim, PacmanSimSimple,
    BarrierAgent, TargetAgent, RunningAgent, ReachTheTargetSim, TargetDone, OnlyAgentLeftDone,
)
from .foraging import Forager, Predator, Resource, ForagingSim  # noqa: F401,E402
from .alternating_battle import AlternatingBattleSim  # noqa: F401,E402
from .king_of_the_hill import KingOfTheHillSim  # noqa: F401,E402
