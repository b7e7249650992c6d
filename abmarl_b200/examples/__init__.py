"""Example simulations (definitions): the four sims named by the BASELINE configs, ReachTheTargetSim, and ForagingSim (a sim
of its own that runs through a step program, abmarl_b200.program)."""
from .sims import (  # noqa: F401
    BattleAgent, TeamBattleSim,
    MazeNavigationAgent, MazeNavigationSim,
    MultiMazeNavigationAgent, MultiMazeNavigationSim, DynamicOrderMultiMazeSim,
    PacmanAgent, WallAgent, FoodAgent, BaddieAgent, PacmanSim, PacmanSimSimple,
    BarrierAgent, TargetAgent, RunningAgent, ReachTheTargetSim, TargetDone, OnlyAgentLeftDone,
)
from .foraging import Forager, Predator, Resource, ForagingSim  # noqa: F401,E402
