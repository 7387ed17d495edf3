"""B200-native per-timestep agent update of rmf_crowdsim (LocationHash2D rebuild + radius query,
Zanlungo social force, Euler integration) behind the reference's own interface.  See DESIGN.md."""
from ._native import RcsError as CrowdsimError  # noqa: F401
from .sim import (  # noqa: F401
    Agent,
    ConstantVelocityPlan,
    CrowdGenerator,
    Duration,
    EventListener,
    HighLevelPlanner,
    LocalPlanner,
    LocationHash2D,
    MonotonicCrowd,
    NoHighLevelPlan,
    NoLocalPlan,
    ParityVelocityPlan,
    PoissonCrowd,
    RouteFollowPlan,
    RouteTablePlan,
    Simulation,
    SourceSink,
    Zanlungo,
)

__all__ = [
    "Agent", "ConstantVelocityPlan", "CrowdGenerator", "CrowdsimError", "Duration", "EventListener",
    "HighLevelPlanner", "LocalPlanner", "LocationHash2D", "MonotonicCrowd", "NoHighLevelPlan", "NoLocalPlan",
    "ParityVelocityPlan", "PoissonCrowd", "RouteFollowPlan", "RouteTablePlan", "Simulation", "SourceSink", "Zanlungo",
]
