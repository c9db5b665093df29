"""primal_ppo_b200 — B200-native batched MAPF environment hot path (step / observe / BFS / GAE).

Host side (this package) mirrors the reference's ``MapfGym`` method surface; all arithmetic runs in hand-written
sm_100a CUDA kernels behind the C ABI of ``include/mapf_b200.h`` (``libmapf_b200.so``).  No CPU fallback.
"""
from .scenario import Scenario, random_scenario, random_actions, looping_trace  # noqa: F401

__all__ = ["Scenario", "random_scenario", "random_actions", "looping_trace", "BatchedMapfGym", "StepOut", "gae", "gae2",
           "sample_actions", "checksum_rows", "decode_results", "unpack_observations", "DeviceScenario",
           "generate_scenario_device"]


def __getattr__(name):
    # torch / CUDA are only needed for the env itself; scenario tooling imports without them
    if name in ("BatchedMapfGym", "StepOut", "gae", "gae2", "sample_actions", "checksum_rows", "decode_results",
                "unpack_observations"):
        from . import vec_env
        return getattr(vec_env, name)
    if name in ("DeviceScenario", "generate_scenario_device"):
        from . import device_scenario
        return getattr(device_scenario, name)
    raise AttributeError(name)
