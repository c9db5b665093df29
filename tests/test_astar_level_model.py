"""The level-synchronous statement of astar_4 (csrc/astar4.cuh, restated in NumPy as tests/astar_util.level_astar) equals
the heap version `episode_io.astar_path` path for path, and the reference's training human walks that path.  CPU only."""
import os

import numpy as np
import pytest

from astar_util import GOLDEN, golden_cases, human_legs, level_astar, random_cases
from primal_ppo_b200.episode_io import astar_path

G = np.load(os.path.join(GOLDEN, "training_env.npz"))


def _same(world, s, g):
    a, b = astar_path(world, s, g), level_astar(world, s, g)
    assert a == b, (world.shape, s, g, a, b)
    return a


def test_level_model_on_reference_paths():
    for world, s, g in golden_cases():
        _same(world, s, g)


@pytest.mark.parametrize("part", range(4))
def test_level_model_on_random_maps(part):
    cases = random_cases()
    kinds = {"none": 0, "empty": 0, "path": 0}
    for world, s, g in cases[part::4]:
        p = _same(world, s, g)
        kinds["none" if p is None else "empty" if p == [] else "path"] += 1
    assert min(kinds.values()) > 0, kinds


def test_level_model_edge_cases():
    world = np.zeros((5, 7), dtype=np.int64)
    assert level_astar(world, (2, 3), (2, 3)) == []
    world[0, 6] = -1
    assert level_astar(world, (4, 0), (0, 6)) is None                          # blocked goal
    world[1, 5] = world[0, 5] = world[1, 6] = -1
    world[0, 6] = 0
    assert level_astar(world, (4, 0), (0, 6)) is None                          # unreachable goal
    world[4, 0] = -1
    _same(world, (4, 0), (2, 2))                                               # a blocked start is still expanded
    # padding a map with walls keeps every path
    rng = np.random.default_rng(5)
    for _ in range(50):
        m = -(rng.random((9, 11)) < 0.25).astype(np.int64)
        pad = np.full((16, 20), -1, dtype=np.int64)
        pad[:9, :11] = m
        s, g = tuple(int(x) for x in rng.integers(0, 9, 2)), tuple(int(x) for x in rng.integers(0, 9, 2))
        assert astar_path(m, s, g) == level_astar(pad, s, g)


def test_training_human_walks_astar_path():
    """In every recorded training world, each out-and-back walk whose turning point is inside the recorded ticks goes
    out along astar_path(map, entrance, turning cell): the reference's training Human plans with exactly this call."""
    legs = 0
    for ci in range(int(G["n_cases"])):
        obst, dims, htrace = G[f"c{ci}_obst"], G[f"c{ci}_dims"], G[f"c{ci}_htrace"]
        for w in range(obst.shape[0]):
            rows, cols = (int(x) for x in dims[w])
            world = -(obst[w, :rows, :cols] != 0).astype(np.int64)
            for ent, turn, out in human_legs(htrace[w]):
                assert astar_path(world, ent, turn) == out, (ci, w, ent, turn)
                legs += 1
    assert legs >= 40
