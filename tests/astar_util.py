"""Shared by the A* tests: a NumPy statement of the level-synchronous astar_4 (what csrc/astar4.cuh computes), the map
set both the CPU model test and the GPU test compare against `episode_io.astar_path`, and the leg finder that reads the
human's out-and-back walks out of a (pos, next) trace."""
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def level_astar(world, start, goal):
    """astar_path(world, start, goal) computed level by level (the four facts of csrc/astar4.cuh): the open cells that
    share the minimum (f, g) expand at once, a reached cell's parent is the highest-index member of the level next to
    it, and the search stops when the goal is in the minimum level."""
    H, Wd = world.shape
    start, goal = (int(start[0]), int(start[1])), (int(goal[0]), int(goal[1]))
    if start == goal:
        return []
    free = (world != -1).ravel()
    s, t = start[0] * Wd + start[1], goal[0] * Wd + goal[1]
    g = np.full(H * Wd, -1, dtype=np.int64)
    parent = np.full(H * Wd, -1, dtype=np.int64)
    closed = np.zeros(H * Wd, dtype=bool)
    g[s] = 0
    open_ = {s}

    def key(c):
        return (g[c] + abs(c // Wd - goal[0]) + abs(c % Wd - goal[1]), g[c])
    while open_:
        best = min(key(c) for c in open_)
        fs = {key(c)[0] for c in open_}
        assert fs <= {best[0], best[0] + 2}, "fact 2: two f values open at a time"
        if t in open_ and key(t) == best:
            path = [t]
            while path[-1] != s:
                path.append(parent[path[-1]])
            return [(int(c) // Wd, int(c) % Wd) for c in path[::-1]]
        lvl = {c for c in open_ if key(c) == best}
        open_ -= lvl
        for m in lvl:
            closed[m] = True
        ng = best[1] + 1
        for m in lvl:
            r, col = divmod(m, Wd)
            for n, ok in ((m - 1, col > 0), (m - Wd, r > 0), (m + 1, col + 1 < Wd), (m + Wd, r + 1 < H)):
                if not ok or not free[n] or closed[n] or 0 <= g[n] < ng:
                    continue
                nr, nc = divmod(n, Wd)
                adj = [a for a, aok in ((n + Wd, nr + 1 < H), (n + 1, nc + 1 < Wd), (n - 1, nc > 0), (n - Wd, nr > 0))
                       if aok and a in lvl]
                g[n], parent[n] = ng, max(adj)
                open_.add(n)
    return None


def golden_cases():
    """The 400 (world, start, goal) triples of tests/golden/astar_paths.npz (paths produced by the reference's astar_4)."""
    d = np.load(os.path.join(GOLDEN, "astar_paths.npz"))
    return [(d[f"world{k}"].astype(np.int64), tuple(int(x) for x in d[f"sg{k}"][0]), tuple(int(x) for x in d[f"sg{k}"][1]))
            for k in range(int(d["count"]))]


def random_cases(n=3000, seed=0, big=3):
    """Maps of density 0 to 0.45, warehouses, open grids (many ties), 1 x n and n x 1 strips, and `big` 128 x 128 maps,
    with a start and a goal each; some goals are blocked, unreachable, or equal to the start."""
    rng = np.random.default_rng(seed)
    wh = np.load(os.path.join(GOLDEN, "warehouse_maps.npz"))
    whs = [wh[k] for k in wh.files]
    out = []
    for i in range(n + big):
        kind = i % 5
        if i >= n:
            H = Wd = 128
            world = -(rng.random((H, Wd)) < rng.uniform(0.0, 0.4)).astype(np.int64)
        elif kind == 0:                                   # density maps
            H, Wd = int(rng.integers(2, 33)), int(rng.integers(2, 33))
            world = -(rng.random((H, Wd)) < rng.uniform(0.0, 0.45)).astype(np.int64)
        elif kind == 1:                                   # warehouses of the training env
            world = -(whs[int(rng.integers(len(whs)))] != 0).astype(np.int64)
        elif kind == 2:                                   # open grids: every shortest path ties
            H, Wd = int(rng.integers(2, 41)), int(rng.integers(2, 41))
            world = np.zeros((H, Wd), dtype=np.int64)
            if rng.random() < 0.5:
                world[rng.random((H, Wd)) < 0.03] = -1
        elif kind == 3:                                   # strips
            L = int(rng.integers(1, 50))
            world = -(rng.random((1, L) if rng.random() < 0.5 else (L, 1)) < 0.1).astype(np.int64)
        else:                                             # small and crowded: many unreachable goals
            H, Wd = int(rng.integers(1, 12)), int(rng.integers(1, 12))
            world = -(rng.random((H, Wd)) < rng.uniform(0.3, 0.6)).astype(np.int64)
        H, Wd = world.shape
        freec = np.argwhere(world == 0)
        pick = lambda: (tuple(int(x) for x in freec[rng.integers(len(freec))]) if len(freec) and rng.random() < 0.95
                        else (int(rng.integers(H)), int(rng.integers(Wd))))
        s, g = pick(), pick()
        if rng.random() < 0.03:
            g = s
        out.append((world, s, g))
    return out


def human_legs(trace):
    """(entrance, turning cell, out-half cells) of every out-and-back walk of a (pos, next) trace [T, 4] whose turning
    point falls inside the trace: a walk leaves the entrance at the last tick of a stay there and turns where the next
    cell equals the previous one."""
    p = [tuple(int(x) for x in row[:2]) for row in trace]
    ent, legs = p[0], []
    for a in range(len(p) - 1):
        if p[a] != ent or p[a + 1] == ent:
            continue
        for b in range(a + 1, len(p) - 1):
            if p[b + 1] == p[b - 1]:
                legs.append((ent, p[b], p[a:b + 1]))
                break
    return legs
