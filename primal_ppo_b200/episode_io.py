"""Evaluation fixtures of the reference (SURVEY.md §8 f4): read / write the `fixed_episode_infos` folder that
`evaluate.py` produces (`evaluate.py:33-35, 104-135`) and turn its episodes into ONE batched `Scenario`, so that a
reference-trained checkpoint can be evaluated on the reference's own fixed episodes with every episode running as a
world of the GPU vector env.

Folder layout (`saveFixedEpisodeInfos`, `evaluate.py:104-121`): `infos.json` with keys `obstacleMap` (file names
`obstacleMap{i}.npy`, int64 arrays with -1 = shelf), `agentsSequence` (per episode, per agent: list of [r, c]; item 0 is the
start, the rest are goals), `humanSequence`, `humanStart`, `humanGoal`, `numEpisodes`.

The human's walk is not stored in the fixture: the reference recomputes it with `astar_4` (`mapf_gym.py:33-37, 80-82`).
To replay the SAME episode the same path is needed, so `astar_path` below restates `astar_4.py:21-109` including its
tie-breaking (heap order on (f, g, cell, parent), neighbour order left / up / right / down, parents overwritten on equal
cost); it is pinned against paths produced by the reference (`tests/golden/astar_paths.npz`).  This is host-side input
preparation, run once per evaluation, not part of the stepped path.
"""
from __future__ import annotations

import json
import os
from heapq import heappop, heappush
from typing import Dict, List, Optional, Sequence as Seq, Tuple

import numpy as np

from .scenario import Scenario

Cell = Tuple[int, int]


# ---- fixture I/O --------------------------------------------------------------------------------------------------
def load_fixed_episode_infos(folder: str) -> Dict:
    """`loadFixedEpisodeInfos` (`evaluate.py:123-135`); agent sequences come back as plain lists of (r, c) tuples."""
    with open(os.path.join(folder, "infos.json")) as f:
        j = json.load(f)
    n = int(j["numEpisodes"])
    return {"obstacleMap": [np.load(os.path.join(folder, j["obstacleMap"][i])) for i in range(n)],
            "agentsSequence": [[[tuple(int(x) for x in it) for it in items] for items in j["agentsSequence"][i]] for i in range(n)],
            "humanSequence": [[tuple(int(x) for x in p) for p in j["humanSequence"][i]] for i in range(n)],
            "humanStart": [tuple(int(x) for x in p) for p in j["humanStart"]],
            "humanGoal": [tuple(int(x) for x in p) for p in j["humanGoal"]],
            "numEpisodes": n}


def save_fixed_episode_infos(infos: Dict, folder: str) -> None:
    """`saveFixedEpisodeInfos` (`evaluate.py:104-121`): same file names, same JSON keys (sorted, indent 4)."""
    os.makedirs(folder, exist_ok=True)
    n = int(infos["numEpisodes"])
    names = []
    for i in range(n):
        name = f"obstacleMap{i}.npy"
        np.save(os.path.join(folder, name), np.asarray(infos["obstacleMap"][i]))
        names.append(name)
    plain = lambda p: [int(p[0]), int(p[1])]
    out = {"obstacleMap": names,
           "agentsSequence": [[[plain(it) for it in getattr(seq, "items", seq)] for seq in infos["agentsSequence"][i]] for i in range(n)],
           "humanSequence": [[plain(p) for p in infos["humanSequence"][i]] for i in range(n)],
           "humanStart": [plain(p) for p in infos["humanStart"][:n]],
           "humanGoal": [plain(p) for p in infos["humanGoal"][:n]],
           "numEpisodes": n}
    with open(os.path.join(folder, "infos.json"), "w", encoding="utf-8") as f:
        json.dump(out, f, ensure_ascii=False, indent=4, sort_keys=True)


# ---- the human's walk -------------------------------------------------------------------------------------------------
def astar_path(world: np.ndarray, start: Cell, goal: Cell) -> Optional[List[Cell]]:
    """Path start -> goal (inclusive) with the exact tie-breaking of `astar_4` (`astar_4.py:21-109`); cells with value -1
    are walls.  Returns [] when start == goal (`:31-32`) and None when no path exists (`:109`)."""
    start, goal = (int(start[0]), int(start[1])), (int(goal[0]), int(goal[1]))
    if start == goal:
        return []
    H, Wd = world.shape
    blocked = world == -1
    heap = [(0, 0, start, None)]                 # (f, g, cell, parent): ties fall through to the cell, then the parent
    closed = set()
    g_best: Dict[Cell, int] = {}
    parent: Dict[Cell, Cell] = {}
    while heap:
        _, g, cur, _ = heappop(heap)
        if cur == goal:
            path = [goal]
            while path[-1] != start:
                path.append(parent[path[-1]])
            return path[::-1]
        if cur in closed:
            continue
        closed.add(cur)
        r, c = cur
        for nr, nc in ((r, c - 1), (r - 1, c), (r, c + 1), (r + 1, c)):          # left, up, right, down (:52-106)
            if not (0 <= nr < H and 0 <= nc < Wd) or blocked[nr, nc] or (nr, nc) in closed:
                continue
            nb = (nr, nc)
            if nb in g_best and g_best[nb] < g + 1:
                par = parent[nb]                                                  # a strictly better route is already known
            else:
                g_best[nb] = g + 1                                                # equal cost overwrites the parent (:56-61)
                parent[nb] = cur
                par = cur
            heappush(heap, (abs(nr - goal[0]) + abs(nc - goal[1]) + g_best[nb], g_best[nb], nb, par))
    return None


def looping_human_ticks(world: np.ndarray, start: Cell, goal: Cell, astar=astar_path) -> np.ndarray:
    """(pos, next) per tick of `LoopingHuman(world, start, goal)` (`mapf_gym.py:52-70`): out along the A* path, back along
    the same cells, then from the top.  i16 [L, 4].  `astar(world, a, b)` plans the walk (`astar_path` or its results
    looked up from the device)."""
    out = astar(world, start, goal)
    if out is None:
        raise ValueError(f"no path from {start} to {goal}")
    if not out:
        raise ValueError("start == goal: the reference's Human indexes an empty path here")
    path = out + out[::-1][1:]
    p = np.asarray(path, dtype=np.int16)
    nxt = np.concatenate([p[1:], p[-1:]], axis=0)
    return np.concatenate([p, nxt], axis=1)


def fixed_path_human_ticks(world: np.ndarray, pose_sequence: Seq[Cell], ticks: int, astar=astar_path):
    """(pos, next) and `path[1:6]` per tick of `FixedPathHuman(world, humanPoseSequence)` (`mapf_gym.py:72-94` on top of
    `Human.nextStep/getNextPos`, `:25-50`) for `ticks` ticks: walk to each pose in turn; once the sequence is exhausted the
    walker jumps back to the start of its last path and repeats it (reference quirk, SURVEY Appendix B).
    `astar` as in `looping_human_ticks`.  Returns (i16 [ticks, 4], i16 [ticks, 5, 2])."""
    seq = [(int(p[0]), int(p[1])) for p in pose_sequence]
    pos, idx = seq[0], 1

    def plan(a, b):
        p = astar(world, a, b)
        if p is None:
            raise ValueError(f"no path from {a} to {b}")
        return p
    path = plan(pos, seq[idx])
    step = 0
    out = np.zeros((ticks, 4), dtype=np.int16)
    hp5 = np.full((ticks, 5, 2), -1, dtype=np.int16)
    for t in range(ticks):
        nxt = path[-1] if step >= len(path) - 1 else path[step + 1]
        out[t] = (pos[0], pos[1], nxt[0], nxt[1])
        seg = path[1:6]
        hp5[t, :len(seg)] = np.asarray(seg, dtype=np.int16).reshape(-1, 2)
        # nextStep (mapf_gym.py:25-31)
        if step >= len(path) - 1:
            idx += 1
            if idx < len(seq):
                path = plan(pos, seq[idx])
            step = 0
        else:
            step += 1
        pos = path[step]
    return out, hp5


# ---- fixture -> batched scenario ------------------------------------------------------------------------------------
def scenario_from_fixed_episode_infos(infos: Dict, *, human_movement_type: int = 0, max_steps: int = 256,
                                      num_channel: int = 6, use_da: bool = False, use_hp: bool = False,
                                      fov: int = 9, episodes: Optional[Seq[int]] = None, device=None) -> Scenario:
    """All (or the selected) fixed episodes as the worlds of one `Scenario` — what `evaluate.py:212-218` passes to
    `FixedMapfGym`, batched.  `human_movement_type` 0 = looping human between humanStart / humanGoal, 1 = the fixed pose
    sequence (`EvalParameters.HUMAN_MOVEMENT_TYPE`, `alg_parameters.py:10`, `evaluate.py:216-217`).
    Maps of different sizes are padded to the largest (`dims` keeps each world's true size); goal sequences of different
    lengths are padded by repeating the last goal, which is what `Sequence.getNext` does (`util.py:33-36`).
    With a CUDA `device`, every A* leg the host would plan is solved in one `mapf_astar4_paths` call (bit-exact with
    `astar_path`) and the same arrays are built from those paths; the result is byte-identical to `device=None` and the
    same errors are raised, for the same legs."""
    eps = list(range(int(infos["numEpisodes"]))) if episodes is None else list(episodes)
    maps = [np.asarray(infos["obstacleMap"][e]) for e in eps]
    W = len(eps)
    H, Wd = max(m.shape[0] for m in maps), max(m.shape[1] for m in maps)
    seqs = [[list(getattr(s, "items", s)) for s in infos["agentsSequence"][e]] for e in eps]
    N = len(seqs[0])
    assert all(len(s) == N for s in seqs), "every episode must have the same number of agents"
    Q = max(len(a) - 1 for s in seqs for a in s)
    obst = np.ones((W, H, Wd), dtype=np.uint8)
    dims = np.zeros((W, 2), dtype=np.int16)
    starts = np.zeros((W, N, 2), dtype=np.int16)
    queue = np.zeros((W, N, Q, 2), dtype=np.int16)
    for w, m in enumerate(maps):
        obst[w, :m.shape[0], :m.shape[1]] = (m != 0)
    traces, hp5s = [], []
    plan = ((lambda w, world, a, b: astar_path(world, a, b)) if device is None else
            _device_planner(infos, eps, maps, obst, human_movement_type, max_steps + 2, device))
    for w, (e, m) in enumerate(zip(eps, maps)):
        dims[w] = m.shape
        for i, items in enumerate(seqs[w]):
            if len(items) < 2:
                raise ValueError(f"episode {e} agent {i}: a start and at least one goal are needed")
            starts[w, i] = items[0]
            g = np.asarray(items[1:], dtype=np.int16).reshape(-1, 2)
            queue[w, i, :len(g)] = g
            queue[w, i, len(g):] = g[-1]
        world = np.where(m != 0, -1, 0)
        if human_movement_type == 0:
            tr = looping_human_ticks(world, infos["humanStart"][e], infos["humanGoal"][e],
                                     lambda world, a, b: plan(w, world, a, b))
            h5 = np.full((5, 2), -1, dtype=np.int16)
            k = min(5, tr.shape[0] - 1)
            h5[:k] = tr[1:1 + k, :2]
            hp5s.append(h5)
        else:
            tr, h5 = fixed_path_human_ticks(world, infos["humanSequence"][e], max_steps + 2,
                                           lambda world, a, b: plan(w, world, a, b))
            hp5s.append(h5)
        traces.append(tr)
    L = max(t.shape[0] for t in traces)
    htrace = np.zeros((W, L, 4), dtype=np.int16)
    hlen = np.zeros((W,), dtype=np.int32)
    for w, t in enumerate(traces):
        htrace[w, :t.shape[0]] = t
        htrace[w, t.shape[0]:] = t[-1]
        hlen[w] = t.shape[0]
    if human_movement_type == 0:
        hp5 = np.stack(hp5s).astype(np.int16)
    else:
        hp5 = np.full((W, L, 5, 2), -1, dtype=np.int16)
        for w, h in enumerate(hp5s):
            hp5[w, :h.shape[0]] = h
            hp5[w, h.shape[0]:] = h[-1]
    sc = Scenario(obst=obst, starts=starts, goal_queue=queue, htrace=htrace, hlen=hlen, hp5=hp5, dims=dims, fov=fov,
                  num_channel=num_channel, use_da=use_da, use_hp=use_hp,
                  meta=dict(kind="fixed_episode_infos", episodes=eps, human_movement_type=human_movement_type))
    sc.validate()
    return sc


def _device_planner(infos, eps, maps, obst, mtype, ticks, device):
    """plan(w, world, a, b) = astar_path(world, a, b) for world w of the batch, answered from one device call that solves
    every leg the host could plan: humanStart -> humanGoal (LoopingHuman), or the consecutive poses of humanSequence a
    FixedPathHuman can reach within `ticks` ticks (leg j starts no earlier than tick 2 (j - 1): every leg lasts at least
    two ticks, and an empty one raises).  A leg with a cell outside its world's own map is malformed input that the
    padded device map cannot represent; it is planned by astar_path itself, so it behaves as on the host."""
    import torch
    from .device_scenario import astar_paths_device
    reqs = {}
    for w, e in enumerate(eps):
        if mtype == 0:
            pairs = [(infos["humanStart"][e], infos["humanGoal"][e])]
        else:
            seq = infos["humanSequence"][e]
            pairs = list(zip(seq[:-1], seq[1:]))[:ticks // 2 + 1]
        for a, b in pairs:
            a, b = (int(a[0]), int(a[1])), (int(b[0]), int(b[1]))
            h, wd = maps[w].shape
            if all(0 <= r < h and 0 <= c < wd for r, c in (a, b)):
                reqs.setdefault((w, a, b), len(reqs))
    keys = list(reqs)
    sg = np.array([[a, b] for _, a, b in keys], dtype=np.int16).reshape(-1, 2, 2)
    dev = torch.device(device)
    widx = torch.tensor([w for w, _, _ in keys], dtype=torch.int64, device=dev)
    paths, lens = astar_paths_device(torch.from_numpy(obst).to(dev)[widx], torch.from_numpy(sg).to(dev))
    paths, lens = paths.cpu().numpy(), lens.cpu().numpy()

    def plan(w, world, a, b):
        i = reqs.get((w, (int(a[0]), int(a[1])), (int(b[0]), int(b[1]))))
        if i is None:
            return astar_path(world, a, b)
        k = int(lens[i])
        return None if k < 0 else [(int(r), int(c)) for r, c in paths[i, :k]]
    return plan


# ---- a plain frame renderer (own design; the reference's `_render` draws cv2 polygons, mapf_gym.py:639-646) --------------
def render_world(obst: np.ndarray, agents: np.ndarray, goals: np.ndarray, human: Cell, scale: int = 12) -> np.ndarray:
    """uint8 [H*scale, Wd*scale, 3] frame: shelves dark, agents as filled squares, their goals as hollow squares of the same
    hue, the human white.  For episode gifs / debugging; not pixel-compatible with the reference's renderer."""
    H, Wd = obst.shape
    img = np.full((H, Wd, 3), 235, dtype=np.uint8)
    img[obst != 0] = (40, 40, 48)
    big = np.repeat(np.repeat(img, scale, axis=0), scale, axis=1)
    n = max(1, len(agents))
    for i, ((ar, ac), (gr, gc)) in enumerate(zip(agents, goals)):
        hue = i / n
        k = int(hue * 6)
        f = hue * 6 - k
        rgb = [(1, f, 0), (1 - f, 1, 0), (0, 1, f), (0, 1 - f, 1), (f, 0, 1), (1, 0, 1 - f)][k % 6]
        col = np.array([int(255 * x) for x in rgb], dtype=np.uint8)
        big[gr * scale:(gr + 1) * scale, gc * scale:(gc + 1) * scale] = col
        big[gr * scale + 2:(gr + 1) * scale - 2, gc * scale + 2:(gc + 1) * scale - 2] = 235
        big[ar * scale + 1:(ar + 1) * scale - 1, ac * scale + 1:(ac + 1) * scale - 1] = col
    hr, hc = int(human[0]), int(human[1])
    big[hr * scale + 2:(hr + 1) * scale - 2, hc * scale + 2:(hc + 1) * scale - 2] = (255, 255, 255)
    big[hr * scale + 4:(hr + 1) * scale - 4, hc * scale + 4:(hc + 1) * scale - 4] = (0, 0, 0)
    return big
