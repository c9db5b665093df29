"""BatchedMapfGym — the reference env's method surface over W lockstep worlds on one B200.

Drop-in for ``MapfGym`` / ``FixedMapfGym`` (``mapf_gym.py:163-669``) as the rollout loop uses them
(``runner.py:30-100``): same method names, same argument order, same values; every array gains a leading world
dimension W and lives on the GPU as a torch tensor.  All arithmetic is done by the hand-written sm_100a kernels
behind the C ABI of ``include/mapf_b200.h``; torch is used for device memory and streams only.  There is no CPU
path: constructing the env without CUDA or without the built library raises.

Reference call                                     | batched call
---------------------------------------------------|---------------------------------------------------------
``env = FixedMapfGym(obst, seqs, hStart, hGoal)``  | ``env = BatchedMapfGym(scenario)``  (``scenario.py``)
``obs, vec = env.getAllObservations()``            | same -> f32 [W,N,C,F,F], f32 [W,N,4]
(bit-packed observations, not in the reference)    | ``getAllObservations(out=(bits, vec))`` with int32 ``env.obs_bits_shape``;
                                                   | ``unpack_observations(bits, C, F)`` -> f32 / bf16 [W,N,C,F,F]
``st = env.getActionStatus(a)``                    | same -> int8 [W,N]
``r, sg = env.calculateActionReward(a, st)``       | same -> f32 [W,N], int32 [W]
``c = env.calculateCostReward(a)``                 | same -> f32 [W,N]
``tv = env.getTrainValid(a)``                      | same -> f32 [W,N,5]
``g, cv = env.jointStep(a, st)``                   | same -> u8 [W,N], u8 [W,N]
(the five calls + ``rewards[g==1] += GOAL_REWARD``)| ``env.step(a)`` -> ``StepOut`` (one fused launch)
``agent.bfsMap``                                   | ``env.bfs_maps()`` -> int16 [W,N,H,Wd]
``env.allGoodActions``                             | same -> uint8 [W,N] 5-bit masks (bit a = action a is good)
``env._render()``                                  | ``env._render(world=0)`` -> uint8 frame of one world

ALIASING.  The reference returns a fresh array from every call.  Here ``getActionStatus`` / ``calculateActionReward`` /
``calculateCostReward`` / ``getTrainValid`` / ``jointStep`` / ``step`` return ENV-OWNED tensors that the next call
overwrites (no allocation on the step path).  A runner that keeps results across steps — ``runner.py:84,93-94`` appends
``trainVal`` / ``rewards`` / ``costRewards`` to lists — must either pass its own storage (``step(a, out=StepOut(...))``
with slices of a rollout buffer, as ``ppo/trainer.py`` does) or construct the env with ``fresh_outputs=True``, which makes
every getter return a clone (the reference's semantics, one extra device copy per call).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch

from . import _cabi
from .scenario import Scenario


@dataclass
class StepOut:
    status: torch.Tensor         # int8  [W,N]
    reward: torch.Tensor         # f32   [W,N]  (goal bonus included)
    cost: torch.Tensor           # f32   [W,N]
    train_valid: torch.Tensor    # f32   [W,N,5]
    goals_reached: torch.Tensor  # uint8 [W,N]
    violated: torch.Tensor       # uint8 [W,N]
    shadow_goals: torch.Tensor   # int32 [W]
    fixed_actions: torch.Tensor  # int8  [W,N]
    good_actions: Optional[torch.Tensor] = None   # uint8 [W,N] allGoodActions masks (mapf_evaluate only)
    packed: Optional[torch.Tensor] = None         # int16 [W,N] all per-agent results in 16 bits (MAPF_PACKED_*; step / step_observe)


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


class BatchedMapfGym:
    def __init__(self, scenario, device=None, seed: int = 1234, use_tape: bool = True,
                 world_offset: int = 0, goal_sampling: bool = False, fresh_outputs: bool = False):
        """goal_sampling: draw the next goal on device at arrival like ``MapfGym.getNextGoal`` (mapf_gym.py:189-190, 626;
        util.getFreeCell) instead of popping the scenario's goal queues (``FixedMapfGym``, :668-669).
        fresh_outputs: getters return clones instead of env-owned tensors (see ALIASING above)."""
        if not torch.cuda.is_available():
            raise _cabi.MapfError("BatchedMapfGym needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self._lib = _cabi.load_library()
        scenario.validate()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        sc = scenario
        self.W, self.H, self.Wd, self.N = sc.num_worlds, sc.height, sc.width, sc.num_agents
        self.F, self.C = sc.fov, sc.num_channel
        self.num_channel, self.use_da, self.use_hp = sc.num_channel, sc.use_da, sc.use_hp
        tape = sc.tape if (use_tape and sc.tape is not None) else None

        up = self._upload
        # scenario arrays are borrowed by the C side: keep them alive here
        self._sc = dict(obst=up(sc.obst), starts=up(sc.starts), goal_queue=up(sc.goal_queue), htrace=up(sc.htrace),
                        hlen=up(sc.hlen), hp5=up(sc.hp5), tape=up(tape),
                        tape_len=up(sc.tape_len) if tape is not None else None, dims=up(sc.dims))
        cfg = _cabi.MapfConfig(num_worlds=self.W, height=self.H, width=self.Wd, num_agents=self.N, fov=self.F,
                               num_channel=self.C, use_da=int(sc.use_da), use_hp=int(sc.use_hp),
                               queue_len=int(sc.goal_queue.shape[2]), trace_len=int(sc.htrace.shape[1]),
                               tape_stride=0 if tape is None else int(tape.shape[1]),
                               hp5_per_tick=int(sc.hp5 is not None and sc.hp5.ndim == 4), seed=seed,
                               device=self.device.index or 0, world_offset=int(world_offset),
                               goal_sampling=int(bool(goal_sampling)), reserved0=0)
        self.goal_sampling, self._fresh = bool(goal_sampling), bool(fresh_outputs)
        h = C.c_void_p()
        _cabi.check(self._lib.mapf_create(C.byref(cfg), C.byref(h)), "mapf_create")
        self._h = h
        W, N, dev = self.W, self.N, self.device
        self._out = StepOut(status=torch.empty((W, N), dtype=torch.int8, device=dev),
                            reward=torch.empty((W, N), dtype=torch.float32, device=dev),
                            cost=torch.empty((W, N), dtype=torch.float32, device=dev),
                            train_valid=torch.empty((W, N, 5), dtype=torch.float32, device=dev),
                            goals_reached=torch.empty((W, N), dtype=torch.uint8, device=dev),
                            violated=torch.empty((W, N), dtype=torch.uint8, device=dev),
                            shadow_goals=torch.empty((W,), dtype=torch.int32, device=dev),
                            fixed_actions=torch.empty((W, N), dtype=torch.int8, device=dev))
        self._obs = None
        self._vec = None
        self._eval_key = None
        self._bfs = None
        self._good = None
        self._zero_actions = None
        self._host_layouts = {}
        self.reset()

    # ------------------------------------------------------------------------------------------------------
    def _upload(self, a):      # numpy arrays are uploaded; tensors of a DeviceScenario are used in place
        if a is None:
            return None
        if isinstance(a, torch.Tensor):
            return a.to(self.device).contiguous()
        return torch.from_numpy(np.ascontiguousarray(a)).to(self.device)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.mapf_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self, scenario=None):
        """``populateMap`` (mapf_gym.py:175-184): back to the scenario's starts / first goals / tick 0.  With ``scenario``
        (same shapes as the one the env was created with) the worlds themselves are replaced — the reference builds a
        fresh ``MapfGym()`` for every rollout (runner.py:30); with a ``DeviceScenario`` this involves no host copy."""
        if scenario is not None:
            scenario.validate()
            sc = scenario
            same = ((sc.num_worlds, sc.height, sc.width, sc.num_agents, sc.fov, sc.num_channel) ==
                    (self.W, self.H, self.Wd, self.N, self.F, self.C)
                    and int(sc.goal_queue.shape[2]) == int(self._sc["goal_queue"].shape[2])
                    and int(sc.htrace.shape[1]) == int(self._sc["htrace"].shape[1])
                    and bool(sc.use_da) == bool(self.use_da) and bool(sc.use_hp) == bool(self.use_hp)
                    and (sc.dims is None) == (self._sc["dims"] is None) and (sc.hp5 is None) == (self._sc["hp5"] is None)
                    and self._sc["tape"] is None and getattr(sc, "tape", None) is None)
            if not same:
                raise ValueError("reset(scenario): the new scenario must have the shapes / flags the env was created with")
            up = self._upload
            self._sc = dict(obst=up(sc.obst), starts=up(sc.starts), goal_queue=up(sc.goal_queue), htrace=up(sc.htrace),
                            hlen=up(sc.hlen), hp5=up(sc.hp5), tape=None, tape_len=None, dims=up(sc.dims))
        s = self._sc
        sc = _cabi.MapfScenario(**{k: (None if v is None else v.data_ptr()) for k, v in s.items()})
        _cabi.check(self._lib.mapf_reset(self._h, C.byref(sc), self._stream()), "mapf_reset")
        self._eval_key = None

    def _actions(self, actions) -> torch.Tensor:
        a = actions if isinstance(actions, torch.Tensor) else torch.as_tensor(np.asarray(actions))
        if a.dtype != torch.int8:
            a = a.to(torch.int8)
        a = a.to(self.device, non_blocking=True).contiguous()
        if tuple(a.shape) != (self.W, self.N):
            raise ValueError(f"actions must have shape {(self.W, self.N)}, got {tuple(a.shape)}")  # mapf_gym.py:437
        return a

    def _step_out(self, o: StepOut, **skip) -> _cabi.MapfStepOut:
        return _cabi.MapfStepOut(status=o.status.data_ptr(), reward=o.reward.data_ptr(), cost=o.cost.data_ptr(),
                                 train_valid=o.train_valid.data_ptr(), goals_reached=o.goals_reached.data_ptr(),
                                 violated=o.violated.data_ptr(), shadow_goals=o.shadow_goals.data_ptr(),
                                 fixed_actions=o.fixed_actions.data_ptr(),
                                 good_actions=None if o.good_actions is None else o.good_actions.data_ptr(),
                                 packed=None if o.packed is None else o.packed.data_ptr())

    def _ret(self, t):
        return t.clone() if self._fresh else t

    # ---- the reference's five step calls (runner.py:64-87) -----------------------------------------------------
    def _evaluate(self, actions):
        a = self._actions(actions)
        key = (a.data_ptr(), a._version, id(actions))
        if self._eval_key != key:
            so = self._step_out(self._out)
            _cabi.check(self._lib.mapf_evaluate(self._h, _ptr(a), C.byref(so), self._stream()), "mapf_evaluate")
            self._eval_key = key
            self._eval_actions = a
        return self._out

    def getActionStatus(self, actions):
        self._eval_key = None
        return self._ret(self._evaluate(actions).status)

    def calculateActionReward(self, actions, actionStatus=None):
        o = self._evaluate(actions)
        return self._ret(o.reward), self._ret(o.shadow_goals)

    def calculateCostReward(self, actions):
        return self._ret(self._evaluate(actions).cost)

    def getTrainValid(self, actions):
        return self._ret(self._evaluate(actions).train_valid)

    @property
    def allGoodActions(self):
        """``MapfGym.allGoodActions`` (mapf_gym.py:169, 635: ``getUnconditionallyGoodActions(returnIsNeeded=True)``) of the
        CURRENT state: uint8 [W,N], bit a set iff action a is unconditionally good for that agent (the reference holds a
        list of sorted action arrays per agent; ``good_actions_lists`` converts).  Recomputed on access (the masks are a
        pure function of the state and are never stored)."""
        if self._good is None:
            self._good = torch.empty((self.W, self.N), dtype=torch.uint8, device=self.device)
            self._zero_actions = torch.zeros((self.W, self.N), dtype=torch.int8, device=self.device)
        so = _cabi.MapfStepOut(good_actions=self._good.data_ptr())
        _cabi.check(self._lib.mapf_evaluate(self._h, _ptr(self._zero_actions), C.byref(so), self._stream()), "mapf_evaluate")
        return self._ret(self._good)

    def good_actions_lists(self, world: int = 0):
        """The reference's representation for one world: a list of N sorted int arrays."""
        m = self.allGoodActions[world].cpu().numpy()
        return [np.flatnonzero([(int(x) >> a) & 1 for a in range(5)]) for x in m]

    def _render(self, world: int = 0, scale: int = 12):
        """``MapfGym._render`` (mapf_gym.py:639-646) for one world: an RGB uint8 frame (own renderer, ``episode_io.render_world``;
        not pixel-compatible with the reference's cv2 drawing)."""
        from .episode_io import render_world
        st = self.state()
        obst = self._sc["obst"][world].cpu().numpy()
        pos, goal = st["pos"][world].cpu().numpy(), st["goal"][world].cpu().numpy()
        human = self.human()[0][world].cpu().numpy()
        return render_world(obst, pos, goal, (int(human[0]), int(human[1])), scale=scale)

    def human(self):
        """``(human.getPos(), human.getNextPos(), tick)`` of every world (mapf_gym.py:25-50): int16 [W,2], int16 [W,2],
        int32 [W]."""
        pn = torch.empty((self.W, 4), dtype=torch.int16, device=self.device)
        tick = torch.empty((self.W,), dtype=torch.int32, device=self.device)
        _cabi.check(self._lib.mapf_get_human(self._h, _ptr(pn), _ptr(tick), self._stream()), "mapf_get_human")
        return pn[:, :2], pn[:, 2:], tick

    def jointStep(self, actions, actionStatus):
        a = self._actions(actions)
        st = actionStatus.to(device=self.device, dtype=torch.int8).contiguous()
        o = self._out
        _cabi.check(self._lib.mapf_joint_step(self._h, _ptr(a), _ptr(st), _ptr(o.goals_reached), _ptr(o.violated),
                                              _ptr(o.fixed_actions), self._stream()), "mapf_joint_step")
        self._eval_key = None
        return self._ret(o.goals_reached), self._ret(o.violated)

    # ---- fused step -------------------------------------------------------------------------------------------
    def step(self, actions, out: Optional[StepOut] = None) -> StepOut:
        """All five calls in one launch plus ``rewards[goalsReached==1] += GOAL_REWARD`` (runner.py:89-91).
        ``out`` lets a rollout buffer receive the results in place (e.g. slices ``buf.reward[t]``)."""
        a = self._actions(actions)
        o = self._out if out is None else out
        so = self._step_out(o)
        _cabi.check(self._lib.mapf_step(self._h, _ptr(a), C.byref(so), self._stream()), "mapf_step")
        self._eval_key = None
        return o

    def step_observe(self, actions, out: Optional[StepOut] = None, obs_out=None):
        """One env step of the rollout loop in ONE launch: ``step(actions)`` then ``getAllObservations()`` of the new
        state (runner.py:64-100), fused per world.  Returns ``(StepOut, obs, vec)``; bit-identical to the two calls."""
        a = self._actions(actions)
        o = self._out if out is None else out
        obs, vec = self._obs_buffers(obs_out)
        so = self._step_out(o)
        fn = {torch.bfloat16: self._lib.mapf_step_observe_bf16, torch.int32: self._lib.mapf_step_observe_bits}.get(
            obs.dtype, self._lib.mapf_step_observe)
        _cabi.check(fn(self._h, _ptr(a), C.byref(so), _ptr(obs), _ptr(vec), self._stream()), "mapf_step_observe")
        self._eval_key = None
        return o, obs, vec

    # ---- observations -----------------------------------------------------------------------------------------
    def _obs_buffers(self, out):
        if out is None:
            if self._obs is None:
                self._obs = torch.empty((self.W, self.N, self.C, self.F, self.F), dtype=torch.float32, device=self.device)
                self._vec = torch.empty((self.W, self.N, 4), dtype=torch.float32, device=self.device)
            return self._obs, self._vec
        obs, vec = out
        assert obs.is_contiguous() and vec.is_contiguous() and vec.dtype == torch.float32
        assert obs.dtype in (torch.float32, torch.bfloat16, torch.int32), \
            "observations are f32 (reference layout) or, optionally, bf16 or bit-packed int32 (obs_bits_shape)"
        if obs.dtype == torch.int32:
            assert tuple(obs.shape) == self.obs_bits_shape, f"bit-packed observations need shape {self.obs_bits_shape}"
        else:
            assert obs.numel() == self.W * self.N * self.C * self.F * self.F
        assert vec.numel() == self.W * self.N * 4
        return obs, vec

    @property
    def obs_bits_shape(self):
        """Shape of the bit-packed observations (int32 [W, N, AW], AW = ``MAPF_OBS_BITS_WORDS(C, F)``): bit k of agent
        (w, i) is ``obs[w, i].flatten()[k]``, in word k // 32 at bit k % 32; ``unpack_observations`` expands them."""
        return (self.W, self.N, _cabi.obs_bits_words(self.C, self.F))

    def getAllObservations(self, out=None):
        """``getAllObservations`` (mapf_gym.py:327-336).  ``out=(obs, vec)`` writes straight into the policy's input
        tensors; otherwise env-owned tensors are (re)used.  ``obs`` selects the format by dtype: f32, bf16, or int32 of
        ``obs_bits_shape`` (one bit per cell)."""
        obs, vec = self._obs_buffers(out)
        fn = {torch.bfloat16: self._lib.mapf_observe_bf16, torch.int32: self._lib.mapf_observe_bits}.get(
            obs.dtype, self._lib.mapf_observe)
        _cabi.check(fn(self._h, _ptr(obs), _ptr(vec), self._stream()), "mapf_observe")
        return obs, vec

    # ---- BFS distance-to-goal maps (agent.bfsMap, mapf_gym.py:211-244) -------------------------------------------
    def bfs_maps(self, agent_ids: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None):
        """All maps [W,N,H,Wd] int16 for the current goals, or the maps of the given flat agent ids (w*N+i)."""
        if agent_ids is None:
            n = self.W * self.N
            shape = (self.W, self.N, self.H, self.Wd)
            lst = None
        else:
            lst = agent_ids.to(device=self.device, dtype=torch.int32).contiguous()
            n = int(lst.numel())
            shape = (n, self.H, self.Wd)
        if out is None:
            out = torch.empty(shape, dtype=torch.int16, device=self.device)
        if n == 0:                         # an empty list is not the C ABI's NULL (= all agents)
            return out
        _cabi.check(self._lib.mapf_bfs(self._h, _ptr(lst), n, _ptr(out), self._stream()), "mapf_bfs")
        return out

    def refresh_bfs(self, bfs_maps: torch.Tensor, goals_reached: Optional[torch.Tensor] = None):
        """In-place refresh of the maps of agents that just received a new goal (mapf_gym.py:627); no host sync."""
        g = self._out.goals_reached if goals_reached is None else goals_reached
        _cabi.check(self._lib.mapf_bfs_refresh(self._h, _ptr(g), _ptr(bfs_maps), self._stream()), "mapf_bfs_refresh")
        return bfs_maps

    # ---- state / counters ---------------------------------------------------------------------------------------
    def state(self):
        W, N, dev = self.W, self.N, self.device
        pos = torch.empty((W, N, 2), dtype=torch.int16, device=dev)
        goal = torch.empty((W, N, 2), dtype=torch.int16, device=dev)
        rep = torch.empty((W, N), dtype=torch.int8, device=dev)
        err = torch.empty((W,), dtype=torch.int32, device=dev)
        _cabi.check(self._lib.mapf_get_state(self._h, _ptr(pos), _ptr(goal), _ptr(rep), _ptr(err), self._stream()),
                    "mapf_get_state")
        return dict(pos=pos, goal=goal, rep=rep, err=err)

    def save_state(self) -> torch.Tensor:
        """Checkpoint of the env's mutable state as an opaque uint8 device tensor (``load_state`` restores it)."""
        n = int(self._lib.mapf_state_bytes(self._h))
        if n < 0:
            _cabi.check(n, "mapf_state_bytes")
        blob = torch.empty((n,), dtype=torch.uint8, device=self.device)
        _cabi.check(self._lib.mapf_save_state(self._h, _ptr(blob), self._stream()), "mapf_save_state")
        return blob

    def load_state(self, blob: torch.Tensor) -> None:
        assert blob.dtype == torch.uint8 and blob.is_contiguous() and blob.numel() == int(self._lib.mapf_state_bytes(self._h))
        _cabi.check(self._lib.mapf_load_state(self._h, _ptr(blob.to(self.device)), self._stream()), "mapf_load_state")
        self._eval_key = None

    def counters(self):
        """OneEpPerformance counters per world (util.py:56-65): int64 [W,6] =
        totalGoals, shadowGoals, staticCollide, humanCollide, agentCollide, constraintViolations."""
        c = torch.empty((self.W, 6), dtype=torch.int64, device=self.device)
        _cabi.check(self._lib.mapf_get_counters(self._h, _ptr(c), self._stream()), "mapf_get_counters")
        return c

    # ---- host-buffer step (what a CPU-side runner calls) ------------------------------------------------------------
    def make_host_buffers(self, with_obs: bool = False, with_train_valid: bool = False, action_slots: int = 1):
        """Pinned host buffers for ``step_observe_host``: the per-agent results the runner's bookkeeping reads on the
        host (runner.py:66-99).  trainValid and the observations are training data consumed on the GPU; they are
        mirrored to the host only on request.

        Everything is carved out of ONE pinned allocation.  Measured on the B200 boxes (`tools/h2d_probe.py`): of eight
        separately pinned 2 MB buffers the sixth to eighth take 73-158 us per host-to-device copy instead of 42 us
        (50 GB/s); slices of a single pinned slab all take 42 us.  ``hb["action_ring"]`` is int8 [action_slots, W, N]
        (a runner that double-buffers its joint actions writes there); ``hb["actions"]`` is slot 0."""
        W, N = self.W, self.N
        fields = [("action_ring", (max(1, action_slots), W, N), torch.int8),
                  ("status", (W, N), torch.int8), ("reward", (W, N), torch.float32), ("cost", (W, N), torch.float32),
                  ("goals_reached", (W, N), torch.uint8), ("violated", (W, N), torch.uint8),
                  ("shadow_goals", (W,), torch.int32)]
        if with_train_valid:
            fields.append(("train_valid", (W, N, 5), torch.float32))
        if with_obs:
            fields.append(("obs", (W, N, self.C, self.F, self.F), torch.float32))
            fields.append(("vec", (W, N, 4), torch.float32))
        offs, total = [], 0
        for _, shape, dt in fields:
            n = torch.empty((), dtype=dt).element_size()
            for d in shape:
                n *= d
            offs.append((total, n))
            total += (n + 255) // 256 * 256
        slab = torch.empty((total,), dtype=torch.uint8, pin_memory=True)
        hb = {}
        for (name, shape, dt), (o, n) in zip(fields, offs):
            hb[name] = slab[o:o + n].view(dt).view(shape)
        hb["action_ring"].zero_()
        hb["actions"] = hb["action_ring"][0]
        hb["_slab"] = slab
        return hb

    def step_observe_host(self, hb: dict, obs_dev: torch.Tensor, vec_dev: torch.Tensor,
                          train_valid_dev: Optional[torch.Tensor] = None, actions: Optional[torch.Tensor] = None):
        """actions (host) -> H2D -> step -> observe -> results D2H, synchronised.  Returns bytes moved (h2d, d2h).
        `actions`: an int8 [W,N] HOST tensor (ideally pinned) to read the joint action from; default ``hb["actions"]``."""
        act = hb["actions"] if actions is None else actions
        assert not act.is_cuda and act.dtype == torch.int8 and act.is_contiguous() and act.numel() == self.W * self.N
        key = (id(hb), hb["status"].data_ptr(), hb["reward"].data_ptr(), len(hb))
        cached = getattr(self, "_host_call_cache", None)
        if cached is None or cached[0] != key:          # the struct and the byte counts only depend on the buffer set
            tvh = hb.get("train_valid")
            so = _cabi.MapfStepOutHost(status=hb["status"].data_ptr(), reward=hb["reward"].data_ptr(),
                                       cost=hb["cost"].data_ptr(), train_valid=None if tvh is None else tvh.data_ptr(),
                                       goals_reached=hb["goals_reached"].data_ptr(), violated=hb["violated"].data_ptr(),
                                       shadow_goals=hb["shadow_goals"].data_ptr(), fixed_actions=None, good_actions=None)
            d2h = sum(hb[k].numel() * hb[k].element_size() for k in hb if k not in ("actions", "action_ring", "_slab"))
            cached = (key, so, d2h, _ptr(hb.get("obs")), _ptr(hb.get("vec")))
            self._host_call_cache = cached
        _, so, d2h, oh, vh = cached
        tvd = self._out.train_valid if train_valid_dev is None else train_valid_dev
        _cabi.check(self._lib.mapf_step_observe_host(self._h, _ptr(act), C.byref(so), _ptr(obs_dev),
                                                     _ptr(vec_dev), _ptr(tvd), oh, vh, self._stream()),
                    "mapf_step_observe_host")
        h2d = act.numel()
        return h2d, d2h


    # ---- split-phase host call: step t's results travel to the host while step t+1 computes -------------------------
    def host_layout(self, with_train_valid: bool = False, compact: bool = False, obs=None) -> "_cabi.MapfHostLayout":
        """``mapf_host_layout``.  obs (None, torch.float32, torch.bfloat16 or "bits"): the slot also carries the step's
        observations in that format and vec (MAPF_HOST_OBS), after ``host_layout(with_train_valid, compact).slot_bytes``."""
        flags = ((_cabi.HOST_TRAIN_VALID if with_train_valid else 0) | (_cabi.HOST_COMPACT if compact else 0)
                 | _host_obs_flags(obs))
        return self._host_layout(flags)

    def _host_layout(self, flags: int) -> "_cabi.MapfHostLayout":
        if flags not in self._host_layouts:
            L = _cabi.MapfHostLayout()
            _cabi.check(self._lib.mapf_host_layout(self._h, flags, C.byref(L)), "mapf_host_layout")
            self._host_layouts[flags] = L
        return self._host_layouts[flags]

    def make_host_ring(self, slots: int = 2, action_slots: int = 2, with_train_valid: bool = False, compact: bool = False,
                       numa_bind: bool = True, obs=None):
        """ONE pinned slab holding `slots` result slots (the layout ``mapf_host_layout`` reports: every per-agent result of
        a step is contiguous, so a step's results come back with one copy) and an int8 [action_slots, W, N] action ring.
        compact=True: the 2-byte-per-agent wire format (``packed`` u16 [W,N] + ``shadow_goals``; ``decode_slot`` expands it
        on the host, bit for bit) instead of the 12-byte-per-agent f32 slab — what keeps eight GPUs of one box off the
        host's PCIe / memory ceiling.  Returns ``{"slots": [dict of views per slot], "action_ring": ..., ...}``.
        numa_bind: allocate while the calling thread is bound to the CPUs next to this GPU (first touch places the pages).
        obs (None, torch.float32, torch.bfloat16 or "bits"): every slot also receives the step's observations in that format
        and vec (MAPF_HOST_OBS), as host views ``obs`` (f32 / bf16 [W,N,C,F,F] or int32 ``obs_bits_shape``) and ``vec``
        (f32 [W,N,4]); ``step_observe_host_begin`` then needs an ``obs_dev`` of that format.  ``unpack_observations``
        expands a bit-packed host ``obs``."""
        L = self.host_layout(with_train_valid, compact, obs)
        obs_flags = _host_obs_flags(obs)
        W, N = self.W, self.N
        sb = int(L.slot_bytes)
        act_bytes = (max(1, action_slots) * W * N + 255) // 256 * 256
        restore = _bind_near_gpu(self.device) if numa_bind else None
        try:
            slab = torch.empty((slots * sb + act_bytes,), dtype=torch.uint8, pin_memory=True)
            slab.zero_()
        finally:
            if restore is not None:
                restore()
        views = []
        for k in range(slots):
            b = slab[k * sb:(k + 1) * sb]

            def f(off, n, dt, shape):
                return b[off:off + n].view(dt).view(shape)
            d = dict(shadow_goals=f(L.off_shadow_goals, W * 4, torch.int32, (W,)), _raw=b)
            if compact:
                d["packed"] = f(L.off_packed, W * N * 2, torch.int16, (W, N))
            else:
                d.update(reward=f(L.off_reward, W * N * 4, torch.float32, (W, N)), cost=f(L.off_cost, W * N * 4, torch.float32, (W, N)),
                         status=f(L.off_status, W * N, torch.int8, (W, N)),
                         goals_reached=f(L.off_goals_reached, W * N, torch.uint8, (W, N)),
                         violated=f(L.off_violated, W * N, torch.uint8, (W, N)),
                         fixed_actions=f(L.off_fixed_actions, W * N, torch.int8, (W, N)))
            if with_train_valid:
                d["train_valid"] = f(L.off_train_valid, W * N * 20, torch.float32, (W, N, 5))
            if obs_flags:
                dt, shape = self._obs_format(obs_flags)
                off_obs = int(self.host_layout(with_train_valid, compact).slot_bytes)
                n_obs = int(np.prod(shape)) * torch.empty((), dtype=dt).element_size()
                d["obs"] = f(off_obs, n_obs, dt, shape)
                d["vec"] = f(off_obs + (n_obs + 255) // 256 * 256, W * N * 16, torch.float32, (W, N, 4))
            views.append(d)
        ring = slab[slots * sb:slots * sb + max(1, action_slots) * W * N].view(torch.int8).view(max(1, action_slots), W, N)
        return {"slots": views, "action_ring": ring, "_slab": slab, "with_train_valid": bool(with_train_valid),
                "compact": bool(compact), "slot_bytes": sb, "obs": obs,
                "flags": (_cabi.HOST_TRAIN_VALID if with_train_valid else 0) | (_cabi.HOST_COMPACT if compact else 0)
                | obs_flags}

    def _obs_format(self, flags: int):
        """(dtype, shape) of observations in the format the MAPF_HOST_OBS_* bits of `flags` select."""
        if flags & _cabi.HOST_OBS_BITS:
            return torch.int32, self.obs_bits_shape
        dt = torch.bfloat16 if flags & _cabi.HOST_OBS_BF16 else torch.float32
        return dt, (self.W, self.N, self.C, self.F, self.F)

    def step_observe_host_begin(self, actions: torch.Tensor, slot: dict, obs_dev: torch.Tensor, vec_dev: torch.Tensor,
                                train_valid_dev: Optional[torch.Tensor] = None, with_train_valid: bool = False):
        """Queue one env step for a HOST runner and return immediately: `actions` (int8 [W,N] host tensor, ideally a slice of
        the ring's pinned slab) -> device, ONE fused step+observe launch into obs_dev / vec_dev, all per-agent results ->
        `slot` (one of ``make_host_ring()["slots"]``; its format — full or compact — is the ring's) with ONE device-to-host
        copy.  ``obs_dev`` selects the observation format by dtype, as in ``step_observe``: f32, bf16, or int32 of
        ``obs_bits_shape``.  A ring made with ``obs=`` also receives obs_dev / vec_dev in the slot's ``obs`` / ``vec``; obs_dev
        must then be in the ring's format.  ``host_wait(age)`` makes a slot readable.  Returns (h2d_bytes, d2h_bytes)."""
        assert not actions.is_cuda and actions.dtype == torch.int8 and actions.is_contiguous() and actions.numel() == self.W * self.N
        obs_dev, vec_dev = self._obs_buffers((obs_dev, vec_dev))
        compact = "packed" in slot
        flags = ((_cabi.HOST_TRAIN_VALID if with_train_valid else 0) | (_cabi.HOST_COMPACT if compact else 0)
                 | _OBS_FORMAT_FLAG[obs_dev.dtype])
        # the trainValid block (and after it the observation block) is placed by the flags: they must be the ring's
        if with_train_valid and "train_valid" not in slot:
            raise _cabi.MapfError("step_observe_host_begin: with_train_valid=True needs a ring made with with_train_valid=True")
        if "obs" in slot and not with_train_valid and "train_valid" in slot:
            raise _cabi.MapfError("step_observe_host_begin: this ring's slots hold train_valid before the observations; "
                                  "pass with_train_valid=True")
        if "obs" in slot:
            if slot["obs"].dtype != obs_dev.dtype:
                raise _cabi.MapfError(f"step_observe_host_begin: the ring holds {slot['obs'].dtype} observations, "
                                      f"obs_dev is {obs_dev.dtype}")
            flags |= _cabi.HOST_OBS
        tvd = train_valid_dev
        if with_train_valid and tvd is None:
            tvd = self._out.train_valid
        _cabi.check(self._lib.mapf_step_observe_host_begin(self._h, _ptr(actions), C.c_void_p(slot["_raw"].data_ptr()), flags,
                                                           _ptr(obs_dev), _ptr(vec_dev), _ptr(tvd), self._stream()),
                    "mapf_step_observe_host_begin")
        self._eval_key = None
        return actions.numel(), int(self._host_layout(flags).slot_bytes)

    def host_wait(self, age: int = 0):
        """Block until the results of the most recent ``step_observe_host_begin`` (age 0) or the one before (age 1) are in
        their host slot."""
        _cabi.check(self._lib.mapf_step_observe_host_wait(self._h, int(age)), "mapf_step_observe_host_wait")


_OBS_FORMAT_FLAG = {torch.float32: 0, torch.bfloat16: _cabi.HOST_OBS_BF16, torch.int32: _cabi.HOST_OBS_BITS}


def _host_obs_flags(obs) -> int:
    """MAPF_HOST_OBS and the format flag for a ring's `obs` argument (None: no observations in the slot)."""
    if obs is None:
        return 0
    if isinstance(obs, str) and obs == "bits":
        return _cabi.HOST_OBS | _cabi.HOST_OBS_BITS
    if obs in (torch.float32, torch.bfloat16):
        return _cabi.HOST_OBS | _OBS_FORMAT_FLAG[obs]
    raise ValueError(f"obs must be None, torch.float32, torch.bfloat16 or 'bits', got {obs!r}")


def decode_results(packed: torch.Tensor, out: Optional[dict] = None) -> dict:
    """``mapf_decode_results_host``: expand a HOST int16 / uint16 tensor of packed per-agent results (a compact slot's
    ``packed``) into the reference's arrays — status i8, reward f32, cost f32, goals_reached u8, violated u8,
    fixed_actions i8 — bit-identical to what the full format carries.  `out` (same keys) is reused when given."""
    lib = _cabi.load_library()
    assert not packed.is_cuda and packed.is_contiguous() and packed.element_size() == 2
    shp = tuple(packed.shape)
    if out is None:
        out = dict(status=torch.empty(shp, dtype=torch.int8), reward=torch.empty(shp, dtype=torch.float32),
                   cost=torch.empty(shp, dtype=torch.float32), goals_reached=torch.empty(shp, dtype=torch.uint8),
                   violated=torch.empty(shp, dtype=torch.uint8), fixed_actions=torch.empty(shp, dtype=torch.int8))
    so = _cabi.MapfStepOutHost(**{k: out[k].data_ptr() for k in ("status", "reward", "cost", "goals_reached", "violated",
                                                                  "fixed_actions") if k in out})
    _cabi.check(lib.mapf_decode_results_host(C.c_void_p(packed.data_ptr()), packed.numel(), C.byref(so)), "mapf_decode_results_host")
    return out


def _bind_near_gpu(device):
    """Bind the calling thread to the CPUs NVML reports as closest to `device`; returns a callable that restores the
    previous affinity, or None when NVML / the affinity call is unavailable."""
    import os
    try:
        import pynvml
        pynvml.nvmlInit()
        idx = device.index or 0
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ent = vis.split(",")[idx].strip()
            idx = int(ent) if ent.isdigit() else idx
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * k + b for k, wd in enumerate(words) for b in range(64) if (int(wd) >> b) & 1}
        prev = os.sched_getaffinity(0)
        cpus &= prev
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return lambda: os.sched_setaffinity(0, prev)
    except Exception:
        return None


def checksum_rows(t: torch.Tensor) -> torch.Tensor:
    """64-bit position-keyed checksum of every row t[r] of a contiguous CUDA tensor of 4-byte-multiple rows
    (``mapf_checksum_rows``): int64 [rows] holding the uint64 bit patterns."""
    lib = _cabi.load_library()
    assert t.is_cuda and t.is_contiguous()
    rows = int(t.shape[0])
    row_bytes = (t.numel() // max(rows, 1)) * t.element_size() if rows else 0
    out = torch.empty((rows,), dtype=torch.int64, device=t.device)
    stream = C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)
    with torch.cuda.device(t.device):
        _cabi.check(lib.mapf_checksum_rows(_ptr(t), rows, row_bytes, _ptr(out), stream), "mapf_checksum_rows")
    return out


def _stream_ptr(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def unpack_observations(bits: torch.Tensor, C: int, F: int, rows: Optional[torch.Tensor] = None,
                        dtype=torch.float32, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Expand bit-packed observations (``mapf_unpack_obs``) into the network's 0/1 values in ONE kernel pass.

    bits: int32 [..., N, AW] (AW = ``MAPF_OBS_BITS_WORDS(C, F)``); its leading dimensions are the source rows.  On the GPU
    the unpack kernel runs; a CPU tensor (a bit-packed host slot of ``make_host_ring(obs="bits")``) is expanded on the host
    by ``mapf_unpack_obs_host``, with the same results.
    rows: optional int64 index into the source rows (a minibatch gather): the result is [len(rows), N, C, F, F], and an
    index outside [0, rows) gives an all-zero row.  Without it the result is bits.shape[:-1] + (C, F, F).
    dtype: torch.float32 or torch.bfloat16.  out: a contiguous tensor of that shape and dtype to write into."""
    lib = _cabi.load_library()
    assert bits.dtype == torch.int32 and bits.is_contiguous() and bits.dim() >= 2
    assert dtype in (torch.float32, torch.bfloat16), "observations expand to f32 or bf16"
    N, AW = int(bits.shape[-2]), int(bits.shape[-1])
    assert AW == _cabi.obs_bits_words(C, F), f"last dimension {AW} is not MAPF_OBS_BITS_WORDS({C}, {F})"
    src_rows = bits.numel() // max(N * AW, 1)
    if rows is None:
        n_rows, shape, idx = src_rows, tuple(bits.shape[:-1]) + (C, F, F), None
    else:
        idx = rows.to(device=bits.device, dtype=torch.int64).contiguous()
        n_rows, shape = int(idx.numel()), (int(idx.numel()), N, C, F, F)
    if out is None:
        out = torch.empty(shape, dtype=dtype, device=bits.device)
    assert out.is_contiguous() and out.dtype == dtype and tuple(out.shape) == shape and out.device == bits.device
    if n_rows == 0:
        return out
    if not bits.is_cuda:
        _cabi.check(lib.mapf_unpack_obs_host(_ptr(bits), src_rows, N, int(C), int(F), _ptr(idx), n_rows,
                                             int(dtype == torch.bfloat16), _ptr(out)), "mapf_unpack_obs_host")
        return out
    stream = _stream_ptr(bits.device)            # (`C` is the channel count here, not the ctypes module)
    with torch.cuda.device(bits.device):
        _cabi.check(lib.mapf_unpack_obs(_ptr(bits), src_rows, N, int(C), int(F), _ptr(idx), n_rows,
                                        int(dtype == torch.bfloat16), _ptr(out), stream), "mapf_unpack_obs")
    return out


def gae(rewards: torch.Tensor, values: torch.Tensor, last_values: torch.Tensor, gamma: float = 0.95,
        lam: float = 0.95, nonterminal: Optional[torch.Tensor] = None, return_advantages: bool = False):
    """GAE + returns (runner.py:120-149) on device.  rewards, values: f32 [T, ...]; last_values: f32 [...]."""
    lib = _cabi.load_library()
    assert rewards.is_cuda and rewards.dtype == torch.float32 and values.dtype == torch.float32
    r, v, lv = rewards.contiguous(), values.contiguous(), last_values.contiguous().to(torch.float32)
    T = int(r.shape[0])
    cols = 1
    for d in r.shape[1:]:
        cols *= int(d)
    assert v.shape == r.shape and lv.numel() == cols
    ret = torch.empty_like(r)
    adv = torch.empty_like(r) if return_advantages else None
    if r.numel() == 0:                      # empty rollout: nothing to scan
        return (ret, adv) if return_advantages else ret
    nt = None if nonterminal is None else nonterminal.to(torch.uint8).contiguous()
    stream = C.c_void_p(torch.cuda.current_stream(r.device).cuda_stream)
    with torch.cuda.device(r.device):
        _cabi.check(lib.mapf_gae(_ptr(r), _ptr(v), _ptr(lv), _ptr(nt), float(gamma), float(lam), T, cols, _ptr(ret),
                                 _ptr(adv), stream), "mapf_gae")
    return (ret, adv) if return_advantages else ret


def gae2(rewards, values, last_values, cost_rewards, cost_values, last_cost_values, gamma: float = 0.95, lam: float = 0.95,
         nonterminal: Optional[torch.Tensor] = None):
    """Both GAE streams of a rollout in one launch (``mapf_gae2``; runner.py:146-149): returns (returns, cost_returns),
    bit-identical to two ``gae`` calls."""
    lib = _cabi.load_library()
    ts = [x.contiguous().to(torch.float32) for x in (rewards, values, last_values, cost_rewards, cost_values, last_cost_values)]
    r, v, lv, cr, cv, lcv = ts
    assert r.is_cuda and v.shape == r.shape and cr.shape == r.shape and cv.shape == r.shape
    T = int(r.shape[0])
    cols = r.numel() // max(T, 1) if T else 0
    assert lv.numel() == cols and lcv.numel() == cols
    ret, cret = torch.empty_like(r), torch.empty_like(r)
    if r.numel() == 0:
        return ret, cret
    nt = None if nonterminal is None else nonterminal.to(torch.uint8).contiguous()
    stream = C.c_void_p(torch.cuda.current_stream(r.device).cuda_stream)
    with torch.cuda.device(r.device):
        _cabi.check(lib.mapf_gae2(_ptr(r), _ptr(v), _ptr(lv), _ptr(cr), _ptr(cv), _ptr(lcv), _ptr(nt), float(gamma), float(lam),
                                  T, cols, _ptr(ret), _ptr(cret), None, None, stream), "mapf_gae2")
    return ret, cret


def sample_actions(ps: torch.Tensor, seed: int = 1234, draw: int = 0, out: Optional[torch.Tensor] = None,
                   chosen_p: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Joint-action sampling on device (model.py:38-40): ps f32 [..., 5] -> int8 [...] actions."""
    lib = _cabi.load_library()
    assert ps.is_cuda and ps.dtype == torch.float32 and ps.shape[-1] == 5
    p = ps.contiguous()
    rows = p.numel() // 5
    if out is None:
        out = torch.empty(p.shape[:-1], dtype=torch.int8, device=p.device)
    assert out.is_contiguous() and out.dtype == torch.int8 and out.numel() == rows
    stream = C.c_void_p(torch.cuda.current_stream(p.device).cuda_stream)
    with torch.cuda.device(p.device):
        _cabi.check(lib.mapf_sample_actions(_ptr(p), rows, int(seed) & (2 ** 64 - 1), int(draw) & 0xffffffff, _ptr(out),
                                            _ptr(chosen_p), stream), "mapf_sample_actions")
    return out
