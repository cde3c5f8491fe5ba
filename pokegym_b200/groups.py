"""Env groups: one batch of envs held as G independent handles that step on G CUDA streams.

Why: the emulation kernel of a step ends with its slowest env (an env-step that runs into a busy stretch of the game
executes ~25 % more instructions than the typical one), so a single handle leaves the GPU partly idle at the end of every
launch.  With the batch split into groups whose kernels are queued on separate streams, the tail of one group's launch is
filled by the other groups' work.  This is what an asynchronous vectoriser does anyway (PufferLib steps one half of its envs
while the policy looks at the other half); nothing about a single env changes -- the groups are ordinary handles of the C ABI
(include/gbenv.h) and env i of the batch is env i - g * n of group g = i // n.

    groups = EnvGroups(lib, 4096, rom, n_groups=2)
    groups.reset(obs)                              # obs u8[E, 23040] on the device
    groups.step(actions, obs, reward, done)        # queues every group's step; returns at once
    groups.join()                                  # the caller's stream now waits for all groups (before reading obs ...)

With obs_format="packed" the observation rows are u8[E, 2304] (include/gbenv.h, VecEnvironment.unpack_obs decodes them).

Measured on B200 (tools/exp_groups.py): 4,096 envs 141.5 k env-steps/s as one group, 152.6 k as two, 144.1 k as four;
32,768 envs (16 per warp: latency bound, a freed SM does not make the remaining warps faster) gain nothing.
"""
from __future__ import annotations

from typing import List, Optional

from . import _capi
from .vec_env import OBS_FORMATS, device_mask, event_counts_from_flags


class EnvGroups:
    def __init__(self, lib: _capi.GbEnvLib, num_envs: int, rom: bytes, n_groups: int = 2, device_id: int = 0, lanes: Optional[int] = None,
                 obs_format: str = "reference"):
        import torch

        if n_groups < 1 or num_envs % n_groups:
            raise ValueError("num_envs must be a multiple of n_groups")
        if obs_format not in OBS_FORMATS:
            raise ValueError(f"obs_format must be one of {OBS_FORMATS}, not {obs_format!r}")
        self.packed = obs_format == "packed"
        self.torch = torch
        self.device = torch.device("cuda", device_id)
        self.num_envs, self.n_groups, self.n = int(num_envs), int(n_groups), int(num_envs) // int(n_groups)
        self.handles: List[_capi.Handle] = [_capi.Handle(lib, self.n, rom, device_id=device_id) for _ in range(n_groups)]
        with torch.cuda.device(self.device):
            self.streams = [torch.cuda.Stream(device=self.device) for _ in range(n_groups)]
            self._ready = [torch.cuda.Event() for _ in range(n_groups)]
            self._done = [torch.cuda.Event() for _ in range(n_groups)]
            self._info_parts = torch.zeros((n_groups, _capi.INFO_SCALARS), dtype=torch.float64, device=self.device)
        self._map_parts = None  # [n_groups, 444, 436] int64, allocated by the first exploration_map_sum
        self._flags = None  # [num_envs, 5] int32, allocated by the first event_counts
        if lanes:
            for h in self.handles:
                h.set_lanes_per_warp(lanes)

    # -- plumbing ------------------------------------------------------------------------------------------------
    def _slice(self, t, g):
        return None if t is None else t[g * self.n:(g + 1) * self.n]

    def _fork(self):
        """every group stream waits for what the caller's stream has queued so far (the inputs of this call)"""
        cur = self.torch.cuda.current_stream(self.device)
        for g, s in enumerate(self.streams):
            self._ready[g].record(cur)
            s.wait_event(self._ready[g])

    def join(self):
        """the caller's current stream waits for everything queued on the group streams"""
        cur = self.torch.cuda.current_stream(self.device)
        for g, s in enumerate(self.streams):
            self._done[g].record(s)
            cur.wait_event(self._done[g])

    def for_each(self, fn):
        """fn(handle, group index, stream handle) for every group (state templates, ticks ...)"""
        for g, (h, s) in enumerate(zip(self.handles, self.streams)):
            fn(h, g, s.cuda_stream)

    # -- the env API, batched over the groups ---------------------------------------------------------------------
    def reset(self, obs, mask=None, **kw):
        self._fork()
        for g, (h, s) in enumerate(zip(self.handles, self.streams)):
            m = self._slice(mask, g)
            if self.packed:
                h.reset_packed(self._slice(obs, g), m, stream=s.cuda_stream, **kw)
            elif m is None:
                h.reset(self._slice(obs, g), stream=s.cuda_stream, **kw)
            else:
                h.reset_dev(self._slice(obs, g), m, stream=s.cuda_stream, **kw)
        self.join()

    def step(self, actions, obs, reward, done, join: bool = False):
        """Queue one env-step of every group (24 frames + reward + observation).  actions u8[E], obs u8[E, 23040] (packed: u8[E, 2304]), reward
        f64[E], done u8[E], all on the device; group g uses rows [g * n, (g + 1) * n).  With join=False the call returns with
        the groups still running: call join() before the caller's stream reads the outputs."""
        self._fork()
        for g, (h, s) in enumerate(zip(self.handles, self.streams)):
            a, o, r, d = (self._slice(t, g) for t in (actions, obs, reward, done))
            if self.packed:
                h.step_packed(a, None, o, r, d, stream=s.cuda_stream)
            else:
                h.step(a, o, r, d, stream=s.cuda_stream)
        if join:
            self.join()

    def reduce_info(self, out, mask=None):
        """sum of the 72-double info rows over every env of every group -> out (on the caller's stream, after a join); with
        `mask` (u8 / bool [E], e.g. the step's done) over the envs with mask[e] != 0 only"""
        mask = device_mask(mask, self.num_envs, self.device, "reduce_info")
        self._fork()
        for g, (h, s) in enumerate(zip(self.handles, self.streams)):
            h.reduce_info_masked(self._info_parts[g], self._slice(mask, g), stream=s.cuda_stream)
        self.join()
        self.torch.sum(self._info_parts, dim=0, out=out)
        return out

    def exploration_map_sum(self, out, mask=None):
        """int64 [444, 436] sum of the heat maps of every env (or those with mask[e] != 0) of every group -> out (on the
        caller's stream, after a join)"""
        mask = device_mask(mask, self.num_envs, self.device, "exploration_map_sum")
        if self._map_parts is None:
            self._map_parts = self.torch.empty((self.n_groups, _capi.COUNTS_H, _capi.COUNTS_W), dtype=self.torch.int64, device=self.device)
        self._fork()
        for g, (h, s) in enumerate(zip(self.handles, self.streams)):
            h.counts_map_sum(self._map_parts[g], self._slice(mask, g), stream=s.cuda_stream)
        self.join()
        self.torch.sum(self._map_parts, dim=0, out=out)
        return out

    def event_counts(self, out, mask=None):
        """int64 [130] count of the envs of every group (or those with mask[e] != 0) that have each event flag set -> out (on
        the caller's stream, after a join)"""
        mask = device_mask(mask, self.num_envs, self.device, "event_counts")
        if self._flags is None:
            self._flags = self.torch.empty((self.num_envs, _capi.EVENT_WORDS), dtype=self.torch.int32, device=self.device)
        self._fork()
        for g, (h, s) in enumerate(zip(self.handles, self.streams)):
            h.event_flags(self._slice(self._flags, g), stream=s.cuda_stream)
        self.join()
        return event_counts_from_flags(self.torch, self._flags, mask, out)

    # -- counters --------------------------------------------------------------------------------------------------
    def counters(self):
        cs = [h.counters() for h in self.handles]
        out = _capi.Counters()
        for name, _ in _capi.Counters._fields_:
            setattr(out, name, sum(getattr(c, name) for c in cs))
        return out

    def kernel_time_total(self, which: int = 0):
        parts = [h.kernel_time_total(which) for h in self.handles]
        return sum(p[0] for p in parts), sum(p[1] for p in parts)

    def lanes_per_warp(self) -> int:
        return self.handles[0].lanes_per_warp()

    def close(self):
        for h in self.handles:
            h.close()
        self.handles = []
