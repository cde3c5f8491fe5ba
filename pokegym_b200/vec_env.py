"""Drop-in Python boundary: `Environment` (pokegym's single-env Gymnasium API) and `VecEnvironment`
(N envs on one GPU, tensors in / tensors out), both over the CUDA library through the C ABI.

Reference interface mirrored here (/root/reference/pokegym/environment.py):
  Environment(rom_path, state_path, headless, save_video, quiet, verbose, **kw)            :437-446
  reset(seed=None, options=None, max_episode_steps=20480, reward_scale=4.0) -> (obs, {})   :1233,1334
  step(action, fast_video=True) -> (obs, reward, done, done, info)                         :1336,1812
  render() -> obs, close(), observation_space Box(0,255,(72,80,4),uint8), action_space Discrete(8)  :154-167,256,412

There is no CPU fallback: constructing either class needs libgbenv.so and a CUDA device.
"""
from __future__ import annotations

import os
from pathlib import Path
from typing import Iterable, Optional, Sequence, Union

import numpy as np

from . import _capi
from .frames import FrameRecorder, check_channels, decode_target, host_env_ids
from .info import INFO_NAMES, build_info, build_info_from_events, info_row_to_dict, unpack_event_words  # noqa: F401

try:  # gymnasium is not installed in this image; use it when it is
    from gymnasium.spaces import Box, Discrete  # type: ignore
except Exception:  # pragma: no cover - exercised implicitly

    class Box:  # minimal stand-in with the attributes vectorisers read
        def __init__(self, low, high, shape=None, dtype=np.uint8):
            self.low, self.high, self.shape, self.dtype = low, high, tuple(shape), np.dtype(dtype)

        def sample(self):
            return np.random.randint(self.low, self.high + 1, size=self.shape).astype(self.dtype)

        def contains(self, x):
            x = np.asarray(x)
            return x.shape == self.shape and x.dtype == self.dtype

    class Discrete:
        def __init__(self, n):
            self.n = int(n)
            self.shape = ()
            self.dtype = np.dtype(np.int64)

        def sample(self):
            return int(np.random.randint(self.n))

        def contains(self, x):
            return 0 <= int(x) < self.n


OBS_SHAPE = (_capi.OBS_H, _capi.OBS_W, _capi.OBS_C)
OBS_FORMATS = ("reference", "packed")
_LIB = None


def _lib() -> _capi.GbEnvLib:
    global _LIB
    if _LIB is None:
        _LIB = _capi.GbEnvLib(_capi.DEFAULT_LIB)  # raises GbEnvError when the CUDA library is missing
    return _LIB


def _default_state() -> Optional[Path]:
    """The save-state pokegym.Environment falls back to when state_path is None (environment.py:119-120 loads the packaged
    current_state/Bulbasaur.state): $POKEGYM_STATE, else that file inside an installed / checked-out pokegym package."""
    env = os.environ.get("POKEGYM_STATE")
    if env and Path(env).exists():
        return Path(env)
    try:
        import importlib.util

        spec = importlib.util.find_spec("pokegym")
        if spec and spec.origin:
            p = Path(spec.origin).parent / "current_state" / "Bulbasaur.state"
            if p.exists():
                return p
    except Exception:
        pass
    p = Path("/root/reference/pokegym/current_state/Bulbasaur.state")
    return p if p.exists() else None


def _read_rom(rom_path: Union[str, os.PathLike, bytes]) -> bytes:
    if isinstance(rom_path, (bytes, bytearray)):
        return bytes(rom_path)
    p = Path(rom_path)
    if p.exists():
        return p.read_bytes()
    env = os.environ.get("POKEGYM_ROM")
    if env and Path(env).exists():
        return Path(env).read_bytes()
    raise FileNotFoundError(
        f"ROM {rom_path!r} not found (pokegym expects a user-supplied pokemon_red.gb; set POKEGYM_ROM, or pass "
        f"pokegym_b200.tools.synth_rom.build_pokelike_rom() for the synthetic test ROM)"
    )


def device_mask(mask, n: int, device, what: str = "mask"):
    """An env mask as the library reads it: a contiguous uint8 tensor of n entries on `device`, or None for all envs.
    Accepts a bool / integer tensor (e.g. the `done` of a step, which then stays on the device) or an array-like."""
    if mask is None:
        return None
    import torch

    if not torch.is_tensor(mask):
        mask = torch.as_tensor(np.ascontiguousarray(mask, dtype=np.uint8), device=device)
    if mask.dtype == torch.bool:
        mask = mask.to(torch.uint8)
    if mask.dtype != torch.uint8 or mask.device != device or not mask.is_contiguous() or mask.numel() != n:
        mask = mask.to(device=device, dtype=torch.uint8).contiguous().view(-1)
        if mask.numel() != n:
            raise ValueError(f"{what} mask must have {n} entries")
    return mask


def event_counts_from_flags(torch, flags, mask, out):
    """int64 [130] `out` = how many rows of `flags` (int32 [n, 5] gbenv_event_flags rows, on the device) with mask[e] != 0
    (mask None: all) have each event flag set.  Device work only: no host synchronisation."""
    k = torch.arange(_capi.EVENT_FLAGS, device=flags.device)
    bits = (flags[:, k >> 5] >> (k & 31).to(torch.int32)) & 1  # [n, 130] int32
    if mask is not None:
        bits = bits * mask.to(torch.int32)[:, None]
    return torch.sum(bits, dim=0, dtype=torch.int64, out=out)


def check_out(torch, out, shape, dtype, device):
    """`out` for a result of `shape` / `dtype`: a new tensor on `device`, or the caller's, checked (raw pointers cross the
    C ABI, so a wrong layout would be out-of-bounds device writes, not an exception)."""
    if out is None:
        return torch.empty(shape, dtype=dtype, device=device)
    if not (torch.is_tensor(out) and out.dtype == dtype and out.device == device and out.is_contiguous() and tuple(out.shape) == tuple(shape)):
        raise ValueError(f"out must be a contiguous {dtype} tensor {list(shape)} on {device}")
    return out


class VecEnvironment:
    """N Game Boy envs on one GPU.  All tensors live on `device`; nothing returns to the host per step.

    obs      uint8 [N, 72, 80, 4]  (a view into `rollout[t]` when a rollout tensor is supplied)
    reward   float64 [N]           (the reference returns Python floats)
    done     bool [N]              (terminated == truncated in the reference)

    obs_format="packed" stores each observation in 2,304 B instead of 23,040 (include/gbenv.h has the layout): reset() and
    step() return uint8 [N, 2304], a rollout is [T, N, 2304], and unpack_obs() turns any set of those rows back into the
    reference observations on the device, bit for bit.
    """

    def __init__(self, num_envs: int, rom_path, state_paths: Union[None, str, bytes, Sequence] = None, device="cuda:0", rollout=None,
                 auto_reset: bool = False, max_episode_steps: int = 20480, reward_scale: float = 4.0, boot_frames: int = 60,
                 validate_actions: bool = False, obs_format: str = "reference"):
        import torch

        if obs_format not in OBS_FORMATS:
            raise ValueError(f"obs_format must be one of {OBS_FORMATS}, not {obs_format!r}")

        self.torch = torch
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _capi.GbEnvError("VecEnvironment runs on CUDA devices only (there is no CPU fallback)")
        self.num_envs = int(num_envs)
        self.handle = _capi.Handle(_lib(), self.num_envs, _read_rom(rom_path), device_id=self.device.index or 0)
        self.packed = obs_format == "packed"
        self._obs_shape = (_capi.OBS_PACKED_BYTES,) if self.packed else OBS_SHAPE  # one env's observation as step() returns it
        self.observation_space = Box(low=0, high=255, shape=self._obs_shape, dtype=np.uint8)
        self.action_space = Discrete(_capi.NUM_ACTIONS)
        self.max_episode_steps, self.reward_scale, self.auto_reset = int(max_episode_steps), float(reward_scale), bool(auto_reset)
        self.rollout = rollout
        self.validate_actions = bool(validate_actions)  # off by default: the check is a device->host sync; the kernel masks actions with & 7
        self._t = 0
        self._recorder = None
        with torch.cuda.device(self.device):
            self._obs = torch.zeros((self.num_envs, *self._obs_shape), dtype=torch.uint8, device=self.device)
            self._reward = torch.zeros(self.num_envs, dtype=torch.float64, device=self.device)
            self._done = torch.zeros(self.num_envs, dtype=torch.uint8, device=self.device)
            self._done_prev = torch.zeros(self.num_envs, dtype=torch.uint8, device=self.device)
            self._info = torch.zeros((self.num_envs, _capi.INFO_SCALARS), dtype=torch.float64, device=self.device)
        if state_paths is None:
            # no save-state: boot the ROM for a few frames so every env sits in its main loop
            self.handle.tick(boot_frames, True, stream=self._stream())
        else:
            blobs = [state_paths] if isinstance(state_paths, (str, bytes, os.PathLike)) else list(state_paths)
            tids = [self.handle.add_state_template(b if isinstance(b, bytes) else Path(b).read_bytes()) for b in blobs]
            if len(tids) == 1:
                self.handle.set_initial_template(tids[0])
            else:  # env i starts from state i mod len(states) (BASELINE.json config 5)
                for k, tid in enumerate(tids):
                    ids = np.arange(k, self.num_envs, len(tids), dtype=np.int32)
                    if ids.size:
                        self.handle.set_initial_template(tid, ids)

    # -- helpers -------------------------------------------------------------
    def _stream(self) -> int:
        return int(self.torch.cuda.current_stream(self.device).cuda_stream)

    def _obs_target(self):
        if self.rollout is None:
            return self._obs
        r = self.rollout
        ok = (self.torch.is_tensor(r) and r.dtype == self.torch.uint8 and r.device == self.device and r.is_contiguous() and r.dim() >= 3
              and r.shape[1] == self.num_envs)
        if self.packed:
            if not (ok and r.dim() == 3 and r.shape[2] == _capi.OBS_PACKED_BYTES):
                raise ValueError(f"rollout must be a contiguous uint8 tensor [T, {self.num_envs}, {_capi.OBS_PACKED_BYTES}] on {self.device}")
            return r[self._t % r.shape[0]]
        ok = ok and r[0, 0].numel() == _capi.OBS_BYTES
        if not ok:  # raw pointers cross the C ABI: a wrong layout would be out-of-bounds device writes, not an exception
            raise ValueError(f"rollout must be a contiguous uint8 tensor [T, {self.num_envs}, 72, 80, 4] (or [T, N, 23040]) on {self.device}")
        return r[self._t % r.shape[0]]

    def _reset_into(self, obs, mask):
        if self.packed:
            self.handle.reset_packed(obs, mask_dev=mask, max_episode_steps=self.max_episode_steps, reward_scale=self.reward_scale,
                                     stream=self._stream())
        else:
            self.handle.reset_dev(obs, mask_dev=mask, max_episode_steps=self.max_episode_steps, reward_scale=self.reward_scale,
                                  obs_stride=_capi.OBS_BYTES, stream=self._stream())

    # -- API -----------------------------------------------------------------
    def reset(self, mask=None, max_episode_steps: Optional[int] = None, reward_scale: Optional[float] = None):
        """Environment.reset for every env (or those with mask[e] != 0).  Returns (obs, {}); obs is [N, 2304] when packed."""
        if max_episode_steps is not None:
            self.max_episode_steps = int(max_episode_steps)
        if reward_scale is not None:
            self.reward_scale = float(reward_scale)
        obs = self._obs_target()
        self._reset_into(obs, device_mask(mask, self.num_envs, self.device, "reset"))
        return obs.view(self.num_envs, *self._obs_shape), {}

    def step(self, actions, skip=None):
        """Environment.step for every env.  `actions`: uint8/int tensor [N] on the device (or array-like).
        `skip` (uint8 device tensor [N], optional): envs with skip[e] != 0 sit this step out -- reward 0, done False, their
        observation row keeps what it holds (e.g. the reset observation just written by reset(mask=...))."""
        torch = self.torch
        if not torch.is_tensor(actions):
            actions = torch.as_tensor(np.asarray(actions), device=self.device)
        if actions.dtype != torch.uint8 or actions.device != self.device or not actions.is_contiguous():
            actions = actions.to(device=self.device, dtype=torch.uint8).contiguous()
        if actions.numel() != self.num_envs:
            raise ValueError(f"expected {self.num_envs} actions, got {actions.numel()}")
        if self.validate_actions and bool((actions >= _capi.NUM_ACTIONS).any()):  # the reference raises IndexError (ACTIONS[action])
            raise IndexError("action out of range 0..7")
        self._t += 1
        obs = self._obs_target()
        if self.packed:
            if skip is not None:
                self._check_skip(skip, obs)
            self.handle.step_packed(actions, skip, obs, self._reward, self._done, stream=self._stream())
        elif skip is None:
            self.handle.step(actions, obs, self._reward, self._done, obs_stride=_capi.OBS_BYTES, stream=self._stream())
        else:
            self._check_skip(skip, obs)
            self.handle.step_masked(actions, skip, obs, self._reward, self._done, obs_stride=_capi.OBS_BYTES, stream=self._stream())
        if self._recorder is not None:  # the frames this step ended on, before an auto-reset below
            self._recorder._capture(self._done, self._stream())
        done = self._done.bool()
        if self.auto_reset:
            # envs that just finished are reset on the device, masked by the done vector the step wrote: their row of `obs`
            # becomes the reset observation, as a vectoriser that resets after `done` would deliver it (no host round trip)
            self._done_prev.copy_(self._done)
            self._reset_into(obs, self._done_prev)
        return obs.view(self.num_envs, *self._obs_shape), self._reward, done, done, {}

    def _check_skip(self, skip, obs):
        if skip.dtype != self.torch.uint8 or skip.device != self.device or not skip.is_contiguous() or skip.numel() != self.num_envs:
            raise ValueError(f"skip must be a contiguous uint8 tensor with {self.num_envs} entries on {self.device}")
        if self.rollout is not None:  # a new rollout slot: the rows of the envs that sit out must carry over
            prev = self.rollout[(self._t - 1) % self.rollout.shape[0]]
            obs.view(self.num_envs, -1)[skip.bool()] = prev.view(self.num_envs, -1)[skip.bool()]

    def unpack_obs(self, packed, out=None):
        """uint8 [..., 2304] packed observations on the device (any leading dims: a step's rows, a rollout, a minibatch gathered
        from it) -> uint8 [..., 72, 80, 4], the reference observations gbenv_step would have written, decoded on the device,
        asynchronously.  compact_view applies to the result."""
        torch = self.torch
        if not (torch.is_tensor(packed) and packed.dtype == torch.uint8 and packed.device == self.device and packed.dim() >= 1
                and packed.shape[-1] == _capi.OBS_PACKED_BYTES):
            raise ValueError(f"packed must be a uint8 tensor [..., {_capi.OBS_PACKED_BYTES}] on {self.device}")
        lead = tuple(packed.shape[:-1])
        out = check_out(torch, out, (*lead, *OBS_SHAPE), torch.uint8, self.device)
        if packed.numel():
            self.handle.unpack_obs(packed.contiguous(), out, stream=self._stream())
        return out

    def screens(self, env_ids=None, channels: int = 3, out=None):
        """uint8 [n, 144, 160, channels] device tensor: the current frame of the envs `env_ids` (None: all), grey
        (channels=1) or RGB (3) exactly as screen() / gbenv_screen gives one env.  Captured and decoded on the device,
        asynchronously; the ids are checked on the host (pass a list or array: a device tensor is copied there first)."""
        torch = self.torch
        channels = check_channels(channels)
        ids = None
        n = self.num_envs
        if env_ids is not None:
            a = host_env_ids(env_ids, self.num_envs)
            n = a.size
            ids = torch.from_numpy(a).pin_memory().to(self.device, non_blocking=True)
        out = decode_target(torch, out, n, channels, self.device)
        packed = torch.empty((n, _capi.FRAME_WORDS), dtype=torch.int32, device=self.device)
        self.handle.capture_frames(packed, ids, stream=self._stream())
        self.handle.frames_to_rgb(packed, out, channels, stream=self._stream())
        return out

    def record_frames(self, env_ids, capacity: Optional[int] = None) -> Optional[FrameRecorder]:
        """Records the frame of the envs `env_ids` on every step() from now on into a new FrameRecorder holding the last
        `capacity` steps (uint32 [capacity, len(env_ids), 1440] packed, 5,760 B per frame), and returns it.  It replaces
        the previous recorder; record_frames(None) stops recording."""
        if env_ids is None:
            self._recorder = None
            return None
        if capacity is None:
            raise ValueError("record_frames needs a capacity (steps held)")
        self._recorder = FrameRecorder(self, env_ids, capacity)
        return self._recorder

    @staticmethod
    def compact_view(obs):
        """Optional 1+1-channel view for new policies (SURVEY.md 8b): the reference's channels 0-2 are the same grey level,
        so `obs[..., 2:]` = (grey, visited) carries everything.  A strided view of the same memory, no copy."""
        return obs[..., 2:]

    def info(self):
        """Per-env info rows: float64 [N, 72] (GBENV_INFO_SCALARS); column names in pokegym_b200.info.INFO_NAMES."""
        self.handle.get_info(self._info, stream=self._stream())
        return self._info

    def info_sum(self, out=None, mask=None):
        """Sum of the info rows over this GPU's envs (the vector multi-GPU runs all-reduce); slot 0 counts the envs summed.
        With `mask` (e.g. the `done` that step() returned), only the envs with mask[e] != 0: their rows are those of their
        last step even after auto_reset, so this is the sum a trainer averages over the episodes that just ended."""
        torch = self.torch
        if out is None:
            out = torch.zeros(_capi.INFO_SCALARS, dtype=torch.float64, device=self.device)
        if mask is None:
            self.handle.reduce_info(out, stream=self._stream())
        else:
            self.handle.reduce_info_masked(out, device_mask(mask, self.num_envs, self.device, "info_sum"), stream=self._stream())
        return out

    def exploration_map_sum(self, mask=None, out=None):
        """int64 [444, 436] device tensor: the sum of the envs' `pokemon_exploration_map`s (environment.py:1624), over the
        envs with mask[e] != 0 (e.g. the `done` of step()) or over all.  Computed on the device, nothing goes to the host."""
        torch = self.torch
        out = check_out(torch, out, (_capi.COUNTS_H, _capi.COUNTS_W), torch.int64, self.device)
        self.handle.counts_map_sum(out, device_mask(mask, self.num_envs, self.device, "exploration_map_sum"), stream=self._stream())
        return out

    def event_flags(self, env_ids=None, out=None):
        """int32 [n, 5] device tensor: the 130 event flags of the envs `env_ids` (None: all), bit k & 31 of word k >> 5 being
        entry k of the event table (pokegym_b200.info.event_table, unpack_event_words).  Gathered on the device,
        asynchronously; the ids are checked on the host (pass a list or array: a device tensor is copied there first)."""
        torch = self.torch
        ids = None
        n = self.num_envs
        if env_ids is not None:
            a = host_env_ids(env_ids, self.num_envs)
            n = a.size
            ids = torch.from_numpy(a).pin_memory().to(self.device, non_blocking=True)
        out = check_out(torch, out, (n, _capi.EVENT_WORDS), torch.int32, self.device)
        self.handle.event_flags(out, ids, stream=self._stream())
        return out

    def event_counts(self, mask=None, out=None):
        """int64 [130] device tensor: how many of the envs with mask[e] != 0 (e.g. the `done` of step(); None: all) have
        each event flag set, in event-table order.  Device work only, no host synchronisation; goes through
        dist.all_reduce_info like info_sum, and info.event_counts_to_means turns it into the reference's event dicts."""
        torch = self.torch
        out = check_out(torch, out, (_capi.EVENT_FLAGS,), torch.int64, self.device)
        return event_counts_from_flags(torch, self.event_flags(), device_mask(mask, self.num_envs, self.device, "event_counts"), out)

    def episode_infos(self, mask) -> dict:
        """{env: info dict} for the envs with mask[e] != 0, typically the `done` of step(), in env order.  Each dict is
        full_info(env)'s with `pokemon_exploration_map` None (exploration_map_sum(mask) is the batched overlay).  Also right
        after auto_reset: a reset leaves the info row as the last step wrote it and writes no event flag.
        Two host synchronisations whatever the number of envs: one to find the ids, one copy of their rows and flags."""
        torch = self.torch
        mask = device_mask(mask, self.num_envs, self.device, "episode_infos")
        ids = torch.nonzero(mask).view(-1).to(torch.int32)
        k = ids.numel()
        if k == 0:
            return {}
        flags = torch.empty((k, _capi.EVENT_WORDS), dtype=torch.int32, device=self.device)
        self.handle.event_flags(flags, ids, stream=self._stream())
        rows = self.info()[ids.long()]
        packed = torch.cat([ids.view(torch.uint8).view(k, 4), rows.view(torch.uint8).view(k, -1), flags.view(torch.uint8).view(k, -1)], 1)
        host = packed.cpu().numpy()
        env_ids = host[:, :4].copy().view(np.int32)[:, 0]
        rows_h = host[:, 4:4 + 8 * _capi.INFO_SCALARS].copy().view(np.float64)
        bits = unpack_event_words(host[:, 4 + 8 * _capi.INFO_SCALARS:].copy().view(np.uint32))
        return {int(e): build_info_from_events(rows_h[i], bits[i], counts_map=None, reward_scale=self.reward_scale) for i, e in enumerate(env_ids)}

    def full_info(self, env: int = 0) -> dict:
        """The reference's complete info dict for one env (environment.py:1621-1810): scalar row + the 130 named
        event flags (gbenv_event_flags) + its counts_map.  Rare path (episode end / every 10,000 steps)."""
        row = self.info()[env].cpu().numpy()
        bits = unpack_event_words(self.event_flags([env]))[0]
        try:
            cm = self.handle.counts_map(env).astype(np.float64)
        except _capi.GbEnvError:  # heat maps switched off (GBENV_COUNTS_MAP=0)
            cm = None
        return build_info_from_events(row, bits, counts_map=cm, reward_scale=self.reward_scale)

    def save_state(self, env: int = 0) -> bytes:
        return self.handle.save_state(env)

    def save_states(self, env_ids=None, out=None):
        """uint8 [n, 142610] device tensor: PyBoy.save_state of the envs `env_ids` (None: all), row i being exactly what
        save_state(env_ids[i]) returns.  Serialised on the device, asynchronously on the current stream; the ids are checked
        on the host (pass a list or array: a device tensor is copied there first).  `rows[i].cpu().numpy().tobytes()` is a
        .state file that PyBoy and load_state() both accept.  Each row is 142,610 B (584 MB for 4,096 envs): pass ids to
        save fewer."""
        torch = self.torch
        ids = None
        n = self.num_envs
        if env_ids is not None:
            a = host_env_ids(env_ids, self.num_envs)
            n = a.size
            ids = torch.from_numpy(a).pin_memory().to(self.device, non_blocking=True)
        out = check_out(torch, out, (n, _capi.STATE_BYTES), torch.uint8, self.device)
        self.handle.save_states(out, ids, stream=self._stream())
        return out

    def load_states(self, rows, env_ids=None):
        """PyBoy.load_state of row i of `rows` (uint8 [n, 142610], the layout save_states returns) into env env_ids[i] (None:
        envs 0..n-1), all in one launch on the device, asynchronously on the current stream.  Returns the int32 [n] status
        tensor: 0 where the row was loaded, -2 (GBENV_E_STATE) where it is not a loadable v9 file and the env was left as it
        was.  Of several rows for one env the last loadable one wins.  The ids are checked on the host; rows in host memory,
        on another device, non-contiguous or not 16-byte aligned (a slice rows[k:] usually is not) are copied first.
        This loads emulator state only: rewards, visited bitmaps and info rows stay as they are, and so does the state an
        env's first reset loads.  To start episodes from the loaded states, reset those envs next (reset(mask)); an env whose
        first reset is still ahead loads its initial state there instead.  One state into k envs:
        load_states(row.expand(k, -1).contiguous(), ids)."""
        torch = self.torch
        if not torch.is_tensor(rows):
            rows = torch.from_numpy(np.ascontiguousarray(rows))
        if rows.dim() != 2 or rows.shape[1] != _capi.STATE_BYTES or rows.dtype != torch.uint8:
            raise ValueError(f"rows must be a uint8 tensor or array [n, {_capi.STATE_BYTES}]")
        n = rows.shape[0]
        ids = None
        if env_ids is not None:
            a = host_env_ids(env_ids, self.num_envs)
            if a.size != n:
                raise ValueError(f"{a.size} env ids for {n} rows")
            ids = torch.from_numpy(a).pin_memory().to(self.device, non_blocking=True)
        elif n > self.num_envs:
            raise ValueError(f"{n} rows for {self.num_envs} envs")
        if rows.device != self.device or not rows.is_contiguous() or rows.data_ptr() % 16:
            rows = torch.empty((n, _capi.STATE_BYTES), dtype=torch.uint8, device=self.device).copy_(rows, non_blocking=rows.device.type != "cpu")
        status = torch.empty(n, dtype=torch.int32, device=self.device)
        self.handle.load_states(rows, ids, status, stream=self._stream())
        return status

    def load_state(self, blob: bytes, env_ids=None):
        """PyBoy.load_state for the listed envs (None: all): pyboy_binding.load_pyboy_state (:65-69)."""
        self.handle.load_template(self.handle.add_state_template(blob), env_ids)

    def close(self):
        self.handle.close()


class Environment:
    """pokegym.Environment on the GPU path: a batch of one (the CUDA library is used even for N = 1)."""

    def __init__(self, rom_path="pokemon_red.gb", state_path=None, headless=True, save_video=False, quiet=False, verbose=False, device="cuda:0", **kwargs):
        if save_video or not headless:
            raise NotImplementedError("video / SDL2 window output is out of scope (SURVEY.md section 8b non-goals)")
        if state_path is None and not isinstance(rom_path, (bytes, bytearray)):
            # environment.py:119-120: the reference falls back to its packaged current_state/Bulbasaur.state.  With a ROM
            # given as bytes (the synthetic test ROMs) there is no such convention and the ROM is booted instead.
            state_path = _default_state()
            if state_path is None:
                raise FileNotFoundError("no state_path given and pokegym's default current_state/Bulbasaur.state was not found "
                                        "(set POKEGYM_STATE or pass state_path)")
        self.vec = VecEnvironment(1, rom_path, state_paths=state_path, device=device)
        self.observation_space = self.vec.observation_space
        self.action_space = self.vec.action_space
        self.verbose = verbose
        self.time = 0
        self.max_episode_steps = 20480
        self._actions = self.vec.torch.zeros(1, dtype=self.vec.torch.uint8, device=self.vec.device)

    def reset(self, seed=None, options=None, max_episode_steps=20480, reward_scale=4.0):
        """Resets the game. Seeding is NOT supported (as in the reference)."""
        self.time = 0
        self.max_episode_steps = max_episode_steps
        obs, _ = self.vec.reset(max_episode_steps=max_episode_steps, reward_scale=reward_scale)
        self._last_obs = obs[0].cpu().numpy()
        return self._last_obs, {}

    def step(self, action, fast_video=True):
        self._actions.fill_(int(action))
        obs, reward, done, _, _ = self.vec.step(self._actions)
        self.time += 1
        d = bool(done[0].item())
        info = {}
        if d or self.time % 10000 == 0:  # environment.py:1621
            info = self.vec.full_info(0)
        self._last_obs = obs[0].cpu().numpy()
        return self._last_obs, float(reward[0].item()), d, d, info

    def render(self):
        """The observation the last reset()/step() returned (environment.py:256-274 rebuilds the same array)."""
        return self._last_obs

    # environment.py:208-227: save_state / load_first_state / load_last_state / load_random_state over self.initial_states
    def save_state(self):
        if not hasattr(self, "initial_states"):
            self.initial_states = []
        self.initial_states.append(self.vec.save_state(0))

    def load_first_state(self):
        return self.initial_states[0]

    def load_last_state(self):
        return self.initial_states[-1]

    def load_random_state(self):
        import random

        return self.initial_states[random.randrange(len(self.initial_states))]

    def close(self):
        self.vec.close()
